"""CPU oracle of ball query (tests/ball_query_oracle.c) and its independent restatements.  TEST INFRASTRUCTURE ONLY.
The C file is compiled on first use into a private temporary directory (the tree may be read-only), with the flags of
oracle/Makefile."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

import knn_oracle as ko
from knn_oracle import _args, _f32p, _i32p, _i64p, _lens, _np32, _ptr

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="ball_query_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libball_query_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                        "-o", so, os.path.join(_HERE, "ball_query_oracle.c"), "-lm"], check=True)
        _lib = ctypes.CDLL(so)
        _lib.ball_query_oracle_forward.restype = ctypes.c_int
    return _lib


def radius2(radius):
    """float32(radius) * float32(radius) rounded to fp32, as pointcloud_b200.ball_query computes it."""
    r = np.float32(radius)
    return np.float32(r * r)


def ball_query_forward(p1, p2, K, r2, lengths1=None, lengths2=None, mode=0):
    """-> (dists (B,P1,K) fp32, idx (B,P1,K) int32) for the fp32 comparison value r2, see ball_query_oracle.c."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, d = a.shape
    n2 = b.shape[1]
    l1, l2 = _lens(lengths1, bsz), _lens(lengths2, bsz)
    dists = np.zeros((bsz, n1, K), np.float32)
    idx = np.zeros((bsz, n1, K), np.int32)
    rc = lib().ball_query_oracle_forward(*_args(a), _ptr(l1, _i64p), *_args(b), _ptr(l2, _i64p), bsz, n1, n2, d, K,
                                         ctypes.c_float(r2), mode, _ptr(dists, _f32p), _ptr(idx, _i32p))
    if rc != 0:
        raise ValueError(f"ball_query_oracle_forward rc={rc}")
    return dists, idx


def ball_query_numpy(p1, p2, K, r2, lengths1=None, lengths2=None):
    """Independent restatement (unfused arithmetic only): the dense fp32 distance matrix in the same operation order,
    then the first K indices with d < r2 per query."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, d = a.shape
    n2 = b.shape[1]
    dists = np.zeros((bsz, n1, K), np.float32)
    idx = np.full((bsz, n1, K), -1, np.int32)
    for n in range(bsz):
        l1 = n1 if lengths1 is None else int(lengths1[n])
        l2 = n2 if lengths2 is None else int(lengths2[n])
        if l1 == 0 or l2 == 0:
            continue
        diff = a[n, :l1, None, :] - b[n, None, :l2, :]
        dm = np.zeros((l1, l2), np.float32)
        for c in range(d):
            dm = dm + diff[..., c] * diff[..., c]
        for i in range(l1):
            js = np.nonzero(dm[i] < np.float32(r2))[0][:K]
            idx[n, i, :len(js)] = js
            dists[n, i, :len(js)] = dm[i, js]
    return dists, idx


def ball_query_from_knn(p1, p2, K, r2, lengths1=None, lengths2=None, mode=0):
    """The kNN oracle with K = P2 (every target, ranked by (distance, index)), filtered to d < r2, re-ordered by index and
    truncated to K."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, _ = a.shape
    n2 = b.shape[1]
    dists = np.zeros((bsz, n1, K), np.float32)
    idx = np.full((bsz, n1, K), -1, np.int32)
    if n2 == 0:
        return dists, idx
    kd, ki = ko.knn_forward(a, b, n2, lengths1, lengths2, mode=mode)
    for n in range(bsz):
        l1 = n1 if lengths1 is None else int(lengths1[n])
        l2 = n2 if lengths2 is None else int(lengths2[n])
        for i in range(l1):
            dd, jj = kd[n, i, :l2], ki[n, i, :l2]
            keep = dd < np.float32(r2)
            order = np.argsort(jj[keep], kind="stable")[:K]
            idx[n, i, :len(order)] = jj[keep][order]
            dists[n, i, :len(order)] = dd[keep][order]
    return dists, idx
