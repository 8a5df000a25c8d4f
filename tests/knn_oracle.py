"""CPU oracle of K-nearest-neighbour search (tests/knn_oracle.c) and its independent numpy restatement.  TEST
INFRASTRUCTURE ONLY.  The C file is compiled on first use into a private temporary directory (the tree may be
read-only), with the flags of oracle/Makefile."""
import atexit
import ctypes
import os
import shutil
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_lib = None

_f32p = ctypes.POINTER(ctypes.c_float)
_i32p = ctypes.POINTER(ctypes.c_int)
_i64p = ctypes.POINTER(ctypes.c_int64)
_u64p = ctypes.POINTER(ctypes.c_uint64)


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="knn_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "libknn_oracle.so")
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        subprocess.run([cc, "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra",
                        "-o", so, os.path.join(_HERE, "knn_oracle.c"), "-lm"], check=True)
        _lib = ctypes.CDLL(so)
        _lib.knn_oracle_forward.restype = ctypes.c_int
        _lib.knn_oracle_backward.restype = ctypes.c_int
    return _lib


def _np32(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().float().numpy()
    a = np.asarray(a, dtype=np.float32)
    if a.strides[-1] != 4:
        a = np.ascontiguousarray(a)
    return a


def _lens(lengths, b):
    if lengths is None:
        return None
    if hasattr(lengths, "detach"):
        lengths = lengths.detach().cpu().numpy()
    a = np.ascontiguousarray(np.asarray(lengths, dtype=np.int64))
    assert a.shape == (b,)
    return a


def _args(x):
    return _ptr(x, _f32p), ctypes.c_long(x.strides[0] // 4), ctypes.c_long(x.strides[1] // 4)


def _ptr(a, t):
    return None if a is None else a.ctypes.data_as(t)


def knn_forward(p1, p2, K, lengths1=None, lengths2=None, mode=0):
    """-> (dists (B,P1,K) fp32, idx (B,P1,K) int32), see knn_oracle.c."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, d = a.shape
    n2 = b.shape[1]
    l1, l2 = _lens(lengths1, bsz), _lens(lengths2, bsz)
    dists = np.zeros((bsz, n1, K), np.float32)
    idx = np.zeros((bsz, n1, K), np.int32)
    scratch = np.zeros(K, np.uint64)
    rc = lib().knn_oracle_forward(*_args(a), _ptr(l1, _i64p), *_args(b), _ptr(l2, _i64p), bsz, n1, n2, d, K, mode,
                                  _ptr(dists, _f32p), _ptr(idx, _i32p), _ptr(scratch, _u64p))
    if rc != 0:
        raise ValueError(f"knn_oracle_forward rc={rc}")
    return dists, idx


def knn_backward(p1, p2, idx, grad_dists, lengths1=None, lengths2=None):
    """-> (grad_p1 (B,P1,D), grad_p2 (B,P2,D)) fp32, sequential accumulation (knn_oracle.c)."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, d = a.shape
    n2 = b.shape[1]
    ix = np.ascontiguousarray(np.asarray(idx, dtype=np.int32))
    g = np.ascontiguousarray(_np32(grad_dists))
    K = ix.shape[2]
    l1, l2 = _lens(lengths1, bsz), _lens(lengths2, bsz)
    g1 = np.zeros((bsz, n1, d), np.float32)
    g2 = np.zeros((bsz, n2, d), np.float32)
    rc = lib().knn_oracle_backward(*_args(a), _ptr(l1, _i64p), *_args(b), _ptr(l2, _i64p), bsz, n1, n2, d, K,
                                   _ptr(ix, _i32p), _ptr(g, _f32p), _ptr(g1, _f32p), _ptr(g2, _f32p))
    assert rc == 0
    return g1, g2


def knn_numpy(p1, p2, K, lengths1=None, lengths2=None):
    """Independent restatement (unfused arithmetic only): the dense fp32 distance matrix in the same operation order,
    then a lexicographic sort by (distance bits with NaN -> 0x7fffffff, index) per query."""
    a, b = _np32(p1), _np32(p2)
    bsz, n1, d = a.shape
    n2 = b.shape[1]
    dists = np.zeros((bsz, n1, K), np.float32)
    idx = np.zeros((bsz, n1, K), np.int32)
    for n in range(bsz):
        l1 = n1 if lengths1 is None else int(lengths1[n])
        l2 = n2 if lengths2 is None else int(lengths2[n])
        if l1 == 0 or l2 == 0:
            continue
        diff = a[n, :l1, None, :] - b[n, None, :l2, :]           # (l1, l2, d) fp32
        dm = np.zeros((l1, l2), np.float32)
        for c in range(d):
            dm = dm + diff[..., c] * diff[..., c]                  # ((0 + dx*dx) + dy*dy) + ..., each op rounded to fp32
        bits = dm.view(np.uint32).copy()
        bits[np.isnan(dm)] = 0x7FFFFFFF
        j = np.broadcast_to(np.arange(l2), (l1, l2))
        order = np.lexsort((j, bits), axis=-1)[:, :K]
        kv = order.shape[1]
        idx[n, :l1, :kv] = order
        dists[n, :l1, :kv] = np.take_along_axis(bits, order, 1).view(np.float32)
    return dists, idx
