"""Build libpcl_b200.so in-tree with nvcc for sm_100a (no JIT cache: the .so travels with the repo)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.environ.get("PCL_LIB_OVERRIDE") or os.path.join(HERE, "libpcl_b200.so")  # override: development A/B builds
SOURCES = ["pcl_api.cu", "pcl_chamfer.cu", "pcl_emd.cu", "pcl_emd_team.cu", "pcl_epilogue.cu", "pcl_sampling.cu", "pcl_knn.cu", "pcl_normals.cu", "pcl_icp.cu", "pcl_volumes.cu", "pcl_raster.cu"]
HEADERS = [os.path.join(CSRC, "pcl_common.cuh"), os.path.join(CSRC, "pcl_nn.cuh"), os.path.join(CSRC, "pcl_emd_core.cuh"), os.path.join(CSRC, "pcl_emd_tasks.cuh"), os.path.join(HERE, "..", "include", "pcl.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--expt-relaxed-constexpr"]


def _nvcc():
    cand = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    return cand if os.path.exists(cand) else "nvcc"


def needs_build() -> bool:
    if os.environ.get("PCL_LIB_OVERRIDE"):
        return False
    if not os.path.exists(LIB):
        return True
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS
    return any(os.path.exists(d) and os.path.getmtime(d) > os.path.getmtime(LIB) for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB
    # several ranks of one node may get here at the same time (torchrun on a fresh checkout): one builds, the others wait
    import fcntl
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not needs_build():
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    objdir = os.path.join(HERE, "_build")
    os.makedirs(objdir, exist_ok=True)
    env = dict(os.environ)
    # the image exports CC=/opt/gcc/bin/gcc; nvcc must use the system host compiler
    ccbin = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [_nvcc(), "-ccbin", ccbin, *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        procs.append((s, obj, subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for s, obj, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {s}")
        objs.append(obj)
    tmp = f"{LIB}.tmp{os.getpid()}"
    cmd = [_nvcc(), "-ccbin", ccbin, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp, *objs]
    subprocess.run(cmd, check=True, env=env)
    os.replace(tmp, LIB)  # atomic: a concurrent reader never sees a half-written library
    return LIB


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
