"""Build libusip_b200.so (the C-ABI library declared in include/usip_b200.h) in-tree with nvcc for
sm_100a.  `python -m usip_b200.build [-f]`.  No torch headers are involved: the kernels only see raw
pointers, so a full rebuild takes a few seconds and cross-compiles without a GPU."""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_DIR = os.path.join(_HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libusip_b200.so")
SOURCES = ["api.cu", "group.cu", "indexmax.cu", "ballquery.cu", "ballgroup.cu", "knngroup.cu", "loss.cu", "nngrid.cu", "mlp.cu", "mlp_tc.cu", "backward.cu", "wgrad_tc.cu", "fps.cu", "nms.cu", "optim.cu", "registration.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
# per-source additions: the registration kernels evaluate one float64 rigid fit in two kernels and need the same bits in
# both, so no multiply-add is contracted there
SOURCE_FLAGS = {"registration.cu": ["-fmad=false"]}


def _nvcc():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.sep not in p or os.path.isfile(p)):
            return p
    raise RuntimeError("nvcc not found")


def _stale(out, deps):
    if not os.path.isfile(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(LIB_DIR, exist_ok=True)
    objdir = os.path.join(LIB_DIR, "obj")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(_HERE, "..", "include", "usip_b200.h"))
    srcs = [s for s in SOURCES if os.path.isfile(os.path.join(CSRC, s))]
    nvcc = _nvcc()

    def compile_one(s):
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + headers):
            cmd = [nvcc] + NVCC_FLAGS + SOURCE_FLAGS.get(s, []) + os.environ.get("USIP_NVCC_EXTRA", "").split() + ["-c", src, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError("nvcc failed on %s:\n%s\n%s" % (s, r.stdout, r.stderr))
            return obj, True
        return obj, False

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        results = list(ex.map(compile_one, srcs))
    objs = [o for o, _ in results]
    if force or any(c for _, c in results) or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcuda"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="-f" in sys.argv, verbose="-v" in sys.argv))
