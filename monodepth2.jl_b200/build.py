"""In-tree nvcc build of libmd2_b200.so (sm_100a only; cross-compiles without a GPU).  Every translation unit is
compiled to its own object file (in parallel, only when stale) and the objects are linked into the shared library."""
import hashlib
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(CSRC, "_obj")
LIB = os.path.join(CSRC, "libmd2_b200.so")
SOURCES = ["md2_fused.cu", "md2_ops.cu", "md2_host.cu", "md2_optim.cu"]
HEADERS = ["md2_math.cuh", "md2_fused.cuh", "md2_march.cuh", "md2_march2.cuh", "md2_common.cuh",
           os.path.join("..", "..", "include", "md2.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--cudart", "shared", "-split-compile", "0"]


def _mtime(f):
    p = os.path.join(CSRC, f)
    return os.path.getmtime(p) if os.path.exists(p) else 0.0


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("MD2_NVCC_EXTRA", "").split()   # tuning experiments, e.g. -DMD2_PREFETCH=0
    missing = [f for f in SOURCES + HEADERS if not os.path.exists(os.path.join(CSRC, f))]
    if missing:
        raise RuntimeError(f"nvcc build: missing source files {missing}")
    tag = hashlib.sha1(" ".join(NVCC_FLAGS + extra).encode()).hexdigest()[:10]    # objects of other flag sets are not reused
    os.makedirs(OBJ, exist_ok=True)
    hdr_t = max(_mtime(h) for h in HEADERS)
    objs, todo = [], []
    for s in SOURCES:
        o = os.path.join(OBJ, f"{os.path.splitext(s)[0]}.{tag}.o")
        objs.append(o)
        if force or not os.path.exists(o) or os.path.getmtime(o) < max(_mtime(s), hdr_t):
            todo.append((s, o))

    def compile_one(job):
        s, o = job
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", o, s]
        return s, subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)

    if todo:
        with ThreadPoolExecutor(max_workers=len(todo)) as ex:
            for s, r in ex.map(compile_one, todo):
                if r.returncode != 0:
                    raise RuntimeError(f"nvcc build of {s} failed:\n" + r.stdout + r.stderr)
                if verbose:
                    print(r.stderr)
    # (the library remembers which flag set it was linked from: a tuning build must not survive as the default library)
    stamp = os.path.join(OBJ, "linked.tag")
    linked = open(stamp).read().strip() if os.path.exists(stamp) else ""
    if todo or linked != tag or not os.path.exists(LIB) or any(os.path.getmtime(o) > os.path.getmtime(LIB) for o in objs):
        r = subprocess.run([nvcc, "-shared", "--cudart", "shared", "-o", LIB] + objs, cwd=CSRC, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link of libmd2_b200.so failed:\n" + r.stdout + r.stderr)
        with open(stamp, "w") as f:
            f.write(tag)
    return LIB


if __name__ == "__main__":
    import sys
    print(build(force="--force" in sys.argv, verbose=True))
