"""In-tree nvcc build of libfgvc_b200.so (sm_100a only; no torch headers, plain C ABI).

``python -m fgvc_b200.build`` or ``__graft_entry__.build()``.  nvcc cross-compiles
without a GPU, so this also runs in the CPU-only build container; the resulting .so
travels to the GPU box with the repo snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libfgvc_b200.so")
STAMP = os.path.join(HERE, ".libfgvc_b200.stamp")
SOURCES = ["capi.cu", "prep.cu", "topk_simt.cu", "topk_tc.cu", "topk_tc16.cu", "gather.cu", "dense.cu", "coords.cu", "c2f.cu", "clip.cu", "cycle.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden", "--use_fast_math=false"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; the fgvc_b200 CUDA library cannot be built")


def _digest():
    h = hashlib.sha256()
    inc = os.path.join(os.path.dirname(HERE), "include", "fgvc_b200.h")
    for p in sorted(os.listdir(CSRC)) + [inc]:
        path = p if os.path.isabs(p) else os.path.join(CSRC, p)
        with open(path, "rb") as f:
            h.update(os.path.basename(p).encode())      # (not the path: the tree moves between boxes)
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def up_to_date():
    """the library exists and was built from the current sources (digest stamp)"""
    try:
        return os.path.exists(LIB) and open(STAMP).read() == _digest()
    except OSError:
        return False


def build(force=False, verbose=False):
    dig = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read() == dig:
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "--use_fast_math=false"]
    if os.environ.get("FGVC_BUILD_DEFS"):          # experiments, e.g. FGVC_BUILD_DEFS=-DFGVC_TC16_STATS
        flags += os.environ["FGVC_BUILD_DEFS"].split()
    procs = []
    for s in SOURCES:
        obj = os.path.join(objdir, s.replace(".cu", ".o"))
        cmd = [nvcc, *flags, "-Xptxas", "-v" if verbose else "-warn-spills", "-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for s, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
        if verbose or "warning" in out:
            print(out, file=sys.stderr)
        objs.append(obj)
    tmp_lib = LIB + f".tmp{os.getpid()}"
    cmd = [nvcc, "-shared", "-o", tmp_lib, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static",
           "-ldl", "-lpthread", "-lrt"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    os.replace(tmp_lib, LIB)            # atomic: a concurrent loader sees the old or the new file, never half of one
    with open(STAMP, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
