"""Builds libscanfold_b200.so (sm_100a) in-tree with nvcc.  Used by __graft_entry__.build()."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.environ.get("SFB_BUILD_OUT") or os.path.join(HERE, "libscanfold_b200.so")   # SFB_BUILD_OUT: debug variants
SOURCES = ["params.cpp", "mfe.cu", "mfe2.cu", "mfe3.cu", "mfe4.cu", "pf.cu", "pf2.cu", "shuffle.cu", "accumulate.cu", "pairprob.cu", "microbench.cu", "api.cu"]
EXTRA = os.environ.get("SFB_NVCC_EXTRA", "").split()
NVCC_FLAGS = EXTRA + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "scanfold_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return OUT
    objdir = os.path.join(HERE, "build" + ("_" + os.path.basename(OUT).split(".")[0] if os.environ.get("SFB_BUILD_OUT") else ""))
    os.makedirs(objdir, exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.rsplit(".", 1)[0] + ".o")
        cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-x", "cu", "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out)
        if p.returncode:
            raise RuntimeError("nvcc failed on " + src)
    cmd = [_nvcc(), "-shared", "-o", OUT] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart_static", "-ldl", "-lpthread", "-lrt"]
    subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
