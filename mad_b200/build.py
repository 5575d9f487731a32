"""Builds libmad_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m mad_b200.build [--force]

The shared library is the C-ABI product (include/mad_b200.h); it is git-ignored but travels
with the source tree to the GPU box.  nvcc cross-compiles without a GPU.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libmad_b200.so")
SOURCES = ["dmap.cu", "density.cu", "scale_space.cu", "detect.cu", "orient.cu", "describe.cu", "match_simt.cu", "match_tc.cu", "match_u8.cu", "match_prep.cu", "repeat.cu", "cloud.cu", "score.cu", "api.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "mad_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every .cu of the package into one shared library; objects are built in parallel."""
    if not force and not needs_build():
        return LIB
    obj_dir = os.path.join(HERE, "build")
    os.makedirs(obj_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(obj_dir, src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((src, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    objs = []
    for src, obj, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            sys.stderr.write(out.decode())
        if p.returncode != 0:
            raise RuntimeError("nvcc failed on %s:\n%s" % (src, out.decode()))
        objs.append(obj)
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s" % r.stdout.decode())
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
