"""Build the CUDA library in-tree: catfish_b200/libcatfish_b200.so (sm_100a only).

    python -m catfish_b200.build            # build if sources are newer than the .so
    python -m catfish_b200.build --force

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the
working tree (e.g. to the GPU box).

Environment (A/B builds, see tools/ab_lib.sh): CF_LIB_OUT = output path, CF_OBJ_TAG = prefix of the
object files, CF_EXTRA_DEFS = extra nvcc flags, CF_PRECISE_ACT = ex2/rcp activations instead of MUFU.TANH.
"""

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(HERE, "..", "include")
LIB = os.environ.get("CF_LIB_OUT") or os.path.join(HERE, "libcatfish_b200.so")
SOURCES = ["api.cu", "k1_normalize.cu", "k6_intervals.cu", "k7_chunks.cu", "k8_split.cu", "k9_validate.cu", "k11_sweep.cu", "k12_train.cu", "k13_curve.cu", "simt_engine.cu", "tc_engine.cu"]
NVCC_FLAGS = (["-DCF_PRECISE_ACT"] if os.environ.get("CF_PRECISE_ACT") else []) + os.environ.get("CF_EXTRA_DEFS", "").split() + ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC,-O2,-Wall", "-Xptxas", "-v"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    return "nvcc"


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, "catfish_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    if not force and not needs_build():
        return LIB
    objs = []
    logs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", os.environ.get("CF_OBJ_TAG", "") + src.replace(".cu", ".o"))
        cmd = [_nvcc()] + NVCC_FLAGS + ["-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        logs.append("== %s\n%s" % (src, out))
        if p.returncode != 0:
            failed = True
    log = "\n".join(logs)
    with open(os.path.join(HERE, "build", "nvcc.log"), "w") as f:
        f.write(log)
    if failed:
        sys.stderr.write(log)
        raise RuntimeError("nvcc failed; see catfish_b200/build/nvcc.log")
    cmd = [_nvcc(), "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("link failed")
    if verbose:
        print(log)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
