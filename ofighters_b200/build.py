"""Build libofb.so (the C-ABI CUDA library) in-tree for sm_100a.

    python -m ofighters_b200.build [--force]

nvcc cross-compiles without a GPU.  The arena translation units are built with
``-fmad=false`` so that no fp64 multiply-add is contracted (bit-exact parity with
CPython's arithmetic); the policy kernels are free to use FMA.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_native")
LIB = os.path.join(OUT_DIR, "libofb.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]

# (source, extra flags)
UNITS = [
    ("ofb_arena.cu", ["-fmad=false"]),
    ("ofb_step.cu", ["-fmad=false"]),
    ("ofb_raster.cu", ["-fmad=false"]),
    ("ofb_replay.cu", ["-fmad=false"]),
    ("ofb_policy.cu", []),
    ("ofb_policy_tc.cu", []),
    ("ofb_policy_tz.cu", []),
    ("ofb_policy_tail.cu", []),
    ("ofb_policy_sp.cu", []),
    ("ofb_policy_st.cu", []),
    ("ofb_train.cu", []),
]


def _deps():
    inc = os.path.join(HERE, "..", "include")
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(inc, f) for f in os.listdir(inc)]


def _compile(src, extra, obj, verbose):
    cmd = ["nvcc"] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + \
          ["-c", os.path.join(CSRC, src), "-o", obj]
    subprocess.check_call(cmd)
    return obj


def build(force=False, verbose=False):
    """Compiles the translation units that are older than any source / header (in parallel) and links libofb.so."""
    from concurrent.futures import ThreadPoolExecutor
    newest = max(os.path.getmtime(p) for p in _deps())
    if not force and os.path.exists(LIB) and os.path.getmtime(LIB) >= newest:
        return LIB
    os.makedirs(OUT_DIR, exist_ok=True)
    hdr_newest = max(os.path.getmtime(p) for p in _deps() if not p.endswith(".cu"))
    jobs, objs = [], []
    for src, extra in UNITS:
        obj = os.path.join(OUT_DIR, src.replace(".cu", ".o"))
        objs.append(obj)
        stale = force or not os.path.exists(obj) or \
            os.path.getmtime(obj) < max(hdr_newest, os.path.getmtime(os.path.join(CSRC, src)))
        if stale:
            jobs.append((src, extra, obj))
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        for f in [ex.submit(_compile, s, e, o, verbose) for s, e, o in jobs]:
            f.result()
    subprocess.check_call(["nvcc"] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcuda"])
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
