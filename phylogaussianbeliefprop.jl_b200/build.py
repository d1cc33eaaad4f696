"""Builds libpgbp_b200.so (CUDA, sm_100a) in-tree with nvcc.

    python phylogaussianbeliefprop.jl_b200/build.py            # the product
    python phylogaussianbeliefprop.jl_b200/build.py --emul     # host emulation of the kernel bodies,
                                                               # used ONLY by CPU tests of the host logic
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
# (source, extra defines, object name): the 78 register-resident message shapes are compiled as three
# translation units in parallel (pgbp_message_t0.cu with -DPGBP_T0_PART=0,1,2)
SOURCES = [("pgbp_plan.cu", [], "pgbp_plan"), ("pgbp_batch.cu", [], "pgbp_batch"), ("pgbp_message.cu", [], "pgbp_message"),
           ("pgbp_message_medium.cu", [], "pgbp_message_medium"), ("pgbp_factors.cu", [], "pgbp_factors"),
           ("pgbp_comm.cu", [], "pgbp_comm"), ("pgbp_marginals.cu", [], "pgbp_marginals"),
           ("pgbp_message_t0.cu", ["PGBP_T0_PART=0"], "pgbp_message_t0_0"),
           ("pgbp_message_t0.cu", ["PGBP_T0_PART=1"], "pgbp_message_t0_1"),
           ("pgbp_message_t0.cu", ["PGBP_T0_PART=2"], "pgbp_message_t0_2"),
           ("pgbp_shared.cu", [], "pgbp_shared"), ("pgbp_simulate.cu", [], "pgbp_simulate")]
HEADERS = ["pgbp_backend.h", "pgbp_internal.h", "pgbp_kernels.cuh", "pgbp_launch.h", "pgbp_shapes.h", "pgbp_msg_t0.cuh",
           "pgbp_coop.cuh", "pgbp_bulk.cuh", "pgbp_factors.cuh", "pgbp_philox.h",
           os.path.join("..", "..", "include", "pgbp_b200.h")]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
              # no implicit mul+add contraction: the only fused operations are the explicit fma() calls, so all
              # kernel variants of one operation are bit-identical to each other
              "-fmad=false"]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def _run(cmd):
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        raise RuntimeError("build failed: " + os.path.basename(cmd[-1]))
    return r.stdout + r.stderr


def build(emul=False, verbose=False, force=False, defines=(), tag=""):
    """tag/defines: experimental variants (lib/libpgbp_b200_<tag>.so built with -D<define>), selected at
    run time with PGBP_B200_LIB=<path>; the default build has neither."""
    os.makedirs(LIBDIR, exist_ok=True)
    objdir = os.path.join(LIBDIR, ("obj_emul" if emul else "obj") + (("_" + tag) if tag else ""))
    os.makedirs(objdir, exist_ok=True)
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    lib = os.path.join(LIBDIR, "libpgbp_emul.so" if emul else ("libpgbp_b200_%s.so" % tag if tag else "libpgbp_b200.so"))
    dflags = ["-D" + d for d in defines]
    objs, jobs = [], []
    for s, sdefs, oname in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(objdir, oname + ".o")
        objs.append(obj)
        sd = ["-D" + d for d in sdefs]
        if force or _stale(obj, [src] + hdrs):
            if emul:
                cmd = ["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-DPGBP_HOST_EMUL"] + sd + ["-x", "c++", "-c", src, "-o", obj]
            else:
                cmd = [NVCC] + NVCC_FLAGS + dflags + sd + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            jobs.append(cmd)
    if jobs:
        with ThreadPoolExecutor(max_workers=min(os.cpu_count() or 4, len(jobs))) as ex:
            for out in ex.map(_run, jobs):
                if verbose:
                    print(out)
    if jobs or not os.path.exists(lib):
        if emul:
            _run(["g++", "-shared", "-o", lib] + objs)
        else:
            _run([NVCC, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"])
    return lib


if __name__ == "__main__":
    defs = [a[2:] for a in sys.argv[1:] if a.startswith("-D")]
    tags = [a[6:] for a in sys.argv[1:] if a.startswith("--tag=")]
    print(build(emul="--emul" in sys.argv, verbose="-v" in sys.argv, force="--force" in sys.argv, defines=defs,
                tag=tags[0] if tags else ""))
