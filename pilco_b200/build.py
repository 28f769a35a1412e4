"""Build the sm_100a shared library in-tree with nvcc (cross-compiles without a GPU).

    python -m pilco_b200.build

Produces ``pilco_b200/libpilco_b200.so`` (git-ignored; travels to the GPU box with the snapshot).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libpilco_b200.so")
SOURCES = ["abi.cu", "mm_forward.cu", "mm_backward.cu", "mm_tape.cu", "closed_forms.cu", "factorize.cu", "rollout.cu",
           "rollout_bwd.cu", "microbench.cu", "gp_predict.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-rdc=false"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "pilco_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, extra_flags=(), lib=None, build_dir=None):
    """``extra_flags``/``lib``/``build_dir``: diagnostics variants (e.g. -DPILCO_TILE_TIMING) built beside the product
    library; the default call builds ``libpilco_b200.so``."""
    if lib is None and not force and not needs_build():
        return LIB
    nvcc = _nvcc()
    objs = []
    build_dir = build_dir or os.path.join(HERE, "build")
    os.makedirs(build_dir, exist_ok=True)
    procs = []
    for src in SOURCES:
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(build_dir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (src, out))
        if verbose and out:
            sys.stderr.write(out)
    out_lib = lib or LIB
    cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out_lib] + objs + ["-lcudart"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout)
    return out_lib


def build_exp256(force=True):
    """Variant library with the bank-conflict-free 256 x 16 exp table (-DPILCO_EXP256), beside the product library:
    select it with PILCO_B200_LIB=<path> (A/B measurements)."""
    return build(force=force, extra_flags=["-DPILCO_EXP256"], lib=os.path.join(HERE, "build_exp256", "libpilco_b200_exp256.so"),
                 build_dir=os.path.join(HERE, "build_exp256"))


if __name__ == "__main__":
    if "--exp256" in sys.argv:
        print(build_exp256())
    elif "--timing" in sys.argv:      # diagnostics variant with per-CTA phase stamps in the tile kernel
        print(build(force=True, extra_flags=["-DPILCO_TILE_TIMING"], lib=os.path.join(HERE, "build_timing", "libpilco_b200_timing.so"),
                    build_dir=os.path.join(HERE, "build_timing")))
    else:
        print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
