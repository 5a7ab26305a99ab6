"""Build libelg_b200.so in-tree with nvcc for sm_100a (no torch headers involved: plain C ABI)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libelg_b200.so")
SOURCES = ["model.cu", "problems.cu", "encoder.cu", "rollout.cu", "rollout_tc.cu", "rollout_stc.cu", "selftest.cu", "train_decode.cu",
           "train_bwd.cu", "generate.cu", "two_opt.cu", "cvrp_ls.cu", "tsp_ls.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--fmad=true"]


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh"))]
    deps.append(os.path.join(HERE, "..", "include", "elg_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


VARIANTS = {"timing": ["-DELG_PHASE_TIMING"]}     # diagnostic builds: libelg_b200_<variant>.so, loaded through ELG_B200_LIB


def build(force=False, verbose=False, variant=None):
    """Compile every CUDA source for sm_100a and link libelg_b200.so next to the sources."""
    if variant is None and not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("ELG_NVCC_EXTRA", "").split()      # e.g. -DELG_PHASE_TIMING for tools/phase_timing.py
    suffix = ""
    if variant:
        extra += VARIANTS[variant]
        suffix = "_" + variant
    out = os.path.join(CSRC, "libelg_b200%s.so" % suffix)
    objs = []
    logs = []
    for src in SOURCES:
        obj = os.path.join(CSRC, src.replace(".cu", suffix + ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        logs.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            sys.stderr.write(logs[-1])
            raise RuntimeError("nvcc failed on " + src)
        objs.append(obj)
    cmd = [nvcc, "-shared", "-o", out] + objs + ["-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    logs.append("$ " + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if r.returncode != 0:
        sys.stderr.write(logs[-1])
        raise RuntimeError("link failed")
    with open(os.path.join(CSRC, "build%s.log" % suffix), "w") as f:
        f.write("\n".join(logs))
    if verbose:
        print("\n".join(logs))
    return out


if __name__ == "__main__":
    var = sys.argv[sys.argv.index("--variant") + 1] if "--variant" in sys.argv else None
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, variant=var))
