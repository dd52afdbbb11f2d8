"""Build libtoued.so (sm_100a) in-tree with nvcc.  Used by __graft_entry__.build() and importable
as ``python -m to_ued_b200.csrc.build``.  One object per .cu so only changed files recompile."""
import os, subprocess, sys, hashlib, shutil

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "..", "libtoued.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC"]
# per-file overrides: the sampling path must round exactly like the oracle (no FMA contraction),
# so rollout.cu adds -fmad=false.
FLAGS = {
    "rollout.cu": ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-fmad=false"],
    "levelgen.cu": ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-fmad=false"],
}


def _nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


# diagnostic variants: name -> extra -D flags; built into libtoued_<name>.so next to the production library
VARIANTS = {
    # random delays in front of every mbarrier wait: schedule fuzzing of the warp-specialised kernels
    "fuzz": ["-DTOUED_FUZZ=1"],
}


def build(verbose=False, force=False, variant=""):
    global OUT
    if variant:
        return _build(verbose, force, os.path.join(HERE, "..", f"libtoued_{variant}.so"),
                      os.path.join(HERE, f"build_{variant}"), VARIANTS[variant])
    return _build(verbose, force, OUT, os.path.join(HERE, "build"), [])


def _build(verbose, force, OUT, objdir, extra):
    srcs = sorted(f for f in os.listdir(HERE) if f.endswith(".cu"))
    hdrs = sorted(f for f in os.listdir(HERE) if f.endswith(".cuh")) + ["../../include/toued.h"]
    hsig = hashlib.sha1(b"".join(open(os.path.join(HERE, h), "rb").read() for h in hdrs)).hexdigest()
    os.makedirs(objdir, exist_ok=True)
    objs, rebuilt = [], False
    for s in srcs:
        src = os.path.join(HERE, s)
        obj = os.path.join(objdir, s[:-3] + ".o")
        flags = list(FLAGS.get(s, COMMON)) + list(extra)
        sig = hashlib.sha1(open(src, "rb").read() + hsig.encode() + " ".join(flags).encode()).hexdigest()
        sigf = obj + ".sig"
        if force or not os.path.exists(obj) or not os.path.exists(sigf) or open(sigf).read() != sig:
            cmd = [_nvcc(), *ARCH, *flags, "-c", src, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas"); cmd.insert(2, "-v")
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
            open(sigf, "w").write(sig)
            rebuilt = True
        objs.append(obj)
    if rebuilt or not os.path.exists(OUT):
        cmd = [_nvcc(), *ARCH, "-shared", "-o", OUT, *objs, "-lcudart"]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
    return os.path.abspath(OUT)


if __name__ == "__main__":
    var = [a.split("=", 1)[1] for a in sys.argv if a.startswith("--variant=")]
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv, variant=var[0] if var else ""))
