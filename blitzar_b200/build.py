"""Builds the in-tree native artefacts (no JIT cache): the product CUDA library for sm_100a, and —
as test infrastructure — the CPU emulation harness, the C oracle port and, when /root/reference
is present, the reference's own CPU path (oracle/_ref)."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "blitzar_b200", "csrc")
LIBDIR = os.path.join(ROOT, "blitzar_b200", "lib")
LIB = os.path.join(LIBDIR, "libblitzar_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = ["-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC"]
UNITS = ["api.cu", "curve_ed25519.cu", "curve_bls12381.cu", "curve_bn254.cu", "curve_grumpkin.cu",
         "sumcheck.cu"]


def _newer(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def _headers():
    return [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))] + \
        [os.path.join(ROOT, "include", "blitzar_b200.h")]


def build_product(verbose=False):
    os.makedirs(LIBDIR, exist_ok=True)
    subprocess.check_call([sys.executable, os.path.join(CSRC, "gen_constants.py")])
    units = [u for u in UNITS if os.path.exists(os.path.join(CSRC, u))]
    objs, procs = [], []
    for u in units:
        src = os.path.join(CSRC, u)
        obj = os.path.join(LIBDIR, u.replace(".cu", ".o"))
        objs.append(obj)
        if _newer(obj, [src] + _headers()):
            cmd = [NVCC] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((u, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for u, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            sys.stderr.write(out.decode())
        if p.returncode:
            raise RuntimeError(f"nvcc failed for {u}")
    if procs or not os.path.exists(LIB):
        subprocess.check_call([NVCC, "-shared", "-o", LIB] + objs +
                              ["-Xlinker", "--version-script=" + os.path.join(CSRC, "export.map")])
    return LIB


def build_emul():
    """CPU emulation harness (test infrastructure): the per-curve units of the product compiled as
    host C++ (-DB200_EMULATE, tests/emul/emul_prefix.h force-included), in parallel."""
    edir = os.path.join(ROOT, "tests", "emul")
    out = os.path.join(edir, "libb200_emul.so")
    objdir = os.path.join(edir, "obj")
    os.makedirs(objdir, exist_ok=True)
    prefix = os.path.join(edir, "emul_prefix.h")
    flags = ["g++", "-std=c++17", "-O1", "-DB200_EMULATE", "-fPIC", "-w", "-include", prefix]
    jobs, objs = [], []
    for u in [x for x in UNITS if x.startswith("curve_")] + ["emul.cpp", "emul_sumcheck.cpp"]:
        src = os.path.join(edir if u.startswith("emul") else CSRC, u)
        obj = os.path.join(objdir, u.rsplit(".", 1)[0] + ".o")
        objs.append(obj)
        if _newer(obj, [src, prefix] + _headers()):
            jobs.append((u, subprocess.Popen(flags + ["-x", "c++", "-c", src, "-o", obj],
                                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT)))
    for u, p in jobs:
        o, _ = p.communicate()
        if p.returncode:
            sys.stderr.write(o.decode())
            raise RuntimeError(f"emulation build failed for {u}")
    if jobs or not os.path.exists(out):
        subprocess.check_call(["g++", "-shared", "-o", out] + objs)
    return out


def build_oracle_port():
    src = os.path.join(ROOT, "oracle", "msm_oracle.c")
    out = os.path.join(ROOT, "oracle", "libmsm_oracle.so")
    if os.path.exists(src) and _newer(out, [src]):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-w", src, "-o", out])
    return out


def build_oracle_ref():
    """Only possible where /root/reference exists (this container); the GPU box uses the prebuilt
    oracle/_ref/libblitzar_ref_cpu.so that travels with the snapshot."""
    if not os.path.isdir("/root/reference/sxt"):
        return None
    ref_build = os.path.join(ROOT, "oracle", "ref_build")
    subprocess.check_call(["make", "-s", "-j8", "-C", ref_build], stdout=subprocess.DEVNULL)
    subprocess.check_call(["make", "-s", "-f", os.path.join(ref_build, "sumcheck.mk")],
                          stdout=subprocess.DEVNULL)
    return os.path.join(ROOT, "oracle", "_ref", "libblitzar_ref_cpu.so")


def build_all(verbose=False):
    build_product(verbose)
    build_emul()
    build_oracle_port()
    build_oracle_ref()


if __name__ == "__main__":
    build_all(verbose="-v" in sys.argv)
