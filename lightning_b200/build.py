"""Build recipes for the engine (nvcc, sm_100a only) and for the test-side artefacts.

Everything is built IN-TREE so that the shared objects travel with a gpurun snapshot:
  lightning_b200/libcln_sigverify.so   the product (CUDA kernels + C ABI)            [nvcc]
  tests/host_emul/libemul.so           kernel headers compiled for the host, tests only [g++]
  tests/host_emul/libemul_recover.so   the same plus the public-key recovery schedules, tests only [g++]
  oracle/libsecp_port.so               the plain-C restatement oracle                 [gcc]
  oracle/_ref/libsecp_ref.so           the unmodified reference, when /root/reference exists [gcc]
"""
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "lightning_b200", "csrc")
LIB = os.path.join(ROOT, "lightning_b200", "libcln_sigverify.so")
EMUL = os.path.join(ROOT, "tests", "host_emul", "libemul.so")
EMUL_RECOVER = os.path.join(ROOT, "tests", "host_emul", "libemul_recover.so")
DAEMON = os.path.join(ROOT, "lightning_b200", "cln_sigverifyd")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    # curve-side kernel variant: inlined field arithmetic + CTA-wide re-convergence barriers (see engine.cu);
    # in the ladder one barrier every 2 windows (measured: per point op 45.7, per window 46.4, per 2 windows 46.5,
    # per 4 windows 46.0, per 8 windows 45.4 M verifies/s — profiles/r1_variants.md)
    "-DSV_FE_INLINE", "-DSV_MAIN_SYNC", "-DSV_SYNC_LEVEL=1", "-DSV_SYNC_WINDOWS=2",
]


def _newer(target, sources):
    if not os.path.exists(target):
        return False
    t = os.path.getmtime(target)
    return all(os.path.getmtime(s) <= t for s in sources)


def _sources(d, exts):
    out = []
    for base, _, files in os.walk(d):
        out += [os.path.join(base, f) for f in files if f.endswith(exts)]
    return out


def build_engine(force=False, verbose=False, extra_flags=()):
    srcs = _sources(CSRC, (".cu", ".cuh", ".c", ".h")) + [os.path.join(ROOT, "include", "cln_sigverify.h"),
                                                   os.path.join(ROOT, "include", "cln_dropin.h")]
    # the flags are part of what the library is: a change of flags (or extra_flags) must rebuild, and so must a stale daemon
    stamp = os.path.join(os.path.dirname(LIB), ".build_flags")
    flags_now = " ".join(NVCC_FLAGS + list(extra_flags))
    same_flags = os.path.exists(stamp) and open(stamp).read() == flags_now
    if not force and same_flags and _newer(LIB, srcs) and _newer(DAEMON, srcs):
        return LIB
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    # host side of the drop-in is plain C (as the reference's bitcoin/signature.c), compiled by gcc
    dropin_o = os.path.join(CSRC, "cln_dropin.o")
    r = subprocess.run(["gcc", "-O2", "-fPIC", "-Wall", "-Wextra", "-std=c11", "-c", os.path.join(CSRC, "cln_dropin.c"),
                        "-o", dropin_o], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("gcc (cln_dropin.c) failed:\n" + r.stdout + r.stderr)
    # the batch-verification kernels are a translation unit of their own, compiled with the field multiplier as real
    # functions (see batch.cu); everything else inlines it
    batch_flags = [f for f in NVCC_FLAGS if f not in ("-shared", "-DSV_FE_INLINE", "-DSV_MAIN_SYNC")] + ["-DSV_NO_SYNC_INLINE", "-c"]
    batch_o = os.path.join(CSRC, "batch.o")
    r = subprocess.run([nvcc] + batch_flags + (["-Xptxas", "-v"] if verbose else []) + ["-o", batch_o, os.path.join(CSRC, "batch.cu")],
                       capture_output=True, text=True)
    if verbose:
        sys.stderr.write(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc (batch.cu) failed:\n" + r.stdout + r.stderr)
    cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + (["-Xptxas", "-v"] if verbose else []) + [
        "-o", LIB, os.path.join(CSRC, "engine.cu"), batch_o, dropin_o]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose:
        sys.stderr.write(r.stderr)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    # verifier subdaemon (row N4): plain C, links the engine
    r = subprocess.run(["gcc", "-O2", "-Wall", "-Wextra", "-std=c11", os.path.join(CSRC, "sigverifyd.c"), "-o", DAEMON,
                        "-L" + os.path.dirname(LIB), "-lcln_sigverify", "-Wl,-rpath,$ORIGIN"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("gcc (sigverifyd.c) failed:\n" + r.stdout + r.stderr)
    open(stamp, "w").write(flags_now)
    return LIB


def _build_emul(out, src, extra_srcs=(), force=False):
    srcs = _sources(CSRC, (".cuh",)) + [src] + list(extra_srcs)
    if not force and _newer(out, srcs):
        return out
    cmd = ["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-pthread", "-Wall", "-Wno-unused-function", "-o", out, src]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"g++ ({os.path.basename(src)}) failed:\n" + r.stdout + r.stderr)
    return out


def build_host_emul(force=False):
    d = os.path.join(ROOT, "tests", "host_emul")
    _build_emul(EMUL_RECOVER, os.path.join(d, "emul_recover.cpp"), [os.path.join(d, "emul.cpp")], force)
    return _build_emul(EMUL, os.path.join(d, "emul.cpp"), force=force)


def build_host_emul_recover(force=False):
    build_host_emul(force)
    return EMUL_RECOVER


def build_oracle():
    r = subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "all"], capture_output=True, text=True,
                       stdin=subprocess.DEVNULL, timeout=900)
    if r.returncode != 0:
        raise RuntimeError("oracle build failed:\n" + r.stdout + r.stderr)


def build_all(force=False, verbose=False):
    build_engine(force=force, verbose=verbose)
    build_host_emul(force=force)
    build_oracle()


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built:", LIB)
