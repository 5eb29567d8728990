"""Build the sm_100a shared library in-tree (nvcc cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")
LIB = os.path.join(HERE, "libbfhe_b200.so")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
CCBIN = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def sources():
    src = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cpp"))]
    if os.path.isdir(HOST):
        src += [os.path.join(HOST, f) for f in sorted(os.listdir(HOST)) if f.endswith(".cpp")]
    return src


def deps():
    d = sources()
    for root in (CSRC, HOST, os.path.join(HERE, "..", "include")):
        if os.path.isdir(root):
            d += [os.path.join(root, f) for f in os.listdir(root) if f.endswith((".h", ".hpp", ".cuh"))]
    return d


def build(force=False, verbose=False):
    if not force and os.path.exists(LIB) and all(os.path.getmtime(s) <= os.path.getmtime(LIB) for s in deps()):
        return LIB
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    common = [NVCC, "-ccbin", CCBIN, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets",
              "-Xcompiler", "-fPIC,-fopenmp,-O3", "-I", os.path.join(HERE, "..", "include")]
    if verbose:
        common += ["-Xptxas", "-v"]
    jobs = []
    for s in sources():
        o = os.path.join(HERE, "build", os.path.basename(s) + ".o")
        if force or not os.path.exists(o) or any(os.path.getmtime(d) > os.path.getmtime(o) for d in deps()):
            jobs.append(common + (["-x", "cu"] if s.endswith(".cpp") else []) + ["-c", s, "-o", o])
        objs.append(o)
    procs = [subprocess.Popen(cmd) for cmd in jobs]  # one nvcc per translation unit, side by side
    failed = [p.args for p in procs if p.wait() != 0]
    if failed:
        raise subprocess.CalledProcessError(1, failed[0])
    subprocess.check_call([NVCC, "-ccbin", CCBIN, "-shared", "-o", LIB] + objs + ["-lgomp", "-ldl", "-cudart", "static"])
    # C++ example written against the reference-shaped headers (host/circuit.h, host/binfhecontext.h)
    for name, flags in (("tb_circuit", []), ("tb_client_server", []), ("tb_omp_gates", ["-fopenmp"])):
        ex = os.path.join(HERE, "examples", name + ".cpp")
        if os.path.exists(ex):
            subprocess.check_call([CCBIN, "-O2", "-std=c++17"] + flags + ["-o", os.path.join(HERE, "examples", name), ex, "-L" + HERE,
                                   "-lbfhe_b200", "-Wl,-rpath," + HERE])
    return LIB


def build_variant(tag, extra_flags):
    """debug/experiment variant of the library (e.g. -DBFHE_PHASE_TIMING): libbfhe_b200_<tag>.so, never used by the product"""
    out = os.path.join(HERE, "libbfhe_b200_%s.so" % tag)
    cmd = [NVCC, "-ccbin", CCBIN, "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets", "-Xcompiler", "-fPIC,-fopenmp,-O3",
           "-I", os.path.join(HERE, "..", "include"), "-shared", "-o", out] + list(extra_flags)
    for s in sources():
        cmd += (["-x", "cu"] if s.endswith(".cpp") else []) + [s]
    subprocess.check_call(cmd + ["-lgomp", "-ldl", "-cudart", "static"])
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
