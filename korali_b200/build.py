"""Builds korali_b200/libkcma.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m korali_b200.build [--force]
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libkcma.so")
OBJ = os.path.join(HERE, "build")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall"] + ARCH
# files whose arithmetic must round like the reference's scalar code (no fused multiply-add)
NO_FMA = {"objective.cu", "update.cu", "constraints.cu", "dea.cu", "mocma.cu", "tmcmc.cu"}
SOURCES = ["api.cu", "gemm.cu", "gemm_tma.cu", "rng.cu", "objective.cu", "sort.cu", "update.cu", "eigen.cu", "constraints.cu", "gemm_batched.cu", "tridiag.cu", "dc.cu", "dea.cu", "mocma.cu", "tmcmc.cu"]


def _newer(src, dst):
    return not os.path.exists(dst) or os.path.getmtime(src) > os.path.getmtime(dst)


def build(force=False, verbose=False):
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    headers.append(os.path.join(HERE, "..", "include", "kcma.h"))
    headers.append(os.path.join(HERE, "..", "include", "kdea.h"))
    headers.append(os.path.join(HERE, "..", "include", "kmocma.h"))
    headers.append(os.path.join(HERE, "..", "include", "ktmcmc.h"))
    objs, rebuilt = [], False
    procs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        objs.append(obj)
        if force or _newer(src, obj) or any(_newer(hd, obj) for hd in headers):
            cmd = ["nvcc", "-c", src, "-o", obj] + COMMON + (["--fmad=false"] if s in NO_FMA else [])
            if verbose:
                cmd += ["-Xptxas", "-v"]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
            rebuilt = True
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (s, out))
        if verbose or out.strip():
            sys.stderr.write(out)
    if rebuilt or not os.path.exists(OUT):
        cmd = ["nvcc", "-shared", "-o", OUT] + objs + ARCH + ["-Xcompiler", "-fPIC", "-ldl"]
        subprocess.check_call(cmd)
    build_host(force)
    return OUT


def build_host(force=False):
    """The pybind11 host shim (korali_b200/_host*.so): Korali's Engine/Experiment surface above the C ABI."""
    import sysconfig
    import pybind11
    src = os.path.join(HERE, "host", "korali_host.cpp")
    out = os.path.join(HERE, "_host" + sysconfig.get_config_var("EXT_SUFFIX"))
    if not (force or _newer(src, out) or _newer(OUT, out) or
            any(_newer(os.path.join(HERE, "..", "include", h), out) for h in ("kcma.h", "kdea.h", "kmocma.h", "ktmcmc.h"))):
        return out
    cmd = ["g++", "-O2", "-shared", "-fPIC", "-std=c++17", "-fvisibility=hidden", "-I", pybind11.get_include(),
           "-I", sysconfig.get_paths()["include"], src, "-o", out, "-L", HERE, "-lkcma", "-Wl,-rpath,$ORIGIN"]
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
