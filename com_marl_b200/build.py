"""Builds lib/libcommarl_b200.so with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(_HERE)
SOURCES = ["env_kernels.cu", "policy_kernel.cu", "policy_tc_kernel.cu", "policy_attn_kernel.cu", "policy_attn_mma_kernel.cu", "policy_cent_kernel.cu", "host_abi.cu", "ppo_kernels.cu", "ppo_net_kernels.cu", "abi.cu"]
OUT = os.path.join(_HERE, "lib", "libcommarl_b200.so")


def nvcc_path():
    for p in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if p and (os.path.exists(p) or p == "nvcc"):
            return p
    return "nvcc"


def needs_build():
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(_HERE, "csrc", f) for f in os.listdir(os.path.join(_HERE, "csrc"))]
    deps.append(os.path.join(ROOT, "include", "commarl_b200.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """every translation unit is compiled on its own (in parallel: the templated kernels take a minute or two each), then linked"""
    if not force and not needs_build():
        return OUT
    from concurrent.futures import ThreadPoolExecutor
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    objdir = os.path.join(_HERE, "lib", "obj")
    os.makedirs(objdir, exist_ok=True)
    common = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(_HERE, "csrc")]
    if verbose:
        common[1:1] = ["-Xptxas", "-v"]

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        subprocess.check_call(common + ["-c", os.path.join(_HERE, "csrc", src), "-o", obj])
        return obj

    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 4)) as pool:
        objs = list(pool.map(compile_one, SOURCES))
    subprocess.check_call([nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", OUT] + objs)
    return OUT


TC_PROBE_SRC = os.path.join(ROOT, "tests", "native", "tc_gemm_probe.cu")
TC_PROBE = os.path.join(ROOT, "tests", "native", "libtc_probe.so")


def build_tc_probe(force=False):
    """tests/native/libtc_probe.so: the tcgen05 GEMM probe over csrc/tc_common.cuh that tests/test_gpu_tc_probe.py loads"""
    deps = (TC_PROBE_SRC, os.path.join(_HERE, "csrc", "tc_common.cuh"))
    if force or not os.path.exists(TC_PROBE) or any(os.path.getmtime(d) > os.path.getmtime(TC_PROBE) for d in deps):
        subprocess.check_call([nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                               "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(_HERE, "csrc"), "-I", os.path.join(ROOT, "include"),
                               "-o", TC_PROBE, TC_PROBE_SRC])
    return TC_PROBE


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print(OUT)
