"""In-tree build of the CUDA library and the calc-witness CLI (nvcc cross-compiles sm_100a without a GPU).

  python circom-witnesscalc_b200/build.py [--force] [--verbose]

Outputs (git-ignored):
  circom-witnesscalc_b200/lib/libcircom_witnesscalc.so   the C-ABI library of include/graph_witness.h
  circom-witnesscalc_b200/bin/calc-witness               CLI with the reference's argv contract
  circom-witnesscalc_b200/bin/calc-witness-batch         batch companion: <graph.bin> <inputs.jsonl> <out_dir> [n_gpus]
  circom-witnesscalc_b200/bin/example-calc-witness       examples/calc_witness.c: <inputs.json> <graph.bin> <out.wtns>
  circom-witnesscalc_b200/bin/wtns-check                 <circuit.r1cs> <witness.wtns> [more.wtns ...] (snarkjs wtns check)
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib", "libcircom_witnesscalc.so")
# the same library with -DGW_PROFILING: per-packet clocks, timing experiments and the fault injection that the watchdog
# test needs (tests/test_gpu_parity.py); loaded through GW_LIB_PATH only
LIB_PROF = os.path.join(HERE, "lib_variants", "libcwc_prof.so")
BIN = os.path.join(HERE, "bin", "calc-witness")
BIN_BATCH = os.path.join(HERE, "bin", "calc-witness-batch")
BIN_WTNS_CHECK = os.path.join(HERE, "bin", "wtns-check")
# the plain-C embedding example of the drop-in ABI (examples/calc_witness.c): the acceptance test of the C ABI runs it
EXAMPLE_SRC = os.path.join(HERE, "..", "examples", "calc_witness.c")
BIN_EXAMPLE = os.path.join(HERE, "bin", "example-calc-witness")
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
SOURCES = ["engine.cu", "r1cs.cu", "ntt.cu", "inputs.cu", "cuda_util.cpp", "graph.cpp", "plan.cpp", "bitplan.cpp", "inputs.cpp", "wtns.cpp", "r1cs.cpp", "capi.cpp"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
# the optimisation flags of every device build (the test-only device harness of tests/csrc is built with them too)
OPT = ["-std=c++17", "-O3", "-lineinfo"]


def _newer(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    os.makedirs(os.path.dirname(BIN), exist_ok=True)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "graph_witness.h")]
    if force or _newer(LIB, deps):
        cmd = [NVCC, "-shared", "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unknown-pragmas,-Wno-misleading-indentation", *OPT, *ARCH,
               "-Xptxas", "-v" if verbose else "-O3", "-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
        if verbose:
            print(" ".join(cmd))
        subprocess.check_call(cmd)
    if force or _newer(LIB_PROF, deps):
        os.makedirs(os.path.dirname(LIB_PROF), exist_ok=True)
        cmd = [NVCC, "-shared", "-Xcompiler", "-fPIC,-O3", *OPT, *ARCH, "-DGW_PROFILING",
               "-o", LIB_PROF] + [os.path.join(CSRC, s) for s in SOURCES]
        subprocess.check_call(cmd)
    if force or _newer(BIN, [LIB, os.path.join(CSRC, "calc_witness_main.cpp")]):
        cmd = ["g++", "-O2", "-std=c++17", "-o", BIN, os.path.join(CSRC, "calc_witness_main.cpp"),
               "-L" + os.path.dirname(LIB), "-lcircom_witnesscalc", "-Wl,-rpath,$ORIGIN/../lib"]
        subprocess.check_call(cmd)
    if force or _newer(BIN_BATCH, [LIB, os.path.join(CSRC, "calc_witness_batch_main.cpp")]):
        cmd = ["g++", "-O2", "-std=c++17", "-o", BIN_BATCH, os.path.join(CSRC, "calc_witness_batch_main.cpp"),
               "-L" + os.path.dirname(LIB), "-lcircom_witnesscalc", "-Wl,-rpath,$ORIGIN/../lib"]
        subprocess.check_call(cmd)
    if force or _newer(BIN_WTNS_CHECK, [LIB, os.path.join(CSRC, "wtns_check_main.cpp")]):
        cmd = ["g++", "-O2", "-std=c++17", "-o", BIN_WTNS_CHECK, os.path.join(CSRC, "wtns_check_main.cpp"),
               "-L" + os.path.dirname(LIB), "-lcircom_witnesscalc", "-Wl,-rpath,$ORIGIN/../lib"]
        subprocess.check_call(cmd)
    header = os.path.join(HERE, "..", "include", "graph_witness.h")
    if force or _newer(BIN_EXAMPLE, [LIB, EXAMPLE_SRC, header]):
        subprocess.check_call(["gcc", "-std=c99", "-O2", "-Wall", "-Wextra", "-o", BIN_EXAMPLE, EXAMPLE_SRC,
                               "-L" + os.path.dirname(LIB), "-lcircom_witnesscalc", "-Wl,-rpath,$ORIGIN/../lib"])
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
