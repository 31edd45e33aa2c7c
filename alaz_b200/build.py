"""Builds libalazgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIB_DIR, "libalazgpu.so")

SOURCES = ["alz_api.cu", "alz_kernels.cu", "alz_ingest.cu", "alz_sort.cu", "alz_comm.cu", "alz_gnn.cu", "alz_sock.cu",
           "alz_history.cu"]
EXTRA = [os.path.join(HERE, "synth", "alz_synth_topo.c")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def _deps():
    out = []
    for d in (CSRC, os.path.join(HERE, "synth"), os.path.join(os.path.dirname(HERE), "include")):
        for f in os.listdir(d):
            if f.endswith((".cu", ".cuh", ".h", ".c", ".cpp")):
                out.append(os.path.join(d, f))
    return out


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(p) > t for p in _deps())


def build(force=False, verbose=False, prof=False):
    """prof=True: libalazgpu_prof.so with per-section cycle counters in the ingest kernel (ALZ_LIB_PATH selects it)."""
    out = LIB.replace("libalazgpu.so", "libalazgpu_prof.so") if prof else LIB
    if not force and not prof and not needs_build():
        return LIB
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = os.environ.get("NVCC", "nvcc")
    srcs = [os.path.join(CSRC, s) for s in SOURCES] + EXTRA
    cmd = [nvcc] + NVCC_FLAGS + (["-DALZ_INGEST_PROF"] if prof else []) + (["-Xptxas", "-v"] if verbose else []) + \
        srcs + ["-o", out + ".tmp", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("nvcc failed building libalazgpu.so")
    os.replace(out + ".tmp", out)   # a snapshot of the tree (gpurun) never sees a half-written library
    if verbose:
        sys.stderr.write(r.stderr)
    return out


SIM_TEST = os.path.join(LIB_DIR, "alaz_sim_test")


def build_sim_test(force=False):
    """g++ build of the C++ host adapter + the reference's simulation scenario (tests/cpp/sim_test.cc)."""
    root = os.path.dirname(HERE)
    srcs = [os.path.join(root, "tests", "cpp", "sim_test.cc"), os.path.join(HERE, "host", "alaz_aggregator.cc")]
    deps = srcs + [os.path.join(HERE, "host", "alaz_aggregator.hpp"), LIB]
    if not os.path.exists(LIB):   # never rebuild a library this process may already have loaded
        build()
    if not force and os.path.exists(SIM_TEST) and all(os.path.getmtime(d) <= os.path.getmtime(SIM_TEST) for d in deps):
        return SIM_TEST
    cmd = ["g++", "-std=c++17", "-O2", "-Wall"] + srcs + ["-L" + LIB_DIR, "-lalazgpu", "-Wl,-rpath," + LIB_DIR,
                                                           "-Wl,-rpath,$ORIGIN", "-o", SIM_TEST]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building alaz_sim_test")
    return SIM_TEST


HOST_UNIT = os.path.join(LIB_DIR, "alaz_host_unit_test")


def build_host_unit_test():
    root = os.path.dirname(HERE)
    srcs = [os.path.join(root, "tests", "cpp", "host_unit_test.cc"), os.path.join(HERE, "host", "alaz_aggregator.cc")]
    if not os.path.exists(LIB):
        build()
    cmd = ["g++", "-std=c++17", "-O1", "-Wall"] + srcs + ["-L" + LIB_DIR, "-lalazgpu", "-Wl,-rpath," + LIB_DIR,
                                                           "-Wl,-rpath,$ORIGIN", "-o", HOST_UNIT]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("g++ failed building alaz_host_unit_test")
    return HOST_UNIT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, prof="--prof" in sys.argv))
