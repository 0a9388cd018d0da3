"""Build recipes: the CUDA C-ABI library (nvcc, sm_100a) and the host-only synthetic generator."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libvloam_b200.so")
SYNTH_LIB = os.path.join(HERE, "libvloam_synth.so")
CU_SOURCES = ["scan_registration.cu", "voxel_grid.cu", "laser_odometry.cu", "laser_mapping.cu", "lm_solver.cu", "stage_inputs.cu", "relocalize.cu", "capi.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # bit-exact parity with the reference's x86-64 arithmetic: no FMA contraction,
    # IEEE division and square root (SURVEY.md 7.2 items 1 and 4)
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-shared", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
]


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_cuda(force=False, verbose=False):
    """One nvcc -c per source file, in parallel, into build/ (git-ignored), then one link step."""
    from concurrent.futures import ThreadPoolExecutor
    srcs = [os.path.join(CSRC, s) for s in CU_SOURCES]
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh", ".hpp"))]
    hdrs.append(os.path.join(ROOT, "include", "vloam_b200.h"))
    hdrs.append(os.path.abspath(__file__))
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    flags = [f for f in NVCC_FLAGS if f != "-shared"]
    objs = [os.path.join(objdir, os.path.basename(s)[:-3] + ".o") for s in srcs]

    def compile_one(i):
        if force or _stale(objs[i], [srcs[i]] + hdrs):
            subprocess.run(["nvcc"] + flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", objs[i], srcs[i]], check=True)
            return True
        return False
    with ThreadPoolExecutor(max_workers=len(srcs)) as ex:
        rebuilt = list(ex.map(compile_one, range(len(srcs))))
    if any(rebuilt) or _stale(LIB, objs):
        subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC", "-o", LIB] + objs, check=True)
    return LIB


def build_synth(force=False):
    src = os.path.join(HERE, "synth", "synth.cpp")
    if force or _stale(SYNTH_LIB, [src]):
        subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", SYNTH_LIB, src], check=True)
    return SYNTH_LIB
