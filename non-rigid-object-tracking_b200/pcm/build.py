"""Builds libpcm_b200.so (the C-ABI library of include/pcm_b200.h) in-tree with nvcc
for sm_100a.  nvcc cross-compiles without a GPU, so this runs in the build container;
the resulting .so travels to the GPU box with the repo snapshot."""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(PKG, "csrc")
LIB = os.environ.get("PCM_LIB_PATH") or os.path.join(PKG, "libpcm_b200.so")
# translation units: (source, extra defines, object name); K1 is instantiated once per tile height in its own unit
UNITS = [("pcm_api.cu", [], "pcm_api.o"),
         ("pcm_score_inst.cu", ["-DPCM_PPT=6"], "pcm_score_ppt6.o"),
         ("pcm_score_inst.cu", ["-DPCM_PPT=7"], "pcm_score_ppt7.o"),
         ("pcm_score_inst.cu", ["-DPCM_PPT=8"], "pcm_score_ppt8.o"),
         ("pcm_host_simd.cpp", [], "pcm_host_simd.o"),
         ("pcm_felzenszwalb.cpp", [], "pcm_felzenszwalb.o"),
         ("pcm_slic.cpp", [], "pcm_slic.o")]
DEPS = ["pcm_api.cu", "pcm_score_inst.cu", "pcm_score_variants.h", "pcm_score.cuh", "pcm_kernels.cuh", "pcm_device.cuh", "pcm_host.h",
        "pcm_host_simd.cpp", "pcm_felzenszwalb.cpp", "pcm_slic.cpp", "pcm_slic.cuh", "pcm_felzenszwalb.cuh", "pcm_quickshift.cuh", "pcm_forest_fit.cuh", "pcm_prior.cuh",
        os.path.join("..", "..", "include", "pcm_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-pthread", "-Xcompiler", "-ffp-contract=off",
    "-Xptxas", "-v",
]


def needs_build():
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(os.path.join(CSRC, d)) > t for d in DEPS)


def build(force=False, verbose=False):
    """Compile if sources are newer than the library (the translation units in parallel).  Returns the library path."""
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "nvcc")
    extra = os.environ.get("PCM_BUILD_DEFS", "").split()      # e.g. "-DPCM_NTHREADS=512" (tuning experiments)
    objdir = os.path.join(PKG, "build", "obj" if LIB.endswith("libpcm_b200.so") else "obj_" + os.path.basename(LIB))
    os.makedirs(objdir, exist_ok=True)
    procs = []
    for src, defs, obj in UNITS:
        cmd = [nvcc] + NVCC_FLAGS + extra + defs + ["-c", "-o", os.path.join(objdir, obj), os.path.join(CSRC, src)]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    log = []
    for cmd, pr in procs:
        out, err = pr.communicate()
        log.append(out + err)
        if verbose or pr.returncode != 0:
            sys.stderr.write(out + err)
        if pr.returncode != 0:
            for _, other in procs:
                if other.poll() is None:
                    other.kill()
            raise RuntimeError("nvcc failed (%d): %s" % (pr.returncode, " ".join(cmd)))
    link = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-pthread", "-o", LIB] + \
           [os.path.join(objdir, obj) for _, _, obj in UNITS]
    res = subprocess.run(link, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("link failed (%d): %s" % (res.returncode, " ".join(link)))
    if LIB.endswith("libpcm_b200.so"):       # registers / spills / shared memory per kernel (ptxas -v), without timings
        with open(os.path.join(PKG, "build", "ptxas_info.txt"), "w") as f:
            f.write("".join(l for text in log for l in text.splitlines(True) if "Compile time" not in l))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
