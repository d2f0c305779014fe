"""In-tree build of libbezgpu.so (nvcc, sm_100a).  Used by __graft_entry__.build().

Translation units
  plan.cu         plan + error plumbing
  constraints.cu  fused constraint kernels (FMA contraction allowed: the
                  reference's BLAS path is not bit-reproducible anyway)
  geometry.cu     split / extrema / GJK / minDist / collCheck -- compiled with
                  -fmad=false so results are bit-identical to the reference's
                  numba/numpy rounding (SURVEY Q13)
"""
import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libbezgpu.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
          "-I", os.path.join(ROOT, "include"), "-I", CSRC]

UNITS = [
    ("plan.cu", []),
    ("constraints.cu", []),
    ("constraints_mma.cu", []),
    ("constraints_mma_pair_a.cu", []),
    ("constraints_mma_pair_b.cu", []),
    ("constraints_mma_pair_c.cu", []),
    ("constraints_mma_pair_d.cu", []),
    ("constraints_mma_speed_a.cu", []),
    ("constraints_mma_speed_b.cu", []),
    ("jacobian.cu", []),
    ("angrate.cu", []),
    ("angrate_jac.cu", []),
    ("curveops.cu", []),
    ("geometry.cu", ["-fmad=false"]),
]


def _nvcc():
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; cannot build libbezgpu.so")
    return nvcc


def _stale(target, sources):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build(force=False, verbose=False):
    """Full build, or -- with BEZGPU_ONLY_N=<degree> in the environment -- a development
    build whose fused kernels are instantiated for that degree only (seconds instead
    of minutes).  The flavor of the linked library is recorded in libbezgpu.flavor so a
    later full build() always relinks over a development library."""
    nvcc = _nvcc()
    only_n = os.environ.get("BEZGPU_ONLY_N", "")
    flavor = "n" + only_n if only_n else "full"
    suffix = "." + flavor + ".o" if only_n else ".o"
    dev = ["-DBEZ_ONLY_N=" + only_n] if only_n else []
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(ROOT, "include", "bezgpu.h"))
    objs = []
    procs = []
    for name, extra in UNITS:
        src = os.path.join(CSRC, name)
        if not os.path.exists(src):
            continue
        obj = os.path.join(CSRC, name[:-3] + suffix)
        objs.append(obj)
        if force or _stale(obj, [src] + hdrs):
            cmd = [nvcc] + ARCH + COMMON + extra + dev + (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj]
            procs.append((name, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for name, cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(out)
        if p.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s" % (name, " ".join(cmd)))
    stamp = os.path.join(PKG, "libbezgpu.flavor")
    linked = open(stamp).read().strip() if os.path.exists(stamp) else ""
    if force or procs or _stale(LIB, objs) or linked != flavor:
        cmd = [nvcc] + ARCH + ["-shared", "-o", LIB] + objs + ["-lcudart"]
        subprocess.check_call(cmd)
        with open(stamp, "w") as f:
            f.write(flavor + "\n")
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
