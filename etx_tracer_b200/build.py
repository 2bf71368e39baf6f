"""Builds the CUDA module in-tree for sm_100a (nvcc cross-compiles without a GPU).

  libetx_b200.so         product build ("fast": FMA contraction, CUDA math library)
  libetx_b200_parity.so  strict-IEEE build (-fmad=false, portable transcendentals) used by the bit-exact parity tests
  libetx_b200_count.so   product build + traversal counters (bench.py roofline pass)

The alternatives measured against "fast" (round 1's IEEE division / sqrt with the CUDA math library; other resident-block counts for the
bounce, connection and gather kernels) are recorded in DESIGN.md §5 and the constants in kernels.cuh; they are not built.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SOURCES = ["module.cu", "bvh_build.cpp", "film_io.cpp", "scene_loader.cpp"]
HEADERS = ["bvh.h", "bvh_build.h", "dcore.cuh", "dscene.cuh", "dimage.cuh", "dbsdf.cuh", "dclosure.cuh", "dtrace.cuh", "dtrav.cuh", "dwide.cuh", "dmedium.cuh", "dsss.cuh", "dvcm.cuh", "dpt.cuh", "kernels.cuh", "kernels_pt.cuh", "portable_math.h", "scene_loader_formats.inl", "scene_loader_build.inl", "scene_loader_atmosphere.inl", "scene_loader_tangents.inl", "scene_loader_nvdb.inl", "scene_loader_jpeg.inl",
           os.path.join("..", "..", "include", "etx_b200.h")]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC,-ffp-contract=off", "-shared", "--expt-relaxed-constexpr", "-Wno-deprecated-gpu-targets"]
FLAVORS = {
    # product build: approximate division / square root (div.approx 2 ulp, no slow-path subroutine at each of the ~500 division sites of a
    # BSDF kernel), flush-to-zero; transcendentals are the special-function unit's (dcore.cuh)
    "fast": (os.path.join(HERE, "libetx_b200.so"), ["-prec-div=false", "-prec-sqrt=false", "-ftz=true"]),
    # "fast" + per-ray node / triangle counters in every traversal (bench.py's roofline pass reads n_node / n_tri from it: SURVEY 8(d) wants the
    # algorithmic bytes with and without the BVH term; the counters cost registers, so the timed build does not carry them)
    "count": (os.path.join(HERE, "libetx_b200_count.so"), ["-prec-div=false", "-prec-sqrt=false", "-ftz=true", "-DETXB_COUNT_TRAVERSAL=1"]),
    "parity": (os.path.join(HERE, "libetx_b200_parity.so"), ["-fmad=false", "-DETXB_PARITY=1"]),
}


def lib_path(flavor="fast"):
    return FLAVORS[flavor][0]


# what each translation unit includes (the per-flavour objects are rebuilt when one of these is newer)
UNIT_DEPS = {
    "module.cu": [h for h in HEADERS if not h.endswith(".inl")],
    "bvh_build.cpp": ["bvh.h", "bvh_build.h"],
    "film_io.cpp": [os.path.join("..", "..", "include", "etx_b200.h")],
    "scene_loader.cpp": ["scene_loader_formats.inl", "scene_loader_build.inl", "scene_loader_atmosphere.inl", "scene_loader_tangents.inl", "scene_loader_nvdb.inl", "scene_loader_jpeg.inl", os.path.join("..", "..", "include", "etx_b200.h")],
}
OBJ_ROOT = os.path.join(HERE, "build")  # git-ignored scratch: objects, one folder per flavour


def _newer(deps, out):
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def _stale(out):
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return _newer(deps, out)


def build(flavors=("fast", "parity", "count"), force=False, verbose=False, extra=()):
    """Every translation unit is compiled to an object per flavour (the CUDA unit takes minutes, the host units seconds), then linked; the shared
    library is written beside its final name and renamed, so a half-written file is never what a loader (or a `gpurun` snapshot) sees."""
    compile_flags = [f for f in COMMON if f != "-shared"]
    jobs = []
    for fl in flavors:
        out, flags = FLAVORS[fl]
        if not force and not _stale(out):
            continue
        odir = os.path.join(OBJ_ROOT, fl)
        os.makedirs(odir, exist_ok=True)
        objs = []
        for src in SOURCES:
            obj = os.path.join(odir, os.path.splitext(src)[0] + ".o")
            objs.append(obj)
            deps = [os.path.join(CSRC, src)] + [os.path.join(CSRC, d) for d in UNIT_DEPS[src]] + [os.path.abspath(__file__)]
            if force or extra or _newer(deps, obj):
                cmd = ["nvcc"] + ARCH + compile_flags + flags + list(extra) + ["-c", os.path.join(CSRC, src), "-o", obj]
                if verbose:
                    cmd.insert(1, "-Xptxas=-v")
                    print(" ".join(cmd), flush=True)
                jobs.append((fl, cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for fl, cmd, p in jobs:
        text, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed for flavor {fl}:\n{' '.join(cmd)}\n{text}")
        if verbose:
            print(text)
    for fl in flavors:
        out, flags = FLAVORS[fl]
        if not force and not _stale(out):
            continue
        objs = [os.path.join(OBJ_ROOT, fl, os.path.splitext(src)[0] + ".o") for src in SOURCES]
        cmd = ["nvcc"] + ARCH + ["-shared", "-Wno-deprecated-gpu-targets"] + objs + ["-o", out + ".tmp"]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"link failed for flavor {fl}:\n{' '.join(cmd)}\n{r.stdout}")
        os.replace(out + ".tmp", out)
    return [FLAVORS[f][0] for f in flavors]


if __name__ == "__main__":
    which = tuple(a for a in sys.argv[1:] if a in FLAVORS) or ("fast", "parity", "count")
    build(which, force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built", [lib_path(f) for f in which])
