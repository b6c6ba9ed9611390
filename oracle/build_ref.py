"""Build the REFERENCE's own CUDA extensions for sm_100a into oracle/_ref/ (git-ignored).

TEST INFRASTRUCTURE ONLY.  Compiles the sources WHERE THEY LIE under <reference>/extensions, a checkout of
facebookresearch/goliath at $GOLIATH_REFERENCE or, by default, at the `reference_path` BASELINE.json records (nothing
is copied into the repo), with the reference's own flags (setup.py of each
extension: -use_fast_math where it says so, -std=c++17, -lineinfo) except the gencode, which is sm_100a.  The outputs
are the reference's pybind modules `sgutilslib`, `utilslib`, `mvpraymarchlib`; tests/golden/make_ref_kernels_golden.py
records their outputs as the fixtures the GPU tests compare our kernels against, and bench.py --ext-compare times them
as the reference arm of the extension-level ratios.  gsplat is third-party and absent: it cannot be built here.

Usage: [GOLIATH_REFERENCE=<goliath checkout>] python oracle/build_ref.py [sgutilslib utilslib mvpraymarchlib]
"""
import json
import os
import subprocess
import sys
import sysconfig
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref")


def reference_dir():
    """$GOLIATH_REFERENCE, else the reference checkout BASELINE.json records."""
    if os.environ.get("GOLIATH_REFERENCE"):
        return os.environ["GOLIATH_REFERENCE"]
    with open(os.path.join(os.path.dirname(HERE), "BASELINE.json")) as f:
        return json.load(f)["reference_path"]


REF = os.path.join(reference_dir(), "extensions")

EXTS = {
    "sgutilslib": dict(dir="sgutils", sources=["sg.cu"], fast_math=True),
    "utilslib": dict(dir="utils", sources=["utils.cpp", "utils_kernel.cu"], fast_math=False),
    "mvpraymarchlib": dict(dir="mvpraymarch", sources=["mvpraymarch.cpp", "mvpraymarch_kernel.cu", "bvh.cu"],
                           fast_math=True),
}


def torch_flags():
    import torch
    from torch.utils import cpp_extension as ce

    inc = ce.include_paths("cuda") if "device_type" in ce.include_paths.__code__.co_varnames else ce.include_paths(True)
    libdir = os.path.join(os.path.dirname(torch.__file__), "lib")
    abi = int(torch._C._GLIBCXX_USE_CXX11_ABI)
    return inc, libdir, abi


def build_one(name):
    spec = EXTS[name]
    inc, libdir, abi = torch_flags()
    os.makedirs(os.path.join(OUT, "obj"), exist_ok=True)
    pyinc = sysconfig.get_paths()["include"]
    common = ["-I" + os.path.join(REF, "include"), "-I" + os.path.join(REF, spec["dir"]), "-I" + pyinc] + \
             ["-I" + p for p in inc] + ["-DTORCH_EXTENSION_NAME=" + name, "-DTORCH_API_INCLUDE_EXTENSION_H",
                                        "-D_GLIBCXX_USE_CXX11_ABI=%d" % abi]
    objs = []
    for src in spec["sources"]:
        path = os.path.join(REF, spec["dir"], src)
        obj = os.path.join(OUT, "obj", name + "_" + src.replace(".", "_") + ".o")
        objs.append(obj)
        if src.endswith(".cu"):
            cmd = ["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-lineinfo", "-O3",
                   "--expt-relaxed-constexpr", "-Xcompiler", "-fPIC", "-D__CUDA_NO_HALF_OPERATORS__",
                   "-D__CUDA_NO_HALF_CONVERSIONS__", "-D__CUDA_NO_HALF2_OPERATORS__"] + \
                  (["-use_fast_math"] if spec["fast_math"] else []) + common + ["-c", path, "-o", obj]
        else:
            cmd = ["g++", "-std=c++17", "-O3", "-fPIC", "-DNDEBUG"]  # setuptools CFLAGS carry -DNDEBUG; utils.cpp:67 only compiles with it
            cmd = cmd + common + ["-c", path, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("%s\n%s" % (" ".join(cmd), r.stderr[-4000:]))
    so = os.path.join(OUT, name + ".so")
    link = ["g++", "-shared", "-o", so] + objs + ["-L" + libdir, "-L/usr/local/cuda/lib64", "-lc10", "-lc10_cuda",
                                                  "-ltorch_cpu", "-ltorch_cuda", "-ltorch", "-ltorch_python",
                                                  "-lcudart", "-Wl,-rpath," + libdir]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("%s\n%s" % (" ".join(link), r.stderr[-4000:]))
    return so


def build(names=None):
    if not os.path.isdir(REF):
        sys.stderr.write("oracle/build_ref.py: no reference checkout at %s (set GOLIATH_REFERENCE): the reference's "
                         "extensions are not built; bench.py --ext-compare and the reference arms of the MVP configs, and "
                         "tests/golden/make_ref_kernels_golden.py need them\n" % os.path.dirname(REF))
        return []
    names = names or list(EXTS)
    with ThreadPoolExecutor(max_workers=3) as ex:
        return list(ex.map(build_one, names))


if __name__ == "__main__":
    print(build(sys.argv[1:] or None))
