"""Build the REFERENCE's own attribute-coder extension (HAC/submodules/arithmetic.zip) into oracle/_ref/arithmetic.so.

TEST INFRASTRUCTURE ONLY.  The sources stay where they are: the zip is unpacked into a temporary directory, compiled with
the reference's own flags (setup.py: -O2) for sm_100a, and only the shared object is kept (oracle/_ref/ is git-ignored and
travels to the GPU box).  tests/test_attr_coder.py and tests/bench_attr_coder.py import it when present to compare the library's
streams and symbols with the reference kernels' on the same B200; nothing in gauspcc_b200/ ever loads it.

    python oracle/build_ref_arithmetic.py <checkout of the reference>
"""
import glob
import os
import shutil
import sys
import tempfile
import zipfile

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "_ref", "arithmetic.so")


def build(reference_root, force=False):
    zpath = os.path.join(reference_root, "src/gs_compress/HAC/submodules/arithmetic.zip")
    if not os.path.exists(zpath):
        return None
    if os.path.exists(OUT) and not force:
        return OUT
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0a")
    from torch.utils.cpp_extension import load
    tmp = tempfile.mkdtemp(prefix="ref_arithmetic_")
    with zipfile.ZipFile(zpath) as z:
        z.extractall(tmp)
    src = os.path.join(tmp, "arithmetic")
    bdir = os.path.join(tmp, "build")
    os.makedirs(bdir)
    load(name="arithmetic", sources=glob.glob(os.path.join(src, "*.cpp")) + glob.glob(os.path.join(src, "*.cu")),
         extra_include_paths=[os.path.join(src, "include")], extra_cflags=["-O2"], extra_cuda_cflags=["-O2"],
         build_directory=bdir, is_python_module=False, verbose=False)
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    shutil.copy(os.path.join(bdir, "arithmetic.so"), OUT)
    shutil.rmtree(tmp, ignore_errors=True)
    return OUT


def load_module():
    """import the built extension as a Python module, or None when it was never built"""
    if not os.path.exists(OUT):
        return None
    import importlib.util
    import torch  # noqa: F401  (libtorch must be loaded first)
    spec = importlib.util.spec_from_file_location("arithmetic", OUT)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    print(build(sys.argv[1], force=True))
