"""Build libagcf.so in-tree (nvcc, sm_100a only):  python -m arlib_b200.build"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))


def _nvcc():
    """nvcc from PATH, else from the CUDA toolkit torch finds (CUDA_HOME / CUDA_PATH / the default install)."""
    if shutil.which("nvcc"):
        return "nvcc"
    from torch.utils.cpp_extension import CUDA_HOME
    if CUDA_HOME is None or not os.path.isfile(os.path.join(CUDA_HOME, "bin", "nvcc")):
        raise RuntimeError("nvcc not found: put the CUDA toolkit's bin/ on PATH or set CUDA_HOME")
    return os.path.join(CUDA_HOME, "bin", "nvcc")


def build(verbose=True, force=False):
    csrc = os.path.join(HERE, "csrc")
    if force:
        subprocess.run(["make", "-C", csrc, "clean"], check=True, stdout=subprocess.DEVNULL)
    res = subprocess.run(["make", "-C", csrc, "-j4", "NVCC=" + _nvcc()], stdout=subprocess.PIPE,
                         stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout[-4000:])
    if res.returncode != 0:
        raise RuntimeError("building libagcf.so failed")
    return os.path.join(HERE, "libagcf.so")


if __name__ == "__main__":
    build(force="--force" in sys.argv)
