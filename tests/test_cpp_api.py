"""include/blsgpu.hpp (the C++ mirror of src/bls.rs): compiles and links against libblsgpu everywhere; without a GPU it
must refuse to run (no CPU fallback); on the B200 box it runs the reference-shaped checks."""
import os, subprocess, tempfile
import pytest
from conftest import ROOT

def _build():
    from bls_verify_gadget_b200 import _lib
    so = _lib.build(); exe = os.path.join(ROOT, "tests", "_hostemu", "test_api")
    try: os.makedirs(os.path.dirname(exe), exist_ok=True)
    except OSError: pass
    if not os.access(os.path.dirname(exe), os.W_OK): exe = os.path.join(tempfile.mkdtemp(prefix="blsgpu-cpp-api-"), "test_api")      # read-only tree
    src = os.path.join(ROOT, "tests", "cpp", "test_api.cpp")
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", os.path.join(ROOT, "include"), src, "-o", exe, "-L", os.path.dirname(so), "-lblsgpu",
                           "-Wl,-rpath," + os.path.dirname(so), "-Wl,-rpath,/usr/local/cuda/lib64"])
    return exe

def test_cpp_api_builds_and_refuses_without_gpu():
    import torch
    exe = _build()
    if torch.cuda.is_available(): pytest.skip("GPU present: covered by the gpu test")
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 3 and "NO_GPU" in r.stdout

@pytest.mark.gpu
def test_cpp_api_on_gpu():
    r = subprocess.run([_build()], capture_output=True, text=True)
    assert r.returncode == 0 and "OK" in r.stdout, r.stdout + r.stderr
