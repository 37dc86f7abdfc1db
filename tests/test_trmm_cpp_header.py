"""The C++ surface of the triangular multiplication (include/dlaf/multiplication/triangular.h) compiled with g++ on the
host, no GPU: dlaf::triangular_multiplication instantiated for the four element types by tests/trmm_header_check.cpp."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def test_triangular_multiplication_header_instantiates(tmp_path):
    exe = tmp_path / "trmm_header_check"
    cmd = ["g++", "-std=c++17", "-O1", "-Wall", f"-I{ROOT}/include", "-I/usr/local/cuda/include", os.path.join(HERE, "trmm_header_check.cpp"),
           "-o", str(exe), f"-L{ROOT}/dla-future_b200/lib", "-ldlaf_b200", "-L/usr/local/cuda/lib64", "-lcudart",
           f"-Wl,-rpath,{ROOT}/dla-future_b200/lib", "-Wl,-rpath,/usr/local/cuda/lib64"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, (r.stdout, r.stderr)
    assert "instantiated for s d c z: ok" in r.stdout
