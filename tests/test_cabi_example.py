"""A plain C program (tests/cpp/abi_example.c) compiles with gcc against include/nvbio_b200.h and links the shared library -- no nvcc,
no C++, no torch: the view a foreign-language binding has of the C ABI -- and reproduces the reference-asserted problems on the GPU."""
import os
import subprocess
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build(out_dir):
    """the example program, built in out_dir: the source tree may be read-only"""
    from nvbio_b200 import build as b
    b.build()
    exe = os.path.join(str(out_dir), "abi_example")
    cmd = ["gcc", "-O1", "-std=c11", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"), "-I/usr/local/cuda/include",
           os.path.join(ROOT, "tests", "cpp", "abi_example.c"), "-o", exe,
           "-L" + os.path.join(ROOT, "nvbio_b200"), "-lnvbio_b200", "-L/usr/local/cuda/lib64", "-lcudart",
           "-Wl,-rpath," + os.path.join(ROOT, "nvbio_b200"), "-Wl,-rpath,/usr/local/cuda/lib64"]
    subprocess.check_call(cmd)
    return exe


def test_c_program_compiles_and_links(tmp_path):
    exe = build(tmp_path)
    assert os.path.exists(exe)


@pytest.mark.gpu
def test_c_program_runs(tmp_path):
    exe = build(tmp_path)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "score -11 sink (165,150)" in r.stdout and "full score 13 sink (18,7)" in r.stdout
