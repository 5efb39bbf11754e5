"""Where the generic kernel finds the pixels of an edge strip (host_params.cpp EncodeSubRect / DecodeSubRect), on a machine
WITHOUT a GPU.  tests/native/subrect_check.cpp enumerates every valid encode and decode description over odd and tiny
sizes, splits each block the way the tuned launchers do (interior of width & ~3 or & ~7, right strip, odd last row) and
checks, with the generic kernels' own indexing, that every pixel of a strip addresses the same host bytes and plane
samples as in the whole block and that the three rectangles cover each pixel once.  A wrong offset would corrupt odd-sized
images only, and only on the GPU."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")


def test_sub_rectangles_address_the_pixels_of_the_whole_block(tmp_path):
    exe = tmp_path / "subrect_check"
    csrc = os.path.join(ROOT, "avif-format_b200", "csrc")
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", CUDA_INCLUDE, "-I", csrc,
                    os.path.join(ROOT, "tests", "native", "subrect_check.cpp"), os.path.join(csrc, "host_params.cpp"), "-o", str(exe)],
                   check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, timeout=600)
    print(out.stdout, out.stderr)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "ALL PASSED" in out.stdout
