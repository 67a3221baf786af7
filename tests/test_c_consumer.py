"""A compiled C host program that includes the REFERENCE's hap.h (oracle/_ref/c_consumer_ref, built by oracle/Makefile
where the reference sources are present) or include/hap.h, and links libhap_b200.so -- the drop-in boundary exercised
the way a C application would."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c_consumer", "consumer.c")
BUILD = os.path.join(ROOT, "tests", "emu", "_build")
LIBDIR = os.path.join(ROOT, "hap_b200")


def build(which: str) -> str:
    if which == "ref":
        exe = os.path.join(ROOT, "oracle", "_ref", "c_consumer_ref")
        return exe if os.path.exists(exe) else ""
    inc = os.path.join(ROOT, "include")
    exe = os.path.join(BUILD, "c_consumer_" + which)
    os.makedirs(BUILD, exist_ok=True)
    subprocess.run(["gcc", "-std=c99", "-O1", "-Wall", "-Werror", "-D_GNU_SOURCE", "-I", inc, SRC, "-o", exe, "-L", LIBDIR,
                    "-l:libhap_b200.so", "-Wl,-rpath," + LIBDIR, "-pthread"], check=True)
    return exe


@pytest.mark.parametrize("which", ["ref", "own"])
def test_c_consumer_container_paths(which):
    import hap_b200
    hap_b200.load()
    exe = build(which)
    if not exe:
        pytest.skip("reference build (oracle/_ref) not present")
    p = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert p.returncode == 0 and "consumer ok" in p.stdout, p.stdout + p.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("which", ["ref", "own"])
def test_c_consumer_gpu_paths(which):
    exe = build(which)
    if not exe:
        pytest.skip("reference build (oracle/_ref) not present")
    p = subprocess.run([exe, "--gpu"], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and "GPU paths" in p.stdout, p.stdout + p.stderr
