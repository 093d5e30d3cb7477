"""The C++ host mirror of the BGZF reader (v2p::VcfText::load_bgzf, include/v2p_host.hpp): builds and links everywhere, the
program itself (a bgzip'd file cut inside the #CHROM line and a cell, the CRC and not-BGZF errors) runs on the GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "vcf_bgzf_host_test.cpp")


@pytest.fixture(scope="module")
def binary(tmp_path_factory):
    from vcf2prot_b200 import _lib

    if not os.path.isfile(_lib.LIB_PATH):
        import __graft_entry__ as g

        g.build()
    out = str(tmp_path_factory.mktemp("cpp") / "vcf_bgzf_host_test")
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-I", os.path.join(ROOT, "include"), SRC, "-o", out,
                           "-L", libdir, "-lv2p_engine", "-Wl,-rpath," + libdir])
    return out


def test_cpp_vcf_bgzf_mirror_builds(binary):
    p = subprocess.run([binary, "--no-gpu"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0 and "OK" in p.stdout, p.stdout


@pytest.mark.gpu
def test_cpp_vcf_bgzf_mirror_on_gpu(binary):
    p = subprocess.run([binary], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert p.returncode == 0 and p.stdout.strip().endswith("OK"), p.stdout
