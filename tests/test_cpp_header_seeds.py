"""k-mer seeding through the header-only C++ API (include/kmer_index.hpp): compiles on CPU, runs on the GPU box."""
import os
import subprocess

import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "cpp", "test_header_seeds.cpp")


def _compile(tmp_path):
    from kmer_index_b200 import build
    build.build()
    exe = str(tmp_path / "test_header_seeds")
    libdir = os.path.join(ROOT, "kmer_index_b200")
    subprocess.run(["g++", "-std=c++20", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe,
                    "-L", libdir, "-lkmer_b200", f"-Wl,-rpath,{libdir}"], check=True)
    return exe


def test_header_seeds_compiles_and_links(tmp_path):
    _compile(tmp_path)


@pytest.mark.gpu
def test_header_seeds_runs(tmp_path):
    exe = _compile(tmp_path)
    out = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr + out.stdout
    assert "all checks passed" in out.stdout
