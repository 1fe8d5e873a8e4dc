"""The header-only C++ API (include/kmer_index.hpp) over the C ABI: compiles on CPU, runs on the GPU box."""
import os
import subprocess

import pytest

from conftest import ROOT

SRC = os.path.join(ROOT, "tests", "cpp", "test_header.cpp")


def _compile(tmp_path):
    from kmer_index_b200 import build
    build.build()
    exe = str(tmp_path / "test_header")
    libdir = os.path.join(ROOT, "kmer_index_b200")
    subprocess.run(["g++", "-std=c++20", "-O2", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), SRC, "-o", exe,
                    "-L", libdir, "-lkmer_b200", f"-Wl,-rpath,{libdir}"], check=True)
    return exe


def test_header_compiles_and_links(tmp_path):
    _compile(tmp_path)


def test_header_bench_tool_compiles(tmp_path):
    """profiles/tools/header_bench.cpp (the drop-in header on a batch held as std::vector<std::vector<dna4>>) stays in
    step with the header: it must compile and link against the library."""
    from kmer_index_b200 import build
    build.build()
    libdir = os.path.join(ROOT, "kmer_index_b200")
    subprocess.run(["g++", "-std=c++20", "-O2", "-Wall", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "profiles", "tools", "header_bench.cpp"), "-o", str(tmp_path / "header_bench"),
                    "-L", libdir, "-lkmer_b200", f"-Wl,-rpath,{libdir}", "-pthread"], check=True)


@pytest.mark.gpu
def test_header_runs(tmp_path):
    exe = _compile(tmp_path)
    import torch
    env = dict(os.environ, KMER_B200_TEST_DEVICES=str(min(torch.cuda.device_count(), 4)))
    out = subprocess.run([exe, str(tmp_path)], capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0, out.stderr + out.stdout
    assert "all checks passed" in out.stdout
