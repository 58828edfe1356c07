"""Shared-memory layouts and the launch plan of the kernels, checked on the host (nvcc needed, no GPU):
tests/stubs/layout_check.cu includes the product's translation unit and verifies, for every series length 3 ... 460, that the
permuted model grid is a bijection with the four loads of a lane lane-contiguous, that the forward-model scratch, the ring
slots and the chain-per-warp regions have the sizes and parities the aligned 16-byte accesses assume, and that what the
kernels carve fits what tc_mcmc_run asks for.  On a B200's numbers it then runs tc_mcmc_run's own plan functions: the
series-length limit of each layout (that of include/tcmcmc.h, 441, for the big one) and of ss_stream_kernel, the kernel,
grid, time slices and solo-SM lag at the chain counts of test_gpu_chain_counts.py, and the partition of chains over 1 ... 8
devices."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_shared_memory_layout_invariants(tmp_path):
    from transcriptioncycleinference_b200 import build
    try:
        nvcc = build.nvcc_path()
    except RuntimeError:
        pytest.skip("nvcc not available")
    exe = str(tmp_path / "layout_check")
    cmd = [nvcc, "-O1", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
           os.path.join(ROOT, "tests", "stubs", "layout_check.cu")]
    if os.path.exists("/usr/bin/g++"):
        cmd += ["-ccbin", "/usr/bin/g++"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-2000:]
    run = subprocess.run([exe], capture_output=True, text=True)
    assert run.returncode == 0, run.stdout[-2000:]
    assert "layout check ok" in run.stdout
    assert "max N: regular 213 (two CTAs per SM 141), big 441, chain-per-warp 144, ss_stream_kernel 152" in run.stdout
    assert "schedules: 20 chain counts" in run.stdout
    assert "partitions: ok" in run.stdout
