"""Differential tests over pseudo-random option sets (tests/fuzz_cases.py): scoring, band, seeding, chaining and
output options, presets, read lengths 36-400, error rates, chimeras, batch sizes.  The CPU half runs the CUDA
kernels in the SIMT emulator, the GPU half the real ones; both must reproduce the reference SAM byte for byte
(or fail with the same exit status on an option set the reference rejects)."""
import os
import subprocess

import pytest

import bwa_b200
from conftest import CUSIMBIN, md5, ref_run, strip_pg
from fuzz_cases import command

# BWA_B200_FUZZ_FROM/TO widen the emulated sweep (e.g. 10..300 after a kernel change); the default keeps the CPU suite short
CPU_CASES = list(range(int(os.environ.get("BWA_B200_FUZZ_FROM", "0")), int(os.environ.get("BWA_B200_FUZZ_TO", "10"))))
REGRESSIONS = [114]   # 114: a tandem-repeat read whose regions merge one by one (146 device rounds in one batch)
CPU_CASES += [k for k in REGRESSIONS if k not in CPU_CASES]
GPU_CASES = list(range(0, 24)) + [114]


def _both(binary, args):
    r = ref_run("bwa", ["mem", "-v", "1"] + args)
    g = subprocess.run([binary, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert (r["rc"] == 0) == (g.returncode == 0), g.stderr.decode()[-2000:]
    if r["rc"] == 0:
        assert md5(strip_pg(g.stdout)) == r["md5"]


@pytest.mark.parametrize("k", CPU_CASES)
def test_emulated_kernels_random_options(data, k):
    _both(CUSIMBIN, command(data, k))


@pytest.mark.gpu
@pytest.mark.parametrize("k", GPU_CASES)
def test_gpu_random_options(data, k):
    _both(bwa_b200.CLI_PATH, command(data, k))
