"""Memory safety of the CUDA kernels and the host glue: the SIMT-emulated kernels (device buffers are heap blocks there)
and the host pipeline built with AddressSanitizer, run over short, paired, long and ragged reads and the kernel variants.
Any report fails the test; the SAM must still equal the reference's."""
import os
import subprocess

import pytest

from conftest import ROOT, md5, ref_sam_md5, strip_pg

ASAN_BIN = os.path.join(ROOT, "tests", "_build", "bwa-b200-cusim-asan")
RUNS = [
    ("stress_pe", "stress", dict(tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05), [], {}),
    ("stress_pe_global_scratch", "stress", dict(tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05), [],
     {"BWA_B200_K4_SM": "0", "BWA_B200_K5_SM": "0"}),
    ("stress_se_table9_dense_sa2", "stress", dict(tag="cs", n=120, seed=33, err=(0.016, 0.002, 0.002), chimeric=0.05), [], {"BWA_B200_KTAB": "9", "BWA_B200_SA_INTV": "2"}),
    ("two_1k", "two", dict(tag="cs1k", n=6, length=1000, seed=35), [], {}),
    ("two_pacbio_4k", "two", dict(tag="cspb", n=3, length=4000, seed=36, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"], {}),
]


@pytest.fixture(scope="module")
def asan_bin():
    r = subprocess.run(["make", "asan"], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0 or not os.path.exists(ASAN_BIN):
        pytest.skip("AddressSanitizer build not available: " + r.stdout.decode()[-300:])
    return ASAN_BIN


@pytest.mark.parametrize("name,ref,kw,extra,env", RUNS, ids=[r[0] for r in RUNS])
def test_emulated_kernels_under_asan(data, asan_bin, name, ref, kw, extra, env):
    fa, fqs = data.reads(ref, **kw)
    args = extra + ["-K", "100000000", "-t", "2", fa] + fqs
    e = dict(os.environ, ASAN_OPTIONS="detect_stack_use_after_return=0:detect_leaks=0", **env)   # fibers switch stacks by hand
    p = subprocess.run([asan_bin, "mem", "-v", "1"] + args, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert b"AddressSanitizer" not in p.stderr, p.stderr.decode()[-3000:]
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    assert md5(strip_pg(p.stdout)) == ref_sam_md5(args)
