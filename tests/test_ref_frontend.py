"""Boundary proof from the reference side (INTEGRATION.md 1-2, SURVEY.md 8b): the reference's OWN front end (main.c,
fastmap.c, kopen.c, utils.c, bwa.c, ... everything of its `bwa` binary except bwamem.o/bwamem_pair.o) and its OWN
library example (example.c), compiled from the reference sources against the reference's headers by oracle/Makefile
(`make frontend[-cusim]`) and LINKED against this repository's library, must print what the unmodified reference
prints.  CPU: the library is the SIMT-emulated build of the CUDA kernels; -m gpu: libbwa_b200.so itself."""
import os
import subprocess

import pytest

from conftest import ROOT, md5, ref_run, ref_sam_md5, strip_pg

REF_DIR = os.path.join(ROOT, "oracle", "_ref")


def _frontend(kind):
    exe = os.path.join(REF_DIR, "ref_frontend_" + kind), os.path.join(REF_DIR, "ref_example_" + kind)
    # built from the reference's sources (oracle/Makefile REF=<lh3/bwa 0.7.19 tree>) when they are there; without them the
    # target keeps what build() made earlier, and the test needs such a build
    target = "frontend" if kind == "b200" else "frontend-cusim"
    subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), target], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    if not all(os.path.exists(e) for e in exe):
        pytest.skip("front ends not built: make -C oracle frontend frontend-cusim needs the reference sources")
    return exe


def _head(src, dst, n_reads):
    with open(src, "rb") as f, open(dst, "wb") as o:
        for i, line in enumerate(f):
            if i >= 4 * n_reads:
                break
            o.write(line)
    return dst


def _mem(exe, args):
    r = subprocess.run([exe, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    return strip_pg(r.stdout)


def _check(kind, data, tmp_path, n_pe, n_ex, extra):
    front, ex_mine = _frontend(kind)
    fa, fqs = data.reads("stress", tag="fe", n=3000, seed=4, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    fqs = [_head(f, str(tmp_path / os.path.basename(f)), n_pe) for f in fqs]
    args = extra + ["-K", "100000000", "-t", "4", fa] + fqs
    assert md5(_mem(front, args)) == ref_sam_md5(args)
    # example.c: mem_align1 + mem_reg2aln per region + free(ar.a), on single-end reads
    fa1, fq1 = data.reads("c1", tag="se", n=2000, seed=11)
    fq = _head(fq1[0], str(tmp_path / "ex.fq"), n_ex)
    want = ref_run("ref_example", [fa1, fq], "raw")
    got = subprocess.run([ex_mine, fa1, fq], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900)
    assert got.returncode == 0, got.stderr.decode()[-2000:]
    assert want["rc"] == 0 and md5(got.stdout) == want["md5"] and want["lines"] >= n_ex // 2


def test_reference_frontend_over_emulated_library(built, data, tmp_path):
    _check("cusim", data, tmp_path, 150, 60, [])


@pytest.mark.gpu
def test_reference_frontend_over_cuda_library(data, tmp_path):
    # with the real library the read-group line set by the reference's own option parser reaches this library's SAM
    # emitter through the interposed globals bwa_rg_id / bwa_pg (bwa.c:42-45)
    _check("b200", data, tmp_path, 3000, 400, ["-R", "@RG\\tID:x\\tSM:y"])
