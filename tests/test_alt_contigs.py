"""ALT contigs (.alt file next to the index, bntseq.c:178-209): is_alt drives a second sort in primary marking, alt_sc / pa:f, XA
limits and the supplementary-ALT record (bwamem.c:560-584, bwamem_extra.c:124-172, bwamem_pair.c:371-378).  Reads over ALT contigs
leave the device post-processing (stage 4 flags them) and take the host path; the SAM must be the reference's either way.
Also: duplicate contig names (the LAST one is marked) and an unterminated last line (ignored), as in the reference's parser."""
import os
import shutil
import subprocess

import numpy as np
import pytest

import bwa_b200
from conftest import CUSIMBIN, index, md5, ref_sam_md5, run_sam


def _make(tmp_path):
    import gen_data
    rng = np.random.default_rng(77)
    base = gen_data.random_contigs(1, 60000, 5)[0]
    alt = base[20000:26000].copy()                      # an ALT haplotype of a stretch of chr1 with 1.5 % divergence
    mut = rng.random(len(alt)) < 0.015
    alt[mut] = gen_data.ACGT[rng.integers(0, 4, size=int(mut.sum()))]
    other = gen_data.random_contigs(1, 8000, 6)[0]
    fa = str(tmp_path / "alt.fa")
    with open(fa, "wb") as f:
        for name, seq in ((b"chr1", base), (b"dup", other[:4000]), (b"chr1_alt", alt), (b"dup", other[4000:])):
            f.write(b">" + name + b"\n" + seq.tobytes() + b"\n")
    index(fa)
    with open(fa + ".alt", "w") as f:
        f.write("@comment line\nchr1_alt\t0\t*\ndup\nchr1")      # last line unterminated: not an ALT contig
    contigs = [base, alt, other]
    r1, r2 = gen_data.gen_reads([base, alt], 300, 150, 3, paired=True)
    fqs = [str(tmp_path / "a_1.fq"), str(tmp_path / "a_2.fq")]
    gen_data.write_fastq(fqs[0], r1); gen_data.write_fastq(fqs[1], r2)
    s1, _ = gen_data.gen_reads([base[19000:27000], other], 200, 150, 4)
    se = str(tmp_path / "a_se.fq")
    gen_data.write_fastq(se, s1)
    return fa, fqs, se


def _check(binary, tmp_path):
    fa, fqs, se = _make(tmp_path)
    for args in (["-K", "100000000", "-t", "3", fa] + fqs, ["-K", "100000000", "-t", "3", fa, se], ["-K", "100000000", "-t", "3", "-a", fa, se]):
        got = run_sam(binary, args)
        assert md5(got) == ref_sam_md5(args)
        assert b"pa:f:" in got or b"XA:Z:" in got or len(args) == 7


def test_alt_contigs_emulated(built, tmp_path):
    _check(CUSIMBIN, tmp_path)


@pytest.mark.gpu
def test_alt_contigs_gpu(tmp_path):
    _check(bwa_b200.CLI_PATH, tmp_path)
