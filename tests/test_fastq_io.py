"""Input formats of bseq_read (bb_fastq.c) against the reference's kseq-based reader: FASTA, multi-line records, gzip,
CR/LF, comments (-C), /1 /2 name suffixes, and paired files of unequal length (warning + truncation, same SAM)."""
import gzip
import os
import subprocess

import pytest

from conftest import TESTBIN, md5, ref_run, strip_pg


def _sam(binary, args):
    r = subprocess.run([binary, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    return r.returncode, strip_pg(r.stdout)


def _records(fq):
    lines = open(fq).read().split("\n")
    return [lines[i:i + 4] for i in range(0, len(lines) - 3, 4)]


@pytest.fixture(scope="module")
def inputs(data, tmp_path_factory):
    d = tmp_path_factory.mktemp("fqio")
    fa, fqs = data.reads("two", tag="io", n=120, seed=5, paired=True)
    r1, r2 = _records(fqs[0]), _records(fqs[1])
    out = {"fa": fa, "r1": fqs[0], "r2": fqs[1]}
    with open(d / "a.fa", "w") as f:                       # FASTA, sequence folded to 60 columns
        for rec in r1:
            f.write(">" + rec[0][1:] + "\n" + "\n".join(rec[1][i:i + 60] for i in range(0, len(rec[1]), 60)) + "\n")
    with gzip.open(d / "a.fq.gz", "wt") as f:
        f.write(open(fqs[0]).read())
    with open(d / "crlf.fq", "w", newline="") as f:
        f.write(open(fqs[0]).read().replace("\n", "\r\n"))
    with open(d / "cmt_1.fq", "w") as f1, open(d / "cmt_2.fq", "w") as f2:   # comments and /1 /2 suffixes
        for a, b in zip(r1, r2):
            f1.write("%s/1 BC:Z:ACGT\n%s\n+\n%s\n" % (a[0], a[1], a[3]))
            f2.write("%s/2 BC:Z:ACGT\n%s\n+\n%s\n" % (b[0], b[1], b[3]))
    with open(d / "short_2.fq", "w") as f:                 # second file has fewer records
        f.write("\n".join("\n".join(r) for r in r2[:70]) + "\n")
    with open(d / "short_1.fq", "w") as f:                 # first file has fewer records
        f.write("\n".join("\n".join(r) for r in r1[:50]) + "\n")
    with open(d / "multi.fq", "w") as f:                   # multi-line FASTQ
        for rec in r1:
            f.write("%s\n%s\n%s\n+\n%s\n%s\n" % (rec[0], rec[1][:70], rec[1][70:], rec[3][:70], rec[3][70:]))
    out["d"] = str(d)
    return out


CASES = {
    "fasta": lambda i: [i["fa"], i["d"] + "/a.fa"],
    "gzip": lambda i: [i["fa"], i["d"] + "/a.fq.gz"],
    "crlf": lambda i: [i["fa"], i["d"] + "/crlf.fq"],
    "multiline": lambda i: [i["fa"], i["d"] + "/multi.fq"],
    "comments": lambda i: ["-C", i["fa"], i["d"] + "/cmt_1.fq", i["d"] + "/cmt_2.fq"],
    "second_shorter": lambda i: ["-K", "9000", i["fa"], i["r1"], i["d"] + "/short_2.fq"],
    "first_shorter": lambda i: ["-K", "9000", i["fa"], i["d"] + "/short_1.fq", i["r2"]],
    "interleaved": lambda i: ["-p", i["fa"], i["d"] + "/cmt_1.fq"],
}


@pytest.mark.parametrize("name", sorted(CASES))
def test_reader_matches_reference(inputs, name):
    args = ["-t", "2"] + CASES[name](inputs)
    rc, sam = _sam(TESTBIN, args)
    want = ref_run("bwa", ["mem", "-v", "1"] + args)
    assert (rc, md5(sam)) == (want["rc"], want["md5"])
