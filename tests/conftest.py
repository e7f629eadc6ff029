import gzip
import hashlib
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
TESTBIN = os.path.join(ROOT, "tests", "_build", "bwa-b200-oracle")
CUSIMBIN = os.path.join(ROOT, "tests", "_build", "bwa-b200-cusim")
DATA = os.path.join(ROOT, "tests", "_build", "data")
GOLDEN = os.path.join(ROOT, "tests", "golden")
# Results of the unmodified reference (lh3/bwa 0.7.19) are stored under tests/golden, so the suite needs no reference build.
# With BWA_B200_RECORD_GOLDEN=<file.json> the tests run the reference binaries of oracle/_ref instead and write what they
# produced to that file (merged into what it holds), to be copied into tests/golden/ref_runs.json deliberately.
RECORD = os.environ.get("BWA_B200_RECORD_GOLDEN")
_recorded = {}


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _sh(cmd, **kw):
    return subprocess.run(cmd, check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE, **kw)


@pytest.fixture(scope="session", autouse=True)
def built():
    """Build the checkers once per session."""
    if not os.path.exists(ORACLE_SO):
        _sh(["make", "-C", os.path.join(ROOT, "oracle"), "-j8", "oracle"])
    if not (os.path.exists(TESTBIN) and os.path.exists(CUSIMBIN)):
        _sh(["make", "-C", ROOT, "-j8", "testbin", "cusim"])
    return True


def strip_pg(b):
    return b"\n".join(l for l in b.split(b"\n") if not l.startswith(b"@PG"))


def _input_key(a):
    """An argument as it enters a golden key: a file by its name and the digest of its content (paths differ from run to run)."""
    if not os.path.isfile(a):
        return a
    b = open(a, "rb").read()
    if a.endswith(".gz"):
        b = gzip.decompress(b)            # the gzip header holds a time stamp
    if os.path.isfile(a + ".alt"):
        b += open(a + ".alt", "rb").read()
    return "%s:%s" % (os.path.basename(a), md5(b)[:16])


def _golden_runs():
    if not hasattr(_golden_runs, "runs"):
        _golden_runs.runs = json.load(open(os.path.join(GOLDEN, "ref_runs.json")))
    return _golden_runs.runs


def ref_run(prog, args, view="sam", keep=None, outputs=()):
    """What the unmodified reference program oracle/_ref/<prog> does with args: {"rc": exit status, "md5": digest of its
    stdout, "lines": newlines in it}.  view "sam": @PG lines removed; "records": header lines removed and trailing newlines
    stripped; "raw": as printed.  keep: a file name under tests/golden that holds the whole output (returned as "out").
    outputs: files the program writes; their digests are returned as "files" ({base name: md5})."""
    key = " ".join([prog, view] + [_input_key(a) for a in args])
    if RECORD:
        r = subprocess.run([os.path.join(ROOT, "oracle", "_ref", prog)] + args, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, timeout=900)
        out = r.stdout
        if view == "sam":
            out = strip_pg(out)
        elif view == "records":
            out = b"\n".join(l for l in out.split(b"\n") if not l.startswith(b"@")).rstrip(b"\n")
        _recorded[key] = {"rc": r.returncode, "md5": md5(out), "lines": out.count(b"\n")}
        if outputs:
            _recorded[key]["files"] = {os.path.basename(f): md5(open(f, "rb").read()) for f in outputs}
        if keep:
            with gzip.GzipFile(os.path.join(GOLDEN, keep), "wb", mtime=0) as f:
                f.write(out)
    runs = _recorded if RECORD else _golden_runs()
    assert key in runs, "no stored result of the reference for %r (BWA_B200_RECORD_GOLDEN records one)" % key
    res = dict(runs[key])
    if keep:
        res["out"] = gzip.open(os.path.join(GOLDEN, keep)).read()
        assert md5(res["out"]) == res["md5"], "tests/golden/%s does not belong to %r" % (keep, key)
    return res


def ref_sam_md5(args, view="sam"):
    """md5 of the SAM of the unmodified reference (bwa mem -v 1 args), @PG removed."""
    r = ref_run("bwa", ["mem", "-v", "1"] + args, view)
    assert r["rc"] == 0
    return r["md5"]


def pytest_sessionfinish(session):
    if RECORD and _recorded:
        old = json.load(open(RECORD)) if os.path.exists(RECORD) else {}
        old.update(_recorded)
        with open(RECORD, "w") as f:
            json.dump(old, f, indent=0, sort_keys=True)


def run_sam(binary, args):
    r = subprocess.run([binary, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-2000:]
    return strip_pg(r.stdout)


def index(fa):
    """The five index files of `bwa index fa`, made by this repository's builder on the CPU; when recording, by the reference
    itself, so that what is recorded does not depend on the builder."""
    if RECORD:
        _sh([os.path.join(ROOT, "oracle", "_ref", "bwa"), "index", fa])
        return
    import bwa_b200.index_build as ib
    ib.build(fa, device="cpu", verbose=False)


class DataSets:
    """Seeded synthetic datasets (tools/gen_data.py), generated and indexed on first use (bwa_b200/index_build.py on the CPU:
    the files of `bwa index`, byte for byte, see test_index_build.py)."""

    def __init__(self):
        os.makedirs(DATA, exist_ok=True)
        self._done = set()

    def ref(self, name):
        import gen_data
        fa = os.path.join(DATA, name + ".fa")
        if name not in self._done:
            if RECORD or not os.path.exists(fa + ".bwt"):
                if name == "c1":
                    contigs = gen_data.random_contigs(1, 1000000, 7)
                elif name == "two":
                    contigs = gen_data.random_contigs(2, 150000, 9)
                elif name == "stress":
                    contigs = gen_data.stress_contigs(1500000, 5)
                else:
                    raise KeyError(name)
                gen_data.write_fasta(fa, contigs)
                index(fa)
            self._done.add(name)
        return fa

    def reads(self, ref, tag, n, length=150, seed=11, paired=False, err=(0.008, 0.001, 0.001), chimeric=0.0):
        import gen_data
        fa = self.ref(ref)
        base = os.path.join(DATA, "%s_%s" % (ref, tag))
        outs = [base + "_1.fq", base + "_2.fq"] if paired else [base + ".fq"]
        if not all(os.path.exists(o) for o in outs):
            contigs = gen_data.read_fasta(fa)
            r1, r2 = gen_data.gen_reads(contigs, n, length, seed, err=err, paired=paired, chimeric=chimeric)
            gen_data.write_fastq(outs[0], r1)
            if paired:
                gen_data.write_fastq(outs[1], r2)
        return fa, outs


@pytest.fixture(scope="session")
def data(built):
    return DataSets()


def md5(b):
    return hashlib.md5(b).hexdigest()
