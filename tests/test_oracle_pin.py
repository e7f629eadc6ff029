"""Pins the CPU oracle (oracle/oracle_*.c) to the UNMODIFIED reference:
  * committed known-answer vectors produced by oracle/_ref/katdump (tests/golden/*.kat.gz, make_golden.sh);
  * katdump runs of the reference's FM-index functions on a generated index (stored: tests/golden/katdump_*.txt.gz);
  * whole-program SAM: host glue + oracle stages (tests/_build/bwa-b200-oracle) vs the md5 of `oracle/_ref/bwa mem`'s.
No GPU needed."""
import ctypes as C
import gzip
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ORACLE_SO, ROOT, TESTBIN, md5, ref_run, ref_sam_md5, run_sam

CODE = {c: i for i, c in enumerate("ACGTN")}


def codes(s):
    return (C.c_uint8 * len(s))(*[CODE[c] for c in s])


def scmat(a, b):
    m = (C.c_int8 * 25)()
    for i in range(5):
        for j in range(5):
            m[i * 5 + j] = -1 if (i == 4 or j == 4) else (a if i == j else -b)
    return m


@pytest.fixture(scope="module")
def orc(built):
    return C.CDLL(ORACLE_SO, mode=C.RTLD_LOCAL)


def test_extend_golden(orc):
    """oracle ksw_extend2 restatement == reference on 1500 seeded cases (scores and all five out-params)."""
    out = [C.c_int() for _ in range(5)]
    n = 0
    for line in gzip.open(os.path.join(ROOT, "tests/golden/extend.kat.gz"), "rt"):
        f = line.split()
        a, b, od, ed, oi, ei, w, eb, zd, h0, ql, tl = map(int, f[1:13])
        q, t = f[13], f[14]
        want = list(map(int, f[16:22]))
        sc = orc.orc_extend_sw(ql, codes(q), tl, codes(t), scmat(a, b), od, ed, oi, ei, w, eb, zd, h0, *[C.byref(o) for o in out], None)
        assert [sc] + [o.value for o in out] == want, line[:80]
        n += 1
    assert n == 1500


class U32V(C.Structure):
    _fields_ = [("n", C.c_size_t), ("m", C.c_size_t), ("a", C.POINTER(C.c_uint32))]


def test_global_golden(orc):
    """oracle ksw_global2 restatement == reference on 1000 seeded cases (score and CIGAR)."""
    n = 0
    for line in gzip.open(os.path.join(ROOT, "tests/golden/global.kat.gz"), "rt"):
        f = line.rstrip("\n").split(" ")
        a, b, od, ed, oi, ei, w, ql, tl = map(int, f[1:10])
        q, t = f[10], f[11]
        want_sc, want_cig = int(f[13]), f[14] if len(f) > 14 else ""
        cv = U32V()
        sc = orc.orc_global(ql, codes(q), tl, codes(t), scmat(a, b), od, ed, oi, ei, w, C.byref(cv), None)
        cig = "".join("%d%s" % (cv.a[i] >> 4, "MIDSH"[cv.a[i] & 15]) for i in range(cv.n))
        assert (sc, cig) == (want_sc, want_cig), line[:80]
        n += 1
    assert n == 1000


class SWR(C.Structure):
    _fields_ = [(k, C.c_int) for k in ("score", "te", "qe", "score2", "te2", "tb", "qb")]


def test_local_golden(built):
    """host local-SW (bb_local_sw, used by mate rescue / seed filter) == reference ksw_align2 on 400 seeded cases."""
    import bwa_b200
    L = bwa_b200.lib()
    L.bb_local_sw.restype = SWR
    n = 0
    for line in gzip.open(os.path.join(ROOT, "tests/golden/local.kat.gz"), "rt"):
        f = line.split()
        a, b, od, ed, oi, ei, xtra, ql, tl = map(int, f[1:10])
        q, t = f[10], f[11]
        want = tuple(map(int, f[13:20]))
        r = L.bb_local_sw(ql, codes(q), tl, codes(t), scmat(a, b), od, ed, oi, ei, xtra)
        assert (r.score, r.te, r.qe, r.score2, r.te2, r.tb, r.qb) == want, line[:60]
        n += 1
    assert n == 400


def test_local_golden_scalar_specification(built):
    """the same vectors through the lane-by-lane scalar version of the routine (the specification of the SSE2 one)"""
    import subprocess
    import sys
    code = "import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import test_oracle_pin as t; t.test_local_golden(None)" % (ROOT, os.path.join(ROOT, "tests"))
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, BWA_B200_SCALAR_SW="1"), stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-2000:]


class Intv(C.Structure):
    _fields_ = [("x0", C.c_uint64), ("x1", C.c_uint64), ("x2", C.c_uint64), ("info", C.c_uint64)]


class IntvV(C.Structure):
    _fields_ = [("n", C.c_size_t), ("m", C.c_size_t), ("a", C.POINTER(Intv))]


def test_fm_index_live(orc, data):
    """oracle bwt_smem1 / bwt_seed_strategy1 / bwt_sa == the reference's on a generated index (every x of 25 reads, 3000 rows)."""
    import bwa_b200
    fa, (fq,) = data.reads("stress", "se", 1200, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05)
    L = bwa_b200.lib()
    idx = L.bwa_idx_load(fa.encode(), 1)
    bwt = idx.contents.bwt
    txt = ref_run("katdump", ["smem", fa, fq, "25"], "raw", keep="katdump_smem.txt.gz")["out"].decode().split("\n")
    seq, mem, one, n_checked = None, IntvV(), Intv(), 0
    reads = {}
    name = None
    for l in open(fq):
        pass
    fql = open(fq).read().split("\n")
    for i in range(0, len(fql) - 3, 4):
        reads[fql[i][1:]] = fql[i + 1]
    orc.orc_sa.restype = C.c_uint64
    for l in txt:
        f = l.split()
        if not f:
            continue
        if f[0] == "R":
            seq = codes(reads[f[1]].replace("a", "A"))
            ln = int(f[2])
        elif f[0] == "S":
            x, mi, ret, n = map(int, f[1:5])
            r = orc.orc_smem1(C.c_void_p(bwt), ln, seq, x, mi, C.byref(mem), None)
            got = ["%d,%d,%d,%d" % (mem.a[k].x0, mem.a[k].x1, mem.a[k].x2, mem.a[k].info) for k in range(mem.n)]
            assert (r, got) == (ret, f[5:]), l[:100]
            n_checked += 1
        elif f[0] == "T":
            x, ret = int(f[1]), int(f[2])
            r = orc.orc_seed_strategy1(C.c_void_p(bwt), ln, seq, x, 19, 20, C.byref(one), None)
            assert (r, "%d,%d,%d,%d" % (one.x0, one.x1, one.x2, one.info)) == (ret, f[3]), l[:100]
    assert n_checked > 5000
    idx2 = L.bwa_idx_load(fa.encode(), 1)
    for l in ref_run("katdump", ["sa", fa, "3000", "99"], "raw", keep="katdump_sa.txt.gz")["out"].decode().split("\n"):
        f = l.split()
        if f:
            assert orc.orc_sa(C.c_void_p(idx2.contents.bwt), C.c_uint64(int(f[1])), None) == int(f[2])


CASES = [
    ("c1_se", "c1", dict(tag="se", n=2000), []),
    ("c1_pe", "c1", dict(tag="pe", n=800, paired=True, seed=12), []),
    ("stress_se", "stress", dict(tag="se", n=1200, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("stress_pe", "stress", dict(tag="pe", n=700, seed=4, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("two_1k", "two", dict(tag="l1k", n=40, length=1000, seed=10), []),
    ("two_pacbio", "two", dict(tag="pb", n=4, length=6000, seed=9, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"]),
    ("c1_len36", "c1", dict(tag="l36", n=500, length=36, seed=21), []),
]


@pytest.mark.parametrize("name,ref,kw,extra", CASES, ids=[c[0] for c in CASES])
def test_host_glue_sam_vs_reference(data, name, ref, kw, extra):
    """Host glue (chaining, dedup, pairing, SAM) over the oracle stages == `bwa mem`, byte for byte, and the
    reference's output itself matches the committed md5 (pins the generators and the oracle build)."""
    fa, fqs = data.reads(ref, **kw)
    args = extra + ["-K", "100000000", "-t", "4", fa] + fqs
    want = ref_sam_md5(args)
    got = run_sam(TESTBIN, args)
    assert md5(got) == want
    pins = json.load(open(os.path.join(ROOT, "tests/golden/sam_md5.json")))
    assert pins[name] == want, "reference SAM changed: regenerate tests/golden/sam_md5.json deliberately"
