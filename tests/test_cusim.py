"""The CUDA kernels themselves, compiled for the CPU SIMT emulator (tests/cusim), against the reference:
same .cu sources, every lane a fiber, warp collectives as rendezvous.  Checks kernel logic without a GPU."""
import pytest

from conftest import CUSIMBIN, md5, ref_sam_md5, run_sam

CASES = [
    ("c1_se", "c1", dict(tag="cs", n=160, seed=31), []),
    ("stress_se", "stress", dict(tag="cs", n=120, seed=33, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("stress_pe", "stress", dict(tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("two_1k", "two", dict(tag="cs1k", n=6, length=1000, seed=35), []),
    # long reads: read bases and DP scratch in global memory (no shared slots), host chaining, seed filter (ksw_align2)
    ("two_pacbio_4k", "two", dict(tag="cspb", n=3, length=4000, seed=36, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"]),
]


@pytest.mark.parametrize("name,ref,kw,extra", CASES, ids=[c[0] for c in CASES])
def test_emulated_kernels_sam_vs_reference(data, name, ref, kw, extra):
    fa, fqs = data.reads(ref, **kw)
    args = extra + ["-K", "100000000", "-t", "2", fa] + fqs
    assert md5(run_sam(CUSIMBIN, args)) == ref_sam_md5(args)


@pytest.mark.parametrize("compact", ["1", "0"])
def test_emulated_seed_stage_buffers_equal_oracle(data, monkeypatch, compact):
    """bwag_seed of the emulated CUDA kernels vs the CPU oracle, buffer by buffer (intervals and SA positions); compact: K1 with its
    short candidates as mask bits (k_smem_c, the default) or with every candidate as a list entry (k_smem)."""
    monkeypatch.setenv("BWA_B200_K1_COMPACT", compact)
    import ctypes as C
    import os
    import bwa_b200
    from conftest import ORACLE_SO, ROOT
    from stage_abi import SeedPar, load_reads_as_codes, seed_stage
    fa, fqs = data.reads("stress", tag="cs", n=120, seed=33, err=(0.016, 0.002, 0.002), chimeric=0.05)
    L = bwa_b200.lib()
    idx = L.bwa_idx_load(fa.encode(), 7).contents
    l_pac = C.cast(idx.bns, C.POINTER(C.c_int64))[0]
    codes, off = load_reads_as_codes(fqs[0], 120)
    par = SeedPar(19, 28, 10, 500, 20)
    S = C.CDLL(os.path.join(ROOT, "tests/_build/libbwa_b200_cusim.so"), mode=C.RTLD_LOCAL)
    O = C.CDLL(ORACLE_SO, mode=C.RTLD_LOCAL)
    t = []
    want = seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par, touches=t)
    assert sum(len(r) for r in want) > 500
    assert seed_stage(S, idx.bwt, l_pac, idx.pac, codes, off, par, touches=t) == want
    for depth in (3, 6):   # with the short-string table: same intervals (x[0], x[1], x[2], info) and positions
        assert seed_stage(S, idx.bwt, l_pac, idx.pac, codes, off, par, ktab=depth, touches=t) == want
    assert len(set(t)) == 1 and t[0] > 0, t   # the Occ-block count (as the reference would touch them) is the oracle's, table or not
    par11 = SeedPar(11, 17, 10, 500, 20)   # a seed length below the table depth + 1: the third pass jumps min_seed_len bases only
    assert seed_stage(S, idx.bwt, l_pac, idx.pac, codes, off, par11, ktab=6) == seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par11)
    t8 = []
    par8 = SeedPar(8, 12, 10, 500, 20)     # a table deeper than the seed length: candidates of 8..10 bases keep their intervals (they can be results)
    assert seed_stage(S, idx.bwt, l_pac, idx.pac, codes, off, par8, ktab=10, touches=t8) == seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par8, touches=t8)
    assert t8[0] == t8[1], t8


def test_batches_in_flight_keep_order_and_content(data, monkeypatch):
    """Several batches aligned at a time (BWA_B200_INFLIGHT): the writer restores input order; PE statistics stay per batch."""
    fa, fqs = data.reads("stress", tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "3000", "-t", "2", fa] + fqs        # ~10 pairs per batch
    want = ref_sam_md5(args)
    for inflight in ("1", "3"):
        monkeypatch.setenv("BWA_B200_INFLIGHT", inflight)
        assert md5(run_sam(CUSIMBIN, args)) == want


def test_default_thread_count_keeps_reference_batches(data):
    """No -t: the batches are the reference's (chunk_size x 1 thread), only the host worker count differs; same SAM."""
    fa, fqs = data.reads("stress", tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    assert md5(run_sam(CUSIMBIN, [fa] + fqs)) == ref_sam_md5([fa] + fqs)


@pytest.mark.parametrize("env", [{"BWA_B200_K4_SM": "0", "BWA_B200_K5_SM": "0"}, {"BWA_B200_K4_FAST": "0", "BWA_B200_K5_FAST": "0"},
                                 {"BWA_B200_K4_SM": "0", "BWA_B200_K5_SM": "0", "BWA_B200_K4_FAST": "0", "BWA_B200_K5_FAST": "0"}],
                         ids=["global_scratch", "first_sweep", "global_scratch_first_sweep"])
def test_emulated_kernel_variants(data, monkeypatch, env):
    """K4/K5 exist in four variants each (scratch in shared or global memory x lean or first row sweep); the default
    run covers shared+lean, this one the others."""
    fa, fqs = data.reads("stress", tag="cspe", n=60, seed=34, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "100000000", "-t", "2", fa] + fqs
    want = ref_sam_md5(args)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    assert md5(run_sam(CUSIMBIN, args)) == want


@pytest.mark.parametrize("ktab", ["0", "3", "5", "8"])
def test_emulated_edge_reads(data, tmp_path, monkeypatch, ktab):
    """Ragged input through the emulated kernels at several short-string table depths: reads shorter than the table depth
    and the seed length, all-N reads, N runs and single Ns (the third pass must fall back to single steps around them),
    mixed lengths, lower case, homopolymers."""
    import numpy as np
    import gen_data
    fa = data.ref("c1")
    c = gen_data.read_fasta(fa)[0]
    recs = []
    rng = np.random.default_rng(5)
    for i, ln in enumerate([1, 2, 3, 5, 6, 8, 9, 18, 19, 20, 33, 150, 151, 400, 149]):
        p = int(rng.integers(0, len(c) - ln))
        recs.append((b"e%d" % i, c[p:p + ln].copy()))
    recs.append((b"allN", np.frombuffer(b"N" * 100, dtype=np.uint8).copy()))
    s = c[5000:5150].copy(); s[40:60] = ord("N"); recs.append((b"nrun", s))
    for i, pos in enumerate([0, 1, 4, 7, 18, 19, 20, 21, 75, 148, 149]):   # a single N at and around every window boundary
        s = c[7000 + 200 * i:7150 + 200 * i].copy(); s[pos] = ord("N"); recs.append((b"n%d" % pos, s))
    s = c[12000:12150].copy(); s[::10] = ord("N"); recs.append((b"nevery10", s))
    recs.append((b"lower", np.frombuffer(c[9000:9150].tobytes().lower(), dtype=np.uint8).copy()))
    recs.append((b"polyA", np.frombuffer(b"A" * 150, dtype=np.uint8).copy()))
    recs.append((b"polyAC", np.frombuffer(b"AC" * 75, dtype=np.uint8).copy()))
    fq = str(tmp_path / "edge.fq")
    gen_data.write_fastq(fq, recs)
    args = ["-K", "100000000", fa, fq]
    want = ref_sam_md5(args)
    monkeypatch.setenv("BWA_B200_KTAB", ktab)
    assert md5(run_sam(CUSIMBIN, args)) == want


def test_startup_selfcheck_passes_and_falls_back(data, monkeypatch):
    """BWA_B200_SELFCHECK=n: when an index goes to the device, n reads drawn from the reference are aligned with the default
    kernels and with the baseline (first row sweeps, no short-string table) and compared.  Agreement is silent; a difference
    (here injected by the test hook) is fatal; with BWA_B200_SELFCHECK_FALLBACK=1 it is reported and the run continues on
    the baseline, with the same SAM."""
    import subprocess
    fa, fqs = data.reads("stress", tag="cs", n=120, seed=33, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "100000000", "-t", "2", fa] + fqs
    want = ref_sam_md5(args)
    monkeypatch.setenv("BWA_B200_SELFCHECK", "24")
    p = subprocess.run([CUSIMBIN, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0 and b"self-check" not in p.stderr
    from conftest import strip_pg
    assert md5(strip_pg(p.stdout)) == want
    monkeypatch.setenv("BWA_B200_SELFCHECK_INJECT", "1")
    p = subprocess.run([CUSIMBIN, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode != 0 and b"records differ" in p.stderr          # a difference is fatal by default
    monkeypatch.setenv("BWA_B200_SELFCHECK_FALLBACK", "1")
    p = subprocess.run([CUSIMBIN, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert p.returncode == 0 and b"staying on the baseline kernels" in p.stderr
    assert md5(strip_pg(p.stdout)) == want


def test_pool_overflow_is_repeated_not_corrupting(data, monkeypatch):
    """The seeding stage sizes its interval / seed pools from typical reads and repeats itself with the sizes the device counters report
    when they overflow (long noisy reads against a large index do that).  The epilogue kernel once sorted slices that did not exist in
    that case (out-of-bounds writes: a crash and a SAM mismatch on the 3 Gbp pacbio workload).  Here the pools start far too small."""
    fa, fqs = data.reads("stress", tag="cs", n=120, seed=33, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "100000000", "-t", "2", fa] + fqs
    want = ref_sam_md5(args)
    monkeypatch.setenv("BWA_B200_TEST_SMALL_POOLS", "1")
    assert md5(run_sam(CUSIMBIN, args)) == want
    # K1's per-lane scratch (candidate-list tails, results of a read): long reads start below the worst case and the stage repeats with more
    monkeypatch.delenv("BWA_B200_TEST_SMALL_POOLS")
    monkeypatch.setenv("BWA_B200_TEST_SMALL_K1", "1")
    monkeypatch.setenv("BWA_B200_KTAB", "6")
    assert md5(run_sam(CUSIMBIN, args)) == want
