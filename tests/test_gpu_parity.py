"""Parity of the CUDA path on a real B200, through the C ABI: SAM from libbwa_b200 / bwa-b200 must equal that of the
unmodified reference binary (oracle/_ref/bwa mem, its md5 stored in tests/golden/ref_runs.json) byte for byte; the seeding stage is additionally compared
buffer by buffer with the CPU oracle through the same device-batch ABI."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import bwa_b200
from conftest import ORACLE_SO, md5, ref_run, ref_sam_md5, run_sam, strip_pg

pytestmark = pytest.mark.gpu

CASES = [
    ("c1_se_10k", "c1", dict(tag="g10k", n=10000, seed=11), []),
    ("c1_pe_5k", "c1", dict(tag="gpe", n=5000, seed=12, paired=True), []),
    ("stress_se", "stress", dict(tag="gse", n=4000, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("stress_pe", "stress", dict(tag="gpe", n=3000, seed=4, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
    ("two_1k", "two", dict(tag="g1k", n=200, length=1000, seed=10), []),
    ("two_pacbio", "two", dict(tag="gpb", n=12, length=8000, seed=9, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"]),
    ("c1_len36", "c1", dict(tag="g36", n=2000, length=36, seed=21), []),
    ("c1_len75", "c1", dict(tag="g75", n=2000, length=75, seed=22), []),
    ("c1_len300", "c1", dict(tag="g300", n=1000, length=300, seed=23), []),
    ("c1_opts", "c1", dict(tag="gopt", n=1500, seed=24), ["-a", "-Y", "-k", "17", "-A", "2", "-T", "50"]),
]


@pytest.mark.parametrize("name,ref,kw,extra", CASES, ids=[c[0] for c in CASES])
def test_cli_sam_identical_to_reference(data, name, ref, kw, extra):
    fa, fqs = data.reads(ref, **kw)
    args = extra + ["-K", "100000000", "-t", "8", fa] + fqs
    assert md5(run_sam(bwa_b200.CLI_PATH, args)) == ref_sam_md5(args)


@pytest.mark.parametrize("ktab", [None, "0", "14"])
def test_edge_reads(data, tmp_path, monkeypatch, ktab):
    """Empty-ish and ragged input: reads shorter than the seed length, all-N reads, N runs, mixed lengths, lower case;
    with the short-string table at its default depth, without it, and at the depth used for 3 Gbp references."""
    if ktab is not None:
        monkeypatch.setenv("BWA_B200_KTAB", ktab)
    fa = data.ref("c1")
    import gen_data
    contigs = gen_data.read_fasta(fa)
    c = contigs[0]
    recs = []
    rng = np.random.default_rng(5)
    for i, ln in enumerate([1, 5, 18, 19, 20, 33, 150, 151, 400, 2, 149]):
        p = int(rng.integers(0, len(c) - ln))
        recs.append((b"e%d" % i, c[p:p + ln].copy()))
    recs.append((b"allN", np.frombuffer(b"N" * 100, dtype=np.uint8).copy()))
    s = c[5000:5150].copy(); s[40:60] = ord("N"); recs.append((b"nrun", s))
    recs.append((b"lower", np.frombuffer(c[9000:9150].tobytes().lower(), dtype=np.uint8).copy()))
    recs.append((b"polyA", np.frombuffer(b"A" * 150, dtype=np.uint8).copy()))
    for i, pos in enumerate([0, 1, 7, 11, 12, 13, 19, 20, 75, 149]):   # a single N at and around the table / seed window boundaries
        s = c[7000 + 200 * i:7150 + 200 * i].copy(); s[pos] = ord("N"); recs.append((b"n%d" % pos, s))
    fq = str(tmp_path / "edge.fq")
    gen_data.write_fastq(fq, recs)
    args = ["-K", "100000000", fa, fq]
    assert md5(run_sam(bwa_b200.CLI_PATH, args)) == ref_sam_md5(args)


def test_batching_and_threads_do_not_change_se_output(data):
    fa, fqs = data.reads("c1", tag="g10k", n=10000, seed=11)
    a = run_sam(bwa_b200.CLI_PATH, ["-K", "100000000", "-t", "8", fa] + fqs)
    b = run_sam(bwa_b200.CLI_PATH, ["-K", "300000", "-t", "3", fa] + fqs)
    assert a == b


def test_library_call_and_dense_sa(data):
    """mem_process_seqs through ctypes (host buffers in, SAM out); a denser on-device SA sample must not change a byte."""
    fa, fqs = data.reads("stress", tag="gse", n=4000, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05)
    want = ref_sam_md5(["-K", "100000000", fa] + fqs, view="records")
    L = bwa_b200.lib()
    idx = bwa_b200.Index(fa)
    os.environ["BWA_B200_SA_INTV"] = "32"      # first pass on the sample of the index files, then denser ones
    try:
        idx.attach()
    finally:
        del os.environ["BWA_B200_SA_INTV"]
    opt = L.mem_opt_init()
    opt.contents.n_threads = 8
    for dense in (0, 8, 2):
        if dense:
            idx.densify_sa(dense)
        batch = bwa_b200.ReadBatch(fqs[0])
        idx.stats(reset=True)
        bwa_b200.mem_process_seqs(opt, idx, batch)
        got = batch.sam().rstrip(b"\n")
        st = idx.stats()
        assert md5(got) == want, "dense=%d" % dense
        assert st["occ_touches"] > 0 and st["ext_cells"] > 0 and st["n_launch"] >= 4
    idx.close()


from stage_abi import SeedPar, load_reads_as_codes, seed_stage


@pytest.mark.parametrize("compact", ["1", "0"])
def test_seed_stage_buffers_equal_oracle(data, monkeypatch, compact):
    """bwag_seed of the CUDA library vs the CPU oracle: every interval (x0,x1,x2,info) and every suffix-array position; with K1's
    compact candidate lists (k_smem_c) and without (k_smem)."""
    monkeypatch.setenv("BWA_B200_K1_COMPACT", compact)
    fa, fqs = data.reads("stress", tag="gse", n=4000, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05)
    L = bwa_b200.lib()
    O = C.CDLL(ORACLE_SO, mode=C.RTLD_LOCAL)
    idx = L.bwa_idx_load(fa.encode(), 7).contents
    l_pac = C.cast(idx.bns, C.POINTER(C.c_int64))[0]
    codes, off = load_reads_as_codes(fqs[0], 1500)
    par = SeedPar(19, 28, 10, 500, 20)
    t = []
    want = seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par, touches=t)
    assert sum(len(r) for r in want) > 5000
    assert seed_stage(L, idx.bwt, l_pac, idx.pac, codes, off, par, touches=t) == want
    for depth in (4, 9, 14):   # with the short-string table (14 = the depth used at 3 Gbp, 5.7 GB): same buffers
        assert seed_stage(L, idx.bwt, l_pac, idx.pac, codes, off, par, ktab=depth, touches=t) == want
    assert len(set(t)) == 1 and t[0] > 0, t   # the roofline's numerator (reference-equivalent Occ-block touches) is the oracle's, table or not
    par11 = SeedPar(11, 17, 10, 500, 20)   # seed length below the table depth: the third pass may only jump min_seed_len bases
    assert seed_stage(L, idx.bwt, l_pac, idx.pac, codes, off, par11, ktab=13) == seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par11)
    t8 = []
    par8 = SeedPar(8, 12, 10, 500, 20)     # candidates of 8..10 bases can be results: they keep their intervals
    assert seed_stage(L, idx.bwt, l_pac, idx.pac, codes, off, par8, ktab=10, touches=t8) == seed_stage(O, idx.bwt, l_pac, idx.pac, codes, off, par8, touches=t8)
    assert t8[0] == t8[1], t8


def test_index_builder_identical_to_bwa_index(data, tmp_path):
    """bwa_b200/index_build.py on the GPU writes the same five files as the reference's `bwa index`."""
    import shutil
    import bwa_b200.index_build as ib
    exts = ("pac", "ann", "amb", "bwt", "sa")
    for name in ("stress", "c1"):
        fa = data.ref(name)
        want = ref_run("bwa", ["index", fa], "raw", outputs=[fa + "." + e for e in exts])["files"]
        mine = str(tmp_path / (name + ".fa"))
        shutil.copy(fa, mine)
        ib.build(mine, verbose=False)
        for ext in exts:
            assert md5(open(mine + "." + ext, "rb").read()) == want[name + ".fa." + ext], (name, ext)


def test_host_chaining_path_still_identical(data, monkeypatch):
    """BWA_B200_DEVICE_CHAIN=0 forces the host chaining path (the one long reads take); default is chaining on the device."""
    monkeypatch.setenv("BWA_B200_DEVICE_CHAIN", "0")
    for ref, kw in (("stress", dict(tag="gse", n=4000, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05)),
                    ("stress", dict(tag="gpe", n=3000, seed=4, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05))):
        fa, fqs = data.reads(ref, **kw)
        args = ["-K", "100000000", "-t", "8", fa] + fqs
        assert md5(run_sam(bwa_b200.CLI_PATH, args)) == ref_sam_md5(args)


@pytest.mark.parametrize("env", [{"BWA_B200_K4_SM": "0", "BWA_B200_K5_SM": "0"}, {"BWA_B200_K4_FAST": "0", "BWA_B200_K5_FAST": "0"},
                                 {"BWA_B200_K4_SM": "0", "BWA_B200_K5_SM": "0", "BWA_B200_K4_FAST": "0", "BWA_B200_K5_FAST": "0"}],
                         ids=["global_scratch", "first_sweep", "global_scratch_first_sweep"])
def test_kernel_variants(data, monkeypatch, env):
    """K4/K5 exist in four variants each (scratch in shared or global memory x lean or first row sweep); the other
    tests run shared+lean for short reads and global+lean for long ones, this one the remaining combinations."""
    fa, fqs = data.reads("stress", tag="gpe", n=3000, seed=4, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "100000000", "-t", "4", fa] + fqs
    want = ref_sam_md5(args)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    assert md5(run_sam(bwa_b200.CLI_PATH, args)) == want


def test_startup_selfcheck_passed(data):
    """Attaching an index runs the start-up self-check (192 reads drawn from the reference: default kernels vs the baseline
    kernels).  It must have passed; had it not, the library would be running on the baseline kernels and every other test
    here would still be green, so this is the test that says so."""
    idx = bwa_b200.Index(data.ref("stress"))
    idx.attach()
    L = bwa_b200.lib()
    L.bb_selfcheck_status.restype = C.c_int
    assert L.bb_selfcheck_status() == 1
    idx.close()


def test_pool_overflow_is_repeated_not_corrupting(data, monkeypatch):
    """Seeding pools that start too small (test hook): the stage is repeated with the sizes the device counters report; no slice of a
    read that did not fit may be touched (once an out-of-bounds sort in the epilogue kernel: crash on the 3 Gbp pacbio workload)."""
    monkeypatch.setenv("BWA_B200_TEST_SMALL_POOLS", "1")
    for ref, kw, extra in (("stress", dict(tag="gse", n=4000, seed=3, err=(0.016, 0.002, 0.002), chimeric=0.05), []),
                           ("two", dict(tag="gpb", n=12, length=8000, seed=9, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"])):
        fa, fqs = data.reads(ref, **kw)
        args = extra + ["-K", "100000000", "-t", "8", fa] + fqs
        assert md5(run_sam(bwa_b200.CLI_PATH, args)) == ref_sam_md5(args)
    monkeypatch.delenv("BWA_B200_TEST_SMALL_POOLS")
    monkeypatch.setenv("BWA_B200_TEST_SMALL_K1", "1")   # K1's per-lane scratch starts too small as well: repeated with the worst-case sizes
    assert md5(run_sam(bwa_b200.CLI_PATH, args)) == ref_sam_md5(args)
