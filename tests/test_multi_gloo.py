"""The N>1 path on CPU: two processes (torch.distributed, gloo), the index blob broadcast from rank 0, batches dealt
round-robin, parts merged by rank 0.  The kernels run in the CPU SIMT emulator build of the library, so the whole
multi-GPU control flow of bwa_b200/multi.py is exercised without a GPU; the merged SAM must equal the reference's."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT, md5, ref_sam_md5

CUSIM_SO = os.path.join(ROOT, "tests/_build/libbwa_b200_cusim.so")


def _launch(world, args, out, port, striped=None, extra_env=None):
    env = dict(os.environ, BWA_B200_LIB=CUSIM_SO, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(port), "-m", "bwa_b200.multi"] + args[:-len(args) + args.index("--")] + ["-o", out] + args[args.index("--") + 1:]
    env.update(extra_env or {})
    r = subprocess.run(cmd, env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
    assert r.returncode == 0, r.stderr.decode()[-3000:]
    if striped is not None:
        assert b"striped ingest:" in r.stderr
        assert (b"batches over" in r.stderr) == striped, r.stderr.decode()[-2000:]
    return open(out, "rb").read()


@pytest.mark.parametrize("paired", [False, True], ids=["se", "pe"])
def test_two_ranks_equal_reference(data, tmp_path, paired):
    fa, fqs = data.reads("stress", tag="mg" + ("pe" if paired else "se"), n=90, seed=77, paired=paired, err=(0.016, 0.002, 0.002), chimeric=0.05)
    opts = ["-K", "6000", "-t", "2"]           # ~40 reads per batch: several batches per rank
    got = _launch(2, opts + ["--", fa] + fqs, str(tmp_path / "out.sam"), 29631 + int(paired), striped=True)
    assert md5(got) == ref_sam_md5(opts + [fa] + fqs)
    assert got.count(b"\n") > 90


def test_three_ranks_striped_and_fallbacks(data, tmp_path):
    """Striped ingest (each rank scans a third of the bytes and parses only its batches) at world 3, the interleaved -p
    input, and the two fallbacks (gzip input; BWA_B200_STRIPED=0): all equal the reference's single-process SAM."""
    import gzip
    fa, fqs = data.reads("stress", tag="mg3", n=75, seed=78, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    opts = ["-K", "5000", "-t", "2"]
    want = ref_sam_md5(opts + [fa] + fqs)
    assert md5(_launch(3, opts + ["--", fa] + fqs, str(tmp_path / "a.sam"), 29641, striped=True)) == want
    assert md5(_launch(2, opts + ["--", fa] + fqs, str(tmp_path / "b.sam"), 29642, striped=False, extra_env={"BWA_B200_STRIPED": "0"})) == want
    gz = []
    for f in fqs:
        g = str(tmp_path / (os.path.basename(f) + ".gz"))
        with gzip.open(g, "wb") as o:
            o.write(open(f, "rb").read())
        gz.append(g)
    assert md5(_launch(2, opts + ["--", fa] + gz, str(tmp_path / "c.sam"), 29643, striped=False)) == ref_sam_md5(opts + [fa] + gz)
    # one interleaved file, odd record count: the lone last record ends the last batch
    r1, r2 = (open(f).read().split("\n") for f in fqs)
    inter = str(tmp_path / "inter.fq")
    with open(inter, "w") as o:
        for k in range(0, len(r1) - 1, 4):
            o.write("\n".join(r1[k:k + 4]) + "\n" + "\n".join(r2[k:k + 4]) + "\n")
        o.write("@lone\nACGTACGTACGTACGTACGTAAACCCGGGTTT\n+\n" + "I" * 32 + "\n")
    assert md5(_launch(3, opts + ["-p", "--", fa, inter], str(tmp_path / "d.sam"), 29644, striped=True)) == ref_sam_md5(opts + ["-p", fa, inter])


def test_merge_parts_orders_batches(tmp_path):
    from bwa_b200.multi import merge_parts, shard_of
    parts = []
    text = {0: b"@HD\n", 1: b""}
    idx = {0: "-1 4\n", 1: "-1 0\n"}
    for b in range(5):
        r = shard_of(b, 2)
        rec = (b"batch%d\n" % b) * (b + 1)
        text[r] += rec
        idx[r] += "%d %d\n" % (b, len(rec))
    for r in (0, 1):
        p, q = tmp_path / ("p%d" % r), tmp_path / ("p%d.idx" % r)
        p.write_bytes(text[r]); q.write_text(idx[r])
        parts.append((str(p), str(q)))
    merge_parts(str(tmp_path / "m"), parts)
    assert (tmp_path / "m").read_bytes() == b"@HD\n" + b"".join((b"batch%d\n" % b) * (b + 1) for b in range(5))


def test_stripe_scan_finds_every_record_once(built, tmp_path):
    """bb_fq_scan_stripe at every cut position of a FASTQ whose quality lines start with '@' and '+': the stripes' records,
    concatenated, are the file's records; wrapped or gzip'd input is declared unfit."""
    import ctypes as C
    import random
    from bwa_b200.multi import Stripe
    L = C.CDLL(CUSIM_SO, mode=C.RTLD_LOCAL)
    L.bb_fq_scan_stripe.argtypes = [C.c_char_p, C.c_int64, C.c_int64, C.POINTER(Stripe)]
    L.bb_fq_stripe_free.argtypes = [C.POINTER(Stripe)]
    rng = random.Random(5)
    recs, text = [], b""
    for k in range(40):
        n = rng.choice([0, 1, 7, 30, 61])
        seq = "".join(rng.choice("ACGTN") for _ in range(n))
        qual = "".join(rng.choice("@+>I#") for _ in range(n))
        recs.append((len(text), n))
        text += ("@r%d extra\n%s\n+%s\n%s\n" % (k, seq, "r%d" % k if k % 3 == 0 else "", qual)).encode()
    fq = tmp_path / "t.fq"
    fq.write_bytes(text)

    def scan(path, beg, end):
        st = Stripe()
        rc = L.bb_fq_scan_stripe(str(path).encode(), beg, end, C.byref(st))
        out = [(st.off[k], st.len[k]) for k in range(st.n)] if rc == 0 else None
        L.bb_fq_stripe_free(C.byref(st))
        return out

    assert scan(fq, 0, len(text)) == recs
    for cut in range(1, len(text)):
        a, b = scan(fq, 0, cut), scan(fq, cut, len(text))
        assert a is not None and b is not None and a + b == recs, cut
    thirds = [scan(fq, len(text) * k // 3, len(text) * (k + 1) // 3) for k in range(3)]
    assert sum(thirds, []) == recs
    # two-line FASTA
    fa = tmp_path / "t.fa"
    fa.write_bytes(b"".join(b">s%d c\n%s\n" % (k, b"ACGT" * k) for k in range(1, 30)))
    size = fa.stat().st_size
    whole = scan(fa, 0, size)
    assert len(whole) == 29 and [n for _, n in whole] == [4 * k for k in range(1, 30)]
    for cut in range(1, size, 7):
        assert scan(fa, 0, cut) + scan(fa, cut, size) == whole
    # unfit inputs
    wrapped = tmp_path / "w.fq"
    wrapped.write_bytes(b"@a\nACGT\nACGT\n+\nIIII\nIIII\n")
    assert scan(wrapped, 0, 100) is None
    trunc = tmp_path / "x.fq"
    trunc.write_bytes(b"@a\nACGT\n+\nIIII\n@b\nAC\n+\n")
    assert scan(trunc, 0, 100) is None
    import gzip
    gz = tmp_path / "g.fq.gz"
    gz.write_bytes(gzip.compress(text))
    assert scan(gz, 0, 100) is None


def test_batch_bounds_follow_the_reader_rule():
    """batch_bounds == simulating bseq_read's loop (bwa.c:79-112) record by record."""
    import random
    from bwa_b200.multi import batch_bounds
    rng = random.Random(9)
    for trial in range(200):
        n = rng.randrange(1, 60)
        lens = [rng.choice([0, 1, 50, 100, 151, 400]) for _ in range(n)]
        chunk = rng.choice([1, 100, 300, 1000, 10 ** 6])
        two_files = trial % 2 == 0
        if two_files and n % 2:
            lens.append(100)
        # reference loop over records (two files: a pair per step; one file: a record per step, the batch ends at even n)
        starts, k = [0], 0
        while k < len(lens):
            size, cnt = 0, 0
            while k < len(lens):
                step = 2 if two_files else 1
                size += sum(lens[k:k + step]); k += step; cnt += step
                if size >= chunk and cnt % 2 == 0:
                    break
            starts.append(k)
        pair = [sum(lens[j:j + 2]) for j in range(0, len(lens), 2)]
        got = [min(2 * s, len(lens)) for s in batch_bounds(pair, chunk)]
        assert got == starts, (lens, chunk, two_files)
