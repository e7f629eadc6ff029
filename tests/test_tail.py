"""Stage 4 (bwag_tail.cu: de-duplication, CIGAR requests, pairing, MAPQ and SAM records on the device) and the
lane-per-read extension kernel (bwag_extend_lane.cu) against the reference binary, with the stage really taken (its
counters say so), with reads it must hand back to the host-side post-processing (repeat-rich reference: XA lists,
supplementary records, mate rescue, region merges), with read groups / comments / FASTA input (no qualities), and with
each of the two switched off (the remaining paths must give the same bytes).  CPU: the SIMT emulator; -m gpu: the B200."""
import os
import re
import subprocess

import pytest

import bwa_b200
from conftest import CUSIMBIN, md5, ref_sam_md5, run_sam, strip_pg


def _counts(binary, args, env=None):
    e = dict(os.environ, BWA_B200_PROFILE="1", BWA_B200_SELFCHECK="0", **(env or {}))   # the start-up self-check would add its own 192 reads to the counters
    p = subprocess.run([binary, "mem", "-v", "1"] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900, env=e)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    took = handed = 0
    for m in re.finditer(rb"stage 4: (\d+) reads, (\d+) handed back", p.stderr):
        took += int(m.group(1)); handed += int(m.group(2))
    _counts.sw = sum(int(m.group(1)) for m in re.finditer(rb"K6: (\d+) local alignments", p.stderr))
    _counts.k5l = sum(int(m.group(1)) for m in re.finditer(rb"lane-per-request kernel made (\d+) of", p.stderr))
    return strip_pg(p.stdout), took, handed, b"lane-per-read kernel" in p.stderr


def _check(binary, data, n_c1, n_stress):
    # unique reference, proper pairs: everything stays on the device
    fa, fqs = data.reads("c1", tag="tl_pe%d" % n_c1, n=n_c1, seed=31, paired=True)
    args = ["-K", "100000000", "-t", "4", "-R", "@RG\\tID:grp1\\tSM:x", fa] + fqs
    sam, took, handed, lane = _counts(binary, args)
    assert md5(sam) == ref_sam_md5(args)
    assert took == 2 * n_c1 and handed * 50 <= took and lane
    # repeat-rich reference, chimeric reads: many reads are handed back, the merged output is still the reference's
    for paired in (True, False):
        fa, fqs = data.reads("stress", tag=("tl_pe%d" if paired else "tl_se%d") % n_stress, n=n_stress, seed=32, paired=paired, err=(0.016, 0.002, 0.002), chimeric=0.05)
        args = ["-K", "100000000", "-t", "4", "-C", fa] + fqs
        sam, took, handed, lane = _counts(binary, args)
        assert md5(sam) == ref_sam_md5(args)
        assert took >= n_stress and 0 < handed < took
        if paired:
            assert _counts.sw > 0          # mate rescue ran its local alignments on the device (K6)
        for env in ({"BWA_B200_TAIL": "0"}, {"BWA_B200_K4_LANE": "0"}, {"BWA_B200_DEVICE_SW": "0"}, {"BWA_B200_K5_LANE": "1"}):
            s2, t2, _, l2 = _counts(binary, args, env)
            assert s2 == sam
            assert (_counts.k5l > 0) == ("BWA_B200_K5_LANE" in env)   # the opt-in lane-per-request global alignment made CIGARs
            assert (t2 == 0) == ("BWA_B200_TAIL" in env) and l2 == ("BWA_B200_K4_LANE" not in env)
            assert (_counts.sw == 0) == ("BWA_B200_DEVICE_SW" in env or not paired)
    # options that keep stage 4 out (-a lists secondary hits, -5 reorders) and options it handles (-M, -Y, -P, -S)
    fa, fqs = data.reads("stress", tag="tl_pe%d" % n_stress, n=n_stress, seed=32, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    for extra, on in ((["-a"], False), (["-5"], False), (["-M", "-Y"], True), (["-P"], True), (["-S"], True), (["-T", "60", "-U", "9"], True)):
        args = extra + ["-K", "100000000", "-t", "4", fa] + fqs
        sam, took, handed, lane = _counts(binary, args)
        assert md5(sam) == ref_sam_md5(args), extra
        assert (took > 0) == on, extra


def test_device_tail_emulated(data):
    _check(CUSIMBIN, data, 96, 64)


def test_device_tail_fasta_input_and_several_chunks(data, tmp_path, monkeypatch):
    """No quality strings (FASTA): QUAL is '*'; chunks smaller than the batch: the insert-size model still sees every pair."""
    fa, fqs = data.reads("c1", tag="tl_fa", n=300, seed=31, paired=True)
    fas = []
    for f in fqs:
        out = str(tmp_path / (os.path.basename(f) + ".fa"))
        with open(f) as i, open(out, "w") as o:
            for k, line in enumerate(i):
                if k % 4 == 0:
                    o.write(">" + line[1:])
                elif k % 4 == 1:
                    o.write(line)
        fas.append(out)
    args = ["-K", "100000000", "-t", "3", fa] + fas
    monkeypatch.setenv("BWA_B200_CHUNK", "64")
    monkeypatch.setenv("BWA_B200_LANES", "2")
    assert md5(run_sam(CUSIMBIN, args)) == ref_sam_md5(args)


@pytest.mark.gpu
def test_device_tail_gpu(data):
    _check(bwa_b200.CLI_PATH, data, 4000, 3000)


def _sb16(binary, data):
    """Occ superblocks of 2^16 symbols (make sb16 / sb16-cuda): a 1 Mbp reference then spans 31 of them, so relative counts,
    per-superblock bases and boundary-crossing rank pairs behave as they do at 2^31 / 2^32 in a 3 Gbp index."""
    if not os.path.exists(binary):
        from conftest import ROOT
        subprocess.run(["make", "-C", ROOT, "sb16" if "cusim" in binary else "sb16-cuda"], check=True, stdout=subprocess.PIPE, stderr=subprocess.PIPE)
    for kw in (dict(tag="sb_se", n=400, seed=41), dict(tag="sb_pe", n=200, seed=42, paired=True)):
        fa, fqs = data.reads("c1", **kw)
        args = ["-K", "100000000", "-t", "4", fa] + fqs
        assert md5(run_sam(binary, args)) == ref_sam_md5(args)


def test_small_superblocks_emulated(data):
    from conftest import ROOT
    _sb16(os.path.join(ROOT, "tests", "_build", "bwa-b200-cusim-sb16"), data)


@pytest.mark.gpu
def test_small_superblocks_gpu(data):
    from conftest import ROOT
    _sb16(os.path.join(ROOT, "tests", "_build", "bwa-b200-sb16"), data)


def _check_seed_filter(binary, data, n_1k, n_pb, pb_len):
    """Reads long enough for the seed-level filter (mem_flt_chained_seeds, >= ~770 bp): K3 lists the local alignments, K6 makes
    them, K3b applies them -- counted, equal to the reference, and equal to chaining + filtering on the host (the switch)."""
    for ref, kw, extra in (("two", dict(tag="sf1k%d" % n_1k, n=n_1k, length=1000, seed=41), []),
                           ("two", dict(tag="sfpb%d" % n_pb, n=n_pb, length=pb_len, seed=42, err=(0.02, 0.05, 0.03)), ["-x", "pacbio"]),
                           ("stress", dict(tag="sfst%d" % n_1k, n=n_1k, length=900, seed=43, err=(0.02, 0.01, 0.01), chimeric=0.1), ["-W", "30"])):
        fa, fqs = data.reads(ref, **kw)
        args = extra + ["-K", "100000000", "-t", "4", fa] + fqs
        sam, _, _, _ = _counts(binary, args)
        assert _counts.sw > 0, (ref, kw)
        assert md5(sam) == ref_sam_md5(args), (ref, kw)
        s2, _, _, _ = _counts(binary, args, {"BWA_B200_DEVICE_SEEDSW": "0"})
        assert _counts.sw == 0 and s2 == sam


def test_seed_filter_on_device_emulated(data):
    _check_seed_filter(CUSIMBIN, data, 8, 3, 3000)


@pytest.mark.gpu
def test_seed_filter_on_device_gpu(data):
    _check_seed_filter(bwa_b200.CLI_PATH, data, 400, 16, 8000)
