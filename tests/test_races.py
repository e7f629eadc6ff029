"""Race detection for the host pipeline: the host glue (worker pool, lanes, batches in flight, buffer caches, order-
restoring writer) built with ThreadSanitizer over the CPU oracle stages, run with several batches, lanes and calls in
flight.  No report may point into the product's host code (the oracle's own statistics counters are not synchronised
and are ignored)."""
import os
import re
import subprocess

import pytest

from conftest import ROOT, md5, ref_sam_md5, strip_pg

TSAN_BIN = os.path.join(ROOT, "tests", "_build", "bwa-b200-tsan")


def test_host_pipeline_is_race_free(data):
    r = subprocess.run(["make", "tsan"], cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    if r.returncode != 0 or not os.path.exists(TSAN_BIN):
        pytest.skip("ThreadSanitizer build not available: " + r.stdout.decode()[-300:])
    fa, fqs = data.reads("stress", tag="tsan", n=400, seed=91, paired=True, err=(0.016, 0.002, 0.002), chimeric=0.05)
    args = ["-K", "12000", "-t", "6", fa] + fqs          # ~40 pairs per batch -> ~10 batches
    env = dict(os.environ, BWA_B200_INFLIGHT="3", BWA_B200_LANES="2", BWA_B200_CHUNK="16", TSAN_OPTIONS="halt_on_error=0 exitcode=0")
    p = subprocess.run([TSAN_BIN, "mem", "-v", "1"] + args, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=800)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    assert md5(strip_pg(p.stdout)) == ref_sam_md5(args)
    reports = re.split(r"WARNING: ThreadSanitizer", p.stderr.decode())[1:]
    ours = []
    for rep in reports:
        top = [l for l in rep.splitlines() if l.strip().startswith("#0")]
        if any("oracle/" not in l for l in top[:2]):      # both accesses of the pair must be outside the oracle to count
            ours.append(rep[:1500])
    assert not ours, "data races in host code:\n" + "\n---\n".join(ours[:3])
