#!/usr/bin/env python
"""bench.py -- reads/sec of the BWA-MEM seed-and-extend hot path on B200 (BASELINE.json metric).

One "step" = one pass of mem_process_seqs (the drop-in boundary) over one batch of synthetic reads:
  e2e    host buffers in, SAM text out, every host<->device copy inside the timed region  (headline)
  value  the same reads / the CUDA-event time of the four kernels (inputs resident in HBM)
  roofline  dominant kernel = SMEM seeding: 64 B x Occ-block touches / its CUDA-event time vs measured HBM peak
  cpu_baseline  the unmodified reference (oracle/_ref/bwa mem -t <cores>) on a bounded sample of the same reads
`--impl reference` times the reference binary alone and prints the same line shape.

Workload (config.workload): synthetic uniform-random reference of --ref-mbp Mbp in contigs of <= 125 Mbp,
150-bp single-end reads with 1 % error (0.8 sub / 0.1 ins / 0.1 del), BASELINE.json configs[1].  The index is
the reference's own on-disk format; for references too large to index with `bwa index` inside a benchmark run it
is produced by this repo's GPU index builder, which is checked byte-for-byte against `bwa index` on small inputs.
Inputs are larger than L2 (index >= hundreds of MB, reads >= 100 MB), so no L2 flush is needed between steps.
The e2e region keeps --inflight calls running from as many host threads and spaces their starts (class Pacer: waits inside the timed region).
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

REF_BWA = os.path.join(ROOT, "oracle", "_ref", "bwa")


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def effective_cpus():
    """CPUs this process may actually use: min(affinity mask, cgroup CPU quota).  GPU boxes of this pool show 128
    logical CPUs but run the container under a CFS quota (cpu.max); oversubscribing the quota gets every thread throttled."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            q, per = open(path).read().split()[:2]
            if q != "max":
                n = min(n, max(1, int(round(int(q) / int(per)))))
        except Exception:
            pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            n = min(n, max(1, int(round(q / per))))
    except Exception:
        pass
    return n


# Other workloads of BASELINE.json (configs 4 and 5) and a repeat-rich reference, selected with --workload; the default (the
# headline) stays 2x150-bp pairs against the 3 Gbp uniform-random reference.  reads = per GPU per step.
WORKLOADS = {
    "pe":      dict(layout="pe", read_len=150, reads=1_000_000),
    "se":      dict(layout="se", read_len=150, reads=1_000_000),
    "len36":   dict(layout="se", read_len=36, reads=2_000_000),
    "len75":   dict(layout="se", read_len=75, reads=2_000_000),
    "len300":  dict(layout="se", read_len=300, reads=500_000),
    "len1000": dict(layout="se", read_len=1000, reads=100_000),
    "pacbio":  dict(layout="se", read_len=10000, reads=2_000, err=(0.02, 0.05, 0.03), mem_args=["-x", "pacbio"]),   # 10 % error: 20 % sub / 50 % ins / 30 % del
    "stress":  dict(layout="pe", read_len=150, reads=100_000, ref="stress", ref_mbp=1000, err=(0.016, 0.002, 0.002), chimeric=0.05),
}


def make_workload(workdir, ref_mbp, n_reads, read_len, seed, rank=0, paired=False, ref="random", err=(0.008, 0.001, 0.001), chimeric=0.0):
    """Reference FASTA + index (once per box) and this rank's reads."""
    import gen_data
    import numpy as np
    os.makedirs(workdir, exist_ok=True)
    if ref == "stress":
        return make_stress_workload(workdir, ref_mbp, n_reads, read_len, seed, rank, paired, err, chimeric)
    fa = os.path.join(workdir, "ref_%d.fa" % ref_mbp)
    contig_len = min(125_000_000, ref_mbp * 1_000_000)
    n_contigs = max(1, (ref_mbp * 1_000_000) // contig_len)
    done = fa + ".done"
    if rank == 0 and not os.path.exists(done):
        t0 = time.time()
        contigs = gen_data.random_contigs(n_contigs, contig_len, 7)
        if ref_mbp <= 60:
            # small enough for the index builder on the CPU (the files of `bwa index`, byte for byte; 60 Mbp: 20 s, 3.8 GB on 8 cores)
            import bwa_b200.index_build as ib
            gen_data.write_fasta(fa, contigs)
            ib.build(fa, device="cpu", verbose=False)
        else:
            # `bwa index` needs hours at this size (bwa.1:767): same files from the GPU builder (bwa_b200/index_build.py,
            # byte-identical to `bwa index` where both can run, see tests/test_gpu_parity.py::test_index_builder)
            # ... in a child process: the builder's torch allocations (tens of GB of cached blocks) must be gone before
            # the aligner places its 34 GB index on the same GPU (a build inside this process ended in cudaMalloc: out of memory)
            del contigs
            code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r); import gen_data, bwa_b200.index_build as ib; "
                    "ib.build_from_contigs(gen_data.random_contigs(%d, %d, 7), %r, verbose=True)" % (ROOT, os.path.join(ROOT, "tools"), n_contigs, contig_len, fa))
            subprocess.run([sys.executable, "-c", code], check=True, stdout=sys.stderr)
        log("[bench] reference %d Mbp generated and indexed in %.1fs" % (ref_mbp, time.time() - t0))
        open(done, "w").write("ok")
    while not os.path.exists(done):
        time.sleep(0.5)
    tag = os.path.join(workdir, "reads_%s%d_%d_e%d_r%d" % ("pe" if paired else "se", n_reads, read_len, int(round(1000 * sum(err))), rank))
    fqs = [tag + "_1.fq", tag + "_2.fq"] if paired else [tag + ".fq"]
    if not all(os.path.exists(f) for f in fqs):
        t0 = time.time()
        # reads are drawn without materialising the FASTA again: regenerate the contigs from the seed
        contigs = gen_data.random_contigs(n_contigs, contig_len, 7)
        r1, r2 = gen_data.gen_reads(contigs, n_reads // 2 if paired else n_reads, read_len, seed + rank, err=err, paired=paired, chimeric=chimeric)
        gen_data.write_fastq(fqs[0], r1)
        if paired:
            gen_data.write_fastq(fqs[1], r2)
        log("[bench] %d reads written in %.1fs" % (n_reads, time.time() - t0))
    return fa, fqs


def make_stress_workload(workdir, ref_mbp, n_reads, read_len, seed, rank, paired, err, chimeric):
    """Repeat-rich reference (tools/gen_data.py stress_contigs: a 1 kb family at 3 % divergence over ~15 % of the sequence, tandem
    repeats, N runs, two contigs), indexed by the GPU builder; reads with 2 % error and 5 % chimeras as in the parity tests."""
    import gen_data
    fa = os.path.join(workdir, "stress_%d.fa" % ref_mbp)
    done = fa + ".done"
    if rank == 0 and not os.path.exists(done):
        t0 = time.time()
        gen_data.write_fasta(fa, gen_data.stress_contigs(ref_mbp * 1_000_000, 5))
        code = ("import sys; sys.path.insert(0, %r); import bwa_b200.index_build as ib; ib.build(%r, verbose=True)" % (ROOT, fa))
        subprocess.run([sys.executable, "-c", code], check=True, stdout=sys.stderr)
        log("[bench] repeat-rich reference %d Mbp generated and indexed in %.1fs" % (ref_mbp, time.time() - t0))
        open(done, "w").write("ok")
    while not os.path.exists(done):
        time.sleep(0.5)
    tag = os.path.join(workdir, "stress_reads_%s%d_%d_r%d" % ("pe" if paired else "se", n_reads, read_len, rank))
    fqs = [tag + "_1.fq", tag + "_2.fq"] if paired else [tag + ".fq"]
    if not all(os.path.exists(f) for f in fqs):
        contigs = gen_data.stress_contigs(ref_mbp * 1_000_000, 5)
        r1, r2 = gen_data.gen_reads(contigs, n_reads // 2 if paired else n_reads, read_len, seed + rank, err=err, paired=paired, chimeric=chimeric)
        gen_data.write_fastq(fqs[0], r1)
        if paired:
            gen_data.write_fastq(fqs[1], r2)
    return fa, fqs


class ClockSampler(threading.Thread):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        self.cmd = ["nvidia-smi", "-i", str(gpu_index), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "200"]
        self.rows = []
        self.p = None

    def run(self):
        try:
            self.p = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.p.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        if self.p:
            self.p.terminate()
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = max([int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()] or [0])
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def time_reference(fa, fqs, n_sample, threads, keep_sam=False, mem_args=()):
    """`bwa mem -t threads` of the unmodified reference on the first n_sample reads; reads/s from its own
    '[M::mem_process_seqs] Processed N reads in X CPU sec, Y real sec' lines (excludes index load and I/O)."""
    samples = []
    per_file = n_sample // len(fqs)
    for fq in fqs:
        sample = fq + ".sample%d" % per_file
        if not os.path.exists(sample):
            with open(fq, "rb") as f, open(sample, "wb") as o:
                for i, line in enumerate(f):
                    if i >= 4 * per_file:
                        break
                    o.write(line)
        samples.append(sample)
    ref_out = samples[0] + ".ref.sam" if keep_sam else os.devnull
    with open(ref_out, "wb") as so:
        r = subprocess.run([REF_BWA, "mem", "-t", str(threads), "-K", "100000000"] + list(mem_args) + [fa] + samples, stdout=so, stderr=subprocess.PIPE, text=True)
    time_reference.last = (samples, ref_out)
    n, real = 0, 0.0
    for m in re.finditer(r"Processed (\d+) reads in ([\d.]+) CPU sec, ([\d.]+) real sec", r.stderr):
        n += int(m.group(1)); real += float(m.group(3))
    if n == 0 or real <= 0:
        raise RuntimeError("reference run produced no timing lines:\n" + r.stderr[-2000:])
    return n / real, n


def dump_outputs(out_dir, sam, n_reads, fa, n_sample=262144):
    """What one mem_process_seqs call returned -- the SAM text of each read -- as arrays DIR/<name>.npy (float64, one row per
    read of a fixed sample of at most n_sample reads, seed 0): fields of the read's first record, its record count and the CRC-32
    of its whole text, so that two builds can be compared output for output.  sam: char *[n_reads] (bb_batch_detach_sam)."""
    import ctypes as C
    import zlib
    import numpy as np
    rows = np.arange(n_reads) if n_reads <= n_sample else np.sort(np.random.default_rng(0).choice(n_reads, n_sample, replace=False))
    names = open(fa + ".ann").read().split("\n")[1::2]
    contig = {l.split()[1]: float(i) for i, l in enumerate(names) if l.strip()}
    p = C.cast(sam, C.POINTER(C.c_char_p))
    cols = {k: np.full(len(rows), -1.0) for k in ("flag", "ref_id", "pos", "mapq", "tlen", "as", "xs", "nm", "n_records", "sam_crc32")}
    for j, i in enumerate(rows):
        text = p[int(i)] or b""
        rec = text.split(b"\n")
        f = rec[0].split(b"\t")
        cols["n_records"][j] = sum(1 for r in rec if r)
        cols["sam_crc32"][j] = zlib.crc32(text)
        if len(f) < 11:
            continue
        cols["flag"][j], cols["pos"][j], cols["mapq"][j], cols["tlen"][j] = int(f[1]), int(f[3]), int(f[4]), int(f[8])
        cols["ref_id"][j] = contig.get(f[2].decode(), -1.0)
        for t in f[11:]:
            if t[:5] in (b"AS:i:", b"XS:i:", b"NM:i:"):
                cols[t[:2].decode().lower()][j] = int(t[5:])
    cols["read_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, v in cols.items():
        np.save(os.path.join(out_dir, k + ".npy"), v)
    log("[bench] outputs of the last timed step (%d of %d reads) written to %s" % (len(rows), n_reads, out_dir))


def supervise(argv):
    """Single-GPU runs happen in a child process under a watchdog: a GPU job that stops making progress must not take the
    whole benchmark with it.  The child prints the JSON line; if it hangs it is killed and the run is repeated once in the
    most conservative configuration (one call in flight), which is recorded in the line."""
    limit = int(os.environ.get("BWA_B200_BENCH_TIMEOUT", "900"))
    for attempt in (0, 1):
        env = dict(os.environ)
        extra = []
        if attempt == 1:
            env["BWA_B200_INFLIGHT"] = "1"
            extra = ["--inflight", "1"]
        p = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker"] + list(argv) + extra, stdout=subprocess.PIPE, env=env, start_new_session=True)
        try:
            out, _ = p.communicate(timeout=limit)
        except subprocess.TimeoutExpired:
            log("[bench] attempt %d made no progress for %d s: killing it" % (attempt, limit))
            try:
                os.killpg(p.pid, 9)
            except Exception:
                p.kill()
            p.communicate()
            continue
        text = out.decode()
        if p.returncode == 0 and attempt == 1:
            try:
                line = json.loads(text.strip().splitlines()[-1])
                line["config"]["watchdog"] = "first attempt hung and was killed; this is the repeat with one call in flight"
                text = json.dumps(line) + "\n"
            except Exception:
                pass
        sys.stdout.write(text)
        sys.stdout.flush()
        return p.returncode
    return 3


class Pacer:
    """Keeps concurrent mem_process_seqs calls out of phase.  Identical calls that start together stay together: they share the GPU
    evenly, reach their host-side phases (encode at the start; insert-size model, text splice at the end) at the same time and
    leave the GPU idle meanwhile -- measured: the chunks of three calls in flight complete within 40 ms of each other, wave after wave
    (profiles/r2_final2_timeline_pe.txt).  A real caller's batches arrive spaced (the command line parses one while the others
    align); this harness hands over all batches at once, so it spaces the STARTS instead: a call may not start sooner than `gap` after
    the previous start, with gap = 0.7 x the mean interval between the last completions (always below the achievable step time, so
    pacing never limits throughput; once the calls are out of phase nobody waits).  Until enough completions exist the gap is a
    small fraction of the shortest call seen.  The waits are inside the timed region."""

    def __init__(self, inflight, enabled=True):
        self.inflight, self.enabled = inflight, enabled and inflight > 1
        self.lock = threading.Lock()
        self.last_start, self.dmin, self.done, self.waited = 0.0, None, [], 0.0

    def new_run(self):
        with self.lock:
            self.done = []

    def gap(self):
        if len(self.done) > self.inflight:
            return min(0.2, 0.7 * (self.done[-1] - self.done[-1 - self.inflight]) / self.inflight)
        return min(0.1, 0.6 * self.dmin / self.inflight) if self.dmin else 0.0

    def before_start(self):
        if not self.enabled:
            return
        with self.lock:
            now = time.perf_counter()
            at = max(now, self.last_start + self.gap())
            self.last_start = at
            self.waited += at - now
        if at > now:
            time.sleep(at - now)

    def after_end(self, duration):
        with self.lock:
            self.done.append(time.perf_counter())
            if self.dmin is None or duration < self.dmin:
                self.dmin = duration


# SASS instructions per DP cell of the kernels' inner loops (cuobjdump -sass, counted by tools/sass_loops.py / by hand from the
# unrolled 8-cell chunk of k_extend_lane: 220 instructions; k_global_sm_fast: 71 per 32-column chunk + per-row work, see profiles/)
SASS_OPS_PER_CELL = {"extend": 27.5, "global": 71.0 / 32}


def roofline_sw(ks, clocks, ksteps):
    """Integer-issue roofline of the two Smith-Waterman kernels (SURVEY.md 8d): achieved cell updates/s against
    (lanes x SMs x measured SM clock) / (SASS instructions per cell of the kernel's cell loop)."""
    mhz = (clocks or {}).get("sm_mhz") or 1965
    lane_ops = 148 * 128 * mhz * 1e6
    out = {"int_lane_ops_per_s": lane_ops, "int_peak_source": "148 SMs x 128 INT32 lanes x SM clock sampled under load (nvidia-smi)"}
    for name, cells, ms in (("extend", ks["ext_cells"], ks["ms_extend"]), ("global", ks["glb_cells"], ks["ms_global"])):
        if ms > 0:
            ach = cells / (ms * 1e-3)
            peak = lane_ops / SASS_OPS_PER_CELL[name]
            out[name] = {"kernel": "k_extend_lane (ksw_extend2)" if name == "extend" else "k_global_sm_fast (ksw_global2 + backtrack, NM, MD)", "achieved": ach / 1e9, "peak": peak / 1e9, "unit": "GCUPS",
                         "frac": ach / peak, "ops_per_cell": SASS_OPS_PER_CELL[name]}
    return out


def selfcheck_status():
    try:
        import ctypes as C
        import bwa_b200
        L = bwa_b200.lib()
        L.bb_selfcheck_status.restype = C.c_int
        return int(L.bb_selfcheck_status())
    except Exception:
        return -1


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-mbp", type=int, default=int(os.environ.get("BWA_B200_BENCH_REF_MBP", "3000")))
    ap.add_argument("--reads", type=int, default=int(os.environ.get("BWA_B200_BENCH_READS", "1000000")))
    ap.add_argument("--read-len", type=int, default=150)
    ap.add_argument("--layout", default=os.environ.get("BWA_B200_BENCH_LAYOUT", "pe"), choices=["pe", "se"], help="pe: 2x150 bp pairs (FR, insert N(400,50)); se: single-end")
    ap.add_argument("--workload", default=None, choices=sorted(WORKLOADS), help="a named workload (overrides --layout/--reads/--read-len): BASELINE.json configs 4-5 and a repeat-rich reference")
    ap.add_argument("--threads", type=int, default=0, help="host threads (0 = all cores / ranks)")
    ap.add_argument("--workdir", default=os.environ.get("BWA_B200_BENCH_DIR", "/tmp/bwa_b200_bench"))
    ap.add_argument("--cpu-sample", type=int, default=None, help="reads of the workload the CPU reference aligns (default: 1 M for the cpu_baseline of the B200 arm, the whole step for --impl reference)")
    ap.add_argument("--inflight", type=int, default=int(os.environ.get("BWA_B200_INFLIGHT", "3")), help="mem_process_seqs calls issued at a time (host threads), as bwa-b200 mem does")
    ap.add_argument("--worker", action="store_true", help="(internal) run the measurement in this process; without it a parent process supervises the run")
    ap.add_argument("--dense-sa", type=int, default=int(os.environ.get("BWA_B200_DENSE_SA", "0")))
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="write what the last timed step returned (per-read SAM fields of a fixed sample) as DIR/<name>.npy")
    a = ap.parse_args()
    a.cpu_sample_given = a.cpu_sample is not None
    if a.cpu_sample is None:
        a.cpu_sample = 1_000_000   # ~10 s of `bwa mem -t 16`: the whole step of the default workload
    wl = dict(WORKLOADS[a.workload]) if a.workload else {}
    if wl:
        a.layout, a.read_len, a.reads = wl["layout"], wl["read_len"], int(os.environ.get("BWA_B200_BENCH_WL_READS", wl["reads"]))
        a.ref_mbp = wl.get("ref_mbp", a.ref_mbp)
        a.cpu_sample = min(a.cpu_sample, max(200, 3_000_000 // a.read_len))
    wl_kw = dict(ref=wl.get("ref", "random"), err=wl.get("err", (0.008, 0.001, 0.001)), chimeric=wl.get("chimeric", 0.0))
    mem_args = wl.get("mem_args", [])

    if a.impl == "b200" and not a.worker and "RANK" not in os.environ:
        return supervise(sys.argv[1:])

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ncores = effective_cpus()
    threads = a.threads or max(1, ncores // max(1, world))
    paired = a.layout == "pe"
    workload = "%d synthetic %s reads per GPU per step (%s), ERRPCT error, vs %d Mbp uniform-random reference" % (
        a.reads, "2x%d-bp PE" % a.read_len if paired else "%d-bp SE" % a.read_len, "%d pairs, FR, insert N(400,50)" % (a.reads // 2) if paired else "single-end", a.ref_mbp)
    workload = workload.replace("ERRPCT", "%g%%" % round(100 * sum(wl_kw["err"]), 2))
    if wl:
        workload += " [--workload %s: error profile sub/ins/del %s%s%s%s]" % (a.workload, wl_kw["err"], ", %.0f %% chimeric reads" % (100 * wl_kw["chimeric"]) if wl_kw["chimeric"] else "",
                                                                          ", repeat-rich reference (gen_data.stress_contigs)" if wl_kw["ref"] == "stress" else "", ", bwa mem " + " ".join(mem_args) if mem_args else "")

    if a.impl == "reference":
        if rank != 0:
            return
        fa, fq = make_workload(a.workdir, a.ref_mbp, a.reads, a.read_len, 1000, 0, paired, **wl_kw)
        # a step = the whole per-step workload (1 M reads: ~10 s on 16 cores) unless --cpu-sample asks for less; the run stops taking
        # further steps once ~4 minutes are used (the steps done are the ones reported)
        n_sample = min(a.reads, a.cpu_sample if a.cpu_sample_given else a.reads)
        vals, t_run = [], time.time()
        for s in range(a.warmup + a.steps):
            t0 = time.time()
            v, n = time_reference(fa, fq, n_sample, ncores, mem_args=mem_args)
            if s >= a.warmup or time.time() - t_run > 240:
                vals.append((v, n, time.time() - t0))
            if time.time() - t_run > 240:   # keep the whole run within minutes
                break
        v = sum(x[0] for x in vals) / len(vals)
        line = {"impl": "reference", "metric": "reads_per_sec", "value": v, "unit": "reads/s", "n_gpus": a.gpus, "steps": len(vals), "warmup": a.warmup,
                "ms_per_step": 1e3 * vals[0][1] / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": {"workload": workload},
                "cpu_baseline": {"value": v, "unit": "reads/s", "cores": ncores, "kind": "reference", "sample": "first %d reads of the workload, bwa mem -t %d, rate from its own Processed-lines" % (n_sample, ncores)},
                "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    import ctypes as C
    import bwa_b200

    # hard deadline for this process: a GPU job that stops making progress becomes a failed run, not a hung box
    deadline = threading.Timer(float(os.environ.get("BWA_B200_BENCH_DEADLINE", "1500")), lambda: (log("[bench] deadline exceeded: giving up"), os._exit(4)))
    deadline.daemon = True
    deadline.start()

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    bound = None
    if os.environ.get("BWA_B200_BIND", "0") == "1":   # opt-in: stay on the GPU's NUMA node (host workers, lanes, pinned buffers); measured at N=2: no gain (profiles/r2_final_n2b_*)
        bound = bwa_b200.bind_to_gpu_node(local_rank)
        log("[bench] rank %d: %s" % (rank, "bound to the %d CPUs of GPU %d's NUMA node" % (len(bound), local_rank) if bound else "NUMA node of the GPU unknown, not bound"))
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    fa, fq = make_workload(a.workdir, a.ref_mbp, a.reads, a.read_len, 1000, rank, paired, **wl_kw)
    if world > 1:
        dist.barrier()

    L = bwa_b200.lib()
    if world > 1:
        # one copy of the index per GPU: rank 0 loads it and fills the blob, a single NCCL broadcast over NVLink replicates it
        from bwa_b200 import multi
        torch.cuda.synchronize()
        t0 = time.time()
        p, keep = multi.replicate_index(L, fa, rank, local_rank, dist, True)
        torch.cuda.synchronize()
        if rank == 0:
            log("[bench] index replicated to %d GPUs (fill + NCCL broadcast) in %.3fs" % (world, time.time() - t0))
        idx = bwa_b200.Index.wrap(p, L, keep)
    else:
        idx = bwa_b200.Index(fa)
    idx.attach()
    if a.dense_sa:
        idx.densify_sa(a.dense_sa)
    index_verified = None
    if a.ref_mbp > 60 and rank == 0 and os.environ.get("BWA_B200_BENCH_VERIFY", "1") != "0":
        # the index files of this workload come from this repository's GPU builder, not from `bwa index`: check EVERY row of the
        # resident BWT / suffix array against the resident text before trusting any alignment made with it (k_index_verify)
        t0 = time.time()
        index_verified = idx.verify(0, 1)
        index_verified["seconds"] = round(time.time() - t0, 2)
        log("[bench] index verified against the text: %r" % (index_verified,))
        if index_verified["bwt_text_sa_mismatches"] or index_verified["order_violations"]:
            raise SystemExit("bench.py: the index does not describe the reference text")

    opt = L.mem_opt_init()
    opt.contents.n_threads = threads
    if mem_args == ["-x", "pacbio"]:   # the preset of the command line (fastmap.c:330-358), applied to the library call
        o = opt.contents
        o.o_del = o.e_del = o.o_ins = o.e_ins = 1
        o.b = 1
        o.split_factor = 10.0
        o.min_chain_weight = 40
        o.min_seed_len = 17
        o.pen_clip5 = o.pen_clip3 = 0
        L.bwa_fill_scmat.argtypes = [C.c_int, C.c_int, C.c_void_p]
        L.bwa_fill_scmat(o.a, o.b, C.addressof(o.mat))
    elif mem_args:
        raise SystemExit("bench.py: no library mapping for bwa mem options %r" % (mem_args,))
    inflight = max(1, min(4, a.inflight))
    batches = [bwa_b200.ReadBatch(*fq) for _ in range(inflight)]     # one host copy of the step's reads per call in flight
    batch = batches[0]
    if paired:
        opt.contents.flag |= bwa_b200.MEM_F_PE
    n_reads = batch.n

    L.bb_batch_detach_sam.restype = C.c_void_p
    L.bb_batch_detach_sam.argtypes = [C.c_int, C.c_void_p]
    L.bb_batch_free_detached.argtypes = [C.c_int, C.c_void_p]
    held = []

    def release():
        while held:
            L.bb_batch_free_detached(batch.n, held.pop())

    def step(b=None):
        b = b or batch
        bwa_b200.mem_process_seqs(opt, idx, b)
        # the SAM text is in host memory now; its release (what fastmap.c:114-119 does after printing) is kept out of the timed region
        held.append(L.bb_batch_detach_sam(b.n, b.seqs))

    pacer = Pacer(inflight, os.environ.get("BWA_B200_BENCH_PACE", "1") != "0")

    def run_steps(n_steps):
        """n_steps calls of mem_process_seqs, `inflight` at a time from as many host threads (ctypes drops the GIL),
        the way the command line keeps two batches in flight (bb_cli.c)."""
        if inflight == 1:
            for _ in range(n_steps):
                step()
            return
        todo = list(range(n_steps))
        lock = threading.Lock()

        pacer.new_run()

        def work(w):
            while True:
                with lock:
                    if not todo:
                        return
                    todo.pop()
                pacer.before_start()
                t_call = time.perf_counter()
                step(batches[w])
                pacer.after_end(time.perf_counter() - t_call)
        ths = [threading.Thread(target=work, args=(w,)) for w in range(inflight)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()

    run_steps(a.warmup)
    release()
    idx.stats(reset=True)
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    pacer.waited = 0.0
    run_steps(a.steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    pacer_waited = pacer.waited
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    st = idx.stats()
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, held[-1], n_reads, fa)   # held[-1]: the SAM of the step that completed last
    release()
    # Kernel-only figures (value, roofline): the timed region above overlaps several chunks on different streams, so
    # per-kernel event times there include waiting for each other.  Two more passes with ONE lane and ONE chunk give
    # each kernel the GPU alone ("timed in isolation", burst peak applies); they are not part of the e2e number.
    pipe_cfg = "chunks of %s reads on %s lanes (streams) per call" % (os.environ.get("BWA_B200_CHUNK", "262144" if paired else "131072"),
                                                                          os.environ.get("BWA_B200_LANES", "2" if inflight > 1 else "3"))
    user_env = {k: os.environ.get(k) for k in ("BWA_B200_LANES", "BWA_B200_CHUNK")}
    os.environ["BWA_B200_LANES"] = "1"
    os.environ["BWA_B200_CHUNK"] = str(1 << 30)
    step()
    release()
    idx.stats(reset=True)
    KSTEPS = 2
    for _ in range(KSTEPS):
        step()
        release()
    torch.cuda.synchronize()
    ks = idx.stats()
    for k, v in user_env.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v
    k_ms = (ks["ms_smem"] + ks["ms_sa"] + ks["ms_chain"] + ks["ms_extend"] + ks["ms_global"] + ks.get("ms_tail", 0.0) + ks.get("ms_localsw", 0.0)) / KSTEPS * a.steps
    vals = torch.tensor([dt, k_ms / 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(vals, op=dist.ReduceOp.MAX)
    dt_max, k_max = float(vals[0]), float(vals[1])
    total_reads = n_reads * a.steps * world

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        smem_gbs = ks["occ_touches"] * 64 / (ks["ms_smem"] * 1e-3) / 1e9 if ks["ms_smem"] > 0 else 0.0
        traffic = None
        try:   # DRAM bytes of the seeding kernels per launch, from the committed ncu --set full captures
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            # captured on the default configuration (short-string table depth 14) of the 3 Gbp / 150-bp workload: valid there only
            k1 = "k_smem" if os.environ.get("BWA_B200_K1_COMPACT") == "0" else "k_smem_c"   # the seeding kernel in use (compact candidate lists by default)
            if a.read_len == 150 and a.ref_mbp == 3000 and os.environ.get("BWA_B200_KTAB") is None:
                traffic = (tr[k1]["dram_bytes_per_read"] + tr["k_smem_fwd"]["dram_bytes_per_read"]) * n_reads
        except Exception:
            pass
        line = {
            "metric": "reads_per_sec", "value": total_reads / k_max if k_max > 0 else None, "unit": "reads/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": 1e3 * dt_max / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
            "config": {"workload": workload, "parallelism": "reads sharded over %d GPU(s), full index copy per GPU" % world, "host_threads_per_rank": threads, "numa_bound_cpus": len(bound) if bound else None,
                       "l2": "inputs larger than L2 (resident index %.1f GB = Occ blocks + SA sample + pac + short-string table, reads %.0f MB per step)" % (
                           os.path.getsize(fa + ".bwt") / 1e9 * (1.25 + 16.0 / (a.dense_sa or int(os.environ.get("BWA_B200_SA_INTV", "2")))) + 5.7, n_reads * a.read_len / 1e6),
                       "value_definition": "reads / summed CUDA-event time of the seeding, SA, chaining, extension, global-alignment and post-processing (stage 4) kernels, inputs resident in HBM, measured in two extra single-stream passes after the timed region",
                       "timed_region_note": "every step re-submits the same host batch (bases already 0..4 codes after the first call: the in-place encode then re-writes them); releasing the SAM strings (what the reference's caller does after printing, fastmap.c:114-119) is outside the timed region",
                       "pipeline": pipe_cfg + ", %d mem_process_seqs calls in flight" % inflight + (", starts paced >= 0.7 x the mean completion interval apart so that the calls stay out of phase (waited %.0f ms in all, inside the timed region)" % (1e3 * pacer_waited) if pacer.enabled else ""),
                       "device_selfcheck": {0: "not run", 1: "passed (192 reads from the reference: default kernels == baseline kernels)", 2: "DIFFERED: the baseline kernels (first row sweeps, no short-string table) are in use"}.get(selfcheck_status(), "?"),
                       "index_verified": index_verified,
                       "sa_interval": a.dense_sa or int(os.environ.get("BWA_B200_SA_INTV", "2")), "sa_interval_note": "index files sample every 32nd row; the device re-samples it at load time"},
            "e2e": {"value": total_reads / dt_max, "unit": "reads/s", "h2d_bytes_per_step": st["h2d_bytes"] // a.steps, "d2h_bytes_per_step": st["d2h_bytes"] // a.steps},
            "gpu_launches": st["n_launch"],
            "clocks": clocks,
            "roofline": {"kernel": "k_smem_fwd + %s + k_seed_post (SMEM seeding over the FM-index)" % ("k_smem" if os.environ.get("BWA_B200_K1_COMPACT") == "0" else "k_smem_c"), "bound": "hbm", "achieved": smem_gbs, "peak": hbm_peak, "unit": "GB/s",
                         "frac": smem_gbs / hbm_peak if hbm_peak else None, "traffic": traffic,
                         "traffic_note": "DRAM bytes of the seeding kernel + k_smem_fwd per launch from the committed ncu --set full capture (profiles/r2_traffic.json), scaled to the reads of one launch; null when the workload is not the captured one",
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if "hbm_gbs" in peaks else "fallback 6650 GB/s",
                         "algorithmic_bytes": "64 B x %d Occ-block touches per step" % (st["occ_touches"] // a.steps)},
            "kernels_ms_per_step": {k: ks.get(k, 0.0) / KSTEPS for k in ("ms_smem", "ms_sa", "ms_chain", "ms_extend", "ms_global", "ms_tail", "ms_localsw", "ms_h2d", "ms_d2h")},
            "device_tail": {"reads": st["tail_reads"] // a.steps, "handed_back_to_host_postprocessing": st["tail_complex"] // a.steps,
                            "note": "stage 4 (bwag_tail.cu): de-duplication, CIGAR requests, pairing, MAPQ and SAM records on the device; reads it hands back are re-aligned with host-side post-processing"},
            "work_per_read": {"occ_touches": st["occ_touches"] / (n_reads * a.steps), "sa_touches": st["sa_touches"] / (n_reads * a.steps),
                              "ext_cells": st["ext_cells"] / (n_reads * a.steps), "glb_cells": st["glb_cells"] / (n_reads * a.steps)},
            "roofline_sw": roofline_sw(ks, clocks, KSTEPS),
            "sw_gcups": {"extend": ks["ext_cells"] / (ks["ms_extend"] * 1e-3) / 1e9 if ks["ms_extend"] > 0 else None,
                         "global": ks["glb_cells"] / (ks["ms_global"] * 1e-3) / 1e9 if ks["ms_global"] > 0 else None,
                         "note": "cells the kernels computed; the extension kernel stops a sweep at the first row after which no output of ksw_extend2 can change "
                                 "(about a third fewer cells than the reference iterates on this workload: 3.78 k per read with BWA_B200_K4_FAST=0)"},
        }
        if world == 1:
            try:
                n_sample = min(a.reads, a.cpu_sample)
                v, n = time_reference(fa, fq, n_sample, ncores, keep_sam=True, mem_args=mem_args)
                line["cpu_baseline"] = {"value": v, "unit": "reads/s", "cores": ncores, "kind": "reference",
                                        "sample": "first %d reads of the workload, oracle/_ref/bwa mem -t %d, rate from its own Processed-lines" % (n, ncores)}
                # the same sample through `bwa-b200 mem` on the full-size index: its SAM must equal the reference's byte for byte
                samples, ref_out = time_reference.last
                mine = samples[0] + ".b200.sam"
                rc = bwa_b200.run_cli(["mem", "-t", str(threads), "-K", "100000000"] + list(mem_args) + [fa] + samples, mine)
                strip = lambda path: b"\n".join(l for l in open(path, "rb").read().split(b"\n") if not l.startswith(b"@PG"))
                line["cpu_baseline"]["sam_identical_on_sample"] = bool(rc == 0 and strip(mine) == strip(ref_out))
                if not line["cpu_baseline"]["sam_identical_on_sample"]:   # say where: first differing record pair, and keep both files for inspection
                    la, lb = strip(ref_out).split(b"\n"), strip(mine).split(b"\n")
                    k = next((i for i, (x, y) in enumerate(zip(la, lb)) if x != y), min(len(la), len(lb)))
                    cut = lambda l: b"\t".join(l.split(b"\t")[:9] + l.split(b"\t")[11:]).decode("latin1")[:600]
                    line["cpu_baseline"]["sam_diff"] = {"rc": rc, "lines_reference": len(la), "lines_b200": len(lb), "differing_lines": sum(1 for x, y in zip(la, lb) if x != y), "first_at": k,
                                                        "reference": cut(la[k]) if k < len(la) else None, "b200": cut(lb[k]) if k < len(lb) else None}
                    import shutil
                    shutil.copy(ref_out, os.path.join(a.workdir, "sam_diff_reference.sam")); shutil.copy(mine, os.path.join(a.workdir, "sam_diff_b200.sam"))
                    line["cpu_baseline"]["sam_diff"]["kept"] = a.workdir
                for f in (mine, ref_out):
                    os.remove(f)
                if not mem_args and a.ref_mbp >= 1000:
                    # the full-size index is the only place where >1 Occ superblock, 33-bit rows and the depth-14 short-string table are live:
                    # one more sample there, single-end with non-default scoring / seeding / output options (host post-processing path: -a)
                    opts = ["-k", "17", "-A", "2", "-B", "5", "-O", "5,7", "-E", "2,1", "-T", "40", "-Y", "-a"]
                    n2 = min(20000, n_sample)
                    one = samples[0] + ".se%d" % n2
                    with open(samples[0], "rb") as f, open(one, "wb") as o:
                        for i, l in enumerate(f):
                            if i >= 4 * n2:
                                break
                            o.write(l)
                    want = subprocess.run([REF_BWA, "mem", "-v", "1", "-t", str(ncores), "-K", "100000000"] + opts + [fa, one], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL).stdout
                    rc2 = bwa_b200.run_cli(["mem", "-v", "1", "-t", str(threads), "-K", "100000000"] + opts + [fa, one], one + ".sam")
                    spg = lambda b: b"\n".join(l for l in b.split(b"\n") if not l.startswith(b"@PG"))
                    line["cpu_baseline"]["sam_identical_on_se_sample_with_options"] = {"options": " ".join(opts), "reads": n2, "identical": bool(rc2 == 0 and spg(open(one + ".sam", "rb").read()) == spg(want))}
                    os.remove(one + ".sam")
            except Exception as e:  # the baseline is reported, never required for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": "reads/s", "cores": ncores, "kind": "reference", "sample": "failed: %s" % e}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.exit(main() or 0)
