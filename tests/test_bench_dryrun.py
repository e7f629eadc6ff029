"""bench.py's B200 arm from end to end without a GPU: the CUDA kernels run in the SIMT emulator (tests/_build/libbwa_b200_cusim.so) and the
few torch.cuda calls the harness makes are stubbed.  Checks the contract of the JSON line (keys, the e2e block, the kernel named in
`roofline`, SAM identity of the CPU-baseline sample against the reference's), that the pacing of the concurrent calls ran, and that
--dump-outputs writes, read by read, the reference's SAM of the step.  Numbers mean nothing here.  SAM is checked against the stored md5
of the reference's; the benchmark's own comparison runs where the reference binary (oracle/_ref/bwa) is built."""
import json
import os
import subprocess
import sys
import zlib

import numpy as np

from conftest import CUSIMBIN, ROOT, md5, ref_sam_md5, run_sam

DRIVER = r'''
import sys, os
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch
torch.cuda.is_available = lambda: True
torch.cuda.set_device = lambda *a, **k: None
torch.cuda.synchronize = lambda *a, **k: None
_tensor = torch.tensor
torch.tensor = lambda *a, **k: _tensor(*a, **{x: y for x, y in k.items() if x != "device"})
import bwa_b200
bwa_b200.LIB_PATH = os.path.join(ROOT, "tests", "_build", "libbwa_b200_cusim.so")
bwa_b200.CLI_PATH = os.path.join(ROOT, "tests", "_build", "bwa-b200-cusim")
import importlib.util
spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
bench = importlib.util.module_from_spec(spec); spec.loader.exec_module(bench)
sys.argv = ["bench.py", "--worker", "--ref-mbp", "1", "--reads", "1200", "--steps", "4", "--warmup", "3", "--cpu-sample", "400", "--workdir", WORKDIR, "--dump-outputs", DUMP]
bench.main()
'''


def test_bench_worker_line_on_the_emulator(tmp_path):
    work, dump = str(tmp_path / "w"), str(tmp_path / "dump")
    code = "ROOT = %r\nWORKDIR = %r\nDUMP = %r\n" % (ROOT, work, dump) + DRIVER
    env = dict(os.environ, BWA_B200_SELFCHECK="0")
    p = subprocess.run([sys.executable, "-c", code], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=800, env=env, cwd=str(tmp_path))
    assert p.returncode == 0, p.stderr.decode()[-3000:]
    d = json.loads(p.stdout.decode().strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "e2e", "gpu_launches", "clocks", "roofline", "roofline_sw", "cpu_baseline", "kernels_ms_per_step"):
        assert k in d, k
    assert d["steps"] == 4 and d["warmup"] == 3 and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["e2e"]["value"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] > 0 and "k_smem_c" in d["roofline"]["kernel"] and d["roofline"]["bound"] == "hbm"
    assert d["cpu_baseline"]["kind"] == "reference"
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "bwa")):
        assert d["cpu_baseline"]["sam_identical_on_sample"] is True
    samples = sorted(os.path.join(work, f) for f in os.listdir(work) if f.endswith(".sample200"))
    assert len(samples) == 2
    args = ["-K", "100000000", "-t", "4", os.path.join(work, "ref_1.fa")] + samples
    assert md5(run_sam(CUSIMBIN, args)) == ref_sam_md5(args)
    # --dump-outputs: the SAM of the last timed step (all 1200 reads, one batch) is the reference's, read by read
    fqs = sorted(os.path.join(work, f) for f in os.listdir(work) if f.startswith("reads_") and f.endswith(".fq"))
    args = ["-K", "100000000", "-t", "4", os.path.join(work, "ref_1.fa")] + fqs
    sam = run_sam(CUSIMBIN, args)
    assert md5(sam) == ref_sam_md5(args)
    reads = []   # the records of each read in input order: the mates of a pair share the name, not the flag bits 0x40/0x80
    for l in sam.split(b"\n"):
        if l and not l.startswith(b"@"):
            f = l.split(b"\t", 2)
            k = (f[0], int(f[1]) & 0xC0)
            if not reads or reads[-1][0] != k:
                reads.append((k, []))
            reads[-1][1].append(l)
    cols = {k: np.load(os.path.join(dump, k + ".npy")) for k in ("flag", "ref_id", "pos", "mapq", "tlen", "as", "xs", "nm", "n_records", "sam_crc32", "read_index")}
    assert all(v.dtype == np.float64 and v.shape == (1200,) for v in cols.values())
    assert cols["read_index"].tolist() == list(range(1200)) and len(reads) == 1200
    assert cols["n_records"].tolist() == [len(r) for _, r in reads]
    assert cols["sam_crc32"].tolist() == [zlib.crc32(b"\n".join(r) + b"\n") for _, r in reads]
    assert cols["pos"].tolist() == [int(r[0].split(b"\t")[3]) for _, r in reads]
    assert "paced" in d["config"]["pipeline"] and "workload" in d["config"]
