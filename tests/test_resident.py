"""An index that stays on the GPU between runs (SURVEY.md 8-f3; the reference's `bwa shm`, bwashm.c): `bwa-b200 shm idx` starts a
keeper process that exports its device copy, `bwa-b200 mem` attaches to it instead of loading and uploading the index, `shm -l`
lists, `shm -d` ends the keeper.  CPU: the emulator build (the three regions travel as POSIX shared memory); -m gpu: CUDA IPC."""
import os
import subprocess
import time

import pytest

import bwa_b200
from conftest import CUSIMBIN, md5, ref_sam_md5, strip_pg


def _flow(binary, data, tmp_path, n):
    fa, fqs = data.reads("two", tag="res%d" % n, n=n, seed=51, paired=True)
    env = dict(os.environ, BWA_B200_SHM_DIR=str(tmp_path))
    run = lambda args: subprocess.run([binary] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=900, env=env)
    args = ["-K", "100000000", "-t", "4", fa] + fqs
    want = ref_sam_md5(args)
    try:
        r = run(["shm", fa])
        assert r.returncode == 0, r.stderr.decode()[-2000:]
        lst = run(["shm", "-l"]).stdout.decode().split("\n")[0].split("\t")
        assert lst[2] == "resident" and int(lst[1]) > 0
        keeper = int(lst[1])
        for _ in range(2):                                  # two clients, one after the other, over the same device copy
            r = run(["mem"] + args)
            assert r.returncode == 0, r.stderr.decode()[-2000:]
            assert b"using the index resident on the GPU" in r.stderr
            assert b".bwt" not in r.stderr                  # the FM-index files were not opened
            assert md5(strip_pg(r.stdout)) == want
        assert b"already resident" in run(["shm", fa]).stderr
    finally:
        run(["shm", "-d"])
    assert run(["shm", "-l"]).stdout == b""
    for _ in range(200):                                    # the keeper is gone and took its descriptor with it
        try:
            os.kill(keeper, 0)
        except ProcessLookupError:
            break
        time.sleep(0.05)
    else:
        raise AssertionError("keeper %d still alive" % keeper)
    assert not [f for f in os.listdir(str(tmp_path)) if f.endswith(".resident")]
    r = run(["mem"] + args)                                 # no keeper: the usual load
    assert r.returncode == 0 and b"resident" not in r.stderr and md5(strip_pg(r.stdout)) == want


def test_resident_index_emulated(built, data, tmp_path):
    _flow(CUSIMBIN, data, tmp_path, 40)


@pytest.mark.gpu
def test_resident_index_gpu(data, tmp_path):
    _flow(bwa_b200.CLI_PATH, data, tmp_path, 2000)
