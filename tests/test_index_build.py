"""bwa_b200/index_build.py (input preparation for 3 Gbp benchmark references, where `bwa index` needs hours) against the
reference's `bwa index`, byte for byte, on small adversarial references: texts whose fwd+revcomp ends in runs of A (a
reference starting with T's), so that several suffixes shorter than the 32-base sort key have identical zero-padded
keys and only their lengths order them; periodic and single-base texts (deep tie refinement)."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from conftest import md5, ref_run

CASES = {
    "tt": "TT", "ttt": "TTT", "ttc": "TTC", "t40": "T" * 40, "aa_tail": "", "period": "", "polyA": "",
}


def _ref(name, rng):
    body = "".join("ACGT"[i] for i in rng.integers(0, 4, 3000))
    if name in ("tt", "ttt", "ttc", "t40"):
        return CASES[name] + body
    if name == "aa_tail":
        return "TTTT" + body + "AAAAAA"
    if name == "period":
        return "TTAGGG" * 300 + body[:500] + "TTAGGG" * 40
    return "A" * 700


def _build_both(tmp_path, name, device):
    import bwa_b200.index_build as ib
    import zlib
    rng = np.random.default_rng(zlib.crc32(name.encode()) % 1000)
    seq = _ref(name, rng)
    fa = str(tmp_path / (name + ".fa"))
    with open(fa, "w") as f:
        f.write(">c1\n%s\n>c2 second contig\n%s\n" % (seq, seq[::-1][:800] if len(seq) > 900 else "ACGTTTGACA" * 7))
    mine = str(tmp_path / (name + "_mine.fa"))
    shutil.copy(fa, mine)
    exts = ("pac", "ann", "amb", "bwt", "sa")
    want = ref_run("bwa", ["index", fa], "raw", outputs=[fa + "." + e for e in exts])["files"]
    recs = ib.read_fasta(mine)
    codes = ib.pack_reference(recs, mine)
    ib.build_from_codes(codes, mine, device=device, verbose=False)
    for ext in exts:
        assert md5(open(mine + "." + ext, "rb").read()) == want[name + ".fa." + ext], (name, ext)


@pytest.mark.parametrize("name", sorted(CASES))
def test_index_builder_cpu_identical_to_bwa_index(built, tmp_path, name):
    _build_both(tmp_path, name, "cpu")


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CASES))
def test_index_builder_gpu_identical_to_bwa_index(tmp_path, name):
    _build_both(tmp_path, name, "cuda")


def _verify(lib_path, data, tmp_path):
    """bwag_ctx_verify: a complete check of the resident BWT / suffix array against the resident text; must pass on an index of
    `bwa index` and on the GPU builder's, and must notice a single flipped BWT symbol or a shifted suffix-array sample."""
    import ctypes as C
    import bwa_b200
    L = C.CDLL(lib_path, mode=C.RTLD_LOCAL) if lib_path else bwa_b200.lib()
    L.bwa_idx_load.restype = C.POINTER(bwa_b200.BwaIdx)
    L.bwa_idx_load.argtypes = [C.c_char_p, C.c_int]
    L.bwag_ctx_create.restype = C.c_void_p
    L.bwag_ctx_create.argtypes = [C.c_int, C.c_void_p, C.c_int64, C.c_void_p]
    L.bwag_ctx_verify.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
    L.bwag_ctx_destroy.argtypes = [C.c_void_p]
    L.bwag_ctx_densify_sa.argtypes = [C.c_void_p, C.c_int]
    fa = data.ref("two")

    def run(prefix, dense):
        idx = L.bwa_idx_load(prefix.encode(), 7).contents
        l_pac = C.cast(idx.bns, C.POINTER(C.c_int64))[0]
        ctx = L.bwag_ctx_create(-1, idx.bwt, l_pac, idx.pac)
        assert ctx
        if dense:
            assert L.bwag_ctx_densify_sa(ctx, 4) == 0
        out = (C.c_uint64 * 4)()
        assert L.bwag_ctx_verify(ctx, 0, 1, out) == 0
        L.bwag_ctx_destroy(ctx)
        return list(out), 2 * l_pac + 1

    good, rows = run(fa, True)
    assert good == [rows, 0, 0, 0]
    bad = str(tmp_path / "bad.fa")
    for ext in ("amb", "ann", "pac", "sa"):
        shutil.copy(fa + "." + ext, bad + "." + ext)
    raw = bytearray(open(fa + ".bwt", "rb").read())
    raw[40 + 64 * 500 + 37] ^= 0x30                   # one symbol of the 500th Occ block
    open(bad + ".bwt", "wb").write(raw)
    res, _ = run(bad, False)
    assert res[1] + res[2] > 0
    shutil.copy(fa + ".bwt", bad + ".bwt")
    raw = bytearray(open(fa + ".sa", "rb").read())
    raw[56 + 8 * 1000] ^= 0x04                        # one suffix-array sample off by 4
    open(bad + ".sa", "wb").write(raw)
    res, _ = run(bad, False)
    assert res[1] + res[2] > 0


def test_index_verification_emulated(built, data, tmp_path):
    from conftest import ROOT
    _verify(os.path.join(ROOT, "tests/_build/libbwa_b200_cusim.so"), data, tmp_path)


@pytest.mark.gpu
def test_index_verification_gpu(data, tmp_path):
    _verify(None, data, tmp_path)
