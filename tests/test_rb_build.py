"""rb_build on the GPU (SURVEY.md §8(f) row 4): the files it writes must be byte-identical to the
unmodified reference rb_build's, and an index opened straight from the raw inputs must answer like one
opened from the serialized files.

CPU part: the sdsl serialization writers alone (decode the committed .rbwt/.tsa/.mab, write them again).
GPU part: raw .bwt/.ssa/.esa/.ma (tests/golden/raw, made by the reference's pfbwt-f64 / mps_to_ma) through
the run-length kernels, the sample sort and the writers."""
import filecmp
import os
import subprocess

import numpy as np
import pytest

from conftest import GOLDEN, ROOT, read_fastx

import rowbowt_b200 as rb

RB_BUILD = os.path.join(ROOT, "rowbowt_b200", "rb_build")
RAW = os.path.join(GOLDEN, "raw", "tiny")
TINY = os.path.join(GOLDEN, "tiny", "tiny")


def _data_prefixes():
    out = [("toy/small.fa", 7), ("tiny/tiny", 7), ("greedy/ref.fa", 3)]
    return out


@pytest.mark.parametrize("pre,parts", _data_prefixes())
def test_writers_reproduce_reference_files(tmp_path, pre, parts):
    """sdsl_writer.hpp: sd_vector (+ both select_support_mcl, slow and fast construction), wt_huff (+ rank_support_v,
    tree), int_vector -- the reference's files come out byte for byte from their decoded contents."""
    src = os.path.join(GOLDEN, pre)
    out = str(tmp_path / "o")
    assert rb.lib().rbg_selftest_rewrite(src.encode(), out.encode(), parts) == 0
    for bit, suf in ((1, ".rbwt"), (2, ".tsa"), (4, ".mab")):
        if parts & bit:
            assert filecmp.cmp(src + suf, out + suf, shallow=False), suf


@pytest.mark.parametrize("cfg", ["small", "medium", "c2"])
def test_writers_reproduce_benchmark_index_files(tmp_path, cfg):
    """Same on the benchmark indexes when they are present (bit vectors beyond 100000 bits take
    select_support_mcl's init_fast path, long superblocks included)."""
    src = os.path.join(ROOT, "data", cfg, cfg)
    if not os.path.exists(src + ".rbwt"):
        pytest.skip("data/%s not built" % cfg)
    if cfg == "c2" and not os.environ.get("RBG_TEST_C2_REWRITE"):
        pytest.skip("rewriting the c2 index takes about a minute; set RBG_TEST_C2_REWRITE=1")
    out = str(tmp_path / "o")
    assert rb.lib().rbg_selftest_rewrite(src.encode(), out.encode(), 7) == 0
    for suf in (".rbwt", ".tsa", ".mab"):
        assert filecmp.cmp(src + suf, out + suf, shallow=False), suf


def test_raw_inputs_without_the_reference_equal_pfbwt_output(tmp_path):
    """tools/synth.write_raw_index (what bench.py and the full-size tests build their index from when data/ is empty)
    writes the reference pfbwt-f64 / mps_to_ma files of the `tiny` panel byte for byte."""
    from tools import synth
    pre = str(tmp_path / "tiny")
    synth.write_raw_index(synth.make_panel(*synth.CONFIGS["tiny"]), pre, markers=True)
    for suf in (".bwt", ".ssa", ".esa", ".ma"):
        assert filecmp.cmp(RAW + suf, pre + suf, shallow=False), suf
    assert filecmp.cmp(TINY + ".docs", pre + ".docs", shallow=False)


@pytest.mark.gpu
def test_build_index_is_byte_identical_to_reference(tmp_path):
    out = str(tmp_path / "b")
    st = rb.build_index(RAW, out, sa=True, markers=True)
    assert st.n == os.path.getsize(RAW + ".bwt") and st.r > 0
    for suf in (".rbwt", ".tsa", ".mab"):
        assert filecmp.cmp(TINY + suf, out + suf, shallow=False), suf


@pytest.mark.gpu
def test_rb_build_binary(tmp_path):
    """Host driver with the reference's command line: -s -m -l -f, then --ftab-only."""
    out = str(tmp_path / "t")
    cmd = [RB_BUILD, "-s", "-m", "-f", "-k", "6", "-o", out, RAW]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    for suf in (".rbwt", ".tsa", ".mab"):
        assert filecmp.cmp(TINY + suf, out + suf, shallow=False), suf
    # the ftab of the built index equals the one made from the serialized index
    ix = rb.GpuIndex.open(TINY)
    ix.build_ftab(6)
    ref_ftab = str(tmp_path / "ref.ftab")
    ix.save_ftab(ref_ftab)
    ix.close()
    assert filecmp.cmp(ref_ftab, out + ".ftab", shallow=False)
    os.remove(out + ".ftab")
    p = subprocess.run([RB_BUILD, "--ftab-only", "-k", "6", "-o", out, RAW], capture_output=True, text=True)
    assert p.returncode == 0 and "loading rbwt file" in p.stderr
    assert filecmp.cmp(ref_ftab, out + ".ftab", shallow=False)
    p = subprocess.run([RB_BUILD, "-s", "-o", out, str(tmp_path / "missing")], capture_output=True, text=True)
    assert p.returncode == 1


@pytest.mark.gpu
def test_open_raw_answers_like_open(tmp_path):
    _, seqs = read_fastx(os.path.join(GOLDEN, "tiny", "noisy.fq"))
    _, more = read_fastx(os.path.join(GOLDEN, "tiny", "marked.fq"))
    seqs += more
    a = rb.GpuIndex.open(TINY, sa=True, markers=True)
    b = rb.GpuIndex.open_raw(RAW, sa=True, markers=True)
    ia, ib = a.info(), b.info()
    assert (ia.n, ia.r, ia.toehold0, list(ia.F)) == (ib.n, ib.r, ib.toehold0, list(ib.F))
    mode = rb.RBG_LOCATE | rb.RBG_MARKERS
    ra, rb_ = a.query(seqs, mode), b.query(seqs, mode)
    for f in ("lo", "hi", "toehold", "loc_off", "locs", "mk_off", "markers"):
        assert np.array_equal(getattr(ra, f), getattr(rb_, f)), f
    a.close()
    b.close()


@pytest.mark.gpu
def test_rle_kernels_on_adversarial_bwt(tmp_path):
    """Run boundaries at every alignment (16-byte vectors, 32 KB tiles, 64 MB chunks are internal): random run
    lengths from 1 to 70000, the zero terminator, a file length that is not a multiple of 16."""
    rng = np.random.default_rng(11)
    lens = np.concatenate([rng.integers(1, 4, 5000), rng.integers(1, 70000, 60), rng.integers(1, 40, 3000), [1, 1, 1, 15, 16, 17]])
    heads = rng.choice(np.frombuffer(b"ACGT", np.uint8), len(lens))
    for j in range(1, len(heads)):                     # adjacent runs must differ
        if heads[j] == heads[j - 1]:
            heads[j] = b"ACGT"[(b"ACGT".index(heads[j]) + 1) % 4]
    heads[len(heads) // 2] = 0                          # the terminator, stored as byte 0 in the file
    lens[len(heads) // 2] = 1
    bwt = np.repeat(heads, lens)
    pre = str(tmp_path / "adv")
    bwt.tofile(pre + ".bwt")
    out = str(tmp_path / "adv_out")
    st = rb.build_index(pre, out)
    assert (st.n, st.r) == (len(bwt), len(lens))
    from oracle import rbformats
    got = rbformats.read_rbwt(out + ".rbwt")
    exp_heads = heads.copy()
    exp_heads[exp_heads == 0] = 1
    assert np.array_equal(got.heads, exp_heads) and np.array_equal(got.lens, lens.astype(np.uint64))
    if os.path.exists(os.path.join(ROOT, "oracle", "_ref", "rb_build")):
        ref = str(tmp_path / "adv_ref")
        subprocess.run([os.path.join(ROOT, "oracle", "_ref", "rb_build"), "-o", ref, pre], check=True, capture_output=True)
        assert filecmp.cmp(ref + ".rbwt", out + ".rbwt", shallow=False)
    bad = str(tmp_path / "ws")
    np.frombuffer(b"ACGT ACGT\n", np.uint8).tofile(bad + ".bwt")
    with pytest.raises(rb.RbgError) as e:
        rb.build_index(bad, out)
    assert e.value.code == -3
