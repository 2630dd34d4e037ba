"""Host-side planning (method expansion, makeConfig, ZPAQL assembler) against the reference itself.
Reference: compressBlock level table Z:20289-20390, makeConfig Z:19615, Compiler Z:15904."""
import pytest

from zpaqfranz_b200 import corpus

EXPLICIT = [
    "x0,0", "x0,1,4,0,7,21,1", "x0,1,5,0,3,20", "x0,2,12,0,7,21,1c0,0,511i2", "x0,3ci1", "x0,0ci1,1,1,1,2am",
    "x0,0ci1,1,1,1,2awm",
    "x0,0w1i1c256ci1,1,1,1,1,1,2ac0,2,0,255i1c0,3,0,0,255i1c0,4,0,0,0,255i1mm16ts19t0",
    "x0,5,4,0,3,20", "x0,6,12,0,7,21,1c0,0,511i2", "x0,7ci1", "x0,4", "x6,3ci1", "x6,7ci1", "x5,1,4,0,7,26,1",
    "x8,1,4,0,7,29,1", "x8,5,4,0,7,29,1",
    "x0,0w2c0,1010,255i1c256ci1,1,1,1,1,1,2ac0,0,1019,255i1c0,20i1c0,2,0,255i1c0,3,0,0,255i1c0,4,0,0,0,255i1mm16ts19t0",
    "00,0", "x4,2,5,0,7,251c0,0,511", "s4,0,0c0,0,255,255i3", "x0,0c0,7i1c1004,0,1256i1s8,32,255",
    "x1,0c2,1100,255,0,128,300,511,1001,1300a24,1,1t16,20", "x0,0c0,0,255i2,13m8,24s", "x2,3w3,97,26,223,20,1i1,2a",
]


@pytest.mark.parametrize("method", EXPLICIT)
def test_explicit_method_bytes_match_reference(zq, ref, method):
    cfg, args = ref.make_config(method)
    hdr, pc = ref.compile(cfg, args)
    p = zq.plan_block(method)
    assert p["args"] == args
    assert p["header"] == hdr
    assert p["pcomp"] == pc


SUFFIXES = ["", ",0,0", ",5,0", ",7,1", ",10,0", ",11,0", ",15,2", ",30,1", ",50,2", ",100,3", ",160,0", ",200,1",
            ",240,0", ",250,0", ",255,3"]


@pytest.mark.parametrize("level", "012345")
def test_digit_method_headers_match_reference(zq, ref, level):
    data = corpus.text_unit(1, 3000)
    for blk_digit in ("", "4", "6"):
        for sfx in SUFFIXES:
            m = level + blk_digit + sfx
            assert zq.plan_block(m, data)["header"] == ref.block_header(data, m, "f", "c"), m


def test_level5_period_analysis_matches_reference(zq, ref):
    # periodic data makes compressBlock add "c0,0,999+P,255i1[c0,Pi1]" models (Z:20367-20387)
    for period, reps in ((37, 300), (300, 60)):
        data = corpus.random_unit(period, period) * reps
        p = zq.plan_block("5", data)
        assert "c0,0,%d,255i1" % (999 + period) in p["method"]
        assert p["header"] == ref.block_header(data, "5", "", "")


def test_bad_methods_raise(zq):
    for m in ("q", "x0,1,2,0,3,20"):  # unknown type letter; LZ77 min match too small is a runtime error later
        try:
            zq.plan_block(m)
        except zq.ZqError:
            continue
        if m == "q":
            raise AssertionError("expected an error for method %r" % m)


def test_file_sort_key(zq):
    # extension bytes (case folded, 5 at most, reset by every '/' and '.'), then descending size in 16 KiB steps
    top = (1 << 24) - 1
    assert zq.file_sort_key("/a/b.txt", 100) == (ord("t") << 56) + (ord("x") << 48) + (ord("t") << 40) + top
    assert zq.file_sort_key("/a/b.TXT", 100) == zq.file_sort_key("/x.y/c.txt", 16383)
    assert zq.file_sort_key("/a/noext", 5 << 14) == top - 5
    assert zq.file_sort_key("/a/b.tar.gz", 0) == (ord("g") << 56) + (ord("z") << 48) + top
    assert zq.file_sort_key("/a/b.jpegxy", 1 << 40) == sum(ord(c) << s for c, s in zip("jpegx", (56, 48, 40, 32, 24)))
