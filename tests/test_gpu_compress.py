"""Parity of the CUDA block compressor (through the C ABI) with the oracle and the reference."""
import numpy as np
import pytest

from zpaqfranz_b200 import corpus

pytestmark = pytest.mark.gpu


def _arena(units):
    lens = np.array([len(u) for u in units], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens.astype(np.uint64))[:-1]]).astype(np.uint64)
    arena = np.frombuffer(b"".join(units) + b"\0", dtype=np.uint8)
    return arena, offs, lens


EDGE_UNITS = [
    b"", b"a", b"ab", b"abc", b"abcd", b"aaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaaa", bytes(5), bytes(4097), bytes(65536),
    bytes([255]) * 70000, b"abcabcabcabcabc" * 10, bytes([0, 0, 1, 0, 0, 0, 1, 0]) * 500,
    corpus.text_unit(1, 65536), corpus.text_unit(2, 65535), corpus.text_unit(3, 65537), corpus.random_unit(4, 20000),
    corpus.repeats_unit(5, 65536), corpus.text_unit(6, 1000), corpus.text_unit(7, 200000), corpus.repeats_unit(8, 300000),
    (corpus.text_unit(9, 30000) * 3), corpus.random_unit(10, 70000) + corpus.random_unit(10, 70000),
]


def test_sha1_many(ctx, oracle):
    arena, offs, lens = _arena(EDGE_UNITS + [corpus.random_unit(s, 1 + 61 * s) for s in range(40)])
    # unaligned starts on purpose: shift the arena by 1..3 bytes
    for shift in (0, 1, 3):
        a2 = np.concatenate([np.zeros(shift, np.uint8), arena])
        dg = ctx.sha1(a2, offs + np.uint64(shift), lens)
        for i in range(len(offs)):
            o, l = int(offs[i]), int(lens[i])
            assert dg[i].tobytes() == oracle.sha1(arena[o:o + l].tobytes()), (shift, i)


def test_suffix_array_matches_oracle(ctx, oracle):
    for u in EDGE_UNITS:
        if not u:
            continue
        sa = ctx.suffix_array(u)
        assert (sa == oracle.suffix_array(u)).all(), len(u)


def _skewed(seed, k, n):
    """n bytes over k byte values, Zipf-like (the shared-memory suffix sort packs them into 1..8 bits per character)"""
    rng = np.random.default_rng(seed)
    vals = rng.choice(256, size=k, replace=False)
    p = 1.0 / np.arange(1, k + 1) ** 1.2
    return vals[rng.choice(k, size=n, p=p / p.sum())].astype(np.uint8).tobytes()


def test_small_alphabets_bit_exact(ctx, ref):
    """k_suffix_sort16's dense form at every character width: blocks over 2 .. 256 byte values, -m2 against the reference."""
    units = [_skewed(10 + k, k, n) for k, n in ((2, 30000), (3, 65536), (5, 50000), (9, 65536), (17, 65536), (33, 40000), (65, 65536),
                                                (129, 65536), (200, 65535), (256, 65536))]
    units += [corpus.text_unit(31, 40000) + corpus.random_unit(31, 25536), bytes(range(256)) * 256]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method="2", filename="", comment="jDC\x01")
    for i, u in enumerate(units):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        assert got == ref.compress_block(u, "2", "", "jDC\x01"), (i, len(u))


@pytest.mark.parametrize("method", ["2", "0", "26,200,1", "x0,0", "x0,1,4,0,7,21,1", "x0,1,4,0,7,21,0", "x0,1,6,0,5,21,2",
                                     "x0,1,4,0,4,21,1"])
def test_unmodeled_blocks_bit_exact(ctx, zq, oracle, ref, method):
    arena, offs, lens = _arena(EDGE_UNITS)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename="nm", comment="jDC\x01")
    for i, u in enumerate(EDGE_UNITS):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        p = zq.plan_block(method, u)
        s = oracle.lz_stream(u, p["args"]) if (p["args"][1] & 3) else u
        want = oracle.block_unmodeled(p["header"], p["pcomp"], b"nm", ("%d jDC\x01" % len(u)).encode(), s, oracle.sha1(u))
        assert got == want, (method, i, len(u))
        assert got == ref.compress_block(u, method, "nm", "jDC\x01"), (method, i, len(u))
    # the concatenation is a valid archive stream: the reference decoder restores every unit
    total = int(ooff[-1]) + int(olen[-1])
    assert ref.decompress(out[:total].tobytes(), int(lens.sum())) == b"".join(EDGE_UNITS)


def test_per_unit_methods_and_names(ctx, ref):
    units = [corpus.text_unit(s, 20000 + 1000 * s) for s in range(6)]
    methods = ["2", "0", "x0,0", "2", "26,200,1", "x0,1,4,0,7,21,1"]
    names = ["f%d" % i for i in range(6)]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=methods, filename=names, comment=["c"] * 6, dosha1=False)
    for i, u in enumerate(units):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        assert got == ref.compress_block(u, methods[i], names[i], "c", dosha1=False), i


def test_batch_of_text_units_m2(ctx, ref):
    n = 296
    arena = corpus.text_corpus(n)
    offs = np.arange(n, dtype=np.uint64) * 65536
    lens = np.full(n, 65536, dtype=np.uint32)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method="2", filename="", comment="")
    for i in list(range(0, n, 37)) + [n - 1]:
        u = arena[i * 65536:(i + 1) * 65536].tobytes()
        assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, "2", "", ""), i
    total = int(ooff[-1]) + int(olen[-1])
    assert ref.decompress(out[:total].tobytes(), n * 65536) == arena.tobytes()


CM_UNITS = [
    b"", b"a", b"abcabcabcabcabc" * 10, bytes(3000), corpus.text_unit(1, 20000), corpus.random_unit(2, 3000),
    corpus.repeats_unit(3, 30000), corpus.text_unit(4, 65536), corpus.mixed_unit(6, 9000),
]


@pytest.mark.parametrize("method", ["3", "36,200,1", "4", "46,200,1", "5", "56,180,1", "3,100,0", "4,30,0",
                                     "x0,0c0,0,255i2,13m8,24s", "x0,0c0,7i1c1004,0,1256i1s8,32,255",
                                     "x0,0c2,1100,255,0,128a24,1,1t16,20", "s0,0c0,0,255,255i3", "x0,3ci1",
                                     "x0,0c8,0,255c0,0,255,255a16,2,2t8", "x0,2,12,0,7,21,1c0,0,511i2"])
def test_modeled_blocks_bit_exact(ctx, zq, oracle, ref, method):
    units = CM_UNITS if method not in ("5", "56,180,1") else CM_UNITS[:7]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename="nm", comment="jDC\x01")
    for i, u in enumerate(units):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        want = ref.compress_block(u, method, "nm", "jDC\x01")
        if got != want:
            k = next((j for j in range(min(len(got), len(want))) if got[j] != want[j]), -1) if isinstance(want, bytes) else -1
            raise AssertionError("method %s unit %d (n=%d): %d vs %d bytes, first difference at %d" %
                                 (method, i, len(u), len(got), len(want), k))
    total = int(ooff[-1]) + int(olen[-1])
    assert ref.decompress(out[:total].tobytes(), int(lens.sum())) == b"".join(units)


@pytest.mark.parametrize("jit", ["0", "1", "2"])
def test_context_program_forms_over_several_waves(zq, ref, monkeypatch, jit):
    # the three forms of the context machine / coder -- ZPAQL interpreter on its own warp (ZQ_CM_JIT=0), HCOMP translated
    # to CUDA C and compiled with NVRTC (=1, the default), generated straight-line coder as well (=2) -- with the work
    # arena cut so small that the batch runs in several waves (the per-wave bookkeeping of the translated path)
    monkeypatch.setenv("ZQ_CM_JIT", jit)
    monkeypatch.setenv("ZQ_MODEL_BUDGET", str(3 << 20))     # ~2 blocks of -m3 per wave
    units = [corpus.text_unit(40 + k, 9000 + 700 * k) for k in range(7)] + [corpus.mixed_unit(9, 8000), b"abc" * 900]
    arena, offs, lens = _arena(units)
    with zq.Context(0) as c2:
        for method in ("3", "36,200,1", "4"):
            out, ooff, olen = c2.compress_blocks(arena, offs, lens, method=method, filename="", comment="")
            for i, u in enumerate(units):
                assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, method, "", ""), (jit, method, i)


def test_modeled_matches_c_oracle(ctx, zq, oracle):
    u = corpus.text_unit(11, 12000)
    arena, offs, lens = _arena([u])
    for method in ("3", "4", "36,200,1"):
        out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename="", comment="")
        p = zq.plan_block(method, u)
        s = oracle.lz_stream(u, p["args"]) if (p["args"][1] & 3) else u
        want = oracle.block_modeled(p["header"], p["pcomp"], b"", b"%d " % len(u), s, oracle.sha1(u))
        assert out[: int(olen[0])].tobytes() == want, method


def _exe_like(seed, n):
    """bytes with many E8/E9 xx xx xx 00/FF patterns so that the E8E9 filter has work to do"""
    rng = np.random.Generator(np.random.PCG64([seed, 5]))
    a = rng.integers(0, 256, n, dtype=np.uint8)
    for pos in rng.integers(0, max(n - 8, 1), n // 24):
        a[pos] = 0xE8 + int(rng.integers(0, 2))
        a[pos + 4] = 0x00 if rng.integers(0, 2) else 0xFF
    return a.tobytes()


HASH_METHODS = ["1", "1,10,0", "1,20,0", "1,40,0", "1,250,0", "2,10,0", "3,10,0", "4,5,0", "14,128,0", "x0,1,4,0,3,20",
                "x0,1,5,0,3,20", "x0,2,6,0,2,18", "x0,2,12,0,5,16", "x0,1,4,0,6,20", "x0,1,4,4,3,20,1", "x0,2,5,7,2,19"]


@pytest.mark.parametrize("method", HASH_METHODS)
def test_hash_lz77_blocks_bit_exact(ctx, ref, method):
    units = EDGE_UNITS[:12] + [corpus.text_unit(1, 65536), corpus.random_unit(4, 20000), corpus.repeats_unit(5, 65536),
                               corpus.text_unit(7, 200000), bytes(1 << 20)]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename="nm", comment="c")
    for i, u in enumerate(units):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        assert got == ref.compress_block(u, method, "nm", "c"), (method, i, len(u))


@pytest.mark.parametrize("method", ["1,128,2", "2,128,2", "3,100,2", "3,200,3", "4,128,2", "0", "x0,4", "x0,5,4,0,3,20",
                                     "x0,6,12,0,7,21,1c0,0,511i2", "x0,7ci1", "x0,4c0,0,255i1"])
def test_e8e9_blocks_bit_exact(ctx, ref, method):
    units = [_exe_like(1, 30000), _exe_like(2, 65536), _exe_like(3, 7), _exe_like(4, 5), b"\xe8\x01\x02\x03\x00" * 30,
             corpus.text_unit(1, 5000), b""]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena.copy(), offs, lens, method=method, filename="x", comment="")
    for i, u in enumerate(units):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        assert got == ref.compress_block(u, method, "x", ""), (method, i, len(u))
    total = int(ooff[-1]) + int(olen[-1])
    assert ref.decompress(out[:total].tobytes(), int(lens.sum())) == b"".join(units)


def test_config1_one_mib_of_zeros_m1(ctx, ref):
    # BASELINE.json configs[0]: single 1 MiB zero-filled buffer, -m1, byte-compare with the reference
    u = bytes(1 << 20)
    arena, offs, lens = _arena([u])
    for m in ("1", "14,0,0"):
        out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=m, filename="", comment="")
        assert out[: int(olen[0])].tobytes() == ref.compress_block(u, m, "", "")


def test_general_parser_is_bit_exact(zq, ref, monkeypatch):
    # the warp-per-block form of the SA parse (k_lz77_sa): serves methods the scan pipeline does not cover (bucket > 127,
    # look-ahead > 1) and, with ZQ_LZ_OLD=1, every block -- same bytes either way
    monkeypatch.setenv("ZQ_LZ_OLD", "1")
    units = EDGE_UNITS[3:] + [corpus.text_unit(21, 65536), corpus.repeats_unit(22, 65536)]
    arena, offs, lens = _arena(units)
    with zq.Context(0) as c2:
        for method in ("2", "x0,2,12,0,7,21,1", "x0,1,4,0,5,21,2"):
            out, ooff, olen = c2.compress_blocks(arena, offs, lens, method=method, filename="", comment="")
            for i, u in enumerate(units):
                assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, method, "", ""), (method, i)


def test_scan_pipeline_shapes(ctx, ref):
    # the position-parallel parse (k_lz_scan -> k_lz_walk -> k_lz_emit) across its code paths: several tiles per block,
    # 16- and 32-bit indices, look-ahead 0 and 1, both code formats, capped LCPs (exact slow path in the walk), streams
    # assembled in shared memory (<= 64 KiB blocks) and in global memory (larger), plus a method it hands to k_lz77_sa
    units = [corpus.text_unit(31, 65536), corpus.text_unit(32, 70001), corpus.repeats_unit(33, 65536), bytes(66000),
             corpus.random_unit(34, 40000), corpus.mixed_unit(6, 100000), b"ab" * 3000 + b"c" + b"ab" * 3000,
             corpus.text_unit(35, 4096), corpus.text_unit(36, 4097), corpus.text_unit(37, 8191), b"", b"x", bytes(range(256)) * 300]
    arena, offs, lens = _arena(units)
    for method in ("2", "x0,2,12,0,7,21,1", "x0,1,4,0,3,21,0", "x0,2,5,0,6,21,1", "x0,1,6,0,7,21,1", "x0,1,4,0,8,21,1", "x0,1,4,0,5,21,2"):
        out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename="", comment="")
        for i, u in enumerate(units):
            assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, method, "", ""), (method, i)


def test_level5_period_models_on_device(ctx, zq, ref):
    # byte-gap analysis (Z:20355-20388) runs on the device: periodic data adds "c0,0,999+P,255i1[c0,Pi1]" models
    units = [corpus.random_unit(37, 37) * 300, corpus.random_unit(300, 300) * 60, corpus.text_unit(3, 9000), bytes(5000)]
    arena, offs, lens = _arena(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method="5", filename="p", comment="")
    for i, u in enumerate(units):
        assert "c0,0,%d" % (999 + 37) in zq.plan_block("5", units[0])["method"]
        assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, "5", "p", ""), i
    # text + two periodic models = 33 components, one more than a warp has lanes: coded by one lane component by
    # component (zq_cm_wide.cuh), bit-exact, and the device decoder restores it; mixed in a batch with ordinary blocks
    wide = [(corpus.random_unit(41, 41) * 200)[:8000], b"".join(b"%06d,abcde,%08d,xyzxyz\n" % (i, i * 7) for i in range(400)),
            corpus.text_unit(5, 6000), b""]
    assert zq.plan_block("56,180,1", wide[0])["header"][6] == 33 and zq.plan_block("56,180,1", wide[1])["header"][6] == 33
    a2, o2, l2 = _arena(wide)
    out, ooff, olen = ctx.compress_blocks(a2, o2, l2, method="56,180,1", filename="w", comment="")
    for i, u in enumerate(wide):
        assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == ref.compress_block(u, "56,180,1", "w", ""), i
    dec, doff, dlen = ctx.decompress_blocks(out, ooff, olen, expect_len=l2)
    for i, u in enumerate(wide):
        assert dec[int(doff[i]): int(doff[i]) + int(dlen[i])].tobytes() == u, i
    # beyond 64 components there is no device path: reported loudly (never a CPU fallback)
    comps = " ".join("%d cm 8 16" % i for i in range(65))
    cfg = "comp 0 0 0 0 66 " + comps + " 65 mix 0 0 65 24 0 hcomp halt end"
    hdr = zq.assemble_config(cfg)["header"]
    a3, o3, l3 = _arena([b"abc" * 100])
    with pytest.raises(zq.ZqError):
        ctx.compress_segments(a3, o3, l3, hdr)


def test_unsupported_is_loud(ctx, zq):
    arena, offs, lens = _arena([corpus.text_unit(1, 5000)])
    with pytest.raises(zq.ZqError):
        ctx.compress_blocks(arena, offs, lens, method="x0,1,2,0,3,20")   # LZ77 min match too small
    with pytest.raises(zq.ZqError):
        ctx.compress_blocks(arena, offs, lens, method="q1")


def test_pipe_matches_synchronous_calls(zq, ctx):
    # batches in flight (zq_pipe_*): same bytes as the synchronous entry point, host and device pointers
    import torch
    units = [corpus.text_unit(s, 30000 + 977 * s) for s in range(24)]
    lens = np.array([len(u) for u in units], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens.astype(np.uint64))[:-1]]).astype(np.uint64)
    arena = np.frombuffer(b"".join(units) + b"\0" * 16, dtype=np.uint8).copy()
    want, woff, wlen = ctx.compress_blocks(arena, offs, lens, method="2", filename="f", comment="c")
    want = want[: int(woff[-1]) + int(wlen[-1])].tobytes()
    pipe = zq.Pipe(0, 2)
    try:
        cap = int(zq.lib.zq_compress_bound(int(lens.max()))) * len(units)
        outs = [np.empty(cap, dtype=np.uint8) for _ in range(3)]
        d_in = torch.from_numpy(arena).cuda()
        d_outs = [torch.empty(cap, dtype=torch.uint8, device="cuda") for _ in range(3)]
        t = [pipe.submit(arena.ctypes.data, offs, lens, outs[k].ctypes.data, cap, method="2", filename="f", comment="c") for k in range(3)]
        td = [pipe.submit(d_in.data_ptr(), offs, lens, d_outs[k].data_ptr(), cap, method="2", filename="f", comment="c", device=True)
              for k in range(3)]
        for k in range(3):
            ooff, olen = pipe.wait(t[k])
            assert outs[k][: int(ooff[-1]) + int(olen[-1])].tobytes() == want
        for k in range(3):
            ooff, olen = pipe.wait(td[k])
            assert d_outs[k][: int(ooff[-1]) + int(olen[-1])].cpu().numpy().tobytes() == want
        assert pipe.launch_count() > 0
    finally:
        pipe.close()
