"""Device decoder (arithmetic decoder + predictor, unmodeled chunk reader, PCOMP post-processor):
blocks written by the REFERENCE and by our compressor are restored bit-exactly."""
import numpy as np
import pytest

from zpaqfranz_b200 import corpus

pytestmark = pytest.mark.gpu

UNITS = [b"", b"a", b"abcabcabcabcabc" * 10, bytes(3000), corpus.text_unit(1, 20000), corpus.random_unit(2, 3000),
         corpus.repeats_unit(3, 30000), corpus.text_unit(4, 65536), corpus.mixed_unit(6, 9000), bytes(70000)]


def _pack(blobs):
    lens = np.array([len(b) for b in blobs], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens.astype(np.uint64))[:-1]]).astype(np.uint64)
    return np.frombuffer(b"".join(blobs) + b"\0", dtype=np.uint8), offs, lens


def _reference_blocks(ctx, ref, units, method, filename, comment, dosha1=True):
    """The blocks the reference writes for `units`: made by the device compressor, each one checked equal to the
    reference's (whose recorded answer for a large block is its digest, not its bytes)."""
    arena, offs, lens = _pack(units)
    out, ooff, olen = ctx.compress_blocks(arena, offs, lens, method=method, filename=filename, comment=comment, dosha1=dosha1)
    blocks = [out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() for i in range(len(units))]
    for i, u in enumerate(units):
        assert blocks[i] == ref.compress_block(u, method, filename, comment, dosha1=dosha1), (method, i, len(u))
    return blocks


@pytest.mark.parametrize("method", ["0", "1", "2", "3", "36,200,1", "4", "46,200,1", "1,128,2", "3,200,3", "x0,4", "x0,7ci1",
                                     "x0,2,12,0,7,21,1c0,0,511i2", "x0,0c0,0,255i2,13m8,24s", "x0,6,12,0,7,21,1c0,0,511i2"])
def test_decode_reference_blocks(ctx, ref, method):
    blocks = _reference_blocks(ctx, ref, UNITS, method, "name", "jDC\x01")
    arena, offs, lens = _pack(blocks)
    out, ooff, olen = ctx.decompress_blocks(arena, offs, lens)
    for i, u in enumerate(UNITS):
        got = out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes()
        assert got == u, (method, i, len(u), len(got))


def test_decode_m5_and_no_checksum(ctx, ref):
    units = UNITS[:7]
    for method, sha in (("5", True), ("2", False), ("4", False)):
        blocks = _reference_blocks(ctx, ref, units, method, "", "c", dosha1=sha)
        arena, offs, lens = _pack(blocks)
        out, ooff, olen = ctx.decompress_blocks(arena, offs, lens, expect_len=[len(u) for u in units])
        for i, u in enumerate(units):
            assert out[int(ooff[i]): int(ooff[i]) + int(olen[i])].tobytes() == u, (method, i)


def test_gpu_round_trip(ctx):
    units = [corpus.mixed_unit(s, 40000 + 1000 * s) for s in range(8)]
    lens = np.array([len(u) for u in units], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens.astype(np.uint64))[:-1]]).astype(np.uint64)
    arena = np.frombuffer(b"".join(units) + b"\0", dtype=np.uint8)
    for method in ("2", "3", "4", "1"):
        comp, coff, clen = ctx.compress_blocks(arena, offs, lens, method=method, filename="", comment="jDC\x01")
        out, ooff, olen = ctx.decompress_blocks(comp, coff, clen)
        assert out[: int(ooff[-1]) + int(olen[-1])].tobytes() == b"".join(units), method


def test_corruption_is_detected(ctx, ref, zq):
    blk = bytearray(_reference_blocks(ctx, ref, [corpus.text_unit(1, 20000)], "3", "", "jDC\x01")[0])
    blk[len(blk) // 2] ^= 0x5A
    arena, offs, lens = _pack([bytes(blk)])
    with pytest.raises(zq.ZqError):
        ctx.decompress_blocks(arena, offs, lens)
