"""Archive-level parity: the data ("d") and fragment-table ("h") blocks of an archive written by the REFERENCE's
own command line (`zpaqfranz a`, recorded by oracle_bindings.Ref.archive_d_h) are reproduced byte for byte by
zq_add_files -- the device fragmenter + SHA-1 + order-1 tables, the host dedup / type heuristics / new-block rule, and
the device block compressor.  (SURVEY §8 a15-a17, §8f rank 2.)"""
import os

import numpy as np
import pytest

import zpaqfranz_b200 as zqmod
from zpaqfranz_b200 import corpus

pytestmark = pytest.mark.gpu
TREES = {
    "small_mixed": {
        "a.txt": corpus.text_unit(1, 300000), "b.bin": corpus.random_unit(2, 100000), "sub/c.txt": corpus.text_unit(1, 300000),
        "empty.dat": b"", "z.dat": bytes(200000), "sub/deep/d.TXT": corpus.text_unit(5, 70000) + corpus.text_unit(1, 300000),
        "noext": corpus.repeats_unit(3, 50000), "e.exe": corpus.mixed_unit(9, 150000), "also_empty.dat": b"",
    },
    "many_blocks": dict(("f%02d.%s" % (i, ("txt", "bin", "dat")[i % 3]),
                         (corpus.text_unit, corpus.random_unit, corpus.repeats_unit)[i % 3](100 + i, 400000 + 37000 * i))
                        for i in range(12)),
}


@pytest.mark.parametrize("tree,flags", [("small_mixed", ["-m2"]), ("small_mixed", ["-m1"]), ("small_mixed", ["-m3"]),
                                        ("small_mixed", ["-m20", "-fragment", "4"]), ("many_blocks", ["-m10"]),
                                        ("many_blocks", ["-m21"]), ("small_mixed", ["-m4"])])
def test_d_and_h_blocks_match_the_reference_archiver(ctx, ref, tree, flags):
    src = "/archived/src"      # any common prefix: the order below depends on the paths below it only
    date14, nblocks, want_d, want_h = ref.archive_d_h(TREES[tree], flags)
    assert want_d and want_h
    # files in the reference's order: sort key, then full path (Z:121735-121754, compareFilename Z:63575)
    files = []
    for rel, data in TREES[tree].items():
        path = os.path.join(src, rel)
        files.append((zqmod.file_sort_key(path, len(data)), path, data))
    files.sort(key=lambda t: (t[0], t[1]))
    lens = np.array([len(f[2]) for f in files], dtype=np.uint64)
    offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64)
    arena = np.frombuffer(b"".join(f[2] for f in files) + b"\0", dtype=np.uint8)
    method = flags[0][2:]
    fragment = int(flags[flags.index("-fragment") + 1]) if "-fragment" in flags else 6
    got = ctx.add_files(arena, offs, lens, method=method, fragment=fragment, date14=date14)
    assert got["nblocks"] == nblocks
    assert got["d"] == want_d
    assert got["h"] == want_h
    # every file is covered by its fragment list, duplicates share ids
    names = [os.path.relpath(f[1], src) for f in files]
    ids = dict(zip(names, got["file_frags"]))
    if tree == "small_mixed":
        assert ids["a.txt"] == ids["sub/c.txt"]
        assert ids["empty.dat"] == ids["also_empty.dat"] and len(ids["empty.dat"]) == 1
