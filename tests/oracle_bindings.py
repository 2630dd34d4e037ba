"""ctypes views of the two CHECKERS under oracle/_ref/ (test infrastructure; never used by the product)."""
import base64
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_DIR = os.path.join(ROOT, "oracle", "_ref")


class Oracle:
    def __init__(self, lib):
        self.lib = lib
        lib.zqo_lz_stream.restype = C.c_longlong
        lib.zqo_block_unmodeled.restype = C.c_longlong
        lib.zqo_fragment.restype = C.c_longlong
        lib.zqo_block_modeled.restype = C.c_longlong

    def sha1(self, data):
        out = C.create_string_buffer(20)
        self.lib.zqo_sha1(bytes(data), C.c_uint64(len(data)), out)
        return out.raw

    def suffix_array(self, data):
        data = bytes(data)
        sa = np.zeros(max(len(data), 1), dtype=np.uint32)
        self.lib.zqo_suffix_array(data, sa.ctypes.data_as(C.c_void_p), C.c_uint32(len(data)))
        return sa[: len(data)]

    def lz_stream(self, data, args, sa=None, tokens=False):
        data = bytes(data)
        a = (C.c_int * 9)(*args)
        cap = len(data) + len(data) // 16 + 1024
        out = C.create_string_buffer(cap)
        tok = np.zeros(3 * (len(data) + 1), dtype=np.uint32)
        ntok = C.c_uint64(0)
        sap = sa.ctypes.data_as(C.c_void_p) if sa is not None else None
        r = self.lib.zqo_lz_stream(data, C.c_uint32(len(data)), a, sap, out, C.c_uint64(cap),
                                   tok.ctypes.data_as(C.c_void_p), C.c_uint64(tok.size), C.byref(ntok))
        if r < 0:
            raise RuntimeError("zqo_lz_stream failed %d" % r)
        if tokens:
            return out.raw[:r], tok[: 3 * ntok.value].reshape(-1, 3)
        return out.raw[:r]

    def e8e9(self, data):
        b = C.create_string_buffer(bytes(data), len(data))
        self.lib.zqo_e8e9(b, C.c_int(len(data)))
        return b.raw

    def block_unmodeled(self, header, pcomp, filename, comment_full, stream, sha1):
        cap = len(stream) + len(stream) // 1000 + len(header) + len(pcomp) + 1024
        out = C.create_string_buffer(cap)
        r = self.lib.zqo_block_unmodeled(bytes(header), C.c_uint32(len(header)), bytes(pcomp), C.c_uint32(len(pcomp)),
                                         filename, comment_full, bytes(stream), C.c_uint64(len(stream)), sha1, out,
                                         C.c_uint64(cap))
        if r < 0:
            raise RuntimeError("zqo_block_unmodeled failed %d" % r)
        return out.raw[:r]

    def block_modeled(self, header, pcomp, filename, comment_full, stream, sha1):
        cap = len(stream) + len(stream) // 8 + len(header) + len(pcomp) + 4096
        out = C.create_string_buffer(cap)
        r = self.lib.zqo_block_modeled(bytes(header), C.c_uint32(len(header)), bytes(pcomp), C.c_uint32(len(pcomp)),
                                       filename, comment_full, bytes(stream), C.c_uint64(len(stream)), sha1, out,
                                       C.c_uint64(cap))
        if r < 0:
            raise RuntimeError("zqo_block_modeled failed %d" % r)
        return out.raw[:r]

    def table_sums(self):
        a, b = C.c_uint32(0), C.c_uint32(0)
        self.lib.zqo_table_sums(C.byref(a), C.byref(b))
        return a.value, b.value

    def fragment(self, data, fragment=6, blocksize=(1 << 26) - 4096):
        data = bytes(data)
        cap = len(data) // 64 + 16
        fl = np.zeros(cap, dtype=np.uint32)
        fh = np.zeros(cap, dtype=np.uint32)
        k = self.lib.zqo_fragment(data, C.c_uint64(len(data)), C.c_int(fragment), C.c_uint32(blocksize),
                                  fl.ctypes.data_as(C.c_void_p), fh.ctypes.data_as(C.c_void_p), C.c_uint64(cap))
        return fl[:k].copy(), fh[:k].copy()


class Ref:
    """The unmodified reference (libzpaq inside zpaqfranz.cpp) behind oracle/ref_shim.cpp."""

    def __init__(self, lib):
        self.lib = lib
        for f in ("zref_compress_block", "zref_decompress", "zref_lz_stream", "zref_fragment", "zref_compress_units_mt", "zref_compress_segment"):
            getattr(lib, f).restype = C.c_longlong
        lib.zref_last_error.restype = C.c_char_p

    def compress_block(self, data, method, filename=None, comment=None, dosha1=True):
        data = bytes(data)
        cap = len(data) + len(data) // 8 + 100000
        out = C.create_string_buffer(cap)
        fn = filename.encode() if isinstance(filename, str) else filename
        cm = comment.encode() if isinstance(comment, str) else comment
        r = self.lib.zref_compress_block(data, C.c_uint(len(data)), method.encode(), fn, cm, C.c_int(1 if dosha1 else 0),
                                         out, C.c_ulonglong(cap))
        if r < 0:
            raise RuntimeError("reference compressBlock failed: %s" % self.lib.zref_last_error().decode(errors="replace"))
        return out.raw[:r]

    def compress_segment(self, data, header=None, level=0, pcomp=b"", filename=None, comment=None, sha1=None, tag=True):
        """libzpaq::Compressor driven directly: writeTag/startBlock(level | header)/startSegment/postProcess/compress/
        endSegment(sha1)/endBlock."""
        data = bytes(data)
        cap = len(data) + len(data) // 8 + 200000
        out = C.create_string_buffer(cap)
        fn = filename.encode() if isinstance(filename, str) else filename
        cm = comment.encode() if isinstance(comment, str) else comment
        r = self.lib.zref_compress_segment(C.c_int(level), bytes(header) if header else None, bytes(pcomp) if pcomp else None,
                                           C.c_int(len(pcomp)), data, C.c_uint(len(data)), fn, cm,
                                           bytes(sha1) if sha1 is not None else None, C.c_int(1 if tag else 0), out, C.c_ulonglong(cap))
        if r < 0:
            raise RuntimeError("reference Compressor failed: %s" % self.lib.zref_last_error().decode(errors="replace"))
        return out.raw[:r]

    def compress_multi(self, segments, header=None, level=0, pcomp=b"", filename="seg", comment="", sha=True):
        """One block with several segments through the reference's Compressor class."""
        import numpy as _np
        data = b"".join(bytes(x) for x in segments)
        lens = _np.array([len(x) for x in segments], dtype=_np.uint32)
        offs = (_np.cumsum(lens, dtype=_np.uint64) - lens).astype(_np.uint64)
        cap = len(data) + len(data) // 8 + 200000 + 400 * len(segments)
        out = C.create_string_buffer(cap)
        self.lib.zref_compress_multi.restype = C.c_longlong
        r = self.lib.zref_compress_multi(C.c_int(level), bytes(header) if header else None, bytes(pcomp) if pcomp else None,
                                         C.c_int(len(pcomp)), C.c_int(len(segments)), data + b"\0", offs.ctypes.data_as(C.c_void_p),
                                         lens.ctypes.data_as(C.c_void_p), filename.encode(), comment.encode(), C.c_int(1 if sha else 0),
                                         out, C.c_ulonglong(cap))
        if r < 0:
            raise RuntimeError("reference Compressor failed: %s" % self.lib.zref_last_error().decode(errors="replace"))
        return out.raw[:r]

    def decompress(self, blob, cap):
        out = C.create_string_buffer(cap + 16)
        r = self.lib.zref_decompress(bytes(blob), C.c_ulonglong(len(blob)), out, C.c_ulonglong(cap + 16))
        if r < 0:
            raise RuntimeError("reference decompress failed: %s" % self.lib.zref_last_error().decode(errors="replace"))
        return out.raw[:r]

    def _digest(self, fn, n, data):
        out = C.create_string_buffer(n)
        fn(bytes(data), C.c_ulonglong(len(data)), out)
        return out.raw

    def sha1(self, d):
        return self._digest(self.lib.zref_sha1, 20, d)

    def sha256(self, d):
        return self._digest(self.lib.zref_sha256, 32, d)

    def xxh3_128(self, d):
        return self._digest(self.lib.zref_xxh3_128, 16, d)

    def blake3(self, d):
        return self._digest(self.lib.zref_blake3, 32, d)

    def md5(self, d):
        return self._digest(self.lib.zref_md5, 16, d)

    def sha3_256(self, d):
        return self._digest(self.lib.zref_sha3_256, 32, d)

    def xxh64(self, d):
        return self._digest(self.lib.zref_xxh64, 8, d)

    def crc32(self, d):
        return self._digest(self.lib.zref_crc32, 4, d)

    def divsufsort(self, data):
        data = bytes(data)
        sa = np.zeros(max(len(data), 1), dtype=np.int32)
        self.lib.zref_divsufsort(data, sa.ctypes.data_as(C.c_void_p), C.c_int(len(data)))
        return sa[: len(data)].astype(np.uint32)

    def make_config(self, method):
        args = (C.c_int * 9)()
        out = C.create_string_buffer(1 << 16)
        r = self.lib.zref_make_config(method.encode(), args, out, 1 << 16)
        if r < 0:
            raise RuntimeError(self.lib.zref_last_error().decode(errors="replace"))
        return out.value.decode(), list(args)

    def compile(self, config, args):
        a = (C.c_int * 9)(*args)
        hdr = C.create_string_buffer(70000)
        pc = C.create_string_buffer(70000)
        hl, pl = C.c_int(0), C.c_int(0)
        r = self.lib.zref_compile(config.encode(), a, hdr, C.byref(hl), pc, C.byref(pl))
        if r < 0:
            raise RuntimeError(self.lib.zref_last_error().decode(errors="replace"))
        return hdr.raw[: hl.value], pc.raw[: pl.value]

    def lz_stream(self, data, args):
        data = bytes(data)
        a = (C.c_int * 9)(*args)
        cap = len(data) + len(data) // 16 + 1024
        out = C.create_string_buffer(cap)
        r = self.lib.zref_lz_stream(data, C.c_uint(len(data)), a, out, C.c_ulonglong(cap))
        if r < 0:
            raise RuntimeError(self.lib.zref_last_error().decode(errors="replace"))
        return out.raw[:r]

    def fragment(self, data, fragment=6):
        data = bytes(data)
        cap = len(data) // 64 + 16
        fl = np.zeros(cap, dtype=np.uint32)
        fh = np.zeros(cap, dtype=np.uint32)
        k = self.lib.zref_fragment(data, C.c_ulonglong(len(data)), C.c_int(fragment), fl.ctypes.data_as(C.c_void_p),
                                   fh.ctypes.data_as(C.c_void_p), C.c_ulonglong(cap))
        return fl[:k].copy(), fh[:k].copy()

    def block_header(self, data, method, filename=None, comment=None):
        """The model header (hsize + HCOMP bytes) of the block compress_block writes."""
        blk = self.compress_block(data, method, filename, comment)
        hs = blk[18] + 256 * blk[19]
        return blk[18:20 + hs]

    def archive_d_h(self, files, flags):
        """`zpaqfranz a <archive> <dir> flags...` (the reference's main(), in a child process) over a directory holding
        `files` ({relative path: bytes}).  Returns (date14 of the transaction, number of d blocks, the d blocks
        concatenated, the h blocks concatenated)."""
        code = ("import ctypes as C, sys\n"
                "lib = C.CDLL(%r)\n"
                "a = [x.encode() for x in sys.argv[1:]]\n"
                "arr = (C.c_char_p * len(a))(*a)\n"
                "lib.zref_main.restype = C.c_int\n"
                "sys.exit(lib.zref_main(len(a), arr))\n") % self.lib._name
        with tempfile.TemporaryDirectory() as tmp:
            src = os.path.join(tmp, "src")
            for rel, data in files.items():
                p = os.path.join(src, rel)
                os.makedirs(os.path.dirname(p), exist_ok=True)
                with open(p, "wb") as f:
                    f.write(data)
            archive = os.path.join(tmp, "t.zpaq")
            r = subprocess.run([sys.executable, "-c", code, "zpaqfranz", "a", archive, src] + list(flags),
                               capture_output=True, text=True, timeout=900)
            if r.returncode != 0:
                raise RuntimeError(r.stdout[-2000:] + r.stderr[-2000:])
            blob = open(archive, "rb").read()
        blocks = split_blocks(blob)
        d = b"".join(b for k, _, b in blocks if k == "d")
        h = b"".join(b for k, _, b in blocks if k == "h")
        return blocks[0][1][3:17], sum(1 for k, _, _ in blocks if k == "d"), d, h


ZPAQ_TAG = bytes([0x37, 0x6b, 0x53, 0x74, 0xa0, 0x31, 0x83, 0xd3, 0x8c, 0xb2, 0x28, 0xb0, 0xd3]) + b"zPQ"


def split_blocks(blob):
    """[(kind, name, block bytes)] of a journaling archive: kind is the letter after the 14-digit date."""
    starts = []
    p = blob.find(ZPAQ_TAG)
    while p >= 0:
        starts.append(p)
        p = blob.find(ZPAQ_TAG, p + 16)
    out = []
    for i, s in enumerate(starts):
        e = starts[i + 1] if i + 1 < len(starts) else len(blob)
        b = blob[s:e]
        q = 18
        q += 2 + b[q] + 256 * b[q + 1]
        assert b[q] == 1
        name = b[q + 1: b.index(b"\0", q + 1)].decode()
        assert name.startswith("jDC")
        out.append((name[17], name, b))
    return out


# ---- the reference's answers as golden data ---------------------------------------------------------------------
# The tests ask the reference through the `ref` fixture: a GoldenRef, which answers from tests/golden/ref/, so that the
# comparisons run wherever the tests do; a RecordingRef around the built reference writes those answers.  Answers are
# keyed by the method name and a digest of the arguments.  Bytes and arrays larger than FULL_BYTES, and strings longer
# than LONG_STR, are kept as length + the first 128 bits of their SHA-256 only (a Digest, which compares equal to the
# value it stands for), except the results of KEEP, which the tests feed to the decoders under test.
GOLDEN_DIR = os.path.join(ROOT, "tests", "golden", "ref")
FULL_BYTES = 160          # small blocks whole: some tests read single bytes of them
LONG_STR = 64
KEEP = ("compress_multi",)


def _sha(b):
    return hashlib.sha256(b).hexdigest()[:32]


class Digest:
    """A value the reference returned -- bytes, an array or a string -- known by its length and digest only."""
    __array_ufunc__ = None          # ndarray == Digest defers to Digest.__eq__
    __hash__ = None

    def __init__(self, n, sha, dtype=None, shape=None, is_str=False):
        self.n, self.sha, self.dtype, self.shape, self.is_str = n, sha, dtype, shape, is_str

    def __eq__(self, other):
        if isinstance(other, Digest):
            return vars(self) == vars(other)
        if isinstance(other, np.ndarray):
            if self.dtype is None or list(other.shape) != self.shape:
                return np.bool_(False)
            return np.bool_(_sha(np.ascontiguousarray(other, dtype=np.dtype(self.dtype)).tobytes()) == self.sha)
        if isinstance(other, str) and self.is_str:
            return len(other) == self.n and _sha(other.encode()) == self.sha
        if isinstance(other, (bytes, bytearray, memoryview)) and self.dtype is None and not self.is_str:
            return len(other) == self.n and _sha(other) == self.sha
        return NotImplemented

    def __ne__(self, other):
        r = self.__eq__(other)
        return r if r is NotImplemented else ~r if isinstance(r, np.bool_) else not r

    def __len__(self):
        return self.n

    def __repr__(self):
        return "Digest(%d %s, sha256 %s...)" % (self.n, "characters" if self.is_str else "bytes", self.sha)


def _canon(x):
    """Canonical text of a call's arguments (large values by digest; a Digest as the string it stands for)."""
    if isinstance(x, (bytes, bytearray, memoryview)):
        return "b%d:%s" % (len(x), hashlib.sha256(x).hexdigest())
    if isinstance(x, np.ndarray):
        return "a%s%s:%s" % (x.dtype.str, list(x.shape), hashlib.sha256(np.ascontiguousarray(x).tobytes()).hexdigest())
    if isinstance(x, (list, tuple)):
        return "[" + ",".join(_canon(v) for v in x) + "]"
    if isinstance(x, dict):
        return "{" + ",".join("%r:%s" % (k, _canon(x[k])) for k in sorted(x)) + "}"
    if isinstance(x, np.integer):
        return repr(int(x))
    if isinstance(x, str) and len(x) > LONG_STR:
        return "s%d:%s" % (len(x), _sha(x.encode()))
    if isinstance(x, Digest) and x.is_str:
        return "s%d:%s" % (x.n, x.sha)
    if x is None or isinstance(x, (bool, int, float, str)):
        return repr(x)
    raise TypeError("no canonical form for %r" % type(x))


def call_key(name, args, kwargs):
    return "%s:%s" % (name, hashlib.sha256(_canon([list(args), kwargs]).encode()).hexdigest()[:16])


def _encode(v, full):
    if isinstance(v, (bytes, bytearray)):
        v = bytes(v)
        if full or len(v) <= FULL_BYTES:
            return {"b64": base64.b64encode(v).decode()}
        return {"len": len(v), "sha": _sha(v)}
    if isinstance(v, np.ndarray):
        raw = np.ascontiguousarray(v).tobytes()
        e = {"dtype": v.dtype.str, "shape": list(v.shape)}
        if full or len(raw) <= FULL_BYTES:
            e["b64"] = base64.b64encode(raw).decode()
        else:
            e.update(len=len(raw), sha=_sha(raw))
        return e
    if isinstance(v, str) and len(v) > LONG_STR:
        return {"str_len": len(v), "sha": _sha(v.encode())}
    if isinstance(v, tuple):
        return {"tuple": [_encode(x, full) for x in v]}
    if isinstance(v, list):
        return [_encode(x, full) for x in v]
    if isinstance(v, np.integer):
        return int(v)
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    raise TypeError("cannot record %r" % type(v))


def _decode(e):
    if isinstance(e, list):
        return [_decode(x) for x in e]
    if not isinstance(e, dict):
        return e
    if "tuple" in e:
        return tuple(_decode(x) for x in e["tuple"])
    if "str_len" in e:
        return Digest(e["str_len"], e["sha"], is_str=True)
    if "dtype" in e:
        if "b64" in e:
            return np.frombuffer(base64.b64decode(e["b64"]), dtype=np.dtype(e["dtype"])).reshape(e["shape"]).copy()
        return Digest(e["len"], e["sha"], e["dtype"], e["shape"])
    if "b64" in e:
        return base64.b64decode(e["b64"])
    return Digest(e["len"], e["sha"])


class GoldenRef:
    """Answers Ref's questions from tests/golden/ref/*.json.  A question that was never recorded fails the test:
    its arguments differ from the ones the reference was asked."""

    def __init__(self, directory=GOLDEN_DIR):
        self.answers = {}
        for f in sorted(os.listdir(directory)):
            if f.endswith(".json"):
                with open(os.path.join(directory, f)) as fh:
                    self.answers.update(json.load(fh))

    def __getattr__(self, name):
        if name.startswith("_") or not callable(getattr(Ref, name, None)):
            raise AttributeError(name)

        def answer(*args, **kwargs):
            key = call_key(name, args, kwargs)
            if key not in self.answers:
                raise AssertionError("no recorded answer of the reference to %s (%s): where oracle/_ref/libzpaqref.so is "
                                     "built, record them with ZQ_RECORD_REF=tests/golden/ref python -m pytest tests" % (name, key))
            return _decode(self.answers[key])
        return answer


class RecordingRef:
    """The reference itself, every answer also kept for tests/golden/ref/<test module>.json."""

    def __init__(self, ref):
        self._ref, self.answers = ref, {}

    def __getattr__(self, name):
        f = getattr(self._ref, name)
        if name.startswith("_") or not callable(f):
            return f

        def record(*args, **kwargs):
            v = f(*args, **kwargs)
            module = os.environ.get("PYTEST_CURRENT_TEST", "unknown").split("::")[0]
            module = os.path.splitext(os.path.basename(module))[0]
            self.answers.setdefault(module, {})[call_key(name, args, kwargs)] = _encode(v, name in KEEP)
            return v
        return record

    def save(self, directory):
        os.makedirs(directory, exist_ok=True)
        for module, answers in self.answers.items():
            with open(os.path.join(directory, module + ".json"), "w") as fh:
                fh.write("{\n" + ",\n".join("%s:%s" % (json.dumps(k), json.dumps(answers[k], sort_keys=True, separators=(",", ":")))
                                             for k in sorted(answers)) + "\n}\n")


def load_oracle():
    return Oracle(C.CDLL(os.path.join(REF_DIR, "libzqoracle.so")))


def load_ref():
    p = os.path.join(REF_DIR, "libzpaqref.so")
    if not os.path.exists(p):
        return None
    return Ref(C.CDLL(p))
