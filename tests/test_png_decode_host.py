"""CPU: the sequential pieces of the PNG decoder (attwarp_b200/csrc/png_inflate.h, compiled for the host by g++
through tests/hostcheck/png_decode_hostcheck.cpp, with the kernel's window decode run one window after another) inflate
the seeded corpus as zlib does and decode it as Pillow does; Pillow and cv2.imdecode agree on every corpus file, so
moving exact_device PNGs from cv2 to the device changes no pixel; the product's attwarp_png_probe accepts the
corpus and refuses other files with their own codes; the decode entry points reject bad arguments without a GPU."""

import ctypes as C
import io
import os
import shutil
import struct
import subprocess
import zlib

import numpy as np
import pytest

import png_corpus as PC

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("png_decode_hostcheck") / "libpngdecodehostcheck.so"
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(HERE, "hostcheck", "png_decode_hostcheck.cpp")])
    return C.CDLL(str(out))


@pytest.fixture(scope="module")
def corpus():
    return PC.corpus()


def _idat_stream(b: bytes) -> bytes:
    off, parts = 8, []
    while off < len(b):
        n, tag = struct.unpack(">I4s", b[off:off + 8])
        if tag == b"IDAT":
            parts.append(b[off + 8:off + 8 + n])
        off += 12 + n
    return b"".join(parts)


def test_corpus_covers_the_subset(corpus):
    names = [n for n, _ in corpus]
    for colour, depth in PC.SUBSET:
        assert any(n.startswith(f"py_c{colour}_d{depth}_") for n in names)
    for lvl in range(10):
        for s in PC.CV2_STRATEGIES:
            assert f"cv2_c{lvl}_{s}" in names
    for k in ("adv_d1_run_2048", "adv_dist_32768", "adv_sync_flush_blocks", "adv_literals_only", "adv_runs_zlib"):
        assert k in names
    assert {w % 16 for w in range(1, 17)} == set(range(16))


def test_inflate_equals_zlib(hc, corpus):
    bad = []
    stats = (C.c_int64 * 3)()
    for name, b in corpus:
        ref = zlib.decompress(_idat_stream(b))
        out = np.zeros(len(ref) + 1, np.uint8)
        n = C.c_int64()
        rc = hc.hc_png_inflate(b, len(b), out.ctypes.data_as(C.c_void_p), out.size, C.byref(n), stats)
        if rc != 0 or n.value != len(ref) or out[:len(ref)].tobytes() != ref:
            bad.append((name, rc))
    assert not bad, bad[:10]


def test_decode_equals_pillow_and_pillow_equals_cv2(hc, corpus):
    bad, differ = [], []
    for name, b in corpus:
        ref = PC.pillow_bgr(b)
        cv = PC.cv2_bgr(b)
        if cv is None or not np.array_equal(cv, ref):
            differ.append(name)
        out = np.zeros_like(ref)
        rc = hc.hc_png_decode(b, len(b), out.ctypes.data_as(C.c_void_p))
        if rc != 0 or not np.array_equal(out, ref):
            bad.append((name, rc))
    assert not bad, bad[:10]
    assert not differ, differ[:10]


def test_window_sync_statistic(hc):
    """Windows of 512 bits until a trajectory started at a window's first bit meets the true one, per writer (the
    numbers DESIGN.md section 6 item 9 records): they meet within a window or two, so the sync rounds of a set are
    few."""
    lists = {"cv2": PC.big_photo_list(1, 2, 300, 400)[0::2], "pillow": PC.big_photo_list(1, 2, 300, 400)[1::2]}
    rng = np.random.default_rng(2)
    lists["zlib_rle"] = [PC.write_png(PC.photo(300, 300, rng), 2, 8, rng, strategy=zlib.Z_RLE)]
    lists["zlib_fixed"] = [PC.write_png(PC.photo(300, 300, rng), 2, 8, rng, strategy=zlib.Z_FIXED)]
    for name, files in lists.items():
        stats = (C.c_int64 * 3)()
        for b in files:
            n = C.c_int64()
            assert hc.hc_png_inflate(b, len(b), None, 0, C.byref(n), stats) == 0
        mean = stats[1] / max(stats[0], 1)
        print(f"window sync {name}: {stats[0]} guessed windows, mean {mean:.3f}, max {stats[2]}")
        assert stats[0] > 100 and mean < 2 and stats[2] <= 16, (name, list(stats))


def _rgb(h=20, w=30, seed=3):
    return PC.photo(h, w, np.random.default_rng(seed))


def _with_ihdr(b: bytes, w: int, h: int) -> bytes:
    """b with IHDR's width and height replaced and its CRC recomputed."""
    ihdr = struct.pack(">II", w, h) + b[24:29]
    return b[:8] + PC.chunk(b"IHDR", ihdr) + b[33:]


def test_probe_codes():
    from attwarp_b200 import ops
    import cv2
    rng = np.random.default_rng(5)
    img = _rgb()
    good = cv2.imencode(".png", img)[1].tobytes()
    assert ops.png_probe(good) == (20, 30, 2, 8, 0)
    sixteen = cv2.imencode(".png", img.astype(np.uint16) * 257)[1].tobytes()
    inter = PC.write_png(img[..., ::-1], 2, 8, rng, interlace=True)
    bad_ihdr = bytearray(good)
    bad_ihdr[29] ^= 1                                      # IHDR CRC
    idx = PC.palette_file(8, 10, 10, rng)
    no_plte = idx.replace(b"PLTE", b"pLTE")                # now an ancillary chunk: a palette file without PLTE
    split = PC.write_png(img[..., ::-1], 2, 8, rng, idat_sizes=[50], extra_chunks=())
    i = split.index(b"IDAT", split.index(b"IDAT") + 4) - 4  # a tEXt chunk between the two IDAT chunks
    split = split[:i] + PC.chunk(b"tEXt", b"k\x00v") + split[i:]
    fdict = PC.write_png(img[..., ::-1], 2, 8, rng, stream=b"\x78\xbb" + b"\x00" * 8)
    codes = {"not_png": ops.png_probe(b"GIF89a" + b"\x00" * 40)[4], "truncated": ops.png_probe(good[:60])[4],
             "sixteen": ops.png_probe(sixteen)[4], "interlaced": ops.png_probe(inter)[4],
             "bad_ihdr": ops.png_probe(bytes(bad_ihdr))[4], "no_plte": ops.png_probe(no_plte)[4],
             "split_idat": ops.png_probe(split)[4], "preset_dict": ops.png_probe(fdict)[4],
             "size": ops.png_probe(_with_ihdr(PC.write_png(np.zeros((1, 1), np.uint8), 0, 8, rng), 1_000_001, 1))[4],
             "size_ok": ops.png_probe(_with_ihdr(PC.write_png(np.zeros((1, 1), np.uint8), 0, 8, rng), 1_000_000, 1))[4]}
    assert codes == {"not_png": 1, "truncated": 2, "sixteen": 3, "interlaced": 4, "bad_ihdr": 5, "no_plte": 6,
                     "split_idat": 6, "preset_dict": 6, "size": 7, "size_ok": 0}
    for c in set(codes.values()) - {0}:
        assert ops.PNG_SUPPORT_REASONS[c]


def test_probe_accepts_the_corpus(corpus):
    from attwarp_b200 import ops
    for name, b in corpus:
        h, w, _, _, sup = ops.png_probe(b)
        assert sup == 0, name
        assert (h, w) == PC.pillow_bgr(b).shape[:2], name


def _file_type():
    class PngFile(C.Structure):
        _fields_ = [("host", C.c_void_p), ("dev", C.c_void_p), ("nbytes", C.c_size_t), ("dst", C.c_void_p),
                    ("H", C.c_int32), ("W", C.c_int32)]
    return PngFile


def test_decode_argument_validation_without_gpu():
    """Invalid arguments are rejected before any CUDA call."""
    import cv2

    from attwarp_b200 import _lib
    lib = _lib.load()
    good = cv2.imencode(".png", _rgb())[1].tobytes()
    inter = PC.write_png(_rgb()[..., ::-1], 2, 8, np.random.default_rng(0), interlace=True)
    gbuf = C.create_string_buffer(good, len(good))
    ibuf = C.create_string_buffer(inter, len(inter))
    scratch = C.create_string_buffer(64)
    table = (_file_type() * 2)()
    for t in table:
        t.host, t.dev, t.nbytes, t.dst, t.H, t.W = C.addressof(gbuf), C.addressof(scratch), len(good), \
            C.addressof(scratch), 20, 30
    ws = lib.attwarp_png_decode_workspace_bytes(table, 2)
    assert ws > 0
    status = C.create_string_buffer(8)
    args = dict(files=table, n=2, ws=C.addressof(scratch), ws_bytes=ws, status=C.addressof(status))

    def call(**kw):
        a = dict(args, **kw)
        return lib.attwarp_decode_png(a["files"], a["n"], a["ws"], a["ws_bytes"], a["status"], None)

    assert call(files=None) == _lib.ERR_INVALID_ARG and b"NULL" in lib.attwarp_last_error()
    assert call(status=None) == _lib.ERR_INVALID_ARG
    assert call(n=0) == _lib.ERR_INVALID_ARG
    assert call(ws=None) == _lib.ERR_WORKSPACE
    assert call(ws_bytes=ws - 1) == _lib.ERR_WORKSPACE and b"too small" in lib.attwarp_last_error()
    for field, value in (("H", 19), ("W", 31), ("host", None), ("dev", None), ("dst", None)):
        saved = getattr(table[1], field)
        setattr(table[1], field, value)
        assert call() == _lib.ERR_INVALID_ARG, (field, value)
        assert b"file 1" in lib.attwarp_last_error()
        setattr(table[1], field, saved)
    table[1].host, table[1].nbytes = C.addressof(ibuf), len(inter)
    assert call() == _lib.ERR_UNSUPPORTED and b"file 1" in lib.attwarp_last_error()
    assert lib.attwarp_png_decode_workspace_bytes(table, 2) == 0
    assert lib.attwarp_png_decode_workspace_bytes(None, 1) == 0
    assert lib.attwarp_png_decode_workspace_bytes(table, 0) == 0
    info = (C.c_int32 * 5)()
    assert lib.attwarp_png_probe(None, 10, info) == _lib.ERR_INVALID_ARG
    assert lib.attwarp_png_probe(gbuf, len(good), None) == _lib.ERR_INVALID_ARG
    assert lib.attwarp_png_probe(gbuf, len(good), info) == _lib.OK and list(info) == [20, 30, 2, 8, 0]


def test_python_entry_point_refuses_without_gpu():
    from attwarp_b200 import ops
    import cv2
    good = cv2.imencode(".png", _rgb())[1].tobytes()
    sixteen = cv2.imencode(".png", _rgb().astype(np.uint16) * 257)[1].tobytes()
    with pytest.raises(ValueError, match="file 1 is not device-decodable: 16-bit samples"):
        ops.decode_png([good, sixteen], device="cuda:0")


def test_split_chunk_crc_equals_zlib(hc):
    """The kernel's CRC of a large IDAT chunk: kThreads pieces (the first one short), each a raw CRC, folded as a
    tree with crc_combine (png_inflate.h crc_piece / crc_raw / crc32_finish)."""
    hc.hc_crc32_split.restype = C.c_uint32
    hc.hc_crc32_split.argtypes = [C.c_char_p, C.c_uint64, C.c_int]
    rng = np.random.default_rng(6)
    for n in (1, 2, 255, 256, 257, 16389, 65536 + 13, 1_000_003):
        b = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
        for pieces in (1, 2, 8, 256):
            assert hc.hc_crc32_split(b, n, pieces) == zlib.crc32(b), (n, pieces)


def test_code_rules_follow_zlib(hc):
    """zlib's inflate_table: a code-length code must be complete; literal/length and distance codes may also be a
    single code of length 1; only the distance code may be empty; an over-subscribed code is never allowed."""
    def build(lens, kind):
        a = np.array(lens, np.uint8)
        return hc.hc_huff_build(a.ctypes.data_as(C.c_void_p), len(lens), kind)

    single = [0] * 5 + [1] + [0] * 13
    complete = [1, 2, 2] + [0] * 16
    over = [1, 1, 1] + [0] * 16
    empty = [0] * 19
    assert [build(single, k) for k in (0, 1, 2)] == [-1, 0, 0]
    assert [build(complete, k) for k in (0, 1, 2)] == [0, 0, 0]
    assert [build(over, k) for k in (0, 1, 2)] == [-1, -1, -1]
    assert [build(empty, k) for k in (0, 1, 2)] == [-1, -1, 0]
    assert [build([2, 2, 2] + [0] * 16, k) for k in (0, 1, 2)] == [-1, -1, -1]     # incomplete, longest code 2
