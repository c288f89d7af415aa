"""CPU: the PNG encoder's C ABI rejects bad arguments without a GPU, and the sequential pieces the kernels run
(attwarp_b200/csrc/png_deflate.h, compiled for the host by g++ through tests/hostcheck/png_hostcheck.cpp) are
checked against zlib: Huffman code lengths (complete, length-limited), the dynamic-block header, the tokeniser run
over many chunks as the CTA's threads run it, and the CRC-32 combination."""

import ctypes
import os
import shutil
import subprocess
import zlib

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("png_hostcheck") / "libpnghostcheck.so"
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(HERE, "hostcheck", "png_hostcheck.cpp")])
    lib = ctypes.CDLL(str(out))
    lib.hc_crc32_chunked.restype = ctypes.c_uint32
    return lib


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _lengths(hc, freq, max_bits=15):
    freq = np.ascontiguousarray(freq, dtype=np.uint32)
    lens = np.full(freq.size, 99, np.uint8)
    hc.hc_huff_lengths(_p(freq), freq.size, max_bits, _p(lens))
    return lens


def _kraft(lens):
    used = lens[lens > 0].astype(np.int64)
    return sum(2.0 ** -int(x) for x in used)


def _fibonacci(n):
    f = [1, 1]
    while len(f) < n:
        f.append(f[-1] + f[-2])
    return np.array(f[:n], np.uint64)


@pytest.mark.parametrize("case", ["random", "one_symbol", "no_symbol", "all_equal", "fibonacci", "sparse"])
@pytest.mark.parametrize("max_bits", [15, 7])
def test_huffman_lengths_complete_and_limited(hc, case, max_bits):
    rng = np.random.default_rng(len(case) * 31 + max_bits)
    n = 286 if max_bits == 15 else 19
    freq = np.zeros(n, np.uint64)
    if case == "random":
        freq[:] = rng.integers(0, 5000, n) * (rng.random(n) < 0.8)
    elif case == "one_symbol":
        freq[n // 2] = 12345
    elif case == "all_equal":
        freq[:] = 7
    elif case == "fibonacci":                 # an unlimited code would be 39 bits deep
        k = min(n, 40)
        freq[:k] = rng.permutation(_fibonacci(k))
    elif case == "sparse":
        freq[[0, 5, n - 1]] = [1, 1000, 3]
    lens = _lengths(hc, freq, max_bits)
    assert lens.max() <= max_bits
    assert _kraft(lens) == 1.0                # complete: every decoder accepts it
    assert np.all(lens[freq > 0] > 0)
    assert (lens > 0).sum() == max(2, int((freq > 0).sum()))
    if case == "fibonacci":
        assert lens.max() == max_bits
    if case in ("random", "all_equal", "sparse"):
        # more frequent symbols never get longer codes
        used = np.nonzero(freq)[0]
        order = used[np.argsort(freq[used], kind="stable")]
        assert np.all(np.diff(lens[order].astype(int)) <= 0)


def _block(hc, data, nchunks):
    data = np.ascontiguousarray(data, dtype=np.uint8)
    out = np.zeros(2 * data.size + 1024, np.uint8)
    nb = hc.hc_deflate_block(_p(data), data.size, nchunks, _p(out))
    return out[:nb].tobytes()


def _fib_bytes(rng):
    counts = _fibonacci(22)
    return rng.permutation(np.repeat(np.arange(22, dtype=np.uint8) * 11, counts.astype(np.int64)))


@pytest.mark.parametrize("kind", ["constant", "noise", "runs", "fibonacci", "one_byte", "two_bytes", "long_runs"])
@pytest.mark.parametrize("nchunks", [1, 3, 256])
def test_dynamic_block_decodes_with_zlib(hc, kind, nchunks):
    rng = np.random.default_rng(5)
    data = {
        "constant": np.full(5000, 9, np.uint8),
        "noise": rng.integers(0, 256, 7000, dtype=np.uint8),
        "runs": np.repeat(rng.integers(0, 5, 700).astype(np.uint8), rng.integers(1, 12, 700)),
        "fibonacci": _fib_bytes(rng),
        "one_byte": np.array([200], np.uint8),
        "two_bytes": np.array([3, 3], np.uint8),
        "long_runs": np.repeat(np.array([1, 2, 1, 7], np.uint8), [258 * 3 + 2, 259, 3, 1000]),
    }[kind]
    blk = _block(hc, data, nchunks)
    d = zlib.decompressobj(-15)
    assert d.decompress(blk) == data.tobytes()
    assert d.eof and d.unused_data == b""
    if kind in ("constant", "long_runs"):
        assert len(blk) < 200                  # the runs became matches


def test_chunked_tokeniser_is_the_sequential_one(hc):
    """Splitting a segment between threads does not change a single bit of the block."""
    rng = np.random.default_rng(9)
    data = np.repeat(rng.integers(0, 3, 3000).astype(np.uint8), rng.integers(1, 300, 3000))[:32768]
    ref = _block(hc, data, 1)
    for nchunks in (2, 7, 64, 256, 1000):
        assert _block(hc, data, nchunks) == ref


def test_crc_combination(hc):
    rng = np.random.default_rng(2)
    for n in (0, 1, 4, 5, 100, 32773):
        data = rng.integers(0, 256, n, dtype=np.uint8)
        for nchunks in (1, 2, 5, 256):
            assert hc.hc_crc32_chunked(_p(data), n, nchunks) == zlib.crc32(data.tobytes())


def test_png_argument_validation_without_gpu():
    """Invalid arguments are rejected before any CUDA call."""
    import ctypes as C
    from attwarp_b200 import _lib
    lib = _lib.load()
    buf = C.create_string_buffer(64)
    table = (_lib_png_image() * 2)()
    table[0].src, table[0].H, table[0].W, table[0].C = C.addressof(buf), 2, 2, 3
    table[1].src, table[1].H, table[1].W, table[1].C = C.addressof(buf), 1, 1, 1
    ok_out = sum(lib.attwarp_png_max_bytes(t.H, t.W, t.C) for t in table)
    ws = lib.attwarp_png_workspace_bytes(table, 2)
    assert ws > 0 and ok_out > 0
    args = dict(images=table, n=2, ws=C.addressof(buf), ws_bytes=ws, out=C.addressof(buf), cap=ok_out,
                offsets=C.addressof(buf))

    def call(**kw):
        a = dict(args, **kw)
        return lib.attwarp_encode_png(a["images"], a["n"], a["ws"], a["ws_bytes"], a["out"], a["cap"], a["offsets"],
                                      None)

    assert call(images=None) == _lib.ERR_INVALID_ARG and b"NULL" in lib.attwarp_last_error()
    assert call(out=None) == _lib.ERR_INVALID_ARG
    assert call(offsets=None) == _lib.ERR_INVALID_ARG
    assert call(n=0) == _lib.ERR_INVALID_ARG
    assert call(cap=ok_out - 1) == _lib.ERR_INVALID_ARG and b"too small" in lib.attwarp_last_error()
    assert call(ws=None) == _lib.ERR_WORKSPACE
    assert call(ws_bytes=ws - 1) == _lib.ERR_WORKSPACE
    for field, value in (("C", 2), ("C", 0), ("C", 5), ("H", 0), ("W", 0), ("W", -3), ("src", None)):
        saved = getattr(table[0], field)
        setattr(table[0], field, value)
        assert call() == _lib.ERR_INVALID_ARG, (field, value)
        setattr(table[0], field, saved)
    for shape in ((0, 4, 3), (4, 0, 3), (4, 4, 2), (4, 4, 0)):
        assert lib.attwarp_png_max_bytes(*shape) == 0
    assert lib.attwarp_png_workspace_bytes(None, 1) == 0
    assert lib.attwarp_png_workspace_bytes(table, 0) == 0


def test_png_max_bytes_is_the_stored_size_plus_overhead():
    from attwarp_b200 import _lib
    lib = _lib.load()
    for h, w, c in ((1, 1, 1), (336, 336, 3), (500, 500, 3), (1, 30000, 3), (7, 5, 4)):
        raw = h * (1 + w * c)
        segs = -(-raw // 32768)
        assert lib.attwarp_png_max_bytes(h, w, c) == raw + 17 * segs + 75


def _lib_png_image():
    import ctypes as C

    class PngImage(C.Structure):
        _fields_ = [("src", C.c_void_p), ("H", C.c_int32), ("W", C.c_int32), ("C", C.c_int32)]
    return PngImage
