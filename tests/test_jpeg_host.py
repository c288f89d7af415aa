"""CPU: the sequential pieces of the JPEG decoder (attwarp_b200/csrc/jpeg_decode.h, compiled for the host by g++
through tests/hostcheck/jpeg_hostcheck.cpp) decode a seeded corpus bit for bit as Pillow does; the product's
attwarp_jpeg_probe accepts exactly that corpus and refuses other files with their own codes; the decode entry
points reject bad arguments without a GPU."""

import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

import jpeg_corpus as JC

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("jpeg_hostcheck") / "libjpeghostcheck.so"
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(HERE, "hostcheck", "jpeg_hostcheck.cpp")])
    return C.CDLL(str(out))


@pytest.fixture(scope="module")
def corpus():
    return JC.corpus()


def _host_decode(hc, b):
    info = (C.c_int32 * 4)()
    hc.hc_jpeg_probe(b, len(b), info)
    out = np.zeros((max(info[0], 1), max(info[1], 1), 3), np.uint8)
    rc = hc.hc_jpeg_decode(b, len(b), out.ctypes.data_as(C.c_void_p), None)
    return rc, out


def test_corpus_covers_the_supported_subset(corpus):
    names = [n for n, _ in corpus]
    for s in JC.SAMPLINGS:
        assert any(n.startswith(f"cv2_{s}_") for n in names)
    for q in JC.QUALITIES:
        assert any(f"_q{q}_" in n for n in names)
    hs = {h % 16 for h, _ in JC.SIZES}
    ws = {w % 16 for _, w in JC.SIZES}
    assert hs == ws == set(range(16))
    assert len(corpus) > 800


def test_sequential_decode_matches_pillow(hc, corpus):
    bad = []
    for name, b in corpus:
        rc, out = _host_decode(hc, b)
        if rc != 0 or not np.array_equal(out, JC.pillow_bgr(b)):
            bad.append((name, rc))
    assert not bad, bad[:10]


def test_probe_accepts_the_corpus(corpus):
    from attwarp_b200 import ops
    for name, b in corpus:
        h, w, c, sup = ops.jpeg_probe(b)
        ref = JC.pillow_bgr(b)
        assert sup == 0, name
        assert (h, w) == ref.shape[:2] and c == (1 if "grey" in name else 3), name


def _photo(h=48, w=40):
    return JC.content("photo", h, w, np.random.default_rng(3))


def test_probe_refuses_other_files_with_their_own_codes():
    from attwarp_b200 import ops
    img = _photo()
    base = JC.pil_jpeg(img, quality=90)
    prog = JC.pil_jpeg(img, quality=90, progressive=True)
    import io

    from PIL import Image
    buf = io.BytesIO()
    Image.fromarray(img[..., ::-1]).convert("CMYK").save(buf, "JPEG", quality=90)
    cmyk = buf.getvalue()
    png = JC.cv2.imencode(".png", img)[1].tobytes()
    a, _ = JC.scan_range(base)
    codes = {
        "progressive": ops.jpeg_probe(prog)[3],
        "cmyk": ops.jpeg_probe(cmyk)[3],
        "truncated_header": ops.jpeg_probe(base[:a - 10])[3],
        "not_jpeg": ops.jpeg_probe(png)[3],
        "random_bytes": ops.jpeg_probe(np.random.default_rng(1).integers(0, 256, 500, dtype=np.uint8).tobytes())[3],
        "data_after_eoi": ops.jpeg_probe(base + b"\x00trailer")[3],
    }
    assert codes["progressive"] == 3
    assert codes["cmyk"] == 7
    assert codes["truncated_header"] == 2
    assert codes["not_jpeg"] == 1 and codes["random_bytes"] == 1
    assert codes["data_after_eoi"] == 9
    assert ops.jpeg_probe(base)[3] == 0
    for name, b in (("cmyk", cmyk), ("progressive", prog)):
        assert ops.JPEG_SUPPORT_REASONS[codes[name]]


def test_host_decode_refuses_malformed_entropy_data(hc):
    b = bytearray(JC.pil_jpeg(_photo(64, 64), quality=90, restart_marker_blocks=2))
    a, e = JC.scan_range(bytes(b))
    # a run of stuffed FF bytes is 64 one-bits: no Huffman code is all ones
    bad_code = bytes(b[:a + 40]) + b"\xff\x00" * 8 + bytes(b[a + 56:])
    assert _host_decode(hc, bad_code)[0] == -2
    i = bytes(b).index(b"\xff\xd3", a)
    no_rst = bytes(b[:i]) + bytes(b[i + 2:])
    assert _host_decode(hc, no_rst)[0] == -4
    short = bytes(b[:a + (e - a) // 2]) + b"\xff\xd9"
    assert _host_decode(hc, short)[0] in (-1, -4)


def _jpeg_image_type():
    class JpegImage(C.Structure):
        _fields_ = [("host", C.c_void_p), ("dev", C.c_void_p), ("nbytes", C.c_size_t), ("dst", C.c_void_p),
                    ("H", C.c_int32), ("W", C.c_int32)]
    return JpegImage


def test_decode_argument_validation_without_gpu():
    """Invalid arguments are rejected before any CUDA call."""
    from attwarp_b200 import _lib
    lib = _lib.load()
    good = JC.pil_jpeg(_photo(), quality=90)
    prog = JC.pil_jpeg(_photo(), quality=90, progressive=True)
    gbuf = C.create_string_buffer(good, len(good))
    pbuf = C.create_string_buffer(prog, len(prog))
    scratch = C.create_string_buffer(64)
    table = (_jpeg_image_type() * 2)()
    for t in table:
        t.host, t.dev, t.nbytes, t.dst, t.H, t.W = C.addressof(gbuf), C.addressof(scratch), len(good), \
            C.addressof(scratch), 48, 40
    ws = lib.attwarp_jpeg_workspace_bytes(table, 2)
    assert ws > 0
    status = C.create_string_buffer(8)
    args = dict(images=table, n=2, ws=C.addressof(scratch), ws_bytes=ws, status=C.addressof(status))

    def call(**kw):
        a = dict(args, **kw)
        return lib.attwarp_decode_jpeg(a["images"], a["n"], a["ws"], a["ws_bytes"], a["status"], None)

    assert call(images=None) == _lib.ERR_INVALID_ARG and b"NULL" in lib.attwarp_last_error()
    assert call(status=None) == _lib.ERR_INVALID_ARG
    assert call(n=0) == _lib.ERR_INVALID_ARG
    assert call(ws=None) == _lib.ERR_WORKSPACE
    assert call(ws_bytes=ws - 1) == _lib.ERR_WORKSPACE and b"too small" in lib.attwarp_last_error()
    for field, value in (("H", 47), ("W", 41), ("host", None), ("dev", None), ("dst", None)):
        saved = getattr(table[1], field)
        setattr(table[1], field, value)
        assert call() == _lib.ERR_INVALID_ARG, (field, value)
        assert b"image 1" in lib.attwarp_last_error()
        setattr(table[1], field, saved)
    table[1].host, table[1].nbytes = C.addressof(pbuf), len(prog)
    assert call() == _lib.ERR_UNSUPPORTED and b"image 1" in lib.attwarp_last_error()
    assert lib.attwarp_jpeg_workspace_bytes(table, 2) == 0
    assert lib.attwarp_jpeg_workspace_bytes(None, 1) == 0
    assert lib.attwarp_jpeg_workspace_bytes(table, 0) == 0
    info = (C.c_int32 * 4)()
    assert lib.attwarp_jpeg_probe(None, 10, info) == _lib.ERR_INVALID_ARG
    assert lib.attwarp_jpeg_probe(gbuf, len(good), None) == _lib.ERR_INVALID_ARG
    assert lib.attwarp_jpeg_probe(gbuf, len(good), info) == _lib.OK and list(info) == [48, 40, 3, 0]


def test_python_entry_points_refuse_without_gpu():
    from attwarp_b200 import image_io, ops
    prog = JC.pil_jpeg(_photo(), quality=90, progressive=True)
    good = JC.pil_jpeg(_photo(), quality=90)
    with pytest.raises(ValueError, match="file 1 is not device-decodable: progressive"):
        ops.decode_jpeg([good, prog], device="cuda:0")
    with pytest.raises(ValueError, match="exclusive"):
        image_io.decode_jpeg_batch([good], device="cuda:0", exact=True, exact_device=True)
