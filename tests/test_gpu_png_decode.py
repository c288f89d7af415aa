"""GPU: ops.decode_png equals Pillow's Image.open(f).convert('RGB') (as BGR) on the seeded corpus and on a fuzz
list; a round trip through ops.encode_png gives the pixels back; a file's pixels depend on nothing else in the
call; the kernel writes each [H, W, 3] buffer at any byte alignment and nothing around it; malformed files are
accepted or rejected as cv2.imdecode (libpng) accepts or rejects them; the whole list takes one kernel launch;
decode_jpeg_batch(exact_device=True) routes every file to an exact decoder; warp_files(exact_decode=True) on PNG
inputs writes the files the cv2 decode gives."""

import ctypes as C
import struct
import zlib

import cv2
import numpy as np
import pytest
import torch

import png_corpus as PC
from gpu_util import need_gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _gpu():
    need_gpu()


def _check_equal(files, outs, names=None):
    bad = []
    for i, (b, t) in enumerate(zip(files, outs)):
        ref = PC.pillow_bgr(b)
        got = t.cpu().numpy()
        if got.shape != ref.shape or not np.array_equal(got, ref):
            bad.append(names[i] if names else i)
    assert not bad, bad[:10]


def test_corpus_equals_pillow():
    from attwarp_b200 import ops
    corpus = PC.corpus()
    files = [b for _, b in corpus]
    _check_equal(files, ops.decode_png(files), [n for n, _ in corpus])


def _fuzz(n, seed, max_side=300):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        colour, depth = PC.SUBSET[int(rng.integers(len(PC.SUBSET)))]
        h, w = int(rng.integers(1, max_side)), int(rng.integers(1, max_side))
        kw = dict(level=int(rng.integers(0, 10)), wbits=int(rng.integers(9, 16)), memlevel=int(rng.integers(1, 10)),
                  strategy=int(rng.choice([zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE,
                                           zlib.Z_FIXED])))
        if k % 3 == 0:
            kw["idat_sizes"] = PC.random_cuts(h * w, rng)
        if colour == 3:
            out.append(PC.palette_file(depth, h, w, rng, out_of_range=k % 2 == 0, **kw))
        else:
            out.append(PC.write_png(PC.random_samples(colour, depth, h, w, rng), colour, depth, rng, **kw))
    return out


def test_fuzz_list_equals_pillow():
    from attwarp_b200 import ops
    files = _fuzz(200, 7) + PC.big_photo_list(3, 6, 600, 1400)
    _check_equal(files, ops.decode_png(files))


def test_round_trip_through_encode_png():
    from attwarp_b200 import image_io, ops
    g = torch.Generator(device="cuda").manual_seed(3)
    imgs = [torch.randint(0, 256, (h, w, c), dtype=torch.uint8, device="cuda", generator=g)
            for h, w, c in ((37, 91, 3), (500, 333, 3), (64, 64, 4), (1, 1, 3), (200, 17, 1))]
    imgs[1] = torch.from_numpy(PC.photo(500, 333, np.random.default_rng(1))).cuda()
    files = image_io.encode_png_device(imgs)
    outs = ops.decode_png(files)
    for im, t in zip(imgs, outs):
        ref = im[..., :3] if im.shape[2] >= 3 else im.expand(-1, -1, 3)
        assert torch.equal(t, ref.contiguous())


def test_output_independent_of_list_position():
    from attwarp_b200 import ops
    files = _fuzz(40, 9, 120)
    alone = [ops.decode_png([b])[0].cpu() for b in files]
    perm = np.random.default_rng(1).permutation(len(files))
    together = ops.decode_png([files[k] for k in perm] + files[:5])
    for j, k in enumerate(perm):
        assert torch.equal(together[j].cpu(), alone[k])
    for j in range(5):
        assert torch.equal(together[len(files) + j].cpu(), alone[j])


def test_rows_at_odd_byte_offsets_and_guard_bytes():
    from attwarp_b200 import _lib, ops
    files = _fuzz(24, 5, 90)
    shapes = [PC.pillow_bgr(b).shape for b in files]
    guard = 37
    sizes = [int(np.prod(s)) for s in shapes]
    starts, at = [], 1
    for sz in sizes:
        at += guard
        at += 1 - at % 2
        starts.append(at)
        at += sz
    buf = torch.full((at + guard,), 0xA5, dtype=torch.uint8, device="cuda")
    lib = _lib.load()
    host = torch.from_numpy(np.frombuffer(b"".join(files), np.uint8).copy()).pin_memory()
    dev = host.cuda()
    offs = np.concatenate([[0], np.cumsum([len(b) for b in files])])
    table = np.zeros(len(files), dtype=ops._PNG_FILE_DTYPE)
    table["host"] = host.data_ptr() + offs[:-1]
    table["dev"] = dev.data_ptr() + offs[:-1]
    table["nbytes"] = [len(b) for b in files]
    table["dst"] = [buf.data_ptr() + s for s in starts]
    table["H"] = [s[0] for s in shapes]
    table["W"] = [s[1] for s in shapes]
    tp = table.ctypes.data_as(C.c_void_p)
    ws = torch.empty(lib.attwarp_png_decode_workspace_bytes(tp, len(files)), dtype=torch.uint8, device="cuda")
    status = torch.full((len(files),), -1, dtype=torch.int32, device="cuda")
    assert lib.attwarp_decode_png(tp, len(files), C.c_void_p(ws.data_ptr()), ws.numel(),
                                  C.c_void_p(status.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)) == 0
    assert not status.cpu().numpy().any()
    hb = buf.cpu().numpy()
    mask = np.ones(hb.size, bool)
    for b, s, sz, shp in zip(files, starts, sizes, shapes):
        assert np.array_equal(hb[s:s + sz].reshape(shp), PC.pillow_bgr(b))
        mask[s:s + sz] = False
    assert np.all(hb[mask] == 0xA5)


def _malformed():
    """name -> file bytes; each malformation of the table in DESIGN.md section 6 item 9."""
    rng = np.random.default_rng(8)
    img = PC.photo(60, 70, rng)
    rgb = img[..., ::-1]
    raw = PC.filter_rows(rgb.reshape(60, -1), 3, rng.integers(0, 5, 60))
    z = zlib.compress(raw, 6)
    good = PC.write_png(rgb, 2, 8, rng, stream=z, idat_sizes=[500])

    def with_stream(stream, **kw):
        return PC.write_png(rgb, 2, 8, rng, stream=stream, **kw)

    def flip_crc(b, tag, nth=0):
        i = -1
        for _ in range(nth + 1):
            i = b.index(tag, i + 1)
        n = struct.unpack(">I", b[i - 4:i])[0]
        b = bytearray(b)
        b[i + 4 + n] ^= 0x55
        return bytes(b)

    bad_adler = z[:-1] + bytes([z[-1] ^ 1])
    bad_filter = bytearray(raw)
    bad_filter[(3 * 70 + 1) * 7] = 5
    pal = PC.palette_file(8, 20, 20, rng)
    return good, {
        "bad_crc_ihdr": flip_crc(good, b"IHDR"),
        "bad_crc_plte": flip_crc(pal, b"PLTE"),
        "bad_crc_idat": flip_crc(good, b"IDAT", 1),
        "bad_adler": with_stream(bad_adler),
        "truncated_zlib": with_stream(z[:len(z) // 2]),
        "too_few_rows": with_stream(zlib.compress(raw[:len(raw) - 2 * (3 * 70 + 1)])),
        "filter_above_4": with_stream(zlib.compress(bytes(bad_filter))),
        "bad_crc_ancillary": PC.write_png(rgb, 2, 8, rng, stream=z, extra_chunks=[(b"tEXt", b"a\x00b")])
        .replace(PC.chunk(b"tEXt", b"a\x00b"), PC.chunk(b"tEXt", b"a\x00b", crc=1)),
        "extra_rows": with_stream(zlib.compress(raw + raw[:3 * (3 * 70 + 1)])),
        "bytes_after_stream": with_stream(z + b"trailing"),
    }


@pytest.mark.parametrize("kind", list(_malformed()[1]))
def test_malformed_files_accepted_and_rejected_as_cv2(kind):
    from attwarp_b200 import image_io, ops
    good, cases = _malformed()
    bad = cases[kind]
    cv_ok = PC.cv2_bgr(bad) is not None
    dev_ok = True
    try:
        outs = image_io.decode_jpeg_batch([good, bad], device="cuda", exact_device=True)
    except ValueError as exc:
        dev_ok = False
        assert "source 1 " in str(exc), str(exc)
    assert dev_ok == cv_ok, (kind, cv_ok)
    if dev_ok:
        assert np.array_equal(outs[1].cpu().numpy(), PC.cv2_bgr(bad))
        if kind != "bad_crc_ancillary":                  # Pillow rejects a bad ancillary CRC before IDAT
            assert np.array_equal(outs[1].cpu().numpy(), PC.pillow_bgr(bad))
    if ops.png_probe(bad)[4] == 0 and not cv_ok:
        with pytest.raises(ValueError, match="file 2 is malformed"):
            ops.decode_png([good, good, bad, good])


def test_one_launch_for_the_list(tmp_path):
    """torch.profiler can miss the first kernel record of a window late in a long session, so the window opens with
    a kernel of its own and a trace without the decode kernel is taken again (as tests/test_gpu_overlay.py does)."""
    import json

    from attwarp_b200 import ops
    files = _fuzz(30, 12, 200)
    ops.decode_png(files)
    kernels = []
    for _ in range(3):
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            torch.ones(1, device="cuda").add_(1)
            ops.decode_png(files)
            torch.cuda.synchronize()
        prof.export_chrome_trace(str(tmp_path / "trace.json"))
        with open(tmp_path / "trace.json") as f:
            events = json.load(f).get("traceEvents", [])
        if not any(e.get("cat") == "kernel" for e in events):
            pytest.skip("torch.profiler reported no CUDA kernel events: the launches are not checked")
        kernels = [e["name"] for e in events if e.get("cat") == "kernel" and "png_decode_kernel" in e["name"]]
        if kernels:
            break
    assert len(kernels) == 1, kernels


def _count_decode_png(monkeypatch):
    """Patches ops.decode_png to record the length of every list it is called with."""
    from attwarp_b200 import ops
    calls, real = [], ops.decode_png

    def counted(buffers, device=None):
        calls.append(len(buffers))
        return real(buffers, device)

    monkeypatch.setattr(ops, "decode_png", counted)
    return calls


def test_decode_jpeg_batch_routes_every_file(tmp_path, monkeypatch):
    import io

    from PIL import Image

    from attwarp_b200 import image_io
    rng = np.random.default_rng(12)
    imgs = [PC.photo(70 + 9 * k, 90 - 7 * k, rng) for k in range(5)]
    jpg = io.BytesIO()
    Image.fromarray(imgs[0][..., ::-1]).save(jpg, "JPEG", quality=90)
    png = cv2.imencode(".png", imgs[1])[1].tobytes()
    png16 = cv2.imencode(".png", imgs[2].astype(np.uint16) * 257)[1].tobytes()
    inter = PC.write_png(imgs[3][..., ::-1], 2, 8, rng, interlace=True)
    pal = PC.palette_file(4, 33, 21, rng)
    srcs = [jpg.getvalue(), png, png16, inter, pal]
    path = tmp_path / "f.png"
    path.write_bytes(png)
    srcs.append(str(path))
    calls = _count_decode_png(monkeypatch)
    outs = image_io.decode_jpeg_batch(srcs, exact_device=True)
    assert calls == [3]                              # png, pal and the path: one call; 16-bit and interlaced to cv2
    for k, (s, t) in enumerate(zip(srcs, outs)):
        b = s if isinstance(s, bytes) else open(s, "rb").read()
        ref = PC.pillow_bgr(b) if k in (0, 1, 3, 4, 5) else PC.cv2_bgr(b)
        assert t.dtype == torch.uint8 and t.is_cuda
        assert np.array_equal(t.cpu().numpy(), ref), k


def test_warp_files_on_png_inputs(tmp_path, monkeypatch):
    from attwarp_b200 import image_io
    rng = np.random.default_rng(21)
    shapes = [(120, 160), (97, 131), (64, 64), (150, 90)]
    pngs = []
    for k, (h, w) in enumerate(shapes):
        p = tmp_path / f"in{k}.png"
        cv2.imwrite(str(p), PC.photo(h, w, rng))
        pngs.append(str(p))
    n = len(shapes)
    tok = torch.rand(n, 24, 24, generator=torch.Generator().manual_seed(1))

    def run(tag, exact):
        outs = [str(tmp_path / f"{tag}_w{k}.png") for k in range(n)]
        ovs = [str(tmp_path / f"{tag}_o{k}.png") for k in range(n)]
        ors = [str(tmp_path / f"{tag}_g{k}.png") for k in range(n)]
        assert all(image_io.warp_files(pngs, tok, outs, overlay_paths=ovs, original_paths=ors, exact_decode=exact,
                                       out_sizes=[(100, 110)] * n))
        return [cv2.imread(p, cv2.IMREAD_UNCHANGED) for p in outs + ovs + ors]

    calls = _count_decode_png(monkeypatch)
    got = run("dev", True)
    assert calls == [n]
    ref = run("ref", False)
    assert calls == [n]
    for k, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(g, r), k


def one_idat(b: bytes) -> bytes:
    """The same file with its IDAT payloads joined into one chunk."""
    off, head, data, tail = 8, [], [], []
    while off < len(b):
        n, tag = struct.unpack(">I4s", b[off:off + 8])
        piece = b[off:off + 12 + n]
        if tag == b"IDAT":
            data.append(b[off + 8:off + 8 + n])
        elif data:
            tail.append(piece)
        else:
            head.append(piece)
        off += 12 + n
    return b[:8] + b"".join(head) + PC.chunk(b"IDAT", b"".join(data)) + b"".join(tail)


def test_single_idat_files_and_their_crc():
    """Files of one large IDAT chunk (as lodepng, stb or the png crate write them): the chunk's CRC is split across
    the CTA; a flipped CRC bit is found there too."""
    from attwarp_b200 import ops
    files = [one_idat(b) for b in PC.big_photo_list(4, 4, 900, 1500)]
    assert all(b.count(b"IDAT") == 1 for b in files)
    _check_equal(files, ops.decode_png(files))
    bad = bytearray(files[1])
    i = bad.index(b"IDAT")
    n = struct.unpack(">I", bad[i - 4:i])[0]
    bad[i + 4 + n + 3] ^= 0x10
    with pytest.raises(ValueError, match="file 2 is malformed: IDAT CRC mismatch"):
        ops.decode_png([files[0], files[2], bytes(bad)])
