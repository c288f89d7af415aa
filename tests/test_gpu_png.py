"""GPU: PNG files encoded on the device (ops.encode_png, image_io.encode_png_device) against the contract in
image_io's docstring: pixel-exact decode with cv2 and Pillow, a valid chunk structure with CRCs and Adler-32
recomputed by zlib, Sub-filtered scanlines in the zlib stream, bytes independent of the batch, sizes within 3 %
of cv2.imencode."""

import io
import struct
import zlib

import numpy as np
import pytest
import torch

from gpu_util import need_gpu

pytestmark = pytest.mark.gpu


def _photo_like(rng, h, w):
    y, x = np.mgrid[0:h, 0:w].astype(np.float64)
    base = np.stack([127 + 100 * np.sin(x / 17 + y / 23), 127 + 90 * np.cos(x / 11 - y / 29), 255 * (x + y) / (h + w)], -1)
    base += rng.normal(0, 6, base.shape)
    base[h // 3: h // 2, w // 4: w // 2] = [230, 40, 60]
    return np.clip(np.rint(base), 0, 255).astype(np.uint8)


def _smooth(h, w):
    y, x = np.mgrid[0:h, 0:w]
    return np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) * 255 // max(h + w - 2, 1)],
                    -1).astype(np.uint8)


def _image(kind, h, w, c, rng):
    if kind == "constant":
        img = np.full((h, w, 3), (17, 200, 99), np.uint8)
    elif kind == "noise":
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    elif kind == "smooth":
        img = _smooth(h, w)
    else:
        img = _photo_like(rng, h, w)
    if c == 0:
        return np.ascontiguousarray(img[..., 1])                     # 2-D
    if c == 1:
        return np.ascontiguousarray(img[..., 1:2])
    if c == 4:
        alpha = (np.arange(h * w).reshape(h, w, 1) * 7 % 256).astype(np.uint8)
        return np.concatenate([img, alpha], -1)
    return img


def _chunks(buf):
    assert buf[:8] == b"\x89PNG\r\n\x1a\n"
    pos, out = 8, []
    while pos < len(buf):
        (n,) = struct.unpack(">I", buf[pos:pos + 4])
        typ, data = buf[pos + 4:pos + 8], buf[pos + 8:pos + 8 + n]
        (crc,) = struct.unpack(">I", buf[pos + 8 + n:pos + 12 + n])
        assert crc == zlib.crc32(typ + data), typ
        out.append((typ, data))
        pos += 12 + n
    assert pos == len(buf)
    return out


def _sub_filtered(img):
    h, w = img.shape[:2]
    c = 1 if img.ndim == 2 else img.shape[2]
    f = img.reshape(h, w, c)
    if c >= 3:
        f = np.concatenate([f[..., 2::-1], f[..., 3:]], -1)          # BGR(A) -> RGB(A)
    row = f.reshape(h, w * c).astype(np.int16)
    d = row.copy()
    d[:, c:] = row[:, c:] - row[:, :-c]
    return np.concatenate([np.ones((h, 1), np.uint8), (d & 255).astype(np.uint8)], 1).tobytes()


def _check_file(buf, img):
    """Contract points 1 and 2 for one file."""
    import cv2
    from PIL import Image
    ch = _chunks(buf)
    assert [t for t, _ in ch][0] == b"IHDR" and [t for t, _ in ch][-1] == b"IEND" and ch[-1][1] == b""
    assert all(t == b"IDAT" for t, _ in ch[1:-1]) and len(ch) >= 4
    ok, ref = cv2.imencode(".png", img)
    assert ok
    assert ch[0][1] == _chunks(ref.tobytes())[0][1]                  # the IHDR cv2 writes
    z = b"".join(d for _, d in ch[1:-1])
    assert z[:2] == b"\x78\x01"
    raw = zlib.decompress(z)
    assert raw == _sub_filtered(img)
    assert struct.unpack(">I", z[-4:])[0] == zlib.adler32(raw)
    got = cv2.imdecode(np.frombuffer(buf, np.uint8), cv2.IMREAD_UNCHANGED)
    want = img[..., 0] if img.ndim == 3 and img.shape[2] == 1 else img
    assert got.dtype == np.uint8 and got.shape == want.shape and np.array_equal(got, want)
    pil = np.array(Image.open(io.BytesIO(buf)))
    if img.ndim == 3 and img.shape[2] >= 3:
        pil = np.concatenate([pil[..., 2::-1], pil[..., 3:]], -1)
    assert np.array_equal(pil, want)
    return len(ref)


def _encode(imgs):
    from attwarp_b200 import image_io
    return image_io.encode_png_device([torch.from_numpy(im).cuda() for im in imgs])


SHAPES = [(1, 1), (1, 77), (93, 1), (5, 7), (37, 333), (300, 301)]


@pytest.mark.parametrize("c", [0, 1, 3, 4])
@pytest.mark.parametrize("kind", ["constant", "noise", "smooth", "photo"])
def test_png_files_decode_exactly(c, kind):
    need_gpu()
    rng = np.random.default_rng(c * 10 + len(kind))
    imgs = [_image(kind, h, w, c, rng) for h, w in SHAPES]
    for buf, img in zip(_encode(imgs), imgs):
        _check_file(buf, img)


@pytest.mark.parametrize("kind", ["photo", "noise", "constant"])
def test_png_large_and_wide(kind):
    """2048^2 (hundreds of segments in one image) and a single 30 000-pixel RGB row (one row over three segments)."""
    need_gpu()
    rng = np.random.default_rng(1)
    imgs = [_image(kind, 2048, 2048, 3, rng), _image(kind, 1, 30000, 3, rng)]
    for buf, img in zip(_encode(imgs), imgs):
        _check_file(buf, img)


def test_png_bytes_do_not_depend_on_the_batch():
    need_gpu()
    from attwarp_b200 import image_io
    rng = np.random.default_rng(4)
    imgs = []
    for k in range(24):
        kind = ["photo", "noise", "smooth", "constant"][k % 4]
        h, w = int(rng.integers(1, 400)), int(rng.integers(1, 400))
        imgs.append(_image(kind, h, w, [0, 1, 3, 4][(k // 4) % 4], rng))
    batch = _encode(imgs)
    again = _encode(imgs[::-1])[::-1]
    assert batch == again
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        on_side = image_io.encode_png_device([torch.from_numpy(im).cuda() for im in imgs])
    assert on_side == batch
    for k, img in enumerate(imgs):
        alone = _encode([img])[0]
        assert alone == batch[k], k
        _check_file(alone, img)


def test_png_batch_tensor_and_empty_list():
    need_gpu()
    from attwarp_b200 import image_io, ops
    rng = np.random.default_rng(6)
    imgs = np.stack([_photo_like(rng, 64, 48) for _ in range(3)])
    files = image_io.encode_png_device(torch.from_numpy(imgs).cuda())
    assert files == _encode(list(imgs))
    assert image_io.encode_png_device([]) == []
    payload, offsets = ops.encode_png([])
    assert payload.numel() == 0 and offsets.tolist() == [0]


@pytest.mark.parametrize("bad", ["cpu", "float", "c2", "5d", "4d_list_item", "not_a_tensor", "empty"])
def test_png_rejects_bad_inputs(bad):
    need_gpu()
    from attwarp_b200 import ops
    good = torch.zeros(4, 4, 3, dtype=torch.uint8, device="cuda")
    arg = {
        "cpu": [good.cpu()],
        "float": [good.float()],
        "c2": [good[..., :2]],
        "5d": good[None, None],
        "4d_list_item": [good[None]],
        "not_a_tensor": [np.zeros((4, 4, 3), np.uint8)],
        "empty": [good[:0]],
    }[bad]
    with pytest.raises(ValueError):
        ops.encode_png(arg)


def test_png_sizes_close_to_cv2():
    """Contract point 4: <= 1.03x cv2.imencode for photo-like, smooth and noise images at 336^2, 500^2, 1344^2 and
    for warped outputs of bench-style batches; noise no larger than stored plus fixed overhead; tiny images within
    64 bytes of cv2."""
    need_gpu()
    import cv2
    from attwarp_b200 import _lib, ops
    rng = np.random.default_rng(12)
    lib = _lib.load()
    imgs, names = [], []
    for s in (336, 500, 1344):
        for kind in ("photo", "smooth", "noise"):
            imgs.append(_image(kind, s, s, 3, rng))
            names.append(f"{kind} {s}^2")
    # warped outputs of a seeded ragged batch (the images the drivers write)
    srcs = [torch.from_numpy(_photo_like(rng, h, w)).cuda() for h, w in ((336, 336), (480, 640), (301, 224))]
    tok = torch.from_numpy((rng.random((3, 24, 24)) ** 3).astype(np.float32)).cuda()
    warped = ops.warp_ragged_from_tokens(tok, srcs, [(500, 500)] * 3)
    for k, t in enumerate(warped):
        imgs.append(t.cpu().numpy())
        names.append(f"warped {k}")
    small = [_image(kind, h, w, 3, rng) for kind in ("photo", "noise", "constant") for h, w in ((1, 1), (8, 8), (40, 60))]
    files = _encode(imgs + small)
    worst = 0.0
    for name, img, buf in zip(names, imgs, files):
        ref = len(cv2.imencode(".png", img)[1])
        ratio = len(buf) / ref
        worst = max(worst, ratio)
        print(f"[png size] {name}: {len(buf)} bytes, cv2 {ref}, ratio {ratio:.4f}")
        assert ratio <= 1.03, name
        if name.startswith("noise"):
            h, w, c = img.shape
            assert len(buf) <= lib.attwarp_png_max_bytes(h, w, c)
    for img, buf in zip(small, files[len(imgs):]):
        ref = len(cv2.imencode(".png", img)[1])
        assert len(buf) <= ref + 64, img.shape
    print(f"[png size] worst ratio {worst:.4f}")


def test_warp_files_with_device_png(tmp_path):
    need_gpu()
    import cv2
    from PIL import Image
    from attwarp_b200 import image_io
    rng = np.random.default_rng(11)
    sizes = [(224, 224), (336, 500), (301, 224)]
    files = []
    for h, w in sizes:
        buf = io.BytesIO()
        Image.fromarray(_photo_like(rng, h, w)).save(buf, format="JPEG", quality=90)
        files.append(buf.getvalue())
    tok = rng.random((3, 24, 24)) ** 3
    tok = torch.from_numpy((tok / tok.sum(axis=(1, 2), keepdims=True)).astype(np.float32))
    out_sizes = [(224, 224), (500, 500), (301, 224)]
    ref_paths = [str(tmp_path / f"ref{k}.png") for k in range(3)]
    dev_paths = [str(tmp_path / f"dev{k}.png") for k in range(3)]
    assert image_io.warp_files(files, tok, ref_paths, out_sizes) == [True] * 3
    assert image_io.warp_files(files, tok, dev_paths, out_sizes, on_device_png=True) == [True] * 3
    for r, d in zip(ref_paths, dev_paths):
        a, b = cv2.imread(r, cv2.IMREAD_UNCHANGED), cv2.imread(d, cv2.IMREAD_UNCHANGED)
        assert a is not None and b is not None and a.shape == b.shape and np.array_equal(a, b)
    assert image_io.encode_png_batch([torch.zeros(2, 2, 3, dtype=torch.uint8, device="cuda")],
                                     [str(tmp_path / "missing_dir" / "x.png")], on_device=True) == [False]
