"""Seeded JPEG files for the decoder tests (tests/test_jpeg_host.py, tests/test_gpu_jpeg.py), written with Pillow
and cv2.imencode (both libjpeg-turbo), and the reference every decode is held to: Pillow's
``Image.open(f).convert('RGB')`` in BGR order."""

import io

import cv2
import numpy as np
from PIL import Image

QUALITIES = (1, 5, 50, 75, 90, 95, 100)
SAMPLINGS = {411: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411, 420: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
             422: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422, 440: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440,
             444: cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444}
CONTENTS = ("noise", "flat", "gradient", "photo")
# every residue mod 16 of both the height and the width, 1 x 1 up
SIZES = [(h, (5 * h + 3) % 16 + 16 * (h % 3) + 1) for h in range(1, 17)] + [(1, 1), (97, 130), (336, 336)]


def content(kind, h, w, rng):
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "flat":
        return np.broadcast_to(rng.integers(0, 256, 3, dtype=np.uint8), (h, w, 3)).copy()
    yy, xx = np.mgrid[0:h, 0:w]
    img = np.stack([xx * 255 // max(w - 1, 1), yy * 255 // max(h - 1, 1), (xx + 2 * yy) % 256], -1).astype(np.uint8)
    if kind == "photo":                     # smooth, with noise and saturated colour blocks (hard chroma edges)
        img = np.clip(img.astype(np.int16) + rng.integers(-10, 11, img.shape), 0, 255).astype(np.uint8)
        img[h // 4:h // 2, w // 5:w // 2] = (0, 0, 255)
        img[h // 2:, w // 2:] = (255, 0, 255)
        img[:h // 3, 2 * w // 3:] = (0, 255, 0)
    return img


def cv2_jpeg(bgr, quality, sampling=420, rst=0, grey=False, optimize=False):
    params = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLINGS[sampling],
              cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize)]
    if rst:
        params += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    img = cv2.cvtColor(bgr, cv2.COLOR_BGR2GRAY) if grey else bgr
    ok, enc = cv2.imencode(".jpg", img, params)
    assert ok
    return enc.tobytes()


def pil_jpeg(bgr, grey=False, **kw):
    im = Image.fromarray(np.ascontiguousarray(bgr[..., ::-1]))
    if grey:
        im = im.convert("L")
    buf = io.BytesIO()
    im.save(buf, "JPEG", **kw)
    return buf.getvalue()


def pillow_bgr(b):
    return np.ascontiguousarray(np.array(Image.open(io.BytesIO(b)).convert("RGB"))[..., ::-1])


def corpus():
    """[(name, bytes)]: every supported sampling at every quality and size, grey, optimised tables, restart
    intervals of 1 block, a few blocks and whole rows, over noise / flat / gradient / photo-like content."""
    rng = np.random.default_rng(20261022)
    out = []
    for si, (h, w) in enumerate(SIZES):
        for qi, q in enumerate(QUALITIES):
            kind = CONTENTS[(si + qi) % 4]
            img = content(kind, h, w, rng)
            for s in SAMPLINGS:
                out.append((f"cv2_{s}_q{q}_{kind}_{h}x{w}", cv2_jpeg(img, q, s)))
            out.append((f"pil_grey_q{q}_{kind}_{h}x{w}", pil_jpeg(img, grey=True, quality=q)))
        img = content(CONTENTS[si % 4], h, w, rng)
        tag = f"{CONTENTS[si % 4]}_{h}x{w}"
        out.append((f"pil_opt_420_{tag}", pil_jpeg(img, quality=85, optimize=True)))
        out.append((f"pil_opt_444_{tag}", pil_jpeg(img, quality=92, optimize=True, subsampling=0)))
        out.append((f"pil_opt_grey_{tag}", pil_jpeg(img, grey=True, quality=80, optimize=True)))
        out.append((f"pil_rst1blk_{tag}", pil_jpeg(img, quality=90, restart_marker_blocks=1)))
        out.append((f"pil_rst5blk_422_{tag}", pil_jpeg(img, quality=75, subsampling=1, restart_marker_blocks=5)))
        out.append((f"pil_rstrow_{tag}", pil_jpeg(img, quality=95, restart_marker_rows=1)))
        out.append((f"pil_rstrow_grey_{tag}", pil_jpeg(img, grey=True, quality=60, restart_marker_rows=1)))
        out.append((f"cv2_rst3_440_{tag}", cv2_jpeg(img, 90, 440, rst=3)))
        out.append((f"cv2_rst1_411_{tag}", cv2_jpeg(img, 50, 411, rst=1)))
        out.append((f"cv2_grey_rst2_{tag}", cv2_jpeg(img, 70, 420, rst=2, grey=True)))
    return out


def fuzz(n=320, seed=7, max_side=700):
    """n files of random size 1..max_side, sampling, quality, optimisation, restart interval, content and grey /
    colour."""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h, w = (int(v) for v in rng.integers(1, max_side + 1, 2))
        img = content(CONTENTS[int(rng.integers(0, 4))], h, w, rng)
        q = int(rng.integers(1, 101))
        grey = bool(rng.random() < 0.2)
        if rng.random() < 0.5:
            rst = int(rng.choice([0, 0, 1, 2, 7, 40]))
            out.append(cv2_jpeg(img, q, int(rng.choice(list(SAMPLINGS))), rst=rst, grey=grey))
        else:
            kw = dict(quality=q, optimize=bool(rng.random() < 0.5), subsampling=int(rng.integers(0, 3)))
            r = rng.random()
            if r < 0.2:
                kw["restart_marker_blocks"] = int(rng.integers(1, 9))
            elif r < 0.35:
                kw["restart_marker_rows"] = int(rng.integers(1, 4))
            try:
                out.append(pil_jpeg(img, grey=grey, **kw))
            except OSError:
                # Pillow's buffer for optimised tables is too small for some noise images: the same file from cv2
                out.append(cv2_jpeg(img, q, (444, 422, 420)[kw["subsampling"]], grey=grey, optimize=kw["optimize"]))
    return out


def scan_range(b):
    """[start, end) of the entropy-coded data of a single-scan file (after the SOS header, before EOI)."""
    p = 2
    while True:
        assert b[p] == 0xFF
        m = b[p + 1]
        ln = (b[p + 2] << 8) | b[p + 3]
        if m == 0xDA:
            return p + 2 + ln, len(b) - 2
        p += 2 + ln
