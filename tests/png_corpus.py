"""A seeded corpus of PNG files for the PNG decoder's tests, generated on the CPU (no downloads): files written by
Pillow (compress_level 0/1/6/9, optimize), by cv2.imencode (compression 0-9 x every IMWRITE_PNG_STRATEGY) and by a
Python writer (zlib.compressobj with varied level, strategy, wbits 9-15 and memLevel 1-9, a random filter type per
row, IDAT chunks cut at random sizes including 1-byte and empty ones, sync / full flushes every few bytes), in
every colour type and bit depth the device decodes, plus adversarial streams (one distance-1 run over a whole
2048^2 image, distance 32768, matches across block and IDAT boundaries, length code 285, literal-only blocks)."""

from __future__ import annotations

import io
import struct
import zlib

import cv2
import numpy as np
from PIL import Image

SUBSET = [(0, 1), (0, 2), (0, 4), (0, 8), (2, 8), (3, 1), (3, 2), (3, 4), (3, 8), (4, 8), (6, 8)]
CHANNELS = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}
CV2_STRATEGIES = {"default": cv2.IMWRITE_PNG_STRATEGY_DEFAULT, "filtered": cv2.IMWRITE_PNG_STRATEGY_FILTERED,
                  "huffman": cv2.IMWRITE_PNG_STRATEGY_HUFFMAN_ONLY, "rle": cv2.IMWRITE_PNG_STRATEGY_RLE,
                  "fixed": cv2.IMWRITE_PNG_STRATEGY_FIXED}


def pillow_bgr(b: bytes) -> np.ndarray:
    return np.ascontiguousarray(np.array(Image.open(io.BytesIO(b)).convert("RGB"))[..., ::-1])


def cv2_bgr(b: bytes):
    return cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR)


def photo(h: int, w: int, rng, c: int = 3) -> np.ndarray:
    """Smooth gradients, a few blobs and mild noise: compresses like a photograph."""
    y, x = np.mgrid[0:h, 0:w].astype(np.float32)
    img = np.zeros((h, w, c), np.float32)
    for k in range(c):
        fx, fy, ph = rng.uniform(0.5, 4.0), rng.uniform(0.5, 4.0), rng.uniform(0, 6.28)
        img[..., k] = 128 + 90 * np.sin(fx * x / max(w, 1) * 6.28 + ph) * np.cos(fy * y / max(h, 1) * 6.28)
    for _ in range(3):
        cy, cx, r = rng.uniform(0, h), rng.uniform(0, w), rng.uniform(4, max(h, w) / 3 + 5)
        img += (((y - cy) ** 2 + (x - cx) ** 2) < r * r)[..., None] * rng.uniform(-60, 60, c)
    img += rng.normal(0, 6, img.shape)
    return np.clip(img, 0, 255).astype(np.uint8)


# ---- a PNG writer of our own ------------------------------------------------------------------------------------
def chunk(tag: bytes, data: bytes, crc: int | None = None) -> bytes:
    c = zlib.crc32(tag + data) if crc is None else crc
    return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", c & 0xFFFFFFFF)


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(raw: np.ndarray, bpp: int, filters) -> bytes:
    """raw: [H, row_bytes] uint8 -> the filtered stream with filters[y] per row."""
    out = []
    prev = np.zeros(raw.shape[1], np.int32)
    for y in range(raw.shape[0]):
        row = raw[y].astype(np.int32)
        a = np.concatenate([np.zeros(bpp, np.int32), row[:-bpp]]) if row.size > bpp else np.zeros_like(row)
        c = np.concatenate([np.zeros(bpp, np.int32), prev[:-bpp]]) if row.size > bpp else np.zeros_like(row)
        if row.size <= bpp:
            a = np.zeros_like(row)
            c = np.zeros_like(row)
        f = int(filters[y])
        pred = [0, a, prev, (a + prev) >> 1, _paeth(a, prev, c)][f]
        out.append(bytes([f]) + ((row - pred) & 255).astype(np.uint8).tobytes())
        prev = row
    return b"".join(out)


def pack_rows(idx: np.ndarray, depth: int) -> np.ndarray:
    """[H, W] samples of `depth` bits -> [H, row_bytes] packed MSB first."""
    if depth == 8:
        return idx.astype(np.uint8)
    h, w = idx.shape
    per = 8 // depth
    rb = (w * depth + 7) // 8
    pad = np.zeros((h, rb * per), np.uint8)
    pad[:, :w] = idx
    pad = pad.reshape(h, rb, per)
    out = np.zeros((h, rb), np.uint8)
    for k in range(per):
        out |= (pad[:, :, k] << (8 - depth * (k + 1))).astype(np.uint8)
    return out


def write_png(samples: np.ndarray, colour: int, depth: int, rng, palette=None, trns=None, level=6,
              strategy=zlib.Z_DEFAULT_STRATEGY, wbits=15, memlevel=8, filters=None, flush_every=0,
              flush_mode=zlib.Z_SYNC_FLUSH, idat_sizes=None, stream=None, extra_chunks=(),
              interlace=False) -> bytes:
    """samples: [H, W] or [H, W, C] in file channel order (RGB / indices / grey).  interlace: Adam7, 8-bit
    samples, every row of every pass with filter 0."""
    h, w = samples.shape[:2]
    ch = CHANNELS[colour]
    bpp = max(1, ch * depth // 8)
    if interlace:
        data = b""
        for x0, y0, dx, dy in ((0, 0, 8, 8), (4, 0, 8, 8), (0, 4, 4, 8), (2, 0, 4, 4), (0, 2, 2, 4), (1, 0, 2, 2),
                               (0, 1, 1, 2)):
            sub = samples[y0::dy, x0::dx]
            if sub.size:
                data += filter_rows(sub.reshape(sub.shape[0], -1).astype(np.uint8), bpp, [0] * sub.shape[0])
    else:
        raw = pack_rows(samples, depth) if ch == 1 else samples.reshape(h, w * ch).astype(np.uint8)
        if filters is None:
            filters = rng.integers(0, 5, h)
        data = filter_rows(raw, bpp, filters)
    if stream is None:
        co = zlib.compressobj(level, zlib.DEFLATED, wbits, memlevel, strategy)
        if flush_every:
            parts = []
            for k in range(0, len(data), flush_every):
                parts.append(co.compress(data[k:k + flush_every]))
                parts.append(co.flush(flush_mode))
            parts.append(co.flush())
            stream = b"".join(parts)
        else:
            stream = co.compress(data) + co.flush()
    out = [b"\x89PNG\r\n\x1a\n", chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, colour, 0, 0, int(interlace)))]
    out += [chunk(t, d) for t, d in extra_chunks]
    if palette is not None:
        out.append(chunk(b"PLTE", bytes(np.asarray(palette, np.uint8).reshape(-1))))
    if trns is not None:
        out.append(chunk(b"tRNS", trns))
    if idat_sizes is None:
        out.append(chunk(b"IDAT", stream))
    else:
        k = 0
        for s in idat_sizes:
            out.append(chunk(b"IDAT", stream[k:k + s]))
            k += s
        if k < len(stream):
            out.append(chunk(b"IDAT", stream[k:]))
    out.append(chunk(b"IEND", b""))
    return b"".join(out)


def random_cuts(n: int, rng) -> list:
    """IDAT sizes summing to less than n: 1-byte, empty and larger pieces."""
    sizes, total = [], 0
    while total < n:
        s = int(rng.choice([0, 1, 1, 2, 7, 100, 1000, 5000]))
        sizes.append(s)
        total += s
    return sizes


def random_samples(colour, depth, h, w, rng, photo_like=True):
    ch = CHANNELS[colour]
    if colour == 3 or depth < 8:
        hi = 1 << depth
        return (photo(h, w, rng, 1)[..., 0].astype(np.int32) * hi // 256).astype(np.uint8)
    img = photo(h, w, rng, ch) if photo_like else rng.integers(0, 256, (h, w, ch), dtype=np.uint8)
    return img if ch > 1 else img[..., 0]


def palette_file(depth, h, w, rng, entries=None, trns=False, out_of_range=False, **kw) -> bytes:
    hi = 1 << depth
    n = int(entries if entries is not None else rng.integers(1, hi + 1))
    idx = (random_samples(3, depth, h, w, rng).astype(np.int32) % n).astype(np.uint8)
    if out_of_range and n < hi:
        idx[rng.random(idx.shape) < 0.1] = hi - 1
    pal = rng.integers(0, 256, (n, 3), dtype=np.uint8)
    tr = bytes(rng.integers(0, 256, int(rng.integers(1, n + 1)), dtype=np.uint8)) if trns else None
    return write_png(idx, 3, depth, rng, palette=pal, trns=tr, **kw)


# ---- the corpus -------------------------------------------------------------------------------------------------
SIZES = [(1, 1), (1, 17), (23, 1), (5, 3)] + [(7 + k, 16 + k) for k in range(16)]


def corpus(seed: int = 0):
    """List of (name, bytes)."""
    rng = np.random.default_rng(seed)
    out = []
    img = photo(48, 61, rng)
    for lvl in (0, 1, 6, 9):
        buf = io.BytesIO()
        Image.fromarray(img[..., ::-1]).save(buf, "PNG", compress_level=lvl)
        out.append((f"pil_l{lvl}", buf.getvalue()))
    for mode in ("L", "RGB", "RGBA", "P", "LA", "1"):
        buf = io.BytesIO()
        src = Image.fromarray(photo(33, 45, rng))
        src = src.convert(mode) if mode != "P" else src.quantize(200)
        src.save(buf, "PNG", optimize=True)
        out.append((f"pil_opt_{mode}", buf.getvalue()))
    for lvl in range(10):
        for sname, s in CV2_STRATEGIES.items():
            im = photo(int(rng.integers(20, 70)), int(rng.integers(20, 70)), rng, int(rng.choice([1, 3, 4])))
            out.append((f"cv2_c{lvl}_{sname}",
                        cv2.imencode(".png", im, [cv2.IMWRITE_PNG_COMPRESSION, lvl, cv2.IMWRITE_PNG_STRATEGY, s])[1]
                        .tobytes()))
    strategies = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FILTERED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE, zlib.Z_FIXED]
    k = 0
    for colour, depth in SUBSET:
        for h, w in SIZES:
            kw = dict(level=int(rng.integers(0, 10)), strategy=strategies[k % 5], wbits=9 + k % 7,
                      memlevel=1 + k % 9)
            if k % 3 == 0:
                kw["idat_sizes"] = random_cuts(4 * h * w + 64, rng)
            if k % 4 == 1:
                kw["flush_every"] = int(rng.integers(1, 40))
                kw["flush_mode"] = zlib.Z_SYNC_FLUSH if k % 8 == 1 else zlib.Z_FULL_FLUSH
            k += 1
            if colour == 3:
                b = palette_file(depth, h, w, rng, trns=k % 2 == 0, out_of_range=k % 3 == 0, **kw)
            else:
                tr = None
                if k % 2 == 0 and colour in (0, 2):
                    vals = rng.integers(0, 1 << depth, 1 if colour == 0 else 3)
                    tr = b"".join(struct.pack(">H", int(v)) for v in vals)
                b = write_png(random_samples(colour, depth, h, w, rng), colour, depth, rng, trns=tr, **kw)
            out.append((f"py_c{colour}_d{depth}_{h}x{w}", b))
    for n in (1, 2, 17, 255, 256):
        out.append((f"py_palette_{n}", palette_file(8, 19, 21, rng, entries=n, trns=n % 2 == 1,
                                                    out_of_range=n < 256)))
    # row bytes at every residue mod 16 for RGB and grey
    for w in range(1, 17):
        out.append((f"py_rgb_w{w}", write_png(photo(9, w, rng), 2, 8, rng)))
    out += adversarial(rng)
    return out


def raw_deflate_stream(blocks: bytes) -> bytes:
    return b"\x78\x01" + blocks


class BitWriter:
    def __init__(self):
        self.acc, self.n, self.out = 0, 0, bytearray()

    def put(self, v, n):
        self.acc |= v << self.n
        self.n += n
        while self.n >= 8:
            self.out.append(self.acc & 255)
            self.acc >>= 8
            self.n -= 8

    def put_rev(self, code, n):       # a Huffman code, most significant bit first
        self.put(int(format(code, f"0{n}b")[::-1], 2), n)

    def flush(self):
        if self.n:
            self.out.append(self.acc & 255)
        self.acc, self.n = 0, 0
        return bytes(self.out)


def fixed_code(sym):
    if sym < 144:
        return 0x30 + sym, 8
    if sym < 256:
        return 0x190 + sym - 144, 9
    if sym < 280:
        return sym - 256, 7
    return 0xC0 + sym - 280, 8


def fixed_block_stream(data: bytes, tokens) -> bytes:
    """A zlib stream of one fixed-Huffman block of `tokens` ((literal,) or (length, distance)) producing `data`."""
    bw = BitWriter()
    bw.put(1, 1)
    bw.put(1, 2)
    for t in tokens:
        if len(t) == 1:
            bw.put_rev(*fixed_code(t[0]))
        else:
            ln, d = t
            if ln == 258:
                sym, ex, nex = 285, 0, 0
            else:
                v = ln - 3
                if v < 8:
                    sym, ex, nex = 257 + v, 0, 0
                else:
                    lg = v.bit_length() - 1
                    nex = lg - 2
                    sym, ex = 261 + 4 * nex + ((v >> nex) - 4), v & ((1 << nex) - 1)
            bw.put_rev(*fixed_code(sym))
            if nex:
                bw.put(ex, nex)
            v = d - 1
            if v < 4:
                dsym, dex, dn = v, 0, 0
            else:
                lg = v.bit_length() - 1
                dn = lg - 1
                dsym, dex = 2 * lg + ((v >> dn) & 1), v & ((1 << dn) - 1)
            bw.put_rev(dsym, 5)
            if dn:
                bw.put(dex, dn)
    bw.put_rev(*fixed_code(256))
    return raw_deflate_stream(bw.flush()) + struct.pack(">I", zlib.adler32(data))


def adversarial(rng):
    out = []
    # a whole 2048^2 grey image as one distance-1 run (length code 285 throughout)
    h = w = 2048
    data = b"\x00" * ((w + 1) * h)
    toks = [(0,)]
    left = len(data) - 1
    while left >= 258:
        toks.append((258, 1))
        left -= 258
    toks += [(0,)] * left
    out.append(("adv_d1_run_2048", write_png(np.zeros((h, w), np.uint8), 0, 8, rng,
                                             stream=fixed_block_stream(data, toks), idat_sizes=[65536] * 200)))
    # distance exactly 32768: 32768 random bytes then a copy of them, as one RGB image
    w = 1024
    rows = (32768 * 2) // (3 * w + 1) + 1
    total = rows * (3 * w + 1)
    first = rng.integers(0, 5, 32768, dtype=np.uint8).tobytes()    # values 0-4: every row starts with a filter type
    data = bytearray(total)
    data[:32768] = first
    for i in range(32768, total):
        data[i] = data[i - 32768]
    data = bytes(data)
    toks = [(b,) for b in data[:32768]]
    left = total - 32768
    while left > 0:
        ln = min(258, left)
        if ln < 3:
            toks += [(data[total - left + j],) for j in range(ln)]
            break
        toks.append((ln, 32768))
        left -= ln
    out.append(("adv_dist_32768", write_png(np.zeros((rows, w, 3), np.uint8), 2, 8, rng,
                                            stream=fixed_block_stream(data, toks), idat_sizes=random_cuts(total, rng))))
    # matches across block and IDAT boundaries: full flushes are not used, sync flushes keep the window
    img = photo(200, 300, rng)
    out.append(("adv_sync_flush_blocks", write_png(img, 2, 8, rng, level=9, flush_every=997,
                                                   idat_sizes=[1, 0, 3] + [257] * 2000)))
    # blocks of literals only
    out.append(("adv_literals_only", write_png(photo(64, 64, rng), 2, 8, rng, strategy=zlib.Z_HUFFMAN_ONLY,
                                               level=9, flush_every=300)))
    # long runs (length code 285 at distance 1 and 3) from zlib
    flat = np.zeros((300, 400, 3), np.uint8)
    flat[100:200] = (10, 200, 30)
    out.append(("adv_runs_zlib", write_png(flat, 2, 8, rng, filters=np.zeros(300, np.int64), level=9)))
    return out


def big_photo_list(seed: int, n: int, lo: int, hi: int):
    """n photo-like RGB files of sides lo..hi, cv2 at its default level and Pillow at level 6 alternately."""
    rng = np.random.default_rng(seed)
    out = []
    for k in range(n):
        h, w = int(rng.integers(lo, hi + 1)), int(rng.integers(lo, hi + 1))
        img = photo(h, w, rng)
        if k % 2 == 0:
            out.append(cv2.imencode(".png", img)[1].tobytes())
        else:
            buf = io.BytesIO()
            Image.fromarray(img[..., ::-1]).save(buf, "PNG", compress_level=6)
            out.append(buf.getvalue())
    return out
