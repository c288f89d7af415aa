"""Stage 5 (remap_quad.cu, remap_stream.cu, remap_f32_stream.cu, remap.cu): every compiled resample kernel bit for bit
against a device restatement of the oracle, at the launch geometry of small, full-size and mixed-size batches.

The resample kernels are persistent: a CTA owns a contiguous range of output rows and walks it in chunks through a ring
of shared-memory stages, carrying the blends of a source-row pair from one chunk into the next, and moving from one
(image, strip) into the next while it holds a stage.  A batch of two images gives every CTA one or two rows and never
reaches that regime; a full batch gives every CTA hundreds of rows.  CASES has one row per compiled instance and launch
configuration, at a small batch (grid = work units) and at a full one (grid = SMs x CTAs per SM, at least three full
chunks per CTA); each row names the kernel it must launch, its block size and its geometry class, all read back from
torch.profiler.  Every image of a batch takes its own map family (production token maps, identity, exact 1/32-pixel
ties, shuffled, minifying jumps, magnification, maps outside the image, flat runs), on random and coordinate-coded
inputs, and every output byte must equal the reference: BASELINE.md section 4 makes stage 5 bit-exact given identical
maps.  Outputs sit in guard bytes (0x5A, or NaN for float32) and start filled with the guard, so an unwritten or
overwritten byte shows.

ref_remap restates oracle.numpy_path.remap_u8 / remap_f32 in torch so that full-size batches can be checked on the
device; test_device_reference_equals_oracle pins it to the oracle and to cv2.remap on the CPU.  plan_ragged restates
the width classes and joins of launch_remap_u8_quad_ragged_prepare, and the mixed-size tests hold the launches to it.
Process-wide switches (ATTWARP_REMAP, ATTWARP_REMAP_F32, ATTWARP_REMAP_QUAD, ATTWARP_REMAP_CPT) run in child processes.

    python -m pytest tests/test_gpu_remap_dispatch.py -m gpu
"""

import ctypes
import json
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import numpy_path as ON

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

U8, F32 = torch.uint8, torch.float32
GUARD_U8 = 0x5A
PAD = 256                                  # guard elements before, between and after outputs
SMS_B200 = 148

# (id, kernel, dtype, layout, C, B, H, W, Ho, Wo, lead, geometry)
#   lead      elements between the guard and the output: a byte lead of 1 - 3 makes a uint8 destination unaligned
#             (the quad kernel's MODE 2)
#   geometry  small: grid = work units (one or a few rows per CTA);  full: persistent grid of SMs x CTAs per SM with at
#             least three full chunks per CTA;  direct: one CTA per 256 columns of a row;  rows: one grid plane per
#             image plane
# quad kernel: ceil(columns / 128) consumer warps (MODE 1, rows 4-byte aligned) or ceil(columns / 127) (MODE 2), at
# least 3: <128,5> <= 3 warps (4 CTAs/SM), <224,2> 4 (3 CTAs/SM) and 5-6 (2), <544,1> 7-9 (2) and 13-16 (1),
# <384,1> 10-11, <416,1> 12
Q = "remap_u8_quad_kernel"
CASES = [
    ("q3-m1-small", Q + "<128,5,1>", U8, "hwc", 3, 2, 48, 100, 40, 96, 0, "small"),
    ("q3-m2-small", Q + "<128,5,2>", U8, "hwc", 3, 2, 48, 101, 40, 95, 0, "small"),
    ("q3-m1-wide-src-small", Q + "<128,5,1>", U8, "hwc", 3, 2, 48, 6000, 40, 300, 0, "small"),
    ("q4-m1-small", Q + "<224,2,1>", U8, "hwc", 3, 2, 48, 452, 40, 448, 0, "small"),
    ("q4-m2-small", Q + "<224,2,2>", U8, "hwc", 3, 2, 48, 449, 40, 446, 0, "small"),
    ("q6-m1-small", Q + "<224,2,1>", U8, "hwc", 3, 2, 48, 701, 40, 700, 0, "small"),
    ("q6-m2-small", Q + "<224,2,2>", U8, "hwc", 3, 2, 48, 700, 40, 701, 0, "small"),
    ("q9-m1-small", Q + "<544,1,1>", U8, "hwc", 3, 2, 48, 1024, 40, 1024, 0, "small"),
    ("q9-m2-small", Q + "<544,1,2>", U8, "hwc", 3, 2, 48, 1022, 40, 1023, 0, "small"),
    ("q11-m1-small", Q + "<384,1,1>", U8, "hwc", 3, 2, 48, 1345, 40, 1344, 0, "small"),
    ("q11-m2-small", Q + "<384,1,2>", U8, "hwc", 3, 2, 48, 1344, 40, 1343, 0, "small"),
    ("q12-m1-small", Q + "<416,1,1>", U8, "hwc", 3, 2, 48, 1500, 40, 1500, 0, "small"),
    ("q12-m2-small", Q + "<416,1,2>", U8, "hwc", 3, 2, 48, 1501, 40, 1499, 0, "small"),
    ("q16-m1-small", Q + "<544,1,1>", U8, "hwc", 3, 2, 48, 2048, 40, 2048, 0, "small"),
    ("q16-m2-small", Q + "<544,1,2>", U8, "hwc", 3, 2, 48, 2031, 40, 2032, 1, "small"),
    ("q11-m1-3strips-small", Q + "<384,1,1>", U8, "hwc", 3, 1, 48, 4100, 40, 4100, 0, "small"),
    # full batches: c2 (256 x 336^2) and c3 (64 x 1344^2) are the benchmark's; the rest fill every warp range
    ("c2-m1", Q + "<128,5,1>", U8, "hwc", 3, 256, 336, 336, 336, 336, 0, "full"),
    ("c2-m2", Q + "<128,5,2>", U8, "hwc", 3, 256, 336, 336, 336, 335, 0, "full"),
    ("c2-m2-lead1", Q + "<128,5,2>", U8, "hwc", 3, 256, 336, 336, 336, 336, 1, "full"),
    ("q3-m1-wide-src-full", Q + "<128,5,1>", U8, "hwc", 3, 192, 400, 3000, 336, 336, 0, "full"),
    ("q4-m1-full", Q + "<224,2,1>", U8, "hwc", 3, 128, 480, 500, 480, 500, 0, "full"),
    ("q4-m2-full", Q + "<224,2,2>", U8, "hwc", 3, 128, 480, 500, 480, 500, 1, "full"),
    ("q6-m1-full", Q + "<224,2,1>", U8, "hwc", 3, 96, 700, 700, 700, 700, 0, "full"),
    ("q6-m2-full", Q + "<224,2,2>", U8, "hwc", 3, 96, 700, 700, 700, 701, 0, "full"),
    ("q9-m1-full", Q + "<544,1,1>", U8, "hwc", 3, 64, 1024, 1024, 1024, 1024, 0, "full"),
    ("q9-m2-full", Q + "<544,1,2>", U8, "hwc", 3, 64, 1024, 1026, 1024, 1023, 0, "full"),
    ("c3-m1", Q + "<384,1,1>", U8, "hwc", 3, 64, 1344, 1344, 1344, 1344, 0, "full"),
    ("c3-m2", Q + "<384,1,2>", U8, "hwc", 3, 64, 1344, 1344, 1344, 1343, 0, "full"),
    ("q12-m1-full", Q + "<416,1,1>", U8, "hwc", 3, 48, 1500, 1500, 1500, 1500, 0, "full"),
    ("q12-m2-full", Q + "<416,1,2>", U8, "hwc", 3, 48, 1500, 1502, 1500, 1499, 0, "full"),
    ("q16-m1-full", Q + "<544,1,1>", U8, "hwc", 3, 32, 1024, 2048, 1024, 2048, 0, "full"),
    ("q16-m2-full", Q + "<544,1,2>", U8, "hwc", 3, 32, 1024, 2046, 1024, 2030, 0, "full"),
    # several strips per row: CTA ranges cross strip boundaries, MODE 2 strips after the first compute their halo
    ("q9-m1-2strips-full", Q + "<544,1,1>", U8, "hwc", 3, 32, 512, 2052, 512, 2052, 0, "full"),
    ("q11-m1-3strips-full", Q + "<384,1,1>", U8, "hwc", 3, 12, 512, 4100, 512, 4100, 0, "full"),
    ("q9-m2-2strips-full", Q + "<544,1,2>", U8, "hwc", 3, 32, 512, 2033, 512, 2033, 0, "full"),
    ("q9-m2-2strips-2049-full", Q + "<544,1,2>", U8, "hwc", 3, 32, 512, 2049, 512, 2049, 0, "full"),
    # streaming uint8 kernel: grey, planar (B x C planes sharing their image's maps) and RGBA
    ("s1-hwc-small", "remap_u8_stream_kernel<1,16,2>", U8, "hwc", 1, 3, 90, 100, 64, 80, 0, "small"),
    ("s1-hwc-full", "remap_u8_stream_kernel<1,16,2>", U8, "hwc", 1, 256, 336, 336, 336, 336, 0, "full"),
    ("s1-chw-small", "remap_u8_stream_kernel<1,16,2>", U8, "chw", 3, 2, 90, 100, 40, 80, 0, "small"),
    ("s1-chw-full", "remap_u8_stream_kernel<1,16,2>", U8, "chw", 3, 256, 336, 336, 336, 336, 0, "full"),
    ("s4-small", "remap_u8_stream_kernel<4,16,1>", U8, "hwc", 4, 3, 90, 100, 40, 80, 0, "small"),
    ("s4-full", "remap_u8_stream_kernel<4,16,1>", U8, "hwc", 4, 256, 336, 336, 336, 336, 1, "full"),
    # float32 streaming kernel: the geometry follows Wo * E (<= 512, <= 1024, above)
    ("f160-small", "remap_f32_stream_kernel<160,4>", F32, "chw", 3, 2, 64, 64, 40, 60, 0, "small"),
    ("f160-c5", "remap_f32_stream_kernel<160,4>", F32, "chw", 3, 128, 512, 512, 512, 512, 0, "full"),
    ("f288-small", "remap_f32_stream_kernel<288,2>", F32, "hwc", 3, 2, 60, 300, 50, 336, 0, "small"),
    ("f288-full", "remap_f32_stream_kernel<288,2>", F32, "hwc", 3, 64, 336, 336, 336, 336, 1, "full"),
    ("f416-small", "remap_f32_stream_kernel<416,1>", F32, "hwc", 3, 1, 60, 1344, 40, 1344, 0, "small"),
    ("f416-full", "remap_f32_stream_kernel<416,1>", F32, "hwc", 3, 16, 1344, 1344, 1344, 1344, 0, "full"),
    # fallbacks reached by their natural routes: 1-pixel source axes, more than 65535 planes, a 1 GiB float32 plane
    ("direct-u8-hwc-h1", "remap_direct_kernel<unsigned char,true>", U8, "hwc", 3, 256, 1, 300, 20, 200, 0, "direct"),
    ("direct-u8-chw-w1", "remap_direct_kernel<unsigned char,false>", U8, "chw", 3, 256, 300, 1, 200, 20, 0, "direct"),
    ("direct-u8-65538-planes", "remap_direct_kernel<unsigned char,false>", U8, "chw", 3, 21846, 8, 8, 8, 8, 0,
     "direct"),
    ("rows-f32-1gib", "remap_f32_rows_kernel<true>", F32, "hwc", 1, 1, 64, 64, 16384, 16384, 0, "rows"),
]
CASE_IDS = [c[0] for c in CASES]

# instances reached only through a process-wide switch (ENV_RUNS)
SWITCH_KERNELS = ("remap_direct_kernel<float,true>", "remap_direct_kernel<float,false>", "remap_f32_rows_kernel<false>",
                  "remap_u8_stream_kernel<3,16,2>", "remap_u8_stream_kernel<3,16,1>", "remap_u8_stream_kernel<1,16,1>")

BASE_NAMES = ("remap_u8_quad_kernel", "remap_u8_stream_kernel", "remap_f32_stream_kernel", "remap_f32_rows_kernel",
              "remap_direct_kernel")
KERNEL_RE = re.compile(r"(?<![A-Za-z_])(" + "|".join(BASE_NAMES) + r")(?![A-Za-z_])(<[^>]*>)?")

FAMILIES = ("tokens", "tokens_cubed", "identity", "ties", "shuffled", "jumps", "magnify", "outside", "flat_runs")


def _norm(name):
    return re.sub(r"\s+", "", name)


def _stage5_kernels(names):
    """The stage-5 kernel instances in a list of (possibly mangled) symbol names, without spaces."""
    tool = shutil.which("c++filt") or shutil.which("cu++filt")
    if tool is not None and names:
        names = subprocess.run([tool], input="\n".join(names) + "\n", capture_output=True, text=True,
                               check=True).stdout.splitlines()
    return [_norm(m.group(0)) for n in names for m in KERNEL_RE.finditer(n)]


# ---------------------------------------------------------------------------------------------- launch geometry
def plan_strips(Wo, max_cols):
    n = -(-Wo // max_cols)
    cols = (-(-Wo // n) + 15) & ~15
    return -(-Wo // cols), cols


def quad_max_cols(aligned):
    return 16 * (128 if aligned else 127) & ~15


def quad_build(cols, aligned):
    """launch_direct_mode: (instance, consumer warps, CTAs per SM wanted) for strips of ``cols`` columns."""
    w = max(3, -(-cols // (128 if aligned else 127)))
    m = 1 if aligned else 2
    if w <= 3:
        return f"{Q}<128,5,{m}>", w, 4
    if w <= 6:
        return f"{Q}<224,2,{m}>", w, 3 if w == 4 else 2
    if w <= 9:
        return f"{Q}<544,1,{m}>", w, 2
    if w <= 11:
        return f"{Q}<384,1,{m}>", w, 1
    if w <= 12:
        return f"{Q}<416,1,{m}>", w, 1
    return f"{Q}<544,1,{m}>", w, 1


def quad_rows(cols, warps, ctas, stages=2):
    """launch_core: rows per chunk of the quad kernel (the shared memory of 1 / ctas of an SM, at most 30)."""
    tab = 64 + 16 * 31
    unit_pitch = (((cols + 1) * 3 + 45 + 15) & ~15) + 16
    budget = (227 * 1024) // ctas - 1024 - stages * tab - 16 * 4 - 256 - (1024 * warps + 16)
    return min((budget - stages * (2 * unit_pitch + 64 + 128)) // (stages * unit_pitch), 30)


def quad_uniform(Wo, lead_bytes):
    """(instance, block, CTAs per SM wanted, rows per chunk, strips) of a uniform 3-channel batch."""
    aligned = ((lead_bytes | (Wo * 3)) & 3) == 0
    n, sc = plan_strips(Wo, quad_max_cols(aligned))
    cols = min(Wo, sc)
    name, w, ctas = quad_build(cols, aligned)
    return name, (w + 1) * 32, ctas, quad_rows(cols, w, ctas), n


def work_units(case):
    """Units the launch splits over its CTAs: output rows x strips (x planes)."""
    _, kern, dt, lay, C, B, H, W, Ho, Wo, lead, _ = case
    planes = B * C if lay == "chw" else B
    if kern.startswith(Q):
        return B * quad_uniform(Wo, lead)[4] * Ho
    if kern.startswith("remap_u8_stream"):
        return planes * plan_strips(Wo, 352)[0] * Ho
    if kern.startswith("remap_f32_stream"):
        E = C if lay == "hwc" else 1
        max_el = 512 if Wo * E <= 512 else (1024 if Wo * E <= 1024 else 1536)
        px = max_el // E
        strip_px = -(-Wo // -(-Wo // px))
        return planes * -(-Wo // strip_px) * Ho
    return None


def chunk_rows(case):
    """Output rows a CTA's first chunks and three full chunks take (a full row must give every CTA at least these)."""
    kern, lead, Wo = case[1], case[10], case[9]
    if kern.startswith(Q):
        R = quad_uniform(Wo, lead)[3]
        return 8 + min(16, R) + 3 * R
    return 3 * 16                          # 16-row chunks of the streaming kernels


def check_geometry(case, grid, block, sms):
    """None if the launch has the case's geometry class, else why not."""
    _, kern, dt, lay, C, B, H, W, Ho, Wo, lead, geo = case
    gx, gy, gz = (list(grid) + [1, 1, 1])[:3]
    if kern.startswith(Q):
        want_block = quad_uniform(Wo, lead)[1]
        if block and block[0] != want_block:
            return f"block {block[0]}, not (warps + 1) * 32 = {want_block}"
    if geo == "direct":
        ok = (gx, gy, gz) == (-(-Wo // 256), Ho, B)
        return None if ok else f"grid {grid}, not (ceil(Wo / 256), Ho, B) = {(-(-Wo // 256), Ho, B)}"
    if geo == "rows":
        planes = B if lay == "hwc" else B * C
        return None if gz == planes else f"grid {grid}, not one plane of the grid per image plane ({planes})"
    units = work_units(case)
    if geo == "small":
        return None if gx == units else f"grid {gx}, not one CTA per work unit ({units})"
    if not (gx < units and gx % sms == 0):
        return f"grid {gx} is not a persistent grid (multiple of {sms} SMs, below {units} units)"
    if units // gx < chunk_rows(case):
        return f"{units // gx} rows per CTA, fewer than three full chunks ({chunk_rows(case)})"
    return None


def _launches(prof, path):
    """(kernel name, grid, block) of every stage-5 launch in the profile's chrome trace."""
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f).get("traceEvents", [])
    out = []
    for e in events:
        if e.get("cat") == "kernel":
            names = _stage5_kernels([e.get("name", "")])
            if names:
                args = e.get("args", {})
                out.append((names[0], tuple(args.get("grid", ())), tuple(args.get("block", ()))))
    return out


def _profiled(fn, path):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                            torch.profiler.ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, _launches(prof, path)


# ---------------------------------------------------------------------------------------------- ragged planner
def plan_ragged(images, min_px=24000000, min_aligned_px=32000000):
    """launch_remap_u8_quad_ragged_prepare's classes, restated.  images: (Ho, Wo, destination address) per image.
    Returns the launches in issue order (biggest class first): dicts of class, instance, block, count, units, px."""
    K = 14
    px = [0] * 2 * K
    cls = []
    for Ho, Wo, addr in images:
        aligned = ((addr | (Wo * 3)) & 3) == 0
        _, sc = plan_strips(Wo, quad_max_cols(aligned))
        c = quad_build(min(Wo, sc), aligned)[1] - 3 + (0 if aligned else K)
        cls.append(c)
        px[c] += Ho * Wo
    join = list(range(2 * K))
    for c in range(K):
        if px[c] == 0 or px[c] >= min_aligned_px or px[c + K] == 0:
            continue
        px[c + K] += px[c]
        px[c] = 0
        join[c] = c + K
    for half in range(2):
        c0, c1 = half * K, half * K + K
        for c in range(c0, c1 - 1):
            if px[c] == 0 or px[c] >= min_px:
                continue
            up = c + 1
            while up < c1 and px[up] == 0:
                up += 1
            if up == c1:
                continue
            px[up] += px[c]
            px[c] = 0
            join[c] = up
    classes = {}
    for (Ho, Wo, addr), c in zip(images, cls):
        while join[c] != c:
            c = join[c]
        aligned = c < K
        n, sc = plan_strips(Wo, quad_max_cols(aligned))
        cols = min(Wo, sc)
        d = classes.setdefault(c, {"class": c, "count": 0, "units": 0, "max_strip": 0, "px": 0})
        d["count"] += 1
        d["units"] += n * Ho * -(-cols // (128 if aligned else 127))
        d["max_strip"] = max(d["max_strip"], cols)
        d["px"] += Ho * Wo
    out = []
    for c, d in classes.items():
        name, w, _ = quad_build(d["max_strip"], c < K)
        out.append(dict(d, kernel=name, block=(w + 1) * 32))
    return sorted(out, key=lambda d: (-d["units"], d["class"]))


# ---------------------------------------------------------------------------------------------- reference
def _quant(m):
    s = torch.round(m.to(torch.float32) * 32.0).to(torch.int64)      # rint, half to even
    return s >> 5, s & 31


def _ref_piece(img, mx, my):
    """img [n, H, W, C]; mx [n, Wo], my [n, h] -> [n, h, Wo, C]"""
    n, H, W, C = img.shape
    ix, ax = _quant(mx)
    iy, ay = _quant(my)
    x0, x1 = ix.clamp(0, W - 1), (ix + 1).clamp(0, W - 1)
    y0, y1 = iy.clamp(0, H - 1), (iy + 1).clamp(0, H - 1)
    b = torch.arange(n, device=img.device)[:, None, None]
    X0, X1, Y0, Y1 = x0[:, None, :], x1[:, None, :], y0[:, :, None], y1[:, :, None]
    p00, p01, p10, p11 = img[b, Y0, X0], img[b, Y0, X1], img[b, Y1, X0], img[b, Y1, X1]
    wx, wy = ax[:, None, :, None], ay[:, :, None, None]
    if img.dtype == U8:
        p00, p01, p10, p11 = (p.to(torch.int64) for p in (p00, p01, p10, p11))
        acc = 32 * ((32 - wx) * (32 - wy) * p00 + wx * (32 - wy) * p01 + (32 - wx) * wy * p10 + wx * wy * p11)
        return ((acc + (1 << 14)) >> 15).to(U8)
    fx = wx.to(F32) * 0.03125
    fy = wy.to(F32) * 0.03125
    w00 = (1.0 - fy) * (1.0 - fx)
    w01 = (1.0 - fy) * fx
    w10 = fy * (1.0 - fx)
    w11 = fy * fx
    t = p00 * w00                          # one op per multiply and add: nothing is contracted
    t = t + p01 * w01
    t = t + p10 * w10
    return t + p11 * w11


def ref_remap(img, mx, my, limit=1 << 25):
    """img [B, H, W, C] uint8 / float32, maps float32 [B, Wo], [B, Ho] -> [B, Ho, Wo, C], oracle.numpy_path.remap
    restated in torch (runs on the CPU or the device), in pieces of at most ``limit`` output elements."""
    B, H, W, C = img.shape
    Ho, Wo = my.shape[1], mx.shape[1]
    out = torch.empty((B, Ho, Wo, C), dtype=img.dtype, device=img.device)
    per_img = Ho * Wo * C
    if per_img <= limit:
        step = max(1, limit // per_img)
        for b0 in range(0, B, step):
            out[b0:b0 + step] = _ref_piece(img[b0:b0 + step], mx[b0:b0 + step], my[b0:b0 + step])
    else:
        rows = max(1, limit // (Wo * C))
        for b in range(B):
            for y0 in range(0, Ho, rows):
                out[b:b + 1, y0:y0 + rows] = _ref_piece(img[b:b + 1], mx[b:b + 1], my[b:b + 1, y0:y0 + rows])
    return out


def _bits(t):
    return t.view(torch.int32) if t.dtype == F32 else t


def compare(got, ref, img, mx, my, what, launches=()):
    """got / ref [B, Ho, Wo, C]: bit-equal, else the first differing (image, y, x, channel) with its taps."""
    diff = _bits(got) != _bits(ref)
    if not bool(diff.any()):
        return
    n_bad = int(diff.sum())
    flat = int(torch.argmax(diff.reshape(-1).to(torch.uint8)))
    B, Ho, Wo, C = got.shape
    b, y, x, c = flat // (Ho * Wo * C), flat // (Wo * C) % Ho, flat // C % Wo, flat % C
    H, W = img.shape[1:3]
    sx = int(torch.round(mx[b, x].float() * 32)), float(mx[b, x])
    sy = int(torch.round(my[b, y].float() * 32)), float(my[b, y])
    x0, x1 = min(max(sx[0] >> 5, 0), W - 1), min(max((sx[0] >> 5) + 1, 0), W - 1)
    y0, y1 = min(max(sy[0] >> 5, 0), H - 1), min(max((sy[0] >> 5) + 1, 0), H - 1)
    taps = [img[b, yy, xx, c].item() for yy in (y0, y1) for xx in (x0, x1)]
    raise AssertionError(
        f"{what}: {n_bad} of {diff.numel()} output elements differ from the reference; first at image {b}, y {y}, "
        f"x {x}, channel {c}: got {got[b, y, x, c].item()!r}, ref {ref[b, y, x, c].item()!r}; map_x {sx[1]!r} "
        f"(x taps {x0}, {x1}, weight {sx[0] & 31}/32), map_y {sy[1]!r} (y taps {y0}, {y1}, weight {sy[0] & 31}/32), "
        f"source p00 p01 p10 p11 = {taps}; launched {list(launches)}")


# ---------------------------------------------------------------------------------------------- inputs
def axis_map(family, n_out, n_src, rng):
    """One axis of a map family (float32 [n_out]) for a source axis of n_src pixels."""
    lin = np.linspace(0, n_src - 1, n_out)
    if family == "identity":
        m = np.arange(n_out) if n_out == n_src else lin
    elif family == "ties":                 # exactly on 1/32-pixel ties: rint rounds half to even
        m = (np.round(np.linspace(0, max((n_src - 1) * 32 - 1, 0), n_out)) + 0.5) / 32
    elif family == "shuffled":             # non-monotone: one-row chunks, lane mapping
        m = rng.permutation(lin)
    elif family == "jumps":                # 7.4 source pixels per output pixel: chunks cut by the stage size
        m = (np.arange(n_out) * 7.37 + rng.uniform(0, n_src)) % max(n_src - 1, 1)
    elif family == "magnify":              # every output pixel on 3 source pixels: pairs carried across chunks
        m = rng.uniform(0, max(n_src - 3, 0)) + np.linspace(0, min(2.5, n_src - 1), n_out)
    elif family == "outside":              # up to 4 image sizes outside on both sides, some rows inside
        m = np.linspace(-4.0 * n_src, 4.0 * n_src, n_out)
        k = rng.integers(0, n_out, n_out // 8)
        m[k] = rng.uniform(-4.0 * n_src, 4.0 * n_src, len(k))
    elif family == "flat_runs":            # runs of one value, then a jump either way
        runs = rng.integers(1, 40, n_out)
        vals = rng.uniform(-2, n_src + 1, n_out)
        m = np.repeat(vals, runs)[:n_out]
    else:
        raise ValueError(family)
    return np.asarray(m, dtype=np.float32)


def make_maps(B, H, W, Ho, Wo, seed, shift=0, device="cuda"):
    """map_x [B, Wo], map_y [B, Ho]: image b takes family FAMILIES[(b + shift) % len]; token maps come from
    ops.maps_from_tokens on random and rand^3 24 x 24 token grids."""
    rng = np.random.default_rng(seed)
    fams = [FAMILIES[(b + shift) % len(FAMILIES)] for b in range(B)]
    mx = np.empty((B, Wo), np.float32)
    my = np.empty((B, Ho), np.float32)
    for b, f in enumerate(fams):
        if not f.startswith("tokens"):
            mx[b] = axis_map(f, Wo, W, rng)
            my[b] = axis_map(f, Ho, H, rng)
    mx, my = torch.from_numpy(mx).to(device), torch.from_numpy(my).to(device)
    tb = [b for b, f in enumerate(fams) if f.startswith("tokens")]
    if tb and H >= 1 and W >= 1:
        from attwarp_b200 import ops
        tok = rng.random((len(tb), min(24, H), min(24, W)), dtype=np.float32)
        cubed = np.array([fams[b] == "tokens_cubed" for b in tb])
        tok[cubed] **= 3
        tx, ty = ops.maps_from_tokens(torch.from_numpy(tok).to(device), (H, W), (Ho, Wo))
        mx[tb], my[tb] = tx, ty
    return mx, my, fams


def make_image(kind, shape_hwc, dtype, seed, device="cuda"):
    """[B, H, W, C]: uniform random values, or coordinate-coded (channel 0 = x & 255, 1 = y & 255,
    2 = (x >> 8) ^ (y >> 8), 3 = (x + y) & 255; float32: x, y, x ^ y, x + y)."""
    B, H, W, C = shape_hwc
    if kind == "random":
        g = torch.Generator(device=device).manual_seed(seed)
        if dtype == U8:
            return torch.randint(0, 256, shape_hwc, generator=g, dtype=U8, device=device)
        return torch.rand(shape_hwc, generator=g, dtype=F32, device=device)
    y = torch.arange(H, device=device)[:, None].expand(H, W)
    x = torch.arange(W, device=device)[None, :].expand(H, W)
    if dtype == U8:
        planes = [x & 255, y & 255, (x >> 8) ^ (y >> 8), (x + y) & 255]
    else:
        planes = [x, y, x ^ y, x + y]
    img = torch.stack([planes[c % 4] for c in range(C)], -1).to(dtype)
    return img[None].expand(B, H, W, C).contiguous()


def guarded(numel, dtype, lead, device="cuda"):
    """(flat buffer filled with the guard, view of ``numel`` elements starting PAD + lead elements in)."""
    flat = torch.full((PAD + lead + numel + PAD,), GUARD_U8 if dtype == U8 else float("nan"), dtype=dtype,
                      device=device)
    return flat, flat[PAD + lead:PAD + lead + numel]


def check_guards(flat, spans, dtype, what):
    """Every element of ``flat`` outside the (start, end) spans still holds the guard."""
    keep = torch.ones(flat.numel(), dtype=torch.bool, device=flat.device)
    for s, e in spans:
        keep[s:e] = False
    g = flat[keep]
    ok = bool((g == GUARD_U8).all()) if dtype == U8 else bool(torch.isnan(g).all())
    if not ok:
        bad = (g != GUARD_U8) if dtype == U8 else ~torch.isnan(g)
        raise AssertionError(f"{what}: {int(bad.sum())} guard elements overwritten")


def run_uniform(case, img_hwc, mx, my):
    """remap_bilinear on the case's layout into a guarded output -> (output as [B, Ho, Wo, C], flat, span)."""
    from attwarp_b200 import ops
    _, kern, dt, lay, C, B, H, W, Ho, Wo, lead, _ = case
    img = img_hwc if lay == "hwc" else img_hwc.permute(0, 3, 1, 2).contiguous()
    shape = (B, Ho, Wo, C) if lay == "hwc" else (B, C, Ho, Wo)
    numel = B * Ho * Wo * C
    flat, view = guarded(numel, dt, lead)
    out = view.view(shape)
    ops.remap_bilinear(img, mx, my, layout=lay, out=out)
    got = out if lay == "hwc" else out.permute(0, 2, 3, 1)
    return got, flat, (PAD + lead, PAD + lead + numel)


def sm_count():
    from attwarp_b200 import _lib
    sm, ma, mi = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    _lib.check(_lib.load().attwarp_device_info(ctypes.byref(sm), ctypes.byref(ma), ctypes.byref(mi)))
    return sm.value


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


# ---------------------------------------------------------------------------------------------- CPU
def test_case_table_names_every_compiled_kernel():
    """The stage-5 instances in the built library are exactly those CASES and the switch runs name: a new instance
    without a row fails here, and so does a row whose kernel is no longer compiled."""
    from attwarp_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(cuobjdump):
        pytest.skip("cuobjdump not available")
    assert os.path.isfile(_lib.lib_path()), "build the library first: python -m attwarp_b200.build"
    out = subprocess.run([cuobjdump, "-symbols", _lib.lib_path()], capture_output=True, text=True, check=True).stdout
    compiled = set(_stage5_kernels(out.splitlines()))
    named = {_norm(c[1]) for c in CASES} | {_norm(k) for k in SWITCH_KERNELS}
    assert {_norm(k) for r in ENV_RUNS for k in r["kernels"]} <= named
    print(f"\n{len(compiled)} stage-5 kernel instances in the library:\n  " + "\n  ".join(sorted(compiled)))
    assert len(compiled) == 24
    assert compiled == named, f"compiled but no case: {sorted(compiled - named)}; named but not compiled: {sorted(named - compiled)}"


def test_case_table_rows():
    """Every quad build x MODE has a small and a full row (<224,2> and <544,1> in both of their CTA-per-SM
    configurations), every float32 streaming geometry and uint8 streaming instance has both, the quad rows launch the
    build the launcher picks, and full rows give every CTA of a B200 grid at least three full chunks."""
    assert len(set(CASE_IDS)) == len(CASE_IDS)
    seen = {}
    for case in CASES:
        cid, kern, dt, lay, C, B, H, W, Ho, Wo, lead, geo = case
        key = _norm(kern)
        if kern.startswith(Q):
            name, block, ctas, R, _ = quad_uniform(Wo, lead)
            assert _norm(name) == key, f"{cid}: the launcher picks {name}"
            assert R >= 2
            key += f"@{ctas}"
            if geo == "full":
                assert work_units(case) // (SMS_B200 * ctas) >= chunk_rows(case), cid
            else:
                assert work_units(case) <= SMS_B200 * ctas, cid
        seen.setdefault(key, set()).add(geo)
    quad = [k for k in seen if k.startswith(Q)]
    assert len(quad) == 14                 # 5 builds, <224,2> and <544,1> at two CTA counts, x 2 MODEs
    for k, geos in seen.items():
        if k.startswith((Q, "remap_u8_stream", "remap_f32_stream")):
            assert {"small", "full"} <= geos, k


def test_ragged_planner_hand_tables():
    """plan_ragged on tables small enough to work out by hand."""
    # a 300- and a 700-column image, both aligned, far below 24 M pixels: the 3-warp class joins the 6-warp one
    p = plan_ragged([(300, 300, 0), (700, 700, 0)])
    assert [(d["class"], d["kernel"], d["block"], d["count"]) for d in p] == [(3, Q + "<224,2,1>", 224, 2)]
    assert p[0]["units"] == 300 * 3 + 700 * 6
    # the same images with the class threshold off: two launches, biggest first
    p = plan_ragged([(300, 300, 0), (700, 700, 0)], min_px=0)
    assert [(d["class"], d["kernel"], d["count"]) for d in p] == [(3, Q + "<224,2,1>", 1), (0, Q + "<128,5,1>", 1)]
    # an aligned 384-column image next to an unaligned 380-column one joins it (MODE 2 then needs 4 warps for 384)
    p = plan_ragged([(10, 384, 0), (10, 380, 1)])
    assert [(d["class"], d["kernel"], d["block"], d["count"], d["max_strip"]) for d in p] == \
        [(14, Q + "<224,2,2>", 160, 2, 384)]
    # without an unaligned sibling of its width the aligned class stays MODE 1
    p = plan_ragged([(10, 384, 0), (10, 700, 1)])
    assert [(d["class"], d["kernel"]) for d in p] == [(17, Q + "<224,2,2>"), (0, Q + "<128,5,1>")]
    # 4100 columns, aligned: three strips of 1376 columns (11 warps) per row
    p = plan_ragged([(5, 4100, 0)])
    assert [(d["class"], d["kernel"], d["units"], d["max_strip"]) for d in p] == [(8, Q + "<384,1,1>", 5 * 3 * 11, 1376)]


def test_device_reference_equals_oracle():
    """ref_remap (torch, here on the CPU) equals oracle.numpy_path.remap on every map family, uint8 and float32, 1, 3
    and 4 channels, and cv2.remap on the meshgrid of a few of them."""
    rng = np.random.default_rng(7)
    fams = [f for f in FAMILIES if not f.startswith("tokens")]
    for k, (H, W, Ho, Wo, C) in enumerate([(37, 53, 41, 29, 3), (16, 90, 33, 45, 1), (50, 20, 17, 64, 4)]):
        for dt in (U8, F32):
            imgs = make_image("random", (1, H, W, C), dt, k, device="cpu")[0].numpy()
            for f in fams + ["production"]:
                if f == "production":
                    att = rng.random((H, W)).astype(np.float32) ** 3
                    mx, my, _, _ = ON.inverse_maps(att, Wo, Ho, "identity")
                    mx, my = np.asarray(mx, np.float32), np.asarray(my, np.float32)
                else:
                    mx, my = axis_map(f, Wo, W, rng), axis_map(f, Ho, H, rng)
                ref = ON.remap(imgs, mx, my)
                got = ref_remap(torch.from_numpy(imgs)[None], torch.from_numpy(mx)[None],
                                torch.from_numpy(my)[None])[0].numpy()
                assert np.array_equal(got.view(np.uint8), ref.reshape(got.shape).view(np.uint8)), (f, dt, H, W)
                if f in ("identity", "ties", "shuffled", "production") and C != 4:
                    cv = ON.remap_cv2(imgs, mx, my)
                    assert np.array_equal(got.reshape(cv.shape).view(np.uint8), cv.view(np.uint8)), ("cv2", f, dt)


# ---------------------------------------------------------------------------------------------- GPU: case table
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_kernel_bit_exact(case, tmp_path):
    """One row of CASES: every output element bit-equal to the reference on random and coordinate-coded inputs,
    with every map family, guards intact, and the launch of the instance, block and geometry class the row names."""
    _need_gpu()
    row = CASES[case]
    cid, kern, dt, lay, C, B, H, W, Ho, Wo, lead, geo = row
    rounds = max(1, -(-len(FAMILIES) // B)) if geo == "small" else 1
    launched = None
    for kind in ("random", "coded"):
        img = make_image(kind, (B, H, W, C), dt, 100 + case)
        for r in range(rounds):
            mx, my, fams = make_maps(B, H, W, Ho, Wo, 1000 * case + r, shift=r * B + (kind == "coded") * 4)
            what = f"{cid} ({kern}) {kind} input"
            if launched is None:
                (got, flat, span), launched = _profiled(lambda: run_uniform(row, img, mx, my), tmp_path / "t.json")
            else:
                got, flat, span = run_uniform(row, img, mx, my)
            check_guards(flat, [span], dt, what)
            ref = ref_remap(img, mx, my)
            compare(got, ref, img, mx, my, what + f" (families of images 0..: {fams[:4]})", launched)
            del got, flat, ref
    if not launched:
        pytest.skip("torch.profiler reported no CUDA kernel events: the launched kernel and its geometry are not checked")
    names = [n for n, _, _ in launched]
    assert names == [_norm(kern)], f"{cid}: expected {kern}, launched {names}"
    _, grid, block = launched[0]
    if not grid:
        pytest.skip(f"{cid}: the trace has no grid for the launch: its geometry is not checked")
    why = check_geometry(row, grid, block, sm_count())
    assert why is None, f"{cid}: {kern} launched grid {grid} block {block}: {why}"


# ---------------------------------------------------------------------------------------------- GPU: chunk and grid sweeps
SWEEP_CASES = [("q6-m1-full", Q + "<224,2,1>", U8, "hwc", 3, 128, 700, 700, 700, 700, 0, "full"),
               ("q6-m2-full", Q + "<224,2,2>", U8, "hwc", 3, 128, 700, 700, 700, 701, 0, "full")]


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(SWEEP_CASES)), ids=[c[0] for c in SWEEP_CASES])
def test_chunk_and_grid_sweeps(case, monkeypatch, tmp_path):
    """One full MODE 1 and one full MODE 2 batch (128 x 700^2, shuffled and production maps among the families) under
    every CTA count, chunk height, first-chunk height, ring depth, row-mapping policy and SM share: each variant
    bit-equal to the reference.  These put chunk and CTA boundaries at every row phase of the same batch."""
    _need_gpu()
    from attwarp_b200 import _lib
    row = SWEEP_CASES[case]
    cid, kern, dt, lay, C, B, H, W, Ho, Wo, lead, geo = row
    img = make_image("coded", (B, H, W, C), dt, 7)
    mx, my, _ = make_maps(B, H, W, Ho, Wo, 77)
    ref = ref_remap(img, mx, my)
    name, block, ctas, R, _ = quad_uniform(Wo, lead)
    sms = sm_count()
    variants = [("ATTWARP_REMAP_CTAS_PER_SM", str(v)) for v in range(1, ctas + 1)]
    variants += [("ATTWARP_QUAD_ROWS", str(v)) for v in (2, 3, 7, R)]
    variants += [("ATTWARP_QUAD_FIRST_ROWS", str(v)) for v in (1, 8, 13)]
    variants += [("ATTWARP_QUAD_RING", str(v)) for v in (2, 3, 4)]
    variants += [("ATTWARP_QUAD_MAP", str(v)) for v in (0, 1, 2)]
    variants += [("sm_share", "2")]
    for var, val in variants:
        lib = _lib.load()
        with monkeypatch.context() as mp:
            if var == "sm_share":
                prev = lib.attwarp_set_sm_share(2)
            else:
                mp.setenv(var, val)
            try:
                (got, flat, span), launched = _profiled(lambda: run_uniform(row, img, mx, my), tmp_path / "t.json")
            finally:
                if var == "sm_share":
                    lib.attwarp_set_sm_share(prev)
        what = f"{cid} with {var}={val}"
        check_guards(flat, [span], dt, what)
        compare(got, ref, img, mx, my, what, launched)
        assert [n for n, _, _ in launched] in ([_norm(kern)], []), (what, launched)
        if var == "ATTWARP_REMAP_CTAS_PER_SM" and launched and launched[0][1]:
            assert launched[0][1][0] == sms * int(val), (what, launched)


# ---------------------------------------------------------------------------------------------- GPU: mixed-size lists
def ragged_outputs(sizes, C, offsets):
    """Guarded outputs carved from one flat buffer, at least PAD guard bytes apart: image i starts offsets[i] bytes
    past a 4-byte boundary -> (flat, outs, spans)."""
    starts, pos = [], 0
    for (ho, wo), off in zip(sizes, offsets):
        pos = ((pos + PAD + 3) & ~3) + off
        starts.append(pos)
        pos += ho * wo * C
    flat = torch.full((pos + PAD,), GUARD_U8, dtype=U8, device="cuda")
    outs = [flat[s:s + ho * wo * C].view(ho, wo, C) for s, (ho, wo) in zip(starts, sizes)]
    return flat, outs, [(s, s + ho * wo * C) for s, (ho, wo) in zip(starts, sizes)]


def attention_map(family, H, W, g):
    if family == "uniform":
        return torch.full((H, W), 77, dtype=U8, device="cuda")
    if family == "random":
        return torch.randint(0, 256, (H, W), generator=g, dtype=U8, device="cuda")
    a = torch.zeros((H, W), dtype=U8, device="cuda")
    if family == "hot_column":
        a[:, int(torch.randint(0, W, (1,), generator=g, device="cuda"))] = 255
    else:
        a[int(torch.randint(0, H, (1,), generator=g, device="cuda"))] = 255
    return a


def run_ragged(sizes, out_sizes, C, offsets, seed, kind="random"):
    """warp_ragged_from_attention on a list -> (imgs, outs, map_xs, map_ys, flat, spans)."""
    from attwarp_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(seed)
    fams = ("random", "uniform", "hot_column", "hot_row")
    imgs = [make_image(kind, (1, h, w, C), U8, seed + i)[0] for i, (h, w) in enumerate(sizes)]
    att = [attention_map(fams[i % 4], h, w, g) for i, (h, w) in enumerate(sizes)]
    flat, outs, spans = ragged_outputs(out_sizes, C, offsets)
    _, mxs, mys = ops.warp_ragged_from_attention(att, imgs, out_sizes, outs=outs, return_maps=True)
    return imgs, outs, mxs, mys, flat, spans


def check_ragged(imgs, outs, mxs, mys, flat, spans, what, launched=()):
    check_guards(flat, spans, U8, what)
    for i, (im, o, mx, my) in enumerate(zip(imgs, outs, mxs, mys)):
        ref = ref_remap(im[None], mx[None], my[None])
        compare(o[None], ref, im[None], mx[None], my[None], f"{what}, image {i} {tuple(im.shape)} -> {tuple(o.shape)}",
                launched)


def _addresses(outs):
    return [(o.shape[0], o.shape[1], o.data_ptr()) for o in outs]


def _check_plan(outs, launched, what, **kw):
    from attwarp_b200 import _lib
    plan = plan_ragged(_addresses(outs), **kw)
    got = sorted((n, b[0] if b else None) for n, _, b in launched)
    want = sorted((_norm(d["kernel"]), d["block"]) for d in plan)
    if launched:
        if not all(b for _, _, b in launched):
            want = sorted((n, None) for n, _ in want)
        assert got == want, f"{what}: launched {got}, the restated planner predicts {want}"
    assert _lib.load().attwarp_ragged_last_launches() - 2 == len(plan), what
    return plan


@pytest.mark.gpu
def test_ragged_configs3_like_list(tmp_path):
    """1024 images with sides uniform in [224, 2048] (BASELINE configs[3]), each output 0 - 3 bytes off its 4-byte
    boundary, warped by uint8 attention maps (random, uniform, one hot column or row): every image bit-equal to the
    reference on the maps the call returns, the launches those of the restated planner, and classes past both
    join thresholds."""
    _need_gpu()
    rng = np.random.default_rng(3)
    n = 1024
    sizes = [tuple(int(v) for v in rng.integers(224, 2049, 2)) for _ in range(n)]
    out_sizes = [s if i % 2 else tuple(int(v) for v in rng.integers(224, 2049, 2)) for i, s in enumerate(sizes)]
    offsets = [int(v) for v in rng.integers(0, 4, n)]
    res, launched = _profiled(lambda: run_ragged(sizes, out_sizes, 3, offsets, 11), tmp_path / "t.json")
    imgs, outs, mxs, mys, flat, spans = res
    plan = _check_plan(outs, launched, "configs[3]-like list")
    assert max(d["px"] for d in plan) >= 32000000, plan
    check_ragged(imgs, outs, mxs, mys, flat, spans, "configs[3]-like list", launched)


def _threshold_list(kind):
    """(sizes, offsets): one class just below or just above a join threshold.
    below24 / above24: 384 x 384 aligned images (3 warps) of 23.9 M / 24.2 M pixels next to 600-column ones;
    below32 / above32: 384 x 384 aligned images of 31.9 M / 32.1 M pixels next to unaligned 380-column ones."""
    n384 = {"below24": 162, "above24": 164, "below32": 216, "above32": 218}[kind]
    sizes = [(384, 384)] * n384
    offsets = [0] * n384
    if kind.endswith("24"):
        sizes += [(300, 600)] * 4
        offsets += [0] * 4
    else:
        sizes += [(300, 380)] * 4
        offsets += [1] * 4
    return sizes, offsets


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["below24", "above24", "below32", "above32"])
def test_ragged_planner_thresholds(kind, monkeypatch, tmp_path):
    """A class just below / above the 24 M-pixel join threshold, and an aligned class just below / above the 32 M
    threshold next to a non-empty unaligned sibling: the launches (instance, block, count across all streams) are
    those of the restated planner, and the outputs stay bit-equal with ATTWARP_QUAD_CLASS_MIN_PX=0 and
    ATTWARP_RAGGED_STREAMS=1."""
    _need_gpu()
    sizes, offsets = _threshold_list(kind)
    for env in ({}, {"ATTWARP_QUAD_CLASS_MIN_PX": "0"}, {"ATTWARP_RAGGED_STREAMS": "1"}):
        with monkeypatch.context() as mp:
            for k, v in env.items():
                mp.setenv(k, v)
            res, launched = _profiled(lambda: run_ragged(sizes, sizes, 3, offsets, 21, kind="coded"),
                                      tmp_path / "t.json")
        imgs, outs, mxs, mys, flat, spans = res
        what = f"{kind} {env or 'defaults'}"
        plan = _check_plan(outs, launched, what, min_px=0 if env.get("ATTWARP_QUAD_CLASS_MIN_PX") else 24000000)
        if not env:
            joined = {"below24": True, "above24": False, "below32": True, "above32": False}[kind]
            assert len(plan) == (1 if joined else 2), (what, plan)
        check_ragged(imgs, outs, mxs, mys, flat, spans, what, launched)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [1, 4])
def test_ragged_stream_lists(C, tmp_path):
    """Grey and RGBA lists take remap_u8_stream_kernel's ragged mode: one launch over the whole list, bit-equal."""
    _need_gpu()
    rng = np.random.default_rng(30 + C)
    n = 40
    sizes = [tuple(int(v) for v in rng.integers(2, 900, 2)) for _ in range(n)]
    out_sizes = [tuple(int(v) for v in rng.integers(2, 900, 2)) for _ in range(n)]
    offsets = [int(v) for v in rng.integers(0, 4, n)]
    res, launched = _profiled(lambda: run_ragged(sizes, out_sizes, C, offsets, 31), tmp_path / "t.json")
    imgs, outs, mxs, mys, flat, spans = res
    want = "remap_u8_stream_kernel<1,16,2>" if C == 1 else "remap_u8_stream_kernel<4,16,1>"
    if launched:
        assert [n_ for n_, _, _ in launched] == [want], launched
    check_ragged(imgs, outs, mxs, mys, flat, spans, f"C = {C} list", launched)


@pytest.mark.gpu
def test_ragged_degenerate_launch_count():
    """A tokens call on a list with a 1 x N image goes through the per-image entry points: it reports 2n launches
    (maps + resample per image), not the count of the call before it."""
    _need_gpu()
    from attwarp_b200 import _lib, ops
    lib = _lib.load()
    g = torch.Generator(device="cuda").manual_seed(5)
    tok = torch.rand((3, 1, 1), generator=g, device="cuda")        # a token grid no larger than a 1 x N image
    normal = [make_image("random", (1, h, w, 3), U8, i)[0] for i, (h, w) in enumerate([(300, 300), (700, 900), (64, 64)])]
    batch = ops.RaggedBatch(normal)
    batch.run(tok)
    torch.cuda.synchronize()
    assert batch.launches == 1 + len(plan_ragged(_addresses(batch.outs)))
    degenerate = [make_image("random", (1, h, w, 3), U8, i)[0] for i, (h, w) in enumerate([(1, 57), (700, 900), (64, 1)])]
    ops.warp_ragged_from_tokens(tok, degenerate)
    torch.cuda.synchronize()
    assert lib.attwarp_ragged_last_launches() == 2 * 3
    batch.run(tok)
    assert batch.launches == 1 + len(plan_ragged(_addresses(batch.outs)))
    deg_batch = ops.RaggedBatch(degenerate)
    deg_batch.run(tok)
    torch.cuda.synchronize()
    assert deg_batch.launches == 2 * 3


# ---------------------------------------------------------------------------------------------- GPU: process-wide switches
# uniform: (dtype, layout, C, B, H, W, Ho, Wo); ragged: C (a 24-image list)
ENV_RUNS = [
    {"env": {"ATTWARP_REMAP": "direct"},
     "uniform": [(U8, "hwc", 3, 256, 336, 336, 336, 336), (U8, "chw", 3, 256, 336, 336, 336, 336),
                 (F32, "hwc", 3, 256, 336, 336, 336, 336), (F32, "chw", 3, 256, 336, 336, 336, 336)],
     "kernels": ["remap_direct_kernel<unsigned char,true>", "remap_direct_kernel<unsigned char,false>",
                 "remap_direct_kernel<float,true>", "remap_direct_kernel<float,false>"], "ragged": []},
    {"env": {"ATTWARP_REMAP_F32": "rows"},
     "uniform": [(F32, "chw", 3, 128, 512, 512, 512, 512), (F32, "hwc", 3, 128, 512, 512, 512, 512)],
     "kernels": ["remap_f32_rows_kernel<false>", "remap_f32_rows_kernel<true>"], "ragged": []},
    {"env": {"ATTWARP_REMAP_QUAD": "0"},
     "uniform": [(U8, "hwc", 3, 256, 336, 336, 336, 336)],
     "kernels": ["remap_u8_stream_kernel<3,16,2>"], "ragged": [3], "ragged_kernels": ["remap_u8_stream_kernel<3,16,2>"]},
    {"env": {"ATTWARP_REMAP_QUAD": "0", "ATTWARP_REMAP_CPT": "1"},
     "uniform": [(U8, "hwc", 3, 256, 336, 336, 336, 336), (U8, "hwc", 1, 256, 336, 336, 336, 336)],
     "kernels": ["remap_u8_stream_kernel<3,16,1>", "remap_u8_stream_kernel<1,16,1>"], "ragged": [3],
     "ragged_kernels": ["remap_u8_stream_kernel<3,16,1>"]},
]


def _env_uniform_inputs(k, j, spec):
    dt, lay, C, B, H, W, Ho, Wo = spec
    img = make_image("random" if j % 2 == 0 else "coded", (B, H, W, C), dt, 500 + 10 * k + j)
    mx, my, _ = make_maps(B, H, W, Ho, Wo, 600 + 10 * k + j, shift=j)
    return img, mx, my


def _env_ragged_sizes(k):
    rng = np.random.default_rng(700 + k)
    sizes = [tuple(int(v) for v in rng.integers(2, 1500, 2)) for _ in range(24)]
    return sizes, [int(v) for v in rng.integers(0, 4, 24)]


def _run_child(k, out_path):
    """Child process of test_process_wide_switches: the switches are read once per process."""
    run = ENV_RUNS[k]
    res = {"uniform": [], "ragged": [], "kernels": []}
    for j, spec in enumerate(run["uniform"]):
        dt, lay, C, B, H, W, Ho, Wo = spec
        img, mx, my = _env_uniform_inputs(k, j, spec)
        case = ("child", "", dt, lay, C, B, H, W, Ho, Wo, 0, "")
        (got, flat, span), launched = _profiled(lambda: run_uniform(case, img, mx, my), out_path + f".u{j}.json")
        check_guards(flat, [span], dt, f"{run['env']} uniform {j}")
        res["uniform"].append(got.cpu())
        res["kernels"].append([n for n, _, _ in launched])
    for j, C in enumerate(run["ragged"]):
        sizes, offsets = _env_ragged_sizes(k)
        r, launched = _profiled(lambda: run_ragged(sizes, sizes, C, offsets, 800 + k), out_path + f".r{j}.json")
        imgs, outs, mxs, mys, flat, spans = r
        check_guards(flat, spans, U8, f"{run['env']} ragged {j}")
        res["ragged"].append({"outs": [o.cpu() for o in outs], "mx": [m.cpu() for m in mxs],
                              "my": [m.cpu() for m in mys]})
        res["kernels"].append([n for n, _, _ in launched])
    torch.save(res, out_path)


@pytest.mark.gpu
def test_process_wide_switches(tmp_path):
    """ATTWARP_REMAP=direct (uint8 and float32, both layouts, c2 size), ATTWARP_REMAP_F32=rows (c5, both layouts),
    ATTWARP_REMAP_QUAD=0 (<3,16,2>, uniform and mixed-size) and ATTWARP_REMAP_QUAD=0 ATTWARP_REMAP_CPT=1 (<3,16,1>,
    <1,16,1>), each in a child process whose outputs are compared here with the reference."""
    _need_gpu()
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_remap_dispatch as m; m._run_child(int(sys.argv[1]), sys.argv[2])" % (HERE, ROOT))
    procs = {}
    for k, run in enumerate(ENV_RUNS):
        env = dict(os.environ, **run["env"])
        procs[k] = subprocess.Popen([sys.executable, "-c", code, str(k), str(tmp_path / f"out_{k}.pt")],
                                    env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        logs = {k: p.communicate(timeout=600)[0] for k, p in procs.items()}
    finally:
        for p in procs.values():
            if p.poll() is None:
                p.kill()
                p.wait()
    for k, run in enumerate(ENV_RUNS):
        assert procs[k].returncode == 0, f"{run['env']}: child failed\n{logs[k]}"
        res = torch.load(tmp_path / f"out_{k}.pt", weights_only=True)
        want = run["kernels"] + run.get("ragged_kernels", [])
        if all(res["kernels"]):
            assert res["kernels"] == [[_norm(w)] for w in want], (run["env"], res["kernels"])
        for j, spec in enumerate(run["uniform"]):
            img, mx, my = _env_uniform_inputs(k, j, spec)
            compare(res["uniform"][j].cuda(), ref_remap(img, mx, my), img, mx, my, f"{run['env']} uniform {spec}",
                    res["kernels"][j])
        for j, C in enumerate(run["ragged"]):
            sizes, _ = _env_ragged_sizes(k)
            r = res["ragged"][j]
            for i, (h, w) in enumerate(sizes):
                im = make_image("random", (1, h, w, C), U8, 800 + k + i)
                mx, my = r["mx"][i].cuda()[None], r["my"][i].cuda()[None]
                compare(r["outs"][i].cuda()[None], ref_remap(im, mx, my), im, mx, my,
                        f"{run['env']} ragged C={C} image {i}", res["kernels"][len(run["uniform"]) + j])
