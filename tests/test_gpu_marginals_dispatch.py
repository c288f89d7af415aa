"""Stage 2 (profiles.cu, mask.cu, torch_path.cu): every compiled reduction kernel against a float64 reference, at the
launch geometry of small and of full-size batches.

The reductions that turn an attention map (or the LANCZOS resize of a token mask) into marginal sums, and the
trainer's pooling, pick their launch geometry from the batch size: rows per CTA of the row-owning marginals kernels
(profiles.cu: rows_per_cta, 64 to 256), the tile height of the tensor-core LANCZOS kernel (mask.cu: mma_geometry),
the tiles per image of the register-window LANCZOS kernel (up_geometry) and the (image, row) pairs per CTA of the
pooling kernel.  CASES has one row per compiled kernel at a small batch and, for every kernel whose geometry depends
on B, one more at the batch the benchmark's driver flow or the trainer runs; each row names the kernel it must launch
and the geometry class it must reach, both read back from the launch through torch.profiler.  Every row runs on the
input families that expose a dropped or doubled row or column (random, one nonzero pixel on a chunk / tile edge,
all-zero images, saturated bytes), with NaN or 255 wherever the kernel must not read.
test_case_table_names_every_compiled_kernel (CPU) keeps CASES and the library in step.

    python -m pytest tests/test_gpu_marginals_dispatch.py -m gpu -s     # -s prints the worst error per family
"""

import json
import os
import re
import shutil
import subprocess

import numpy as np
import pytest
import torch

from oracle import numpy_path as ON
from oracle import torch_path as OT

U8, F32, F64 = np.uint8, np.float32, np.float64
MARGIN = 64                                # guard elements before and after every input (NaN, or 255 for bytes)
LEAD = {"dense": 0, "offset": 1, "offset4": 4}   # elements between the guard and the input: 16-byte aligned or not
POOL = (24, 24)                            # the trainer's pooled grid (trainer.py:197)
EXP = (1e-3, 3.0)                          # exp_scale, exp_divisor: exp of values up to 1e4 stays finite

# (entry, dtype, transform, B, shape, layout, kernel, geometry)
#   entry   maps: ops.maps_from_attention to (H + 3, W + 5)   gt: checkpoint_utils.gt_marginals
#           pool / pool_sqrt: checkpoint_utils.pool_attention without / with the per-sample sqrt prologue
#           resize: ops.resize_lanczos_u8 (shape h, w, Ho, Wo)
#           mota: ops.maps_from_mota_tokens, fused, token grid h x w -> image Ho x Wo -> maps (Ho + 3, Wo + 5)
#   geometry  rows64: one CTA per 64 rows (the small-batch launch); tall: fewer, taller row chunks;
#           rows256: chunks of 256 rows (the bound of the 16-bit column lanes / the row-kernel maximum);
#           mma_short / mma_tall: tensor-core tiles of <= 48 / > 48 output rows; up_tiles / up_one: several tiles
#           per image / one; resize: 32-row tiles; pool_one / pool_multi: one (image, row) pair per CTA / several
CASES = [
    # generic marginals: float64 maps, float32 / uint8 maps whose rows or base miss the alignment of the row kernels
    ("maps", F64, "identity", 2, (130, 1100), "dense", "marginals_partial_kernel<double, 0>", "rows64"),
    ("maps", F64, "square", 3, (70, 203), "offset", "marginals_partial_kernel<double, 1>", "rows64"),
    ("maps", F64, "sqrt", 2, (65, 336), "dense", "marginals_partial_kernel<double, 2>", "rows64"),
    ("maps", F64, "exp", 3, (64, 333), "dense", "marginals_partial_kernel<double, 3>", "rows64"),
    ("maps", F64, "log", 2, (129, 516), "dense", "marginals_partial_kernel<double, 4>", "rows64"),
    ("gt", F32, None, 3, (67, 333), "dense", "marginals_partial_kernel<float, -1>", "rows64"),
    ("maps", F32, "identity", 3, (130, 336), "offset", "marginals_partial_kernel<float, 0>", "rows64"),
    ("maps", F32, "square", 2, (70, 203), "dense", "marginals_partial_kernel<float, 1>", "rows64"),
    ("maps", F32, "sqrt", 3, (65, 1344), "offset", "marginals_partial_kernel<float, 2>", "rows64"),
    ("maps", F32, "exp", 2, (64, 333), "dense", "marginals_partial_kernel<float, 3>", "rows64"),
    ("maps", F32, "log", 3, (129, 1030), "dense", "marginals_partial_kernel<float, 4>", "rows64"),
    ("maps", U8, "identity", 3, (130, 203), "dense", "marginals_partial_kernel<unsigned char, 8>", "rows64"),
    # row-owning float64 kernel: aligned float32 maps per transform, gt_marginals, uint8 maps off the integer kernel
    ("gt", F32, None, 3, (130, 512), "dense", "marginals_f32_rows_kernel<float, -1>", "rows64"),
    ("gt", F32, None, 128, (512, 512), "dense", "marginals_f32_rows_kernel<float, -1>", "rows256"),
    ("maps", F32, "identity", 3, (200, 1344), "dense", "marginals_f32_rows_kernel<float, 0>", "rows64"),
    ("maps", F32, "identity", 64, (1344, 1344), "dense", "marginals_f32_rows_kernel<float, 0>", "tall"),
    ("maps", F32, "square", 2, (65, 512), "dense", "marginals_f32_rows_kernel<float, 1>", "rows64"),
    ("maps", F32, "square", 256, (336, 336), "dense", "marginals_f32_rows_kernel<float, 1>", "tall"),
    ("maps", F32, "sqrt", 2, (130, 516), "dense", "marginals_f32_rows_kernel<float, 2>", "rows64"),
    ("maps", F32, "sqrt", 64, (1344, 1344), "dense", "marginals_f32_rows_kernel<float, 2>", "tall"),
    ("maps", F32, "exp", 3, (70, 1028), "dense", "marginals_f32_rows_kernel<float, 3>", "rows64"),
    ("maps", F32, "exp", 256, (336, 336), "dense", "marginals_f32_rows_kernel<float, 3>", "tall"),
    ("maps", F32, "log", 2, (129, 516), "dense", "marginals_f32_rows_kernel<float, 4>", "rows64"),
    ("maps", F32, "log", 256, (336, 336), "dense", "marginals_f32_rows_kernel<float, 4>", "tall"),
    ("maps", U8, "sqrt", 3, (70, 336), "dense", "marginals_f32_rows_kernel<unsigned char, 8>", "rows64"),
    ("maps", U8, "identity", 2, (65, 512), "offset4", "marginals_f32_rows_kernel<unsigned char, 8>", "rows64"),
    ("maps", U8, "square", 256, (336, 336), "dense", "marginals_f32_rows_kernel<unsigned char, 8>", "tall"),
    # integer kernel: uint8 identity maps with 16-byte rows; tile columns <= 512 / <= 1024 / <= 1536
    ("maps", U8, "identity", 3, (336, 336), "dense", "marginals_u8_identity_kernel<1, 4>", "rows64"),
    ("maps", U8, "identity", 256, (336, 336), "dense", "marginals_u8_identity_kernel<1, 4>", "tall"),
    ("maps", U8, "identity", 592, (256, 512), "dense", "marginals_u8_identity_kernel<1, 4>", "rows256"),
    ("maps", U8, "identity", 3, (200, 1024), "dense", "marginals_u8_identity_kernel<2, 2>", "rows64"),
    ("maps", U8, "identity", 256, (300, 1024), "dense", "marginals_u8_identity_kernel<2, 2>", "tall"),
    ("maps", U8, "identity", 3, (130, 1552), "dense", "marginals_u8_identity_kernel<3, 2>", "rows64"),
    ("maps", U8, "identity", 64, (1344, 1344), "dense", "marginals_u8_identity_kernel<3, 2>", "tall"),
    # LANCZOS up-scaling on the tensor cores: fused into the marginals (driver flow) / writing the mask
    ("mota", F32, "identity", 5, (24, 24, 336, 336), "dense", "resize_lanczos_up_mma_kernel<true>", "mma_short"),
    ("mota", F32, "identity", 256, (24, 24, 336, 336), "dense", "resize_lanczos_up_mma_kernel<true>", "mma_tall"),
    ("mota", F32, "identity", 5, (48, 48, 1344, 1344), "dense", "resize_lanczos_up_mma_kernel<true>", "mma_short"),
    ("mota", F32, "identity", 64, (48, 48, 1344, 1344), "dense", "resize_lanczos_up_mma_kernel<true>", "mma_tall"),
    ("resize", U8, None, 5, (24, 24, 336, 336), "dense", "resize_lanczos_up_mma_kernel<false>", "mma_short"),
    ("resize", U8, None, 256, (24, 24, 336, 336), "dense", "resize_lanczos_up_mma_kernel<false>", "mma_tall"),
    ("resize", U8, None, 5, (48, 48, 1344, 1344), "dense", "resize_lanczos_up_mma_kernel<false>", "mma_short"),
    ("resize", U8, None, 64, (48, 48, 1344, 1344), "dense", "resize_lanczos_up_mma_kernel<false>", "mma_tall"),
    # register-window LANCZOS kernel: token grids wider than 1024 (fused), output rows that are not 16-byte groups
    ("mota", F32, "identity", 3, (4, 1040, 96, 1100), "dense", "resize_lanczos_up_kernel<7, true>", "up_tiles"),
    ("mota", F32, "identity", 296, (4, 1040, 96, 1100), "dense", "resize_lanczos_up_kernel<7, true>", "up_one"),
    ("resize", U8, None, 3, (24, 24, 336, 338), "dense", "resize_lanczos_up_kernel<7, false>", "up_tiles"),
    ("resize", U8, None, 296, (24, 24, 336, 340), "dense", "resize_lanczos_up_kernel<7, false>", "up_one"),
    # any other resize: down-scaling
    ("resize", U8, None, 3, (336, 336, 24, 24), "dense", "resize_lanczos_u8_kernel", "resize"),
    ("resize", U8, None, 4, (100, 90, 37, 41), "offset", "resize_lanczos_u8_kernel", "resize"),
    # adaptive pooling to 24 x 24: float4 rows (W % 4 == 0, aligned) and scalar rows
    ("pool", F32, None, 2, (512, 512), "dense", "adaptive_avg_pool2d_kernel<0>", "pool_one"),
    ("pool", F32, None, 3, (130, 333), "dense", "adaptive_avg_pool2d_kernel<0>", "pool_one"),
    ("pool", F32, None, 128, (512, 512), "dense", "adaptive_avg_pool2d_kernel<0>", "pool_multi"),
    ("pool_sqrt", F32, None, 2, (512, 512), "dense", "adaptive_avg_pool2d_kernel<1>", "pool_one"),
    ("pool_sqrt", F32, None, 3, (97, 512), "offset", "adaptive_avg_pool2d_kernel<1>", "pool_one"),
    ("pool_sqrt", F32, None, 128, (512, 512), "dense", "adaptive_avg_pool2d_kernel<1>", "pool_multi"),
]

BASE_NAMES = ("marginals_partial_kernel", "marginals_f32_rows_kernel", "marginals_u8_identity_kernel",
              "resize_lanczos_up_mma_kernel", "resize_lanczos_up_kernel", "resize_lanczos_u8_kernel",
              "adaptive_avg_pool2d_kernel")
KERNEL_RE = re.compile(r"(?<![A-Za-z_])(" + "|".join(BASE_NAMES) + r")(?![A-Za-z_])(<[^>]*>)?")
CNAME = {U8: "u8", F32: "f32", F64: "f64"}
CASE_IDS = [f"{e}-{CNAME[dt]}-{tr or 'none'}-B{B}-{'x'.join(map(str, s))}-{lay}"
            for e, dt, tr, B, s, lay, k, g in CASES]
WORST = {}                                 # (kernel family, input family) -> worst err / bar


def _families(entry, dt):
    if entry == "mota":                    # an all-zero token map has no min-max normalisation
        return ["random", "single_pixel"]
    if dt == U8:
        return ["random", "single_pixel", "zero_image", "saturated"]
    return ["random", "single_pixel", "zero_image"]


def _norm(name):
    return re.sub(r"\s+", "", name)


def _stage2_kernels(names):
    """The stage-2 kernel instances in a list of (possibly mangled) symbol names, without spaces."""
    tool = shutil.which("c++filt") or shutil.which("cu++filt")
    if tool is not None and names:
        names = subprocess.run([tool], input="\n".join(names) + "\n", capture_output=True, text=True,
                               check=True).stdout.splitlines()
    return [_norm(m.group(0)) for n in names for m in KERNEL_RE.finditer(n)]


# ---------------------------------------------------------------------------------------------- inputs
def _edges(n, steps):
    """Coordinates 0, n - 1 and the first and last coordinate of every block of each length in ``steps``."""
    out = {0, n - 1}
    for s in steps:
        for k in range(s, n, s):
            out |= {k - 1, k}
    return sorted(out)


def make_input(family, dt, shape, rng, ys, xs, transform=None, signed=False, scaled=True):
    """[B, H, W] values of dtype dt.  ``ys`` / ``xs``: the rows / columns the single pixels sit on (chunk and tile
    edges).  ``signed``: float values with negatives (clamped by the kernels).  ``scaled``: float rows scaled over
    10^+-4 (else uniform in [0, 1))."""
    B, H, W = shape
    if family == "saturated":
        return np.full(shape, 255, U8)
    if family == "single_pixel":
        x = np.zeros(shape, dt)
        for b in range(B):
            y, c = ys[(b * 7) % len(ys)], xs[(b * 5) % len(xs)]
            if b == 0:
                y, c = 0, 0
            elif b == B - 1:
                y, c = H - 1, W - 1
            x[b, y, c] = rng.integers(1, 256) if dt == U8 else 10.0 ** rng.uniform(-3, 3)
        return x
    if dt == U8:
        x = rng.integers(0, 256, shape, dtype=U8)
    else:
        x = rng.random(shape, dtype=F32)
        if signed:
            x -= F32(0.2)
        if scaled:
            x *= (10.0 ** rng.uniform(-4, 4, (B, H, 1))).astype(F32)
        if transform == "log":             # log(x + 1e-5) >= 0: monotone knots
            x += F32(1.0)
        x = x.astype(dt)
    if family == "zero_image":
        x[::3] = 0
    return x


def on_device(x, layout):
    """x inside a guard of NaN (floats) or 255 (bytes), ``LEAD[layout]`` elements past a 16-byte boundary."""
    guard = 255 if x.dtype == U8 else np.nan
    lead = MARGIN + LEAD[layout]
    flat = torch.from_numpy(np.concatenate([np.full(lead, guard, x.dtype), x.ravel(), np.full(MARGIN, guard, x.dtype)]))
    return flat.cuda()[lead:lead + x.size].view(x.shape)


# ---------------------------------------------------------------------------------------------- references
def ref_maps(x, transform, Wo, Ho, es=1.0, ed=1.0):
    """float64 maps of every image of x (new_method.py:207-261): the marginals summed in float64 (exact int64
    sums for identity bytes), then the oracle's profile tail, knots and np.interp."""
    B, H, W = x.shape
    mx, my = np.empty((B, Wo)), np.empty((B, Ho))
    for s in range(0, B, 16):
        c = x[s:s + 16]
        if c.dtype == U8 and transform == "identity":
            px = c.sum(1, dtype=np.int64) + H * ON.BASE_ATTENTION
            py = c.sum(2, dtype=np.int64) + W * ON.BASE_ATTENTION
            mean = c.sum((1, 2), dtype=np.int64) / (H * W) + ON.BASE_ATTENTION
        else:
            a = ON.forward_transform(np.maximum(c.astype(F64), 0), transform, es, ed) + ON.BASE_ATTENTION
            px, py, mean = a.sum(1), a.sum(2), a.mean((1, 2))
        for k in range(len(c)):
            prof = ON.finish_profiles(px[k], py[k], mean[k], transform, es, ed)
            mx[s + k], my[s + k], _, _ = ON.maps_from_profiles(*prof[:4], Wo, Ho)
    return mx, my


def ref_gt(x):
    """gt_marginals in float64, mx held in float32 as the finish kernel (and the reference) does."""
    out = []
    for axis in (1, 2):
        m = np.concatenate([np.maximum(x[s:s + 16].astype(F64), 0).sum(axis) for s in range(0, len(x), 16)])
        m32 = m.astype(F32).astype(F64)
        denom = np.maximum(m32.sum(1, keepdims=True).astype(F32), F32(1e-6)).astype(F64)
        out.append(m32 / denom)
    return out


def ref_pool(x, take_sqrt):
    """Window means in float64 of the float32 values (of float32 sqrt(max(v, 0)) for images with take_sqrt)."""
    B, H, W = x.shape
    ys, ye = OT.pool_windows(H, POOL[0])
    xs, xe = OT.pool_windows(W, POOL[1])
    out = np.empty((B,) + POOL)
    for b in range(B):
        v = x[b]
        if take_sqrt is not None:
            v = np.maximum(v, F32(0))
            if take_sqrt[b]:
                v = np.sqrt(v)
        v = v.astype(F64)
        rs = np.stack([v[ys[i]:ye[i]].sum(0) for i in range(POOL[0])])
        for j in range(POOL[1]):
            out[b, :, j] = rs[:, xs[j]:xe[j]].sum(1) / ((ye - ys) * (xe[j] - xs[j]))
    return out


def pil_resize(x, Ho, Wo):
    from PIL import Image
    return np.stack([np.array(Image.fromarray(m, mode="L").resize((Wo, Ho), Image.LANCZOS)) for m in x])


def check_maps(got, ref, what):
    """|map - ref| <= 1e-4 px * max(1, n / 1000) (BASELINE.md section 4) -> worst err / bar."""
    got = got.cpu().numpy().astype(F64)
    bar = 1e-4 * max(1.0, ref.shape[1] / 1000)
    err = np.abs(got - ref)
    bad = ~(err <= bar)
    if bad.any():
        b, i = (int(v) for v in np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} map entries off the float64 reference, first "
                             f"at image {b} index {i}: got {got[b, i]!r}, ref {ref[b, i]!r} (bar {bar:.3g} px)")
    return float(err.max() / bar)


def check_rel(got, ref, rel, what):
    """|got - ref| <= rel |ref| (a zero reference must give exactly 0) -> worst err / bar."""
    got = got.cpu().numpy().astype(F64).reshape(ref.shape)
    err = np.abs(got - ref)
    bar = rel * np.abs(ref)
    bad = ~(err <= bar)
    if bad.any():
        idx = tuple(int(v) for v in np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} outputs off the float64 reference, first at "
                             f"{idx}: got {got[idx]!r}, ref {ref[idx]!r}")
    return float(np.max(np.where(bar > 0, err / np.where(bar > 0, bar, 1), 0)))


def ulp_diff(a, b):
    return np.abs(a.cpu().numpy().view(np.int32).astype(np.int64) - b.cpu().numpy().view(np.int32).astype(np.int64))


# ---------------------------------------------------------------------------------------------- launch geometry
def _launches(prof, path):
    """(kernel name, grid) of every stage-2 launch in the profile's chrome trace."""
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        events = json.load(f).get("traceEvents", [])
    out = []
    for e in events:
        if e.get("cat") == "kernel":
            names = _stage2_kernels([e.get("name", "")])
            if names:
                out.append((names[0], tuple(e.get("args", {}).get("grid", ()))))
    return out


def _consistent_rows(n, chunks, lo, hi, step):
    """Chunk heights in [lo, hi] (multiples of step) that split n rows into ``chunks`` chunks."""
    return [r for r in range(lo, hi + 1, step) if -(-n // r) == chunks]


def check_geometry(geo, grid, B, H, Ho):
    gx, gy, gz = (list(grid) + [1, 1, 1])[:3]
    c64 = -(-H // 64)
    if geo == "rows64":
        ok = gy == c64
    elif geo == "tall":
        ok = gy < c64
    elif geo == "rows256":
        ok = gy == -(-H // 256) < c64
    elif geo in ("mma_short", "mma_tall"):
        rows = _consistent_rows(Ho, gy, 16, 512, 16)
        ok = bool(rows) and (max(rows) <= 48 if geo == "mma_short" else min(rows) > 48)
    elif geo == "up_tiles":
        ok = gx > 1 and gy == B
    elif geo == "up_one":
        ok = gx == 1 and gy == B
    elif geo == "resize":
        ok = gx == -(-Ho // 32) and gy == B
    elif geo == "pool_one":
        ok = gx == B * POOL[0]
    elif geo == "pool_multi":
        ok = gx < B * POOL[0]
    else:
        raise ValueError(geo)
    return ok


@pytest.fixture(scope="module", autouse=True)
def _print_worst():
    yield
    if WORST:
        print("\nstage-2 worst error per kernel and input family (err / bar must be <= 1):")
        for (kern, fam), bar in sorted(WORST.items()):
            print(f"  {kern:30s} {fam:13s} err/bar {bar:.3g}")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


# ---------------------------------------------------------------------------------------------- CPU
def test_case_table_names_every_compiled_kernel():
    """The stage-2 kernel instances in the built library are exactly the kernels CASES names: a new instance without
    a case fails here, and so does a row whose kernel is no longer compiled."""
    from attwarp_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(cuobjdump):
        pytest.skip("cuobjdump not available")
    assert os.path.isfile(_lib.lib_path()), "build the library first: python -m attwarp_b200.build"
    out = subprocess.run([cuobjdump, "-symbols", _lib.lib_path()], capture_output=True, text=True, check=True).stdout
    compiled = set(_stage2_kernels(out.splitlines()))
    named = {_norm(k) for *_, k, _ in CASES}
    print(f"\n{len(compiled)} stage-2 kernel instances in the library:\n  " + "\n  ".join(sorted(compiled)))
    assert len(compiled) >= 29
    assert compiled == named, f"compiled but no case: {sorted(compiled - named)}; named but not compiled: {sorted(named - compiled)}"


def test_case_table_rows():
    """Every kernel whose geometry depends on B has a small-batch and a large-batch row, and no case id repeats."""
    assert len(set(CASE_IDS)) == len(CASE_IDS)
    by_kernel = {}
    for e, dt, tr, B, s, lay, k, g in CASES:
        by_kernel.setdefault(_norm(k), set()).add(g)
    for k, geos in by_kernel.items():
        if k.startswith(("marginals_f32_rows", "marginals_u8_identity")):
            assert "rows64" in geos and geos & {"tall", "rows256"}, k
        elif k.startswith("resize_lanczos_up_mma"):
            assert geos == {"mma_short", "mma_tall"}, k
        elif k.startswith("resize_lanczos_up_kernel"):
            assert geos == {"up_tiles", "up_one"}, k
        elif k.startswith("adaptive_avg_pool2d"):
            assert geos == {"pool_one", "pool_multi"}, k


# ---------------------------------------------------------------------------------------------- GPU
def _run(entry, dt, transform, x, layout, shape):
    """One call of the row's entry point on x (numpy) -> its outputs (device tensors)."""
    from attwarp_b200 import checkpoint_utils as CU, ops
    d = on_device(x, layout)
    if entry == "maps":
        H, W = shape
        es, ed = EXP if transform == "exp" else (1.0, 1.0)
        return ops.maps_from_attention(d, (H + 3, W + 5), transform, es, ed)
    if entry == "gt":
        return CU.gt_marginals(d[:, None])
    if entry == "pool":
        return CU.pool_attention(d[:, None], None, POOL)
    if entry == "pool_sqrt":
        return CU.pool_attention(d[:, None], ["sqrt" if b % 2 == 0 else "iden" for b in range(len(x))], POOL)
    if entry == "resize":
        return ops.resize_lanczos_u8(d, shape[2:])
    if entry == "mota":
        Ho, Wo = shape[2:]
        return ops.maps_from_mota_tokens(d, (Ho, Wo), (Ho + 3, Wo + 5))
    raise ValueError(entry)


def _check(entry, dt, transform, x, layout, shape, got, what):
    """Compare one call's outputs with the reference -> worst err / bar."""
    from attwarp_b200 import ops
    if entry == "maps":
        H, W = shape
        es, ed = EXP if transform == "exp" else (1.0, 1.0)
        rx, ry = ref_maps(x, transform, W + 5, H + 3, es, ed)
        return max(check_maps(got[0], rx, what + " map_x"), check_maps(got[1], ry, what + " map_y"))
    if entry == "gt":
        rx, ry = ref_gt(x)
        return max(check_rel(got[0], rx, 3e-7, what + " px"), check_rel(got[1], ry, 3e-7, what + " py"))
    if entry in ("pool", "pool_sqrt"):
        sq = None if entry == "pool" else [b % 2 == 0 for b in range(len(x))]
        return check_rel(got, ref_pool(x, sq), 2.5e-7, what)
    if entry == "resize":
        ref = pil_resize(x, *shape[2:])
        g = got.cpu().numpy()
        for b in range(len(x)):
            assert np.array_equal(g[b], ref[b]), (f"{what}: image {b} differs from PIL in "
                                                  f"{int((g[b] != ref[b]).sum())} bytes")
        return 0.0
    if entry == "mota":
        h, w, Ho, Wo = shape
        tok = on_device(x, layout)
        _, u8 = ops.revise_mask(tok, return_u8=True)
        mask = pil_resize(u8.cpu().numpy(), Ho, Wo)          # the mask the fused kernel never writes
        rx, ry = ref_maps(mask, "identity", Wo + 5, Ho + 3)
        two = ops.maps_from_mota_tokens(tok, (Ho, Wo), (Ho + 3, Wo + 5), fused=False)
        for a, b_, ax in zip(got, two, "xy"):
            u = ulp_diff(a, b_)
            assert u.max() <= 1, f"{what}: fused map_{ax} {int(u.max())} float32 ulp from the two-step path"
        return max(check_maps(got[0], rx, what + " map_x"), check_maps(got[1], ry, what + " map_y"))
    raise ValueError(entry)


@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_kernel_vs_float64(case, tmp_path):
    """One case of CASES on every input family against the float64 reference (bit-equality with PIL for the
    resize), and the launch of the kernel and geometry class the table names."""
    _need_gpu()
    entry, dt, transform, B, shape, layout, kernel, geo = CASES[case]
    kern_family = KERNEL_RE.search(kernel).group(1)
    rng = np.random.default_rng(2000 + case)
    if entry in ("resize", "mota"):        # single pixels / tokens at the corners and on a few source rows
        h, w, Ho, Wo = shape
        H = Ho
        x_shape = (B, h, w)
        ys, xs = _edges(h, (max(h // 3, 1),)), _edges(w, (max(w // 3, 1),))
    else:
        H, W = shape
        Ho = H + 3
        x_shape = (B, H, W)
        ys, xs = _edges(H, (64,)), _edges(W, (512, 1536))
        if entry in ("pool", "pool_sqrt"):     # the first and last row / column of every pooling window
            (y0, y1), (x0, x1) = OT.pool_windows(H, POOL[0]), OT.pool_windows(W, POOL[1])
            ys, xs = sorted(set(y0.tolist()) | set((y1 - 1).tolist())), sorted(set(x0.tolist()) | set((x1 - 1).tolist()))
    signed = entry in ("gt", "pool_sqrt") or (entry == "maps" and dt != U8 and transform != "log")
    launched = None
    for fam in _families(entry, dt):
        x = make_input(fam, dt, x_shape, rng, ys, xs, transform, signed, scaled=entry != "mota")
        what = f"{CASE_IDS[case]} ({kernel}) family {fam}"
        if launched is None:
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                    torch.profiler.ProfilerActivity.CUDA]) as prof:
                got = _run(entry, dt, transform, x, layout, shape)
                torch.cuda.synchronize()
            launched = _launches(prof, tmp_path / "trace.json")
            mine = [g for n, g in launched if n == _norm(kernel)]
            if len(mine) == 1 and len(mine[0]) >= 2 and geo in ("rows64", "tall", "rows256"):
                # the next families put their single pixels on the edges of the row chunks this launch used
                ys = _edges(H, _consistent_rows(H, mine[0][1], 64, 256, 8) or (64,))
        else:
            got = _run(entry, dt, transform, x, layout, shape)
        bar = _check(entry, dt, transform, x, layout, shape, got, what)
        WORST[(kern_family, fam)] = max(WORST.get((kern_family, fam), 0.0), bar)
    if not launched:
        pytest.skip("torch.profiler reported no CUDA kernel events: the launched kernel and its geometry are not checked")
    names = [n for n, _ in launched]
    assert names == [_norm(kernel)], f"{CASE_IDS[case]}: expected {kernel}, launched {names}"
    grid = launched[0][1]
    if not grid:
        pytest.skip(f"{CASE_IDS[case]}: the trace has no grid for the launch: its geometry is not checked")
    assert check_geometry(geo, grid, B, H, Ho), f"{CASE_IDS[case]}: {kernel} launched grid {grid}, not geometry {geo}"
