"""Oracle: NumPy restatement of the attention overlay ``save_warped_image`` writes as
``masked_overlay_save_path`` (new_method.py; mirrored in ``attwarp_b200/new_method.py:save_warped_image``).

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

For a uint8 BGR image (grey replicated to BGR) and a 2-D attention map ``a`` of the image's size, the reference
computes ``cv2.addWeighted(applyColorMap(uint8(n * 255), JET), alpha, base, 1 - alpha, 0)`` with
``n = (a - lo) / (hi - lo) if hi > lo + 1e-9 else 0``.  Written out here step by step, each in the precision
NumPy 2 promotion gives the map's dtype, with no reliance on that promotion:

* uint8: ``a - lo`` in uint8; the comparison, the division and ``* 255`` in float64;
* float32: every step in float32, ``lo + 1e-9`` too (the Python float is a weak scalar);
* float64: every step in float64;
* ``min`` / ``max`` propagate NaN, and a NaN map takes the zero branch;
* ``uint8(x)`` truncates;
* ``cv2.addWeighted`` on uint8 (OpenCV 4.13): ``saturate(rint(fmaf(heat, a32, base * b32)))`` with
  ``a32 = float32(alpha)``, ``b32 = float32(1 - alpha)`` (``1 - alpha`` in double) and ``base * b32`` rounded
  to float32; ``fmaf`` is computed exactly here (``fma_f32``).

``JET`` is ``cv2.applyColorMap``'s 256-entry BGR table.  ``tests/test_overlay_host.py`` checks all of this against
the real cv2 / NumPy expression.
"""

from __future__ import annotations

import numpy as np

from .numpy_path import EPSILON, upsample_tokens_nearest

# cv2.applyColorMap(arange(256), COLORMAP_JET) (OpenCV 4.13), BGR bytes
JET = np.frombuffer(bytes.fromhex(
    "8000008400008800008c00009000009400009800009c0000a00000a40000a80000ac0000b00000b40000b80000bc0000"
    "c00000c40000c80000cc0000d00000d40000d80000dc0000e00000e40000e80000ec0000f00000f40000f80000fc0000"
    "ff0000ff0400ff0800ff0c00ff1000ff1400ff1800ff1c00ff2000ff2400ff2800ff2c00ff3000ff3400ff3800ff3c00"
    "ff4000ff4400ff4800ff4c00ff5000ff5400ff5800ff5c00ff6000ff6400ff6800ff6c00ff7000ff7400ff7800ff7c00"
    "ff8000ff8400ff8800ff8c00ff9000ff9400ff9800ff9c00ffa000ffa400ffa800ffac00ffb000ffb400ffb800ffbc00"
    "ffc000ffc400ffc800ffcc00ffd000ffd400ffd800ffdc00ffe000ffe400ffe800ffec00fff000fff400fff800fffc00"
    "feff02faff06f6ff0af2ff0eeeff12eaff16e6ff1ae2ff1edeff22daff26d6ff2ad2ff2eceff32caff36c6ff3ac2ff3e"
    "beff42baff46b6ff4ab2ff4eaeff52aaff56a6ff5aa2ff5e9eff629aff6696ff6a92ff6e8eff728aff7686ff7a82ff7e"
    "7eff827aff8676ff8a72ff8e6eff926aff9666ff9a62ff9e5effa25affa656ffaa52ffae4effb24affb646ffba42ffbe"
    "3effc23affc636ffca32ffce2effd22affd626ffda22ffde1effe21affe616ffea12ffee0efff20afff606fffa01fffe"
    "00fcff00f8ff00f4ff00f0ff00ecff00e8ff00e4ff00e0ff00dcff00d8ff00d4ff00d0ff00ccff00c8ff00c4ff00c0ff"
    "00bcff00b8ff00b4ff00b0ff00acff00a8ff00a4ff00a0ff009cff0098ff0094ff0090ff008cff0088ff0084ff0080ff"
    "007cff0078ff0074ff0070ff006cff0068ff0064ff0060ff005cff0058ff0054ff0050ff004cff0048ff0044ff0040ff"
    "003cff0038ff0034ff0030ff002cff0028ff0024ff0020ff001cff0018ff0014ff0010ff000cff0008ff0004ff0000ff"
    "0000fc0000f80000f40000f00000ec0000e80000e40000e00000dc0000d80000d40000d00000cc0000c80000c40000c0"
    "0000bc0000b80000b40000b00000ac0000a80000a40000a000009c00009800009400009000008c000088000084000080"
), dtype=np.uint8).reshape(256, 3)


def _trunc_u8(x):
    """uint8(x) of values in [0, 255] (NaN -> 0, as the x86 conversion gives)."""
    x = np.nan_to_num(np.trunc(x), nan=0.0)
    return np.clip(x, 0, 255).astype(np.uint8)


def heat_index(att) -> np.ndarray:
    """uint8 [H, W]: the JET index ``uint8((a - lo) / (hi - lo) * 255)`` of every pixel, or 0 everywhere when
    ``hi <= lo + 1e-9`` (NaN included), in the dtype's own precision (module docstring)."""
    a = np.asarray(att)
    if a.ndim != 2:
        raise ValueError(f"attention map must be 2-D, got {a.shape}")
    if a.dtype == np.uint8:
        lo, hi = int(a.min()), int(a.max())
        if not (np.float64(hi) > np.float64(lo) + np.float64(EPSILON)):
            return np.zeros(a.shape, np.uint8)
        d = (a.astype(np.int64) - lo).astype(np.uint8).astype(np.float64)
        return _trunc_u8(d / np.float64(hi - lo) * np.float64(255))
    if a.dtype in (np.float32, np.float64):
        t = a.dtype.type
        lo, hi = t(np.min(a)), t(np.max(a))                      # NaN-propagating
        if not (hi > t(lo + t(EPSILON))):
            return np.zeros(a.shape, np.uint8)
        with np.errstate(invalid="ignore", over="ignore"):
            n = (a - lo) / t(hi - lo)
            return _trunc_u8(n * t(255))
    raise ValueError(f"attention dtype {a.dtype} is outside the contract (uint8, float32, float64)")


def fma_f32(x, y, z) -> np.ndarray:
    """Correctly rounded float32 ``x * y + z`` for float32 arrays (what the device's ``fmaf`` computes)."""
    x, y, z = (np.asarray(v, np.float32).astype(np.float64) for v in (x, y, z))
    p = x * y                                   # exact: two 24-bit significands fit in 53 bits
    s = p + z
    bp = s - z                                  # TwoSum: p + z == s + e exactly
    e = (p - bp) + (z - (s - bp))
    f = s.astype(np.float32)                    # round to nearest even from s
    toward = np.where(s > f.astype(np.float64), np.float32(np.inf), np.float32(-np.inf))
    g = np.nextafter(f, toward)
    # s was a tie between f and g: the exact value decides, on whichever side of s it lies
    tie = (s != f.astype(np.float64)) & (s == (f.astype(np.float64) + g.astype(np.float64)) / 2)
    away = tie & (e != 0) & (np.sign(e) == np.sign(s - f.astype(np.float64)))
    return np.where(away, g, f)


def add_weighted(heat, base, alpha) -> np.ndarray:
    """``cv2.addWeighted(heat, alpha, base, 1 - alpha, 0)`` on uint8 arrays of one shape."""
    a32 = np.float32(alpha)
    b32 = np.float32(1.0 - float(alpha))
    hb = np.asarray(heat).astype(np.float32)
    bb = np.asarray(base).astype(np.float32)
    v = fma_f32(hb, a32, (bb * b32).astype(np.float32))
    return np.clip(np.rint(v), 0, 255).astype(np.uint8)


def as_bgr(image) -> np.ndarray:
    """uint8 [H, W] / [H, W, 1] (grey, replicated as cv2.cvtColor(GRAY2BGR) does) or [H, W, 3] -> [H, W, 3]."""
    im = np.asarray(image)
    if im.dtype != np.uint8:
        raise ValueError(f"image must be uint8, got {im.dtype}")
    if im.ndim == 3 and im.shape[2] == 1:
        im = im[..., 0]
    if im.ndim == 2:
        return np.repeat(im[..., None], 3, -1)
    if im.ndim == 3 and im.shape[2] == 3:
        return im
    raise ValueError(f"image must be [H, W], [H, W, 1] or [H, W, 3], got {im.shape}")


def attention_overlay(image, att, alpha: float = 0.5) -> np.ndarray:
    """uint8 [H, W, 3] BGR: the overlay of an attention map of the image's own size."""
    base = as_bgr(image)
    a = np.asarray(att)
    if a.shape != base.shape[:2]:
        raise ValueError(f"attention map {a.shape} is not the image's size {base.shape[:2]}")
    return add_weighted(JET[heat_index(a)], base, alpha)


def attention_overlay_tokens(image, tok, alpha: float = 0.5) -> np.ndarray:
    """The overlay of a float32 [gh, gw] token map, index-upsampled to the image (``(y * gh) // H``,
    ``(x * gw) // W``); lo and hi are those of the upsampled map, i.e. of the tokens it reaches."""
    base = as_bgr(image)
    H, W = base.shape[:2]
    full = upsample_tokens_nearest(np.asarray(tok, np.float32), H, W)
    return attention_overlay(base, full, alpha)
