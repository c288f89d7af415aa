"""Oracle: float64 NumPy restatement of the reference's NumPy warp path.

TEST INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

Follows ``/root/reference/Attention Guided Warping/new_method.py``:

* transform registry + inverses ............ ``new_method.py:133-188``
* constants ``EPSILON = BASE_ATTENTION = 1e-9`` ``new_method.py:194-195``
* ``warp_image_by_attention`` ............... ``new_method.py:198-283``

and restates the two third-party routines it relies on:

* ``numpy.interp`` (NumPy ``compiled_base.c: arr_interp``; unpinned, 2.3.5 here) --
  ``interp_restated``;
* ``cv2.remap(..., INTER_LINEAR, BORDER_REPLICATE)`` (OpenCV ``imgwarp.cpp:
  remapBilinear`` with the 1/32-pixel ``INTER_TAB_SIZE`` coordinate quantisation and 15-bit
  fixed-point weights; unpinned, 4.13.0 here) -- ``remap_u8`` / ``remap_f32``.

Every function here is checked against the real reference / real cv2 in
``tests/test_oracle_vs_golden.py``.
"""

from __future__ import annotations

import numpy as np

EPSILON = 1e-9          # new_method.py:194
BASE_ATTENTION = 1e-9   # new_method.py:195

TRANSFORM_NAMES = ("identity", "square", "sqrt", "exp", "log")


# --------------------------------------------------------------------------------------
# transforms (new_method.py:133-188)
# --------------------------------------------------------------------------------------
def resolve_transform(name):
    """Unknown names silently become identity (new_method.py:399-402)."""
    return name if name in TRANSFORM_NAMES else "identity"


def forward_transform(x, name, exp_scale=1.0, exp_divisor=1.0):
    x = np.asarray(x, dtype=np.float64)
    if name == "identity":
        return x
    if name == "square":
        return x ** 2
    if name == "sqrt":
        return np.sqrt(np.maximum(x, 0))
    if name == "exp":
        return np.exp(exp_scale * x) / exp_divisor
    if name == "log":
        with np.errstate(divide="ignore", invalid="ignore"):
            return np.log(x + 1e-5)
    raise ValueError(name)


def inverse_transform(x, name, exp_scale=1.0, exp_divisor=1.0):
    x = np.asarray(x, dtype=np.float64)
    if name == "identity":
        return x
    if name == "square":               # inverse of square is sqrt
        return np.sqrt(np.maximum(x, 0))
    if name == "sqrt":                 # inverse of sqrt is square
        return x ** 2
    if name == "exp":
        return np.log(np.maximum(x * exp_divisor, 1e-9)) / exp_scale
    if name == "log":
        return np.exp(x) - 1e-5
    raise ValueError(name)


# --------------------------------------------------------------------------------------
# stage 2b: marginal profiles (new_method.py:207-239)
# --------------------------------------------------------------------------------------
def axis_profiles(att_map, transform="sqrt", exp_scale=1.0, exp_divisor=1.0,
                  apply_inverse=False):
    """Returns (profile_x[w], profile_y[h], total_x, total_y, used_fallback)."""
    a = np.maximum(np.asarray(att_map).astype(np.float64), 0)           # :207-208
    biased = forward_transform(a, transform, exp_scale, exp_divisor) + BASE_ATTENTION  # :210-212
    return finish_profiles(biased.sum(axis=0), biased.sum(axis=1),      # :215-216
                           biased.mean(), transform, exp_scale, exp_divisor, apply_inverse)


def finish_profiles(prof_x, prof_y, biased_mean, transform="sqrt", exp_scale=1.0, exp_divisor=1.0,
                    apply_inverse=False):
    """The rest of ``axis_profiles`` from the raw marginal sums of the biased map (column sums ``prof_x[w]``, row
    sums ``prof_y[h]``) and its mean: inverse transform, totals, fallback."""
    h, w = len(prof_y), len(prof_x)
    if apply_inverse:                                                   # :219-226
        prof_x = inverse_transform(prof_x - BASE_ATTENTION * h, transform, exp_scale,
                                   exp_divisor) + BASE_ATTENTION * h
        prof_y = inverse_transform(prof_y - BASE_ATTENTION * w, transform, exp_scale,
                                   exp_divisor) + BASE_ATTENTION * w
    tot_x = prof_x.sum()                                                # :228
    tot_y = prof_y.sum()                                                # :229
    fallback = bool(tot_x < EPSILON or tot_y < EPSILON)                 # :231
    if fallback:                                                        # :233-239
        prof_x = np.ones(w, dtype=np.float64)
        prof_y = np.ones(h, dtype=np.float64)
        m = biased_mean
        tot_x = max(w * (m * h), EPSILON)
        tot_y = max(h * (m * w), EPSILON)
    return prof_x, prof_y, float(tot_x), float(tot_y), fallback


# --------------------------------------------------------------------------------------
# stage 3: CDF -> forward knots (new_method.py:242-255)
# --------------------------------------------------------------------------------------
def forward_knots(profile, total, n_out):
    """xp[0]=0, xp[i+1]=cumsum(profile)[i]/total*n_out, xp[-1] forced to n_out (float64)."""
    cdf = np.cumsum(np.asarray(profile, dtype=np.float64)) / total
    xp = np.concatenate(([0.0], cdf)) * n_out
    xp[-1] = n_out
    return xp


# --------------------------------------------------------------------------------------
# stage 4: np.interp restated (inverse CDF)
# --------------------------------------------------------------------------------------
def interp_restated(x, xp):
    """``np.interp(x, xp, fp)`` with ``fp = [0, 1, ..., len(xp)-1]`` in float64.

    Semantics of NumPy's ``arr_interp``: ``x < xp[0] -> fp[0]``; ``x > xp[-1] -> fp[-1]``;
    otherwise ``j`` = last index with ``xp[j] <= x`` (bisection); ``j == n-1`` or an exact knot
    hit returns ``fp[j]``; else ``slope*(x-xp[j]) + fp[j]`` with
    ``slope = (fp[j+1]-fp[j])/(xp[j+1]-xp[j])`` evaluated as separate float64 operations.
    """
    x = np.asarray(x, dtype=np.float64)
    xp = np.asarray(xp, dtype=np.float64)
    n = xp.shape[0]
    j = np.searchsorted(xp, x, side="right") - 1
    out = np.empty_like(x)
    left = x < xp[0]
    right = x > xp[-1]
    jc = np.clip(j, 0, n - 2)
    with np.errstate(divide="ignore", invalid="ignore"):
        slope = 1.0 / (xp[jc + 1] - xp[jc])
        val = slope * (x - xp[jc]) + jc.astype(np.float64)
    exact = (j >= n - 1) | (xp[np.clip(j, 0, n - 1)] == x)
    out[:] = np.where(exact, np.clip(j, 0, n - 1).astype(np.float64), val)
    out[left] = 0.0
    out[right] = float(n - 1)
    return out


def interp_scalar_numpy_algorithm(x, xp):
    """Pure-Python transliteration of the *published* NumPy algorithm including its
    ``binary_search_with_guess`` (matters only for non-monotone ``xp``; small cases)."""
    xp = [float(v) for v in xp]
    n = len(xp)
    out = []
    guess = 0
    for key in x:
        key = float(key)
        if key > xp[n - 1]:
            j = n
        elif key < xp[0]:
            j = -1
        elif n <= 4:
            i = 1
            while i < n and key >= xp[i]:
                i += 1
            j = i - 1
        else:
            g = min(max(guess, 1), n - 3)
            imin, imax = 0, n
            done = None
            if key < xp[g]:
                if key < xp[g - 1]:
                    imax = g - 1
                    if g > 8 and key >= xp[g - 8]:
                        imin = g - 8
                else:
                    done = g - 1
            else:
                if key < xp[g + 1]:
                    done = g
                elif key < xp[g + 2]:
                    done = g + 1
                else:
                    imin = g + 2
                    if g < n - 8 - 1 and key < xp[g + 8]:
                        imax = g + 8
            if done is None:
                while imin < imax:
                    imid = imin + ((imax - imin) >> 1)
                    if key >= xp[imid]:
                        imin = imid + 1
                    else:
                        imax = imid
                done = imin - 1
            j = done
        guess = j
        if j == -1:
            out.append(0.0)
        elif j == n:
            out.append(float(n - 1))
        elif j == n - 1 or xp[j] == key:
            out.append(float(j))
        else:
            slope = 1.0 / (xp[j + 1] - xp[j])
            out.append(slope * (key - xp[j]) + float(j))
    return np.asarray(out, dtype=np.float64)


def inverse_maps(att_map, new_width, new_height, transform="sqrt", exp_scale=1.0,
                 exp_divisor=1.0, apply_inverse=False):
    """Stages 2b-4 of the NumPy path: returns float64 (map_x[new_w], map_y[new_h], xp, yp)."""
    return maps_from_profiles(*axis_profiles(att_map, transform, exp_scale, exp_divisor, apply_inverse)[:4],
                              new_width, new_height)


def maps_from_profiles(px, py, tx, ty, new_width, new_height):
    """Stages 3-4 from ``axis_profiles``' profiles and totals: float64 (map_x, map_y, xp, yp)."""
    xp = forward_knots(px, tx, new_width)
    yp = forward_knots(py, ty, new_height)
    map_x = interp_restated(np.arange(new_width), xp)      # new_method.py:258-260
    map_y = interp_restated(np.arange(new_height), yp)     # new_method.py:259-261
    return map_x, map_y, xp, yp


# --------------------------------------------------------------------------------------
# stage 5: cv2.remap(INTER_LINEAR, BORDER_REPLICATE) restated
# --------------------------------------------------------------------------------------
def quantise_coord(m):
    """float32 map value -> (integer pixel, 5-bit fraction): ``s = rint(m*32)`` (half-even)."""
    s = np.rint(np.asarray(m, dtype=np.float32) * np.float32(32.0)).astype(np.int64)
    return s >> 5, s & 31


def _taps(map_x, map_y, H, W):
    ix, ax = quantise_coord(map_x)
    iy, ay = quantise_coord(map_y)
    if ix.ndim == 1:                       # separable maps -> broadcast to a grid
        ix, ax = ix[None, :], ax[None, :]
        iy, ay = iy[:, None], ay[:, None]
    x0 = np.clip(ix, 0, W - 1)
    x1 = np.clip(ix + 1, 0, W - 1)
    y0 = np.clip(iy, 0, H - 1)
    y1 = np.clip(iy + 1, 0, H - 1)
    return x0, x1, y0, y1, ax, ay


def remap_u8(image, map_x, map_y):
    """uint8 image [H,W] or [H,W,C]; float32 maps (1-D separable or 2-D)."""
    img = np.asarray(image)
    assert img.dtype == np.uint8
    H, W = img.shape[:2]
    x0, x1, y0, y1, ax, ay = _taps(map_x, map_y, H, W)
    src = img.astype(np.int64)
    if img.ndim == 3:
        ax, ay = ax[..., None], ay[..., None]
    p00, p01 = src[y0, x0], src[y0, x1]
    p10, p11 = src[y1, x0], src[y1, x1]
    acc = 32 * ((32 - ax) * (32 - ay) * p00 + ax * (32 - ay) * p01
                + (32 - ax) * ay * p10 + ax * ay * p11)
    return ((acc + (1 << 14)) >> 15).astype(np.uint8)


def remap_f32(image, map_x, map_y):
    """float32 image; same coordinate quantisation, float32 weights, no FMA contraction."""
    img = np.asarray(image)
    assert img.dtype == np.float32
    H, W = img.shape[:2]
    x0, x1, y0, y1, ax, ay = _taps(map_x, map_y, H, W)
    scale = np.float32(1.0 / 32.0)
    fx = ax.astype(np.float32) * scale
    fy = ay.astype(np.float32) * scale
    one = np.float32(1.0)
    w00 = (one - fy) * (one - fx)
    w01 = (one - fy) * fx
    w10 = fy * (one - fx)
    w11 = fy * fx
    if img.ndim == 3:
        w00, w01, w10, w11 = (w[..., None] for w in (w00, w01, w10, w11))
    p00, p01 = img[y0, x0], img[y0, x1]
    p10, p11 = img[y1, x0], img[y1, x1]
    return ((p00 * w00 + p01 * w01) + p10 * w10) + p11 * w11


def remap(image, map_x, map_y):
    if image.dtype == np.uint8:
        return remap_u8(image, map_x, map_y)
    if image.dtype == np.float32:
        return remap_f32(image, map_x, map_y)
    raise TypeError(f"unsupported image dtype {image.dtype}")


def remap_cv2(image, map_x, map_y):
    """The reference's actual call (new_method.py:263-271): meshgrid + cv2.remap.
    Used as the timed CPU baseline and to pin ``remap_u8``/``remap_f32``."""
    import cv2
    gx, gy = np.meshgrid(map_x, map_y)
    return cv2.remap(image, gx.astype(np.float32), gy.astype(np.float32),
                     interpolation=cv2.INTER_LINEAR, borderMode=cv2.BORDER_REPLICATE)


# --------------------------------------------------------------------------------------
# end to end (new_method.py:198-283)
# --------------------------------------------------------------------------------------
def warp_image_by_attention(image, att_map, new_width, new_height, transform="sqrt",
                            exp_scale=1.0, exp_divisor=1.0, apply_inverse=False,
                            remap_backend="restated", return_maps=False):
    map_x, map_y, _, _ = inverse_maps(att_map, new_width, new_height, transform, exp_scale,
                                      exp_divisor, apply_inverse)
    mx32 = map_x.astype(np.float32)        # new_method.py:264-265
    my32 = map_y.astype(np.float32)
    fn = remap if remap_backend == "restated" else remap_cv2
    out = fn(np.ascontiguousarray(image), mx32, my32)
    if return_maps:
        return out, mx32, my32
    return out


def upsample_tokens_nearest(tok, H, W):
    """Token grid [gh,gw] -> [H,W] by index ``(y*gh)//H, (x*gw)//W`` (== np.repeat when H,W are
    multiples of the grid).  Not a reference function: it is the synthetic 'upsample to image
    resolution' step of BASELINE.json configs[1]/[2] (SURVEY.md section 8(d))."""
    tok = np.asarray(tok)
    gh, gw = tok.shape
    yi = (np.arange(H) * gh) // H
    xi = (np.arange(W) * gw) // W
    return tok[yi][:, xi]


# --------------------------------------------------------------------------------------
# the wrapper the drivers call (new_method.py:405-506), array level
# --------------------------------------------------------------------------------------
def save_warped_image_arrays(image_rgb, att_map, width=500, height=500, transform="identity", exp_scale=1.0,
                             exp_divisor=1.0, apply_inverse=False, remap_backend="restated"):
    """What ``save_warped_image`` hands to ``cv2.imwrite(output_path, ...)`` for an image given as a PIL / RGB
    array: RGB -> BGR (new_method.py:421-422; a 2-D image is replicated to three channels by cvtColor), the
    attention map coerced to 2-D (:432-452: list -> first element, [h,w,c] -> mean over c), the IMAGE resized to
    the attention map's size with ``cv2.resize(INTER_LINEAR)`` when they differ (:478, :355-376 -- the real cv2
    call: this step is host-side scaffolding in the product too), then ``warp_image_by_attention`` with the
    named transform (:483-486).  Returns the BGR array."""
    import cv2
    image = np.asarray(image_rgb)
    bgr = np.repeat(image[..., None], 3, -1) if image.ndim == 2 else image[..., ::-1]
    bgr = np.ascontiguousarray(bgr)
    if isinstance(att_map, list):
        att_map = np.asarray(att_map[0]) if len(att_map) > 0 else np.ones((height, width), np.float32) * 128
    att = np.asarray(att_map)
    if att.ndim == 3:
        att = np.mean(att, axis=2)
    elif att.ndim != 2:
        raise ValueError(f"Attention map must be 2D, got shape {att.shape}")
    if bgr.shape[:2] != att.shape[:2]:
        bgr = cv2.resize(bgr, (att.shape[1], att.shape[0]), interpolation=cv2.INTER_LINEAR)
    return warp_image_by_attention(bgr, att, width, height, resolve_transform(transform), exp_scale, exp_divisor,
                                   apply_inverse, remap_backend)
