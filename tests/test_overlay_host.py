"""CPU: ``oracle/overlay.py`` -- the NumPy restatement of the attention overlay ``save_warped_image`` writes -- against
the host expression itself (real cv2 and NumPy): random uint8, float32 and float64 maps, negative values, each
dtype's zero branch near 1e-9, NaN maps, grey images; the restated ``cv2.addWeighted`` over every byte pair; the
baked JET table against ``cv2.applyColorMap``."""

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from attwarp_b200.new_method import EPSILON  # noqa: E402
from oracle import numpy_path as ON  # noqa: E402
from oracle import overlay as OV  # noqa: E402

ALPHAS = (0.0, 0.3, 0.5, 0.7, 1.0)


def host_expression(image, att_map, alpha=0.5):
    """The overlay lines of save_warped_image (attwarp_b200/new_method.py), verbatim."""
    in_h, in_w = image.shape[:2]
    base = image.copy()
    if base.ndim == 2:
        base = cv2.cvtColor(base, cv2.COLOR_GRAY2BGR)
    att_r = cv2.resize(att_map.copy(), (in_w, in_h), interpolation=cv2.INTER_LINEAR)
    lo, hi = np.min(att_r), np.max(att_r)
    att_n = (att_r - lo) / (hi - lo) if hi > lo + EPSILON else np.zeros_like(att_r)
    heat = cv2.applyColorMap((att_n * 255).astype(np.uint8), cv2.COLORMAP_JET)
    return cv2.addWeighted(heat, alpha, base, 1 - alpha, 0)


def test_jet_table_equals_cv2():
    ramp = np.arange(256, dtype=np.uint8).reshape(1, 256)
    assert np.array_equal(OV.JET, cv2.applyColorMap(ramp, cv2.COLORMAP_JET)[0])


@pytest.mark.parametrize("alpha", ALPHAS)
@pytest.mark.parametrize("width", [1, 3, 7, 16, 33, 256])
def test_add_weighted_every_byte_pair(alpha, width):
    """All 65 536 (heat, base) pairs, laid out as rows of `width` BGR pixels (cv2's SIMD body and scalar tail)."""
    h, b = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
    h, b = h.reshape(-1), b.reshape(-1)
    per_row = 3 * width
    pad = -len(h) % per_row
    h, b = np.concatenate([h, h[:pad]]), np.concatenate([b, b[:pad]])
    heat, base = h.reshape(-1, width, 3), b.reshape(-1, width, 3)
    want = cv2.addWeighted(heat, alpha, base, 1 - alpha, 0)
    got = OV.add_weighted(heat, base, alpha)
    assert np.array_equal(got, want), f"{int((got != want).sum())} mismatches"


def test_fma_is_exact():
    """fma_f32 rounds once: a tie of the double sum is broken by the exact value."""
    x = y = np.float32(1 + 2.0 ** -12)           # x * y = 1 + 2^-11 + 2^-24: a float32 tie, exact in double
    z = np.float32(2.0 ** -80)                   # lost in the double sum, yet it puts the exact value above the tie
    want = np.nextafter(np.float32(1 + 2.0 ** -11), np.float32(2))
    assert OV.fma_f32(x, y, z) == want
    assert OV.fma_f32(x, y, -z) == np.float32(1 + 2.0 ** -11)
    rng = np.random.default_rng(5)
    a, b, c = (rng.standard_normal(4096).astype(np.float32) for _ in range(3))
    ref = [float(np.float32(np.longdouble(p) * np.longdouble(q) + np.longdouble(r))) for p, q, r in zip(a, b, c)]
    if np.finfo(np.longdouble).nmant >= 63:                  # x87 extended: p * q + r is exact for these ranges
        assert np.array_equal(OV.fma_f32(a, b, c), np.asarray(ref, np.float32))


def _maps(dtype, H, W, rng):
    """(name, map) families for one dtype."""
    out = []
    if dtype == np.uint8:
        out.append(("random", rng.integers(0, 256, (H, W), dtype=np.uint8)))
        out.append(("narrow", rng.integers(100, 103, (H, W), dtype=np.uint8)))
        out.append(("two_values", np.where(rng.random((H, W)) < 0.5, 7, 8).astype(np.uint8)))
        out.append(("constant", np.full((H, W), 42, np.uint8)))
        return out
    t = np.dtype(dtype).type
    out.append(("random", (rng.random((H, W)) ** 3).astype(dtype)))
    out.append(("negative", (rng.standard_normal((H, W)) * 100 - 50).astype(dtype)))
    out.append(("constant", np.full((H, W), 0.25, dtype)))
    # hi - lo around 1e-9: float64 takes the zero branch below it; float32 (lo + 1e-9 == lo for |lo| >> 1e-9)
    # takes the normalising branch for any hi > lo
    lo = t(1.0)
    for k, step in enumerate((np.nextafter(lo, t(2)) - lo, t(5e-10), t(2e-9))):
        m = np.full((H, W), lo, dtype)
        m[rng.random((H, W)) < 0.3] = t(lo + t(step))
        out.append((f"near_eps_{k}", m))
    tiny = np.full((H, W), t(1e-12), dtype)                 # |lo| tiny: lo + 1e-9 differs from lo in float32 too
    tiny[rng.random((H, W)) < 0.3] = t(1e-12 + 5e-10)
    out.append(("tiny_below_eps", tiny))
    tiny2 = tiny.copy()
    tiny2[tiny2 != t(1e-12)] = t(1e-12 + 2e-9)
    out.append(("tiny_above_eps", tiny2))
    nan = (rng.random((H, W))).astype(dtype)
    nan[H // 2, W // 3] = np.nan
    out.append(("nan", nan))
    return out


@pytest.mark.parametrize("dtype", [np.uint8, np.float32, np.float64])
@pytest.mark.parametrize("shape", [(37, 53, 3), (64, 80, 3), (40, 50), (1, 17, 3), (23, 1)])
def test_oracle_equals_host_expression(dtype, shape):
    rng = np.random.default_rng(hash((np.dtype(dtype).str, shape)) % 2 ** 32)
    image = rng.integers(0, 256, shape, dtype=np.uint8)
    H, W = shape[:2]
    import warnings
    for name, att in _maps(dtype, H, W, rng):
        for alpha in ALPHAS:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore", RuntimeWarning)
                want = host_expression(image, att, alpha)
            got = OV.attention_overlay(image, att, alpha)
            assert np.array_equal(got, want), f"{name} alpha={alpha}: {int((got != want).any(-1).sum())} pixels"


@pytest.mark.parametrize("grid,hw", [((24, 24), (336, 336)), ((48, 48), (97, 53)), ((24, 24), (1, 40)),
                                     ((24, 24), (40, 1)), ((48, 48), (500, 375))])
def test_token_oracle_equals_host_expression_of_upsampled_map(grid, hw):
    rng = np.random.default_rng(grid[0] * 1000 + hw[0])
    tok = (rng.random(grid) ** 4).astype(np.float32)
    image = rng.integers(0, 256, hw + (3,), dtype=np.uint8)
    full = ON.upsample_tokens_nearest(tok, *hw)
    assert np.array_equal(OV.attention_overlay_tokens(image, tok), host_expression(image, full, 0.5))


@pytest.mark.parametrize("name", ["path_list_sqrt", "att_3d_mean", "pil_att_exp_inv", "gray_input"])
def test_oracle_reproduces_the_reference_overlays(name):
    """The overlays the unmodified reference wrote (tests/golden/save_warped.npz), with save_warped_image's coercions:
    RGB -> BGR (a grey image comes back replicated), a 3-D map averaged over its last axis."""
    import os
    from conftest import GOLDEN_DIR
    gs = np.load(os.path.join(GOLDEN_DIR, "save_warped.npz"))
    image = cv2.cvtColor(gs[name + "/image_rgb"], cv2.COLOR_RGB2BGR)
    att = gs[name + "/att"]
    if att.ndim == 3:
        att = np.mean(att, axis=2)
    assert np.array_equal(OV.attention_overlay(image, att), gs[name + "/overlay_bgr"])


def test_oracle_rejects_outside_contract():
    img = np.zeros((4, 5, 3), np.uint8)
    with pytest.raises(ValueError):
        OV.attention_overlay(img, np.zeros((4, 6), np.float32))
    with pytest.raises(ValueError):
        OV.attention_overlay(img, np.zeros((4, 5), np.int32))
    with pytest.raises(ValueError):
        OV.attention_overlay(np.zeros((4, 5, 4), np.uint8), np.zeros((4, 5), np.float32))
