"""GPU parity, NumPy path (stages 2b-5): CUDA kernels vs golden vectors recorded from the real
reference and vs the oracle.  Tolerances: BASELINE.md section 4 -- maps <= 1e-4 px, uint8 remap
given identical maps 0 LSB, end-to-end uint8 +-1 LSB (we assert 0 where the reference's own
maps are used and +-1 end to end)."""

import numpy as np
import pytest
import torch

from conftest import numpy_case_names
from gpu_util import dev, hwc, need_gpu
from oracle import numpy_path as ON

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("name", numpy_case_names())
def test_remap_given_reference_maps_is_bit_equal(golden_numpy, name):
    need_gpu()
    from attwarp_b200 import ops
    c = golden_numpy.case(name)
    img = hwc(c["image"])
    out = ops.remap_bilinear(dev(img)[None], dev(c["map_x"])[None], dev(c["map_y"])[None], "hwc")
    got = out[0].cpu().numpy()
    assert np.array_equal(got, hwc(c["out"]))


@pytest.mark.parametrize("name", numpy_case_names())
def test_maps_and_end_to_end(golden_numpy, name):
    need_gpu()
    from attwarp_b200 import ops, new_method
    c = golden_numpy.case(name)
    tname = ON.resolve_transform(c["transform"])
    att = c["att"]
    att_t = dev(att if att.dtype in (np.uint8, np.float32, np.float64) else att.astype(np.float64))
    mx, my = ops.maps_from_attention(att_t[None], (c["new_h"], c["new_w"]), tname, c["exp_scale"],
                                     c["exp_divisor"], c["apply_inverse"])
    assert np.abs(mx[0].cpu().numpy() - c["map_x"]).max() <= 1e-4
    assert np.abs(my[0].cpu().numpy() - c["map_y"]).max() <= 1e-4
    # the drop-in NumPy entry point (host buffers in / out), module-level transform state
    new_method.set_transform_function(c["transform"], c["exp_scale"], c["exp_divisor"],
                                      c["apply_inverse"])
    out = new_method.warp_image_by_attention(c["image"], att, c["new_w"], c["new_h"])
    assert out.shape == c["out"].shape and out.dtype == c["out"].dtype
    diff = np.abs(out.astype(np.int32) - c["out"].astype(np.int32))
    assert diff.max() <= 1, f"max LSB diff {diff.max()}"
    assert (diff != 0).mean() <= 1e-3


@pytest.mark.parametrize("layout", ["hwc", "chw"])
@pytest.mark.parametrize("dtype", [np.uint8, np.float32])
@pytest.mark.parametrize("C", [1, 3, 4])
def test_remap_random_maps_vs_oracle(layout, dtype, C):
    need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(100 + C)
    B, H, W, Ho, Wo = 3, 45, 67, 52, 71
    img = (rng.integers(0, 256, (B, H, W, C)).astype(np.uint8) if dtype == np.uint8
           else rng.random((B, H, W, C)).astype(np.float32))
    mx = np.sort(rng.random((B, Wo)) * (W + 4) - 2, axis=1).astype(np.float32)
    my = np.sort(rng.random((B, Ho)) * (H + 4) - 2, axis=1).astype(np.float32)
    mx[:, :3] = [0.0, 1.0 / 64, 3.0 / 64]            # exact rounding ties
    src = dev(img if layout == "hwc" else np.transpose(img, (0, 3, 1, 2)))
    out = ops.remap_bilinear(src, dev(mx), dev(my), layout).cpu().numpy()
    if layout == "chw":
        out = np.transpose(out, (0, 2, 3, 1))
    for b in range(B):
        ref = hwc(ON.remap(img[b], mx[b], my[b]))
        assert np.array_equal(out[b], ref)


@pytest.mark.parametrize("gh,gw,H,W,Ho,Wo,transform", [
    (24, 24, 336, 336, 336, 336, "identity"), (24, 24, 336, 336, 500, 500, "sqrt"),
    (48, 48, 1344, 1344, 1344, 1344, "identity"), (24, 24, 100, 130, 90, 140, "square"),
    (7, 5, 97, 53, 64, 200, "exp")])
def test_maps_from_tokens_vs_oracle(gh, gw, H, W, Ho, Wo, transform):
    need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(gh * 1000 + W)
    B = 3
    tok = (rng.random((B, gh, gw)) ** 3).astype(np.float32)
    tok /= tok.sum(axis=(1, 2), keepdims=True)
    mx, my = ops.maps_from_tokens(dev(tok), (H, W), (Ho, Wo), transform, 2.0, 3.0)
    for b in range(B):
        full = ON.upsample_tokens_nearest(tok[b], H, W)
        rx, ry, _, _ = ON.inverse_maps(full, Wo, Ho, transform, 2.0, 3.0)
        assert np.abs(mx[b].cpu().numpy() - rx.astype(np.float32)).max() <= 1e-4
        assert np.abs(my[b].cpu().numpy() - ry.astype(np.float32)).max() <= 1e-4


def test_large_image_end_to_end_vs_oracle():
    """1344x1344 (BASELINE configs[2] size) and a non-square large case, noise images."""
    need_gpu()
    from attwarp_b200 import new_method
    rng = np.random.default_rng(5)
    for (h, w, nh, nw) in [(1344, 1344, 1344, 1344), (700, 2048, 900, 1500)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        att = rng.integers(0, 256, (h, w), dtype=np.uint8)
        out = new_method.warp_image_by_attention(img, att, nw, nh, transform="identity")
        ref = ON.warp_image_by_attention(img, att, nw, nh, "identity")
        diff = np.abs(out.astype(np.int32) - ref.astype(np.int32))
        assert diff.max() <= 1 and (diff != 0).mean() <= 1e-3


def test_error_behaviour(tmp_path):
    need_gpu()
    from attwarp_b200 import new_method
    img = np.zeros((8, 9, 3), np.uint8)
    with pytest.raises(ValueError):
        new_method.warp_image_by_attention(img, np.zeros((8, 8), np.float32), 9, 8)
    with pytest.raises(TypeError):
        new_method.warp_image_by_attention(img.astype(np.int32), np.zeros((8, 9)), 9, 8)
    assert new_method.set_transform_function("nope") == "identity"
    out = tmp_path / "x.png"
    assert new_method.save_warped_image("/nonexistent.png", np.zeros((4, 4)), None, None, str(out)) is False
    assert not out.exists()


@pytest.mark.parametrize("H,W", [(1, 16), (63, 336), (64, 336), (65, 1024), (200, 1040), (130, 1344), (70, 2064)])
def test_u8_identity_marginals_fast_path(H, W):
    """uint8 attention maps with rows of 16-byte multiples take the integer marginals kernel; it must
    agree with the float64 oracle profile sums and with the generic kernel (same map as float32)."""
    need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(H * 31 + W)
    B = 3
    att = rng.integers(0, 256, (B, H, W), dtype=np.uint8)
    att[1] = 0                                             # all-zero map: + 1e-9 only -> identity warp
    att[2, :, : W // 2] = 0
    Ho, Wo = max(H, 2) + 3, W + 5
    mx, my = ops.maps_from_attention(dev(att), (Ho, Wo), "identity")
    gx, gy = ops.maps_from_attention(dev(att.astype(np.float32)), (Ho, Wo), "identity")
    assert np.abs(mx.cpu().numpy() - gx.cpu().numpy()).max() <= 1e-4
    assert np.abs(my.cpu().numpy() - gy.cpu().numpy()).max() <= 1e-4
    for b in range(B):
        _, rx, ry = ON.warp_image_by_attention(np.zeros((H, W, 3), np.uint8), att[b], Wo, Ho, "identity",
                                               return_maps=True)
        assert np.abs(mx[b].cpu().numpy() - rx).max() <= 1e-4
        assert np.abs(my[b].cpu().numpy() - ry).max() <= 1e-4


@pytest.mark.parametrize("H,W,transform", [(1, 4, "identity"), (63, 336, "sqrt"), (130, 512, "identity"),
                                            (70, 516, "square"), (129, 1028, "identity"), (66, 1344, "sqrt"),
                                            (40, 333, "identity")])
def test_f32_marginals_rows_kernel(H, W, transform):
    """float32 attention maps with rows of 4-float multiples take the row-owning float64 kernel (W = 333
    keeps the generic one): maps must match the float64 oracle; gt_marginals must match its definition."""
    need_gpu()
    from attwarp_b200 import ops, checkpoint_utils as CU
    rng = np.random.default_rng(H * 17 + W)
    B = 3
    att = (rng.random((B, H, W)) ** 3).astype(np.float32)
    att[1, :, W // 3:] = 0.0
    att[2] -= 0.2                                          # negatives are clamped
    Ho, Wo = max(H, 2) + 3, W + 5
    mx, my = ops.maps_from_attention(dev(att), (Ho, Wo), transform)
    for b in range(B):
        _, rx, ry = ON.warp_image_by_attention(np.zeros((H, W, 3), np.uint8), att[b], Wo, Ho, transform,
                                               return_maps=True)
        assert np.abs(mx[b].cpu().numpy() - rx).max() <= 1e-4
        assert np.abs(my[b].cpu().numpy() - ry).max() <= 1e-4
    px, py = CU.gt_marginals(dev(att)[:, None])
    a = np.maximum(att.astype(np.float64), 0.0)
    rpx = a.sum(1) / np.maximum(a.sum(1).sum(1, keepdims=True), 1e-6)
    rpy = a.sum(2) / np.maximum(a.sum(2).sum(1, keepdims=True), 1e-6)
    assert np.abs(px.cpu().numpy() - rpx).max() <= 1e-5 * rpx.max() + 1e-9
    assert np.abs(py.cpu().numpy() - rpy).max() <= 1e-5 * rpy.max() + 1e-9


@pytest.mark.parametrize("dtype", ["u8", "f32", "f64"])
@pytest.mark.parametrize("transform", ["identity", "square", "sqrt", "exp", "log"])
@pytest.mark.parametrize("H,W", [(48, 336), (37, 203)])
def test_marginals_every_transform_and_dtype(dtype, transform, H, W):
    """The marginals kernels are instantiated once per transform (float32 / float64 maps) and uint8 maps go
    through a 256-entry table of the transformed values: every (dtype, transform) pair, on rows the row-owning
    kernels take (W = 336) and on rows only the generic kernel takes (W = 203), against the float64 oracle
    (new_method.py:207-216 with the registry of :133-188)."""
    need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(H * 7 + W + len(transform))
    B = 2
    if dtype == "u8":
        att = rng.integers(0, 256, (B, H, W), dtype=np.uint8)
        att[1, :, : W // 2] = 0
    else:
        att = (rng.random((B, H, W)) ** 3).astype(np.float32 if dtype == "f32" else np.float64)
        att[1] -= 0.2                                      # negatives are clamped
    # exp of byte values needs a scale that keeps float64 finite and the profile non-degenerate
    es, ed = (0.02, 3.0) if dtype == "u8" else (2.0, 3.0)
    Ho, Wo = H + 3, W + 5
    mx, my = ops.maps_from_attention(dev(att), (Ho, Wo), transform, es, ed)
    for b in range(B):
        _, rx, ry = ON.warp_image_by_attention(np.zeros((H, W, 3), np.uint8), att[b], Wo, Ho, transform, es, ed,
                                               return_maps=True)
        assert np.abs(mx[b].cpu().numpy() - rx).max() <= 1e-4
        assert np.abs(my[b].cpu().numpy() - ry).max() <= 1e-4


@pytest.mark.parametrize("transform", ["sqrt", "square", "identity"])
def test_f32_marginals_extreme_values(transform):
    """The float32-pair evaluation of sqrt / square (profiles.cu: sqrt_pair) on the inputs that leave its
    fast path: zeros, denormals, values below 1e-27, large finite values -- maps still match the float64 oracle."""
    need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(11)
    H, W = 40, 336
    att = (rng.random((3, H, W)) ** 3).astype(np.float32)
    att[0, ::3, ::5] = 0.0
    att[0, 1::7, 2::11] = 1e-40            # denormal
    att[0, 2::7, 3::11] = 3e-30            # normal, below the fast path's range
    att[1] *= 1e-20                        # a whole map of tiny values (sqrt ~1e-10, square underflows to ~0)
    att[2] *= 1e15 if transform == "square" else 1e30
    Ho, Wo = H + 5, W + 7
    mx, my = ops.maps_from_attention(dev(att), (Ho, Wo), transform)
    for b in range(3):
        _, rx, ry = ON.warp_image_by_attention(np.zeros((H, W, 3), np.uint8), att[b], Wo, Ho, transform,
                                               return_maps=True)
        assert np.abs(mx[b].cpu().numpy() - rx).max() <= 1e-4
        assert np.abs(my[b].cpu().numpy() - ry).max() <= 1e-4


def test_host_entry_point_from_several_threads():
    """new_method.warp_image_by_attention keeps per-thread device and pinned scratch (api.cu: HostArena) that regrows
    when the sizes change: six threads, sizes changing from call to call, every result within 1 LSB of the oracle."""
    need_gpu()
    import threading
    from attwarp_b200 import new_method
    rng = np.random.default_rng(1)
    cases = [(rng.integers(0, 256, (H, W, 3), dtype=np.uint8), rng.integers(0, 256, (H, W), dtype=np.uint8), Wo, Ho)
             for (H, W, Wo, Ho) in ((336, 336, 336, 336), (200, 333, 500, 400), (64, 48, 90, 70), (500, 500, 336, 336))]
    refs = [ON.warp_image_by_attention(i, a, wo, ho, "identity") for i, a, wo, ho in cases]
    bad = []

    def work(tid):
        for k in range(24):
            j = (tid + k) % len(cases)
            i, a, wo, ho = cases[j]
            out = new_method.warp_image_by_attention(i, a, wo, ho, transform="identity")
            if out.shape != refs[j].shape or np.abs(out.astype(int) - refs[j].astype(int)).max() > 1:
                bad.append((tid, k, j))

    threads = [threading.Thread(target=work, args=(t,)) for t in range(6)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    assert not bad, bad[:5]
