"""GPU: the attention overlay of ``save_warped_image`` on the device (``ops.attention_overlay``,
``image_io.warp_files(overlay_paths=..., original_paths=...)``).  Every comparison is bit-equal: against the
unmodified reference's overlays in tests/golden/save_warped.npz, and against ``oracle/overlay.py`` (itself held to the
host expression with real cv2 by tests/test_overlay_host.py) on the driver sizes, token maps on odd and misaligned
images, mixed-size lists, the whole JET table, an alpha sweep, each dtype's zero branch and NaN maps.  Each launch
path the launcher can choose is asserted through torch.profiler."""

import io
import json
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from gpu_util import need_gpu
from oracle import numpy_path as ON
from oracle import overlay as OV

pytestmark = pytest.mark.gpu

ALPHAS = (0.0, 0.3, 0.5, 0.7, 1.0)
MM_CHUNK, BLEND_PIX = 65536, 4096           # attention values per min/max CTA, pixels per blend CTA (overlay.cu)
KERNEL_RE = re.compile(r"(overlay_(?:minmax|minmax_tokens|blend|blend_tokens)_kernel)(<[^>]*>)?")
_LUTS = {}


def _ops():
    need_gpu()
    from attwarp_b200 import ops
    return ops


def _pair_lut(alpha):
    """[256, 256] uint8: the oracle's addWeighted of every (heat, base) byte pair (it is elementwise)."""
    if alpha not in _LUTS:
        h, b = np.meshgrid(np.arange(256, dtype=np.uint8), np.arange(256, dtype=np.uint8), indexing="ij")
        _LUTS[alpha] = OV.add_weighted(h, b, alpha)
    return _LUTS[alpha]


def oracle(image, att, alpha=0.5):
    """OV.attention_overlay through the pair table: same bytes, fast enough for 1344^2 batches."""
    base = OV.as_bgr(image)
    att = np.asarray(att)
    assert att.shape == base.shape[:2]
    return _pair_lut(alpha)[OV.JET[OV.heat_index(att)], base]


def oracle_tokens(image, tok, alpha=0.5):
    H, W = OV.as_bgr(image).shape[:2]
    return oracle(image, ON.upsample_tokens_nearest(np.asarray(tok, np.float32), H, W), alpha)


_TORCH = {np.dtype(np.uint8): torch.uint8, np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64}


def _misaligned(a, offset):
    """A CUDA copy of `a` whose base lies `offset` bytes (a multiple of its item size) past a 512-byte boundary."""
    a = np.ascontiguousarray(a)
    buf = torch.empty(a.nbytes + offset + 16, dtype=torch.uint8, device="cuda")
    view = buf[offset:offset + a.nbytes]
    view.copy_(torch.from_numpy(a.reshape(-1).view(np.uint8)).cuda())
    return view.view(_TORCH[a.dtype]).view(a.shape)


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _assert_equal(got, want, what):
    got = got.cpu().numpy()
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    if not np.array_equal(got, want):
        bad = np.argwhere((got != want).any(-1))
        y, x = bad[0]
        raise AssertionError(f"{what}: {len(bad)} pixels differ, first at ({y}, {x}): {got[y, x]} vs {want[y, x]}")


def _image(rng, h, w, c=3):
    return rng.integers(0, 256, (h, w, c) if c else (h, w), dtype=np.uint8)


def _launches(events):
    """(kernel, template args, grid) of every overlay launch among a trace's events."""
    out = []
    for e in events:
        if e.get("cat") == "kernel":
            m = KERNEL_RE.search(e.get("name", ""))
            if m:
                out.append((m.group(1), (m.group(2) or "").replace(" ", ""), tuple(e.get("args", {}).get("grid", ()))))
    return out


def _has_both_launches(launched):
    names = [n for n, _, _ in launched]
    return any("minmax" in n for n in names) and any("blend" in n for n in names)


def _profiled(fn, path, complete=lambda events: _has_both_launches(_launches(events)), attempts=3):
    """(fn's result, the trace's events).  torch.profiler can miss a kernel record of its window (seen on the first
    launch of a window inside a long session), so the window opens with a kernel of its own, and a trace in which
    `complete` finds a launch missing is taken again, up to `attempts` times; what the launches must be is asserted
    by the caller."""
    for _ in range(attempts):
        torch.cuda.synchronize()
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                torch.profiler.ProfilerActivity.CUDA]) as prof:
            torch.ones(1, device="cuda").add_(1)
            res = fn()
            torch.cuda.synchronize()
        prof.export_chrome_trace(str(path))
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
        if not any(e.get("cat") == "kernel" for e in events):
            pytest.skip("torch.profiler reported no CUDA kernel events: the launched kernels are not checked")
        if complete(events):
            break
    return res, events


# ---------------------------------------------------------------------------------------------- 1. golden cases
@pytest.mark.parametrize("name", ["path_list_sqrt", "att_3d_mean", "pil_att_exp_inv", "gray_input"])
def test_golden_overlays_of_the_unmodified_reference(name):
    ops = _ops()
    import cv2
    gs = np.load(os.path.join(GOLDEN_DIR, "save_warped.npz"))
    image_rgb, att = gs[name + "/image_rgb"], gs[name + "/att"]
    image = cv2.cvtColor(image_rgb, cv2.COLOR_RGB2BGR)          # save_warped_image's coercions
    if att.ndim == 3:
        att = np.mean(att, axis=2)
    want = gs[name + "/overlay_bgr"]
    got = ops.attention_overlay([_cuda(image)], att=[_cuda(att)])
    torch.cuda.synchronize()
    _assert_equal(got[0], want, name)
    if image_rgb.ndim == 2:                                      # the grey image itself: C = 1, replicated
        _assert_equal(ops.attention_overlay([_cuda(image_rgb)], att=[_cuda(att)])[0], want, name + " (grey input)")


# ---------------------------------------------------------------------------------------------- 2. driver sizes
@pytest.mark.parametrize("B,gh,H", [(256, 24, 336), (64, 48, 1344)])
def test_mota_masks_at_driver_sizes(B, gh, H):
    ops = _ops()
    rng = np.random.default_rng(B + H)
    tok = torch.from_numpy((rng.random((B, gh, gh)) ** 3).astype(np.float32)).cuda()
    mask = ops.mota_mask(tok, (H, H))
    imgs = torch.from_numpy(rng.integers(0, 256, (B, H, H, 3), dtype=np.uint8)).cuda()
    got = ops.attention_overlay(imgs, att=mask)
    torch.cuda.synchronize()
    m, im = mask.cpu().numpy(), imgs.cpu().numpy()
    for b in range(B):
        _assert_equal(got[b], oracle(im[b], m[b]), f"mota mask {B} x {H}^2, image {b}")


TOKEN_SIZES = [(336, 336), (1344, 1344), (500, 375), (97, 53), (1, 77), (61, 1), (1, 1), (337, 333), (35, 334),
               (36, 335), (5, 2)]


@pytest.mark.parametrize("grid", [24, 48])
@pytest.mark.parametrize("offset", [0, 1, 7, 15])
def test_token_maps_on_odd_sizes_and_misaligned_bases(grid, offset):
    ops = _ops()
    rng = np.random.default_rng(grid * 100 + offset)
    imgs = [_image(rng, h, w) for h, w in TOKEN_SIZES]
    tok = (rng.random((len(imgs), grid, grid)) ** 3).astype(np.float32)
    dev = [_misaligned(im, (offset + k) % 16 if offset else 0) for k, im in enumerate(imgs)]
    got = ops.attention_overlay(dev, tok=_cuda(tok))
    torch.cuda.synchronize()
    for k, im in enumerate(imgs):
        _assert_equal(got[k], oracle_tokens(im, tok[k]), f"tokens {grid}^2 -> {im.shape[:2]}, offset {offset}")


@pytest.mark.parametrize("dtype", [np.uint8, np.float32, np.float64])
@pytest.mark.parametrize("offset", [0, 3])
def test_maps_on_odd_sizes_and_misaligned_bases(dtype, offset):
    ops = _ops()
    rng = np.random.default_rng(offset + np.dtype(dtype).itemsize)
    sizes = [(336, 336), (500, 375), (97, 53), (1, 77), (61, 1), (337, 333), (35, 334), (36, 335)]
    imgs = [_image(rng, h, w) for h, w in sizes]
    atts = [(rng.integers(0, 256, s, dtype=np.uint8) if dtype == np.uint8 else (rng.standard_normal(s) * 3).astype(dtype))
            for s in sizes]
    got = ops.attention_overlay([_misaligned(im, offset + k % 5 if offset else 0) for k, im in enumerate(imgs)],
                                att=[_misaligned(a, offset * (1 + k % 3) * a.itemsize) for k, a in enumerate(atts)])
    torch.cuda.synchronize()
    for k in range(len(sizes)):
        _assert_equal(got[k], oracle(imgs[k], atts[k]), f"{np.dtype(dtype)} map {sizes[k]}, offset {offset}")


def _random_sizes(rng, n):
    hs = rng.integers(1, 900, n)
    ws = rng.integers(1, 900, n)
    return [(int(h), int(w)) for h, w in zip(hs, ws)]


@pytest.mark.parametrize("kind", ["tokens", "f32", "u8"])
def test_64_random_sizes_in_one_call_and_batch_independence(kind):
    ops = _ops()
    rng = np.random.default_rng({"tokens": 1, "f32": 2, "u8": 3}[kind])
    sizes = _random_sizes(rng, 64)
    imgs = [_image(rng, h, w, c=0 if k % 7 == 3 else 3) for k, (h, w) in enumerate(sizes)]
    dev = [_cuda(im) for im in imgs]
    if kind == "tokens":
        tok = (rng.random((64, 24, 24)) ** 2).astype(np.float32)
        tok[5] = 0.5                                          # a constant map: the zero branch, next to others
        got = ops.attention_overlay(dev, tok=_cuda(tok))
        want = [oracle_tokens(im, tok[k]) for k, im in enumerate(imgs)]
        single = [ops.attention_overlay([dev[k]], tok=_cuda(tok[k:k + 1]))[0] for k in range(64)]
    else:
        atts = [(rng.random(s) ** 3).astype(np.float32) if kind == "f32" else rng.integers(0, 256, s, dtype=np.uint8)
                for s in sizes]
        got = ops.attention_overlay(dev, att=[_cuda(a) for a in atts])
        want = [oracle(im, atts[k]) for k, im in enumerate(imgs)]
        single = [ops.attention_overlay([dev[k]], att=[_cuda(atts[k])])[0] for k in range(64)]
    torch.cuda.synchronize()
    for k in range(64):
        _assert_equal(got[k], want[k], f"{kind} list, image {k} {sizes[k]}")
        assert torch.equal(got[k], single[k]), f"{kind}: image {k} differs from its single-image call"


# ---------------------------------------------------------------------------------------------- 4-6. table, alpha, branches
def test_whole_jet_table():
    ops = _ops()
    import cv2
    ramp = np.arange(256, dtype=np.uint8).reshape(1, 256)
    base = np.zeros((1, 256, 3), np.uint8)
    got = ops.attention_overlay([_cuda(base)], att=[_cuda(ramp)], alpha=1.0)[0]
    torch.cuda.synchronize()
    _assert_equal(got, cv2.applyColorMap(ramp, cv2.COLORMAP_JET), "alpha 1 on the 0..255 ramp")


@pytest.mark.parametrize("alpha", ALPHAS + (0.25, 0.9, -0.5, 1.5))
def test_alpha_sweep(alpha):
    ops = _ops()
    rng = np.random.default_rng(int(alpha * 100) + 1000)
    imgs = [_image(rng, 129, 131), _image(rng, 64, 64, c=0)]
    atts = [rng.random((129, 131)).astype(np.float32), rng.integers(0, 256, (64, 64), dtype=np.uint8)]
    got = ops.attention_overlay([_cuda(imgs[0])], att=[_cuda(atts[0])], alpha=alpha)
    got += ops.attention_overlay([_cuda(imgs[1])], att=[_cuda(atts[1])], alpha=alpha)
    tok = (rng.random((2, 24, 24)) ** 3).astype(np.float32)
    got_t = ops.attention_overlay([_cuda(im) for im in imgs], tok=_cuda(tok), alpha=alpha)
    torch.cuda.synchronize()
    for k in range(2):
        _assert_equal(got[k], oracle(imgs[k], atts[k], alpha), f"alpha {alpha}, map {k}")
        _assert_equal(got_t[k], oracle_tokens(imgs[k], tok[k], alpha), f"alpha {alpha}, tokens {k}")


def _branch_maps(dtype, H, W, rng):
    if dtype == np.uint8:
        two = np.where(rng.random((H, W)) < 0.5, 7, 8).astype(np.uint8)
        return {"constant": np.full((H, W), 42, np.uint8), "two_values": two}
    t = np.dtype(dtype).type
    out = {"constant": np.full((H, W), 0.25, dtype)}
    one = t(1.0)
    for name, step in (("one_ulp", np.nextafter(one, t(2)) - one), ("below_eps", t(5e-10)), ("above_eps", t(2e-9))):
        m = np.full((H, W), one, dtype)
        m[rng.random((H, W)) < 0.3] = t(one + t(step))
        out[name] = m
    tiny = np.full((H, W), t(1e-12), dtype)
    sel = rng.random((H, W)) < 0.3
    tiny[sel] = t(1e-12 + 5e-10)
    out["tiny_below_eps"] = tiny
    tiny2 = np.full((H, W), t(1e-12), dtype)
    tiny2[sel] = t(1e-12 + 2e-9)
    out["tiny_above_eps"] = tiny2
    nan = (rng.random((H, W)) * 10 - 3).astype(dtype)
    nan[H - 1, W - 1] = np.nan                               # in the last min/max chunk of the image
    out["nan_last"] = nan
    nan0 = (rng.random((H, W)) * 10 - 3).astype(dtype)
    nan0[0, 0] = np.nan
    out["nan_first"] = nan0
    out["all_nan"] = np.full((H, W), np.nan, dtype)
    return out


@pytest.mark.parametrize("dtype", [np.uint8, np.float32, np.float64])
@pytest.mark.parametrize("hw", [(61, 67), (400, 401)])
def test_zero_branch_and_nan_maps(dtype, hw):
    ops = _ops()
    rng = np.random.default_rng(hw[0] + np.dtype(dtype).itemsize)
    maps = _branch_maps(dtype, *hw, rng)
    img = _image(rng, *hw)
    names = list(maps)
    got = ops.attention_overlay([_cuda(img)] * len(names), att=[_cuda(maps[k]) for k in names])
    torch.cuda.synchronize()
    for k, name in enumerate(names):
        _assert_equal(got[k], oracle(img, maps[name]), f"{np.dtype(dtype)} {name} {hw}")
    if dtype == np.float32:                                  # NaN token maps: NaN in a reached token
        tok = rng.random((2, 24, 24)).astype(np.float32)
        tok[0, 23, 23] = np.nan
        tok[1] = 0.5
        got = ops.attention_overlay([_cuda(img)] * 2, tok=_cuda(tok))
        torch.cuda.synchronize()
        for k in range(2):
            _assert_equal(got[k], oracle_tokens(img, tok[k]), f"token map {k} {hw}")


def test_tokens_the_upsampling_never_reaches_are_ignored():
    """An image smaller than its token grid reads a subset of the tokens: lo and hi are theirs only."""
    ops = _ops()
    rng = np.random.default_rng(9)
    img = _image(rng, 7, 5)
    tok = rng.random((1, 48, 48)).astype(np.float32)
    reached_y = set(((np.arange(7) * 48) // 7).tolist())
    reached_x = set(((np.arange(5) * 48) // 5).tolist())
    ys = [y for y in range(48) if y not in reached_y]
    xs = [x for x in range(48) if x not in reached_x]
    tok[0, ys[0], :] = 1e6
    tok[0, :, xs[-1]] = -1e6
    tok[0, ys[1], xs[1]] = np.nan
    got = ops.attention_overlay([_cuda(img)], tok=_cuda(tok))[0]
    torch.cuda.synchronize()
    want = oracle_tokens(img, tok[0])
    assert np.unique(OV.heat_index(ON.upsample_tokens_nearest(tok[0], 7, 5))).size > 10
    _assert_equal(got, want, "7 x 5 image, 48^2 tokens")


# ---------------------------------------------------------------------------------------------- 7. launch paths
def _path_case(rng, dtype, vec, hw):
    imgs = [_image(rng, *hw), _image(rng, 33, 35, c=0)]
    shapes = [hw, (33, 35)]
    if dtype == "tokens":
        atts = (rng.random((2, 24, 24)) ** 2).astype(np.float32)
    elif dtype == np.uint8:
        atts = [rng.integers(0, 256, s, dtype=np.uint8) for s in shapes]
    else:
        atts = [(rng.standard_normal(s)).astype(dtype) for s in shapes]
        for a in atts:                                        # the extremes in the image's last min/max chunk
            a.reshape(-1)[-1] = 40.0
            a.reshape(-1)[-2] = -40.0
    if dtype == np.uint8:
        for a in atts:
            a[a == 0] = 1
            a[a == 255] = 254
            a.reshape(-1)[-1] = 255
            a.reshape(-1)[-2] = 0
    off = 0 if vec else 1
    dev_imgs = [_misaligned(im, off) for im in imgs]
    if dtype == "tokens":
        return imgs, atts, dev_imgs, dict(tok=_cuda(atts))
    return imgs, atts, dev_imgs, dict(att=[_misaligned(a, 0) for a in atts])


PATHS = [(dt, vec, hw) for dt in (np.uint8, np.float32, np.float64, "tokens") for vec in (True, False)
         for hw in ((200, 300), (1344, 1344))]


@pytest.mark.parametrize("dtype,vec,hw", PATHS, ids=[f"{d if isinstance(d, str) else np.dtype(d).name}-"
                                                     f"{'vec' if v else 'bytes'}-{h[0]}x{h[1]}" for d, v, h in PATHS])
def test_launch_paths(dtype, vec, hw, tmp_path):
    """4-pixel vs byte path (chosen by the bases' alignment), one vs several min/max CTAs per image (200 x 300 =
    60 000 values fit one CTA, 1344^2 takes 28): the launched kernels and grids, and the bytes."""
    ops = _ops()
    rng = np.random.default_rng(hash((str(dtype), vec, hw)) % 2 ** 32)
    imgs, atts, dev_imgs, kw = _path_case(rng, dtype, vec, hw)
    got, events = _profiled(lambda: ops.attention_overlay(dev_imgs, **kw), tmp_path / "trace.json")
    launched = _launches(events)
    tokens = dtype == "tokens"
    tname = {np.uint8: "unsignedchar", np.float32: "float", np.float64: "double"}.get(dtype)
    if tokens:
        want_names = [("overlay_minmax_tokens_kernel", ""), ("overlay_blend_tokens_kernel", f"<{str(vec).lower()}>")]
        mm_grid = 2
    else:
        want_names = [("overlay_minmax_kernel", f"<{tname}>"), ("overlay_blend_kernel", f"<{tname},{str(vec).lower()}>")]
        mm_grid = -(-hw[0] * hw[1] // MM_CHUNK) + 1
    assert [(n, t) for n, t, _ in launched] == want_names, launched
    grids = [g for _, _, g in launched]
    if grids[0] and grids[1]:
        assert grids[0][0] == mm_grid, f"min/max grid {grids[0]}, expected {mm_grid}"
        assert grids[1][0] == -(-hw[0] * hw[1] // BLEND_PIX) + -(-33 * 35 // BLEND_PIX), grids[1]
    for k in range(2):
        want = oracle_tokens(imgs[k], atts[k]) if tokens else oracle(imgs[k], atts[k])
        _assert_equal(got[k], want, f"path {dtype} vec={vec} {hw} image {k}")


def test_large_image_extremes_in_every_chunk():
    """A 1344^2 float32 map whose min and max sit in different, late min/max chunks, and a NaN in the 27th."""
    ops = _ops()
    rng = np.random.default_rng(77)
    img = _image(rng, 1344, 1344)
    base = rng.random((1344, 1344)).astype(np.float32)
    a, b, c = base.copy(), base.copy(), base.copy()
    a.reshape(-1)[20 * MM_CHUNK + 5] = 3.0
    a.reshape(-1)[27 * MM_CHUNK + 9] = -2.0
    b.reshape(-1)[26 * MM_CHUNK] = np.nan
    c.reshape(-1)[-1] = 7.0
    got = ops.attention_overlay([_cuda(img)] * 3, att=[_cuda(x) for x in (a, b, c)])
    torch.cuda.synchronize()
    for k, m in enumerate((a, b, c)):
        _assert_equal(got[k], oracle(img, m), f"1344^2 map {k}")


# ---------------------------------------------------------------------------------------------- 8. warp_files
def _jpegs(rng, sizes):
    from PIL import Image
    files = []
    for h, w in sizes:
        y, x = np.mgrid[0:h, 0:w].astype(np.float64)
        img = np.stack([127 + 100 * np.sin(x / 17 + y / 23), 127 + 90 * np.cos(x / 11 - y / 29),
                        255 * (x + y) / (h + w)], -1) + rng.normal(0, 6, (h, w, 3))
        buf = io.BytesIO()
        Image.fromarray(np.clip(np.rint(img), 0, 255).astype(np.uint8)).save(buf, format="JPEG", quality=90)
        files.append(buf.getvalue())
    return files


@pytest.mark.parametrize("on_device_png", [False, True])
def test_warp_files_writes_overlay_and_original(on_device_png, tmp_path):
    need_gpu()
    import cv2
    from attwarp_b200 import image_io
    rng = np.random.default_rng(31)
    sizes = [(224, 224), (336, 500), (301, 223), (97, 53)]
    n = len(sizes)
    files = _jpegs(rng, sizes)
    tok = rng.random((n, 24, 24)) ** 3
    tok = torch.from_numpy((tok / tok.sum(axis=(1, 2), keepdims=True)).astype(np.float32))
    out_sizes = [(224, 224), (500, 500), (301, 223), (60, 40)]
    p = lambda kind: [str(tmp_path / f"{kind}{k}.png") for k in range(n)]   # noqa: E731
    assert image_io.warp_files(files, tok, p("plain"), out_sizes, on_device_png=on_device_png) == [True] * n
    run = lambda: image_io.warp_files(files, tok, p("warped"), out_sizes, on_device_png=on_device_png,  # noqa: E731
                                      overlay_paths=p("overlay"), original_paths=p("orig"))
    if on_device_png:
        res, events = _profiled(run, tmp_path / "trace.json", complete=lambda ev: _has_both_launches(_launches(ev)) and any(
            e.get("cat") == "kernel" and "png_segment_kernel" in e.get("name", "") for e in ev))
    else:
        res = run()
    assert res == [True] * (3 * n)
    decoded = [t.cpu().numpy() for t in image_io.decode_jpeg_batch(files)]
    for k in range(n):
        with open(p("plain")[k], "rb") as f1, open(p("warped")[k], "rb") as f2:
            assert f1.read() == f2.read(), f"warped file {k} differs from a run without the new keywords"
        orig = cv2.imread(p("orig")[k], cv2.IMREAD_UNCHANGED)
        assert np.array_equal(orig, decoded[k]), f"original {k}"
        ov = cv2.imread(p("overlay")[k], cv2.IMREAD_UNCHANGED)
        assert np.array_equal(ov, oracle_tokens(decoded[k], tok[k].numpy())), f"overlay {k}"
    if on_device_png:
        segs = [e for e in events if e.get("cat") == "kernel" and "png_segment_kernel" in e.get("name", "")]
        assert len(segs) == 1, f"{len(segs)} png_segment_kernel launches for {3 * n} files"
    # overlays only, and the keyword counts are checked
    assert image_io.warp_files(files, tok, p("w2"), out_sizes, on_device_png=on_device_png,
                               overlay_paths=p("o2"), overlay_alpha=0.3) == [True] * (2 * n)
    ov = cv2.imread(p("o2")[1], cv2.IMREAD_UNCHANGED)
    assert np.array_equal(ov, oracle_tokens(decoded[1], tok[1].numpy(), 0.3))
    with pytest.raises(ValueError):
        image_io.warp_files(files, tok, p("w3"), out_sizes, overlay_paths=p("o3")[:2])
    with pytest.raises(ValueError):
        image_io.warp_files(files, tok, p("w3"), out_sizes, original_paths=p("r3")[:1])


# ---------------------------------------------------------------------------------------------- 9. errors
def test_every_value_error():
    ops = _ops()
    img = torch.zeros(4, 5, 3, dtype=torch.uint8, device="cuda")
    att = torch.zeros(4, 5, dtype=torch.float32, device="cuda")
    tok = torch.zeros(1, 3, 3, dtype=torch.float32, device="cuda")
    bad = [
        dict(images=[img], att=[torch.zeros(4, 6, device="cuda")]),                       # shape mismatch
        dict(images=[img], att=[torch.zeros(24, 24, device="cuda")]),                     # resize: out of scope
        dict(images=[torch.zeros(4, 5, 4, dtype=torch.uint8, device="cuda")], att=[att]),  # C = 4
        dict(images=[torch.zeros(4, 5, 2, dtype=torch.uint8, device="cuda")], att=[att]),  # C = 2
        dict(images=[img.float()], att=[att]),                                             # non-uint8 image
        dict(images=[img], att=[att.to(torch.float16)]),                                  # attention dtype
        dict(images=[img], att=[att.to(torch.int32)]),
        dict(images=[img], tok=tok.double()),                                             # token dtype
        dict(images=[img], att=[att], tok=tok),                                           # both
        dict(images=[img]),                                                               # neither
        dict(images=[img], tok=torch.zeros(2, 3, 3, device="cuda")),                     # token count
        dict(images=[img], att=[att, att]),                                               # map count
        dict(images=[img], att=[att.cpu()]),                                              # mixed devices
        dict(images=[img.cpu()], att=[att.cpu()]),                                        # not on a CUDA device
        dict(images=[img], att=[att], alpha=float("nan")),                                # alpha
        dict(images=[img], att=[att], alpha=float("inf")),
        dict(images=[img, img], att=[att, att.double()]),                                 # mixed map dtypes
        dict(images=img, att=[att]),                                                      # 3-D tensor of images
    ]
    for k, kw in enumerate(bad):
        with pytest.raises(ValueError):
            ops.attention_overlay(**kw)
    assert ops.attention_overlay([], att=[]) == []
    assert ops.attention_overlay([], tok=torch.zeros(0, 3, 3, device="cuda")) == []
