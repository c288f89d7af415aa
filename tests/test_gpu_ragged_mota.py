"""``ops.warp_ragged_from_mota_tokens`` / ``attwarp_warp_ragged_from_mask``: a mixed-size list warped by the drivers'
own attention -- per image blend_mask's mask (revise_mask, then Pillow's LANCZOS resize to that image's size) and
save_warped_image(..., "identity") -- with one fused LANCZOS + marginals launch for the whole list.

Bars: an image the fused kernel takes (an up-scaling whose tiles fit the tensor-core kernel) has maps and pixels
bit-identical to ``ops.maps_from_mota_tokens`` + ``ops.remap_bilinear`` on that image alone; one it does not take
(down-scaling, smaller than or close to the token grid) bit-identical to ``ops.warp_ragged_from_attention`` on its
``ops.mota_mask`` alone, and within one float32 ulp of ``maps_from_mota_tokens`` (the float64 sums are added in
another order).  Against the host oracle (Pillow's LANCZOS restated, the reference's warp_image_by_attention):
maps within 1e-3 px, pixels equal to the cv2.remap restatement fed the returned maps.

    python -m pytest tests/test_gpu_ragged_mota.py -m gpu
"""

import ctypes as C
import os

import numpy as np
import pytest
import torch

from oracle import mask_path as OM
from oracle import numpy_path as ON

GH = GW = 24

# (H, W, Ho, Wo): fused up-scalings (odd sizes, W % 4 != 0, H != W, outputs of other sizes, 24..2048 per axis);
# images the fused kernel does not take: down-scaled (20 x 16), one axis at the grid (24 x 500), close to the grid
# (30 x 40: an up-scaling the tensor-core tiles do not fit), tiny (3 x 5)
FUSED = [(336, 336, 336, 336), (500, 333, 500, 500), (2048, 224, 1000, 300), (97, 1501, 97, 1500), (1344, 1344, 700, 700),
         (613, 2047, 613, 2047), (225, 226, 250, 190), (1999, 61, 1999, 61)]
UNFUSED = [(20, 16, 20, 16), (24, 500, 30, 500), (30, 40, 32, 41), (3, 5, 7, 5)]


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _tok(n, seed):
    rng = np.random.default_rng(seed)
    return torch.from_numpy(rng.random((n, GH, GW)).astype(np.float32) ** 2).cuda()


def _image(H, W, Cc, rng):
    return torch.from_numpy(rng.integers(0, 256, (H, W, Cc), dtype=np.uint8)).cuda()


def _fused(H, W):
    """Whether the fused kernel takes an image of these test lists: an up-scaling of both axes whose 16-row tiles tap
    at most 16 of the 24 token rows (H >= 48 is enough; the lists keep every other image below 44 rows or 25 columns)."""
    return H >= 48 and W > GW


def _per_image(ops, tok, img, Ho, Wo, inv, fused):
    """The same image warped on its own: the uniform fused call, or (not fused) the ragged-attention call on its mask."""
    H, W = img.shape[:2]
    if fused:
        mx, my = ops.maps_from_mota_tokens(tok[None], (H, W), (Ho, Wo), apply_inverse=inv)
        return ops.remap_bilinear(img[None], mx, my)[0], mx[0], my[0]
    mask = ops.mota_mask(tok[None], (H, W))[0]
    outs, mxs, mys = ops.warp_ragged_from_attention([mask], [img], [(Ho, Wo)], apply_inverse=inv, return_maps=True)
    return outs[0], mxs[0], mys[0]


def _bits(t):
    return t.cpu().numpy().view(np.int32)


def _check_list(ops, tok, imgs, sizes, inv):
    outs, mxs, mys = ops.warp_ragged_from_mota_tokens(tok, imgs, [(s[2], s[3]) for s in sizes], apply_inverse=inv,
                                                      return_maps=True)
    for k, (img, s) in enumerate(zip(imgs, sizes)):
        fused = _fused(s[0], s[1])
        ref, rx, ry = _per_image(ops, tok[k], img, s[2], s[3], inv, fused)
        assert np.array_equal(_bits(mxs[k]), _bits(rx)), (k, s, "map_x")
        assert np.array_equal(_bits(mys[k]), _bits(ry)), (k, s, "map_y")
        assert torch.equal(outs[k], ref), (k, s, "pixels")
        if not fused:        # and within one float32 ulp of the uniform call, whose sums run in another order
            ux, uy = ops.maps_from_mota_tokens(tok[k][None], (s[0], s[1]), (s[2], s[3]), apply_inverse=inv)
            for got, want in ((mxs[k], ux[0]), (mys[k], uy[0])):
                ulp = np.abs(_bits(got).astype(np.int64) - _bits(want).astype(np.int64))
                assert ulp.max() <= 1, (k, s, int(ulp.max()))
    return outs, mxs, mys


@pytest.mark.gpu
@pytest.mark.parametrize("Cc", [1, 3, 4])
@pytest.mark.parametrize("inv", [False, True])
def test_mixed_list_matches_per_image_calls(Cc, inv):
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(Cc * 10 + inv)
    sizes = FUSED + UNFUSED
    order = rng.permutation(len(sizes))
    sizes = [sizes[i] for i in order]
    tok = _tok(len(sizes), Cc + 100 * inv)
    imgs = [_image(s[0], s[1], Cc, rng) for s in sizes]
    _check_list(ops, tok, imgs, sizes, inv)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_random_mixed_sizes(seed):
    """Seeded lists of sizes 48..2048 per axis, outputs of other sizes, and one small image."""
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(1000 + seed)
    sizes = []
    for _ in range(10):
        H, W = (int(v) for v in rng.integers(48, 2049, 2))
        Ho, Wo = (int(v) for v in rng.integers(16, 1200, 2))
        sizes.append((H, W, Ho, Wo))
    sizes += [(int(rng.integers(2, 24)), int(rng.integers(2, 60)), 33, 21)]
    tok = _tok(len(sizes), seed)
    imgs = [_image(s[0], s[1], 3, rng) for s in sizes]
    _check_list(ops, tok, imgs, sizes, bool(seed & 1))


@pytest.mark.gpu
def test_position_and_neighbours_do_not_matter():
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(7)
    sizes = FUSED + UNFUSED
    tok = _tok(len(sizes), 7)
    imgs = [_image(s[0], s[1], 3, rng) for s in sizes]
    outs, mxs, mys = ops.warp_ragged_from_mota_tokens(tok, imgs, [(s[2], s[3]) for s in sizes], return_maps=True)
    perm = rng.permutation(len(sizes))
    sub = perm[: len(sizes) // 2]                 # a permuted half: other positions and other neighbours
    for idx in (perm, sub):
        o2, x2, y2 = ops.warp_ragged_from_mota_tokens(tok[torch.from_numpy(idx).cuda()], [imgs[i] for i in idx],
                                                      [(sizes[i][2], sizes[i][3]) for i in idx], return_maps=True)
        for j, i in enumerate(idx):
            assert torch.equal(o2[j], outs[i]) and torch.equal(x2[j], mxs[i]) and torch.equal(y2[j], mys[i]), (i, j)


@pytest.mark.gpu
@pytest.mark.parametrize("s", [FUSED[0], FUSED[2], UNFUSED[0], UNFUSED[3]])
def test_list_of_one(s):
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(s[0])
    _check_list(ops, _tok(1, s[1]), [_image(s[0], s[1], 3, rng)], [s], False)


@pytest.mark.gpu
@pytest.mark.parametrize("hw", [(336, 336), (500, 375)])
def test_same_size_list_equals_uniform_batch(hw):
    """Every image of one size: the maps of the uniform batch call (at these sizes its tiles are those of a single
    image) and its remap, bit for bit."""
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(hw[1])
    n, out_hw = 6, (400, 300)
    tok = _tok(n, hw[0])
    imgs = [_image(hw[0], hw[1], 3, rng) for _ in range(n)]
    outs, mxs, mys = ops.warp_ragged_from_mota_tokens(tok, imgs, [out_hw] * n, return_maps=True)
    ux, uy = ops.maps_from_mota_tokens(tok, hw, out_hw)
    ref = ops.remap_bilinear(torch.stack(imgs), ux, uy)
    for k in range(n):
        assert torch.equal(mxs[k], ux[k]) and torch.equal(mys[k], uy[k]) and torch.equal(outs[k], ref[k]), k


@pytest.mark.gpu
def test_list_without_shared_sizes_against_the_oracle():
    """Pillow's LANCZOS and warp_image_by_attention restated on the host, for a list whose images share no size."""
    _need_gpu()
    from attwarp_b200 import ops
    rng = np.random.default_rng(11)
    sizes = [(336, 336, 336, 336), (401, 97, 300, 120), (130, 517, 130, 517), (20, 16, 20, 16), (30, 40, 32, 41),
             (613, 255, 500, 500)]
    tok = _tok(len(sizes), 11)
    imgs = [_image(s[0], s[1], 3, rng) for s in sizes]
    for inv in (False, True):
        outs, mxs, mys = ops.warp_ragged_from_mota_tokens(tok, imgs, [(s[2], s[3]) for s in sizes], apply_inverse=inv,
                                                          return_maps=True)
        for k, s in enumerate(sizes):
            m = OM.mota_mask(tok[k].cpu().numpy(), (s[0], s[1]))
            ox, oy, _, _ = ON.inverse_maps(m, s[3], s[2], "identity", apply_inverse=inv)
            gx, gy = mxs[k].cpu().numpy(), mys[k].cpu().numpy()
            assert np.abs(gx - ox).max() <= 1e-3 and np.abs(gy - oy).max() <= 1e-3, (k, s, inv)
            want = ON.remap(imgs[k].cpu().numpy(), gx, gy)
            assert np.array_equal(outs[k].cpu().numpy(), want), (k, s, inv)


@pytest.mark.gpu
def test_launches_do_not_grow_with_the_list():
    _need_gpu()
    from attwarp_b200 import _lib, ops
    rng = np.random.default_rng(5)
    counts = []
    for n in (4, 64):
        sizes = [(int(h), int(w)) for h, w in rng.integers(100, 700, (n, 2))]
        ops.warp_ragged_from_mota_tokens(_tok(n, n), [_image(h, w, 3, rng) for h, w in sizes])
        counts.append(int(_lib.load().attwarp_ragged_last_launches()))
    assert counts[1] <= 2 + 28 and counts[1] - counts[0] <= 28, counts     # fused + finish + stage-5 classes


@pytest.mark.gpu
def test_warp_files_mota_matches_save_warped_image(tmp_path):
    """warp_files(mask="mota") against the reference flow per image: blend_mask (GPU, Pillow-exact mask) then
    save_warped_image(..., "identity") -- the warped files decode to the same pixels and the overlay files are the
    ones save_warped_image writes."""
    _need_gpu()
    import cv2
    from PIL import Image

    from attwarp_b200 import attention_extraction as AE
    from attwarp_b200 import image_io, new_method
    rng = np.random.default_rng(3)
    sizes = [(300, 200), (97, 413), (520, 333), (20, 30), (64, 64)]
    out_sizes = [(500, 500), (97, 413), (300, 301), (20, 30), (80, 50)]
    paths = []
    for k, (h, w) in enumerate(sizes):
        p = str(tmp_path / f"in{k}.png")        # PNG: decoded exactly on the host by both sides
        cv2.imwrite(p, rng.integers(0, 256, (h, w, 3), dtype=np.uint8))
        paths.append(p)
    tok = _tok(len(sizes), 3)
    outs = [str(tmp_path / f"warp{k}.png") for k in range(len(sizes))]
    ovls = [str(tmp_path / f"ovl{k}.png") for k in range(len(sizes))]
    ok = image_io.warp_files(paths, tok, outs, out_sizes, overlay_paths=ovls, mask="mota")
    assert all(ok)
    for k, (p, (ho, wo)) in enumerate(zip(paths, out_sizes)):
        pil = Image.open(p).convert("RGB")
        _, mask_img = AE.blend_mask(pil, tok[k], 10, 3, Image.LANCZOS, 0.5)
        ref_w, ref_o = str(tmp_path / f"ref_warp{k}.png"), str(tmp_path / f"ref_ovl{k}.png")
        assert new_method.save_warped_image(pil, mask_img, None, ref_o, ref_w, width=wo, height=ho,
                                            transform="identity")
        for got, want in ((outs[k], ref_w), (ovls[k], ref_o)):
            a, b = cv2.imread(got, cv2.IMREAD_UNCHANGED), cv2.imread(want, cv2.IMREAD_UNCHANGED)
            assert a.shape == b.shape and np.array_equal(a, b), (k, got)


def test_warp_files_mask_switch_is_checked():
    from attwarp_b200 import image_io
    with pytest.raises(ValueError, match="mask"):
        image_io.warp_files(["x.png"], torch.zeros(1, 2, 2), ["y.png"], mask="lanczos")
    with pytest.raises(ValueError, match="identity"):
        image_io.warp_files(["x.png"], torch.zeros(1, 2, 2), ["y.png"], transform="sqrt", mask="mota")
    with pytest.raises(ValueError, match="token maps"):
        image_io.warp_files(["x.png"], None, ["y.png"], att=[np.zeros((2, 2), np.uint8)], mask="mota")


# ---- the C ABI's argument checks: no device needed (nothing is enqueued before they pass) ----------------------------
_TABLE = np.dtype([("src", np.uint64), ("dst", np.uint64), ("H", np.int32), ("W", np.int32), ("Ho", np.int32),
                   ("Wo", np.int32)])


def _abi():
    from attwarp_b200 import _lib
    if not os.path.isfile(_lib.lib_path()):
        pytest.skip("library not built")
    return _lib, _lib.load()


def _table(sizes):
    t = np.zeros(len(sizes), dtype=_TABLE)
    t["src"] = [0x10000 + 0x1000 * k for k in range(len(sizes))]      # never dereferenced: the checks fail first
    t["dst"] = [0x90000 + 0x1000 * k for k in range(len(sizes))]
    for k, s in enumerate(sizes):
        t["H"][k], t["W"][k], t["Ho"][k], t["Wo"][k] = s
    return t


@pytest.mark.parametrize("case,status,msg", [
    ("square", "ERR_UNSUPPORTED", "identity transform only"),
    ("log_inverse", "ERR_UNSUPPORTED", "identity transform only"),
    ("bad_transform", "ERR_INVALID_ARG", "unknown transform"),
    ("small_ws", "ERR_WORKSPACE", "workspace too small"),
    ("small_ws_inverse", "ERR_WORKSPACE", "workspace too small"),
    ("empty_H", "ERR_INVALID_ARG", "sizes must be positive"),
    ("empty_W", "ERR_INVALID_ARG", "sizes must be positive"),
    ("empty_out", "ERR_INVALID_ARG", "sizes must be positive"),
    ("huge", "ERR_INVALID_ARG", "below 65536"),
    ("C2", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("C0", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("C5", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("null_mask", "ERR_INVALID_ARG", "NULL pointer"),
    ("null_ws", "ERR_INVALID_ARG", "NULL pointer"),
    ("n0", "ERR_INVALID_ARG", "must be positive"),
    ("same_src_dst", "ERR_INVALID_ARG", "bad pointers"),
])
def test_abi_rejects_without_a_device(case, status, msg):
    _lib, lib = _abi()
    sizes = [(336, 336, 336, 336), (20, 16, 20, 16)]
    if case == "empty_H":
        sizes[1] = (0, 16, 20, 16)
    elif case == "empty_W":
        sizes[0] = (336, 0, 336, 336)
    elif case == "empty_out":
        sizes[1] = (20, 16, 20, 0)
    elif case == "huge":
        sizes[1] = (70000, 16, 20, 16)
    t = _table(sizes)
    if case == "same_src_dst":
        t["dst"][1] = t["src"][1]
    tp = {"square": _lib.make_transform("square"), "log_inverse": _lib.make_transform("log", apply_inverse=True),
          "small_ws_inverse": _lib.make_transform("identity", apply_inverse=True)}.get(case, _lib.make_transform())
    if case == "bad_transform":
        tp.transform = 9
    n = 0 if case == "n0" else len(sizes)
    Cc = {"C2": 2, "C0": 0, "C5": 5}.get(case, 3)
    tp_ = C.byref(tp)
    need = lib.attwarp_ragged_mask_workspace_bytes(t.ctypes.data_as(C.c_void_p), 2, GH, GW)
    ws_bytes = need - 1 if case.startswith("small_ws") else need
    rc = lib.attwarp_warp_ragged_from_mask(t.ctypes.data_as(C.c_void_p), None if case == "null_mask" else C.c_void_p(0x5000),
                                           n, GH, GW, Cc, tp_, None if case == "null_ws" else C.c_void_p(0x7000000),
                                           ws_bytes, None, None, None)
    assert rc == getattr(_lib, status), (rc, lib.attwarp_last_error())
    assert msg in lib.attwarp_last_error().decode()


def test_abi_workspace_bytes_without_a_device():
    _, lib = _abi()
    ok = _table([(336, 336, 336, 336), (20, 16, 20, 16), (2048, 224, 1000, 300)])
    p = ok.ctypes.data_as(C.c_void_p)
    assert lib.attwarp_ragged_mask_workspace_bytes(p, 3, GH, GW) > 0
    assert lib.attwarp_ragged_mask_workspace_bytes(p, 0, GH, GW) == 0
    assert lib.attwarp_ragged_mask_workspace_bytes(p, 3, 0, GW) == 0
    assert lib.attwarp_ragged_mask_workspace_bytes(None, 3, GH, GW) == 0
    bad = _table([(336, 336, 336, 336), (20, 0, 20, 16)])
    assert lib.attwarp_ragged_mask_workspace_bytes(bad.ctypes.data_as(C.c_void_p), 2, GH, GW) == 0
