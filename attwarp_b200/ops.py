"""Device-resident batched operators over the C ABI (torch tensors in, torch tensors out).

These are the siblings SURVEY.md section 8(b) asks for next to the NumPy-signature drop-ins:
inputs stay in HBM, outputs are allocated with torch's caching allocator, all work is enqueued
on the current CUDA stream, nothing synchronises.  torch is plumbing only (memory + streams);
every arithmetic step runs in libattwarp_sm100.so.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import (LAYOUT_CHW, LAYOUT_HWC, TORCH_DTYPE_IDS, check, current_stream, load,
                   make_transform, ptr, require_cuda)

_ws_cache = {}

# attwarp_ragged_image (include/attwarp.h)
_RAGGED_DTYPE = np.dtype([("src", np.uint64), ("dst", np.uint64), ("H", np.int32), ("W", np.int32),
                          ("Ho", np.int32), ("Wo", np.int32)])


_ws_scope = None     # a dict while a GraphedCall warms up / captures: that graph's private scratch


def _workspace(nbytes: int, device) -> torch.Tensor:
    """A reusable uint8 scratch tensor of at least ``nbytes`` on ``device`` (stream-ordered
    reuse is safe because all kernels of this package run on the caller's current stream).
    A captured graph keeps scratch of its own (it lives and dies with the GraphedCall object): graphs may
    be replayed concurrently on different streams, whatever stream they were captured on."""
    if _ws_scope is not None:
        cache, key = _ws_scope, torch.device(device).index
    else:
        cache, key = _ws_cache, (torch.device(device).index, torch.cuda.current_stream(device).cuda_stream)
    buf = cache.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        cache[key] = buf
    return buf


def _check_out(name, t, shape, dtype, device):
    """Caller-provided output / scratch tensors are written through raw pointers: anything but the exact
    dense tensor would corrupt memory silently."""
    if (tuple(t.shape) != tuple(shape) or t.dtype != dtype or t.device != device or not t.is_contiguous()):
        raise ValueError(f"{name}: expected a contiguous {dtype} tensor of shape {tuple(shape)} on {device}, got "
                         f"{t.dtype} {tuple(t.shape)} on {t.device} (contiguous={t.is_contiguous()})")


def _tp(transform, exp_scale, exp_divisor, apply_inverse):
    if isinstance(transform, _lib.TransformParams):
        return transform
    return make_transform(transform, exp_scale, exp_divisor, apply_inverse)


class GraphedCall:
    """Capture ``fn()`` -- a callable that only enqueues work of this package on the current
    stream, on pre-allocated tensors -- into a CUDA graph; ``replay()`` launches the whole
    sequence with one driver call (the per-kernel launch gaps of a 150 us step disappear)."""

    def __init__(self, fn, warmup: int = 2, device=None):
        global _ws_scope
        dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self._scratch = {}                   # device index -> this graph's scratch tensor
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        prev, _ws_scope = _ws_scope, self._scratch
        try:
            with torch.cuda.stream(side):
                for _ in range(warmup):          # kernel attribute opt-ins, this graph's scratch
                    fn()
            torch.cuda.current_stream(dev).wait_stream(side)
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph):
                fn()
        finally:
            _ws_scope = prev

    def replay(self):
        self.graph.replay()


# --------------------------------------------------------------------------------------------
# stage 1
# --------------------------------------------------------------------------------------------
def _token_window(name, tok_start, B, K, T, device):
    """Check that every image's token window [start, start + T) lies inside its row of K tokens and return
    ``tok_start`` as a contiguous int32 tensor on ``device`` (None stays None).  The kernels read the window
    through raw pointers, so a window past the row reads another row, another image or past the tensor.
    A CUDA ``tok_start`` is not copied back to be checked: only its length is, its values are the caller's."""
    if T < 1:
        raise ValueError(f"{name}: the token window must hold at least one token, got T={T}")
    if tok_start is None:
        if T > K:
            raise ValueError(f"{name}: T={T} tokens requested from rows of K={K} (pass tok_start for a window)")
        return None
    starts = torch.as_tensor(tok_start)        # list / CPU tensor / CUDA tensor of per-sample offsets
    if starts.numel() != B:
        raise ValueError(f"{name}: tok_start holds {starts.numel()} values for a batch of {B}")
    if not starts.is_cuda and B > 0:
        lo, hi = int(starts.min()), int(starts.max())
        if lo < 0 or hi > K - T:
            raise ValueError(f"{name}: tok_start values in [{lo}, {hi}] put a window of T={T} tokens outside rows "
                             f"of K={K} (each start must lie in [0, {K - T}])")
    return starts.to(device=device, dtype=torch.int32).contiguous()


def aggregate_attention(attn: torch.Tensor, tok_start: torch.Tensor | None = None,
                        num_tokens: int | None = None, out: torch.Tensor | None = None,
                        accumulate: bool = False, out_scale: float = 1.0,
                        eps: float = 1e-12) -> torch.Tensor:
    """attn [B, L, Hh, K] (bf16/fp16/fp32, last dim contiguous, other dims arbitrarily strided)
    -> float32 [B, T]:  mean over L and Hh of  a[..., st:st+T] / (sum + eps).
    Reference: llava.py:94-132, 385-411 (L = hooked steps).

    T is ``num_tokens`` (default K).  ``tok_start`` (B offsets) selects the window [st, st + T) of image b's
    rows; without it T must not exceed K.  A list or CPU tensor of offsets is checked against [0, K - T]
    (ValueError); a CUDA tensor is used as it is, and keeping its values in that range is the caller's
    responsibility."""
    lib = load()
    require_cuda(attn, out)
    assert attn.dim() == 4, "attn must be [B, L, Hh, K]"
    if attn.stride(3) != 1:
        raise ValueError("attention rows must be contiguous along the token axis")
    B, L, Hh, K = attn.shape
    T = K if num_tokens is None else int(num_tokens)
    tok_start = _token_window("aggregate_attention", tok_start, B, K, T, attn.device)
    if out is None:
        out = torch.empty(B, T, dtype=torch.float32, device=attn.device)
        accumulate = False
    else:
        _check_out("aggregate_attention: out", out, (B, T), torch.float32, attn.device)
    wsb = lib.attwarp_aggregate_workspace_bytes(B, L, Hh, T)
    ws = _workspace(wsb, attn.device)
    with torch.cuda.device(attn.device):
        check(lib.attwarp_aggregate_attention(
            ptr(attn), TORCH_DTYPE_IDS[attn.dtype], B, L, Hh, T, attn.stride(0), attn.stride(1),
            attn.stride(2), ptr(tok_start), eps, ptr(ws), ws.numel(), ptr(out),
            1 if accumulate else 0, float(out_scale), current_stream(attn.device)))
    return out


# --------------------------------------------------------------------------------------------
# mask post-processing of the driver flow (between stage 1 and stage 2b)
# --------------------------------------------------------------------------------------------
def revise_mask(tok: torch.Tensor, kernel_size: int = 3, enhance_coe: float = 10.0, return_u8: bool = False):
    """tok [B,gh,gw] float32 -> revise_mask(tok) [B,gh,gw] float32 (llava.py:207-238); with
    ``return_u8`` also the uint8 image ToPILImage makes of it (truncation of v * 255)."""
    lib = load()
    require_cuda(tok)
    tok = tok.contiguous().float()
    B, gh, gw = tok.shape
    rev = torch.empty_like(tok)
    u8 = torch.empty(B, gh, gw, dtype=torch.uint8, device=tok.device) if return_u8 else None
    with torch.cuda.device(tok.device):
        check(lib.attwarp_revise_mask(ptr(tok), B, gh, gw, int(kernel_size), float(enhance_coe), ptr(rev),
                                      ptr(u8), current_stream(tok.device)))
    return (rev, u8) if return_u8 else rev


def resize_lanczos_u8(img: torch.Tensor, out_hw) -> torch.Tensor:
    """img [B,h,w] uint8 -> [B,Ho,Wo], bit-identical to PIL.Image.resize((Wo,Ho), LANCZOS) in mode 'L'."""
    lib = load()
    require_cuda(img)
    assert img.dtype == torch.uint8 and img.dim() == 3
    img = img.contiguous()
    B, h, w = img.shape
    Ho, Wo = int(out_hw[0]), int(out_hw[1])
    out = torch.empty(B, Ho, Wo, dtype=torch.uint8, device=img.device)
    with torch.cuda.device(img.device):
        check(lib.attwarp_resize_lanczos_u8(ptr(img), B, h, w, Ho, Wo, ptr(out), current_stream(img.device)))
    return out


def mota_mask(tok: torch.Tensor, image_hw, kernel_size: int = 3, enhance_coe: float = 10.0) -> torch.Tensor:
    """tok [B,gh,gw] -> the uint8 [B,H,W] mask blend_mask returns at image size (llava.py:240-256):
    revise_mask -> ToPILImage -> resize(LANCZOS) -> 'L'.  It is the att_map the drivers pass to
    save_warped_image (main.py:361, 520): feed it to ``maps_from_attention``."""
    _, u8 = revise_mask(tok, kernel_size, enhance_coe, return_u8=True)
    return resize_lanczos_u8(u8, image_hw)


def maps_from_mota_tokens(tok: torch.Tensor, image_hw, out_size=None, kernel_size: int = 3, enhance_coe: float = 10.0,
                          apply_inverse: bool = False, fused: bool = True):
    """tok [B,gh,gw] -> (map_x, map_y) of the driver flow ``blend_mask`` -> ``save_warped_image(..., "identity")``
    (llava.py:240-256 then new_method.py:207-261) for callers that only warp.  ``fused=True``: the image-size uint8
    mask is never written, its marginals are summed where the LANCZOS resize computes it, on the tensor cores (saves the
    B x H x W buffer and time: 37 us vs 43 us for the two steps at 256 x 336^2, 73 us vs 93 us at 64 x 1344^2).
    Same maps as ``maps_from_attention(mota_mask(tok, image_hw), out_size)``, which ``fused=False`` runs."""
    lib = load()
    _, u8 = revise_mask(tok, kernel_size, enhance_coe, return_u8=True)
    B, gh, gw = u8.shape
    H, W = int(image_hw[0]), int(image_hw[1])
    Ho, Wo = (H, W) if out_size is None else (int(out_size[0]), int(out_size[1]))
    wsb = lib.attwarp_maps_from_mask_workspace_bytes(B, gh, gw, H, W) if fused else 0
    if wsb == 0:        # not fused, or not an up-scaling the fused kernel takes: the two device steps
        return maps_from_attention(resize_lanczos_u8(u8, (H, W)), (Ho, Wo), apply_inverse=apply_inverse)
    tp = _tp("identity", 1.0, 1.0, apply_inverse)
    map_x = torch.empty(B, Wo, dtype=torch.float32, device=tok.device)
    map_y = torch.empty(B, Ho, dtype=torch.float32, device=tok.device)
    ws = _workspace(wsb, tok.device)
    with torch.cuda.device(tok.device):
        check(lib.attwarp_maps_from_mask(ptr(u8), B, gh, gw, H, W, Wo, Ho, C.byref(tp), ptr(ws), ws.numel(),
                                         ptr(map_x), ptr(map_y), current_stream(tok.device)))
    return map_x, map_y


# --------------------------------------------------------------------------------------------
# stages 2b-4
# --------------------------------------------------------------------------------------------
def maps_from_attention(att: torch.Tensor, out_size, transform="identity", exp_scale=1.0,
                        exp_divisor=1.0, apply_inverse=False):
    """att [B,H,W] (uint8/float32/float64) -> (map_x [B,Wo], map_y [B,Ho]) float32.
    Reference: new_method.py:207-261."""
    lib = load()
    require_cuda(att)
    att = att.contiguous()
    B, H, W = att.shape
    Ho, Wo = out_size
    tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
    map_x = torch.empty(B, Wo, dtype=torch.float32, device=att.device)
    map_y = torch.empty(B, Ho, dtype=torch.float32, device=att.device)
    wsb = lib.attwarp_maps_workspace_bytes(B, H, W)
    ws = _workspace(wsb, att.device)
    with torch.cuda.device(att.device):
        check(lib.attwarp_maps_from_attention(ptr(att), TORCH_DTYPE_IDS[att.dtype], B, H, W, Wo, Ho,
                                              C.byref(tp), ptr(ws), ws.numel(), ptr(map_x),
                                              ptr(map_y), current_stream(att.device)))
    return map_x, map_y


def maps_from_tokens(tok: torch.Tensor, image_size, out_size=None, transform="identity",
                     exp_scale=1.0, exp_divisor=1.0, apply_inverse=False, out=None):
    """tok [B,gh,gw] float32, index-upsampled on the fly to image_size=(H,W)."""
    lib = load()
    require_cuda(tok)
    tok = tok.contiguous().float()
    B, gh, gw = tok.shape
    H, W = image_size
    Ho, Wo = (H, W) if out_size is None else out_size
    tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
    if out is not None:
        map_x, map_y = out
        _check_out("maps_from_tokens: out[0] (map_x)", map_x, (B, Wo), torch.float32, tok.device)
        _check_out("maps_from_tokens: out[1] (map_y)", map_y, (B, Ho), torch.float32, tok.device)
    else:
        map_x = torch.empty(B, Wo, dtype=torch.float32, device=tok.device)
        map_y = torch.empty(B, Ho, dtype=torch.float32, device=tok.device)
    with torch.cuda.device(tok.device):
        check(lib.attwarp_maps_from_tokens(ptr(tok), B, gh, gw, H, W, Wo, Ho, C.byref(tp),
                                           ptr(map_x), ptr(map_y), current_stream(tok.device)))
    return map_x, map_y


def maps_from_cdf(Fx: torch.Tensor, Fy: torch.Tensor, out_size=None):
    """Fx [B,W], Fy [B,H] float32 CDFs -> (map_x [B,Wo], map_y [B,Ho]).
    Reference: checkpoint_utils.py:157-189."""
    lib = load()
    require_cuda(Fx, Fy)
    Fx = Fx.contiguous().float()
    Fy = Fy.contiguous().float()
    B, W = Fx.shape
    H = Fy.shape[1]
    Ho, Wo = (H, W) if out_size is None else out_size
    map_x = torch.empty(B, Wo, dtype=torch.float32, device=Fx.device)
    map_y = torch.empty(B, Ho, dtype=torch.float32, device=Fx.device)
    with torch.cuda.device(Fx.device):
        check(lib.attwarp_maps_from_cdf(ptr(Fx), ptr(Fy), B, H, W, Wo, Ho, ptr(map_x), ptr(map_y),
                                        current_stream(Fx.device)))
    return map_x, map_y


# --------------------------------------------------------------------------------------------
# stage 5
# --------------------------------------------------------------------------------------------
def remap_bilinear(img: torch.Tensor, map_x: torch.Tensor, map_y: torch.Tensor,
                   layout: str = "hwc", out: torch.Tensor | None = None) -> torch.Tensor:
    """img [B,H,W,C] (layout 'hwc') or [B,C,H,W] ('chw'), uint8/float32; maps [B,Wo], [B,Ho].
    cv2.remap(INTER_LINEAR, BORDER_REPLICATE) semantics (new_method.py:268-271)."""
    lib = load()
    require_cuda(img, map_x, map_y, out)
    img = img.contiguous()
    map_x = map_x.contiguous().float()
    map_y = map_y.contiguous().float()
    if layout == "hwc":
        B, H, W, Cc = img.shape
        lay = LAYOUT_HWC
    elif layout == "chw":
        B, Cc, H, W = img.shape
        lay = LAYOUT_CHW
    else:
        raise ValueError(f"layout must be 'hwc' or 'chw', got {layout!r}")
    Wo, Ho = map_x.shape[1], map_y.shape[1]
    assert map_x.shape[0] == B and map_y.shape[0] == B
    shape = (B, Ho, Wo, Cc) if layout == "hwc" else (B, Cc, Ho, Wo)
    if out is None:
        out = torch.empty(shape, dtype=img.dtype, device=img.device)
    else:
        _check_out("remap_bilinear: out", out, shape, img.dtype, img.device)
    with torch.cuda.device(img.device):
        check(lib.attwarp_remap_bilinear(ptr(img), ptr(out), TORCH_DTYPE_IDS[img.dtype], lay, B, Cc,
                                         H, W, Ho, Wo, ptr(map_x), ptr(map_y),
                                         current_stream(img.device)))
    return out


# --------------------------------------------------------------------------------------------
# fused batch driver (BASELINE configs[1]/[2])
# --------------------------------------------------------------------------------------------
def warp_from_attention_tokens(attn: torch.Tensor, images: torch.Tensor, grid_hw, out_size=None,
                               layout: str = "hwc", tok_start: torch.Tensor | None = None,
                               transform="identity", exp_scale=1.0, exp_divisor=1.0,
                               apply_inverse=False, out: torch.Tensor | None = None,
                               return_aux: bool = False, aux: tuple | None = None,
                               stage_events=None):
    """Stages 1-5 for a uniform batch in one host call:
    attn [B,L,Hh,K] -> token map [B,gh*gw] -> separable maps -> warped images.

    Without ``tok_start`` K must equal gh*gw; with it, image b's tokens are [st_b, st_b + gh*gw) of its rows,
    checked as in ``aggregate_attention`` (a CUDA ``tok_start`` is the caller's responsibility)."""
    lib = load()
    require_cuda(attn, images, out)
    assert attn.dim() == 4 and attn.stride(3) == 1
    images = images.contiguous()
    B, L, Hh, K = attn.shape
    gh, gw = grid_hw
    if tok_start is None and K != gh * gw:
        raise ValueError(f"warp_from_attention_tokens: attention row length K={K} must equal gh*gw={gh * gw} "
                         "unless tok_start is given")
    tok_start = _token_window("warp_from_attention_tokens", tok_start, B, K, gh * gw, attn.device)
    if layout == "hwc":
        Bi, H, W, Cc = images.shape
        lay = LAYOUT_HWC
    else:
        Bi, Cc, H, W = images.shape
        lay = LAYOUT_CHW
    assert Bi == B
    Ho, Wo = (H, W) if out_size is None else out_size
    shape = (B, Ho, Wo, Cc) if layout == "hwc" else (B, Cc, Ho, Wo)
    dev = images.device
    if out is None:
        out = torch.empty(shape, dtype=images.dtype, device=dev)
    else:
        _check_out("warp_from_attention_tokens: out", out, shape, images.dtype, dev)
    if aux is not None:                      # caller-provided (tok, map_x, map_y) buffers
        tok, map_x, map_y = aux
        _check_out("warp_from_attention_tokens: aux[0] (token map)", tok.view(B, -1) if tok.is_contiguous() else tok,
                   (B, gh * gw), torch.float32, dev)
        _check_out("warp_from_attention_tokens: aux[1] (map_x)", map_x, (B, Wo), torch.float32, dev)
        _check_out("warp_from_attention_tokens: aux[2] (map_y)", map_y, (B, Ho), torch.float32, dev)
    else:
        tok = torch.empty(B, gh * gw, dtype=torch.float32, device=dev)
        map_x = torch.empty(B, Wo, dtype=torch.float32, device=dev)
        map_y = torch.empty(B, Ho, dtype=torch.float32, device=dev)
    ev = None
    if stage_events is not None:             # 4 recorded torch.cuda.Event(enable_timing=True)
        ev = (C.c_void_p * 4)(*[e.cuda_event for e in stage_events])
    tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
    wsb = lib.attwarp_aggregate_workspace_bytes(B, L, Hh, gh * gw)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_warp_from_attention_tokens(
            ptr(attn), TORCH_DTYPE_IDS[attn.dtype], B, L, Hh, attn.stride(0), attn.stride(1),
            attn.stride(2), ptr(tok_start), gh, gw, ptr(images), ptr(out),
            TORCH_DTYPE_IDS[images.dtype], lay, Cc, H, W, Ho, Wo, C.byref(tp), ptr(ws), ws.numel(),
            ptr(tok), ptr(map_x), ptr(map_y), ev, current_stream(dev)))
    if return_aux:
        return out, tok.view(B, gh, gw), map_x, map_y
    return out


# --------------------------------------------------------------------------------------------
# predicted PDFs -> warped images (BASELINE configs[4])
# --------------------------------------------------------------------------------------------
def warp_from_pdfs(img: torch.Tensor, px: torch.Tensor, py: torch.Tensor, alpha: float = 0.0,
                   out_size=None, layout: str = "chw", eps: float = 1e-8, out: torch.Tensor | None = None,
                   return_aux: bool = False):
    """MarginalNet PDFs px [B,Nx], py [B,Ny] + images -> warped images, three launches:
    (mix_with_uniform + upsample_pdf_right_inverse + clamp_min(0) + cdf_from_density) for both axes,
    inverse-CDF maps, resample.  Same arithmetic as calling the mirrors in checkpoint_utils / model one
    after the other (trainer.py:212-218, 285-289)."""
    from .checkpoint_utils import right_inverse_matrix
    lib = load()
    require_cuda(img, px, py, out)
    img = img.contiguous()
    if layout == "chw":
        B, Cc, H, W = img.shape
        lay = LAYOUT_CHW
    else:
        B, H, W, Cc = img.shape
        lay = LAYOUT_HWC
    Ho, Wo = (H, W) if out_size is None else (int(out_size[0]), int(out_size[1]))
    dev = img.device
    px = px.detach().to(device=dev, dtype=torch.float32).contiguous()
    py = py.detach().to(device=dev, dtype=torch.float32).contiguous()
    assert px.shape[0] == B and py.shape[0] == B and px.dim() == 2 and py.dim() == 2
    Mx = right_inverse_matrix(W, px.shape[1], eps, dev)
    My = right_inverse_matrix(H, py.shape[1], eps, dev)
    shape = (B, Cc, Ho, Wo) if layout == "chw" else (B, Ho, Wo, Cc)
    if out is None:
        out = torch.empty(shape, dtype=img.dtype, device=dev)
    else:
        _check_out("warp_from_pdfs: out", out, shape, img.dtype, dev)
    Fx = torch.empty(B, W, dtype=torch.float32, device=dev)
    Fy = torch.empty(B, H, dtype=torch.float32, device=dev)
    map_x = torch.empty(B, Wo, dtype=torch.float32, device=dev)
    map_y = torch.empty(B, Ho, dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_warp_from_pdfs(ptr(px), ptr(py), B, px.shape[1], py.shape[1], float(alpha),
                                         ptr(Mx), ptr(My), ptr(img), ptr(out), TORCH_DTYPE_IDS[img.dtype],
                                         lay, Cc, H, W, Ho, Wo, ptr(Fx), ptr(Fy), ptr(map_x), ptr(map_y),
                                         current_stream(dev)))
    if return_aux:
        return out, Fx, Fy, map_x, map_y
    return out


# --------------------------------------------------------------------------------------------
# ragged batches (mixed resolutions, BASELINE configs[3])
# --------------------------------------------------------------------------------------------
def _ragged_list(name, images, out_sizes, outs, anchor):
    """The list of a ragged call: the images made contiguous, the outputs (allocated when ``outs`` is None), the output
    sizes as ints -- default the input sizes -- and the descriptor table (attwarp_ragged_image [n]) of them all.  Every
    image must be a uint8 [H, W, C] tensor with one C on ``anchor``'s device, every output a contiguous uint8
    [Ho, Wo, C] tensor there.  The library writes each image through its table row at that row's size, and NumPy
    broadcasts a one-element list into every row, so lists of the wrong length are refused before anything else."""
    n = len(images)
    if out_sizes is not None and len(out_sizes) != n:
        raise ValueError(f"{name}: {len(out_sizes)} output sizes for {n} images")
    if outs is not None and len(outs) != n:
        raise ValueError(f"{name}: {len(outs)} outputs for {n} images")
    require_cuda(anchor, *images)
    dev, index = anchor.device, anchor.get_device()      # get_device(): no torch.device built per tensor
    imgs = [im.contiguous() for im in images]
    Cc = imgs[0].shape[2] if imgs[0].dim() == 3 else 0
    for im in imgs:
        if im.dtype != torch.uint8 or im.dim() != 3 or im.shape[2] != Cc or im.get_device() != index:
            raise ValueError(f"{name}: images must be uint8 HWC tensors with the same channel count on one device, got "
                             f"{im.dtype} {tuple(im.shape)} on {im.device} (expected C={Cc} on {dev})")
    if out_sizes is None:
        out_sizes = [(im.shape[0], im.shape[1]) for im in imgs]
    else:
        out_sizes = [(int(ho), int(wo)) for ho, wo in out_sizes]
    if outs is None:
        outs = [torch.empty(ho, wo, Cc, dtype=torch.uint8, device=dev) for ho, wo in out_sizes]
    else:
        outs = list(outs)
        for k, (o, (ho, wo)) in enumerate(zip(outs, out_sizes)):
            if o.dtype != torch.uint8 or o.shape != (ho, wo, Cc) or not o.is_contiguous() or o.get_device() != index:
                raise ValueError(f"{name}: outputs must be contiguous [Ho, Wo, C] uint8 tensors on {dev}: output {k} "
                                 f"is {o.dtype} {tuple(o.shape)} on {o.device}, expected {(ho, wo, Cc)}")
    # one structured array (a ctypes struct per image costs ~3 us each)
    table = np.empty(n, dtype=_RAGGED_DTYPE)
    table["src"] = [im.data_ptr() for im in imgs]
    table["dst"] = [o.data_ptr() for o in outs]
    table["H"] = [im.shape[0] for im in imgs]
    table["W"] = [im.shape[1] for im in imgs]
    table["Ho"] = [hw[0] for hw in out_sizes]
    table["Wo"] = [hw[1] for hw in out_sizes]
    return imgs, outs, out_sizes, table


def warp_ragged_from_tokens(tok: torch.Tensor, images, out_sizes=None, grid_hw=None,
                            transform="identity", exp_scale=1.0, exp_divisor=1.0,
                            apply_inverse=False, outs=None):
    """Stages 2-5 for n images of different shapes with ONE launch per stage.

    tok     [n, gh, gw] (or [n, gh*gw] with ``grid_hw``) float32 token maps on the device
    images  sequence of n uint8 HWC tensors [H_i, W_i, C] on the same device
    out_sizes  sequence of (Ho_i, Wo_i), default = input sizes
    Returns the list of warped images.  Replaces the per-image loops of AGW/main.py:395-533 and
    AGW/main_batched.py:243-287 (one warp_image_by_attention call per image)."""
    lib = load()
    n = len(images)
    if tok.shape[0] != n:
        raise ValueError(f"warp_ragged_from_tokens: {tok.shape[0]} token maps for {n} images")
    if n == 0:                      # the reference's per-image loop over an empty list does nothing
        return []
    imgs, outs, _, table = _ragged_list("warp_ragged_from_tokens", images, out_sizes, outs, tok)
    dev = tok.device
    if tok.dim() == 3:
        gh, gw = tok.shape[1], tok.shape[2]
    else:
        gh, gw = grid_hw
    tok = tok.reshape(n, gh * gw).to(torch.float32).contiguous()
    table_p = table.ctypes.data_as(C.c_void_p)           # `table` stays alive until the call returns
    tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
    wsb = lib.attwarp_ragged_workspace_bytes(table_p, n)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_warp_ragged_from_tokens(ptr(tok), n, gh, gw, table_p, imgs[0].shape[2], C.byref(tp),
                                                  ptr(ws), ws.numel(), current_stream(dev)))
    return outs


# attwarp_ragged_attention (include/attwarp.h)
_RAGGED_ATT_DTYPE = np.dtype([("att", np.uint64), ("map_x", np.uint64), ("map_y", np.uint64)])
_RAGGED_MAP_DTYPES = (torch.uint8, torch.float32, torch.float64)


def warp_ragged_from_attention(att, images, out_sizes=None, transform="identity", exp_scale=1.0, exp_divisor=1.0,
                               apply_inverse=False, outs=None, return_maps=False):
    """Stages 2b-5 for n images of different shapes, each warped by its OWN attention map -- the reference's
    ``warp_image_by_attention(image, att_map, w, h)`` (new_method.py:198-283) per image -- in one marginals launch
    for all maps, one finish launch and the stage-5 launches of ``warp_ragged_from_tokens``.

    att     sequence of n CUDA tensors [H_i, W_i] of one dtype: uint8 (e.g. ``blend_mask`` / ``mota_mask``),
            float32 or float64.  Any strides of a 2-D view are taken (non-dense ones are copied first); rows may
            start at any byte offset.
    images  sequence of n uint8 HWC tensors [H_i, W_i, C], C in {1, 3, 4}, on the same device
    out_sizes  sequence of (Ho_i, Wo_i), default = input sizes
    Returns the list of warped images, and with ``return_maps`` also the lists of map_x [Wo_i] and map_y [Ho_i].
    An image's maps depend on its own map only: they are bit-identical to those of a call on that image alone."""
    lib = load()
    n = len(images)
    if not isinstance(att, (list, tuple)):
        raise ValueError(f"warp_ragged_from_attention: att must be a sequence of [H, W] tensors, got {type(att).__name__}")
    if len(att) != n:
        raise ValueError(f"warp_ragged_from_attention: {len(att)} attention maps for {n} images")
    if n == 0:
        return ([], [], []) if return_maps else []
    imgs, outs, out_sizes, table = _ragged_list("warp_ragged_from_attention", images, out_sizes, outs, images[0])
    dev = imgs[0].device
    Cc = imgs[0].shape[2]
    if Cc not in (1, 3, 4):
        raise ValueError(f"warp_ragged_from_attention: images must be uint8 [H, W, C] with C in (1, 3, 4), got "
                         f"{tuple(imgs[0].shape)}")
    maps = []
    for k, (a, im) in enumerate(zip(att, imgs)):
        if not isinstance(a, torch.Tensor):
            raise ValueError(f"warp_ragged_from_attention: attention map {k} is a {type(a).__name__}, not a tensor")
        if a.dim() != 2:
            raise ValueError(f"warp_ragged_from_attention: attention map {k} must be 2-D [H, W], got {tuple(a.shape)}")
        if a.dtype not in _RAGGED_MAP_DTYPES:
            raise ValueError(f"warp_ragged_from_attention: attention map {k} has dtype {a.dtype}; uint8, float32 and "
                             "float64 are supported")
        if a.device != dev:
            raise ValueError(f"warp_ragged_from_attention: attention map {k} is on {a.device}, image 0 on {dev}: all "
                             "tensors must be on one CUDA device")
        if tuple(a.shape) != tuple(im.shape[:2]):
            raise ValueError(f"warp_ragged_from_attention: attention map {k} is {tuple(a.shape)}, image {k} is "
                             f"{tuple(im.shape[:2])}: the map must have its image's size")
        maps.append(a if a.is_contiguous() else a.contiguous())
    if len({a.dtype for a in maps}) > 1:
        raise ValueError("warp_ragged_from_attention: all attention maps must have one dtype, got "
                         f"{sorted({str(a.dtype) for a in maps})}")
    atab = np.zeros(n, dtype=_RAGGED_ATT_DTYPE)
    atab["att"] = [a.data_ptr() for a in maps]
    map_xs = map_ys = None
    if return_maps:
        map_xs = [torch.empty(wo, dtype=torch.float32, device=dev) for _, wo in out_sizes]
        map_ys = [torch.empty(ho, dtype=torch.float32, device=dev) for ho, _ in out_sizes]
        atab["map_x"] = [m.data_ptr() for m in map_xs]
        atab["map_y"] = [m.data_ptr() for m in map_ys]
    table_p = table.ctypes.data_as(C.c_void_p)           # the tables stay alive until the call returns
    atab_p = atab.ctypes.data_as(C.c_void_p)
    tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
    wsb = lib.attwarp_ragged_attention_workspace_bytes(table_p, n)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_warp_ragged_from_attention(table_p, atab_p, n, TORCH_DTYPE_IDS[maps[0].dtype], Cc,
                                                     C.byref(tp), ptr(ws), ws.numel(), current_stream(dev)))
    return (outs, map_xs, map_ys) if return_maps else outs


def warp_ragged_from_mota_tokens(tok: torch.Tensor, images, out_sizes=None, kernel_size: int = 3,
                                 enhance_coe: float = 10.0, apply_inverse: bool = False, return_maps: bool = False):
    """The drivers' flow for a mixed-size list: per image ``blend_mask`` (revise_mask -> uint8 -> Pillow LANCZOS resize
    to that image's own size, llava.py:240-256) then ``save_warped_image(..., "identity")`` -- one ``revise_mask``
    launch for all token maps, then ``attwarp_warp_ragged_from_mask``: one fused LANCZOS + marginals launch, one finish
    launch and the stage-5 launches of ``warp_ragged_from_tokens``.

    tok     [n, gh, gw] float32 token maps on the device
    images  sequence of n uint8 HWC tensors [H_i, W_i, C], C in {1, 3, 4}, on the same device
    out_sizes  sequence of (Ho_i, Wo_i), default = input sizes
    Returns the list of warped images, and with ``return_maps`` also the lists of map_x [Wo_i] and map_y [Ho_i].
    An image's maps are bit-identical to ``maps_from_mota_tokens`` on that image alone (images the fused kernel does not
    take -- down-scaling, smaller than the token grid -- are resized first, as that call does)."""
    lib = load()
    n = len(images)
    if not isinstance(tok, torch.Tensor) or tok.dim() != 3:
        raise ValueError("warp_ragged_from_mota_tokens: tok must be a [n, gh, gw] tensor")
    if tok.shape[0] != n:
        raise ValueError(f"warp_ragged_from_mota_tokens: {tok.shape[0]} token maps for {n} images")
    if n == 0:
        return ([], [], []) if return_maps else []
    imgs, outs, out_sizes, table = _ragged_list("warp_ragged_from_mota_tokens", images, out_sizes, None, tok)
    dev = tok.device
    Cc = imgs[0].shape[2]
    if Cc not in (1, 3, 4):
        raise ValueError(f"warp_ragged_from_mota_tokens: images must be uint8 [H, W, C] with C in (1, 3, 4), got "
                         f"{tuple(imgs[0].shape)}")
    _, u8 = revise_mask(tok, kernel_size, enhance_coe, return_u8=True)
    gh, gw = int(u8.shape[1]), int(u8.shape[2])
    map_x = map_y = None
    if return_maps:
        map_x = torch.empty(int(table["Wo"].sum()), dtype=torch.float32, device=dev)
        map_y = torch.empty(int(table["Ho"].sum()), dtype=torch.float32, device=dev)
    table_p = table.ctypes.data_as(C.c_void_p)           # `table` stays alive until the call returns
    tp = _tp("identity", 1.0, 1.0, apply_inverse)
    wsb = lib.attwarp_ragged_mask_workspace_bytes(table_p, n, gh, gw)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_warp_ragged_from_mask(table_p, ptr(u8), n, gh, gw, Cc, C.byref(tp), ptr(ws), ws.numel(),
                                                ptr(map_x), ptr(map_y), current_stream(dev)))
    if not return_maps:
        return outs
    return (outs, list(map_x.split([wo for _, wo in out_sizes])), list(map_y.split([ho for ho, _ in out_sizes])))


class RaggedBatch:
    """A mixed-resolution batch whose buffers stay put across calls (the steady state of a driver that re-uses its
    image and output buffers): the descriptor table, the output tensors and a private workspace are built ONCE,
    ``run(tok)`` is a single library call with no per-image Python work (building the table for 1024 images costs
    more host time than the GPU needs to warp them).

        batch = RaggedBatch(images, out_sizes)        # uint8 HWC device tensors
        warped = batch.run(tok)                       # tok [n, gh, gw] float32 on the device -> batch.outs
    """

    def __init__(self, images, out_sizes=None, outs=None):
        lib = load()
        n = len(images)
        assert n > 0
        self.images, self.outs, self.out_sizes, table = _ragged_list("RaggedBatch", images, out_sizes, outs, images[0])
        self.device = self.images[0].device
        self.C = int(self.images[0].shape[2])
        self._table = table
        self._table_p = table.ctypes.data_as(C.c_void_p)
        self.n = n
        self.launches = 0            # kernels the last run() enqueued (maps + one resample launch per class)
        self._ws = torch.empty(max(int(lib.attwarp_ragged_workspace_bytes(self._table_p, n)), 256), dtype=torch.uint8,
                               device=self.device)

    def run(self, tok: torch.Tensor, grid_hw=None, transform="identity", exp_scale=1.0, exp_divisor=1.0,
            apply_inverse=False):
        """Stages 2-5 over the batch, enqueued on the current stream; returns ``self.outs``."""
        lib = load()
        if tok.dim() == 3:
            gh, gw = tok.shape[1], tok.shape[2]
        else:
            gh, gw = grid_hw
        if tok.shape[0] != self.n or tok.device != self.device:
            raise ValueError(f"RaggedBatch.run: {self.n} token maps on {self.device} expected")
        if tok.dtype != torch.float32 or not tok.is_contiguous():
            tok = tok.to(torch.float32).contiguous()
        tp = _tp(transform, exp_scale, exp_divisor, apply_inverse)
        with torch.cuda.device(self.device):
            check(lib.attwarp_warp_ragged_from_tokens(ptr(tok), self.n, gh, gw, self._table_p, self.C, C.byref(tp),
                                                      ptr(self._ws), self._ws.numel(), current_stream(self.device)))
            self.launches = int(lib.attwarp_ragged_last_launches())      # kernels this call enqueued
        return self.outs


# --------------------------------------------------------------------------------------------
# PNG encode (the warped images' way to disk)
# --------------------------------------------------------------------------------------------
# attwarp_png_image (include/attwarp.h)
_PNG_DTYPE = np.dtype([("src", np.uint64), ("H", np.int32), ("W", np.int32), ("C", np.int32), ("pad", np.int32)])


def encode_png(images):
    """PNG files of n uint8 device images of any shapes, in two launches on the current stream (nothing
    synchronises).

    images  a sequence of uint8 CUDA tensors [H, W] or [H, W, C] with C in {1, 3, 4} -- channel order as
            cv2.imwrite takes it: BGR(A) is stored as RGB(A), one channel as grey -- or a [B, H, W, C] tensor
    Returns (payload, offsets): uint8 [capacity] and int64 [n + 1] device tensors; file i is
    payload[offsets[i]:offsets[i + 1]].  A file's bytes depend only on its image's pixels; they are not cv2's
    bytes, the decoded pixels are the same (every row Sub-filtered, deflate of run-length matches in 32 KiB
    segments, within a few per mille of cv2's sizes on photo-like, smooth and noise images)."""
    lib = load()
    if isinstance(images, torch.Tensor):
        if images.dim() != 4:
            raise ValueError(f"encode_png: a tensor argument must be [B, H, W, C], got {tuple(images.shape)}")
        images = list(images.unbind(0))
    elif not isinstance(images, (list, tuple)):
        raise ValueError(f"encode_png: expected a sequence of image tensors or a [B, H, W, C] tensor, got {type(images)}")
    imgs = []
    for k, t in enumerate(images):
        if (not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or not t.is_cuda or t.dim() not in (2, 3)
                or (t.dim() == 3 and t.shape[2] not in (1, 3, 4)) or t.numel() == 0):
            desc = f"{t.dtype} {tuple(t.shape)} on {t.device}" if isinstance(t, torch.Tensor) else type(t).__name__
            raise ValueError(f"encode_png: image {k} must be a non-empty uint8 CUDA tensor [H, W] or [H, W, C] with "
                             f"C in (1, 3, 4), got {desc}")
        imgs.append(t.contiguous())
    n = len(imgs)
    dev = imgs[0].device if n else torch.device("cuda", torch.cuda.current_device())
    if any(t.device != dev for t in imgs):
        raise ValueError("encode_png: all images must be on one device")
    if n == 0:
        return torch.empty(0, dtype=torch.uint8, device=dev), torch.zeros(1, dtype=torch.int64, device=dev)
    table = np.zeros(n, dtype=_PNG_DTYPE)
    table["src"] = [t.data_ptr() for t in imgs]
    table["H"] = [t.shape[0] for t in imgs]
    table["W"] = [t.shape[1] for t in imgs]
    table["C"] = [t.shape[2] if t.dim() == 3 else 1 for t in imgs]
    table_p = table.ctypes.data_as(C.c_void_p)           # `table` stays alive until the call returns
    cap = sum(int(lib.attwarp_png_max_bytes(int(h), int(w), int(c))) for h, w, c in zip(table["H"], table["W"], table["C"]))
    payload = torch.empty(cap, dtype=torch.uint8, device=dev)
    offsets = torch.empty(n + 1, dtype=torch.int64, device=dev)
    wsb = lib.attwarp_png_workspace_bytes(table_p, n)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_encode_png(table_p, n, ptr(ws), ws.numel(), ptr(payload), cap, ptr(offsets),
                                     current_stream(dev)))
    return payload, offsets


# --------------------------------------------------------------------------------------------
# Baseline JPEG decode, bit-identical to Pillow (the reference drivers' reader)
# --------------------------------------------------------------------------------------------
# attwarp_jpeg_info / attwarp_jpeg_image (include/attwarp.h)
_JPEG_INFO_DTYPE = np.dtype([("H", np.int32), ("W", np.int32), ("components", np.int32), ("support", np.int32)])
_JPEG_DTYPE = np.dtype([("host", np.uint64), ("dev", np.uint64), ("nbytes", np.uint64), ("dst", np.uint64),
                        ("H", np.int32), ("W", np.int32)])
JPEG_SUPPORT_REASONS = {1: "not a JPEG file", 2: "truncated markers", 3: "progressive", 4: "arithmetic-coded",
                        5: "lossless or hierarchical", 6: "12-bit samples or 16-bit quantisation tables",
                        7: "colour space other than grey / YCbCr", 8: "sampling factors",
                        9: "multi-scan, DNL or data after EOI", 10: "missing or invalid table", 11: "size"}
JPEG_STATUS_REASONS = {1: "entropy-coded data ends before the last block", 2: "invalid Huffman code",
                       3: "coefficient index past 63", 4: "restart marker missing or out of order",
                       5: "unexpected marker inside the entropy-coded data"}


def jpeg_probe(buf) -> tuple:
    """(H, W, components, support) of a file's bytes from its markers, on the host (no GPU).  support 0: the file
    is one ``decode_jpeg`` takes; otherwise a key of ``JPEG_SUPPORT_REASONS``."""
    data = np.frombuffer(bytes(buf), dtype=np.uint8)
    info = np.zeros(1, dtype=_JPEG_INFO_DTYPE)
    check(load().attwarp_jpeg_probe(data.ctypes.data_as(C.c_void_p), data.size, info.ctypes.data_as(C.c_void_p)))
    return tuple(int(info[0][k]) for k in ("H", "W", "components", "support"))


def decode_jpeg(buffers, device=None):
    """Baseline JPEG files (a sequence of bytes-like objects) -> list of uint8 [H, W, 3] **BGR** CUDA tensors,
    bit-identical to ``np.array(Image.open(f).convert('RGB'))[..., ::-1]`` (Pillow's libjpeg-turbo: ISLOW IDCT,
    fancy up-sampling); grey files come out as three equal channels.  The whole list is decoded on the GPU in seven
    launches: only the compressed bytes are copied to the device (one copy from pinned memory).

    Raises ValueError naming the first file ``jpeg_probe`` does not accept (see include/attwarp.h for the subset),
    and, after one synchronisation that reads the per-file status, the first file whose entropy-coded data is
    malformed (no pixels of such a file are returned)."""
    lib = load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    bufs = [bytes(b) for b in buffers]
    n = len(bufs)
    if n == 0:
        return []
    infos = [jpeg_probe(b) for b in bufs]
    for i, (_, _, _, sup) in enumerate(infos):
        if sup != 0:
            raise ValueError(f"decode_jpeg: file {i} is not device-decodable: "
                             f"{JPEG_SUPPORT_REASONS.get(sup, sup)} (support code {sup})")
    sizes = [len(b) for b in bufs]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    host = torch.empty(int(offs[-1]), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    for b, o in zip(bufs, offs[:-1]):
        hv[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
    with torch.cuda.device(dev):
        data = host.to(dev, non_blocking=True)
        outs = [torch.empty((h, w, 3), dtype=torch.uint8, device=dev) for h, w, _, _ in infos]
        status = torch.empty(n, dtype=torch.int32, device=dev)
        table = np.zeros(n, dtype=_JPEG_DTYPE)
        table["host"] = host.data_ptr() + offs[:-1]
        table["dev"] = data.data_ptr() + offs[:-1]
        table["nbytes"] = sizes
        table["dst"] = [t.data_ptr() for t in outs]
        table["H"] = [h for h, _, _, _ in infos]
        table["W"] = [w for _, w, _, _ in infos]
        table_p = table.ctypes.data_as(C.c_void_p)
        wsb = lib.attwarp_jpeg_workspace_bytes(table_p, n)
        ws = _workspace(wsb, dev)
        check(lib.attwarp_decode_jpeg(table_p, n, ptr(ws), ws.numel(), ptr(status), current_stream(dev)))
        st = status.cpu().numpy()                      # synchronises: the decode (and the upload) have run
    bad = np.nonzero(st)[0]
    if bad.size:
        i = int(bad[0])
        raise ValueError(f"decode_jpeg: file {i} has malformed entropy-coded data: "
                         f"{JPEG_STATUS_REASONS.get(int(st[i]), int(st[i]))} (status {int(st[i])})")
    return outs


# --------------------------------------------------------------------------------------------
# PNG decode, pixel for pixel as Pillow's convert('RGB')
# --------------------------------------------------------------------------------------------
# attwarp_png_info / attwarp_png_file (include/attwarp.h)
_PNG_INFO_DTYPE = np.dtype([("H", np.int32), ("W", np.int32), ("colour_type", np.int32), ("bit_depth", np.int32),
                            ("support", np.int32)])
_PNG_FILE_DTYPE = _JPEG_DTYPE
PNG_SUPPORT_REASONS = {1: "not a PNG file", 2: "truncated", 3: "16-bit samples", 4: "interlaced",
                       5: "bad CRC on a critical chunk", 6: "chunk structure, IHDR or zlib header", 7: "size"}
PNG_STATUS_REASONS = {1: "invalid deflate block type", 2: "invalid Huffman code", 3: "distance too far back",
                      4: "stored block length mismatch", 5: "zlib stream ends early", 6: "Adler-32 mismatch",
                      7: "IDAT CRC mismatch", 8: "invalid filter type", 9: "too little image data"}


class PngDecodeError(ValueError):
    """A file ``decode_png`` refuses: ``file`` is its index in the call's list, ``reason`` what is wrong with it."""

    def __init__(self, file: int, reason: str):
        super().__init__(f"decode_png: file {file} {reason}")
        self.file, self.reason = file, reason


def png_probe(buf) -> tuple:
    """(H, W, colour_type, bit_depth, support) of a file's bytes from its chunks, on the host (no GPU).  support 0:
    the file is one ``decode_png`` takes; otherwise a key of ``PNG_SUPPORT_REASONS``."""
    data = np.frombuffer(bytes(buf), dtype=np.uint8)
    info = np.zeros(1, dtype=_PNG_INFO_DTYPE)
    check(load().attwarp_png_probe(data.ctypes.data_as(C.c_void_p), data.size, info.ctypes.data_as(C.c_void_p)))
    return tuple(int(info[0][k]) for k in ("H", "W", "colour_type", "bit_depth", "support"))


def decode_png(buffers, device=None):
    """PNG files (a sequence of bytes-like objects) -> list of uint8 [H, W, 3] **BGR** CUDA tensors, equal to
    ``np.array(Image.open(f).convert('RGB'))[..., ::-1]``.  The whole list is decoded on the GPU in one launch:
    only the file bytes are copied to the device (one copy from pinned memory).

    Raises ``PngDecodeError`` (a ValueError) naming the first file ``png_probe`` does not accept (see
    include/attwarp.h for the subset), and, after one synchronisation that reads the per-file status, the first
    malformed file (no pixels of such a file are returned)."""
    lib = load()
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    bufs = [bytes(b) for b in buffers]
    n = len(bufs)
    if n == 0:
        return []
    infos = [png_probe(b) for b in bufs]
    for i, info in enumerate(infos):
        sup = info[4]
        if sup != 0:
            raise PngDecodeError(i, f"is not device-decodable: {PNG_SUPPORT_REASONS.get(sup, sup)} "
                                    f"(support code {sup})")
    sizes = [len(b) for b in bufs]
    offs = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    host = torch.empty(int(offs[-1]), dtype=torch.uint8, pin_memory=True)
    hv = host.numpy()
    for b, o in zip(bufs, offs[:-1]):
        hv[o:o + len(b)] = np.frombuffer(b, dtype=np.uint8)
    with torch.cuda.device(dev):
        data = host.to(dev, non_blocking=True)
        outs = [torch.empty((info[0], info[1], 3), dtype=torch.uint8, device=dev) for info in infos]
        status = torch.empty(n, dtype=torch.int32, device=dev)
        table = np.zeros(n, dtype=_PNG_FILE_DTYPE)
        table["host"] = host.data_ptr() + offs[:-1]
        table["dev"] = data.data_ptr() + offs[:-1]
        table["nbytes"] = sizes
        table["dst"] = [t.data_ptr() for t in outs]
        table["H"] = [info[0] for info in infos]
        table["W"] = [info[1] for info in infos]
        table_p = table.ctypes.data_as(C.c_void_p)
        wsb = lib.attwarp_png_decode_workspace_bytes(table_p, n)
        ws = _workspace(wsb, dev)
        check(lib.attwarp_decode_png(table_p, n, ptr(ws), ws.numel(), ptr(status), current_stream(dev)))
        st = status.cpu().numpy()                      # synchronises: the decode (and the upload) have run
    bad = np.nonzero(st)[0]
    if bad.size:
        i = int(bad[0])
        raise PngDecodeError(i, f"is malformed: {PNG_STATUS_REASONS.get(int(st[i]), int(st[i]))} "
                                f"(status {int(st[i])})")
    return outs


# --------------------------------------------------------------------------------------------
# Attention overlay (save_warped_image's masked_overlay_save_path image)
# --------------------------------------------------------------------------------------------
# attwarp_overlay_image (include/attwarp.h)
_OVERLAY_DTYPE = np.dtype([("src", np.uint64), ("att", np.uint64), ("dst", np.uint64), ("H", np.int32),
                           ("W", np.int32), ("C", np.int32), ("pad", np.int32)])
_OVERLAY_MAP, _OVERLAY_TOKENS = 0, 1
_OVERLAY_ATT_DTYPES = (torch.uint8, torch.float32, torch.float64)


def attention_overlay(images, att=None, tok=None, alpha: float = 0.5):
    """The JET attention overlay ``save_warped_image`` writes (``masked_overlay_save_path``) for n images of any
    sizes, in two launches on the current stream (nothing synchronises).  Bit-identical to that host expression:
    ``cv2.addWeighted(applyColorMap(uint8(n * 255), JET), alpha, base, 1 - alpha, 0)`` with
    ``n = (a - lo) / (hi - lo) if hi > lo + 1e-9 else 0`` in the precision NumPy gives the map's dtype (the
    contract: INTEGRATION.md section B.5b, include/attwarp.h).

    images  a sequence of uint8 CUDA tensors [H, W, 3] (BGR) or [H, W] / [H, W, 1] (grey, replicated to BGR as
            cv2.cvtColor(GRAY2BGR) does), or a [B, H, W, C] tensor
    att     per-image attention maps of each image's own size: a sequence of [H, W] tensors or a [B, H, W] tensor,
            uint8, float32 or float64 (e.g. the uint8 mask ``mota_mask`` / ``blend_mask`` gives)
    tok     or [n, gh, gw] float32 token maps, index-upsampled to each image as ``maps_from_tokens`` does
            (``(y * gh) // H``, ``(x * gw) // W``); lo and hi are those of the upsampled map
    alpha   the heat map's weight (finite); the image's is 1 - alpha
    Returns a list of uint8 [H, W, 3] BGR CUDA tensors (views of one buffer).  Exactly one of ``att`` / ``tok``.
    A map of another size than its image is refused: the reference resizes it with cv2.resize(INTER_LINEAR),
    whose float result is not reproducible bit for bit."""
    lib = load()
    if (att is None) == (tok is None):
        raise ValueError("attention_overlay: give exactly one of att (per-image maps) or tok (token maps)")
    if isinstance(images, torch.Tensor):
        if images.dim() != 4:
            raise ValueError(f"attention_overlay: a tensor argument must be [B, H, W, C], got {tuple(images.shape)}")
        images = list(images.unbind(0))
    elif not isinstance(images, (list, tuple)):
        raise ValueError(f"attention_overlay: expected a sequence of image tensors or a [B, H, W, C] tensor, "
                         f"got {type(images)}")
    try:
        alpha = float(alpha)
    except (TypeError, ValueError):
        raise ValueError(f"attention_overlay: alpha must be a finite number, got {alpha!r}") from None
    if not np.isfinite(alpha):
        raise ValueError(f"attention_overlay: alpha must be finite, got {alpha}")
    imgs, chans = [], []
    for k, t in enumerate(images):
        if not isinstance(t, torch.Tensor):
            raise ValueError(f"attention_overlay: image {k} is a {type(t).__name__}, not a tensor")
        if t.dtype != torch.uint8:
            raise ValueError(f"attention_overlay: image {k} must be uint8, got {t.dtype}")
        if t.dim() == 3 and t.shape[2] == 4:
            raise ValueError(f"attention_overlay: image {k} has 4 channels; the reference's cv2.addWeighted of a "
                             "3-channel heat map fails on them too")
        if t.dim() not in (2, 3) or (t.dim() == 3 and t.shape[2] not in (1, 3)) or t.numel() == 0:
            raise ValueError(f"attention_overlay: image {k} must be a non-empty [H, W], [H, W, 1] or [H, W, 3] "
                             f"tensor, got {tuple(t.shape)}")
        imgs.append(t.contiguous())
        chans.append(3 if t.dim() == 3 and t.shape[2] == 3 else 1)
    n = len(imgs)
    if tok is not None:
        if not isinstance(tok, torch.Tensor) or tok.dim() != 3:
            raise ValueError("attention_overlay: tok must be a [n, gh, gw] tensor")
        if tok.dtype != torch.float32:
            raise ValueError(f"attention_overlay: tok must be float32, got {tok.dtype}")
        if tok.shape[0] != n:
            raise ValueError(f"attention_overlay: {tok.shape[0]} token maps for {n} images")
        if tok.shape[1] == 0 or tok.shape[2] == 0:
            raise ValueError(f"attention_overlay: empty token grid {tuple(tok.shape[1:])}")
        atts = list(tok.contiguous().unbind(0)) if n else []
    else:
        if isinstance(att, torch.Tensor):
            if att.dim() != 3:
                raise ValueError(f"attention_overlay: an att tensor must be [B, H, W], got {tuple(att.shape)}")
            att = list(att.unbind(0))
        elif not isinstance(att, (list, tuple)):
            raise ValueError(f"attention_overlay: att must be a sequence of [H, W] tensors or a [B, H, W] tensor")
        if len(att) != n:
            raise ValueError(f"attention_overlay: {len(att)} attention maps for {n} images")
        atts = []
        for k, (a, im) in enumerate(zip(att, imgs)):
            if not isinstance(a, torch.Tensor):
                raise ValueError(f"attention_overlay: attention map {k} is a {type(a).__name__}, not a tensor")
            if a.dtype not in _OVERLAY_ATT_DTYPES:
                raise ValueError(f"attention_overlay: attention map {k} has dtype {a.dtype}; uint8, float32 and "
                                 "float64 are supported")
            if tuple(a.shape) != tuple(im.shape[:2]):
                raise ValueError(f"attention_overlay: attention map {k} is {tuple(a.shape)}, image {k} is "
                                 f"{tuple(im.shape[:2])}: a map of another size would need the reference's "
                                 "cv2.resize(INTER_LINEAR), whose float result is not reproducible bit for bit; "
                                 "resize it to the image first")
            atts.append(a.contiguous())
        if len({a.dtype for a in atts}) > 1:
            raise ValueError("attention_overlay: all attention maps must have one dtype")
    if n == 0:
        return []
    dev = imgs[0].device
    if not imgs[0].is_cuda or any(t.device != dev for t in imgs + atts):
        raise ValueError("attention_overlay: images and attention must all be on one CUDA device")
    for k, t in enumerate(imgs):
        if t.shape[0] > 65535 or t.shape[1] > 65535:
            raise ValueError(f"attention_overlay: image {k} is {tuple(t.shape[:2])}; H and W must be at most 65535")
    if tok is not None and (tok.shape[1] > 65535 or tok.shape[2] > 65535):
        raise ValueError(f"attention_overlay: token grid {tuple(tok.shape[1:])} above 65535")
    # outputs: one buffer, each image at a 16-byte aligned offset
    sizes = [int(t.shape[0]) * int(t.shape[1]) * 3 for t in imgs]
    offs = np.zeros(n + 1, dtype=np.int64)
    offs[1:] = np.cumsum([(s + 15) // 16 * 16 for s in sizes])
    buf = torch.empty(int(offs[-1]), dtype=torch.uint8, device=dev)
    outs = [buf[int(o):int(o) + s].view(int(t.shape[0]), int(t.shape[1]), 3) for o, s, t in zip(offs, sizes, imgs)]
    table = np.zeros(n, dtype=_OVERLAY_DTYPE)
    table["src"] = [t.data_ptr() for t in imgs]
    table["att"] = [a.data_ptr() for a in atts]
    table["dst"] = [o.data_ptr() for o in outs]
    table["H"] = [t.shape[0] for t in imgs]
    table["W"] = [t.shape[1] for t in imgs]
    table["C"] = chans
    table_p = table.ctypes.data_as(C.c_void_p)           # `table` stays alive until the call returns
    kind = _OVERLAY_TOKENS if tok is not None else _OVERLAY_MAP
    gh, gw = (int(tok.shape[1]), int(tok.shape[2])) if tok is not None else (0, 0)
    wsb = lib.attwarp_overlay_workspace_bytes(table_p, n, kind)
    ws = _workspace(wsb, dev)
    with torch.cuda.device(dev):
        check(lib.attwarp_attention_overlay(table_p, n, TORCH_DTYPE_IDS[atts[0].dtype], kind, gh, gw, alpha,
                                            ptr(ws), ws.numel(), current_stream(dev)))
    return outs
