"""On-disk formats either side of the warp (SURVEY.md section 8(f) N3): the reference drivers read JPEG files
(``Image.open(path).convert('RGB')``, AGW/main.py:152, main_batched.py:98), hand PIL images to ``save_warped_image``,
which flips them to BGR (new_method.py:421-422) and writes PNG files with ``cv2.imwrite`` (:491).  With the warp at
~0.1 ms per batch those two steps ARE the driver's run time, so this module moves the decode onto the GPU and
batches the rest:

* ``decode_jpeg_batch(sources)``     JPEG bytes / paths -> uint8 HWC **BGR** device tensors, the layout stage 5
  reads (nvJPEG through ``torchvision.io.decode_jpeg(device=...)`` -- library code, like calling cuBLAS).
  NOT bit-identical to libjpeg: IDCT and chroma up-sampling differ between decoders.  Measured against Pillow (the
  reader the reference drivers use) on the B200 box, synthetic photo-like images with a saturated colour block,
  quality 90 (tests/test_image_io.py holds these bounds): 4:4:4 files: max 4 LSB, mean 0.5 LSB; 4:2:0 files: mean
  1.9 LSB, 99 % of the bytes within ~10 LSB, but up to ~100 LSB on the one-pixel rim of a saturated colour edge
  (nvJPEG replicates chroma samples where libjpeg's "fancy" up-sampling interpolates them).  ``exact=True`` decodes
  on the host with Pillow instead -- bit-identical to ``Image.open(path).convert('RGB')`` -- for runs that must
  reproduce the reference's pixels.  Anything that is not a JPEG (PNG, ...) is decoded on the host, exactly.
  ``exact_device=True`` gives the same pixels as ``exact=True`` with the JPEG decode on the GPU (``ops.decode_jpeg``,
  csrc/jpeg.cu: seven launches for the whole mixed-size list, only the compressed bytes cross PCIe): libjpeg-turbo's
  Huffman decode, ISLOW IDCT with its range-limit table, fancy h2v1 / h2v2 / h1v2 up-sampling (replication for
  4:1:1 and for chroma 2 samples wide or less) and ycc_rgb_convert, restated.  It takes baseline / extended
  sequential Huffman files with 8-bit samples, one interleaved scan (or one grey component), YCbCr (JFIF, or
  component IDs 1/2/3) or grey, luma sampling 4:4:4, 4:2:2, 4:2:0, 4:4:0 or 4:1:1, any restart interval, any
  tables, APPn / COM / EXIF skipped (no rotation, like Pillow's open).  Other JPEGs (progressive, arithmetic,
  12-bit, CMYK / YCCK / RGB, multi-scan, ...) go to Pillow and other formats to cv2, both exact; ``ops.jpeg_probe``
  tells which path a file takes.  A file whose entropy-coded data is malformed raises ValueError naming it (Pillow
  would recover from some such files with a warning; the device decoder never guesses pixels).
  PNGs go the same way under ``exact_device=True``: the ones ``ops.png_probe`` accepts (not interlaced; 8-bit
  grey / RGB / palette / grey + alpha / RGBA, 1/2/4-bit grey and palette) are decoded on the GPU in one
  ``ops.decode_png`` call (csrc/png_decode.cu: one launch for the whole mixed-size list, the inflate of each file
  split across a CTA), giving the pixels cv2.imdecode and Pillow give them; they accept and reject the malformed
  files libpng does (bad IDAT CRC, Adler-32, truncated stream, too few rows, a filter type above 4 rejected; a bad
  ancillary CRC, extra rows, bytes after the stream accepted).  Other PNGs stay with cv2.  Known gap: for 16-bit
  grey files cv2 (which decodes them on that path) shifts samples right by 8 where Pillow's ``convert('RGB')``
  clips them to 255, so under ``exact_device=True`` those files are not Pillow's pixels (DESIGN.md section 6 item 9).
* ``encode_png_batch(images, paths)`` device tensors -> PNG files: device -> pinned host copy, then
  ``cv2.imwrite`` in a thread pool -- the reference's own encoder, so the files decode to the same bytes.
  ``on_device=True`` encodes on the GPU instead (``encode_png_device``, ``ops.encode_png``: two launches for the
  whole mixed-size list) and only the compressed bytes cross PCIe.  Like ``decode_jpeg_batch(exact=...)`` the
  keyword trades byte identity for speed, here of the FILE bytes only: PNG is lossless and the pixels are the
  same.  What the device encoder's files satisfy:
    1. ``cv2.imdecode(buf, cv2.IMREAD_UNCHANGED)`` returns the input array exactly (Pillow: the same pixels in
       RGB(A) order): HWC BGR is stored as RGB (colour type 2), BGRA as RGBA (6), [H, W] / [H, W, 1] as grey (0);
       bit depth 8, no interlace -- the IHDR cv2.imencode writes.
    2. Signature, IHDR, IDAT chunks, IEND with a correct CRC-32 each; the IDAT payloads are one zlib stream
       (78 01, deflate blocks, Adler-32) of the filtered scanlines.
    3. A file's bytes depend only on its pixels (not on the batch, the position in it, the stream or the run).
    4. Sizes: every row Sub-filtered, like cv2 4.13; the stream cut into 32 KiB segments, each one deflate block of
       distance-1 matches (zlib's Z_RLE, what cv2 evidently uses at level 1) under its own dynamic Huffman code, or
       stored when that is not smaller.  Measured on the CPU with the encoder's own block builder against
       cv2.imencode 4.13: 0.998x on photo-like, 1.000-1.003x on smooth gradients, 0.999x on noise (336^2, 500^2,
       1344^2); noise never exceeds the stored size plus 17 bytes per 32 KiB and 75 bytes per file.
* ``warp_files(...)``                the driver loop of main_batched.py:243-287 for a whole list of files: decode
  -> one ragged launch per stage -> encode (``on_device_png=True``: the device encoder above).  With
  ``overlay_paths`` / ``original_paths`` it also writes the other two files ``save_warped_image`` writes: the JET
  attention overlay (``ops.attention_overlay``, bit-identical to the host expression) and the decoded image.
"""

from __future__ import annotations

import concurrent.futures as cf
import os
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import ops


def _read_bytes(src) -> bytes:
    if isinstance(src, (bytes, bytearray, memoryview)):
        return bytes(src)
    with open(os.fspath(src), "rb") as f:
        return f.read()


def _is_jpeg(buf: bytes) -> bool:
    return len(buf) > 3 and buf[0] == 0xFF and buf[1] == 0xD8


def _is_png(buf: bytes) -> bool:
    return buf[:8] == b"\x89PNG\r\n\x1a\n"


def _pillow_bgr(b: bytes, dev) -> torch.Tensor:
    import io

    from PIL import Image
    rgb = np.array(Image.open(io.BytesIO(b)).convert("RGB"))
    return torch.from_numpy(np.ascontiguousarray(rgb[..., ::-1])).to(dev, non_blocking=True)


def decode_jpeg_batch(sources: Sequence, device=None, exact: bool = False,
                      exact_device: bool = False) -> List[torch.Tensor]:
    """Paths or encoded bytes -> list of uint8 [H, W, 3] BGR tensors on ``device`` (cv2.imread's channel order, the
    one ``save_warped_image`` warps in).  JPEG files are decoded on the GPU in one batched nvJPEG call; grey JPEGs
    come out as three equal channels (like ``Image.convert('RGB')``).  ``exact=True``: host decode with Pillow,
    bit-identical to the reference's reader, then one copy to the device.  ``exact_device=True``: bit-identical too,
    with the JPEGs ``ops.jpeg_probe`` accepts decoded on the GPU in one ``ops.decode_jpeg`` call and the PNGs
    ``ops.png_probe`` accepts in one ``ops.decode_png`` call; other JPEGs (progressive, CMYK, ...) are decoded by
    Pillow and other files (16-bit or interlaced PNGs, ...) by cv2, as without the keyword."""
    if exact and exact_device:
        raise ValueError("decode_jpeg_batch: exact and exact_device are exclusive")
    dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    bufs = [_read_bytes(s) for s in sources]
    out: List[Optional[torch.Tensor]] = [None] * len(bufs)
    if exact:
        for i, b in enumerate(bufs):
            out[i] = _pillow_bgr(b, dev)
        return out  # type: ignore[return-value]
    if exact_device:
        jpegs = [i for i, b in enumerate(bufs) if _is_jpeg(b)]
        dev_idx = [i for i in jpegs if ops.jpeg_probe(bufs[i])[3] == 0]
        if dev_idx:
            for i, t in zip(dev_idx, ops.decode_jpeg([bufs[i] for i in dev_idx], dev)):
                out[i] = t
        for i in jpegs:
            if out[i] is None:
                out[i] = _pillow_bgr(bufs[i], dev)
        png_idx = [i for i, b in enumerate(bufs) if _is_png(b) and ops.png_probe(b)[4] == 0]
        if png_idx:
            try:
                decoded = ops.decode_png([bufs[i] for i in png_idx], dev)
            except ops.PngDecodeError as exc:
                raise ValueError(f"decode_jpeg_batch: source {png_idx[exc.file]} {exc.reason}") from exc
            for i, t in zip(png_idx, decoded):
                out[i] = t
        return _decode_others(bufs, out, dev)
    from torchvision.io import ImageReadMode, decode_jpeg
    jpeg_idx = [i for i, b in enumerate(bufs) if _is_jpeg(b)]
    if jpeg_idx:
        datas = [torch.frombuffer(bytearray(bufs[i]), dtype=torch.uint8) for i in jpeg_idx]
        decoded = decode_jpeg(datas, mode=ImageReadMode.RGB, device=dev)          # list of [3, H, W] RGB
        for i, t in zip(jpeg_idx, decoded):
            out[i] = t.flip(0).permute(1, 2, 0).contiguous()                      # -> [H, W, 3] BGR
    return _decode_others(bufs, out, dev)


def _decode_others(bufs, out, dev) -> List[torch.Tensor]:
    """cv2.imdecode (exact) of the sources not decoded yet."""
    for i, b in enumerate(bufs):
        if out[i] is None:
            import cv2
            img = cv2.imdecode(np.frombuffer(b, dtype=np.uint8), cv2.IMREAD_COLOR)
            if img is None:
                raise ValueError(f"decode_jpeg_batch: source {i} is not a decodable image")
            out[i] = torch.from_numpy(img).to(dev)
    return out  # type: ignore[return-value]


def encode_png_device(images) -> List[bytes]:
    """uint8 device images ([H, W] or [H, W, C], C in {1, 3, 4}, mixed shapes; or a [B, H, W, C] tensor) -> the
    bytes of their PNG files, encoded on the GPU (``ops.encode_png``).  The offsets come to the host first, then
    the files in one copy to pinned memory; blocks until they are there."""
    payload, offsets = ops.encode_png(images)
    offs = offsets.cpu().tolist()                    # synchronises: the encode has run
    total = offs[-1]
    host = torch.empty(total, dtype=torch.uint8, pin_memory=True)
    if total:
        host.copy_(payload[:total], non_blocking=True)
        torch.cuda.current_stream(payload.device).synchronize()
    buf = host.numpy()
    return [buf[offs[k]:offs[k + 1]].tobytes() for k in range(len(offs) - 1)]


def _write_file(path, data: bytes) -> bool:
    try:
        with open(os.fspath(path), "wb") as f:
            f.write(data)
        return True
    except OSError:
        return False


def encode_png_batch(images: Sequence[torch.Tensor], paths: Sequence[str], workers: int = 8,
                     on_device: bool = False) -> List[bool]:
    """uint8 [H, W, 3] (BGR) or [H, W] device tensors -> PNG files with ``cv2.imwrite`` (the reference's encoder,
    new_method.py:491).  The device -> host copies are enqueued first (pinned staging), the encodes run in a
    thread pool (OpenCV releases the GIL).  Returns cv2.imwrite's result per file.
    ``on_device=True``: the files are encoded on the GPU (``encode_png_device``; also [H, W, 1] and BGRA [H, W, 4])
    and written with plain file writes; False for a file that cannot be written, like cv2.imwrite.  Same pixels,
    different file bytes (module docstring)."""
    assert len(images) == len(paths)
    if on_device:
        return [_write_file(p, b) for p, b in zip(paths, encode_png_device(list(images)))]
    import cv2
    host = []
    for t in images:
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t, non_blocking=True)
        host.append(h)
    if images:
        torch.cuda.current_stream(images[0].device).synchronize()

    def write(k):
        return bool(cv2.imwrite(os.fspath(paths[k]), host[k].numpy()))

    if workers <= 1 or len(paths) <= 1:
        return [write(k) for k in range(len(paths))]
    with cf.ThreadPoolExecutor(max_workers=min(workers, len(paths))) as ex:
        return list(ex.map(write, range(len(paths))))


def _mota_masks(tok: torch.Tensor, imgs: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    """blend_mask's uint8 mask of each image's size (``ops.mota_mask`` per image): one revise_mask launch, then one
    LANCZOS resize per distinct image size."""
    _, u8 = ops.revise_mask(tok, return_u8=True)
    groups = {}
    for k, im in enumerate(imgs):
        groups.setdefault((int(im.shape[0]), int(im.shape[1])), []).append(k)
    masks: List[Optional[torch.Tensor]] = [None] * len(imgs)
    for hw, idx in groups.items():
        for k, m in zip(idx, ops.resize_lanczos_u8(u8[idx], hw).unbind(0)):
            masks[k] = m
    return masks  # type: ignore[return-value]


def warp_files(image_sources: Sequence, tok: Optional[torch.Tensor], output_paths: Sequence[str], out_sizes=None,
               transform: str = "identity", exp_scale: float = 1.0, exp_divisor: float = 1.0,
               apply_inverse: bool = False, device=None, workers: int = 8, on_device_png: bool = False,
               overlay_paths: Optional[Sequence[str]] = None, original_paths: Optional[Sequence[str]] = None,
               overlay_alpha: float = 0.5, att=None, mask: str = "index", exact_decode: bool = False) -> List[bool]:
    """The per-image loop of the batched driver (main_batched.py:243-287: ``save_warped_image(image, mask, ...,
    width, height, "identity")`` per sample) for a list of image files and their token maps: GPU decode -> stages
    2-5 for the whole (mixed-resolution) list in one launch per stage -> PNG files.

    tok         [n, gh, gw] float32 token maps (the aggregated attention of each sample), index-upsampled to each
                image on the fly (BASELINE configs[3])
    att         or per-image attention maps of each decoded image's size ([H_i, W_i] CUDA tensors or NumPy arrays,
                uint8 / float32 / float64, one dtype): the reference's own input, e.g. ``blend_mask``'s uint8 mask or
                ``ops.mota_mask`` per image; warped with ``ops.warp_ragged_from_attention``.  Exactly one of
                ``tok`` / ``att``.
    mask        how ``tok`` becomes each image's attention: ``"index"`` upsamples the token map (nearest index, as
                above); ``"mota"`` is the drivers' own ``blend_mask`` mask -- revise_mask, then Pillow's LANCZOS
                resize to each image's size -- warped with ``ops.warp_ragged_from_mota_tokens`` (identity transform
                only), and the overlays are drawn from that mask as ``save_warped_image`` draws them
    out_sizes   per-image (height, width) of the warped files, default = the input sizes (the drivers pass the
                sample's own size, main_batched.py:276-287)
    on_device_png  encode the files on the GPU (``encode_png_batch(on_device=True)``): same pixels, other bytes
    overlay_paths  also write, per image, the JET attention overlay save_warped_image writes as
                   ``masked_overlay_save_path``: ``ops.attention_overlay`` of the decoded image and its attention
                   (``att``, or the token map index-upsampled like the warp's attention), weight ``overlay_alpha``
                   (the drivers' 0.5)
    original_paths also write, per image, the decoded image: save_warped_image's ``original_image_save_path``.
                   With nvJPEG decode these are nvJPEG's pixels (module docstring), not libjpeg's
    exact_decode   decode with ``decode_jpeg_batch(exact_device=True)``: the images are Pillow's pixels, bit for bit,
                   so the warped, overlay and original files are those of the reference's reader
    Every file goes through one encoder call (one ``ops.encode_png`` with ``on_device_png``, else one cv2.imwrite
    pool).  Returns one bool per file written, grouped per kind: the n warped files, then the n overlays if
    ``overlay_paths`` is given, then the n originals if ``original_paths`` is given -- a list of n, 2n or 3n."""
    n = len(image_sources)
    if (tok is None) == (att is None):
        raise ValueError("warp_files: give exactly one of tok (token maps) or att (per-image attention maps)")
    if att is not None and len(att) != n:
        raise ValueError(f"warp_files: {len(att)} attention maps for {n} images")
    for name, paths in (("overlay_paths", overlay_paths), ("original_paths", original_paths)):
        if paths is not None and len(paths) != n:
            raise ValueError(f"warp_files: {len(paths)} {name} for {n} images")
    if mask not in ("index", "mota"):
        raise ValueError(f"warp_files: mask must be 'index' or 'mota', got {mask!r}")
    if mask == "mota" and (tok is None or transform != "identity"):
        raise ValueError("warp_files: mask='mota' takes token maps and the identity transform (blend_mask's flow)")
    if n == 0:
        return []
    imgs = decode_jpeg_batch(image_sources, device, exact_device=exact_decode)
    dev = imgs[0].device
    if att is not None:
        maps = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) if isinstance(a, np.ndarray) else a.to(dev)
                for a in att]
        outs = ops.warp_ragged_from_attention(maps, imgs, out_sizes, transform=transform, exp_scale=exp_scale,
                                              exp_divisor=exp_divisor, apply_inverse=apply_inverse)
    elif mask == "mota":
        tok = tok.to(dev).reshape(n, tok.shape[-2], tok.shape[-1]).float()
        outs = ops.warp_ragged_from_mota_tokens(tok, imgs, out_sizes, apply_inverse=apply_inverse)
    else:
        tok = tok.to(dev)
        outs = ops.warp_ragged_from_tokens(tok, imgs, out_sizes, transform=transform, exp_scale=exp_scale,
                                           exp_divisor=exp_divisor, apply_inverse=apply_inverse)
    images, paths = list(outs), list(output_paths)
    if overlay_paths is not None:
        if att is not None:
            images += ops.attention_overlay(imgs, att=maps, alpha=overlay_alpha)
        elif mask == "mota":
            images += ops.attention_overlay(imgs, att=_mota_masks(tok, imgs), alpha=overlay_alpha)
        else:
            images += ops.attention_overlay(imgs, tok=tok.reshape(n, tok.shape[-2], tok.shape[-1]).float(),
                                            alpha=overlay_alpha)
        paths += list(overlay_paths)
    if original_paths is not None:
        images += list(imgs)
        paths += list(original_paths)
    return encode_png_batch(images, paths, workers, on_device=on_device_png)
