"""Ragged image-resolution marginals (profiles.cu, marginals_ragged_*) and the whole ops.warp_ragged_from_attention call.

    python profiles/ragged_attention_probe.py [--out result.json]

Cases (DESIGN.md section 4.2):
  a      64 x 1344^2 uint8 masks as a list, against maps_from_attention on the stacked tensor (the integer kernel)
  b      the same at 1344 x 1343 (rows off the 16-byte phase: the uniform path takes the generic kernel)
  c      the c4 size list (square sides from default_rng(1237).integers(224, 2049, 1024)), uint8 masks
  d-id   c4 with float32 maps, identity;  d-sqrt: the same with sqrt
Per case: the marginals launch's time (torch.profiler, a pass of its own), its GB/s over the map bytes and the share of
a device-to-device copy peak taken in the same run; the whole call (CUDA events, inputs rotated so that they do not
fit the 126 MB L2) against warp_ragged_from_tokens (24 x 24 tokens) on the same list and against a per-image loop of
maps_from_attention + remap_bilinear.  The card's name and power limit are read in the same run.
"""

import argparse
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from attwarp_b200 import ops  # noqa: E402

dev = torch.device("cuda")
gen = torch.Generator(device=dev).manual_seed(1)
L2_BYTES = 126 << 20
MARG_KEYS = ("marginals_ragged", "marginals_u8_identity", "marginals_partial", "marginals_f32_rows")


def case_list():
    c4 = [(int(s), int(s)) for s in np.random.default_rng(1237).integers(224, 2049, 1024)]
    return [("a", [(1344, 1344)] * 64, torch.uint8, "identity"),
            ("b", [(1344, 1343)] * 64, torch.uint8, "identity"),
            ("c", c4, torch.uint8, "identity"),
            ("d-id", c4, torch.float32, "identity"),
            ("d-sqrt", c4, torch.float32, "sqrt")]


def make_batch(sizes, dtype):
    imgs = [torch.randint(0, 256, (h, w, 3), device=dev, dtype=torch.uint8, generator=gen) for h, w in sizes]
    uniform = len(set(sizes)) == 1
    if dtype == torch.uint8:
        draw = lambda shape: torch.randint(0, 256, shape, device=dev, dtype=torch.uint8, generator=gen)
    else:
        draw = lambda shape: torch.rand(shape, device=dev, generator=gen)
    if uniform:                                  # one stacked tensor; the list holds views of it
        stacked = draw((len(sizes),) + sizes[0])
        maps = list(stacked.unbind(0))
    else:
        stacked = None
        maps = [draw(hw) for hw in sizes]
    tok = torch.rand((len(sizes), 24, 24), device=dev, generator=gen)
    return dict(imgs=imgs, maps=maps, stacked=stacked, tok=tok)


def copy_peak():
    a = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    return 2 * a.numel() * 10 / (e0.elapsed_time(e1) / 1e3)


def time_events(fn, batches, reps):
    for b in batches:
        fn(b)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for r in range(reps):
        fn(batches[r % len(batches)])
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


def marginals_time(fn, batches, reps=4):
    """Seconds per call of the marginals launch(es) fn enqueues, from torch.profiler, and their kernel names."""
    fn(batches[0])
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for r in range(reps):
            fn(batches[r % len(batches)])
        torch.cuda.synchronize()
    tot, names = 0.0, set()
    for e in prof.key_averages():
        if any(k in e.key for k in MARG_KEYS):
            tot += e.device_time_total
            names.add(re.search(r"marginals_\w+?_kernel(<[^>]*>)?", e.key).group(0))
    return tot / reps / 1e6, sorted(names)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    card = q[0] if q else torch.cuda.get_device_name(dev)
    peak = copy_peak()
    print(f"GPU: {card}\ndevice-to-device copy peak (1 GiB, read + write): {peak / 1e9:.0f} GB/s\n")
    res = dict(card=card, copy_peak_gbs=peak / 1e9, cases={})
    for name, sizes, dtype, transform in case_list():
        es = torch.tensor([], dtype=dtype).element_size()
        map_bytes = sum(h * w for h, w in sizes) * es
        img_bytes = sum(h * w for h, w in sizes) * 3
        copies = max(1, -(-2 * L2_BYTES // (map_bytes + 2 * img_bytes)))
        batches = [make_batch(sizes, dtype) for _ in range(copies)]
        hw = list(sizes)
        ragged = lambda b: ops.warp_ragged_from_attention(b["maps"], b["imgs"], hw, transform)
        tokens = lambda b: ops.warp_ragged_from_tokens(b["tok"], b["imgs"], hw, transform=transform)

        def loop(b):
            for m, im in zip(b["maps"], b["imgs"]):
                mx, my = ops.maps_from_attention(m[None], m.shape, transform)
                ops.remap_bilinear(im[None], mx, my)

        r = {"images": len(sizes), "map_MB": map_bytes / 1e6, "copies": copies}
        t_marg, names = marginals_time(ragged, batches)
        r.update(ragged_kernels=names, ragged_marg_us=t_marg * 1e6, ragged_marg_gbs=map_bytes / t_marg / 1e9,
                 ragged_marg_peak=map_bytes / t_marg / peak)
        if batches[0]["stacked"] is not None:
            uni = lambda b: ops.maps_from_attention(b["stacked"], sizes[0], transform)
            t_uni, unames = marginals_time(uni, batches)
            r.update(uniform_kernels=unames, uniform_marg_us=t_uni * 1e6, uniform_marg_gbs=map_bytes / t_uni / 1e9,
                     ragged_over_uniform=t_marg / t_uni)
        reps = 20 if len(sizes) <= 64 else 6
        r["call_us"] = time_events(ragged, batches, reps) * 1e6
        r["tokens_call_us"] = time_events(tokens, batches, reps) * 1e6
        r["loop_call_us"] = time_events(loop, batches, 3) * 1e6
        r["call_over_tokens"] = r["call_us"] / r["tokens_call_us"]
        r["loop_over_call"] = r["loop_call_us"] / r["call_us"]
        res["cases"][name] = r
        line = (f"{name:7s} {len(sizes):5d} maps {map_bytes / 1e6:8.1f} MB | marginals {t_marg * 1e6:8.1f} us "
                f"{r['ragged_marg_gbs']:6.0f} GB/s {r['ragged_marg_peak']:5.2f} of peak {names}")
        if "uniform_marg_us" in r:
            line += (f" | uniform {r['uniform_marg_us']:8.1f} us {r['uniform_marg_gbs']:6.0f} GB/s {r['uniform_kernels']}"
                     f" ragged/uniform {r['ragged_over_uniform']:.3f}")
        line += (f" | call {r['call_us']:8.1f} us, tokens {r['tokens_call_us']:8.1f} us (x{r['call_over_tokens']:.2f}),"
                 f" per-image loop {r['loop_call_us']:9.1f} us (x{r['loop_over_call']:.1f} of the call)")
        print(line, flush=True)
        del batches
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
