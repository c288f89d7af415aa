#!/usr/bin/env python
"""bench.py -- warped images/s of the attention-guided warp hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c3|c4|c5] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input:
  c2 (default; BASELINE.json configs[1]): 256 x 336^2 RGB uint8 + bf16 attention
      [256, 32, 32, 576]  -> stage 1 aggregation -> 24x24 token map -> marginals / CDF /
      inverse-CDF maps -> bilinear resample (cv2.remap semantics) to 336^2.
  c3 (configs[2]): 64 x 1344^2 RGB uint8 + 48x48 token maps -> maps -> resample.
  c4 (configs[3]): 1024 mixed-resolution images, LPT-sharded over the ranks (strong scaling), ragged launches.
  c5 (configs[4]): 128 x 3 x 512^2 float32 images + PDFs [128,24] x 2 -> fused PDF->CDF -> maps -> resample.
For N > 1 (launched under torchrun, one rank per GPU) every rank processes its own batch
(weak scaling, images sharded by index, no data-path collective); NCCL only gathers timings and
checksums.  Rank 0 prints ONE JSON line.

`value`  : whole-job images/s, inputs resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : the same metric through the host-buffer pipeline (pinned host -> H2D -> kernels -> D2H).
`roofline`: the dominant kernel's algorithmic bytes / its CUDA-event duration vs the measured
            HBM copy peak (MEASURED_PEAKS.json).
`cpu_baseline`: the oracle port of the reference CPU path on this box's host cores (bounded sample).
`--impl reference`: only the CPU arm, same metric/config, `"impl": "reference"`.
`--dump-outputs DIR`: after the timed steps, rank 0 writes what the last timed step of each workload returned to
            its caller as DIR/<workload>_<array>.npy (float32; a fixed, seeded sample of the elements of an array
            larger than DUMP_ELEMENTS).  Inputs are seeded, so two builds can be compared output for output.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "warped_images_per_sec"
UNIT = "images/s"

WORKLOADS = {
    "c2": dict(name="c2: LLaVA-1.5 batch 256x336^2 RGB u8 + bf16 attention [256,32,32,576] "
                    "aggregation + 24x24 token map -> inverse-CDF warp -> 336^2",
               B=256, L=32, Hh=32, grid=24, side=336, C=3, has_attention=True),
    "c3": dict(name="c3: Qwen-VL-style batch 64x1344^2 RGB u8 + 48x48 token map upsample + "
                    "inverse-CDF warp -> 1344^2",
               B=64, L=0, Hh=0, grid=48, side=1344, C=3, has_attention=False),
    "c4": dict(name="c4: mixed-resolution batch of 1024 RGB u8 images (sides uniform in [224, 2048]) + 24x24 "
                    "token maps -> inverse-CDF warp at input size, ragged launches, LPT-sharded over the GPUs",
               B=1024, L=0, Hh=0, grid=24, side=0, C=3, has_attention=False, ragged=True),
    "c5": dict(name="c5: MarginalNet-style PDFs (2 x [128,24], softmax of seeded logits, alpha=0.1) -> fused "
                    "PDF->CDF + inverse-CDF maps + float32 resample of 128x3x512^2 images (NCHW)",
               B=128, L=0, Hh=0, grid=24, side=512, C=3, has_attention=False, pdf=True),
}


class _StdoutToStderr:
    """OS-level redirect of fd 1 to fd 2 while libraries that printf() to stdout initialise (NCCL prints its
    version banner with a raw printf at NCCL_DEBUG=VERSION): stdout must carry the ONE JSON line only."""

    def __enter__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        os.close(self.saved)
        return False


def init_nccl(dev):
    import torch.distributed as dist
    with _StdoutToStderr():
        dist.init_process_group("nccl", device_id=dev)
        dist.barrier()                       # communicator creation (and its banner) happens here at the latest


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured copy, burst)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md; MEASURED_PEAKS.json absent)"


def ncu_traffic(kernel, workload):
    """Per-launch DRAM bytes of `kernel` from the committed ncu capture, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload, {}).get(kernel)
    except Exception:
        return None


# ------------------------------------------------------------------------------------------
# --dump-outputs
# ------------------------------------------------------------------------------------------
DUMP_ELEMENTS = 4_000_000          # per array: 16 MB of float32; a run of all workloads writes < 64 MB
DUMP_BYTES_MAX = 64 * 10**6


def dump_sample(tensors, n=DUMP_ELEMENTS, seed=0):
    """float32 host copy of the elements of `tensors` (flattened and concatenated in order): all of them when
    there are at most n, else n of them at sorted positions drawn with a fixed seed (the same positions in every
    run of the same workload, whatever the build)."""
    import numpy as np
    import torch
    sizes = [t.numel() for t in tensors]
    total = sum(sizes)
    if total <= n:
        return torch.cat([t.reshape(-1).float() for t in tensors]).cpu().numpy()
    idx = np.sort(np.random.default_rng(seed).integers(0, total, n))
    starts = np.cumsum([0] + sizes)
    parts = []
    for t, lo, hi, start in zip(tensors, np.searchsorted(idx, starts[:-1]), np.searchsorted(idx, starts[1:]),
                                starts[:-1]):
        if hi > lo:
            parts.append(t.reshape(-1)[torch.from_numpy(idx[lo:hi] - start).to(t.device)].float())
    return torch.cat(parts).cpu().numpy()


def write_dumps(path, dumps):
    """dumps: {workload: {array name: float32 ndarray}} -> path/<workload>_<array>.npy"""
    import numpy as np
    total = sum(a.nbytes for d in dumps.values() for a in d.values())
    if total > DUMP_BYTES_MAX:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed {DUMP_BYTES_MAX}")
    os.makedirs(path, exist_ok=True)
    for wl_key, d in dumps.items():
        for name, a in d.items():
            np.save(os.path.join(path, f"{wl_key}_{name}.npy"), a)


# ------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------
def _gpu_uuid(index):
    try:
        import torch
        return str(torch.cuda.get_device_properties(index).uuid)
    except Exception:
        return None


class ClockSampler:
    """SM clock and clock-event (throttle) reasons DURING the timed region.  The region is a few
    milliseconds long, so the sampler is an NVML polling thread (a sample every ~0.2 ms; every NVML
    call releases the GIL); `nvidia-smi -lms` (50 ms period) is the fallback when NVML cannot be loaded."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index, uuid=None):
        self.proc = None
        self.path = None
        self.gpu_index = gpu_index
        self.uuid = uuid
        self.thread = None
        self.samples = []
        self._stop = False
        self.nvml = None
        self.handle = None

    def _nvml_init(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if self.uuid:
                for cand in (self.uuid, "GPU-" + self.uuid):
                    try:
                        h = pynvml.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                        break
                    except Exception:
                        h = None
            if h is None:
                idx = self.gpu_index
                vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
                try:
                    if vis:
                        idx = int(vis.split(",")[self.gpu_index])
                except Exception:
                    pass
                h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.nvml, self.handle = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            return True
        except Exception:
            self.nvml = None
            return False

    def _poll(self):
        nv, h = self.nvml, self.handle
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons", None)
        while not self._stop:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                bits = int(get_reasons(h)) if get_reasons else 0
                self.samples.append((mhz, bits))
            except Exception:
                pass
            time.sleep(0.0002)

    def start(self):
        if self._nvml_init():
            import threading
            # the main thread enqueues steps in a tight Python loop: with the default 5 ms GIL switch interval
            # the polling thread would get one sample per 5 ms
            self._switch = sys.getswitchinterval()
            sys.setswitchinterval(1e-4)
            self._stop = False
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-i", str(self.gpu_index), "-lms", "50"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=2)
            sys.setswitchinterval(self._switch)
            nv = self.nvml
            table = {}
            for nm, attrs in (("hw_slowdown", ("nvmlClocksEventReasonHwSlowdown", "nvmlClocksThrottleReasonHwSlowdown")),
                              ("hw_thermal_slowdown", ("nvmlClocksEventReasonHwThermalSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown")),
                              ("sw_thermal_slowdown", ("nvmlClocksEventReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwThermalSlowdown")),
                              ("sw_power_cap", ("nvmlClocksEventReasonSwPowerCap", "nvmlClocksThrottleReasonSwPowerCap"))):
                for a in attrs:
                    if hasattr(nv, a):
                        table[nm] = int(getattr(nv, a))
                        break
            if not self.samples:
                return None
            sm = sorted(s[0] for s in self.samples)
            reasons = sorted(nm for nm, bit in table.items() if any(s[1] & bit for s in self.samples))
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(sm), "how": "NVML polled during the timed region"}
        if self.proc is None:
            return None
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for k, nm in enumerate(names):
                    if f[5 + k].lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return None
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons),
                "samples": len(sm), "how": "nvidia-smi -lms 50 during the timed region"}



# ------------------------------------------------------------------------------------------
# workload descriptions (identical in both arms: `config` is a function of the workload and the world size)
# ------------------------------------------------------------------------------------------
def workload_config(wl_key, world):
    wl = WORKLOADS[wl_key]
    B, side, C = wl["B"], wl["side"], wl["C"]
    if wl.get("ragged"):
        return {"workload": wl["name"], "images_total": B, "transform": "identity",
                "l2_policy": "inputs larger than L2: a rank's shard is >= 1.2 GB in + as much out (126 MB L2)",
                "parallelism": f"one batch of {B} images LPT-sharded by pixels in + out over {world} GPU(s) "
                               "(strong scaling), no data-path collective"}
    if wl.get("pdf"):
        by = B * C * side * side * 4 * 2
        return {"workload": wl["name"], "images_per_step_per_gpu": B, "transform": "n/a (PDFs in)",
                "l2_policy": f"inputs larger than L2: one batch is {by / 1e6:.0f} MB in+out > 126 MB L2; the GPU arm "
                             "rotates over resident buffer sets",
                "parallelism": f"images sharded by index over {world} GPU(s) (weak scaling), no data-path collective"}
    by = B * side * side * C * 2 + (B * wl["L"] * wl["Hh"] * wl["grid"] ** 2 * 2 if wl["has_attention"] else 0)
    return {"workload": wl["name"], "images_per_step_per_gpu": B, "transform": "identity",
            "l2_policy": f"inputs larger than L2: one batch ({'attention + ' if wl['has_attention'] else ''}images in + out) "
                         f"is {by / 1e6:.0f} MB > 126 MB L2; the GPU arm rotates over resident buffer sets",
            "parallelism": f"images sharded by index over {world} GPU(s) (weak scaling: every rank its own batch), "
                           "no data-path collective"}


# ------------------------------------------------------------------------------------------
# CPU arm (the reference's own CPU path: unmodified reference from baseline/_ref when present, else the oracle port)
# ------------------------------------------------------------------------------------------
def cpu_arm(wl_key, steps, warmup, budget_s, rows=False):
    """Times the reference CPU path on the host cores.  Each step = one pass over a bounded sample of
    the workload (the full batch when it is cheap enough)."""
    from oracle import cpu_baseline as CB
    wl = WORKLOADS[wl_key]
    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # calibrate on a few images, single process
    if wl["has_attention"]:
        attn, imgs = CB.make_c2_sample(4, wl["L"], wl["Hh"], wl["grid"], wl["side"])
        tok = None
    else:
        tok, imgs = CB.make_c3_sample(4, wl["grid"], wl["side"])
        attn = None
    r = CB.CpuRunner(attn, tok, imgs, wl["grid"], (wl["side"], wl["side"]), workers=1)
    kind = r.kind
    thread_rows = r.threading_rows(4, 2) if rows else None
    r.step()
    t1, _ = r.step()
    per_img = t1 / 4
    r.close()
    total_steps = steps + warmup
    # images per step so that the whole run fits the budget (assume ~70 % parallel efficiency)
    n = int(budget_s / max(total_steps, 1) / per_img * avail * 0.7)
    n = max(min(n, wl["B"]), min(avail, wl["B"]), 1)
    if wl["has_attention"]:
        attn, imgs = CB.make_c2_sample(n, wl["L"], wl["Hh"], wl["grid"], wl["side"])
    else:
        tok, imgs = CB.make_c3_sample(n, wl["grid"], wl["side"])
    runner = CB.CpuRunner(attn, tok, imgs, wl["grid"], (wl["side"], wl["side"]))
    for _ in range(warmup):
        runner.step()
    t = 0.0
    for _ in range(steps):
        dt, _ = runner.step()
        t += dt
    runner.close()
    value = n * steps / t
    import cv2
    import numpy
    what = ("the UNMODIFIED reference functions (MaskHookLogger._process_attention/finalize, set_transform_function, "
            "warp_image_by_attention) imported from baseline/_ref" if kind == "reference"
            else "the oracle port (no copy of the reference present)")
    info = {"value": value, "unit": UNIT, "cores": runner.workers, "kind": kind,
            "sample": f"{n} of {wl['B']} images per step x {steps} steps ({warmup} warm-up); {what}; "
                      f"{runner.workers} fork()ed workers x 1 image at a time, cv2.setNumThreads(1), torch 1 thread; "
                      f"single-process cost {per_img * 1e3:.2f} ms/image; numpy {numpy.__version__}, "
                      f"cv2 {cv2.__version__}; host cpus visible {avail}"}
    if thread_rows is not None:
        info["rows"] = thread_rows
    return info, t / steps * 1e3


def run_reference(args, rank, world):
    if rank != 0:
        return 0
    key = "c2" if args.workload == "all" else args.workload
    wl = WORKLOADS[key]
    if wl.get("ragged") or wl.get("pdf"):
        print(json.dumps({"impl": "reference", "unavailable": "the CPU arm covers the bench workloads c2 and c3; "
                          "c4 and c5 are parity/scaling configurations"}), flush=True)
        return 0
    info, ms_per_step = cpu_arm(key, args.steps, args.warmup, budget_s=100.0 if args.workload == "all" else 120.0,
                                rows=True)
    line = {"impl": "reference", "metric": METRIC, "value": info["value"], "unit": UNIT,
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": DTYPES[key], "data": "synthetic",
            "config": workload_config(key, world),
            "run": {"timing": "wall clock around each CPU step", "arm": "reference CPU path on the host cores"},
            "cpu_baseline": info,
            "e2e": {"value": info["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                    "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    if args.workload == "all":
        # 1344^2 (configs[2]) on the same host cores, a smaller sample
        i3, ms3 = cpu_arm("c3", max(2, min(args.steps, 3)), 1, budget_s=40.0)
        line["workloads"] = {"c3": {"metric": METRIC, "value": i3["value"], "unit": UNIT, "ms_per_step": ms3,
                                    "config": workload_config("c3", world), "cpu_baseline": i3,
                                    "e2e": {"value": i3["value"], "unit": UNIT, "h2d_bytes_per_step": 0,
                                            "d2h_bytes_per_step": 0}}}
    print(json.dumps(line), flush=True)
    return 0


DTYPES = {"c2": "bf16->fp32 (stage 1), f64 (stages 2-4), u8 fixed-point (stage 5)",
          "c3": "f64 (stages 2-4), u8 fixed-point (stage 5)",
          "c4": "f64 (stages 2-4), u8 fixed-point (stage 5)",
          "c5": "f32 (PDF/CDF rows), f64 (inversion), f32 (resample)"}


# ------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, rank, local_rank, world):
        import torch
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        if world > 1:
            init_nccl(self.dev)
        self.peak, self.peak_src = measured_peak()

    def barrier(self):
        import torch
        import torch.distributed as dist
        torch.cuda.synchronize()
        if self.world > 1:
            dist.barrier()
        torch.cuda.synchronize()


def timed_steps(ctx, step, n_steps, first_index, fork=None, join=None):
    """barrier + synchronize, CUDA events around exactly n_steps calls of step(i), synchronize + barrier.
    Returns (elapsed ms on this rank, launches)."""
    import torch
    ctx.barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches = 0
    ev0.record()
    if fork is not None:
        fork()                                    # every ring stream starts after ev0 ...
    for i in range(n_steps):
        launches += step(first_index + i)
    if join is not None:
        join()                                    # ... and ev1 waits for all of them
    ev1.record()
    ctx.barrier()
    return ev0.elapsed_time(ev1), launches


def pick_roofline(ctx, kernels, workload, total_bytes):
    """`roofline` = the kernel that dominates the step; when two kernels are within 15 % of each other in time
    (a margin wider than the 10 % box-to-box spread of the two c2 kernels, so that the choice does not flip between
    runs), the one FURTHER from the peak.  `worst` = the kernel furthest below peak of all, `worst_streaming` = among the
    kernels that move >= 5 % of the step's bytes (the others are latency-bound: a few KB per image)."""
    streaming = {k: v for k, v in kernels.items() if v["algorithmic_bytes"] >= 0.05 * total_bytes}
    dom_ms = max(v["ms"] for v in streaming.values())
    cands = [k for k, v in streaming.items() if v["ms"] >= 0.85 * dom_ms]
    dom = min(cands, key=lambda k: kernels[k]["frac"])
    worst = min(kernels, key=lambda k: kernels[k]["frac"])
    worst_s = min(streaming, key=lambda k: kernels[k]["frac"])
    return {"bound": "hbm", "kernel": dom, "achieved": kernels[dom]["achieved_gbs"], "peak": ctx.peak,
            "unit": "GB/s", "frac": kernels[dom]["frac"], "traffic": ncu_traffic(dom, workload),
            "peak_source": ctx.peak_src, "algorithmic_bytes_per_launch": kernels[dom]["algorithmic_bytes"],
            "kernel_ms": kernels[dom]["ms"],
            "selection": "dominant kernel by CUDA-event time; of kernels within 15 % in time, the lower fraction",
            "worst": {"kernel": worst, "frac": kernels[worst]["frac"], "achieved": kernels[worst]["achieved_gbs"],
                      "note": "latency-bound launch (a few KB per image)" if worst not in streaming else "streaming kernel"},
            "worst_streaming": {"kernel": worst_s, "frac": kernels[worst_s]["frac"],
                                "achieved": kernels[worst_s]["achieved_gbs"]}}


def bench_uniform(ctx, wl_key, with_clocks=True):
    """configs[1] / configs[2]: uniform batches, every rank its own batch (weak scaling)."""
    import torch

    from attwarp_b200 import _lib, ops, sharding
    from attwarp_b200.batched import HostBatchPipeline, HostCopyProbe, HostTokenPipeline, StreamRing

    args, dev, world, rank = ctx.args, ctx.dev, ctx.world, ctx.rank
    wl = WORKLOADS[wl_key]
    B, side, C, grid = wl["B"], wl["side"], wl["C"], wl["grid"]
    L, Hh, T = wl["L"], wl["Hh"], wl["grid"] ** 2
    R = args.rotate if args.rotate > 0 else (8 if wl["has_attention"] else 4)
    gen = torch.Generator(device=dev).manual_seed(1235 + rank + (0 if wl["has_attention"] else 7919))
    sets = []
    for _ in range(R):
        s = {}
        if wl["has_attention"]:
            chunks = []
            for lo in range(0, B, 64):                 # bounded fp32 temporaries
                z = torch.randn(min(64, B - lo), L, Hh, T, device=dev, generator=gen) * 2
                chunks.append(torch.softmax(z, -1).to(torch.bfloat16))
            s["attn"] = torch.cat(chunks)
            del chunks, z
        else:
            tok = torch.rand(B, grid, grid, device=dev, generator=gen) ** 3
            s["tok"] = (tok / tok.sum(dim=(1, 2), keepdim=True)).contiguous()
        s["img"] = torch.randint(0, 256, (B, side, side, C), device=dev, dtype=torch.uint8, generator=gen)
        s["out"] = torch.empty(B, side, side, C, device=dev, dtype=torch.uint8)
        s["aux"] = (torch.empty(B, T, device=dev), torch.empty(B, side, device=dev),
                    torch.empty(B, side, device=dev))
        sets.append(s)
    side_hw = (side, side)

    def enqueue(s, evs=None):
        """One step on buffer set `s`: every kernel of the hot path, on the current stream."""
        if wl["has_attention"]:
            ops.warp_from_attention_tokens(s["attn"], s["img"], (grid, grid), None, "hwc",
                                           transform="identity", out=s["out"], aux=s["aux"],
                                           stage_events=evs)
            return 3
        mx, my = s["aux"][1], s["aux"][2]
        ops.maps_from_tokens(s["tok"], side_hw, None, "identity", out=(mx, my))
        ops.remap_bilinear(s["img"], mx, my, "hwc", out=s["out"])
        return 2

    # Consecutive steps are independent batches: they go round-robin over a few streams so that the
    # HBM-bound stage 1 of one step shares the GPU with the issue-bound stage 5 of the previous one.
    n_streams = args.streams if args.streams > 0 else (4 if wl["has_attention"] else 3)
    n_streams = max(1, min(n_streams, R))        # concurrent steps need distinct buffer sets
    ring = StreamRing(n_streams, dev) if n_streams > 1 else None
    # ... and for them to be CO-RESIDENT on an SM each launch may fill only half of it (attwarp_set_sm_share; the
    # grid size is part of a captured graph, so the graphs of the overlapped steps are captured in that mode)
    lib = _lib.load()
    sm_share = args.sm_share if args.sm_share > 0 else (2 if (wl["has_attention"] and ring is not None) else 1)

    # one CUDA graph per resident buffer set: a step is ONE driver launch of its 2-3 kernels
    launches_per_step = 3 if wl["has_attention"] else 2
    graphs = graphs_single = None
    if not args.no_graph:
        prev_share = lib.attwarp_set_sm_share(sm_share)
        graphs = [ops.GraphedCall(lambda s=s: enqueue(s), device=dev) for s in sets]
        lib.attwarp_set_sm_share(prev_share)
        # the single-stream figure runs graphs captured with whole-SM launches
        graphs_single = graphs if sm_share == 1 else [ops.GraphedCall(lambda s=s: enqueue(s), device=dev) for s in sets[:3]]

    def run_step(i):
        if graphs is not None:
            graphs[i % R].replay()
        else:
            enqueue(sets[i % R])

    def run_step_single(i):
        if graphs_single is not None:
            graphs_single[i % len(graphs_single)].replay()
        else:
            enqueue(sets[i % R])

    def step(i):
        if ring is not None:
            ring.submit(lambda: run_step(i))
        else:
            run_step(i)
        return launches_per_step

    fork = ring.fork if ring is not None else None
    join = ring.join if ring is not None else None
    if args.no_graph and sm_share > 1:
        lib.attwarp_set_sm_share(sm_share)             # eager launches read the mode at every launch
    if fork:
        fork()
    for i in range(args.warmup):
        step(i)
    if join:
        join()
    torch.cuda.synchronize()

    sampler = ClockSampler(ctx.local_rank, _gpu_uuid(ctx.local_rank))
    if rank == 0 and with_clocks:
        sampler.start()
    elapsed_ms, launches = timed_steps(ctx, step, args.steps, args.warmup, fork, join)
    clocks = sampler.stop() if (rank == 0 and with_clocks) else None
    lib.attwarp_set_sm_share(1)

    last = sets[(args.warmup + args.steps - 1) % R]
    dump = None
    if args.dump_outputs and rank == 0:
        dump = {"out": dump_sample([last["out"]])}
        if wl["has_attention"]:
            dump["tokens"] = dump_sample([last["aux"][0]])
        dump.update(map_x=dump_sample([last["aux"][1]]), map_y=dump_sample([last["aux"][2]]))
    chk = sharding.checksum64(last["out"][:8])
    stats = sharding.gather_stats(elapsed_ms, B * args.steps, chk, dev)
    value = sharding.aggregate_throughput(stats)
    worst_ms = max(s[0] for s in stats)

    # single-stream figure (one batch at a time: nothing of another step to overlap with)
    one_ms, _ = timed_steps(ctx, lambda i: (run_step_single(i), launches_per_step)[1], args.steps, 0)
    one_stats = sharding.gather_stats(one_ms, B * args.steps, 0, dev)

    # ---- per-kernel durations, outside the timed region ---------------------------------------------
    # each kernel alone, launched back to back over the rotating sets (the launch of kernel n+1 overlaps
    # kernel n, so events around the whole run / N is the kernel duration, fill and drain included)
    kernels = {}
    kreps = max(10, min(args.steps, 30))

    def back_to_back(fn):
        # one CUDA graph holding a pass over the resident sets (eager launches through ctypes cost ~10 us of host
        # time each: a 12 us kernel would be timed at the host's enqueue rate, not the device's)
        n_sets = min(R, 4)
        if args.no_graph:
            run = lambda: [fn(sets[i]) for i in range(n_sets)]            # noqa: E731
        else:
            g = ops.GraphedCall(lambda: [fn(sets[i]) for i in range(n_sets)], device=dev)
            run = g.replay
        passes = (kreps + n_sets - 1) // n_sets
        run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(passes):
            run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (passes * n_sets)

    how = f">= {kreps} back-to-back launches over the rotating sets" + ("" if args.no_graph else " (graph replay)")

    def add(name, ms, by, extra=None):
        kernels[name] = {"ms": ms, "algorithmic_bytes": by, "achieved_gbs": by / ms / 1e6,
                         "frac": by / ms / 1e6 / ctx.peak, "how": how}
        if extra:
            kernels[name].update(extra)

    if wl["has_attention"]:
        add("aggregate_rows_tma_kernel", back_to_back(lambda s: ops.aggregate_attention(s["attn"], out=s["aux"][0])),
            B * (L * Hh * T * 2 + T * 4), {"note": "includes its 4 us finalize launch"})
        tokmap = lambda s: s["aux"][0].view(B, grid, grid)          # noqa: E731
    else:
        tokmap = lambda s: s["tok"]                                  # noqa: E731
    add("maps_from_tokens_kernel",
        back_to_back(lambda s: ops.maps_from_tokens(tokmap(s), side_hw, None, "identity", out=(s["aux"][1], s["aux"][2]))),
        B * (T * 4 + 2 * side * 4))
    add("remap_u8_quad_kernel",
        back_to_back(lambda s: ops.remap_bilinear(s["img"], s["aux"][1], s["aux"][2], "hwc", out=s["out"])),
        B * side * side * C * 2)
    step_bytes = sum(k["algorithmic_bytes"] for k in kernels.values())
    roofline = pick_roofline(ctx, kernels, wl_key, step_bytes)
    roofline["whole_step"] = {"algorithmic_bytes": step_bytes,
                              "achieved": step_bytes / (worst_ms / args.steps) / 1e6,
                              "frac": step_bytes / (worst_ms / args.steps) / 1e6 / ctx.peak,
                              "note": f"all kernels of a step, {n_streams} steps in flight"}

    # ---- the reference drivers' flow at this size (a labelled extra, not the headline): token map -> revise_mask ->
    # Pillow-exact LANCZOS mask at image size + its marginals (one kernel, vertical pass on the tensor cores, the mask
    # never written) -> maps -> stage 5; "Attention Guided Warping/main.py":361 -> 520.  Device-resident, graph replay.
    driver_flow = None
    try:
        ms_maps = back_to_back(lambda s: ops.maps_from_mota_tokens(tokmap(s), side_hw))

        def flow_step(s):
            mx_, my_ = ops.maps_from_mota_tokens(tokmap(s), side_hw)
            ops.remap_bilinear(s["img"], mx_, my_, "hwc", out=s["out"])
        ms_flow = back_to_back(flow_step)
        driver_flow = {"what": "tokens -> revise_mask -> LANCZOS mask + marginals (fused) -> maps -> resample, "
                               "one batch at a time on one stream",
                       "maps_from_mota_tokens_ms": ms_maps, "step_ms": ms_flow, "images_per_s": B / ms_flow * 1e3,
                       "how": how}
    except Exception as e:                                   # an extra must never cost the headline
        driver_flow = {"error": repr(e)[:200]}

    # ---- e2e: pinned host buffers -> H2D -> kernels -> D2H, per step -----------------------------
    e2e = None
    if not args.no_e2e:
        h_img = torch.empty(B, side, side, C, dtype=torch.uint8).pin_memory()
        h_out = torch.empty(B, side, side, C, dtype=torch.uint8).pin_memory()
        h_img.copy_(sets[0]["img"])
        chunk = args.e2e_chunk if args.e2e_chunk > 0 else (64 if wl["has_attention"] else 16)
        if wl["has_attention"]:
            h_in = torch.empty(B, L, Hh, T, dtype=torch.bfloat16).pin_memory()
            h_in.copy_(sets[0]["attn"])
            pipe = HostBatchPipeline(chunk, L, Hh, (grid, grid), (side, side, C), device=dev)
            api = "attwarp_b200.batched.HostBatchPipeline.run (pinned host in/out)"
        else:
            h_in = torch.empty(B, grid, grid, dtype=torch.float32).pin_memory()
            h_in.copy_(sets[0]["tok"])
            pipe = HostTokenPipeline(chunk, (grid, grid), (side, side, C), device=dev)
            api = "attwarp_b200.batched.HostTokenPipeline.run (pinned host in/out)"
        probe = HostCopyProbe(pipe)
        ke = args.steps

        def time_e2e(fn):
            for _ in range(2):
                fn()
            ms, _ = timed_steps(ctx, lambda i: (fn(), 0)[1], ke, 0)
            return ms

        ems = time_e2e(lambda: pipe.run(h_in, h_img, h_out))
        est = sharding.gather_stats(ems, B * ke, int(h_out[:4].to(torch.int64).sum()), dev)
        cms = time_e2e(lambda: probe.run((h_in, h_img), h_out))
        cst = sharding.gather_stats(cms, B * ke, 0, dev)
        e2e_ms, copy_ms = max(s[0] for s in est) / ke, max(s[0] for s in cst) / ke
        e2e = {"value": sharding.aggregate_throughput(est), "unit": UNIT,
               "h2d_bytes_per_step": h_in.numel() * h_in.element_size() + h_img.numel(),
               "d2h_bytes_per_step": h_out.numel(), "steps": ke, "chunk": chunk,
               "ms_per_step": e2e_ms, "api": api,
               "copy_only_ms_per_step": copy_ms, "frac_of_copy_ceiling": copy_ms / e2e_ms,
               "copy_only_note": "the same chunks, bytes, streams and pinned buffers without the kernels, all ranks "
                                 "copying at the same time: what PCIe + host memory deliver on this box at this N",
               "pcie_gbs_per_gpu": {"h2d": (h_in.numel() * h_in.element_size() + h_img.numel()) / e2e_ms / 1e6,
                                    "d2h": h_out.numel() / e2e_ms / 1e6}}
        if wl["has_attention"]:
            # second variant, labelled: in the real pipeline the attention tensor is born on the GPU (it is the
            # output of the model's attention layer); only the images cross PCIe
            d_attn = sets[0]["attn"]
            tpipe = HostBatchPipeline(chunk, L, Hh, (grid, grid), (side, side, C), device=dev)

            def run_resident():
                caller = torch.cuda.current_stream(dev)
                for s_ in tpipe.streams:
                    s_.wait_stream(caller)
                k = 0
                for lo in range(0, B, chunk):
                    hi = min(lo + chunk, B)
                    slot, st = tpipe.slots[k % 2], tpipe.streams[k % 2]
                    with torch.cuda.stream(st):
                        slot["img"][:hi - lo].copy_(h_img[lo:hi], non_blocking=True)
                        ops.warp_from_attention_tokens(d_attn[lo:hi], slot["img"][:hi - lo], (grid, grid), None, "hwc",
                                                       transform="identity", out=slot["out"][:hi - lo],
                                                       aux=tuple(a[:hi - lo] for a in slot["aux"]))
                        h_out[lo:hi].copy_(slot["out"][:hi - lo], non_blocking=True)
                    k += 1
                for s_ in tpipe.streams:
                    caller.wait_stream(s_)

            rms = time_e2e(run_resident)
            rst = sharding.gather_stats(rms, B * ke, 0, dev)
            e2e["attention_device_resident"] = {
                "value": sharding.aggregate_throughput(rst), "unit": UNIT, "ms_per_step": max(s[0] for s in rst) / ke,
                "h2d_bytes_per_step": h_img.numel(), "d2h_bytes_per_step": h_out.numel(),
                "note": "NOT the headline e2e: attention already in HBM (as inside a real generate()), images only over PCIe"}
            del tpipe
        del pipe, probe, h_in, h_img, h_out

    res = {"value": value, "ms_per_step": worst_ms / args.steps, "per_rank_ms": [s[0] for s in stats],
           "launches": launches * world, "kernels": kernels, "roofline": roofline, "e2e": e2e, "clocks": clocks,
           "driver_flow": driver_flow, "dump": dump,
           "single_stream": {"ms_per_step": max(s[0] for s in one_stats) / args.steps,
                             "value": sharding.aggregate_throughput(one_stats),
                             "note": "one batch at a time on one stream (no overlap between steps)"},
           "run": {"rotate": R, "streams": n_streams, "sm_share": sm_share,
                   "launch": ("one CUDA graph replay per step" if graphs is not None else "eager launches") +
                             (f"; consecutive steps round-robin over {n_streams} CUDA streams (independent batches: "
                              "the early stages of one step overlap stage 5 of the previous one)" if ring is not None else "") +
                             ("; every launch of stage 1 / stage 5 fills half of each SM so that two steps are co-resident "
                              "(attwarp_set_sm_share(2)); the single-stream figure and the per-kernel timings use whole-SM "
                              "launches" if sm_share > 1 else "")}}
    del sets, graphs, graphs_single
    torch.cuda.empty_cache()
    return res


def c4_image(i, side, C, dev, gen):
    """Image i of the configs[3] batch: the same bytes whichever rank generates it."""
    import torch
    gen.manual_seed(1237 * 1000003 + int(i))
    return torch.randint(0, 256, (int(side), int(side), C), device=dev, dtype=torch.uint8, generator=gen)


def bench_ragged(ctx):
    """configs[3]: ONE batch of 1024 mixed-resolution images split over the ranks by greedy LPT on
    pixels in + pixels out (strong scaling, no data-path collective); a step = stages 2-5 over the
    rank's shard through the ragged entry point (one launch per stage).  After the timed region the per-image
    checksums of all ranks are merged and compared with an UNSHARDED pass over the whole batch."""
    import numpy as np
    import torch

    from attwarp_b200 import multi_gpu, ops, sharding

    args, dev, world, rank = ctx.args, ctx.dev, ctx.world, ctx.rank
    wl = WORKLOADS["c4"]
    B, C, grid = wl["B"], wl["C"], wl["grid"]
    steps = args.steps if args.c4_steps <= 0 else args.c4_steps
    sides = np.random.default_rng(1237).integers(224, 2049, size=B)
    sizes = [(int(s), int(s)) for s in sides]
    plan = multi_gpu.plan_ragged(sizes, world=world)
    mine = plan.shards[rank]
    gen = torch.Generator(device=dev)
    imgs = [c4_image(i, sides[i], C, dev, gen) for i in mine]
    outs = [torch.empty_like(t) for t in imgs]
    tok_all = torch.rand(B, grid, grid, generator=torch.Generator().manual_seed(1237)) ** 3
    tok_all = (tok_all / tok_all.sum(dim=(1, 2), keepdim=True)).contiguous()
    tok = tok_all[torch.as_tensor(mine)].to(dev)
    my_bytes = 2 * sum(t.numel() for t in imgs)

    # the descriptor table is a function of the buffers: built once (ops.RaggedBatch), re-used by every step
    batch = ops.RaggedBatch(imgs, outs=outs)

    def step(i):
        batch.run(tok)
        return batch.launches                    # maps + one resample launch per class (counted by the library)

    step(0)
    launches_per_step = batch.launches

    for i in range(args.warmup):
        step(i)
    elapsed_ms, launches = timed_steps(ctx, step, steps, 0)
    dump = {"out": dump_sample(outs)} if args.dump_outputs and rank == 0 else None
    stats = sharding.gather_stats(elapsed_ms, len(mine) * steps, 0, dev)
    bstats = sharding.gather_stats(elapsed_ms, my_bytes // 1024, 0, dev)
    value = sharding.aggregate_throughput(stats)
    worst_ms = max(s[0] for s in stats)

    # ---- sharded == unsharded -------------------------------------------------------------------
    table = multi_gpu.gather_image_checksums(plan, mine, outs)
    check = {"images_checked": 0}
    if rank == 0:
        if world > 1:
            del imgs, outs, batch
            torch.cuda.empty_cache()
            whole_in = [c4_image(i, sides[i], C, dev, gen) for i in range(B)]
            whole = ops.warp_ragged_from_tokens(tok_all.to(dev), whole_in)
            ref = torch.tensor([sharding.checksum64(o) for o in whole], dtype=torch.int64)
            how = f"rank 0 re-ran the whole batch in one unsharded launch and compared {B} per-image checksums"
        else:
            # one rank: compare against the two shards of a 2-way LPT plan run one after the other
            plan2 = multi_gpu.plan_ragged(sizes, world=2)
            ref = torch.zeros(B, dtype=torch.int64)
            for r in range(2):
                idx = plan2.shards[r]
                o2 = ops.warp_ragged_from_tokens(tok_all[torch.as_tensor(idx)].to(dev), [imgs[i] for i in idx])
                for i, o in zip(idx, o2):
                    ref[i] = sharding.checksum64(o)
                del o2
            how = "one rank: its single launch compared with the two shards of a 2-way LPT plan run in turn"
        same = bool(torch.equal(ref.cpu(), table.cpu()))
        if not same:
            bad = (ref.cpu() != table.cpu()).nonzero().flatten().tolist()[:8]
            raise RuntimeError(f"c4: sharded and unsharded results differ for images {bad}")
        check = {"images_checked": B, "sharded_equals_unsharded": same, "how": how}
    ctx.barrier()
    total_bytes = sum(b[1] for b in bstats) * 1024
    gbs = total_bytes / (worst_ms / steps) / 1e6 / world
    loads = plan.load()
    res = {"value": value, "ms_per_step": worst_ms / steps, "per_rank_ms": [s[0] / steps for s in stats],
           "steps": steps, "launches": launches * world, "images_per_rank": [len(s) for s in plan.shards],
           "shard_imbalance": max(loads) / (sum(loads) / world),
           "roofline": {"bound": "hbm", "kernel": "maps_from_tokens_ragged + remap_u8_quad per width class (whole step)",
                        "achieved": gbs, "peak": ctx.peak, "unit": "GB/s", "frac": gbs / ctx.peak, "traffic": None,
                        "peak_source": ctx.peak_src, "algorithmic_bytes_per_launch": total_bytes // world,
                        "note": "per GPU: the slowest rank's step time over its share of the bytes"},
           "check": check, "e2e": None, "dump": dump,
           "run": {"launch": "one maps launch + one resample launch per class of images (grouped by the consumer warps "
                             "their strips need, 3..16, and by whether their rows are 4-byte aligned; classes fan out "
                             "over three streams) per step over the rank's shard; descriptor table planned once per "
                             "buffer set (ops.RaggedBatch)",
                   "launches_per_step": launches_per_step}}
    torch.cuda.empty_cache()
    return res


def bench_pdf(ctx):
    """configs[4]: predicted PDFs feeding the fused CDF + resample path (trainer.py:212-218, 285-289 chain):
    a step = attwarp_warp_from_pdfs over one batch of 128 float32 NCHW images (three launches)."""
    import torch

    from attwarp_b200 import ops, sharding
    from attwarp_b200.batched import StreamRing

    args, dev, world, rank = ctx.args, ctx.dev, ctx.world, ctx.rank
    wl = WORKLOADS["c5"]
    B, C, side, N = wl["B"], wl["C"], wl["side"], wl["grid"]
    R = args.rotate if args.rotate > 0 else 3
    gen = torch.Generator(device=dev).manual_seed(1238 + rank)
    sets = []
    for _ in range(R):
        sets.append(dict(px=torch.softmax(torch.randn(B, N, device=dev, generator=gen) * 1.5, -1),
                         py=torch.softmax(torch.randn(B, N, device=dev, generator=gen) * 1.5, -1),
                         img=torch.rand(B, C, side, side, device=dev, generator=gen),
                         out=torch.empty(B, C, side, side, device=dev)))

    def enqueue(s):
        ops.warp_from_pdfs(s["img"], s["px"], s["py"], alpha=0.1, layout="chw", out=s["out"])

    graphs = None if args.no_graph else [ops.GraphedCall(lambda s=s: enqueue(s), device=dev) for s in sets]
    n_streams = max(1, min(args.streams if args.streams > 0 else 3, R))
    ring = StreamRing(n_streams, dev) if n_streams > 1 else None

    def run_step(i):
        if graphs is not None:
            graphs[i % R].replay()
        else:
            enqueue(sets[i % R])

    def step(i):
        if ring is not None:
            ring.submit(lambda: run_step(i))
        else:
            run_step(i)
        return 3

    fork = ring.fork if ring is not None else None
    join = ring.join if ring is not None else None
    if fork:
        fork()
    for i in range(args.warmup):
        step(i)
    if join:
        join()
    torch.cuda.synchronize()
    sampler = ClockSampler(ctx.local_rank, _gpu_uuid(ctx.local_rank))
    if rank == 0:
        sampler.start()
    elapsed_ms, launches = timed_steps(ctx, step, args.steps, args.warmup, fork, join)
    clocks = sampler.stop() if rank == 0 else None
    dump = None
    if args.dump_outputs and rank == 0:
        dump = {"out": dump_sample([sets[(args.warmup + args.steps - 1) % R]["out"]])}
    stats = sharding.gather_stats(elapsed_ms, B * args.steps, 0, dev)
    value = sharding.aggregate_throughput(stats)
    worst_ms = max(s[0] for s in stats)
    by = B * C * side * side * 4 * 2
    kreps = max(10, min(args.steps, 30))

    def kernel_ms(mx, my):
        for i in range(3):
            ops.remap_bilinear(sets[i % R]["img"], mx, my, "chw", out=sets[i % R]["out"])
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(kreps):
            ops.remap_bilinear(sets[i % R]["img"], mx, my, "chw", out=sets[i % R]["out"])
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / kreps

    # the resample kernel alone on two families of maps: the PDF maps of the step (softmax PDFs mixed with
    # alpha = 0.1: close to the identity) and the harder maps of rand^3 token grids (strong local scale changes)
    _, _, _, mx, my = ops.warp_from_pdfs(sets[0]["img"], sets[0]["px"], sets[0]["py"], alpha=0.1, layout="chw",
                                         out=sets[0]["out"], return_aux=True)
    tokr = torch.rand(B, N, N, device=dev, generator=gen) ** 3
    hx, hy = ops.maps_from_tokens((tokr / tokr.sum(dim=(1, 2), keepdim=True)).contiguous(), (side, side))
    kms, hms = kernel_ms(mx, my), kernel_ms(hx, hy)
    kernels = {"remap_f32_stream_kernel": {"ms": kms, "algorithmic_bytes": by, "achieved_gbs": by / kms / 1e6,
                                         "frac": by / kms / 1e6 / ctx.peak, "maps": "PDF maps of the step (alpha = 0.1)"},
               "remap_f32_stream_kernel@rand3_token_maps": {"ms": hms, "algorithmic_bytes": by,
                                                          "achieved_gbs": by / hms / 1e6, "frac": by / hms / 1e6 / ctx.peak,
                                                          "maps": "maps of rand^3 24x24 token grids"}}
    hard = max(kernels, key=lambda k: kernels[k]["ms"])
    res = {"value": value, "ms_per_step": worst_ms / args.steps, "per_rank_ms": [s[0] for s in stats],
           "launches": launches * world, "kernels": kernels, "clocks": clocks, "e2e": None, "dump": dump,
           "roofline": {"bound": "hbm", "kernel": "remap_f32_stream_kernel", "achieved": kernels[hard]["achieved_gbs"],
                        "peak": ctx.peak, "unit": "GB/s", "frac": kernels[hard]["frac"],
                        "traffic": ncu_traffic("remap_f32_stream_kernel", "c5"), "peak_source": ctx.peak_src,
                        "algorithmic_bytes_per_launch": by, "kernel_ms": kernels[hard]["ms"],
                        "selection": "the slower of the two map families (" + kernels[hard]["maps"] + ")"},
           "run": {"rotate": R, "streams": n_streams,
                   "launch": ("one CUDA graph replay per step" if graphs is not None else "eager launches") +
                             (f"; consecutive steps round-robin over {n_streams} CUDA streams" if ring is not None else "")}}
    del sets, graphs
    torch.cuda.empty_cache()
    return res


def run_gpu(args, rank, local_rank, world):
    head_key = "c2" if args.workload == "all" else args.workload
    cpu_info = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline and not WORKLOADS[head_key].get("ragged") \
            and not WORKLOADS[head_key].get("pdf"):
        # before CUDA is initialised (the pool forks)
        cpu_info, _ = cpu_arm(head_key, steps=3, warmup=1, budget_s=20.0, rows=True)

    import torch.distributed as dist

    ctx = Ctx(args, rank, local_rank, world)
    wl = WORKLOADS[head_key]
    if wl.get("ragged"):
        head = bench_ragged(ctx)
    elif wl.get("pdf"):
        head = bench_pdf(ctx)
    else:
        head = bench_uniform(ctx, head_key)
    dumps = {head_key: head["dump"]}
    extra = {}
    if args.workload == "all":
        for key in ("c3", "c4"):
            r = bench_uniform(ctx, key, with_clocks=False) if key == "c3" else bench_ragged(ctx)
            dumps[key] = r["dump"]
            entry = {"metric": METRIC, "unit": UNIT, "value": r["value"], "ms_per_step": r["ms_per_step"],
                     "scaling": "strong" if key == "c4" else "weak", "dtype": DTYPES[key],
                     "config": workload_config(key, world), "roofline": r["roofline"], "e2e": r["e2e"],
                     "per_rank_ms": r["per_rank_ms"], "gpu_launches": r["launches"], "run": r["run"]}
            for k in ("kernels", "single_stream", "driver_flow", "images_per_rank", "shard_imbalance", "check", "steps"):
                if k in r:
                    entry[k] = r[k]
            extra[key] = entry
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    if args.dump_outputs:
        write_dumps(args.dump_outputs, dumps)
    line = {"metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world,
            "steps": head.get("steps", args.steps), "warmup": args.warmup, "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "strong" if wl.get("ragged") else "weak", "vs_baseline": None,
            "dtype": DTYPES[head_key], "data": "synthetic", "config": workload_config(head_key, world),
            "run": head["run"], "clocks": head.get("clocks"), "e2e": head["e2e"], "gpu_launches": head["launches"],
            "roofline": head["roofline"], "cpu_baseline": cpu_info, "per_rank_ms": head["per_rank_ms"]}
    for k in ("kernels", "single_stream", "driver_flow", "images_per_rank", "shard_imbalance", "check"):
        if k in head:
            line[k] = head[k]
    if extra:
        line["workloads"] = extra
    print(json.dumps(line), flush=True)
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="default 200 (a single c4 run: 10)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="all", choices=sorted(WORKLOADS) + ["all"],
                    help="all (default): c2 is the headline line, c3 (1344^2) and c4 (mixed resolutions) ride in "
                         "`workloads`; or one workload alone")
    ap.add_argument("--rotate", type=int, default=0, help="resident input buffer sets to rotate over (default 8 with attention, else 4)")
    ap.add_argument("--streams", type=int, default=0, help="CUDA streams consecutive steps alternate over (default 4 with attention, else 3)")
    ap.add_argument("--sm-share", type=int, default=0, help="attwarp_set_sm_share for the overlapped steps (default 2 with attention and several streams, else 1)")
    ap.add_argument("--e2e-chunk", type=int, default=0, help="images per host-pipeline chunk (default 64 at 336^2, 16 at 1344^2)")
    ap.add_argument("--c4-steps", type=int, default=0, help="steps of the c4 workload (default: --steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch the kernels eagerly instead of by graph replay")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step returned as DIR/<workload>_<array>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 10 if args.workload == "c4" else 200
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank, local_rank, world = env_int("RANK", 0), env_int("LOCAL_RANK", 0), env_int("WORLD_SIZE", 1)
    # stdout carries the ONE JSON line and nothing else: NCCL's own logging (its version banner, NCCL_DEBUG
    # output) goes to stderr
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if args.impl == "reference":
        return run_reference(args, rank, world)
    if world == 1 and args.gpus > 1:
        print(f"bench.py: --gpus {args.gpus} needs torchrun (one rank per GPU); running 1 rank",
              file=sys.stderr)
    return run_gpu(args, rank, local_rank, world)


if __name__ == "__main__":
    sys.exit(main())
