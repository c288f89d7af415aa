"""Stage 1 (aggregate.cu, aggregate_tma.cu): every compiled row kernel against a float64 reference.

The launcher picks one of 30 kernels from dtype, layout, alignment and row length T.  CASES names one input per
kernel at the lengths where the choice changes (the last T a variant takes and the first T the next one takes),
the layout that reaches it, and the kernel it must launch; each case is checked against a float64 reference on
inputs that expose a wrong normalisation (row sums over eight decades, zero rows, sums near eps, subnormal values,
a single nonzero at either end of a row), with NaN wherever the kernel must not read, and its launch is read back
from torch.profiler.  test_case_table_names_every_compiled_kernel (CPU) keeps CASES and the library in step.

    python -m pytest tests/test_gpu_aggregate_dispatch.py -m gpu -s     # -s prints the worst error per family
"""

import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

BF16, F16, F32 = torch.bfloat16, torch.float16, torch.float32
VE = {BF16: 8, F16: 8, F32: 4}             # elements per 16-byte vector
EPS = 1e-12                                # the eps of ops.aggregate_attention and of the fused warp path
MARGIN = 64                                # NaN elements before and after every input (a multiple of 16 bytes)
EXTRA = 13                                 # row length beyond T in the tok_start layout

# Layouts (all inside a NaN margin):
#   gap     dense rows; storage [B, L + 1, Hh, T] with NaN at index L, the view is [:, :L]
#   pad     rows padded to T + VE with NaN, the view is [..., :T]
#   window  rows of K = T + EXTRA, a tok_start window of T tokens per image, NaN outside it
#   offset  dense rows from a base one element past a 16-byte boundary
# (dtype, B, L, Hh, T, layout, kernel)
CASES = [
    # TMA: no tok_start, rows of an image contiguous, 16-byte aligned, T <= 576; NP = ceil(T / 64)
    (BF16, 3, 3, 7, 8, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 2, false>"),
    (BF16, 1, 9, 37, 128, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 2, false>"),
    (BF16, 600, 3, 7, 136, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 5, false>"),
    (BF16, 2, 5, 7, 320, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 5, false>"),
    (BF16, 3, 1, 37, 328, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 9, false>"),
    (BF16, 2, 3, 17, 568, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 9, false>"),
    (BF16, 4, 7, 11, 576, "gap", "aggregate_rows_tma_kernel<__nv_bfloat16, 9, true>"),
    (F16, 2, 7, 13, 8, "gap", "aggregate_rows_tma_kernel<__half, 2, false>"),
    (F16, 3, 3, 17, 128, "gap", "aggregate_rows_tma_kernel<__half, 2, false>"),
    (F16, 1, 9, 37, 136, "gap", "aggregate_rows_tma_kernel<__half, 5, false>"),
    (F16, 4, 5, 11, 320, "gap", "aggregate_rows_tma_kernel<__half, 5, false>"),
    (F16, 2, 3, 7, 328, "gap", "aggregate_rows_tma_kernel<__half, 9, false>"),
    (F16, 3, 5, 19, 568, "gap", "aggregate_rows_tma_kernel<__half, 9, false>"),
    (F16, 2, 1, 53, 576, "gap", "aggregate_rows_tma_kernel<__half, 9, true>"),
    (F32, 2, 3, 7, 4, "gap", "aggregate_rows_tma_kernel<float, 2, false>"),
    (F32, 3, 5, 7, 128, "gap", "aggregate_rows_tma_kernel<float, 2, false>"),
    (F32, 2, 1, 37, 132, "gap", "aggregate_rows_tma_kernel<float, 5, false>"),
    (F32, 1, 9, 37, 320, "gap", "aggregate_rows_tma_kernel<float, 5, false>"),
    (F32, 4, 3, 17, 324, "gap", "aggregate_rows_tma_kernel<float, 9, false>"),
    (F32, 2, 7, 13, 572, "gap", "aggregate_rows_tma_kernel<float, 9, false>"),
    (F32, 3, 3, 19, 576, "gap", "aggregate_rows_tma_kernel<float, 9, true>"),
    # vec: no tok_start, 16-byte aligned rows that miss TMA (padded, or T > 576); NV = ceil(T / VE / 32) <= 9
    (BF16, 2, 3, 7, 8, "pad", "aggregate_rows_vec_kernel<__nv_bfloat16, 1>"),
    (BF16, 1, 9, 37, 256, "pad", "aggregate_rows_vec_kernel<__nv_bfloat16, 1>"),
    (BF16, 3, 5, 7, 264, "pad", "aggregate_rows_vec_kernel<__nv_bfloat16, 2>"),
    (BF16, 2, 3, 17, 512, "pad", "aggregate_rows_vec_kernel<__nv_bfloat16, 2>"),
    (BF16, 4, 1, 37, 520, "pad", "aggregate_rows_vec_kernel<__nv_bfloat16, 3>"),
    (BF16, 2, 7, 11, 768, "gap", "aggregate_rows_vec_kernel<__nv_bfloat16, 3>"),
    (BF16, 3, 3, 19, 776, "gap", "aggregate_rows_vec_kernel<__nv_bfloat16, 5>"),
    (BF16, 2, 5, 11, 1280, "gap", "aggregate_rows_vec_kernel<__nv_bfloat16, 5>"),
    (BF16, 1, 7, 13, 1288, "gap", "aggregate_rows_vec_kernel<__nv_bfloat16, 9>"),
    (BF16, 2, 3, 7, 2304, "gap", "aggregate_rows_vec_kernel<__nv_bfloat16, 9>"),
    (F16, 3, 7, 13, 8, "pad", "aggregate_rows_vec_kernel<__half, 1>"),
    (F16, 2, 3, 17, 256, "pad", "aggregate_rows_vec_kernel<__half, 1>"),
    (F16, 600, 3, 7, 264, "pad", "aggregate_rows_vec_kernel<__half, 2>"),
    (F16, 1, 9, 37, 512, "pad", "aggregate_rows_vec_kernel<__half, 2>"),
    (F16, 2, 5, 7, 520, "pad", "aggregate_rows_vec_kernel<__half, 3>"),
    (F16, 3, 1, 53, 768, "gap", "aggregate_rows_vec_kernel<__half, 3>"),
    (F16, 2, 3, 7, 776, "gap", "aggregate_rows_vec_kernel<__half, 5>"),
    (F16, 2, 7, 11, 1280, "gap", "aggregate_rows_vec_kernel<__half, 5>"),
    (F16, 3, 5, 11, 1288, "gap", "aggregate_rows_vec_kernel<__half, 9>"),
    (F16, 1, 3, 19, 2304, "gap", "aggregate_rows_vec_kernel<__half, 9>"),
    (F32, 2, 5, 7, 4, "pad", "aggregate_rows_vec_kernel<float, 1>"),
    (F32, 3, 3, 7, 128, "pad", "aggregate_rows_vec_kernel<float, 1>"),
    (F32, 1, 9, 37, 132, "pad", "aggregate_rows_vec_kernel<float, 2>"),
    (F32, 2, 3, 17, 256, "pad", "aggregate_rows_vec_kernel<float, 2>"),
    (F32, 4, 7, 11, 260, "pad", "aggregate_rows_vec_kernel<float, 3>"),
    (F32, 2, 1, 37, 384, "pad", "aggregate_rows_vec_kernel<float, 3>"),
    (F32, 3, 5, 19, 388, "pad", "aggregate_rows_vec_kernel<float, 5>"),
    (F32, 2, 3, 19, 640, "gap", "aggregate_rows_vec_kernel<float, 5>"),
    (F32, 2, 7, 13, 644, "gap", "aggregate_rows_vec_kernel<float, 9>"),
    (F32, 1, 5, 11, 1152, "gap", "aggregate_rows_vec_kernel<float, 9>"),
    # generic: tok_start, a misaligned base, or rows too long for the vector kernels (8 T floats <= 200 KB)
    (BF16, 3, 3, 7, 1, "window", "aggregate_rows_generic_kernel<__nv_bfloat16>"),
    (F16, 2, 5, 7, 7, "window", "aggregate_rows_generic_kernel<__half>"),
    (F32, 2, 3, 17, 577, "window", "aggregate_rows_generic_kernel<float>"),
    (BF16, 1, 9, 37, 577, "window", "aggregate_rows_generic_kernel<__nv_bfloat16>"),
    (F16, 3, 3, 7, 128, "offset", "aggregate_rows_generic_kernel<__half>"),
    (F32, 2, 1, 37, 132, "offset", "aggregate_rows_generic_kernel<float>"),
    (BF16, 2, 1, 21, 6400, "gap", "aggregate_rows_generic_kernel<__nv_bfloat16>"),
    (F32, 1, 3, 7, 6400, "window", "aggregate_rows_generic_kernel<float>"),
]

CNAME = {BF16: "bf16", F16: "f16", F32: "f32"}
CASE_IDS = [f"{k.split('_')[2]}-{CNAME[dt]}-T{T}-B{B}-{lay}" for dt, B, L, Hh, T, lay, k in CASES]
FAMILIES = ["scaled", "zero_rows", "tiny_sums", "subnormal", "edge_columns"]
WORST = {}                                 # (kernel family, input family) -> (worst err / bar, worst relative err)


def _families(dt):
    # f16 cannot hold row sums near 1e-12, and its subnormals are normal floats
    return [f for f in FAMILIES if dt != F16 or f not in ("tiny_sums", "subnormal")]


def _exact(x, dt):
    """x rounded to dt, as float64: the values the kernel reads."""
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float64)).to(dt).double().numpy()


def make_input(family, dt, shape, rng):
    """A float64 [B, L, Hh, T] array whose values dt holds exactly."""
    B, L, Hh, T = shape
    if family == "scaled":                 # positive rows scaled by 10^U(-4, 4); <= 1e4 stays inside f16
        x = rng.uniform(0.05, 1.0, shape) * 10.0 ** rng.uniform(-4, 4, (B, L, Hh, 1))
    elif family == "zero_rows":            # some rows all zero; with B > 1 image 0 is all zero
        x = rng.uniform(0.05, 1.0, shape) * 10.0 ** rng.uniform(-2, 2, (B, L, Hh, 1))
        x[rng.random((B, L, Hh)) < 0.3] = 0.0
        x[B - 1, 0, 0] = 0.0
        if B > 1:
            x[0] = 0.0
    elif family == "tiny_sums":            # row sums 1e-12 * U(0.5, 2): eps is about half of each denominator
        p = rng.uniform(0.05, 1.0, shape)
        x = p / p.sum(-1, keepdims=True) * 1e-12 * rng.uniform(0.5, 2.0, (B, L, Hh, 1))
    elif family == "subnormal":            # every value subnormal in dt (bf16: m * 2^-133, f32: m * 2^-149)
        x = rng.integers(1, 128, shape) * 2.0 ** -133 if dt == BF16 else rng.integers(1, 1 << 23, shape) * 2.0 ** -149
    elif family == "edge_columns":         # one nonzero per row, in column 0 or column T - 1
        x = np.zeros(shape)
        col = np.where(rng.random((B, L, Hh)) < 0.5, 0, T - 1)
        np.put_along_axis(x, col[..., None], (rng.uniform(0.5, 2.0, (B, L, Hh)) * 10.0 ** rng.uniform(-3, 3, (B, L, Hh)))[..., None], -1)
    else:
        raise ValueError(family)
    x = _exact(x, dt)
    if family == "subnormal":
        assert 0 < x.min() and x.max() < np.finfo(np.float32).tiny
    return x


def reference(x):
    """float64: mean over l, h of a / (sum_t a + 1e-12)."""
    return (x / (x.sum(-1, keepdims=True) + EPS)).mean(axis=(1, 2))


def place(x, dt, layout, rng):
    """Lay x out as ``layout`` in a NaN-filled host buffer.  -> (flat dt tensor, view shape, view strides, storage
    offset, tok_start or None); ``on_device`` turns it into the CUDA view the kernel reads."""
    B, L, Hh, T = x.shape
    starts = None
    if layout == "gap":
        store = np.full((B, L + 1, Hh, T), np.nan)
        store[:, :L] = x
        shape = x.shape
    elif layout == "pad":
        store = np.full((B, L, Hh, T + VE[dt]), np.nan)
        store[..., :T] = x
        shape = x.shape
    elif layout == "window":
        store = np.full((B, L, Hh, T + EXTRA), np.nan)
        starts = rng.integers(0, EXTRA + 1, B)
        starts[0], starts[-1] = 0, EXTRA            # windows at both ends of the row
        for b in range(B):
            store[b, ..., starts[b]:starts[b] + T] = x[b]
        starts = [int(s) for s in starts]
        shape = store.shape
    elif layout == "offset":
        store = np.ascontiguousarray(x)
        shape = x.shape
    else:
        raise ValueError(layout)
    lead = MARGIN + (1 if layout == "offset" else 0)
    flat = np.concatenate([np.full(lead, np.nan), store.ravel(), np.full(MARGIN, np.nan)])
    strides = tuple(s // store.itemsize for s in store.strides)
    return torch.from_numpy(flat).to(dt), shape, strides, lead, starts


def on_device(flat, shape, strides, offset):
    return flat.cuda().as_strided(shape, strides, offset)


def check(got, ref, what):
    """|got - ref| <= 1e-5 |ref| + 1e-7 max|ref_b| per image b (an all-zero image must give exactly 0).
    -> (worst err / bar, worst relative err)."""
    got = got.double().cpu().numpy()
    err = np.abs(got - ref)
    bar = 1e-5 * np.abs(ref) + 1e-7 * np.abs(ref).max(axis=1, keepdims=True)
    bad = ~(err <= bar)                             # NaN fails
    if bad.any():
        b, t = (int(i) for i in np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} outputs off the float64 reference, first at "
                             f"image {b} token {t}: got {got[b, t]!r}, ref {ref[b, t]!r}, bar {bar[b, t]:.3g}")
    nz = ref != 0
    return (float(np.max(np.where(bar > 0, err / np.where(bar > 0, bar, 1), 0))),
            float(np.max(err[nz] / np.abs(ref[nz]))) if nz.any() else 0.0)


def _demangle(names):
    tool = shutil.which("c++filt") or shutil.which("cu++filt")
    if tool is None or not names:
        return list(names)
    res = subprocess.run([tool], input="\n".join(names) + "\n", capture_output=True, text=True, check=True)
    return res.stdout.splitlines()


def _row_kernels(names):
    """The aggregate_rows_* template instances in a list of (possibly mangled) symbol names, without spaces."""
    found = []
    for n in _demangle(names):
        found += [re.sub(r"\s+", "", m) for m in re.findall(r"aggregate_rows_\w+?_kernel<[^>]*>", n)]
    return found


def _nsplit(lib, B, L, Hh, T):
    return lib.attwarp_aggregate_workspace_bytes(B, L, Hh, T) // (4 * B * T)


@pytest.fixture(scope="module", autouse=True)
def _print_worst():
    yield
    if WORST:
        print("\nstage-1 worst error per kernel and input family (err / bar must be <= 1):")
        for (kern, fam), (bar, rel) in sorted(WORST.items()):
            print(f"  {kern:8s} {fam:13s} err/bar {bar:.3g}   max rel err {rel:.3g}")


def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


# ---------------------------------------------------------------------------------------------- CPU
def test_case_table_names_every_compiled_kernel():
    """The aggregate_rows_* instantiations in the built library are exactly the kernels CASES names: a new variant
    without a case fails here."""
    from attwarp_b200 import _lib
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.isfile(cuobjdump):
        pytest.skip("cuobjdump not available")
    assert os.path.isfile(_lib.lib_path()), "build the library first: python -m attwarp_b200.build"
    out = subprocess.run([cuobjdump, "-symbols", _lib.lib_path()], capture_output=True, text=True, check=True).stdout
    compiled = set(_row_kernels(out.splitlines()))
    named = {re.sub(r"\s+", "", k) for *_, k in CASES}
    print(f"\n{len(compiled)} aggregate_rows_* instantiations in the library:\n  " + "\n  ".join(sorted(compiled)))
    assert len(compiled) >= 30
    assert compiled == named, f"compiled but no case: {sorted(compiled - named)}; named but not compiled: {sorted(named - compiled)}"


# ---------------------------------------------------------------------------------------------- GPU
@pytest.mark.gpu
@pytest.mark.parametrize("case", range(len(CASES)), ids=CASE_IDS)
def test_kernel_vs_float64(case):
    """One case of CASES on every input family: the float64 bar per image, nothing read outside the view (NaN
    there), and the launch of the kernel the table names."""
    _need_gpu()
    from attwarp_b200 import _lib, ops
    dt, B, L, Hh, T, layout, kernel = CASES[case]
    kern_family = kernel.split("_")[2]
    n_rows = L * Hh
    nsplit = _nsplit(_lib.load(), B, L, Hh, T)
    # the table's shapes must give CTAs of uneven length, and B >= 593 a single split (4 CTAs per SM, 148 SMs)
    assert n_rows % 8 and (nsplit == 1 or n_rows % nsplit), (n_rows, nsplit)
    if B >= 593:
        assert nsplit == 1, nsplit
    rng = np.random.default_rng(1000 + case)
    launched = None
    for fam in _families(dt):
        x = make_input(fam, dt, (B, L, Hh, T), rng)
        flat, shape, strides, offset, starts = place(x, dt, layout, rng)
        attn = on_device(flat, shape, strides, offset)
        if launched is None:
            with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CPU,
                                                    torch.profiler.ProfilerActivity.CUDA]) as prof:
                got = ops.aggregate_attention(attn, tok_start=starts, num_tokens=T)
                torch.cuda.synchronize()
            launched = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
        else:
            got = ops.aggregate_attention(attn, tok_start=starts, num_tokens=T)
        ref = reference(x)
        what = f"{CASE_IDS[case]} ({kernel}, nsplit {nsplit}) family {fam}"
        bar, rel = check(got, ref, what)
        if fam == "zero_rows" and B > 1:
            assert torch.count_nonzero(got[0]).item() == 0, f"{what}: the all-zero image gave nonzero output"
        if fam == "subnormal":              # a flush-to-zero kernel returns exactly 0
            assert torch.count_nonzero(got).item() == got.numel(), f"{what}: zeros from subnormal input"
        w = WORST.get((kern_family, fam), (0.0, 0.0))
        WORST[(kern_family, fam)] = (max(w[0], bar), max(w[1], rel))
    if not launched:
        pytest.skip("torch.profiler reported no CUDA kernel events: the launched kernel is not checked")
    rows = _row_kernels(launched)
    assert rows == [re.sub(r"\s+", "", kernel)], f"{CASE_IDS[case]}: expected {kernel}, launched {launched}"


def _dense(dt, shape, seed, layout="gap"):
    rng = np.random.default_rng(seed)
    x = make_input("scaled", dt, shape, rng)
    flat, vshape, strides, offset, starts = place(x, dt, layout, rng)
    return x, on_device(flat, vshape, strides, offset), starts


@pytest.mark.gpu
def test_out_accumulate_and_scale():
    """out= with accumulate=True adds out_scale * mean into the prefilled output; three accumulated calls with
    out_scale = 1/3 give the running mean (the hook loggers' use)."""
    _need_gpu()
    from attwarp_b200 import ops
    for dt, layout, shape in ((BF16, "gap", (3, 3, 7, 576)), (F32, "pad", (2, 5, 7, 260)), (F16, "window", (3, 1, 37, 77))):
        x, attn, starts = _dense(dt, shape, 11, layout)
        B, T = shape[0], shape[3]
        out0 = np.random.default_rng(12).uniform(0.5, 2.0, (B, T)).astype(np.float32)
        out = torch.from_numpy(out0).cuda()
        res = ops.aggregate_attention(attn, tok_start=starts, num_tokens=T, out=out, accumulate=True, out_scale=0.37)
        assert res.data_ptr() == out.data_ptr()
        check(out, out0.astype(np.float64) + 0.37 * reference(x), f"{dt} {layout} accumulate out_scale=0.37")
        run = torch.zeros(B, T, device="cuda")
        refs = []
        for k in range(3):
            x, attn, starts = _dense(dt, shape, 20 + k, layout)
            ops.aggregate_attention(attn, tok_start=starts, num_tokens=T, out=run, accumulate=True, out_scale=1 / 3)
            refs.append(reference(x))
        check(run, np.mean(refs, axis=0), f"{dt} {layout} running mean of three calls")


@pytest.mark.gpu
@pytest.mark.parametrize("dt,shape,grid,layout", [(BF16, (3, 3, 7, 576), (24, 24), "gap"),
                                                  (F16, (2, 5, 7, 264), (12, 22), "pad"),
                                                  (F32, (3, 3, 17, 77), (7, 11), "window")],
                         ids=["tma", "vec", "tok_start"])
def test_fused_token_map_bit_equal(dt, shape, grid, layout):
    """The token map warp_from_attention_tokens hands back is aggregate_attention's, bit for bit: both sum the split
    partials in order and then scale."""
    _need_gpu()
    from attwarp_b200 import ops
    x, attn, starts = _dense(dt, shape, 31, layout)
    B, T = shape[0], shape[3]
    imgs = torch.from_numpy(np.random.default_rng(32).integers(0, 256, (B, 40, 48, 3), dtype=np.uint8)).cuda()
    _, tok, _, _ = ops.warp_from_attention_tokens(attn, imgs, grid, tok_start=starts, return_aux=True)
    agg = ops.aggregate_attention(attn, tok_start=starts, num_tokens=T)
    assert torch.equal(tok.reshape(B, T), agg), layout
    check(agg, reference(x), f"{layout} aggregate_attention")


# (dtype, L, Hh, T, layout) run with every forced split count: 9 * 23 = 207 rows, up to 13 CTAs of uneven length
SPLIT_CASES = [(F32, 9, 23, 320, "gap"), (BF16, 9, 23, 264, "pad"), (F16, 9, 23, 7, "window")]
SPLIT_VALUES = [1, 3, 7, 1000]


def _run_child(in_path, out_path):
    """Child process of test_forced_split_counts: ATTWARP_AGG_NSPLIT is read once per process."""
    from attwarp_b200 import _lib, ops
    lib = _lib.load()
    res = []
    for c in torch.load(in_path, weights_only=True):
        attn = on_device(c["flat"], c["shape"], c["strides"], c["offset"])
        B, L, Hh, _ = c["shape"]
        out = ops.aggregate_attention(attn, tok_start=c["starts"], num_tokens=c["T"])
        res.append({"out": out.cpu(), "nsplit": _nsplit(lib, B, L, Hh, c["T"])})
    torch.save(res, out_path)


@pytest.mark.gpu
def test_forced_split_counts(tmp_path):
    """ATTWARP_AGG_NSPLIT = 1, 3, 7 and 1000 (clamped to ceil(L Hh / 16)): one TMA, one vec and one tok_start case
    per split count, each in a child process, against the float64 reference."""
    _need_gpu()
    inputs, refs = [], []
    for k, (dt, L, Hh, T, layout) in enumerate(SPLIT_CASES):
        rng = np.random.default_rng(40 + k)
        x = make_input("scaled", dt, (2, L, Hh, T), rng)
        flat, shape, strides, offset, starts = place(x, dt, layout, rng)
        inputs.append({"flat": flat, "shape": list(shape), "strides": list(strides), "offset": offset,
                       "starts": starts, "T": T})
        refs.append(reference(x))
    in_path = tmp_path / "inputs.pt"
    torch.save(inputs, in_path)
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import test_gpu_aggregate_dispatch as m; m._run_child(sys.argv[1], sys.argv[2])" % (HERE, ROOT))
    procs = {}
    for v in SPLIT_VALUES:
        env = dict(os.environ, ATTWARP_AGG_NSPLIT=str(v))
        procs[v] = subprocess.Popen([sys.executable, "-c", code, str(in_path), str(tmp_path / f"out_{v}.pt")],
                                    env=env, cwd=ROOT, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        logs = {v: p.communicate(timeout=300)[0] for v, p in procs.items()}
    finally:
        for p in procs.values():
            if p.poll() is None:
                p.kill()
                p.wait()
    for v, p in procs.items():
        assert p.returncode == 0, f"ATTWARP_AGG_NSPLIT={v}: child failed\n{logs[v]}"
        res = torch.load(tmp_path / f"out_{v}.pt", weights_only=True)
        for (dt, L, Hh, T, layout), r, ref in zip(SPLIT_CASES, res, refs):
            assert r["nsplit"] == min(v, -(-L * Hh // 16)), (v, r["nsplit"])
            check(r["out"], ref, f"ATTWARP_AGG_NSPLIT={v} ({r['nsplit']} CTAs per image) {dt} T={T} {layout}")


@pytest.mark.gpu
def test_row_longer_than_generic_kernel_is_rejected():
    """T = 6401 needs 8 T floats > 200 KB of shared memory in the generic kernel: the library refuses it."""
    _need_gpu()
    from attwarp_b200 import ops
    from attwarp_b200._lib import AttWarpError
    attn = torch.full((1, 1, 3, 6401), 1.0, dtype=F32, device="cuda")
    with pytest.raises(AttWarpError, match="exceeds the supported row length"):
        ops.aggregate_attention(attn)
    with pytest.raises(AttWarpError, match="exceeds the supported row length"):
        ops.aggregate_attention(attn, tok_start=[0], num_tokens=6401)


@pytest.mark.gpu
def test_token_range_is_validated():
    """A token window that is not inside the row raises ValueError before any launch, in both ops entry points."""
    _need_gpu()
    from attwarp_b200 import ops
    B, L, Hh, K = 2, 1, 3, 64
    attn = torch.ones(B, L, Hh, K, dtype=BF16, device="cuda")
    imgs = torch.zeros(B, 16, 16, 3, dtype=torch.uint8, device="cuda")
    agg = lambda **kw: ops.aggregate_attention(attn, **kw)                                    # noqa: E731
    warp = lambda grid, **kw: ops.warp_from_attention_tokens(attn, imgs, grid, **kw)          # noqa: E731
    bad = [
        ("fewer starts than images", lambda: agg(tok_start=[0], num_tokens=8)),
        ("more starts than images (CUDA)", lambda: agg(tok_start=torch.zeros(B + 1, dtype=torch.int32, device="cuda"),
                                                       num_tokens=8)),
        ("T < 1", lambda: agg(num_tokens=0)),
        ("T < 1 with tok_start", lambda: agg(tok_start=[0, 0], num_tokens=0)),
        ("T > K", lambda: agg(num_tokens=K + 1)),
        ("negative start", lambda: agg(tok_start=[0, -1], num_tokens=8)),
        ("start + T > K", lambda: agg(tok_start=torch.tensor([K - 8, K - 7]), num_tokens=8)),
        ("warp: fewer starts than images", lambda: warp((2, 4), tok_start=[0])),
        ("warp: more starts than images (CUDA)", lambda: warp((2, 4), tok_start=torch.zeros(B + 1, dtype=torch.int32,
                                                                                             device="cuda"))),
        ("warp: T < 1", lambda: warp((0, 4), tok_start=[0, 0])),
        ("warp: T > K", lambda: warp((5, 13))),
        ("warp: negative start", lambda: warp((2, 4), tok_start=torch.tensor([-3, 0]))),
        ("warp: start + T > K", lambda: warp((2, 4), tok_start=[K - 8, K - 7])),
    ]
    for what, call in bad:
        with pytest.raises(ValueError):
            call()
            pytest.fail(what)
    # the edges of the valid range are accepted
    x = _exact(np.random.default_rng(50).uniform(0.05, 1.0, (B, L, Hh, K)), BF16)
    attn.copy_(torch.from_numpy(x).to(BF16))
    got = ops.aggregate_attention(attn, tok_start=[0, K - 8], num_tokens=8)
    check(got, np.stack([reference(x[:1, ..., :8])[0], reference(x[1:, ..., K - 8:])[0]]), "valid edge windows")
    _, tok, _, _ = ops.warp_from_attention_tokens(attn, imgs, (2, 4), tok_start=[K - 8, 0], return_aux=True)
    check(tok.reshape(B, 8), np.stack([reference(x[:1, ..., K - 8:])[0], reference(x[1:, ..., :8])[0]]),
          "warp: valid edge windows")
