"""The list checks the three ragged calls share, in the torch wrappers and in the C ABI.

A wrapper writes every image through its row of the descriptor table at that row's output size, and NumPy broadcasts a
one-element list into every row of a structured field: a list of outputs or output sizes of the wrong length must be
refused before any table is built.  The C ABI refuses invalid lists before it enqueues anything, and every call that
uploads descriptor tables from host memory refuses a stream that is being captured into a CUDA graph.

    python -m pytest tests/test_ragged_lists.py              # the checks that need no device
    python -m pytest tests/test_ragged_lists.py -m gpu       # graph-capture refusals
"""

import ctypes as C
import os

import numpy as np
import pytest
import torch

from gpu_util import need_gpu

U8 = torch.uint8
SIZES = [(20, 30), (12, 8), (9, 40)]


def _abi():
    from attwarp_b200 import _lib
    if not os.path.isfile(_lib.lib_path()):
        pytest.skip("library not built")
    return _lib, _lib.load()


# ---- wrappers: lists of the wrong length (CPU tensors: the length checks come before the device checks) ------------
def _cpu_list():
    imgs = [torch.zeros(h, w, 3, dtype=U8) for h, w in SIZES]
    return imgs, [torch.empty_like(i) for i in imgs], list(SIZES)


def _tokens(imgs, outs=None, out_sizes=None):
    from attwarp_b200 import ops
    return ops.warp_ragged_from_tokens(torch.zeros(len(imgs), 4, 4), imgs, out_sizes, outs=outs)


def _attention(imgs, outs=None, out_sizes=None):
    from attwarp_b200 import ops
    return ops.warp_ragged_from_attention([torch.zeros(i.shape[:2], dtype=U8) for i in imgs], imgs, out_sizes,
                                          outs=outs)


def _batch(imgs, outs=None, out_sizes=None):
    from attwarp_b200 import ops
    return ops.RaggedBatch(imgs, out_sizes, outs=outs)


@pytest.mark.parametrize("keep", [1, len(SIZES) - 1])
@pytest.mark.parametrize("call", [_tokens, _attention, _batch], ids=["tokens", "attention", "RaggedBatch"])
def test_outs_of_the_wrong_length_are_refused(call, keep):
    _abi()
    imgs, outs, _ = _cpu_list()
    with pytest.raises(ValueError, match=f"{keep} outputs for {len(imgs)} images"):
        call(imgs, outs=outs[:keep])


@pytest.mark.parametrize("keep", [1, len(SIZES) - 1])
@pytest.mark.parametrize("call", [_tokens, _attention], ids=["tokens", "attention"])
def test_out_sizes_of_the_wrong_length_are_refused(call, keep):
    _abi()
    imgs, _, sizes = _cpu_list()
    with pytest.raises(ValueError, match=f"{keep} output sizes for {len(imgs)} images"):
        call(imgs, out_sizes=sizes[:keep])


# ---- C ABI: invalid lists refused before anything is enqueued (fake pointers, no device) --------------------------
_TABLE = np.dtype([("src", np.uint64), ("dst", np.uint64), ("H", np.int32), ("W", np.int32), ("Ho", np.int32),
                   ("Wo", np.int32)])
_ATT = np.dtype([("att", np.uint64), ("map_x", np.uint64), ("map_y", np.uint64)])
_FAKE_WS = 0x7000000               # never dereferenced: every case fails first


def _fake_table(sizes):
    t = np.zeros(len(sizes), dtype=_TABLE)
    t["src"] = [0x10000 + 0x1000 * k for k in range(len(sizes))]
    t["dst"] = [0x90000 + 0x1000 * k for k in range(len(sizes))]
    for k, s in enumerate(sizes):
        t["H"][k], t["W"][k], t["Ho"][k], t["Wo"][k] = s
    return t


_CASES = [
    ("null_table", "ERR_INVALID_ARG", "NULL pointer"),
    ("null_ws", "ERR_INVALID_ARG", "NULL pointer"),
    ("n0", "ERR_INVALID_ARG", "must be positive"),
    ("C0", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("C2", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("C5", "ERR_INVALID_ARG", "C must be 1, 3 or 4"),
    ("empty_H", "ERR_INVALID_ARG", "sizes must be positive"),
    ("empty_W", "ERR_INVALID_ARG", "sizes must be positive"),
    ("empty_out", "ERR_INVALID_ARG", "sizes must be positive"),
    ("huge", "ERR_INVALID_ARG", "below 65536"),
    ("same_src_dst", "ERR_INVALID_ARG", "bad pointers"),
    ("small_ws", "ERR_WORKSPACE", "workspace too small"),
]


_OK = [(336, 336, 336, 336), (20, 16, 40, 30)]


def _fake_args(case):
    sizes = list(_OK)
    if case == "empty_H":
        sizes[1] = (0, 16, 20, 16)
    elif case == "empty_W":
        sizes[0] = (336, 0, 336, 336)
    elif case == "empty_out":
        sizes[1] = (20, 16, 20, 0)
    elif case == "huge":
        sizes[1] = (70000, 16, 20, 16)
    t = _fake_table(sizes)
    if case == "same_src_dst":
        t["dst"][1] = t["src"][1]
    return t, 0 if case == "n0" else len(sizes), {"C0": 0, "C2": 2, "C5": 5}.get(case, 3)


@pytest.mark.parametrize("case,status,msg", _CASES)
def test_tokens_abi_rejects_without_a_device(case, status, msg):
    _lib, lib = _abi()
    t, n, Cc = _fake_args(case)
    tp = _lib.make_transform()
    need = lib.attwarp_ragged_workspace_bytes(_fake_table(_OK).ctypes.data_as(C.c_void_p), 2)
    rc = lib.attwarp_warp_ragged_from_tokens(C.c_void_p(0x5000), n, 24, 24,
                                             None if case == "null_table" else t.ctypes.data_as(C.c_void_p), Cc,
                                             C.byref(tp), None if case == "null_ws" else C.c_void_p(_FAKE_WS),
                                             need - 1 if case == "small_ws" else need, None)
    assert rc == getattr(_lib, status), (rc, lib.attwarp_last_error())
    assert msg in lib.attwarp_last_error().decode()


@pytest.mark.parametrize("case,status,msg", _CASES + [
    ("null_map", "ERR_INVALID_ARG", "NULL attention map"),
    ("unaligned_map", "ERR_INVALID_ARG", "aligned"),
    ("bad_dtype", "ERR_INVALID_ARG", "attention dtype"),
])
def test_attention_abi_rejects_without_a_device(case, status, msg):
    _lib, lib = _abi()
    t, n, Cc = _fake_args(case)
    a = np.zeros(2, dtype=_ATT)
    a["att"] = [0x200000, 0 if case == "null_map" else 0x300001 if case == "unaligned_map" else 0x300000]
    dtype = {"unaligned_map": _lib.F32, "bad_dtype": _lib.BF16}.get(case, _lib.U8)
    tp = _lib.make_transform()
    need = lib.attwarp_ragged_attention_workspace_bytes(_fake_table(_OK).ctypes.data_as(C.c_void_p), 2)
    rc = lib.attwarp_warp_ragged_from_attention(None if case == "null_table" else t.ctypes.data_as(C.c_void_p),
                                                a.ctypes.data_as(C.c_void_p), n, dtype, Cc, C.byref(tp),
                                                None if case == "null_ws" else C.c_void_p(_FAKE_WS),
                                                need - 1 if case == "small_ws" else need, None)
    assert rc == getattr(_lib, status), (rc, lib.attwarp_last_error())
    assert msg in lib.attwarp_last_error().decode()


def test_tokens_workspace_bytes_refuse_invalid_sizes():
    _, lib = _abi()
    ok = _fake_table(_OK)
    assert lib.attwarp_ragged_workspace_bytes(ok.ctypes.data_as(C.c_void_p), 2) > 0
    assert lib.attwarp_ragged_workspace_bytes(ok.ctypes.data_as(C.c_void_p), 0) == 0
    assert lib.attwarp_ragged_workspace_bytes(None, 2) == 0
    for bad in ((0, 16, 40, 30), (20, -1, 40, 30), (20, 16, 0, 30), (20, 16, 40, -5), (65536, 16, 40, 30)):
        t = _fake_table([(336, 336, 336, 336), bad])
        assert lib.attwarp_ragged_workspace_bytes(t.ctypes.data_as(C.c_void_p), 2) == 0, bad


# ---- GPU: the six calls with host-side descriptor tables refuse CUDA-graph capture, before enqueueing anything ----
def _ragged_table(imgs, outs):
    t = np.zeros(len(imgs), dtype=_TABLE)
    t["src"] = [i.data_ptr() for i in imgs]
    t["dst"] = [o.data_ptr() for o in outs]
    t["H"] = [i.shape[0] for i in imgs]
    t["W"] = [i.shape[1] for i in imgs]
    t["Ho"] = [o.shape[0] for o in outs]
    t["Wo"] = [o.shape[1] for o in outs]
    return t


def _gpu_list():
    imgs = [torch.randint(0, 256, (h, w, 3), dtype=U8, device="cuda") for h, w in SIZES]
    return imgs, [torch.empty_like(i) for i in imgs]


def _tokens_call(_lib, lib):
    imgs, outs = _gpu_list()
    t = _ragged_table(imgs, outs)
    tok = torch.rand(len(imgs), 16, device="cuda")
    tp = _lib.make_transform()
    ws = torch.empty(int(lib.attwarp_ragged_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(imgs))), dtype=U8,
                     device="cuda")
    return lambda st: lib.attwarp_warp_ragged_from_tokens(_lib.ptr(tok), len(imgs), 4, 4, t.ctypes.data_as(C.c_void_p),
                                                          3, C.byref(tp), _lib.ptr(ws), ws.numel(), st)


def _attention_call(_lib, lib):
    imgs, outs = _gpu_list()
    t = _ragged_table(imgs, outs)
    maps = [torch.rand(i.shape[:2], device="cuda") for i in imgs]
    a = np.zeros(len(imgs), dtype=_ATT)
    a["att"] = [m.data_ptr() for m in maps]
    tp = _lib.make_transform()
    ws = torch.empty(int(lib.attwarp_ragged_attention_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(imgs))),
                     dtype=U8, device="cuda")
    return lambda st: lib.attwarp_warp_ragged_from_attention(t.ctypes.data_as(C.c_void_p), a.ctypes.data_as(C.c_void_p),
                                                             len(imgs), _lib.F32, 3, C.byref(tp), _lib.ptr(ws),
                                                             ws.numel(), st)


def _mask_call(_lib, lib):
    imgs, outs = _gpu_list()
    t = _ragged_table(imgs, outs)
    mask = torch.randint(0, 256, (len(imgs), 4, 4), dtype=U8, device="cuda")
    tp = _lib.make_transform()
    ws = torch.empty(int(lib.attwarp_ragged_mask_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(imgs), 4, 4)),
                     dtype=U8, device="cuda")
    return lambda st: lib.attwarp_warp_ragged_from_mask(t.ctypes.data_as(C.c_void_p), _lib.ptr(mask), len(imgs), 4, 4,
                                                        3, C.byref(tp), _lib.ptr(ws), ws.numel(), None, None, st)


def _png_call(_lib, lib):
    from attwarp_b200.ops import _PNG_DTYPE
    imgs, _ = _gpu_list()
    t = np.zeros(len(imgs), dtype=_PNG_DTYPE)
    t["src"] = [i.data_ptr() for i in imgs]
    t["H"] = [i.shape[0] for i in imgs]
    t["W"] = [i.shape[1] for i in imgs]
    t["C"] = 3
    cap = sum(int(lib.attwarp_png_max_bytes(i.shape[0], i.shape[1], 3)) for i in imgs)
    out = torch.empty(cap, dtype=U8, device="cuda")
    offsets = torch.empty(len(imgs) + 1, dtype=torch.int64, device="cuda")
    ws = torch.empty(int(lib.attwarp_png_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(imgs))), dtype=U8,
                     device="cuda")
    return lambda st: lib.attwarp_encode_png(t.ctypes.data_as(C.c_void_p), len(imgs), _lib.ptr(ws), ws.numel(),
                                             _lib.ptr(out), cap, _lib.ptr(offsets), st)


def _jpeg_call(_lib, lib):
    import jpeg_corpus as JC
    from attwarp_b200.ops import _JPEG_DTYPE
    files = [JC.pil_jpeg(JC.content("photo", h, w, np.random.default_rng(k)), quality=90)
             for k, (h, w) in enumerate(SIZES)]
    host = [np.frombuffer(f, dtype=np.uint8) for f in files]
    data = [torch.from_numpy(h.copy()).cuda() for h in host]
    outs = [torch.empty(h, w, 3, dtype=U8, device="cuda") for h, w in SIZES]
    status = torch.empty(len(files), dtype=torch.int32, device="cuda")
    t = np.zeros(len(files), dtype=_JPEG_DTYPE)
    t["host"] = [h.ctypes.data for h in host]
    t["dev"] = [d.data_ptr() for d in data]
    t["nbytes"] = [len(f) for f in files]
    t["dst"] = [o.data_ptr() for o in outs]
    t["H"] = [h for h, _ in SIZES]
    t["W"] = [w for _, w in SIZES]
    ws = torch.empty(int(lib.attwarp_jpeg_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(files))), dtype=U8,
                     device="cuda")
    return lambda st: lib.attwarp_decode_jpeg(t.ctypes.data_as(C.c_void_p), len(files), _lib.ptr(ws), ws.numel(),
                                              _lib.ptr(status), st)


def _overlay_call(_lib, lib):
    from attwarp_b200.ops import _OVERLAY_DTYPE, _OVERLAY_MAP
    imgs, outs = _gpu_list()
    maps = [torch.randint(0, 256, i.shape[:2], dtype=U8, device="cuda") for i in imgs]
    t = np.zeros(len(imgs), dtype=_OVERLAY_DTYPE)
    t["src"] = [i.data_ptr() for i in imgs]
    t["att"] = [m.data_ptr() for m in maps]
    t["dst"] = [o.data_ptr() for o in outs]
    t["H"] = [i.shape[0] for i in imgs]
    t["W"] = [i.shape[1] for i in imgs]
    t["C"] = 3
    ws = torch.empty(max(int(lib.attwarp_overlay_workspace_bytes(t.ctypes.data_as(C.c_void_p), len(imgs),
                                                                 _OVERLAY_MAP)), 1), dtype=U8, device="cuda")
    return lambda st: lib.attwarp_attention_overlay(t.ctypes.data_as(C.c_void_p), len(imgs), _lib.U8, _OVERLAY_MAP, 0,
                                                    0, 0.5, _lib.ptr(ws), ws.numel(), st)


@pytest.mark.gpu
@pytest.mark.parametrize("prefix,make", [
    ("warp_ragged", _tokens_call),
    ("warp_ragged_from_attention", _attention_call),
    ("warp_ragged_from_mask", _mask_call),
    ("encode_png", _png_call),
    ("decode_jpeg", _jpeg_call),
    ("attention_overlay", _overlay_call),
], ids=lambda v: v if isinstance(v, str) else "")
def test_host_table_calls_refuse_graph_capture(prefix, make):
    need_gpu()
    _lib, lib = _abi()
    call = make(_lib, lib)
    assert call(_lib.current_stream()) == _lib.OK, lib.attwarp_last_error()       # the same arguments run uncaptured
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph(keep_graph=True)
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            rc = call(C.c_void_p(s.cuda_stream))
    assert rc == _lib.ERR_UNSUPPORTED
    assert lib.attwarp_last_error().decode().startswith(f"{prefix}: cannot be captured into a CUDA graph")
    nodes = C.c_size_t(1 << 30)
    assert C.CDLL("libcuda.so.1").cuGraphGetNodes(C.c_void_p(g.raw_cuda_graph()), None, C.byref(nodes)) == 0
    assert nodes.value == 0                                                          # nothing was enqueued
