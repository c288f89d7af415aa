"""GPU: ops.decode_jpeg equals Pillow's Image.open(f).convert('RGB') (as BGR) bit for bit on the seeded corpus, a
mixed-size fuzz list and large files without restart markers; an image's output depends on nothing else in the
call; the kernels write each [H, W, 3] buffer at any byte alignment and nothing around it; malformed entropy data
raises ValueError naming the file; decode_jpeg_batch(exact_device=True) routes every file to an exact decoder;
warp_files(exact_decode=True) writes the files the exact host decode gives."""

import ctypes as C
import os

import cv2
import numpy as np
import pytest
import torch

import jpeg_corpus as JC
from gpu_util import need_gpu

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def _gpu():
    need_gpu()


def _check_equal(files, outs, names=None):
    bad = []
    for i, (b, t) in enumerate(zip(files, outs)):
        ref = JC.pillow_bgr(b)
        got = t.cpu().numpy()
        if got.shape != ref.shape or not np.array_equal(got, ref):
            diff = int(np.abs(got.astype(int) - ref.astype(int)).max()) if got.shape == ref.shape else -1
            bad.append((names[i] if names else i, diff))
    assert not bad, bad[:10]


def test_corpus_equals_pillow():
    from attwarp_b200 import ops
    corpus = JC.corpus()
    files = [b for _, b in corpus]
    _check_equal(files, ops.decode_jpeg(files), [n for n, _ in corpus])


def test_fuzz_list_equals_pillow():
    from attwarp_b200 import ops
    files = JC.fuzz(320)
    _check_equal(files, ops.decode_jpeg(files))


def test_large_files_without_restart_markers():
    """Tens of thousands of synchronisation windows in one scan."""
    from attwarp_b200 import ops
    rng = np.random.default_rng(11)
    files = [JC.pil_jpeg(JC.content("photo", 1344, 1344, rng), quality=90),
             JC.cv2_jpeg(JC.content("noise", 3000, 4000, rng), 100, 444),
             JC.pil_jpeg(JC.content("photo", 1344, 1344, rng), grey=True, quality=95, optimize=True),
             JC.cv2_jpeg(JC.content("gradient", 2001, 1999, rng), 75, 411)]
    assert len(files[1]) > 20_000_000
    _check_equal(files, ops.decode_jpeg(files))


def test_output_independent_of_list_position_and_stream():
    from attwarp_b200 import ops
    files = JC.fuzz(40, seed=3)
    ref = [t.cpu() for t in ops.decode_jpeg(files)]
    perm = np.random.default_rng(0).permutation(len(files))
    for k, t in zip(perm, ops.decode_jpeg([files[k] for k in perm])):
        assert torch.equal(t.cpu(), ref[k])
    for k in (0, 17, 39):
        assert torch.equal(ops.decode_jpeg([files[k]])[0].cpu(), ref[k])
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        outs = ops.decode_jpeg(files[::-1])
    s.synchronize()
    for k, t in enumerate(outs[::-1]):
        assert torch.equal(t.cpu(), ref[k])


def _decode_into(files, dsts, shapes):
    """attwarp_decode_jpeg straight into the given device addresses."""
    from attwarp_b200 import _lib, ops
    lib = _lib.load()
    n = len(files)
    blob = np.frombuffer(b"".join(files), dtype=np.uint8).copy()
    dev = torch.from_numpy(blob).cuda()
    offs = np.concatenate([[0], np.cumsum([len(b) for b in files])])
    table = np.zeros(n, dtype=ops._JPEG_DTYPE)
    table["host"] = blob.ctypes.data + offs[:-1]
    table["dev"] = dev.data_ptr() + offs[:-1]
    table["nbytes"] = [len(b) for b in files]
    table["dst"] = dsts
    table["H"] = [s[0] for s in shapes]
    table["W"] = [s[1] for s in shapes]
    tp = table.ctypes.data_as(C.c_void_p)
    ws = torch.empty(lib.attwarp_jpeg_workspace_bytes(tp, n), dtype=torch.uint8, device="cuda")
    status = torch.full((n,), -7, dtype=torch.int32, device="cuda")
    _lib.check(lib.attwarp_decode_jpeg(tp, n, _lib.ptr(ws), ws.numel(), _lib.ptr(status), _lib.current_stream()))
    torch.cuda.synchronize()
    return status.cpu().numpy()


def test_rows_at_odd_byte_offsets_and_guard_bytes():
    files = JC.fuzz(24, seed=5, max_side=90)
    shapes = [JC.pillow_bgr(b).shape for b in files]
    guard = 37
    sizes = [int(np.prod(s)) for s in shapes]
    starts, at = [], 1                                  # every buffer at an odd offset, guards between them
    for sz in sizes:
        at += guard
        at += 1 - at % 2
        starts.append(at)
        at += sz
    buf = torch.full((at + guard,), 0xA5, dtype=torch.uint8, device="cuda")
    status = _decode_into(files, [buf.data_ptr() + s for s in starts], shapes)
    assert not status.any()
    host = buf.cpu().numpy()
    mask = np.ones(host.size, bool)
    for b, s, sz, shp in zip(files, starts, sizes, shapes):
        assert np.array_equal(host[s:s + sz].reshape(shp), JC.pillow_bgr(b))
        mask[s:s + sz] = False
    assert np.all(host[mask] == 0xA5)


def _corruptions():
    img = JC.content("photo", 120, 136, np.random.default_rng(8))
    plain = JC.pil_jpeg(img, quality=90)
    rst = JC.pil_jpeg(img, quality=90, restart_marker_blocks=3)
    a, e = JC.scan_range(plain)
    bad_code = plain[:a + 200] + b"\xff\x00" * 8 + plain[a + 216:]
    short = plain[:a + (e - a) // 3] + b"\xff\xd9"
    i = rst.index(b"\xff\xd4", JC.scan_range(rst)[0])
    no_rst = rst[:i] + rst[i + 2:]
    ra, _ = JC.scan_range(rst)
    swapped = bytearray(rst)
    j = rst.index(b"\xff\xd1", ra)
    k = rst.index(b"\xff\xd2", ra)
    swapped[j + 1], swapped[k + 1] = 0xD2, 0xD1
    return plain, {"bad_code": (bad_code, 2), "short": (short, 1), "no_rst": (no_rst, 4),
                   "rst_out_of_order": (bytes(swapped), 4)}


@pytest.mark.parametrize("kind", ["bad_code", "short", "no_rst", "rst_out_of_order"])
def test_malformed_entropy_data_names_the_file(kind):
    from attwarp_b200 import ops
    plain, cases = _corruptions()
    bad, code = cases[kind]
    with pytest.raises(ValueError, match=f"file 2 has malformed entropy-coded data.*status {code}"):
        ops.decode_jpeg([plain, plain, bad, plain])


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    """The sequential decode of tests/hostcheck/jpeg_hostcheck.cpp (jpeg_decode.h on the host)."""
    import shutil
    import subprocess
    gxx = shutil.which("g++")
    if gxx is None:
        pytest.skip("g++ not available")
    out = tmp_path_factory.mktemp("jpeg_hostcheck") / "libjpeghostcheck.so"
    subprocess.check_call([gxx, "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                           os.path.join(os.path.dirname(os.path.abspath(__file__)), "hostcheck", "jpeg_hostcheck.cpp")])
    return C.CDLL(str(out))


# Largest |coefficient x quantisation step| a forward DCT of 8-bit samples gives is about 1024 (the DC of a flat
# block); twice that leaves room for encoder rounding.
DCT_RANGE = 2048


def test_flipped_bytes_never_give_silent_pixels(hc):
    """A flipped byte inside the scan either fails with ValueError or is a valid stream of other codes.  The device
    then equals the sequential restatement of libjpeg's C code, and Pillow too while the coefficients stay in the
    range a forward DCT of 8-bit samples yields.

    Finding: beyond that range (|coefficient x step| of 3241 and more here; valid encoder output stays near 1024)
    Pillow's libjpeg-turbo differs from its own C ISLOW IDCT -- its SIMD IDCT keeps 16-bit intermediates -- and the
    device follows the C code.  No file an encoder writes from 8-bit samples reaches that range."""
    from attwarp_b200 import ops
    rng = np.random.default_rng(4)
    img = JC.content("photo", 96, 112, rng)
    base = JC.pil_jpeg(img, quality=85)
    a, e = JC.scan_range(base)
    failed = same = beyond = 0
    for _ in range(60):
        b = bytearray(base)
        p = int(rng.integers(a + 1, e - 1))
        if b[p] == 0xFF or b[p - 1] == 0xFF:
            continue
        b[p] = int(rng.integers(0, 255))
        if b[p] == 0xFF:
            continue
        b = bytes(b)
        try:
            out = ops.decode_jpeg([b])[0].cpu().numpy()
        except ValueError as exc:
            assert "file 0 has malformed" in str(exc)
            failed += 1
            continue
        ref = np.zeros_like(out)
        mx = C.c_int32()
        assert hc.hc_jpeg_decode(b, len(b), ref.ctypes.data_as(C.c_void_p), C.byref(mx)) == 0
        assert np.array_equal(out, ref)
        if mx.value <= DCT_RANGE:
            assert np.array_equal(out, JC.pillow_bgr(b))
            same += 1
        else:
            beyond += 1
    assert failed > 0 and same > 0 and beyond > 0


def test_decode_jpeg_batch_routes_every_file_to_an_exact_decoder(tmp_path):
    import io

    from PIL import Image

    from attwarp_b200 import image_io
    rng = np.random.default_rng(12)
    imgs = [JC.content("photo", 70 + 9 * k, 90 - 7 * k, rng) for k in range(6)]
    cmyk = io.BytesIO()
    Image.fromarray(imgs[2][..., ::-1]).convert("CMYK").save(cmyk, "JPEG", quality=90)
    png = cv2.imencode(".png", imgs[3])[1].tobytes()
    srcs = [JC.pil_jpeg(imgs[0], quality=90), JC.pil_jpeg(imgs[1], quality=90, progressive=True), cmyk.getvalue(),
            png, JC.cv2_jpeg(imgs[4], 80, 422), JC.pil_jpeg(imgs[5], grey=True, quality=70)]
    path = tmp_path / "f.jpg"
    path.write_bytes(srcs[4])
    srcs[4] = str(path)
    outs = image_io.decode_jpeg_batch(srcs, exact_device=True)
    for k, (s, t) in enumerate(zip(srcs, outs)):
        b = s if isinstance(s, bytes) else open(s, "rb").read()
        ref = cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR) if k == 3 else JC.pillow_bgr(b)
        assert t.dtype == torch.uint8 and t.is_cuda
        assert np.array_equal(t.cpu().numpy(), ref), k


@pytest.mark.parametrize("mode", ["index", "mota", "att"])
def test_warp_files_exact_decode_writes_the_exact_decodes_files(tmp_path, mode):
    from attwarp_b200 import image_io
    rng = np.random.default_rng(21)
    shapes = [(120, 160), (97, 131), (64, 64), (150, 90)]
    jpgs, pngs = [], []
    for k, (h, w) in enumerate(shapes):
        b = JC.pil_jpeg(JC.content("photo", h, w, rng), quality=88, subsampling=2 if k % 2 else 0)
        p = tmp_path / f"in{k}.jpg"
        p.write_bytes(b)
        jpgs.append(str(p))
        q = tmp_path / f"in{k}.png"              # Pillow's pixels, losslessly: what the exact host decode gives
        cv2.imwrite(str(q), JC.pillow_bgr(b))
        pngs.append(str(q))
    n = len(shapes)
    tok = torch.rand(n, 24, 24, generator=torch.Generator().manual_seed(1)) if mode != "att" else None
    att = [rng.integers(0, 256, s, dtype=np.uint8) for s in shapes] if mode == "att" else None
    kw = dict(mask="mota" if mode == "mota" else "index", att=att, out_sizes=[(100, 110)] * n)

    def run(srcs, tag, exact):
        outs = [str(tmp_path / f"{tag}_w{k}.png") for k in range(n)]
        ovs = [str(tmp_path / f"{tag}_o{k}.png") for k in range(n)]
        ors = [str(tmp_path / f"{tag}_g{k}.png") for k in range(n)]
        ok = image_io.warp_files(srcs, tok, outs, overlay_paths=ovs, original_paths=ors, exact_decode=exact, **kw)
        assert all(ok)
        return [cv2.imread(p, cv2.IMREAD_UNCHANGED) for p in outs + ovs + ors]

    got = run(jpgs, "dev", True)
    ref = run(pngs, "ref", False)
    for k, (g, r) in enumerate(zip(got, ref)):
        assert np.array_equal(g, r), k
    for k, b in enumerate(jpgs):
        assert np.array_equal(got[2 * n + k], JC.pillow_bgr(open(b, "rb").read()))
