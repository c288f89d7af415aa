"""CPU: the host-side pieces of bench.py that do not need a GPU -- workload table, the stdout guard used
around NCCL initialisation, the --dump-outputs sampler, and the clock sampler degrading to None when neither
NVML nor nvidia-smi exists."""

import importlib.util
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


def _bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_workloads_cover_the_baseline_configs():
    b = _bench()
    assert set(b.WORKLOADS) == {"c2", "c3", "c4", "c5"}
    assert b.WORKLOADS["c2"]["B"] == 256 and b.WORKLOADS["c2"]["side"] == 336 and b.WORKLOADS["c2"]["has_attention"]
    assert b.WORKLOADS["c3"]["B"] == 64 and b.WORKLOADS["c3"]["side"] == 1344
    assert b.WORKLOADS["c4"]["B"] == 1024 and b.WORKLOADS["c4"].get("ragged")
    assert b.WORKLOADS["c5"]["B"] == 128 and b.WORKLOADS["c5"]["side"] == 512 and b.WORKLOADS["c5"].get("pdf")


def test_stdout_guard_sends_library_output_to_stderr():
    code = (
        "import importlib.util, os, sys\n"
        f"spec = importlib.util.spec_from_file_location('b', r'{os.path.join(ROOT, 'bench.py')}')\n"
        "b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b)\n"
        "print('line-1')\n"
        "with b._StdoutToStderr():\n"
        "    os.write(1, b'banner from a C library\\n')\n"
        "print('line-2')\n")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    assert r.stdout.split() == ["line-1", "line-2"]
    assert "banner from a C library" in r.stderr


def test_dump_sample_is_a_fixed_sample_of_the_concatenated_outputs(tmp_path):
    import numpy as np
    import torch
    b = _bench()
    g = torch.Generator().manual_seed(0)
    ts = [torch.randint(0, 256, (s, s + 1, 3), dtype=torch.uint8, generator=g) for s in (3, 40, 7)]
    flat = np.concatenate([t.numpy().reshape(-1) for t in ts]).astype(np.float32)
    assert np.array_equal(b.dump_sample(ts, flat.size), flat)
    got = b.dump_sample(ts, 500)
    assert got.dtype == np.float32 and got.size == 500
    assert np.array_equal(got, b.dump_sample(ts, 500))                  # the same positions in every run
    assert np.array_equal(got, flat[np.sort(np.random.default_rng(0).integers(0, flat.size, 500))])
    b.write_dumps(str(tmp_path), {"c4": {"out": got}})
    assert np.array_equal(np.load(tmp_path / "c4_out.npy"), got)


def test_clock_sampler_without_a_gpu_is_none_not_an_error():
    b = _bench()
    s = b.ClockSampler(0, None)
    s.start()
    out = s.stop()
    assert out is None or ("sm_mhz" in out and "reasons" in out)
