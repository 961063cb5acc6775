"""bench.py on a machine without a GPU: the CUDA arm refuses to run (no CPU fallback), the reference arm
(the unmodified reference on the host cores, oracle/_ref) prints the one JSON line of the contract."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_the_contract_line():
    from oracle.pyoracle import ref_available
    if not ref_available():
        pytest.skip("oracle/_ref not built")
    out = run_bench("--impl", "reference", "--steps", "1", "--warmup", "1")
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "Mrays/s" and d["higher_is_better"] is True
    assert d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["value"] == d["value"] == d["e2e"]["value"]
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_cuda_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is visible")
    out = run_bench("--steps", "1", "--warmup", "1")
    assert out.returncode != 0
    assert "no CPU fallback" in (out.stdout + out.stderr)
    assert not any(l.startswith("{") for l in out.stdout.splitlines())


def test_gather_form_follows_the_rank_count():
    """bench.py --gather auto: the delivery form of the fused gather is chosen by the number of ranks as measured
    (DESIGN.md §7), an explicit request is taken literally, one rank and `nccl` mean the NCCL / plain path."""
    sys.path.insert(0, ROOT)
    import bench
    assert bench.gather_candidates(1, "auto") == [] and bench.gather_candidates(8, "nccl") == []
    assert bench.gather_candidates(2, "auto")[0] == "multicast"
    assert bench.gather_candidates(3, "auto")[0] == "direct" and bench.gather_candidates(4, "auto")[0] == "direct"
    assert bench.gather_candidates(8, "auto") == ["multicast_staged", "peer", "direct"]        # falls back when there is no multicast address
    for mode in ("multicast", "multicast_staged", "peer", "direct"):
        assert bench.gather_candidates(8, mode) == [mode]


def test_dump_outputs_writes_a_fixed_sample_as_floats(tmp_path):
    """bench.py --dump-outputs: float32 / float64 arrays only, at most 64 MB, and for a batch larger than DUMP_MAX_RAYS the
    same seeded sample every time, each record next to the index of its ray."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from bvh_b200.api import HIT3F
    n = bench.DUMP_MAX_RAYS + 4321
    rec = np.zeros(n, HIT3F)
    rec["prim_id"] = np.arange(n)
    rec["prim_id"][::7] = 0xFFFFFFFF
    rec["t"], rec["u"], rec["v"] = np.arange(n) * 0.5, np.arange(n) * 0.25, np.arange(n) * 0.125
    hits = torch.from_numpy(rec.view(np.int32).reshape(n, 4))
    for out in ("a", "b"):
        bench.dump_outputs(str(tmp_path / out), hits, HIT3F)
    total = 0
    got = {}
    for name in ("prim_id", "t", "u", "v", "ray_index"):
        a, b = np.load(tmp_path / "a" / f"{name}.npy"), np.load(tmp_path / "b" / f"{name}.npy")
        assert a.dtype in (np.float32, np.float64) and a.shape == (bench.DUMP_MAX_RAYS,) and np.array_equal(a, b)
        total += a.nbytes
        got[name] = a
    assert total <= 64 << 20
    index = got["ray_index"].astype(np.int64)
    assert (np.diff(index) > 0).all() and index[-1] < n
    assert np.array_equal(got["prim_id"], rec["prim_id"][index].astype(np.float64))
    assert (got["prim_id"][index % 7 == 0] == 0xFFFFFFFF).all()
    for name in ("t", "u", "v"):
        assert np.array_equal(got[name], rec[name][index])
