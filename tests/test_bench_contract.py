"""Checks of bench.py: the size/byte helpers against SURVEY App. C / 8(d), the JSON line of the
`--impl reference` arm (the CPU restatement on a tiny sample), rank > 0 staying silent, the loud
failure of the product arm without a GPU, and what --dump-outputs writes."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import bp4_oracle as O

from helpers import rel_l2, single

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_module():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_size_and_byte_helpers():
    b = _bench_module()
    # SURVEY App. C: (p, s) -> DoFs, cells
    assert b.n_dofs_of(3, 15) == (2738019, 32768)
    assert b.n_dofs_of(4, 18) == (50923779, 262144)
    assert b.n_dofs_of(6, 18) == (171199875, 262144)
    assert b.n_dofs_of(4, 22) == (809244675, 1 << 22)
    # SURVEY 8(d): merged Q4 60.2 B/DoF/it, plain 138.67 B/DoF + metadata
    nd, nc = b.n_dofs_of(4, 18)
    assert abs(b.algorithmic_bytes_per_iteration(4, 18) / nd - 60.2) < 0.05
    assert abs(b.algorithmic_bytes_per_iteration(4, 18, merged=False) / nd - (138.667 + 300.0 * nc / nd)) < 1e-2


def _run(extra_env=None, *args):
    env = dict(os.environ)
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          env=env, timeout=600, cwd=ROOT)


def test_reference_arm_json_line(c_oracle_lib):
    r = _run(None, "--impl", "reference", "--steps", "1", "--warmup", "1", "--degree", "3", "--s", "6", "--cpu-s", "6")
    assert r.returncode == 0, r.stderr
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "GDoF/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["n_gpus"] == 1
    assert d["dtype"] == "f64" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and "s=6" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GDoF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_are_silent():
    r = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--impl", "reference", "--gpus", "2", "--steps", "1",
             "--warmup", "1", "--degree", "3", "--s", "6", "--cpu-s", "6")
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_fails_loudly_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = _run({"CUDA_VISIBLE_DEVICES": ""}, "--steps", "1", "--warmup", "1", "--degree", "3", "--s", "6",
             "--no-cpu-baseline")
    assert r.returncode != 0          # no CPU fallback, no JSON line
    assert not any(ln.startswith("{") for ln in r.stdout.splitlines())


def test_dump_outputs_files(tmp_path):
    """float64 .npy files of 64 MB at most; a long solution is sampled at the same positions on
    every call, a short one is written whole"""
    b = _bench_module()
    x = np.arange(3 * b.DUMP_MAX_ENTRIES, dtype=np.float64)
    for d in ("a", "b"):
        b.dump_outputs(str(tmp_path / d), x, 37)
    xa, xb = np.load(tmp_path / "a" / "x.npy"), np.load(tmp_path / "b" / "x.npy")
    assert xa.dtype == np.float64 and xa.size == b.DUMP_MAX_ENTRIES and np.array_equal(xa, xb)
    assert np.all(np.diff(xa) > 0) and 0 <= xa[0] and xa[-1] < x.size     # distinct entries of x
    it = np.load(tmp_path / "a" / "iterations.npy")
    assert it.dtype == np.float64 and it.tolist() == [37.0]
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 64 << 20
    short = np.random.default_rng(1).standard_normal(1000)
    b.dump_outputs(str(tmp_path / "c"), short, 5)
    assert np.array_equal(np.load(tmp_path / "c" / "x.npy"), short)


def test_dump_outputs_rejected_for_reference_arm(tmp_path):
    r = _run(None, "--impl", "reference", "--dump-outputs", str(tmp_path / "d"))
    assert r.returncode != 0 and "--dump-outputs" in r.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_dump_outputs_hold_the_solution(tmp_path, c_oracle_lib):
    """bench.py --dump-outputs on a small mesh: the dumped solution and iteration count are those
    of the C oracle's merged CG, and --steps sets the number of timed solves"""
    out = tmp_path / "dump"
    r = _run(None, "--steps", "2", "--warmup", "1", "--degree", "3", "--s", "6", "--sweep", "none",
             "--no-cpu-baseline", "--dump-outputs", str(out))
    assert r.returncode == 0, r.stderr
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][-1])
    x, it = np.load(out / "x.npy"), np.load(out / "iterations.npy")
    assert d["steps"] == 2 and abs(d["iterations_per_step"] - int(it[0])) <= 1
    rd, co = single(3, 6)
    xo, ito, _ = co.cg(rd.rhs, O.finish_inverse_diagonal(O.inverse_diagonal(rd)), merged=True)
    assert abs(int(it[0]) - ito) <= 1
    assert rel_l2(x, xo) <= (1e-8 if ito < 100 else 1e-6)
