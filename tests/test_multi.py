"""Multi-process tests of the N > 1 path: a gloo world_size-2 run on CPU (host logic + exchange
plan under real message passing) and, when at least two GPUs are visible, the NCCL path against
the oracle's virtual ranks."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import bp4_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _torchrun(script, nproc, port, timeout=600):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", script)]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, cwd=ROOT)


def test_gloo_world_size_2_exchange_plan():
    from mf_data_locality_b200 import build
    build.build_all()
    r = _torchrun("gloo_worker.py", 2, 29731)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert "gloo ok" in r.stdout


def test_virtual_ranks_equal_single_rank():
    """oracle self-consistency: N virtual ranks with emulated exchange == 1 rank on the same field"""
    p, s = 3, 6
    t = O.make_tables(p)
    rd1 = O.build_problem(p, s)[0]
    rng = np.random.default_rng(0)
    field = np.zeros((rd1.node_of_local.max() + 1, 3))
    field[rd1.node_of_local] = rng.standard_normal((len(rd1.node_of_local), 3))
    y1 = np.zeros_like(field)
    y1[rd1.node_of_local] = O.vmult(rd1, t, field[rd1.node_of_local].ravel()).reshape(-1, 3)
    for nr in (2, 4):
        rds = O.build_problem(p, s, n_ranks=nr)
        srcs = [np.concatenate([field[rd.node_of_local[: rd.n_owned // 3]].ravel(), np.zeros(rd.n_ghost)]) for rd in rds]
        ys = O.multi_vmult(rds, t, srcs)
        for y, rd in zip(ys, rds):
            assert np.allclose(y[: rd.n_owned].reshape(-1, 3), y1[rd.node_of_local[: rd.n_owned // 3]], atol=1e-12)


@pytest.mark.gpu
def test_nccl_two_gpus_against_virtual_rank_oracle():
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    r = _torchrun("mgpu_worker.py", 2, 29741, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    assert r.stdout.count("mgpu ok") == 4
