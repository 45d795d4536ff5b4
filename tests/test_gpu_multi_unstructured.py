"""Unstructured tube meshes on several GPUs (skipped on boxes with fewer GPUs): partitioned Jacobian against the
serial oracle with NCCL and peer-memory halos, and the partitioned Newton-Krylov-p-MG solve with Jacobi-PCG and with
the redundant AMG coarse solve against the one-GPU run.  One torchrun rank per GPU (tests/mgpu_unstructured_check.py)."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(world, *args):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--local-addr", "127.0.0.1", "--nnodes=1",
           f"--nproc-per-node={world}", os.path.join(ROOT, "tests", "mgpu_unstructured_check.py")] + list(args)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert len(lines) == 1, r.stdout[-3000:]
    return json.loads(lines[0][len("RESULT "):])


@pytest.mark.parametrize("halo", ["nccl", "p2p"])
@pytest.mark.parametrize("world", [2, 4, 8])
def test_partitioned_tube_jacobian_matches_oracle(world, halo):
    rec = _run(world, "jacobian", halo)
    assert rec["rel_err"] <= 1e-12, rec
    assert rec["covered"] and rec["bc_rows_zero"] and not rec["halo_failed"], rec
    assert rec["shared_dofs"] > 0 and rec["bitwise"], rec


@pytest.mark.parametrize("coarse", ["pcg", "amg"])
def test_partitioned_tube_solve_matches_one_gpu(coarse):
    two = _run(2, "solve", coarse)
    one = _run(1, "solve", coarse)
    assert two["ran"] == ("RedundantAMG" if coarse == "amg" else "pcg"), two
    assert one["converged"] and two["converged"], (one, two)
    assert two["snes_its"] == one["snes_its"], (one, two)
    assert abs(two["ksp_its"] - one["ksp_its"]) <= 0.25 * one["ksp_its"], (one, two)
    assert abs(two["strain_energy"] - one["strain_energy"]) <= 1e-8 * abs(one["strain_energy"]), (one, two)


@pytest.mark.parametrize("world", [1, 2, 4])
def test_redundant_amg_on_the_device_equals_the_one_rank_amg_bit_for_bit(world):
    rec = _run(world, "redundant")
    assert rec["levels"] >= 2 and rec["bit_identical"], rec


def test_partitioned_tube_amg_solve_is_bit_identical_in_deterministic_mode():
    rec = _run(2, "solve", "amg", "deterministic")
    assert rec["converged"] and rec["bit_identical_rerun"], rec
