"""Partitioned runs on an unstructured tube mesh, one rank per GPU; rank 0 prints one JSON line.

    torchrun --standalone --nproc-per-node 2 tests/mgpu_unstructured_check.py jacobian nccl
    torchrun --standalone --nproc-per-node 2 tests/mgpu_unstructured_check.py solve amg [deterministic]
    torchrun --standalone --nproc-per-node 1 tests/mgpu_unstructured_check.py redundant

jacobian HALO: the hyperFS p = 2 Jacobian MatMult on a coordinate-bisected tube (masked layout, interface-first element
order, halo overlapped) against the serial CPU oracle, and whether the interface copies are bit-identical.
solve COARSE: the hyperFS p = 2 Newton-Krylov-p-MG solve on tube:4,32,24 with the given coarse solve (pcg or amg);
with "deterministic" on /gpu/b200:deterministic, solved twice, and whether the two solutions are bit-identical.
redundant: the redundant AMG's hierarchy and V-cycle against the one-rank AMG of the global mesh, bit for bit.
Used by tests/test_gpu_multi_unstructured.py (which also runs it with one rank).
"""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _dofs(nodes):
    return (np.asarray(nodes)[:, None] * 3 + np.arange(3)[None, :]).reshape(-1)


def _gather_on_rank0(world, item):
    if world == 1:
        return [item]
    parts = [None] * world
    dist.all_gather_object(parts, item)
    return parts


def jacobian(rank, world, local, halo_mode, p=2, repeats=5):
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200 import matops, setuplibceed
    from ceedpetscsolid_b200.exodus import tube_mesh
    from ceedpetscsolid_b200.halo import Halo
    from ceedpetscsolid_b200.mesh import grid_for, smooth_displacement
    gmesh = tube_mesh(4, 32, 8, r0=0.6, r1=1.0, length=1.5)
    grid = grid_for(world)
    mesh = gmesh.brick(grid, rank, interface_first=True)
    ceed = libceed.Ceed(f"/gpu/b200:device_id={local}")
    degrees, data, phys = setuplibceed.setup_all(ceed, mesh, "hyperFS", p)
    fine = len(degrees) - 1
    halo = Halo(gmesh, grid, rank, p, dist)
    if halo_mode == "p2p" and not halo.enable_p2p():
        raise RuntimeError(f"peer-memory halo could not be set up: {halo._p2p_error}")
    dm = matops.LevelDM(mesh, p, bc_faces="all", halo=halo, masked=True)
    user = matops.setup_jacobian_ctx(dm, ceed, data[fine], phys)
    matops.OVERLAP_MIN_INTERIOR = 0      # exercise the overlapped exchange on this small mesh
    assert 0 < mesh.n_interface < mesh.nelem
    u = torch.from_numpy(smooth_displacement(mesh.node_coords(p)).reshape(-1)).cuda()
    uc, rc = ceed.Vector(u.numel()), ceed.Vector(u.numel())
    r = torch.zeros_like(u)
    uc.set_array(u); rc.set_array(r)
    data[fine].opApply.apply(uc, rc)
    uc.take_array(); rc.take_array()
    gdof = _dofs(mesh.node_ids(p))
    xglob = np.random.default_rng(5).standard_normal(gmesh.lsize(p))
    gbc = np.repeat(gmesh.boundary_mask(p, "all"), 3)
    xglob[gbc] = 0.0
    X, Y = dm.create_global_vector(), dm.create_global_vector()
    X.copy_(torch.from_numpy(xglob[gdof]))
    for _ in range(repeats):
        matops.ApplyJacobian_Ceed(user, X, Y)
    torch.cuda.synchronize()
    failed = halo.p2p_failed_anywhere()
    parts = _gather_on_rank0(world, (gdof, Y.cpu().numpy()))
    halo.close()
    if rank != 0:
        return None
    from helpers import OracleProblem, rel_err
    yref = OracleProblem("hyperFS", None, p, mesh=gmesh).jacobian(xglob)
    ypar = np.full_like(yref, np.nan)
    seen = np.zeros(yref.size, dtype=int)
    bitwise = True
    for d, v in parts:
        again = seen[d] > 0
        bitwise = bitwise and bool(np.array_equal(ypar[d][again], v[again]))
        ypar[d] = v
        seen[d] += 1
    free = ~gbc
    return {"check": "jacobian", "world": world, "halo": halo_mode, "elements": gmesh.nelem,
            "n_interface": mesh.n_interface, "rel_err": float(rel_err(ypar[free], yref[free])),
            "covered": bool(np.all(seen >= 1)), "bc_rows_zero": bool(np.all(ypar[gbc] == 0.0)),
            "bitwise": bitwise, "halo_failed": bool(failed), "shared_dofs": int((seen > 1).sum())}


def redundant(rank, world, local):
    """RedundantAMG on the device against SmoothedAggregationAMG of the global mesh, same element matrices (oracle):
    the hierarchy and the per-rank V-cycle output must be bit-identical (works with one rank too)"""
    from ceedpetscsolid_b200 import matops
    from ceedpetscsolid_b200.amg import RedundantAMG, SmoothedAggregationAMG
    from ceedpetscsolid_b200.exodus import tube_mesh
    from ceedpetscsolid_b200.halo import Halo
    from ceedpetscsolid_b200.mesh import grid_for
    from amg_helpers import CoarseStub, Coo, oracle_element_matrices

    def coo(mesh):
        c = Coo(mesh, oracle_element_matrices(mesh))
        c.elem_nodes, c._v = c.elem_nodes.cuda(), c._v.cuda()
        return c
    m = tube_mesh(4, 32, 8, r0=0.6, r1=1.0, length=1.5)
    grid = grid_for(world)
    sub = m.brick(grid, rank, interface_first=True)
    dm = matops.LevelDM(sub, 1, bc_faces=[1], halo=Halo(m, grid, rank, 1, dist), device="cuda", masked=True)
    amg = RedundantAMG(dm, sub, m, [1], dist, max_coarse=60)
    amg.setup(CoarseStub(coo(sub)))
    gdm = matops.LevelDM(m, 1, bc_faces=[1], device="cuda", masked=True)
    ref = SmoothedAggregationAMG(gdm, m, max_coarse=60)
    ref.setup(CoarseStub(coo(m)))
    bg = torch.from_numpy(np.random.default_rng(11).standard_normal(m.lsize(1))).cuda()
    gdm.zero_constrained(bg)
    xg = torch.zeros_like(bg)
    ref.solve(bg, xg)
    gdof = torch.from_numpy(_dofs(sub.node_ids(1))).cuda()
    b = bg[gdof].contiguous()
    x = torch.zeros_like(b)
    amg.solve(b, x)
    same = torch.tensor([1 if (len(amg.levels) == len(ref.levels) and torch.equal(x, xg[gdof]) and
                               all(torch.equal(a.A.vals, r.A.vals) for a, r in zip(amg.levels, ref.levels))) else 0],
                        device="cuda")
    if world > 1:
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
    return {"check": "redundant", "world": world, "levels": len(ref.levels), "bit_identical": bool(same.item())}


def solve(rank, world, local, coarse, deterministic):
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    from ceedpetscsolid_b200.exodus import tube_mesh
    m = tube_mesh(4, 32, 24)
    ext = float(np.ptp(m.vertices, axis=0).max())
    app = AppCtx(problem="hyperFS", degree=2, num_steps=2, mesh=m,
                 clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.05 * ext, 0.1 * ext, 0, 0, 1, 0]})
    el = Elasticity(app, dist=dist if world > 1 else None, rank=rank, world=world, device_id=local, coarse=coarse,
                    deterministic=deterministic)
    out = el.solve()
    energy = el.strain_energy()
    rec = {"check": "solve", "world": world, "coarse": coarse, "ran": type(el.pc.amg).__name__ if el.pc.amg else "pcg",
           "deterministic": deterministic, "converged": out["converged"], "snes_its": out["snes_its"],
           "ksp_its": out["ksp_its"], "strain_energy": energy, "time_s": out["time_s"]}
    if deterministic:
        U1 = el.U.clone()
        out2 = el.solve()
        same = torch.tensor([1 if (torch.equal(U1, el.U) and el.strain_energy() == energy
                                   and out2["ksp_its"] == out["ksp_its"]) else 0], device="cuda")
        if world > 1:
            dist.all_reduce(same, op=dist.ReduceOp.MIN)
        rec["bit_identical_rerun"] = bool(same.item())
    el.close()
    return rec if rank == 0 else None


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    if world > 1 or sys.argv[1] == "redundant":
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if sys.argv[1] == "redundant":
        rec = redundant(rank, world, local)
    elif sys.argv[1] == "jacobian":
        rec = jacobian(rank, world, local, sys.argv[2])
    else:
        rec = solve(rank, world, local, sys.argv[2], "deterministic" in sys.argv[3:])
    if rank == 0:
        rec["gpu"] = torch.cuda.get_device_name(local)
        print("RESULT " + json.dumps(rec), flush=True)
    if dist.is_initialized():
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
