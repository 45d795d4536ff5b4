#!/usr/bin/env python
"""Cost of CeedOperatorLinearAssembleDiagonal for user QFunctions (K14) at C3 (hyperFS, p = 4, 64^3 box; the three
p-multigrid levels (P, Q) = (5, 5), (3, 5), (2, 5)), in one run on one card:

  * K3, the built-in diagonal from the Jacobian cache;
  * K14 around oracle/qf_port.c:port_HyperFSdF, at 2, 3 and 4 blocks per SM asked of ptxas (B200_JIT_DIAG_CTAS);
  * the generic path on the same QFunction: the operator built with its passive vectors (qdata, gradu) in a plain
    [elem][comp][q] layout, which K12 does not take (9 unit-input passes of K11 and an accumulation each);
  * the relative differences of the diagonals, K14 vs K3 and K14 vs generic;
  * the NVRTC compile time of the K14 program, cold and cached;
  * device-wide free memory (torch.cuda.mem_get_info) before and after the first diagonal, K14 vs generic;
  * Newton and CG counts of a tube:8,64,48 solve (degree 4, 4 load steps, coarse="amg") with the port_HyperFS*
    models, run twice in one process (the first run compiles), beside the built-in model's.
Timings are the best of 3 alternating batches after a warm-up.  Prints the card name and power limit and one JSON
line; --out appends it to a file.
  python tools/jit_diag_time.py [--n 64] [--reps 5] [--out profiles/jit_diag_c3.jsonl]"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ceedpetscsolid_b200 import ceed as libceed  # noqa: E402
from ceedpetscsolid_b200 import setuplibceed  # noqa: E402
from ceedpetscsolid_b200.ceed import BASIS_COLLOCATED, EVAL_GRAD, EVAL_NONE, VECTOR_ACTIVE  # noqa: E402
from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement  # noqa: E402

QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
LOCS = {"apply": f"{QF_PORT}:port_HyperFSF", "jacob": f"{QF_PORT}:port_HyperFSdF"}
CTAS = [2, 3, 4]


def timeit(fn, reps, warm=1):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else f"{torch.cuda.get_device_name(0)} (nvidia-smi unavailable)"


def compile_times():
    """cold: a copy of qf_port.c under a fresh path (another #line, so another program); cached: the same again"""
    tmp = tempfile.mkdtemp(prefix="jit_diag_time_")
    try:
        out = {}
        for tag in ("first", "second"):
            src = os.path.join(tmp, f"qf_port_{tag}.c")
            shutil.copy(QF_PORT, src)
            t0 = time.perf_counter()
            libceed.jit_diag_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 5, 5)
            out[f"k14_compile_cold_{tag}_s"] = time.perf_counter() - t0
        n0 = libceed.jit_compile_count()
        t0 = time.perf_counter()
        for _ in range(100):
            libceed.jit_diag_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 5, 5)
        out["k14_compile_cached_s"] = (time.perf_counter() - t0) / 100
        assert libceed.jit_compile_count() == n0
        return out
    finally:
        shutil.rmtree(tmp)


def diag_vec(ceed, n):
    d = torch.zeros(n, dtype=torch.float64, device="cuda")
    dc = ceed.Vector(n)
    dc.set_array(d)
    return d, dc


def stack(mesh, u, jit):
    """set-up at p = 4 with its levels; the fine residual applied at u (gradu of the linearisation point)"""
    ceed = libceed.Ceed("/gpu/b200:jit" if jit else "/gpu/b200")
    degrees, data, phys = setuplibceed.setup_all(ceed, mesh, "hyperFS", 4, qf_locators=LOCS if jit else None)
    assert degrees == [1, 2, 4]
    for d in data:
        assert d.opJacob.is_jit_fused if jit else d.opJacob.is_fused
    r = torch.zeros_like(u)
    uc, rc = ceed.Vector(u.numel()), ceed.Vector(u.numel())
    uc.set_array(u)
    rc.set_array(r)
    data[-1].opApply.apply(uc, rc)
    diags = [diag_vec(ceed, 3 * mesh.num_nodes(deg)) for deg in degrees]
    torch.cuda.synchronize()
    return SimpleNamespace(ceed=ceed, data=data, phys=phys, ops=[d.opJacob for d in data], diags=diags,
                           keep=(uc, rc, r))


def generic_ops(S, mesh):
    """the port Jacobian of every level of stack S with qdata and gradu re-laid [elem][comp][q] on explicitly strided
    restrictions: K12 refuses such passive vectors, so the operators run on the generic path"""
    fine = S.data[-1]
    nelem, nq = mesh.nelem, 125
    ceed = S.ceed
    plain = {}
    for name, r, v, nc in (("qdata", fine.Erestrictqdi, fine.qdata, 10), ("gradu", fine.ErestrictGradui, fine.gradu, 9)):
        ev = ceed.Vector(nelem * nc * nq)
        r.apply(v, ev)                     # the E-vector of a backend-strided restriction is [elem][comp][q]
        rp = ceed.StridedElemRestriction(nelem, nq, nc, nelem * nc * nq, strides=[1, nq, nc * nq])
        plain[name] = (rp, ev)
    ops = []
    for d in S.data:
        qf = ceed.QFunction(1, LOCS["jacob"])
        qf.add_input("deltadu", 9, EVAL_GRAD)
        qf.add_input("qdata", 10, EVAL_NONE)
        qf.add_input("gradu", 9, EVAL_NONE)
        qf.add_output("deltadv", 9, EVAL_GRAD)
        qf.set_context(S.phys)
        op = ceed.Operator(qf)
        op.set_field("deltadu", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
        op.set_field("qdata", plain["qdata"][0], BASIS_COLLOCATED, plain["qdata"][1])
        op.set_field("gradu", plain["gradu"][0], BASIS_COLLOCATED, plain["gradu"][1])
        op.set_field("deltadv", d.Erestrictu, d.basisu, VECTOR_ACTIVE)
        assert not op.is_jit_fused and not op.is_fused
        ops.append((op, qf))
    return ops, plain


def first_diag_memory(ops, diags):
    """device-wide free memory before and after the first diagonal of every level"""
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info()[0]
    for op, (_, dc) in zip(ops, diags):
        op.linear_assemble_diagonal(dc)
    torch.cuda.synchronize()
    return (free0 - torch.cuda.mem_get_info()[0]) / 1e9


def tube_solves():
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    from ceedpetscsolid_b200.exodus import tube_mesh
    m = tube_mesh(8, 64, 48)
    ext = float(np.ptp(m.vertices, axis=0).max())
    out = {}
    # the port models from a copy of qf_port.c under a path of their own: programs this process has not compiled yet,
    # so the first port run pays every NVRTC compile of a fresh solve and the second finds them cached
    tmp = tempfile.mkdtemp(prefix="jit_diag_tube_")
    src = os.path.join(tmp, "qf_port.c")
    shutil.copy(QF_PORT, src)
    locs_t = {"apply": f"{src}:port_HyperFSF", "jacob": f"{src}:port_HyperFSdF"}
    for tag, locs in (("builtin", None), ("port_first", locs_t), ("port_second", locs_t)):
        app = AppCtx(problem="hyperFS", degree=4, num_steps=4, mesh=m,
                     clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.05 * ext, 0.1 * ext, 0, 0, 1, 0]})
        n0 = libceed.jit_compile_count()
        t0 = time.perf_counter()
        el = Elasticity(app, coarse="amg", qf_locators=locs)
        build = time.perf_counter() - t0
        r = el.solve()
        out[tag] = dict(snes_its=r["snes_its"], ksp_its=r["ksp_its"], converged=r["converged"], time_s=r["time_s"],
                        stack_build_s=build, nvrtc_compiles=libceed.jit_compile_count() - n0)
        out[tag]["U"] = el.U.clone()
        del el
    for tag in ("port_first", "port_second"):
        out[f"rel_diff_U_{tag}"] = (torch.linalg.norm(out[tag]["U"] - out["builtin"]["U"]) /
                                    torch.linalg.norm(out["builtin"]["U"])).item()
    for tag in ("builtin", "port_first", "port_second"):
        del out[tag]["U"]
    shutil.rmtree(tmp)
    return out


def rel(a, b):
    return (torch.linalg.norm(a - b) / torch.linalg.norm(b)).item()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-tube", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/jit_diag_time.py measures on the GPU"
    card = gpu_info()
    print("card:", card, flush=True)
    res = {"case": f"C3 hyperFS p=4 {a.n}^3, levels (P, Q) = (5, 5), (3, 5), (2, 5)", "card": card}
    res.update(compile_times())

    mesh = BoxMesh(n=(a.n,) * 3, perturb=0.08, seed=0)
    res["elements"] = mesh.nelem
    u = torch.from_numpy(smooth_displacement(mesh.node_coords(4)).reshape(-1)).cuda()
    runs = {"k3_builtin": stack(mesh, u, False)}
    for R in runs.values():
        for op, (_, dc) in zip(R.ops, R.diags):
            op.linear_assemble_diagonal(dc)
    env0 = os.environ.get("B200_JIT_DIAG_CTAS")
    for ctas in CTAS:   # read by the K14 compile at each operator's first diagonal
        os.environ["B200_JIT_DIAG_CTAS"] = str(ctas)
        tag = f"k14_ctas{ctas}"
        runs[tag] = stack(mesh, u, True)
        mem = first_diag_memory(runs[tag].ops, runs[tag].diags)
        if ctas == CTAS[0]:
            res["first_diagonal_device_mem_gb_device_wide"] = {"k14": mem}
    if env0 is None:
        os.environ.pop("B200_JIT_DIAG_CTAS", None)
    else:
        os.environ["B200_JIT_DIAG_CTAS"] = env0
    G = runs[f"k14_ctas{CTAS[0]}"]
    gops, plain = generic_ops(G, mesh)
    gdiags = [diag_vec(G.ceed, d.numel()) for d, _ in G.diags]
    runs["generic"] = SimpleNamespace(ops=[op for op, _ in gops], diags=gdiags)
    res["first_diagonal_device_mem_gb_device_wide"]["generic"] = first_diag_memory(runs["generic"].ops, gdiags)

    names = ["(5,5)", "(3,5)", "(2,5)"]
    levels = [2, 1, 0]
    t = {f"{tag} {names[i]}": [] for tag in runs for i in range(3)}
    for _ in range(3):                     # alternate every variant and level
        for tag, R in runs.items():
            for i, lv in enumerate(levels):
                op, (_, dc) = R.ops[lv], R.diags[lv]
                t[f"{tag} {names[i]}"].append(timeit(lambda: op.linear_assemble_diagonal(dc), a.reps))
    res["diagonal_ms"] = {k: min(v) for k, v in t.items()}
    res["diagonal_ms_all"] = t
    for i, lv in enumerate(levels):
        for tag, R in runs.items():            # one more diagonal each, into fresh values, for the comparison
            R.diags[lv][0].zero_()
            R.ops[lv].linear_assemble_diagonal(R.diags[lv][1])
        torch.cuda.synchronize()
        k3 = runs["k3_builtin"].diags[lv][0]
        for tag in runs:
            if tag.startswith("k14"):
                res[f"rel_diff_{tag}_vs_k3 {names[i]}"] = rel(runs[tag].diags[lv][0], k3)
        res[f"rel_diff_k14_vs_generic {names[i]}"] = rel(G.diags[lv][0], runs["generic"].diags[lv][0])
    del runs, G, gops, plain
    torch.cuda.empty_cache()
    if not a.no_tube:
        res["tube_8_64_48_amg_p4"] = tube_solves()
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
