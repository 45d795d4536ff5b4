#!/usr/bin/env python
"""Cost of CeedOperatorLinearAssemble for user QFunctions (K13) at C3 (hyperFS, p = 4, 64^3 box; the p = 1 level,
P = 2, Q = 5, 262 144 elements), in one run on one card:

  * K8, the element matrices of the built-in Jacobian from its cache;
  * K13 around oracle/qf_port.c:port_HyperFSdF, in variants: blocks per SM asked of ptxas (B200_JIT_ASSEMBLE_CTAS)
    and the 9 unit-input calls unrolled or rolled (B200_JIT_ASSEMBLE_UNROLL);
  * the colouring K13 replaces for the same JIT operator: 81 K12 applies through ColoredCoarseMatrix.assemble;
  * the relative difference of the K13 and K8 matrices;
  * the NVRTC compile time of the K13 program, cold and cached;
  * Newton, CG and seconds of a tube:8,64,48 solve (degree 4, 4 load steps, coarse="amg") with the port_HyperFS*
    models beside the built-in model's.
Timings are the best of 3 alternating batches after a warm-up.  Prints the card name and power limit and one JSON
line; --out appends it to a file.
  python tools/jit_assemble_time.py [--n 64] [--reps 5] [--out profiles/jit_assemble_c3.jsonl]"""
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
from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement  # noqa: E402
from ceedpetscsolid_b200.solver import ColoredCoarseMatrix  # noqa: E402

QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
LOCS = {"apply": f"{QF_PORT}:port_HyperFSF", "jacob": f"{QF_PORT}:port_HyperFSdF"}
VARIANTS = [(2, 0), (2, 1), (3, 0), (3, 1)]   # (blocks per SM, unrolled)


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
    tmp = tempfile.mkdtemp(prefix="jit_assemble_time_")
    try:
        out = {}
        for tag in ("first", "second"):
            src = os.path.join(tmp, f"qf_port_{tag}.c")
            shutil.copy(QF_PORT, src)
            t0 = time.perf_counter()
            libceed.jit_assemble_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 2, 5)
            out[f"k13_compile_cold_{tag}_s"] = time.perf_counter() - t0
        n0 = libceed.jit_compile_count()
        t0 = time.perf_counter()
        for _ in range(100):
            libceed.jit_assemble_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 2, 5)
        out["k13_compile_cached_s"] = (time.perf_counter() - t0) / 100
        assert libceed.jit_compile_count() == n0
        return out
    finally:
        shutil.rmtree(tmp)


def level(mesh, u, jit):
    """set-up at p = 4 with the p = 1 level; the fine residual applied at u (gradu of the linearisation point)"""
    ceed = libceed.Ceed("/gpu/b200:jit" if jit else "/gpu/b200")
    degrees, data, _ = setuplibceed.setup_all(ceed, mesh, "hyperFS", 4, qf_locators=LOCS if jit else None)
    assert degrees[0] == 1
    op = data[0].opJacob
    assert op.is_jit_fused if jit else op.is_fused
    r = torch.zeros_like(u)
    uc, rc = ceed.Vector(u.numel()), ceed.Vector(u.numel())
    uc.set_array(u)
    rc.set_array(r)
    data[-1].opApply.apply(uc, rc)
    nelem = mesh.nelem
    vals = torch.zeros(nelem * 576, dtype=torch.float64, device="cuda")
    vc = ceed.Vector(vals.numel())
    vc.set_array(vals)
    torch.cuda.synchronize()
    return SimpleNamespace(ceed=ceed, data=data, op=op, vals=vals, vc=vc, keep=(uc, rc, r))


def tube_solves():
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    from ceedpetscsolid_b200.exodus import tube_mesh
    m = tube_mesh(8, 64, 48)
    ext = float(np.ptp(m.vertices, axis=0).max())
    out = {}
    for tag, locs in (("builtin", None), ("port", LOCS)):
        app = AppCtx(problem="hyperFS", degree=4, num_steps=4, mesh=m,
                     clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.05 * ext, 0.1 * ext, 0, 0, 1, 0]})
        t0 = time.perf_counter()
        el = Elasticity(app, coarse="amg", qf_locators=locs)
        build = time.perf_counter() - t0
        r = el.solve()
        out[tag] = dict(snes_its=r["snes_its"], ksp_its=r["ksp_its"], converged=r["converged"], time_s=r["time_s"],
                        stack_build_s=build, coarse_matrix_from="K13" if locs else "K8")
        out[tag]["U"] = el.U.clone()
        del el
    out["rel_diff_U"] = (torch.linalg.norm(out["port"]["U"] - out["builtin"]["U"]) /
                         torch.linalg.norm(out["builtin"]["U"])).item()
    for tag in ("builtin", "port"):
        del out[tag]["U"]
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-tube", action="store_true")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/jit_assemble_time.py measures on the GPU"
    card = gpu_info()
    print("card:", card, flush=True)
    res = {"case": f"C3 hyperFS p=4 {a.n}^3, level p=1 (P=2, Q=5)", "card": card}
    res.update(compile_times())

    mesh = BoxMesh(n=(a.n,) * 3, perturb=0.08, seed=0)
    res["elements"] = mesh.nelem
    u = torch.from_numpy(smooth_displacement(mesh.node_coords(4)).reshape(-1)).cuda()
    runs = {"k8_builtin": level(mesh, u, False)}
    env0 = {k: os.environ.get(k) for k in ("B200_JIT_ASSEMBLE_CTAS", "B200_JIT_ASSEMBLE_UNROLL")}
    for ctas, unroll in VARIANTS:   # read by the K13 compile at each operator's first assemble, in the warm-up
        os.environ["B200_JIT_ASSEMBLE_CTAS"], os.environ["B200_JIT_ASSEMBLE_UNROLL"] = str(ctas), str(unroll)
        tag = f"k13_ctas{ctas}_{'unrolled' if unroll else 'rolled'}"
        runs[tag] = level(mesh, u, True)
        runs[tag].op.linear_assemble(runs[tag].vc)
        torch.cuda.synchronize()
    for k, v in env0.items():
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = v

    # colouring of the JIT operator (the default variant's set-up): 81 K12 applies into the 27-point stencil
    R = runs["k13_ctas2_rolled"]
    lsize = 3 * mesh.num_nodes(1)
    xc, yc = R.ceed.Vector(lsize), R.ceed.Vector(lsize)

    def local_apply(x, y):
        xc.set_array(x)
        yc.set_array(y)
        y.zero_()
        R.op.apply(xc, yc)
        xc.take_array()
        yc.take_array()
    dm = SimpleNamespace(mesh=mesh, lsize=lsize, device="cuda")
    colour = ColoredCoarseMatrix(dm, local_apply)

    t = {tag: [] for tag in list(runs) + ["colouring_k12"]}
    for _ in range(3):                     # alternate every variant
        for tag, Rv in runs.items():
            t[tag].append(timeit(lambda: Rv.op.linear_assemble(Rv.vc), a.reps))
        t["colouring_k12"].append(timeit(colour.assemble, 1))
    res["assemble_ms"] = {k: min(v) for k, v in t.items()}
    res["assemble_ms_all"] = t
    kb = runs["k8_builtin"].vals
    for tag, Rv in runs.items():
        if tag != "k8_builtin":
            res[f"rel_diff_{tag}_vs_k8"] = (torch.linalg.norm(Rv.vals - kb) / torch.linalg.norm(kb)).item()
    best = min((k for k in runs if k != "k8_builtin"), key=lambda k: res["assemble_ms"][k])
    res["k13_best"] = best
    res["k13_over_k8"] = res["assemble_ms"][best] / res["assemble_ms"]["k8_builtin"]
    res["colouring_over_k13"] = res["assemble_ms"]["colouring_k12"] / res["assemble_ms"][best]
    del runs, colour, R
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
