"""Newton-Krylov-p-MG solve on one GPU with a chosen coarse solve; one JSON line per case.

    python tools/amg_solve.py --mesh tube:4,32,24 --coarse pcg amg
    python tools/amg_solve.py --box 64 --coarse hmg amg

Per case: Newton steps and outer CG iterations, what coarse solve actually ran, coarse iterations (Jacobi-PCG
iterations or V-cycles) per coarse solve, solve time and launches (un-instrumented run), then in a second, instrumented
run with a device synchronise around every coarse solve: the coarse solve's share of the solve time.  For AMG also the
symbolic set-up (host, once), the numeric set-up per Newton step, one V-cycle, the level-0 SpMV rate and the levels.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def timed_cuda(fn, reps):
    import torch
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / reps


def run(args, coarse):
    import numpy as np
    import torch
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    from ceedpetscsolid_b200.exodus import tube_mesh
    if args.mesh:
        m = tube_mesh(*[int(v) for v in args.mesh[5:].split(",")])
        ext = float(np.ptp(m.vertices, axis=0).max())
        app = AppCtx(problem="hyperFS", degree=args.degree, num_steps=args.load_steps, mesh=m,
                     clamp={1: [0, 0, 0, 0, 0, 1, 0], 2: [0, -0.05 * ext, 0.1 * ext, 0, 0, 1, 0]})
        label = args.mesh
    else:
        n = (args.box,) * 3
        app = AppCtx(problem="hyperFS", degree=args.degree, n=n, num_steps=args.load_steps, perturb=0.05,
                     clamp={(2, 0): [0, 0, 0, 0, 0, 1, 0], (2, 1): [0, 0, -0.1, 0, 0, 1, 0]})
        label = f"box:{args.box}"
    t0 = time.perf_counter()
    el = Elasticity(app, coarse=coarse)
    build_s = time.perf_counter() - t0
    pc = el.pc
    ran = "amg" if pc.amg is not None else ("hmg" if pc.hmg is not None else "pcg")
    libceed.launch_count_reset()
    torch.cuda.synchronize()
    out = el.solve()
    launches = int(libceed.launch_count())
    rec = {"case": label, "coarse_requested": coarse, "coarse": ran, "problem": "hyperFS", "degree": args.degree,
           "load_steps": args.load_steps, "elements": el.mesh.nelem, "dofs_unconstrained": out["dofs_global_unconstrained"],
           "snes_its": out["snes_its"], "ksp_its": out["ksp_its"], "converged": out["converged"],
           "coarse_solves": out["coarse_solves"], "coarse_its": out["coarse_its"],
           "coarse_its_per_solve": out["coarse_its"] / max(out["coarse_solves"], 1),
           "time_s": out["time_s"], "gpu_launches": launches, "stack_build_s": build_s}
    # instrumented run: device time of every coarse solve
    csum = [0.0]
    inner = pc._coarse_solve

    def coarse_timed(b, x):
        torch.cuda.synchronize()
        t = time.perf_counter()
        inner(b, x)
        torch.cuda.synchronize()
        csum[0] += time.perf_counter() - t
    pc._coarse_solve = coarse_timed
    pc.coarse_its = pc.coarse_solves = 0
    out2 = el.solve()
    pc._coarse_solve = inner
    rec.update({"instrumented_time_s": out2["time_s"], "coarse_solve_s": csum[0],
                "coarse_share": csum[0] / out2["time_s"]})
    if pc.amg is not None:
        amg = pc.amg
        setup_s = timed_cuda(lambda: amg.setup(pc.coarse if pc.coarse is not None else pc.levels[0]), 3)
        b = torch.randn(el.dms[0].nglobal, dtype=torch.float64, device="cuda")
        el.dms[0].zero_constrained(b)
        x = torch.zeros_like(b)
        vc_s = timed_cuda(lambda: amg.solve(b, x), 20)
        A0 = amg.levels[0].A
        xa = torch.randn(A0.n, dtype=torch.float64, device="cuda")
        ya = torch.zeros_like(xa)
        sp_s = timed_cuda(lambda: A0.mult(xa, ya), 50)
        nbytes = A0.vals.numel() * 8 + A0.colidx.numel() * 4 + A0.rowptr.numel() * 4 + 2 * A0.n * 8
        rec.update({"amg_symbolic_ms": amg.symbolic_s * 1e3, "amg_numeric_setup_ms_per_newton": setup_s * 1e3,
                    "amg_vcycle_ms": vc_s * 1e3, "amg_levels": amg.level_info(), "amg_pairs": amg.pair_counts(),
                    "spmv_level0_ms": sp_s * 1e3, "spmv_level0_GBps_min_traffic": nbytes / sp_s / 1e9})
    rec["gpu"] = torch.cuda.get_device_name(0)
    try:
        import subprocess
        rec["power_limit"] = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"],
                                            capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        rec["power_limit"] = f"unavailable ({type(e).__name__})"
    del el
    torch.cuda.empty_cache()
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--mesh", default=None, help="tube:NR,NT,NZ (side set 1 clamped, side set 2 moved)")
    ap.add_argument("--box", type=int, default=None, help="box of N^3 elements instead of a tube")
    ap.add_argument("--coarse", nargs="+", default=["pcg", "amg"], choices=["hmg", "pcg", "amg"])
    ap.add_argument("--degree", type=int, default=4)
    ap.add_argument("--load-steps", type=int, default=4)
    ap.add_argument("--out", default=None, help="append the lines to this file too")
    args = ap.parse_args()
    if (args.mesh is None) == (args.box is None):
        ap.error("give exactly one of --mesh and --box")
    import torch
    if not torch.cuda.is_available():
        sys.exit("tools/amg_solve.py measures on a GPU; no CUDA device found")
    for c in args.coarse:
        line = json.dumps(run(args, c))
        print(line, flush=True)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")


if __name__ == "__main__":
    main()
