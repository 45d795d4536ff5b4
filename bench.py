#!/usr/bin/env python
"""Benchmark of the hot path: GDoF/s of the hyperFS (finite-strain Neo-Hookean) Jacobian
MatMult at p = 4 on a synthetic box mesh (BASELINE.json metric; SURVEY.md 8(d)).

    python bench.py --gpus N --steps K --warmup W            # /gpu/b200 arm
    python bench.py --impl reference --gpus N ...            # CPU arm (restated /cpu/self)

One "step" = one MatShell MatMult of the fine-level Jacobian: ApplyJacobian_Ceed
(/root/reference/src/matops.c:98-112) = zero Dirichlet inputs, DMGlobalToLocal (+ halo),
zero Yloc, CeedOperatorApply (ONE fused kernel), DMLocalToGlobal (+ halo).
Workload at N = 1: BASELINE.json configs[2], box 64^3, degree 4 (262 144 elements,
50.9 M DoFs).  N > 1: weak scaling, one 64^3 brick per GPU (2x1x1, 2x2x1, 2x2x2 bricks),
NCCL halo exchange; `--scaling strong` shards the ~100 M-DoF 80^3 box of configs[3] instead.
Inputs (4.5 GB of per-quadrature-point data per GPU) are far larger than L2, so no explicit
L2 flush is needed between timed iterations.
"""
import argparse
import json
import os
import sys
import threading
import time

# stdout must carry exactly ONE JSON line.  Libraries write banners to the C-level stdout (NCCL prints its version
# there at NCCL_DEBUG=VERSION, which the image exports, and at WARN): file descriptor 1 is pointed at stderr for the
# whole run and the result line is written to the saved descriptor.
if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
    os.environ["NCCL_DEBUG"] = "WARN"
sys.stdout.flush()
_RESULT_FD = os.dup(1)
os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_RESULT_FD, (json.dumps(line) + "\n").encode())


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True   # the benchmark may run from a read-only tree: no __pycache__ next to the sources

import numpy as np  # noqa: E402

DUMP_ENTRIES = 1 << 22   # --dump-outputs: at most 4 Mi float64 values (32 MB) over all ranks


def dump_output(out_dir, name, y, world):
    """Write a result vector as out_dir/name.npy (float64).  A vector longer than this rank's share of DUMP_ENTRIES is
    sampled at sorted indices drawn with a fixed seed: the same length gives the same indices in every run."""
    import torch
    k = DUMP_ENTRIES // world
    if y.numel() > k:
        idx = np.sort(np.random.default_rng(0).choice(y.numel(), k, replace=False))
        y = y[torch.from_numpy(idx).to(y.device)]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, name + ".npy"), y.detach().to(torch.float64).cpu().numpy())


def alg_bytes(problem, p, qextra=0):
    """SURVEY.md 8(d): 8 Q^3 (10 + g) + 4 P^3 + 48 p^3 bytes per element (22 572 for hyperFS p = 4)."""
    P, Q = p + 1, p + 1 + qextra
    g = 0 if problem == "linElas" else 9
    return 8 * Q ** 3 * (10 + g) + 4 * P ** 3 + 48 * p ** 3


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons of one GPU through NVML during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag = index, [], set(), False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.02)

    def result(self):
        self.stop_flag = True
        self.join(timeout=1)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def cpu_leg(problem, p, n_cpu, steps, warmup):
    """Times the CPU oracle (restated /cpu/self operator) on a bounded sample of the workload with ALL host threads
    (set explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers).  Timing build: the operator loops at
    -O3 -march=native compiled on this box (oracle/_native), calling the reference's own QFunctions at
    -O3 -march=x86-64-v3 (oracle/_ref/libref_qf_fast.so, built from /root/reference where it is mounted) -- or the
    ported ones where that library is absent.  The -ffp-contract=off parity builds are not what is timed."""
    from helpers import OracleProblem
    from oracle import oracle
    try:
        oracle.native_lib()
        native = True
    except Exception:   # no compiler on the box: time the parity build and say so
        native = False
    which = "ref_fast" if oracle.have_ref_fast() else ("port_native" if native else oracle.default_which())
    threads = os.cpu_count() or 1
    oracle.set_num_threads(threads)                    # set-up of the sample (parity build)
    threads = oracle.set_num_threads(threads, native=native)
    pr = OracleProblem(problem, n_cpu, p, which=oracle.default_which())
    x = np.random.default_rng(1).standard_normal(pr.lsize)
    y = np.zeros_like(x)

    def apply():
        return oracle.operator_apply(problem, True, (0.3, 1.0), pr.nelem, pr.P, pr.Q, pr.B, pr.D, pr.offsets,
                                     pr.qdata, pr.gradu, x, which, y, native=native)
    for _ in range(max(1, warmup)):
        apply()
    t0 = time.perf_counter()
    for _ in range(steps):
        apply()
    dt = (time.perf_counter() - t0) / steps
    dofs = pr.lsize
    qf = {"ref_fast": "the reference QFunctions compiled from /root/reference at -O3 -march=x86-64-v3 (oracle/_ref/libref_qf_fast.so)",
          "ref": "the reference QFunctions compiled from /root/reference (oracle/_ref, parity build)",
          "port_native": "the ported QFunctions (oracle/qf_port.c) at -O3 -march=native",
          "port": "the ported QFunctions (oracle/qf_port.c, parity build)"}[which]
    return {"value": dofs / dt / 1e9, "unit": "GDoF/s", "cores": int(threads), "kind": "port",
            "sample": f"{problem} p={p} Jacobian apply on a {n_cpu}^3 box ({pr.nelem} elements, {dofs} DoFs), "
                      f"{steps} applies after {max(1, warmup)} warm-up, restated /cpu/self operator (oracle/ceed_oracle.c, OpenMP over "
                      f"elements, {'-O3 -march=native build of this box' if native else 'parity build'}) calling {qf}",
            "ms_per_apply": dt * 1e3, "elements": int(pr.nelem), "dofs": int(dofs), "omp_threads": int(threads),
            "host_cpus": os.cpu_count()}


def run_solve(args, rank, world, local_rank, dist, n_box, scaling):
    """BASELINE configs[4]: full Newton-Krylov-p-MG solve, hyperFS, 10 load steps, Chebyshev/Jacobi smoothing
    with GPU diagonal assembly; wall time of the load-increment loop only, max over ranks
    (/root/reference/elasticity.c:632-676,755-764).  Returns the record (same on every rank)."""
    import torch
    from ceedpetscsolid_b200 import ceed as libceed
    from ceedpetscsolid_b200.elasticity import AppCtx, Elasticity
    from ceedpetscsolid_b200.mesh import BoxMesh, grid_for
    grid = grid_for(world)
    n = (n_box * grid[0], n_box * grid[1], n_box * grid[2]) if scaling == "weak" else (n_box,) * 3
    lengths = tuple(float(g) for g in grid) if scaling == "weak" else (1.0, 1.0, 1.0)
    umesh = None
    if args.mesh:
        from ceedpetscsolid_b200.exodus import HexMesh, tube_mesh
        umesh = tube_mesh(*[int(v) for v in args.mesh[5:].split(",")]) if args.mesh.startswith("tube:") else HexMesh.from_file(args.mesh)
    app = AppCtx(problem=args.problem, degree=args.degree, n=n, num_steps=args.load_steps, perturb=0.05,
                 clamp={(2, 0): [0, 0, 0, 0, 0, 1, 0], (2, 1): [0, 0, -0.1 * lengths[2], 0, 0, 1, 0]})
    gmesh = BoxMesh(n=n, perturb=app.perturb, seed=0, lengths=lengths)
    if umesh is not None:
        ids = [int(v) for v in args.clamp_sets.split(",")]
        ext = float(np.ptp(umesh.vertices, axis=0).max())
        app.mesh, gmesh = umesh, None
        app.clamp = {ids[0]: [0, 0, 0, 0, 0, 1, 0], ids[1]: [0, -0.05 * ext, 0.1 * ext, 0, 0, 1, 0]}
    el = Elasticity(app, dist=dist if world > 1 else None, rank=rank, world=world, device_id=local_rank, gmesh=gmesh,
                    coarse_rtol=args.coarse_rtol, coarse=args.coarse, assemble=args.assemble, masked=args.dm == "masked",
                    halo=args.halo, overlap=not args.no_overlap, deterministic=args.deterministic)
    el.pc.coarse_maxit = args.coarse_maxit
    libceed.launch_count_reset()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    out = el.solve(log=(lambda m: print(m, file=sys.stderr)) if (rank == 0 and args.verbose) else None)
    t = torch.tensor([out["time_s"]], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    clocks = sampler.result()
    launches = int(libceed.launch_count())
    energy = el.strain_energy()   # elasticity.c:820-830: printed by the reference after the solve (all ranks: reduction)
    rec = {"time_s": float(t.item()), "snes_its": out["snes_its"], "ksp_its": out["ksp_its"], "converged": out["converged"],
           "workload": f"{args.problem} degree {args.degree} Newton-Krylov-pMG solve, box {n_box}^3 "
                       f"{'per GPU' if scaling == 'weak' else 'sharded'}, {args.load_steps} load steps, levels {el.degrees}"
                       + (f", mesh {args.mesh}" if args.mesh else ""),
           "scaling": scaling, "bricks": "x".join(map(str, grid)), "elements_per_gpu": el.mesh.nelem,
           "dofs_unconstrained": out["dofs_global_unconstrained"], "mdofs_per_sec_in_snes": out["mdofs_per_sec_in_snes"],
           "coarse_pcg_its": out["coarse_its"], "coarse": args.coarse, "assemble": args.assemble,
           "coarse_rtol": args.coarse_rtol, "strain_energy": energy, "gpu_launches": launches, "clocks": clocks,
           "halo": "none (1 GPU)" if world == 1 else args.halo, "deterministic": bool(args.deterministic)}
    el.close()
    del el
    torch.cuda.empty_cache()
    return rec


def solve_bench(args, rank, world, local_rank, dist, config):
    """`bench.py --solve`: the solve alone, as its own JSON line."""
    rec = run_solve(args, rank, world, local_rank, dist, args.n, args.scaling)
    if rank == 0:
        config.update({"workload": rec["workload"], "elements_per_gpu": rec["elements_per_gpu"], "bricks": rec["bricks"]})
        line = {"metric": "SNES solve time", "value": rec["time_s"], "unit": "s", "n_gpus": world, "steps": 1,
                "warmup": 0, "ms_per_step": rec["time_s"] * 1e3, "higher_is_better": False,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config}
        line.update({k: v for k, v in rec.items() if k not in ("time_s", "workload", "scaling", "bricks", "elements_per_gpu")})
        emit(line)
    if world > 1:
        dist.destroy_process_group()


class MatMultProblem:
    """One rank's share of a (partitioned) box: libCEED objects, DM stand-in, MatShell context, state at the smooth
    displacement of SURVEY.md 8(d) (the residual has been evaluated once: gradu and the Jacobian cache are current)."""

    def __init__(self, args, rank, world, local_rank, dist, n_box, scaling, dm_kind, halo_kind, overlap):
        import torch
        from ceedpetscsolid_b200 import ceed as libceed
        from ceedpetscsolid_b200 import matops, setuplibceed
        from ceedpetscsolid_b200.mesh import BoxMesh, grid_for, smooth_displacement
        problem, p = args.problem, args.degree
        self.grid = grid = grid_for(world)
        if scaling == "weak":
            self.gmesh = BoxMesh(n=(n_box * grid[0], n_box * grid[1], n_box * grid[2]), perturb=0.08, seed=0,
                                 lengths=tuple(float(g) for g in grid))  # the domain grows with the mesh: cubic elements
        else:
            self.gmesh = BoxMesh(n=(n_box,) * 3, perturb=0.08, seed=0)
        masked = dm_kind == "masked"
        self.mesh = self.gmesh.brick(grid, rank, interface_first=masked and overlap) if world > 1 else self.gmesh
        self.ceed = libceed.Ceed(f"/gpu/b200:device_id={local_rank}" + (":deterministic" if args.deterministic else ""))
        self.degrees, self.data, self.phys = setuplibceed.setup_all(self.ceed, self.mesh, problem, p)
        self.fine = len(self.degrees) - 1
        self.halo = None
        if world > 1:
            from ceedpetscsolid_b200.halo import Halo
            self.halo = Halo(self.gmesh, grid, rank, p, dist)
            if halo_kind == "p2p" and not self.halo.enable_p2p():
                raise RuntimeError(f"peer-memory halo set-up failed: {self.halo._p2p_error}")
        # N > 1: shared-dof global vectors -> one symmetric sum-and-share halo exchange per MatMult
        self.dm = matops.LevelDM(self.mesh, p, bc_faces="all", halo=self.halo, shared=True, masked=masked)
        self.user = matops.setup_jacobian_ctx(self.dm, self.ceed, self.data[self.fine], self.phys)
        self.user.overlap = overlap
        # state: smooth admissible displacement -> residual fills gradu (SURVEY.md 8(d))
        u = torch.from_numpy(smooth_displacement(self.mesh.node_coords(p)).reshape(-1)).cuda()
        self.uc, self.rc = self.ceed.Vector(u.numel()), self.ceed.Vector(u.numel())
        self.u, self.r = u, torch.zeros_like(u)
        self.evaluate_residual()
        self.X, self.Y = self.dm.create_global_vector(), self.dm.create_global_vector()
        self.X.copy_(torch.from_numpy(np.random.default_rng(1 + rank).standard_normal(self.dm.nglobal)))
        self.dm.zero_constrained(self.X)

    def evaluate_residual(self):
        self.uc.set_array(self.u); self.rc.set_array(self.r)
        self.data[self.fine].opApply.apply(self.uc, self.rc)
        self.uc.take_array(); self.rc.take_array()

    def matmult(self):
        from ceedpetscsolid_b200 import matops
        matops.ApplyJacobian_Ceed(self.user, self.X, self.Y)

    def close(self):
        if self.halo is not None:
            self.halo.check_p2p()   # a timed-out peer-memory exchange invalidates the run: fail loudly
            self.halo.close()


def timed(fn, steps, warmup, world, dist):
    """W untimed + exactly K timed calls, CUDA events on the launching stream, barrier + synchronize on both sides,
    max over ranks.  Returns total milliseconds of the K calls."""
    import torch

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(warmup):
        fn()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    return ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--problem", default="hyperFS")
    ap.add_argument("--degree", type=int, default=4)
    ap.add_argument("--box", "--n", dest="n", type=int, default=64, help="elements per direction per GPU (weak) / of the whole box (strong)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--cpu-box", "--n-cpu", dest="n_cpu", type=int, default=32, help="box size of the bounded CPU sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extras", action="store_true",
                    help="main MatMult line only: skip parity, compressed-DM, strong C4 and SNES-solve legs")
    ap.add_argument("--no-solve", action="store_true", help="skip the snes_solve leg")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong_c4 leg")
    ap.add_argument("--strong-box", type=int, default=80, help="BASELINE configs[3]: box sharded over the GPUs (80^3 = 99.2 M DoFs)")
    ap.add_argument("--solve-box", type=int, default=None, help="elements per direction per GPU of the snes_solve leg (default: --box)")
    ap.add_argument("--solve", action="store_true",
                    help="time the full Newton-Krylov-p-MG solve (BASELINE configs[4]) instead of the MatMult")
    ap.add_argument("--load-steps", type=int, default=10)
    ap.add_argument("--mesh", default=None, help="--solve on an unstructured hex8 mesh: an Exodus II file (-mesh, "
                    "setupdm.c:40-68) or 'tube:NR,NT,NZ' (synthetic); side sets --clamp-sets are clamped")
    ap.add_argument("--clamp-sets", default="1,2", help="side-set ids: first fixed, second translated by (0,-0.05,0.1) x length scale")
    ap.add_argument("--coarse-rtol", type=float, default=1e-2)
    ap.add_argument("--coarse-maxit", type=int, default=500)
    ap.add_argument("--dm", default="masked", choices=["masked", "compressed"],
                    help="global-vector layout of the DM stand-in (matops.LevelDM)")
    ap.add_argument("--no-overlap", action="store_true",
                    help="N > 1: do not run the interface elements first / overlap the halo exchange with the interior ones")
    ap.add_argument("--overlap", action="store_true", help="(default now; kept for old command lines)")
    ap.add_argument("--halo", default="p2p", choices=["nccl", "p2p"],
                    help="N > 1: interface exchange stored straight into the neighbours' windows over NVLink peer memory "
                         "(csrc/b200_halo.cu, default) or through NCCL send/recv")
    ap.add_argument("--deterministic", action="store_true", help="/gpu/b200:deterministic (ordered, atomic-free scatter)")
    ap.add_argument("--assemble", default="coo", choices=["coo", "color"], help="p=1 matrix: CeedOperatorLinearAssemble element matrices, or 81 coloured applies (misc.c:151-183)")
    ap.add_argument("--coarse", default="hmg", choices=["hmg", "pcg"], help="coarse solve on the assembled p=1 level: h-multigrid (GAMG stand-in) or Jacobi-PCG")
    ap.add_argument("--verbose", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed MatMults, write the product Y of the last one (this rank's global vector) as "
                         "DIR/y.npy (DIR/y_rank<r>.npy for N > 1), float64; longer vectors as a fixed seeded sample")
    args = ap.parse_args()
    if args.dump_outputs and (args.solve or args.impl != "b200"):
        ap.error("--dump-outputs writes the result of the /gpu/b200 MatMult: not with --solve or --impl reference")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    problem, p = args.problem, args.degree
    overlap = not args.no_overlap
    workload = (f"{problem} degree {p} Jacobian MatMult, box {args.n}^3 per GPU" if args.scaling == "weak"
                else f"{problem} degree {p} Jacobian MatMult, box {args.n}^3 sharded")
    halo_desc = ("none (1 GPU)" if world == 1 else
                 ("NVLink peer-memory windows (CUDA IPC), one rank-ordered sum-and-share per MatMult, no NCCL on the data path"
                  if args.halo == "p2p" else "NCCL send/recv, one rank-ordered sum-and-share per MatMult")
                 + (", overlapped with the interior elements" if (overlap and args.dm == "masked" and not args.deterministic) else ""))
    config = {"workload": workload, "problem": problem, "degree": p, "levels": "fine level of {1,2,4}",
              "elements_per_gpu": None,
              "scatter": "deterministic: E-vector + ordered gather" if args.deterministic else "fp64 atomics",
              "l2": "inputs larger than L2 (no flush needed)", "bricks": None, "halo": halo_desc}

    # ------------------------------------------------------------------ CPU reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        from ceedpetscsolid_b200.mesh import grid_for
        # the b200 arm's workload is one 64^3 box per GPU; one step of THIS arm is a bounded sample of it: one Jacobian
        # MatMult on an n_cpu^3 box of the same problem / degree / geometry, all host cores of the box
        cb = cpu_leg(problem, p, args.n_cpu, args.steps, args.warmup)
        config["workload"] = (f"{problem} degree {p} Jacobian MatMult, CPU sample: box {args.n_cpu}^3 ({cb['elements']} elements, "
                              f"{cb['dofs']} DoFs) of the b200 arm's box {args.n}^3 per GPU")
        config["elements_per_gpu"] = cb["elements"]
        config["bricks"] = "1x1x1"
        config["halo"] = "none (host cores of one box)"
        config["scatter"] = "serial (as /cpu/self)"
        config["same_config_as_b200_arm"] = False
        config["b200_arm_workload"] = workload
        line = {"impl": "reference", "metric": "GDoF/s of hyperFS Jacobian MatMult at p=4", "value": cb["value"],
                "unit": "GDoF/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": cb["ms_per_apply"], "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "cpu_baseline": cb,
                "e2e": {"value": cb["value"], "unit": "GDoF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "omp_threads": cb["omp_threads"], "host_cpus": cb["host_cpus"]}
        emit(line)
        return

    # ------------------------------------------------------------------ /gpu/b200 arm
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    if args.solve:
        return solve_bench(args, rank, world, local_rank, dist, config)
    from ceedpetscsolid_b200 import ceed as libceed

    # ---- parity first: a small partitioned problem against the serial CPU oracle, through the same code path
    parity = None
    if not args.no_extras:
        from mgpu_check import partitioned_parity
        err, ok, bitwise, desc = partitioned_parity(rank, world, local_rank, layout=args.dm if args.dm == "masked" else "1",
                                                    halo_mode=args.halo, overlap=overlap)
        parity = {"rel_err": err, "tolerance": 1e-12, "ok": ok, "interface_copies_bit_identical": bitwise,
                  "halo": "none (1 GPU)" if world == 1 else args.halo, "what": desc}
        if not ok and world > 1 and args.halo == "p2p":
            # the peer-memory exchange is the default; if it cannot be set up or does not pass on this box, say so and
            # measure through NCCL instead (every rank takes this branch: the verdict is broadcast)
            first = parity
            args.halo = "nccl"
            err, ok, bitwise, desc = partitioned_parity(rank, world, local_rank, layout=args.dm if args.dm == "masked" else "1",
                                                        halo_mode="nccl", overlap=overlap)
            parity = {"rel_err": err, "tolerance": 1e-12, "ok": ok, "interface_copies_bit_identical": bitwise,
                      "halo": "nccl", "what": desc, "fallback_from_p2p": first}
            config["halo"] = "NCCL send/recv, one rank-ordered sum-and-share per MatMult (peer-memory path failed its check: see parity.fallback_from_p2p)"
        if not ok:
            raise SystemExit(f"bench.py: parity check failed before timing: {parity}")

    pr = MatMultProblem(args, rank, world, local_rank, dist, args.n, args.scaling, args.dm, args.halo, overlap)
    mesh, gmesh, dm, data, fine = pr.mesh, pr.gmesh, pr.dm, pr.data, pr.fine
    config["elements_per_gpu"] = mesh.nelem
    config["bricks"] = "x".join(map(str, pr.grid))
    config["dm"] = ("masked constrained dofs: Krylov vectors have the L-vector layout, no G2L/L2G copies" if args.dm == "masked"
                    else "compressed global vectors: G2L gather + L2G scatter around every apply (PETSc DM style)")

    pr.matmult()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    sampler.start()
    libceed.launch_count_reset()
    launches_before = 0
    # count the launches of the timed region only: reset after the warm-up inside timed() is not possible, so count
    # one call's launches separately (same code path, same count every call)
    ms = timed(pr.matmult, args.steps, args.warmup, world, dist)
    clocks = sampler.result()
    if args.dump_outputs:
        dump_output(args.dump_outputs, "y" if world == 1 else f"y_rank{rank}", pr.Y, world)
    libceed.launch_count_reset()
    pr.matmult()
    torch.cuda.synchronize()
    launches = int(libceed.launch_count()) * args.steps
    dofs = 3 * gmesh.num_nodes(p)
    dofs_unconstrained = 3 * int(np.prod([gmesh.n[d] * p - 1 for d in range(3)]))
    value = dofs * args.steps / (ms * 1e-3) / 1e9

    # ---- dominant kernel alone (fused Jacobian apply), CUDA events on the launching stream
    xl, yl = dm.create_local_vector(), dm.create_local_vector()
    xl.copy_(torch.from_numpy(np.random.default_rng(7).standard_normal(dm.lsize)))
    xc, yc = data[fine].xceed, data[fine].yceed
    xc.set_array(xl); yc.set_array(yl)
    nk = args.steps
    kms = timed(lambda: data[fine].opJacob.apply_add(xc, yc), nk, 3, 1, None) / nk
    # Jacobian cache: rebuilt lazily after every residual evaluation (new linearisation point)
    pr.evaluate_residual()
    torch.cuda.synchronize()
    j0, j1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    j0.record()
    data[fine].opJacob.apply_add(xc, yc)
    j1.record()
    torch.cuda.synchronize()
    jcache_build_ms = max(j0.elapsed_time(j1) - kms, 0.0)
    xc.take_array(); yc.take_array()
    peak, peak_src = measured_peaks()
    ab = alg_bytes(problem, p) * mesh.nelem
    achieved = ab / (kms * 1e-3) / 1e9
    from ceedpetscsolid_b200.ceed import lib as _lib
    nj = int(_lib.b200_jcache_ncomp({"linElas": 0, "hyperSS": 1, "hyperFS": 2}[problem]))
    Qn = p + 1
    moved = (8 * Qn ** 3 * nj + 4 * (p + 1) ** 3 + 48 * p ** 3) * mesh.nelem
    roofline = {"bound": "hbm", "kernel": "k_fused_apply<P=5,Q=5,hyperFS,Jacobian>", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": None, "peak_source": peak_src,
                "kernel_ms": kms, "algorithmic_bytes_per_launch": ab,
                "algorithmic_bytes_per_element": alg_bytes(problem, p),
                "bytes_the_kernel_must_move_per_launch": moved, "frac_of_bytes_moved": moved / (kms * 1e-3) / 1e9 / peak,
                "jacobian_cache_doubles_per_point": nj,
                "kernel_gdofs": 3 * mesh.num_nodes(p) / (kms * 1e-3) / 1e9}
    # FP64 cross-check (SURVEY.md 8(d)): DFMA-class instructions the kernel executes per element (12 line stages x
    # 3 Q^4 + Q^3 x ~150 for the cached hyperFS Jacobian; DESIGN.md section 3) against a DFMA microbenchmark run now
    if problem == "hyperFS" and p == 4:
        try:
            import ctypes as C
            rate = C.c_double(0.0)
            libceed.b2(libceed.lib.b200_fp64_probe(C.byref(rate)))
            dfma_elem = 12 * 3 * Qn ** 4 + Qn ** 3 * 150
            roofline["fp64"] = {"fp64_instr_per_element": dfma_elem, "kernel_tdfma_per_s": dfma_elem * mesh.nelem / (kms * 1e-3) / 1e12,
                                "probe_tdfma_per_s": rate.value / 1e12,
                                "frac": dfma_elem * mesh.nelem / (kms * 1e-3) / rate.value}
        except Exception as exc:  # the probe is informational: never fail the bench on it
            roofline["fp64"] = {"error": str(exc)}
    traffic_path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(traffic_path):
        with open(traffic_path) as f:
            tj = json.load(f)
        # one `ncu --set full` capture of this kernel; DRAM bytes per element scaled to this launch
        roofline["traffic"] = tj.get("dram_bytes_per_element", 0) * mesh.nelem or None
        roofline["traffic_source"] = tj.get("source")

    # ---- e2e: the libCEED boundary with HOST buffers (-memtype host): SetArray(HOST), Apply, TakeArray(HOST)
    e2e = None
    if not args.no_e2e:
        xh = torch.empty(dm.lsize, dtype=torch.float64).pin_memory()
        yh = torch.zeros(dm.lsize, dtype=torch.float64).pin_memory()
        xh.copy_(xl.cpu())

        def host_barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
        nrep = args.steps
        for it in range(2 + nrep):
            if it == 2:
                host_barrier()
                t0 = time.perf_counter()
            xc.set_array(xh, libceed.MEM_HOST)
            yc.set_array(yh, libceed.MEM_HOST)
            data[fine].opJacob.apply(xc, yc)
            xc.take_array(libceed.MEM_HOST)
            yc.take_array(libceed.MEM_HOST)
        host_barrier()
        dt = (time.perf_counter() - t0) / nrep
        # the floor under it: the same bytes over PCIe in both directions at once, no kernel, ALL ranks concurrently
        # (they share the host's memory controllers and PCIe root complexes)
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()

        def copies():
            with torch.cuda.stream(s1):
                xl.copy_(xh, non_blocking=True)
            with torch.cuda.stream(s2):
                yh.copy_(yl, non_blocking=True)
        copies()
        host_barrier()
        t1 = time.perf_counter()
        for _ in range(3):
            copies()
        host_barrier()
        floor = (time.perf_counter() - t1) / 3
        if world > 1:
            t = torch.tensor([dt, floor], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt, floor = float(t[0].item()), float(t[1].item())
        e2e = {"value": dofs / dt / 1e9, "unit": "GDoF/s", "h2d_bytes_per_step": int(dm.lsize * 8),
               "d2h_bytes_per_step": int(dm.lsize * 8), "ms_per_step": dt * 1e3,
               "pcie_floor_ms": floor * 1e3,
               "pcie_floor_what": "H2D of x and D2H of y (same pinned buffers, two streams, no kernel) on all ranks at once, max over ranks",
               "what": "CeedVectorSetArray(HOST,USE_POINTER) + CeedOperatorApply + CeedVectorTakeArray(HOST) on pinned host "
                       "L-vectors (per rank; N > 1: every rank its own brick, no halo exchange in this leg)"}
        del xh, yh

    # ---- the same MatMult with PETSc-style compressed global vectors (G2L gather + L2G scatter around the kernel)
    extra = {"jcache_build_ms": jcache_build_ms}
    if not args.no_extras:
        from ceedpetscsolid_b200 import matops
        other = "compressed" if args.dm == "masked" else "masked"
        dm2 = matops.LevelDM(mesh, p, bc_faces="all", halo=pr.halo, shared=True, masked=other == "masked")
        user2 = matops.setup_jacobian_ctx(dm2, pr.ceed, data[fine], pr.phys)
        user2.overlap = False   # the brick keeps the element order of the main run; the compressed layout has no overlap path
        X2, Y2 = dm2.create_global_vector(), dm2.create_global_vector()
        X2.copy_(torch.from_numpy(np.random.default_rng(1 + rank).standard_normal(dm2.nglobal)))
        ms2 = timed(lambda: matops.ApplyJacobian_Ceed(user2, X2, Y2), args.steps, args.warmup, world, dist)
        extra["value_" + other + "_dm"] = {"value": dofs * args.steps / (ms2 * 1e-3) / 1e9, "unit": "GDoF/s",
                                            "ms_per_step": ms2 / args.steps,
                                            "what": "same MatMult, " + ("PETSc-style compressed global vectors (G2L gather + L2G "
                                                    "scatter around the kernel)" if other == "compressed" else "masked layout")}
        del dm2, user2, X2, Y2
    pr.close()
    del pr, data, dm, xl, yl, xc, yc
    torch.cuda.empty_cache()

    # ---- BASELINE configs[3]: the ~100 M-DoF box sharded over the N GPUs (strong scaling; N = 1: one GPU holds it)
    if not (args.no_extras or args.no_strong):
        ps = MatMultProblem(args, rank, world, local_rank, dist, args.strong_box, "strong", args.dm, args.halo, overlap)
        mss = timed(ps.matmult, args.steps, args.warmup, world, dist)
        sd = 3 * ps.gmesh.num_nodes(p)
        xs, ys = ps.dm.create_local_vector(), ps.dm.create_local_vector()
        xs.normal_()
        xcs, ycs = ps.data[ps.fine].xceed, ps.data[ps.fine].yceed
        xcs.set_array(xs); ycs.set_array(ys)
        ks = min(timed(lambda: ps.data[ps.fine].opJacob.apply_add(xcs, ycs), args.steps, 3, world, dist) / args.steps
                 for _ in range(2))
        xcs.take_array(); ycs.take_array()
        extra["strong_c4"] = {"value": sd * args.steps / (mss * 1e-3) / 1e9, "unit": "GDoF/s", "ms_per_step": mss / args.steps,
                              "scaling": "strong", "dofs": sd, "elements_per_gpu": ps.mesh.nelem, "bricks": "x".join(map(str, ps.grid)),
                              "interface_elements": int(ps.mesh.n_interface), "kernel_ms_whole_brick": ks,
                              "exposed_ms_per_step": max(mss / args.steps - ks, 0.0),
                              "exposed_what": "step minus the fused kernel over the whole brick timed separately (zeroing of Y, Dirichlet "
                                              "mask, launches, halo exchange not hidden); the two timings see slightly different clocks",
                              "workload": f"{problem} degree {p} Jacobian MatMult, box {args.strong_box}^3 ({sd} DoFs) sharded over {world} GPU(s)"}
        ps.close()
        del ps, xs, ys, xcs, ycs
        torch.cuda.empty_cache()

    # ---- second half of the metric: SNES solve time at this N (BASELINE configs[4])
    if not (args.no_extras or args.no_solve):
        extra["snes_solve"] = run_solve(args, rank, world, local_rank, dist, args.solve_box or args.n, args.scaling)

    if rank == 0:
        cb = None
        if world == 1 and not args.no_cpu:
            cb = cpu_leg(problem, p, args.n_cpu, 5, 2)
        line = {"metric": "GDoF/s of hyperFS Jacobian MatMult at p=4", "value": value, "unit": "GDoF/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64",
                "data": "synthetic", "config": config, "dofs": dofs, "dofs_unconstrained": dofs_unconstrained,
                "value_unconstrained_dofs": dofs_unconstrained * args.steps / (ms * 1e-3) / 1e9,
                "roofline": roofline, "cpu_baseline": cb, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks, "parity": parity}
        line.update(extra)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
