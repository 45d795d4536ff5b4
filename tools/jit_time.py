#!/usr/bin/env python
"""Cost of user QFunctions through "/gpu/b200:jit" at C3 (hyperFS, p = 4, 64^3 box), in one run on one card:

  * the Jacobian apply (CeedOperatorApply on device L-vectors) of the built-in fused kernel against the same operator
    with oracle/qf_port.c:port_HyperFSdF compiled by NVRTC, which runs on K12, the fused kernel generated around the
    user function; the residual apply (gradu written) with port_HyperFSF likewise.  K12 is built with 2, 3 and 4
    blocks per SM asked of ptxas (B200_JIT_FUSED_CTAS), and all variants are timed in alternating batches;
  * the products checked against the built-in ones;
  * K12's bytes from the shapes and its share of the HBM bound (7.7 TB/s, the HGX B200 data sheet figure for one GPU);
  * the NVRTC compile time of the point program (K11) and of the fused programs, cold (programs this process has not
    compiled) and cached.

The generic path (restriction, basis, K11 point kernel, transposes) that JIT operators took before K12 is recorded
in profiles/jit_time_c3.jsonl.  Prints the card name and power limit and one JSON line; --out appends it to a file.
  python tools/jit_time.py [--n 64] [--reps 10] [--out profiles/jit_fused_time_c3.jsonl]"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ceedpetscsolid_b200 import ceed as libceed  # noqa: E402
from ceedpetscsolid_b200 import setuplibceed  # noqa: E402
from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement  # noqa: E402

QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
HBM_BYTES_PER_S = 7.7e12
DP = 8
CTAS = (2, 3, 4)


def timeit(fn, reps, warm=2):
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
    tmp = tempfile.mkdtemp(prefix="jit_time_")
    try:
        out = {}
        for tag in ("first", "second"):
            src = os.path.join(tmp, f"qf_port_{tag}.c")
            shutil.copy(QF_PORT, src)
            t0 = time.perf_counter()
            libceed.jit_compile(src, "port_HyperFSdF", [9, 10, 9], [9])
            out[f"compile_cold_{tag}_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            libceed.jit_fused_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 5, 5)
            out[f"fused_jacobian_compile_cold_{tag}_s"] = time.perf_counter() - t0
            t0 = time.perf_counter()
            libceed.jit_fused_compile(src, "port_HyperFSF", [9, 10], [9, 9], 0, 0, 5, 5)
            out[f"fused_residual_compile_cold_{tag}_s"] = time.perf_counter() - t0
        n0 = libceed.jit_compile_count()
        t0 = time.perf_counter()
        for _ in range(100):
            libceed.jit_fused_compile(src, "port_HyperFSdF", [9, 10, 9], [9], 0, 0, 5, 5)
        out["fused_compile_cached_s"] = (time.perf_counter() - t0) / 100
        assert libceed.jit_compile_count() == n0
        return out
    finally:
        shutil.rmtree(tmp)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=64)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "tools/jit_time.py measures on the GPU"
    card = gpu_info()
    print("card:", card, flush=True)
    res = {"case": f"C3 hyperFS p=4 {a.n}^3", "card": card}
    res.update(compile_times())          # first: includes opening NVRTC

    mesh = BoxMesh(n=(a.n,) * 3, perturb=0.08, seed=0)
    u = torch.from_numpy(smooth_displacement(mesh.node_coords(4)).reshape(-1)).cuda()
    x = torch.randn_like(u)
    locs = {"apply": f"{QF_PORT}:port_HyperFSF", "jacob": f"{QF_PORT}:port_HyperFSdF"}
    runs = {}
    env0 = os.environ.get("B200_JIT_FUSED_CTAS")
    for tag in ["builtin"] + [f"k12_ctas{c}" for c in CTAS]:
        jit = tag != "builtin"
        if jit:   # read by the fused compile at the operators' first apply, below
            os.environ["B200_JIT_FUSED_CTAS"] = tag[len("k12_ctas"):]
        ceed = libceed.Ceed("/gpu/b200:jit" if jit else "/gpu/b200")
        _, data, _ = setuplibceed.setup_all(ceed, mesh, "hyperFS", 4, multigrid="none", qf_locators=locs if jit else None)
        d = data[-1]
        assert (d.opJacob.is_jit_fused and d.opApply.is_jit_fused) if jit else (d.opJacob.is_fused and d.opApply.is_fused)
        r, y = torch.zeros_like(u), torch.zeros_like(u)
        uc, rc, xc, yc = (ceed.Vector(u.numel()) for _ in range(4))
        uc.set_array(u); rc.set_array(r); xc.set_array(x); yc.set_array(y)
        d.opApply.apply(uc, rc)          # gradu of the linearisation point; compiles K12's residual program
        d.opJacob.apply(xc, yc)          # compiles K12's Jacobian program
        torch.cuda.synchronize()
        runs[tag] = dict(ceed=ceed, d=d, r=r, y=y, uc=uc, rc=rc, xc=xc, yc=yc)
    if env0 is None:
        os.environ.pop("B200_JIT_FUSED_CTAS", None)
    else:
        os.environ["B200_JIT_FUSED_CTAS"] = env0

    t = {("jacobian", tag): [] for tag in runs}
    t.update({("residual", tag): [] for tag in runs})
    for _ in range(3):                   # alternate every variant, several rounds
        for tag, R in runs.items():
            t[("jacobian", tag)].append(timeit(lambda: R["d"].opJacob.apply(R["xc"], R["yc"]), a.reps))
            t[("residual", tag)].append(timeit(lambda: R["d"].opApply.apply(R["uc"], R["rc"]), a.reps))
    torch.cuda.synchronize()
    for kind in ("jacobian", "residual"):
        res[f"{kind}_ms"] = {tag: min(t[(kind, tag)]) for tag in runs}
        res[f"{kind}_ms_all"] = {tag: t[(kind, tag)] for tag in runs}
    rb = runs["builtin"]
    gb = rb["d"].gradu.to_numpy()
    for tag, R in runs.items():
        if tag == "builtin":
            continue
        res[f"rel_diff_jacobian_{tag}"] = (torch.linalg.norm(R["y"] - rb["y"]) / torch.linalg.norm(rb["y"])).item()
        res[f"rel_diff_residual_{tag}"] = (torch.linalg.norm(R["r"] - rb["r"]) / torch.linalg.norm(rb["r"])).item()
        g = R["d"].gradu.to_numpy()
        res[f"max_abs_diff_gradu_{tag}"] = float(abs(g - gb).max())
    best = min((f"k12_ctas{c}" for c in CTAS), key=lambda k: res["jacobian_ms"][k] + res["residual_ms"][k])
    res["k12_best"] = best
    res["k12_jacobian_over_builtin"] = res["jacobian_ms"][best] / res["jacobian_ms"]["builtin"]
    res["k12_residual_over_builtin"] = res["residual_ms"][best] / res["residual_ms"]["builtin"]
    # K12 bytes from the shapes: offsets (4 B per node of every element), the passive per-point fields (Jacobian:
    # qdata 10 + gradu 9 read; residual: qdata 10 read, gradu 9 written), x read once, y read and written once
    nelem, P3, Q3, lsize = mesh.nelem, 5 ** 3, 5 ** 3, u.numel()
    for kind, npt in (("jacobian", 19), ("residual", 19)):
        b = nelem * (P3 * 4 + npt * Q3 * DP) + 3 * lsize * DP
        ms = res[f"{kind}_ms"][best]
        res[f"k12_{kind}_bytes"] = b
        res[f"k12_{kind}_tb_per_s"] = b / (ms * 1e-3) / 1e12
        res[f"k12_{kind}_share_of_hbm_bound"] = b / HBM_BYTES_PER_S / (ms * 1e-3)
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")
    for tag in runs:
        if tag != "builtin":
            assert res[f"rel_diff_jacobian_{tag}"] <= 1e-12 and res[f"rel_diff_residual_{tag}"] <= 1e-12, tag


if __name__ == "__main__":
    main()
