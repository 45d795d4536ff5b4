#!/usr/bin/env python
"""Cost of running the Jacobian QFunction through "/gpu/b200:jit" at C3 (hyperFS, p = 4, 64^3 box), in one run:

  * the built-in fused Jacobian apply (CeedOperatorApply on device L-vectors) against the same operator with
    oracle/qf_port.c:port_HyperFSdF compiled by NVRTC, which runs on the generic path (restriction, basis, K11 point
    kernel, transposed basis, transposed restriction); both products are checked against each other;
  * the K11 point kernel alone on the operator's own Q-vectors, with its bytes from the shapes and its share of the
    HBM bound (7.7 TB/s, the HGX B200 data sheet figure for one GPU);
  * the NVRTC compile time, cold (a program this process has not compiled) and cached.

Prints the card name and power limit and one JSON line; --out also writes that line to a file.
  python tools/jit_time.py [--n 64] [--reps 10] [--out profiles/jit_time_c3.jsonl]"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ceedpetscsolid_b200 import ceed as libceed  # noqa: E402
from ceedpetscsolid_b200 import setuplibceed  # noqa: E402
from ceedpetscsolid_b200.mesh import BoxMesh, smooth_displacement  # noqa: E402

QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
HBM_BYTES_PER_S = 7.7e12
DP = 8


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
        n0 = libceed.jit_compile_count()
        t0 = time.perf_counter()
        for _ in range(100):
            libceed.jit_compile(src, "port_HyperFSdF", [9, 10, 9], [9])
        out["compile_cached_s"] = (time.perf_counter() - t0) / 100
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
    ops = {}
    for tag, resource, locs in (("builtin", "/gpu/b200", None),
                                ("jit", "/gpu/b200:jit", {"jacob": f"{QF_PORT}:port_HyperFSdF"})):
        ceed = libceed.Ceed(resource)
        degrees, data, phys = setuplibceed.setup_all(ceed, mesh, "hyperFS", 4, multigrid="none", qf_locators=locs)
        d = data[-1]
        uc, rc = ceed.Vector(u.numel()), ceed.Vector(u.numel())
        r = torch.zeros_like(u)
        uc.set_array(u); rc.set_array(r)
        d.opApply.apply(uc, rc)          # gradu of the linearisation point
        uc.take_array(); rc.take_array()
        ops[tag] = (ceed, d, phys)
        torch.cuda.synchronize()
    assert ops["builtin"][1].opJacob.is_fused and not ops["jit"][1].opJacob.is_fused

    x = torch.randn_like(u)
    ys = {}
    for tag, (ceed, d, _) in ops.items():
        y = torch.zeros_like(u)
        xc, yc = ceed.Vector(u.numel()), ceed.Vector(u.numel())
        xc.set_array(x); yc.set_array(y)
        ys[tag] = (y, xc, yc, d)
    t = {"builtin": [], "jit": []}
    for _ in range(3):                   # alternate the two, several rounds
        for tag, (y, xc, yc, d) in ys.items():
            t[tag].append(timeit(lambda: d.opJacob.apply(xc, yc), a.reps))
    yb, yj = ys["builtin"][0], ys["jit"][0]
    rel = (torch.linalg.norm(yj - yb) / torch.linalg.norm(yb)).item()
    res.update({"fused_jacobian_ms": min(t["builtin"]), "jit_jacobian_ms": min(t["jit"]),
                "fused_jacobian_ms_all": t["builtin"], "jit_jacobian_ms_all": t["jit"],
                "jit_over_fused": min(t["jit"]) / min(t["builtin"]), "rel_diff_jit_vs_fused": rel})

    # K11 alone on the operator's own Q-vectors: deltadu (9), qdata (10), gradu (9) -> deltadv (9)
    ceed, d, phys = ops["jit"]
    nelem, nq = mesh.nelem, 5 ** 3
    def evec(rstr, vec, ncomp):
        ev = ceed.Vector(nelem * ncomp * nq)
        rstr.apply(vec, ev)
        return ev
    qd_e, gu_e = evec(d.Erestrictqdi, d.qdata, 10), evec(d.ErestrictGradui, d.gradu, 9)
    ddu = (torch.randn(nelem * 9 * nq, dtype=torch.float64, device="cuda") * 1e-2)
    out = torch.empty_like(ddu)
    h = libceed.jit_compile(QF_PORT, "port_HyperFSdF", [9, 10, 9], [9])   # the operator's program: cached
    import ctypes as C
    pin = (C.c_void_p * 3)(ddu.data_ptr(), qd_e.device_ptr(), gu_e.device_ptr())
    pout = (C.c_void_p * 1)(out.data_ptr())
    lib = libceed.lib
    lib.b200_jit_apply.argtypes = [C.c_int, C.c_void_p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                   C.c_void_p]
    def k11():
        libceed.b2(lib.b200_jit_apply(h, C.addressof(phys), C.sizeof(phys), nelem, nq, 3, pin, 1, pout))
    kt = min(timeit(k11, a.reps * 3) for _ in range(3))
    kbytes = nelem * nq * (9 + 10 + 9 + 9) * DP
    res.update({"k11_ms": kt, "k11_bytes": kbytes, "k11_tb_per_s": kbytes / (kt * 1e-3) / 1e12,
                "k11_share_of_hbm_bound": kbytes / HBM_BYTES_PER_S / (kt * 1e-3),
                "qvector_gb": nelem * nq * 9 * DP / 1e9})
    line = json.dumps(res)
    print(line, flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "a") as f:
            f.write(line + "\n")
    assert rel <= 1e-12, rel


if __name__ == "__main__":
    main()
