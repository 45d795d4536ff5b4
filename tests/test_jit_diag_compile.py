"""The compile half of K14, the operator-diagonal kernel generated around a JIT-compiled user QFunction
(csrc/b200_jit_diag.cuh, csrc/b200_jit.cu), which needs no device."""
import ctypes as C
import re

import pytest

from ceedpetscsolid_b200 import ceed as libceed
from jit_models import EXTRA_FIELDS, EXTRA_IN, EXTRA_OUT
from test_jit_fused_compile import PQ, QF_PORT, ptxas_log

JACOBIANS = {"port_LinElasdF": ([9, 10], [9]), "port_HyperSSdF": ([9, 10, 9], [9]), "port_HyperFSdF": ([9, 10, 9], [9])}
LATTICE = ("SY", "SZ", "SC", "SE", "EB", "NT")


def diag(name, P, Q, path=QF_PORT, ins=None, outs=None, ai=0, ao=0):
    ins, outs = (ins, outs) if ins is not None else JACOBIANS[name]
    return libceed.jit_diag_compile(path, name, ins, outs, ai, ao, P, Q)


@pytest.mark.parametrize("P,Q", PQ)
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_stock_jacobians_compile_at_every_pq_with_the_k12_lattice(name, P, Q):
    prog = libceed.jit_program(diag(name, P, Q))
    assert f"b200_jit_diag_{name}(" in prog and f"b200_jit_diag_tail_{name}(" in prog
    assert f'#line 1 "{QF_PORT}"' in prog          # NVRTC messages name the user's file
    assert f"#define B200_K14_P {P}\n" in prog and f"#define B200_K14_Q {Q}\n" in prog
    got = [int(re.search(rf"#define B200_K14_{k} (\d+)\n", prog).group(1)) for k in LATTICE]
    want = (C.c_int * 6)()
    assert libceed.lib.b200_apply_smem_layout(P, Q, want) == 0
    assert got == list(want)
    k12 = libceed.jit_program(libceed.jit_fused_compile(QF_PORT, name, *JACOBIANS[name], 0, 0, P, Q))
    assert got == [int(re.search(rf"#define B200_K12_{k} (\d+)\n", k12).group(1)) for k in LATTICE]


def test_a_model_whose_active_fields_are_not_field_0_compiles(tmp_path):
    (tmp_path / "extra.h").write_text(EXTRA_FIELDS)
    prog = libceed.jit_program(diag("ExtraF", 5, 5, tmp_path / "extra.h", EXTRA_IN, EXTRA_OUT, 1, 1))
    generated = prog.split('#line 1 "b200_jit_diag_prefix"')[1]
    # only the passive inputs 0 (1 component) and 2 (10) are loaded and prefetched; the unit vectors go to input 1
    assert "f.in[0] + grp * 1 + pos" in generated and "f.in[2] + grp * 10 + pos" in generated
    assert "f.in[1]" not in generated
    assert "b200_k14_l2(f.in[0] + grp * 1, npts * 1)" in generated
    assert "b200_k14_l2(f.in[2] + grp * 10, npts * 10)" in generated
    assert "in1[c] = c == m * 3 + comp ? 1.0 : 0.0" in generated
    # output 1 is the tangent; passive outputs are never stored
    assert "comp == 0 ? out1[kk * 3]" in generated
    assert "f.out" not in generated


def test_hyperfs_jacobian_at_p5_q5_has_no_stack_frame_or_spills():
    """the backend's K14 program for port_HyperFSdF at (5, 5), recompiled with ptxas -v: both kernels (full groups and
    the tail group) keep the user function's arrays in registers"""
    log = ptxas_log(libceed.jit_program(diag("port_HyperFSdF", 5, 5)))
    for kernel in ("b200_jit_diag_port_HyperFSdF", "b200_jit_diag_tail_port_HyperFSdF"):
        block = log.split(f"Compiling entry function '{kernel}'")[1].split("Compiling entry function")[0]
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in block, block


def test_identical_requests_compile_once(tmp_path):
    src = tmp_path / "qf_port_copy.c"
    src.write_text(open(QF_PORT).read())
    ins, outs = JACOBIANS["port_HyperSSdF"]
    n0 = libceed.jit_compile_count()
    h1 = diag("port_HyperSSdF", 3, 5, path=src)
    h2 = diag("port_HyperSSdF", 3, 5, path=src)
    assert h1 == h2 and libceed.jit_compile_count() == n0 + 1
    assert diag("port_HyperSSdF", 2, 5, path=src) != h1       # another (P, Q): another program
    # the fused apply and the assembly programs of the same function are other programs too
    assert libceed.jit_fused_compile(src, "port_HyperSSdF", ins, outs, 0, 0, 2, 5) != h1
    assert libceed.jit_assemble_compile(src, "port_HyperSSdF", ins, outs, 0, 0, 2, 5) != h1
    assert libceed.jit_compile_count() == n0 + 4


def test_shapes_without_a_fused_layout_and_other_field_widths_are_refused():
    with pytest.raises(libceed.CeedError, match=r"b200_jit_diag_compile: \(P, Q\) = \(5, 6\) is not instantiated"):
        diag("port_HyperFSdF", 5, 6)
    with pytest.raises(libceed.CeedError, match="active input and output must be fields of 9 components"):
        diag("port_HyperFSdF", 5, 5, ai=1)
    with pytest.raises(libceed.CeedError, match="active input and output must be fields of 9 components"):
        diag("port_HyperFSdF", 5, 5, ins=[9, 10, 8], outs=[9], ai=2)
