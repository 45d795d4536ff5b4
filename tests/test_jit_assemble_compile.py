"""The compile half of K13, the element-matrix kernel of a trilinear level generated around a JIT-compiled user
QFunction (csrc/b200_jit_assemble.cuh, csrc/b200_jit.cu), which needs no device."""
import re

import pytest

from ceedpetscsolid_b200 import ceed as libceed
from jit_models import EXTRA_FIELDS, EXTRA_IN, EXTRA_OUT
from test_jit_fused_compile import QF_PORT, ptxas_log

JACOBIANS = {"port_LinElasdF": ([9, 10], [9]), "port_HyperSSdF": ([9, 10, 9], [9]), "port_HyperFSdF": ([9, 10, 9], [9])}


def assemble(name, Q, path=QF_PORT, ins=None, outs=None, ai=0, ao=0, P=2):
    ins, outs = (ins, outs) if ins is not None else JACOBIANS[name]
    return libceed.jit_assemble_compile(path, name, ins, outs, ai, ao, P, Q)


@pytest.mark.parametrize("Q", [2, 3, 4, 5])
@pytest.mark.parametrize("name", sorted(JACOBIANS))
def test_stock_jacobians_compile_at_every_q(name, Q):
    prog = libceed.jit_program(assemble(name, Q))
    assert f"b200_jit_assemble_{name}(" in prog and f"b200_jit_assemble_tail_{name}(" in prog
    assert f'#line 1 "{QF_PORT}"' in prog
    EB = libceed.lib.b200_elems_per_block(Q)
    assert f"#define B200_K13_Q {Q}\n" in prog and f"#define B200_K13_EB {EB}\n" in prog
    assert f"#define B200_K13_NT {24 * EB}\n" in prog


def test_a_model_whose_active_fields_are_not_field_0_compiles(tmp_path):
    (tmp_path / "extra.h").write_text(EXTRA_FIELDS)
    prog = libceed.jit_program(assemble("ExtraF", 5, tmp_path / "extra.h", EXTRA_IN, EXTRA_OUT, 1, 1))
    # passive inputs 0 (1 component) and 2 (10) are loaded, the unit vectors go to input 1, output 1 is the tangent
    assert "f.in[0] + grp * 1 + pos" in prog and "f.in[2] + grp * 10 + pos" in prog
    assert "in1[c] = c == s ? 1.0 : 0.0" in prog and "d[s * 9 + o] = out1[o]" in prog
    # passive outputs are never stored
    assert "f.out" not in prog.split('#line 1 "b200_jit_assemble_prefix"')[1]


def test_hyperfs_jacobian_at_q5_has_no_stack_frame_or_spills():
    """the backend's K13 program for port_HyperFSdF at (2, 5), recompiled with ptxas -v: both kernels (full groups and
    the tail group) keep the user function's arrays and the 24 row sums in registers"""
    log = ptxas_log(libceed.jit_program(assemble("port_HyperFSdF", 5)))
    for kernel in ("b200_jit_assemble_port_HyperFSdF", "b200_jit_assemble_tail_port_HyperFSdF"):
        block = log.split(f"Compiling entry function '{kernel}'")[1].split("Compiling entry function")[0]
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in block, block
        assert int(re.search(r"Used (\d+) registers", block).group(1)) <= 255


def test_identical_requests_compile_once(tmp_path):
    src = tmp_path / "qf_port_copy.c"
    src.write_text(open(QF_PORT).read())
    n0 = libceed.jit_compile_count()
    h1 = assemble("port_HyperSSdF", 4, path=src)
    h2 = assemble("port_HyperSSdF", 4, path=src)
    assert h1 == h2 and libceed.jit_compile_count() == n0 + 1
    assert assemble("port_HyperSSdF", 5, path=src) != h1      # another Q: another program
    # the fused apply program of the same function and (P, Q) is another program too
    assert libceed.jit_fused_compile(src, "port_HyperSSdF", *JACOBIANS["port_HyperSSdF"], 0, 0, 2, 5) != h1
    assert libceed.jit_compile_count() == n0 + 3


def test_other_levels_and_field_widths_are_refused():
    with pytest.raises(libceed.CeedError, match=r"trilinear \(P = 2\) levels only, not P = 3"):
        assemble("port_HyperFSdF", 5, P=3)
    with pytest.raises(libceed.CeedError, match=r"\(P, Q\) = \(2, 6\) is not instantiated"):
        assemble("port_HyperFSdF", 6)
    with pytest.raises(libceed.CeedError, match="active input and output must be fields of 9 components"):
        assemble("port_HyperFSdF", 5, ai=1)
