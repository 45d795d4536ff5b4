"""The compile half of K12, the fused operator kernel generated around a JIT-compiled user QFunction
(csrc/b200_jit_fused.cuh, csrc/b200_jit.cu), which needs no device."""
import ctypes as C
import os
import re

import pytest

from ceedpetscsolid_b200 import ceed as libceed
from jit_models import EXTRA_FIELDS, EXTRA_IN, EXTRA_OUT

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")
PQ = [(2, 2), (2, 3), (3, 3), (2, 4), (3, 4), (4, 4), (2, 5), (3, 5), (4, 5), (5, 5)]   # B200_FOR_PQ
# the stock residual and Jacobian shapes (setuplibceed.py): inputs, outputs; the active fields are the first ones
STOCK = {
    "port_LinElasF": ([9, 10], [9]), "port_LinElasdF": ([9, 10], [9]),
    "port_HyperSSF": ([9, 10], [9, 9]), "port_HyperSSdF": ([9, 10, 9], [9]),
    "port_HyperFSF": ([9, 10], [9, 9]), "port_HyperFSdF": ([9, 10, 9], [9]),
}


def fused(name, P, Q, path=QF_PORT, ins=None, outs=None, ai=0, ao=0):
    ins, outs = (ins, outs) if ins is not None else STOCK[name]
    return libceed.jit_fused_compile(path, name, ins, outs, ai, ao, P, Q)


@pytest.mark.parametrize("P,Q", PQ)
@pytest.mark.parametrize("name", sorted(STOCK))
def test_stock_fused_programs_compile_at_every_pq(name, P, Q):
    prog = libceed.jit_program(fused(name, P, Q))
    assert f"b200_jit_fused_{name}(" in prog and f"b200_jit_fused_tail_{name}(" in prog
    assert f'#line 1 "{QF_PORT}"' in prog          # NVRTC messages name the user's file
    assert f"#define B200_K12_P {P}\n" in prog and f"#define B200_K12_Q {Q}\n" in prog


@pytest.mark.parametrize("P,Q", PQ)
def test_emitted_lattice_constants_are_the_builtin_layout(P, Q):
    prog = libceed.jit_program(fused("port_LinElasdF", P, Q))
    got = [int(re.search(rf"#define B200_K12_{k} (\d+)\n", prog).group(1)) for k in ("SY", "SZ", "SC", "SE", "EB", "NT")]
    want = (C.c_int * 6)()
    assert libceed.lib.b200_apply_smem_layout(P, Q, want) == 0
    assert got == list(want)


def ptxas_log(prog):
    nv = None
    for lib in ("libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12"):
        try:
            nv = C.CDLL(lib)
            break
        except OSError:
            pass
    assert nv is not None, "NVRTC not found"
    p = C.c_void_p()
    hdr = b"typedef int CeedInt;\ntypedef double CeedScalar;\n"
    assert nv.nvrtcCreateProgram(C.byref(p), prog.encode(), QF_PORT.encode(), 3, (C.c_char_p * 3)(hdr, hdr, b"\n"),
                                 (C.c_char_p * 3)(b"ceed.h", b"ceed/ceed.h", b"math.h")) == 0
    opts = [b"--gpu-architecture=sm_100a", b"-default-device", b"--std=c++17", b"--ptxas-options=-v"]
    rc = nv.nvrtcCompileProgram(p, len(opts), (C.c_char_p * len(opts))(*opts))
    n = C.c_size_t()
    nv.nvrtcGetProgramLogSize(p, C.byref(n))
    log = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(p, log)
    nv.nvrtcDestroyProgram(C.byref(p))
    assert rc == 0, log.value.decode()
    return log.value.decode()


def test_fused_hyperfs_jacobian_at_p5_q5_has_no_stack_frame_or_spills():
    """the backend's K12 program for port_HyperFSdF at (5, 5), recompiled with ptxas -v: both kernels (full groups
    and the tail group) keep the user function's arrays in registers"""
    log = ptxas_log(libceed.jit_program(fused("port_HyperFSdF", 5, 5)))
    for kernel in ("b200_jit_fused_port_HyperFSdF", "b200_jit_fused_tail_port_HyperFSdF"):
        block = log.split(f"Compiling entry function '{kernel}'")[1].split("Compiling entry function")[0]
        assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in block, block


def test_a_model_with_extra_passive_input_and_output_compiles(tmp_path):
    (tmp_path / "extra.h").write_text(EXTRA_FIELDS)
    h = libceed.jit_fused_compile(tmp_path / "extra.h", "ExtraF", EXTRA_IN, EXTRA_OUT, 1, 1, 4, 5)
    prog = libceed.jit_program(h)
    # passive fields by declaration order: input 0 (1 component), input 2 (10), output 0 (3), output 2 (1)
    assert "f.in[0] + grp * 1 + pos" in prog and "f.in[2] + grp * 10 + pos" in prog
    assert "f.out[0] + grp * 3 + pos" in prog and "f.out[2] + grp * 1 + pos" in prog
    assert "in1[d * 3 + c] = H[c][d]" in prog and "W[c][kk] = out1[kk * 3 + c]" in prog


def test_identical_requests_compile_once(tmp_path):
    src = tmp_path / "qf_port_copy.c"
    src.write_text(open(QF_PORT).read())
    n0 = libceed.jit_compile_count()
    h1 = fused("port_HyperSSdF", 3, 4, path=src)
    h2 = fused("port_HyperSSdF", 3, 4, path=src)
    assert h1 == h2 and libceed.jit_compile_count() == n0 + 1
    assert fused("port_HyperSSdF", 3, 5, path=src) != h1      # another (P, Q): another program
    assert libceed.jit_compile_count() == n0 + 2


def test_shapes_without_a_fused_layout_are_refused():
    with pytest.raises(libceed.CeedError, match=r"\(P, Q\) = \(5, 6\) has no fused lattice layout"):
        fused("port_HyperFSdF", 5, 6)
    with pytest.raises(libceed.CeedError, match="active input and output must be fields of 9 components"):
        fused("port_HyperFSdF", 5, 5, ai=1)
