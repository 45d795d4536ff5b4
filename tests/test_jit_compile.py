"""The compile half of "/gpu/b200:jit" (csrc/b200_jit_src.c, csrc/b200_jit.cu), which needs no device: user QFunction
sources are read with their quoted includes inlined and compiled by NVRTC for sm_100a, with the generated kernel."""
import ctypes as C
import os
import subprocess

import pytest

from ceedpetscsolid_b200 import ceed as libceed

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QF_PORT = os.path.join(ROOT, "oracle", "qf_port.c")

# the stock field sizes of every QFunction of oracle/qf_port.c (setuplibceed.py: inputs, outputs)
STOCK = {
    "port_SetupGeo": ([9, 1], [10]),
    "port_LinElasF": ([9, 10], [9]), "port_LinElasdF": ([9, 10], [9]),
    "port_HyperSSF": ([9, 10], [9, 9]), "port_HyperSSdF": ([9, 10, 9], [9]),
    "port_HyperFSF": ([9, 10], [9, 9]), "port_HyperFSdF": ([9, 10, 9], [9]),
    "port_SetupConstantForce": ([3, 10], [3]), "port_SetupMMSForce": ([3, 10], [3]), "port_MMSTrueSoln": ([3], [3]),
    "port_LinElasEnergy": ([9, 10], [1]), "port_HyperSSEnergy": ([9, 10], [1]), "port_HyperFSEnergy": ([9, 10], [1]),
    "port_LinElasDiagnostic": ([3, 9, 10], [8]), "port_HyperSSDiagnostic": ([3, 9, 10], [8]),
    "port_HyperFSDiagnostic": ([3, 9, 10], [8]),
}


@pytest.mark.parametrize("name", sorted(STOCK))
def test_every_qf_port_function_compiles_for_sm100a(name):
    ins, outs = STOCK[name]
    h = libceed.jit_compile(QF_PORT, name, ins, outs)
    assert h >= 0
    prog = libceed.jit_program(h)
    assert f"b200_jit_{name}(" in prog and f'#line 1 "{QF_PORT}"' in prog


def test_identical_programs_are_compiled_once():
    libceed.jit_compile(QF_PORT, "port_HyperSSdF", [9, 10, 9], [9])
    n = libceed.jit_compile_count()
    h1 = libceed.jit_compile(QF_PORT, "port_HyperSSdF", [9, 10, 9], [9])
    h2 = libceed.jit_compile(QF_PORT, "port_HyperSSdF", [9, 10, 9], [9])
    assert h1 == h2 and libceed.jit_compile_count() == n
    libceed.jit_compile(QF_PORT, "port_HyperSSdF", [9, 10, 9, 1], [9])  # other field sizes: another kernel
    assert libceed.jit_compile_count() == n + 1


def _nvrtc():
    for name in ("libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12"):
        try:
            return C.CDLL(name)
        except OSError:
            pass
    pytest.fail("NVRTC not found")


def test_generated_hyperfs_jacobian_kernel_has_no_stack_frame_or_spills():
    """the backend's program for port_HyperFSdF, recompiled with ptxas -v: per-field register arrays stay in registers"""
    prog = libceed.jit_program(libceed.jit_compile(QF_PORT, "port_HyperFSdF", [9, 10, 9], [9])).encode()
    nv = _nvrtc()
    p = C.c_void_p()
    hdr = b"typedef int CeedInt;\ntypedef double CeedScalar;\n"
    assert nv.nvrtcCreateProgram(C.byref(p), prog, QF_PORT.encode(), 3, (C.c_char_p * 3)(hdr, hdr, b"\n"),
                                 (C.c_char_p * 3)(b"ceed.h", b"ceed/ceed.h", b"math.h")) == 0
    opts = [b"--gpu-architecture=sm_100a", b"-default-device", b"--std=c++17", b"--ptxas-options=-v"]
    rc = nv.nvrtcCompileProgram(p, len(opts), (C.c_char_p * len(opts))(*opts))
    n = C.c_size_t()
    nv.nvrtcGetProgramLogSize(p, C.byref(n))
    log = C.create_string_buffer(n.value)
    nv.nvrtcGetProgramLog(p, log)
    nv.nvrtcDestroyProgram(C.byref(p))
    text = log.value.decode()
    assert rc == 0, text
    assert "b200_jit_port_HyperFSdF" in text
    assert "0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads" in text, text


HELPER = """#ifndef MY_HELPER_H
#define MY_HELPER_H
static inline CeedScalar twice(CeedScalar x) { return 2 * x; }
#endif
"""

USER = """#include <ceed.h>
#include <math.h>
#include "sub/helper.h"
#include "sub/helper.h"
CEED_QFUNCTION(Scale)(void *ctx, const CeedInt Q, const CeedScalar *const *in, CeedScalar *const *out) {
  const CeedScalar (*u)[CEED_Q_VLA] = (const CeedScalar(*)[CEED_Q_VLA])in[0];
  CeedScalar (*v)[CEED_Q_VLA] = (CeedScalar(*)[CEED_Q_VLA])out[0];
  const CeedScalar s = *(const CeedScalar *)ctx;
  CeedPragmaSIMD
  for (CeedInt i = 0; i < Q; i++)
    for (int c = 0; c < 3; c++) v[c][i] = s * twice(sqrt(fabs(u[c][i])));
  return 0;
}
"""


def test_a_header_with_a_local_helper_header_compiles(tmp_path):
    (tmp_path / "sub").mkdir()
    (tmp_path / "sub" / "helper.h").write_text(HELPER)
    (tmp_path / "user.h").write_text(USER)
    prog = libceed.jit_program(libceed.jit_compile(tmp_path / "user.h", "Scale", [3], [3]))
    helper = str(tmp_path / "sub" / "helper.h")
    assert prog.count(f'#line 1 "{helper}"') == 2     # inlined where it is included, guard and all
    assert f'#line 4 "{tmp_path / "user.h"}"' in prog  # back in the user file after the first include
    assert "#include <ceed.h>" in prog                 # angle includes stay for NVRTC's in-memory headers


def test_a_syntax_error_names_the_user_file_and_line(tmp_path):
    (tmp_path / "sub").mkdir()
    (tmp_path / "sub" / "helper.h").write_text(HELPER.replace("return 2 * x;", "return 2 * x  /* no semicolon */"))
    (tmp_path / "user.h").write_text(USER)
    with pytest.raises(libceed.CeedError) as e:
        libceed.jit_compile(tmp_path / "user.h", "Scale", [3], [3])
    msg = str(e.value)
    assert "NVRTC could not compile" in msg and f"{tmp_path / 'sub' / 'helper.h'}(3)" in msg, msg
    (tmp_path / "sub" / "helper.h").write_text(HELPER)
    (tmp_path / "user.h").write_text(USER.replace("v[c][i] = s *", "v[c][i] = s * undeclared_name *"))
    with pytest.raises(libceed.CeedError, match=r"user\.h\(11\).*undeclared_name"):
        libceed.jit_compile(tmp_path / "user.h", "Scale", [3], [3])


def test_a_missing_file_is_named(tmp_path):
    missing = tmp_path / "nowhere" / "model.h"
    with pytest.raises(libceed.CeedError, match=f"cannot read the QFunction source file \"{missing}\""):
        libceed.jit_compile(missing, "Model", [9], [9])


def test_bad_names_and_field_sizes_are_refused(tmp_path):
    (tmp_path / "sub").mkdir()
    (tmp_path / "sub" / "helper.h").write_text(HELPER)
    (tmp_path / "user.h").write_text(USER)
    with pytest.raises(libceed.CeedError, match="not a C identifier"):
        libceed.jit_compile(tmp_path / "user.h", "Scale; int x", [3], [3])
    with pytest.raises(libceed.CeedError, match="65 components"):
        libceed.jit_compile(tmp_path / "user.h", "Scale", [65], [3])


def test_the_library_has_no_link_time_dependency_on_nvrtc():
    out = subprocess.run(["readelf", "-d", libceed.LIBPATH], capture_output=True, text=True, check=True).stdout
    needed = [line for line in out.splitlines() if "(NEEDED)" in line]
    assert needed and not any("nvrtc" in line for line in needed), needed
