// K11: user QFunctions compiled at run time with NVRTC ("/gpu/b200:jit").
//
// One generated kernel per (program text, QFunction name, field sizes): one thread per (element, point), grid-stride.
// Each input field is loaded from its Q-vector [elem][comp][nq] into a register array (coalesced across q), the user
// function is called with Q = 1, and the outputs are stored the same way.  All parameters are __grid_constant__: the
// context bytes (up to B200_JIT_MAX_CTX, copied from the caller's host pointer at every launch), the field pointers,
// nelem and nq.  The user function's return code is ignored, as libCEED's CUDA backends do.
//
// Compile half (b200_jit_compile): needs no device.  NVRTC is opened with dlopen on first use, so libceed_b200.so has
// no link-time dependency on it.  Each distinct program (text plus options) is compiled once per process.
// Load half (b200_jit_apply): the cubin is loaded once with cudaLibraryLoadData.  A cudaLibrary_t is
// context-independent: the runtime loads its kernel into each device's context on first use there.
//
// K12 (b200_jit_fused_compile / b200_jit_fused_apply): the same user program with the fused operator kernel of
// b200_jit_fused.cuh around it, for one (P, Q) of B200_FOR_PQ and one assignment of the fields to the active gradient
// and the passive q-blocked vectors.  The template is embedded at build time (b200_jit_fused.inc, a raw string made
// from the header by the Makefile); the lattice constants come from b200_apply_smem_layout, so the built-in and the
// generated kernels cannot disagree on the layout.
//
// K13 (b200_jit_assemble_compile / b200_jit_assemble_apply): the same user program with b200_jit_assemble.cuh around
// it, the element matrices of a trilinear (P = 2) level in the CeedOperatorLinearAssemble layout, from the point
// tangents the user function gives for the 9 unit active inputs.  Embedded the same way (b200_jit_assemble.inc).
//
// K14 (b200_jit_diag_compile / b200_jit_diag_apply): the same user program with b200_jit_diag.cuh around it, the
// operator diagonal (CeedOperatorLinearAssembleDiagonal) at one (P, Q) of B200_FOR_PQ, from 3 unit-input calls of the
// user function per point and component, contracted as the built-in diagonal (K3) does.  The lattice constants come
// from b200_apply_smem_layout, as for K12.  Embedded the same way (b200_jit_diag.inc).
//
// The four kinds share the host code: the emitters of the parts of the program text they have in common, one compile
// path (checks, cache), one apply prologue (handle, lazy load, shared-memory limit, context) and, for K12 to K14, one
// launcher of the full element groups and the one-CTA tail.
#include <dlfcn.h>
#include <limits.h>
#include <nvrtc.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "b200_common.cuh"

namespace {

const char *const kOptions[] = {"--gpu-architecture=sm_100a", "-default-device", "--std=c++17"};
const int kNumOptions = 3;
const size_t kMaxLog = 4096;

// libCEED's user-QFunction vocabulary for the device (Q = 1 per call, so CEED_Q_VLA is 1)
const char *const kCeedHeader =
    "#ifndef B200_JIT_CEED_H\n"
    "#define B200_JIT_CEED_H\n"
    "typedef int CeedInt;\n"
    "typedef double CeedScalar;\n"
    "#define CEED_QFUNCTION(name) static int name\n"
    "#define CEED_QFUNCTION_HELPER static inline\n"
    "#define CEED_Q_VLA 1\n"
    "#define CeedPragmaSIMD\n"
    "#define CEED_ERROR_SUCCESS 0\n"
    "#endif\n";
// the math functions are NVRTC built-ins
const char *const kMathHeader = "/* math functions: NVRTC built-ins */\n";

struct Nvrtc {
  bool tried = false;
  void *h = nullptr;
  nvrtcResult (*create)(nvrtcProgram *, const char *, const char *, int, const char *const *, const char *const *);
  nvrtcResult (*compile)(nvrtcProgram, int, const char *const *);
  nvrtcResult (*log_size)(nvrtcProgram, size_t *);
  nvrtcResult (*log)(nvrtcProgram, char *);
  nvrtcResult (*cubin_size)(nvrtcProgram, size_t *);
  nvrtcResult (*cubin)(nvrtcProgram, char *);
  nvrtcResult (*destroy)(nvrtcProgram *);
  const char *(*errstr)(nvrtcResult);
};

// the device templates (b200_jit_fused.cuh, b200_jit_assemble.cuh, b200_jit_diag.cuh) as strings
const char *const kFusedTemplate =
#include "b200_jit_fused.inc"
    ;
const char *const kAssembleTemplate =
#include "b200_jit_assemble.inc"
    ;
const char *const kDiagTemplate =
#include "b200_jit_diag.inc"
    ;

// K12 blocks per SM asked of ptxas for the full-group kernel (__launch_bounds__ min blocks): 128 threads x 3 blocks
// leave 168 registers a thread.  Measured at P = Q = 5, C3 (profiles/jit_fused_ctas_ab.txt): the fastest setting at
// which port_HyperFSdF neither spills nor has a stack frame; 4 blocks (128 registers) ran 7 % faster with 112 bytes of
// spills.  B200_JIT_FUSED_CTAS overrides it (tuning runs).
const int kFusedCtas = 3;

// K13 blocks per SM asked of ptxas for the full-group kernel, and whether the 9 unit-input calls of the user function
// are unrolled (NVCC may then share their input-independent part) or kept rolled.  Chosen by measurement at Q = 5,
// C3 (profiles/jit_assemble_ab.txt); B200_JIT_ASSEMBLE_CTAS and B200_JIT_ASSEMBLE_UNROLL override them (tuning runs).
const int kAssembleCtas = 2;
const int kAssembleUnroll = 0;
// most point tangents a K13 CTA holds in shared memory at once (81 doubles each)
const int kAssembleMaxChunk = 128;

// K14 blocks of 128 threads per SM asked of ptxas for the full-group kernel.  Measured on the three levels of C3
// (profiles/jit_diag_ab.txt): the fastest setting at which port_HyperFSdF neither spills nor has a stack frame
// (162 registers at P = Q = 5); 4 blocks (128 registers) ran 6 to 7 % faster with 88 bytes of spills.
// B200_JIT_DIAG_CTAS overrides it (tuning runs).
const int kDiagCtas = 2;

// K11 (point kernel), K12 (fused apply), K13 (p = 1 assembly), K14 (operator diagonal)
enum Kind { kPoint, kFused, kAssemble, kDiag };
// per kind: the name in its kernels and files (b200_jit_<name>_<Name>, b200_jit_<name>.cuh), the tag of its device
// types (b200_<tag>_fields_t) and its device template
struct KindInfo {
  const char *name, *tag, *tmpl;
};
const KindInfo kKinds[] = {{"", "jit", nullptr},
                           {"fused", "k12", kFusedTemplate},
                           {"assemble", "k13", kAssembleTemplate},
                           {"diag", "k14", kDiagTemplate}};

struct Entry {
  std::string key;  // options + program text
  Kind kind = kPoint;
  // b200_jit_<Name> (K11), or b200_jit_<kind>_<Name> for the full element groups and b200_jit_<kind>_tail_<Name> for
  // the partial group at the end of a range
  std::string kernel, kernel_tail;
  std::vector<char> cubin;
  int nin = 0, nout = 0, in_size[B200_JIT_MAXF] = {}, out_size[B200_JIT_MAXF] = {};
  cudaLibrary_t lib = nullptr;
  cudaKernel_t fn = nullptr, fn_tail = nullptr;
  // K12 to K14: the basis, the active fields, EB elements a group on NT threads a CTA, the dynamic shared memory
  int P = 0, Q = 0, ai = -1, ao = -1, EB = 0, NT = 0;
  size_t smem = 0;
  unsigned long long smem_set = 0;  // devices on which the dynamic shared-memory limit was raised
};

std::mutex g_mu;
Nvrtc g_nv;
std::vector<Entry *> g_entries;
unsigned long long g_compiles = 0;

// the kernel parameters, laid out as the generated kernel declares them (K13 and K14 take only `in`)
struct alignas(16) JitCtx { unsigned char b[B200_JIT_MAX_CTX]; };
struct JitFields { const double *in[B200_JIT_MAXF]; double *out[B200_JIT_MAXF]; };

// b200::set_error_msg of "<fn>: <the formatted message>"
__attribute__((format(printf, 2, 3))) int error(const char *fn, const char *fmt, ...) {
  char msg[320];
  const int n = snprintf(msg, sizeof msg, "%s: ", fn);
  va_list a;
  va_start(a, fmt);
  vsnprintf(msg + n, sizeof msg - n, fmt, a);
  va_end(a);
  return b200::set_error_msg(msg);
}

template <class F>
bool sym(F &f, const char *name) {
  f = reinterpret_cast<F>(dlsym(g_nv.h, name));
  return f != nullptr;
}

int open_nvrtc() {
  if (g_nv.h) return 0;
  if (!g_nv.tried) {
    g_nv.tried = true;
    const char *names[] = {"libnvrtc.so.12", "/usr/local/cuda/lib64/libnvrtc.so.12"};
    for (const char *n : names)
      if ((g_nv.h = dlopen(n, RTLD_NOW | RTLD_LOCAL))) break;
    if (g_nv.h && !(sym(g_nv.create, "nvrtcCreateProgram") && sym(g_nv.compile, "nvrtcCompileProgram") &&
                    sym(g_nv.log_size, "nvrtcGetProgramLogSize") && sym(g_nv.log, "nvrtcGetProgramLog") &&
                    sym(g_nv.cubin_size, "nvrtcGetCUBINSize") && sym(g_nv.cubin, "nvrtcGetCUBIN") &&
                    sym(g_nv.destroy, "nvrtcDestroyProgram") && sym(g_nv.errstr, "nvrtcGetErrorString"))) {
      dlclose(g_nv.h);
      g_nv.h = nullptr;
    }
  }
  if (!g_nv.h)
    return b200::set_error_msg("b200_jit: NVRTC is not available (tried libnvrtc.so.12 and "
                               "/usr/local/cuda/lib64/libnvrtc.so.12)");
  return 0;
}

bool is_identifier(const char *s) {
  if (!s || !((*s >= 'A' && *s <= 'Z') || (*s >= 'a' && *s <= 'z') || *s == '_')) return false;
  for (; *s; s++)
    if (!((*s >= 'A' && *s <= 'Z') || (*s >= 'a' && *s <= 'z') || (*s >= '0' && *s <= '9') || *s == '_')) return false;
  return true;
}

// ---- the generated program text ----------------------------------------------------------------------------------

// the text under construction; add appends one printf-formatted piece of any length
struct Text {
  std::string s;
  __attribute__((format(printf, 2, 3))) void add(const char *fmt, ...) {
    va_list a, b;
    va_start(a, fmt);
    va_copy(b, a);
    const int n = vsnprintf(nullptr, 0, fmt, a);
    const size_t at = s.size();
    s.resize(at + n + 1);
    vsnprintf(&s[at], n + 1, fmt, b);
    s.resize(at + n);
    va_end(b);
    va_end(a);
  }
};

// the context and field structs the kernels take (JitCtx, JitFields); K13 and K14 have no output fields
void emit_structs(Text &t, const Entry &en) {
  t.add("struct alignas(16) b200_jit_ctx_t { unsigned char b[%d]; };\n", B200_JIT_MAX_CTX);
  if (en.kind == kPoint || en.kind == kFused)
    t.add("struct b200_%s_fields_t { const double *in[%d]; double *out[%d]; };\n", kKinds[en.kind].tag, B200_JIT_MAXF,
          B200_JIT_MAXF);
  else
    t.add("struct b200_%s_fields_t { const double *in[%d]; };\n", kKinds[en.kind].tag, B200_JIT_MAXF);
}

// K12, K14: the basis and the lattice of b200_apply_smem_layout {SY, SZ, SC, SE, EB, NT} as B200_<K>_* constants
void emit_lattice(Text &t, const char *K, const Entry &en, const int *lay) {
  t.add("#define B200_%s_P %d\n#define B200_%s_Q %d\n", K, en.P, K, en.Q);
  const char *const names[6] = {"SY", "SZ", "SC", "SE", "EB", "NT"};
  for (int j = 0; j < 6; j++) t.add("#define B200_%s_%s %d\n", K, names[j], lay[j]);
}

// K12 to K14: the register array of every input at indent ind.  A passive input is loaded with ld from its q-blocked
// slab at group offset grp, lane pos and component stride cs; the active one gets `active` (a format taking its index).
void emit_inputs(Text &t, const Entry &en, int ind, const char *ld, const char *active) {
  for (int i = 0; i < en.nin; i++) {
    t.add("%*sdouble in%d[%d];\n", ind, "", i, en.in_size[i]);
    if (i == en.ai)
      t.add(active, i);
    else
      t.add("%*s{ const double *p = f.in[%d] + grp * %d + pos;\n#pragma unroll\n"
            "%*sfor (int c = 0; c < %d; c++) in%d[c] = %s(p + c * cs); }\n",
            ind, "", i, en.in_size[i], ind + 2, "", en.in_size[i], i, ld);
  }
}

// the zeroed output arrays, the ins / outs arrays and the call of the user function with Q = 1, at indent ind
void emit_call(Text &t, const Entry &en, const char *name, int ind) {
  for (int i = 0; i < en.nout; i++) t.add("%*sdouble out%d[%d] = {};\n", ind, "", i, en.out_size[i]);
  t.add("%*sconst double *ins[] = {", ind, "");
  for (int i = 0; i < en.nin; i++) t.add("%sin%d", i ? ", " : "", i);
  t.add("};\n%*sdouble *outs[] = {", ind, "");
  for (int i = 0; i < en.nout; i++) t.add("%sout%d", i ? ", " : "", i);
  t.add("};\n%*s(void)%s((void *)ctx.b, 1, ins, outs);\n", ind, "", name);
}

// K12 to K14: the kind's device template, then its kernel for full element groups (`blocks` blocks of NT threads per
// SM asked of ptxas) and its tail kernel, which runs as one CTA: occupancy is moot there, so it gets every register it
// wants.  params: the parameters after nelem; args: their names, passed on to b200_<tag>_body.
void emit_kernels(Text &t, const Entry &en, const char *name, int blocks, const char *params, const char *args) {
  const KindInfo &k = kKinds[en.kind];
  t.add("#line 1 \"b200_jit_%s.cuh\"\n", k.name);
  t.s += k.tmpl;
  t.add("\n#line 1 \"b200_jit_%s_kernels\"\n", k.name);
  for (int v = 0; v < 2; v++)
    t.add("extern \"C\" __global__ void __launch_bounds__(%d, %d) b200_jit_%s_%s%s(\n"
          "    const __grid_constant__ b200_%s_mats_t m, const __grid_constant__ b200_jit_ctx_t ctx,\n"
          "    const __grid_constant__ b200_%s_fields_t f, const int nelem, %s) {\n"
          "  b200_%s_body<%s>(m, ctx, f, nelem, %s);\n}\n",
          en.NT, v ? 1 : blocks, k.name, v ? "tail_" : "", name, k.tag, k.tag, params, k.tag, v ? "false" : "true",
          args);
}

// K11: the grid-stride point kernel
std::string generated_kernel(const char *name, const Entry &en) {
  Text t;
  t.s += "\n#line 1 \"b200_jit_kernel\"\n";
  emit_structs(t, en);
  t.add("extern \"C\" __global__ void __launch_bounds__(128) b200_jit_%s(const __grid_constant__ b200_jit_ctx_t ctx,\n"
        "    const __grid_constant__ b200_jit_fields_t f, const int nelem, const int nq) {\n", name);
  t.s += "  const long long total = (long long)nelem * nq;\n"
         "  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;\n"
         "       t += (long long)gridDim.x * blockDim.x) {\n"
         "    const long long e = t / nq, q = t - e * nq;\n";
  for (int i = 0; i < en.nin; i++)
    t.add("    double in%d[%d];\n"
          "    { const double *p = f.in[%d] + e * %dLL * nq + q;\n"
          "#pragma unroll\n"
          "      for (int c = 0; c < %d; c++) in%d[c] = p[(long long)c * nq]; }\n",
          i, en.in_size[i], i, en.in_size[i], en.in_size[i], i);
  emit_call(t, en, name, 4);
  for (int i = 0; i < en.nout; i++)
    t.add("    { double *p = f.out[%d] + e * %dLL * nq + q;\n"
          "#pragma unroll\n"
          "      for (int c = 0; c < %d; c++) p[(long long)c * nq] = out%d[c]; }\n",
          i, en.out_size[i], en.out_size[i], i);
  t.s += "  }\n}\n";
  return t.s;
}

// K12: the prefix the template expects (constants, parameter structs, the point adapter that maps H to the active
// input and the active output to W, and stores or adds the passive outputs), the template, the kernels
std::string generated_fused(const char *name, const Entry &en, const int *lay, int ctas) {
  Text t;
  t.s += "\n#line 1 \"b200_jit_fused_prefix\"\n";
  emit_lattice(t, "K12", en, lay);
  emit_structs(t, en);
  t.s += "__device__ __forceinline__ void b200_k12_point(const b200_jit_ctx_t &ctx, const b200_k12_fields_t &f,\n"
         "    const size_t grp, const size_t pos, const size_t cs, const double H[3][3], double W[3][3], const int padd) {\n";
  emit_inputs(t, en, 2, "__ldcs",
              "#pragma unroll\n  for (int d = 0; d < 3; d++)\n#pragma unroll\n"
              "    for (int c = 0; c < 3; c++) in%d[d * 3 + c] = H[c][d];\n");
  emit_call(t, en, name, 2);
  for (int i = 0; i < en.nout; i++) {
    if (i == en.ao)
      t.add("#pragma unroll\n  for (int kk = 0; kk < 3; kk++)\n#pragma unroll\n"
            "    for (int c = 0; c < 3; c++) W[c][kk] = out%d[kk * 3 + c];\n", i);
    else
      t.add("  { double *p = f.out[%d] + grp * %d + pos;\n"
            "    if (padd) {\n#pragma unroll\n      for (int c = 0; c < %d; c++) p[c * cs] += out%d[c];\n"
            "    } else {\n#pragma unroll\n      for (int c = 0; c < %d; c++) __stcs(p + c * cs, out%d[c]);\n    } }\n",
            i, en.out_size[i], en.out_size[i], i, en.out_size[i], i);
  }
  t.s += "}\n";
  emit_kernels(t, en, name, ctas,
               "const int *__restrict__ offsets,\n"
               "    const double *__restrict__ x, double *__restrict__ y, double *__restrict__ evec, const int padd",
               "offsets, x, y, evec, padd");
  return t.s;
}

// K13: the prefix b200_jit_assemble.cuh expects (constants, parameter structs, the point-tangent adapter: the 9
// unit-input calls), the template, the kernels
std::string generated_assemble(const char *name, const Entry &en, int CH, int ctas, int unroll) {
  Text t;
  t.s += "\n#line 1 \"b200_jit_assemble_prefix\"\n";
  t.add("#define B200_K13_Q %d\n#define B200_K13_EB %d\n#define B200_K13_NT %d\n#define B200_K13_CH %d\n", en.Q, en.EB,
        en.NT, CH);
  emit_structs(t, en);
  t.s += "__device__ __forceinline__ void b200_k13_point(const b200_jit_ctx_t &ctx, const b200_k13_fields_t &f,\n"
         "    const size_t grp, const size_t pos, const size_t cs, double *__restrict__ d) {\n";
  emit_inputs(t, en, 2, "__ldcs", "");
  t.s += unroll ? "#pragma unroll\n" : "#pragma unroll 1\n";
  t.s += "  for (int s = 0; s < 9; s++) {\n";
  t.add("#pragma unroll\n    for (int c = 0; c < 9; c++) in%d[c] = c == s ? 1.0 : 0.0;\n", en.ai);
  emit_call(t, en, name, 4);
  t.add("#pragma unroll\n    for (int o = 0; o < 9; o++) d[s * 9 + o] = out%d[o];\n", en.ao);
  t.s += "  }\n}\n";
  // 384 threads (Q <= 3, EB = 16) leave at most 168 registers a thread whatever is asked: one block per SM
  emit_kernels(t, en, name, en.NT > 128 ? 1 : ctas, "double *__restrict__ values", "values");
  return t.s;
}

// K14: the prefix b200_jit_diag.cuh expects (constants, parameter structs, the slab prefetch, the adapter that gives
// one component's point tangent from 3 unit-input calls), the template, the kernels
std::string generated_diag(const char *name, const Entry &en, const int *lay, int ctas) {
  Text t;
  t.s += "\n#line 1 \"b200_jit_diag_prefix\"\n";
  emit_lattice(t, "K14", en, lay);
  emit_structs(t, en);
  // the bulk prefetch wants a 16-byte aligned range: the slab's 16-byte granules that lie inside it
  t.s += "__device__ __forceinline__ void b200_k14_l2(const double *p, const size_t n) {\n"
         "  const unsigned long long a0 = ((unsigned long long)p + 15) & ~15ull, a1 = (unsigned long long)(p + n) & ~15ull;\n"
         "  if (a1 > a0) asm volatile(\"cp.async.bulk.prefetch.L2.global [%0], %1;\" ::\"l\"(a0), \"r\"((unsigned)(a1 - a0)) : \"memory\");\n"
         "}\n";
  t.s += "__device__ __forceinline__ void b200_k14_prefetch(const b200_k14_fields_t &f, const size_t grp, const size_t npts) {\n";
  for (int i = 0; i < en.nin; i++)
    if (i != en.ai) t.add("  b200_k14_l2(f.in[%d] + grp * %d, npts * %d);\n", i, en.in_size[i], en.in_size[i]);
  t.s += "}\n";
  t.s += "template <class Fold>\n"
         "__device__ __forceinline__ void b200_k14_point(const b200_jit_ctx_t &ctx, const b200_k14_fields_t &f,\n"
         "    const size_t grp, const size_t pos, const size_t cs, const int comp, Fold &&fold) {\n";
  t.s += "#pragma unroll 1\n  for (int m = 0; m < 3; m++) {\n";
  emit_inputs(t, en, 4, "__ldg", "");
  t.add("#pragma unroll\n    for (int c = 0; c < 9; c++) in%d[c] = c == m * 3 + comp ? 1.0 : 0.0;\n", en.ai);
  emit_call(t, en, name, 4);
  // selects, not run-time indices: the outputs stay in registers
  t.add("    double v[3];\n#pragma unroll\n    for (int kk = 0; kk < 3; kk++)\n"
        "      v[kk] = comp == 0 ? out%d[kk * 3] : comp == 1 ? out%d[kk * 3 + 1] : out%d[kk * 3 + 2];\n"
        "    fold(m, v);\n", en.ao, en.ao, en.ao);
  t.s += "  }\n}\n";
  // ctas blocks of 128 threads' worth per SM: 160-thread CTAs (Q = 3) ask for fewer blocks, as K3 does, so that a
  // thread keeps the registers the user function needs
  const int full = en.NT > 128 && ctas * 128 / en.NT >= 1 ? ctas * 128 / en.NT : ctas;
  emit_kernels(t, en, name, full, "const int *__restrict__ offsets,\n    double *__restrict__ diag, double *__restrict__ evec",
               "offsets, diag, evec");
  return t.s;
}

// ---- compile -----------------------------------------------------------------------------------------------------

int compile_locked(Entry &en, const char *src_name) {
  if (int rc = open_nvrtc()) return rc;
  const std::string &text = en.key;
  const size_t skip = text.find('\n') + 1;  // the key's first line holds the options
  nvrtcProgram prog;
  const char *hdr[] = {kCeedHeader, kCeedHeader, kMathHeader};
  const char *hdr_names[] = {"ceed.h", "ceed/ceed.h", "math.h"};
  nvrtcResult r = g_nv.create(&prog, text.c_str() + skip, src_name, 3, hdr, hdr_names);
  if (r != NVRTC_SUCCESS) return error("b200_jit", "nvrtcCreateProgram: %s", g_nv.errstr(r));
  r = g_nv.compile(prog, kNumOptions, kOptions);
  g_compiles++;
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    g_nv.log_size(prog, &n);
    std::string log(n ? n : 1, '\0');
    if (n) g_nv.log(prog, &log[0]);
    log.resize(strlen(log.c_str()));
    if (log.size() > kMaxLog) log = log.substr(0, kMaxLog) + "\n[... NVRTC log truncated]";
    std::string msg = std::string("NVRTC could not compile the QFunction (") + g_nv.errstr(r) + "):\n" + log;
    g_nv.destroy(&prog);
    return b200::set_error_msg(msg.c_str());
  }
  size_t n = 0;
  g_nv.cubin_size(prog, &n);
  en.cubin.resize(n);
  if (n) g_nv.cubin(prog, en.cubin.data());
  g_nv.destroy(&prog);
  if (!n) return b200::set_error_msg("b200_jit: NVRTC produced no cubin");
  return 0;
}

// the entry of en's program; compiles unless the same program was compiled before in this process
int find_or_compile(Entry &&en, const char *src_name, int *handle) {
  std::lock_guard<std::mutex> lock(g_mu);
  for (size_t i = 0; i < g_entries.size(); i++)
    if (g_entries[i]->key == en.key) {
      *handle = (int)i;
      return 0;
    }
  if (int rc = compile_locked(en, src_name && src_name[0] ? src_name : "qfunction")) return rc;
  g_entries.push_back(new Entry(std::move(en)));
  *handle = (int)g_entries.size() - 1;
  return 0;
}

int check_fields(const char *fn, const char *name, int nin, const int *in_sizes, int nout, const int *out_sizes) {
  if (!is_identifier(name)) return error(fn, "QFunction name \"%.128s\" is not a C identifier", name);
  if (nin < 0 || nout < 1 || nin > B200_JIT_MAXF || nout > B200_JIT_MAXF)
    return error(fn, "need 0..8 input and 1..8 output fields");
  for (int i = 0; i < nin + nout; i++) {
    const int s = i < nin ? in_sizes[i] : out_sizes[i - nin];
    if (s < 1 || s > B200_JIT_MAX_FIELD)
      return error(fn, "%s field %d of QFunction %.128s has %d components; a JIT QFunction field holds 1 to %d",
                   i < nin ? "input" : "output", i < nin ? i : i - nin, name, s, B200_JIT_MAX_FIELD);
  }
  return 0;
}

std::string options_line() {
  std::string key;
  for (int i = 0; i < kNumOptions; i++) key += std::string(kOptions[i]) + " ";
  return key + "\n";
}

// a tuning override, read at every compile because it is part of the program text and so of its key: the variable's
// value if it is set and at least lo, else dflt
int env_int(const char *name, int dflt, int lo) {
  const char *s = getenv(name);
  return s && s[0] && atoi(s) >= lo ? atoi(s) : dflt;
}

// every compile: the checks, the entry, then per kind its (P, Q) check, tuning, program and shared memory
int compile(Kind kind, const char *fn, const char *text, const char *src_name, const char *name, int nin,
            const int *in_sizes, int nout, const int *out_sizes, int ai, int ao, int P, int Q, int *handle) {
  *handle = -1;
  if (!text || !name) return error(fn, "NULL program text or name");
  if (int rc = check_fields(fn, name, nin, in_sizes, nout, out_sizes)) return rc;
  if (kind != kPoint && (ai < 0 || ai >= nin || ao < 0 || ao >= nout || in_sizes[ai] != 9 || out_sizes[ao] != 9))
    return error(fn, "the active input and output must be fields of 9 components");
  Entry en;
  en.kind = kind;
  en.nin = nin;
  en.nout = nout;
  for (int i = 0; i < nin; i++) en.in_size[i] = in_sizes[i];
  for (int i = 0; i < nout; i++) en.out_size[i] = out_sizes[i];
  en.ai = ai;
  en.ao = ao;
  en.P = P;
  en.Q = Q;
  int lay[6];
  std::string gen;
  switch (kind) {
    case kPoint:
      gen = generated_kernel(name, en);
      break;
    case kFused:
      if (b200_apply_smem_layout(P, Q, lay)) return error(fn, "(P, Q) = (%d, %d) has no fused lattice layout", P, Q);
      en.EB = lay[4];
      en.NT = lay[5];
      // no (P, Q) of the table needs more than 48 KB today
      en.smem = sizeof(double) * (size_t)en.EB * lay[3] + sizeof(int) * (size_t)en.EB * P * P * P;
      gen = generated_fused(name, en, lay, env_int("B200_JIT_FUSED_CTAS", kFusedCtas, 1));
      break;
    case kAssemble: {
      if (P != 2) return error(fn, "element matrices are assembled on trilinear (P = 2) levels only, not P = %d", P);
      if (!b200_fused_supported(P, Q)) return error(fn, "(P, Q) = (%d, %d) is not instantiated", P, Q);
      en.EB = b200::elems_per_block(Q);
      en.NT = 24 * en.EB;
      const int CH = en.NT < kAssembleMaxChunk ? en.NT : kAssembleMaxChunk;
      en.smem = sizeof(double) * 81 * (size_t)CH;  // the point tangents of a chunk: 62 to 83 KB
      gen = generated_assemble(name, en, CH, env_int("B200_JIT_ASSEMBLE_CTAS", kAssembleCtas, 1),
                               env_int("B200_JIT_ASSEMBLE_UNROLL", kAssembleUnroll, INT_MIN) != 0);
      break;
    }
    case kDiag:
      if (!b200_fused_supported(P, Q) || b200_apply_smem_layout(P, Q, lay))
        return error(fn, "(P, Q) = (%d, %d) is not instantiated", P, Q);
      en.EB = lay[4];
      en.NT = lay[5];
      en.smem = sizeof(double) * (size_t)en.EB * lay[3];  // nine lattices per element: 70 KB at Q = 4 (EB = 8)
      gen = generated_diag(name, en, lay, env_int("B200_JIT_DIAG_CTAS", kDiagCtas, 1));
      break;
  }
  en.key = options_line() + text + gen;
  if (kind == kPoint) {
    en.kernel = std::string("b200_jit_") + name;
  } else {
    en.kernel = std::string("b200_jit_") + kKinds[kind].name + "_" + name;
    en.kernel_tail = std::string("b200_jit_") + kKinds[kind].name + "_tail_" + name;
  }
  return find_or_compile(std::move(en), src_name, handle);
}

// ---- apply -------------------------------------------------------------------------------------------------------

// what an apply launches with: the entry, the context and the field pointers (the active ones blank)
struct Call {
  Entry *en;
  JitCtx ctx;
  JitFields f;
};

// every apply, before it launches: the handle's entry, which must be of `kind`, its kernels loaded at first use and its
// dynamic shared-memory limit raised once per device; the field counts (K13 and K14 take no outputs: nout = -1) and
// the context checked
int prologue(Call &c, Kind kind, const char *fn, int handle, const void *h_ctx, size_t ctx_bytes, int nin,
             const double *const *d_in, int nout, double *const *d_out) {
  Entry *en;
  {
    std::lock_guard<std::mutex> lock(g_mu);
    if (handle < 0 || handle >= (int)g_entries.size() || (kind != kPoint && g_entries[handle]->kind != kind))
      return error(fn, "bad handle");
    en = c.en = g_entries[handle];
    if (en->kind != kind) return error(fn, "the handle names a fused operator, assembly or diagonal program");
    if (!en->lib) {
      B200_CHECK(cudaLibraryLoadData(&en->lib, en->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
      B200_CHECK(cudaLibraryGetKernel(&en->fn, en->lib, en->kernel.c_str()));
      if (kind != kPoint) B200_CHECK(cudaLibraryGetKernel(&en->fn_tail, en->lib, en->kernel_tail.c_str()));
    }
    if (en->smem > 48 * 1024) {
      int dev;
      B200_CHECK(cudaGetDevice(&dev));
      if (dev >= 0 && dev < 64 && !(en->smem_set >> dev & 1)) {
        B200_CHECK(cudaKernelSetAttributeForDevice(en->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
        B200_CHECK(cudaKernelSetAttributeForDevice(en->fn_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
        en->smem_set |= 1ull << dev;
      }
    }
  }
  if (nin != en->nin || (nout >= 0 && nout != en->nout)) return error(fn, "field count differs from the compiled one");
  if (ctx_bytes > B200_JIT_MAX_CTX)
    return error(fn, "context of %zu bytes; a JIT QFunction takes at most %d", ctx_bytes, B200_JIT_MAX_CTX);
  if (ctx_bytes && !h_ctx) return error(fn, "NULL context");
  memset(&c.ctx, 0, sizeof c.ctx);
  if (ctx_bytes) memcpy(c.ctx.b, h_ctx, ctx_bytes);
  memset(&c.f, 0, sizeof c.f);
  for (int i = 0; i < nin; i++) c.f.in[i] = i == en->ai ? nullptr : d_in[i];
  for (int i = 0; i < nout; i++) c.f.out[i] = i == en->ao ? nullptr : d_out[i];
  return 0;
}

// K12 to K14 on elements [0, nelem): the full element groups in one launch, the partial group at the end in one CTA of
// the tail kernel, which takes the group extent at run time.  The kernel parameters are (mats, ctx, fields, nelem,
// rest...): the field pointers are shifted here to the launch's first element e0, and rest(e0, a) points a[0], a[1],
// ... at the remaining parameters for a range that starts at e0.
template <class Rest>
int launch_groups(const char *fn, Call &c, void *mats, int nelem, Rest &&rest) {
  const Entry &en = *c.en;
  const int nfull = nelem / en.EB, ntail = nelem - nfull * en.EB;
  const size_t Q3 = (size_t)en.Q * en.Q * en.Q;
  for (int tail = 0; tail < 2; tail++) {
    int n = tail ? ntail : nfull * en.EB;
    if (!n) continue;
    const size_t e0 = tail ? (size_t)nfull * en.EB : 0;
    JitFields f = c.f;
    for (int i = 0; i < en.nin; i++)
      if (f.in[i]) f.in[i] += e0 * en.in_size[i] * Q3;
    for (int i = 0; i < en.nout; i++)
      if (f.out[i]) f.out[i] += e0 * en.out_size[i] * Q3;
    void *args[9] = {mats, &c.ctx, &f, &n};
    rest(e0, args + 4);
    B200_CHECK(cudaLaunchKernel((const void *)(tail ? en.fn_tail : en.fn), dim3(tail ? 1 : nfull), dim3(en.NT), args,
                                en.smem, b200::g_stream));
    char what[64];
    snprintf(what, sizeof what, tail ? "%s(tail)" : "%s", fn);
    B200_LAUNCH_CHECK(what);
  }
  return 0;
}

}  // namespace

extern "C" int b200_jit_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                                int nout, const int *out_sizes, int *handle) {
  return compile(kPoint, "b200_jit_compile", text, src_name, name, nin, in_sizes, nout, out_sizes, -1, -1, 0, 0, handle);
}

extern "C" int b200_jit_fused_compile(const char *text, const char *src_name, const char *name, int nin,
                                      const int *in_sizes, int nout, const int *out_sizes, int active_in,
                                      int active_out, int P, int Q, int *handle) {
  return compile(kFused, "b200_jit_fused_compile", text, src_name, name, nin, in_sizes, nout, out_sizes, active_in,
                 active_out, P, Q, handle);
}

extern "C" int b200_jit_assemble_compile(const char *text, const char *src_name, const char *name, int nin,
                                         const int *in_sizes, int nout, const int *out_sizes, int active_in,
                                         int active_out, int P, int Q, int *handle) {
  return compile(kAssemble, "b200_jit_assemble_compile", text, src_name, name, nin, in_sizes, nout, out_sizes,
                 active_in, active_out, P, Q, handle);
}

extern "C" int b200_jit_diag_compile(const char *text, const char *src_name, const char *name, int nin,
                                     const int *in_sizes, int nout, const int *out_sizes, int active_in, int active_out,
                                     int P, int Q, int *handle) {
  return compile(kDiag, "b200_jit_diag_compile", text, src_name, name, nin, in_sizes, nout, out_sizes, active_in,
                 active_out, P, Q, handle);
}

extern "C" unsigned long long b200_jit_compile_count(void) {
  std::lock_guard<std::mutex> lock(g_mu);
  return g_compiles;
}

extern "C" const char *b200_jit_program(int handle) {
  std::lock_guard<std::mutex> lock(g_mu);
  if (handle < 0 || handle >= (int)g_entries.size()) return nullptr;
  const std::string &k = g_entries[handle]->key;
  return k.c_str() + k.find('\n') + 1;
}

extern "C" int b200_jit_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, int nq, int nin,
                              const double *const *d_in, int nout, double *const *d_out) {
  Call c;
  if (int rc = prologue(c, kPoint, "b200_jit_apply", handle, h_ctx, ctx_bytes, nin, d_in, nout, d_out)) return rc;
  const size_t total = (size_t)nelem * nq;
  if (!total) return 0;
  const int nt = 128;
  const size_t nb = (total + nt - 1) / nt, cap = 148 * 32;
  void *args[] = {&c.ctx, &c.f, &nelem, &nq};
  B200_CHECK(cudaLaunchKernel((const void *)c.en->fn, dim3((unsigned)(nb < cap ? nb : cap)), dim3(nt), args, 0,
                              b200::g_stream));
  B200_LAUNCH_CHECK("b200_jit_apply");
  return 0;
}

extern "C" int b200_jit_fused_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                                    const double *h_grad1d, const int *d_offsets, const double *d_x, double *d_y,
                                    double *d_evec, int nin, const double *const *d_in, int nout, double *const *d_out,
                                    int passive_add) {
  Call c;
  if (int rc = prologue(c, kFused, "b200_jit_fused_apply", handle, h_ctx, ctx_bytes, nin, d_in, nout, d_out)) return rc;
  if (nelem <= 0) return 0;
  const int P = c.en->P, Q = c.en->Q, P3 = P * P * P;
  // B and Gc as the kernel parameter b200_k12_mats_t (sized for this (P, Q))
  double mats[8 * 8 + 8 * 8];
  for (int i = 0; i < Q * P; i++) mats[i] = h_interp1d[i];
  if (b200::collocated_grad_1d(P, Q, h_interp1d, h_grad1d, mats + Q * P))
    return b200::set_error_msg("basis: no collocated gradient with Gc*B = D (rank-deficient interp1d)");
  const int *off;
  double *ev;
  return launch_groups("b200_jit_fused_apply", c, mats, nelem, [&](size_t e0, void **a) {
    off = d_offsets + e0 * P3;
    ev = d_evec ? d_evec + e0 * 3 * P3 : nullptr;
    a[0] = &off, a[1] = &d_x, a[2] = &d_y, a[3] = &ev, a[4] = &passive_add;
  });
}

extern "C" int b200_jit_assemble_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem,
                                       const double *h_interp1d, const double *h_grad1d, int nin,
                                       const double *const *d_in, double *d_values) {
  Call c;
  if (int rc = prologue(c, kAssemble, "b200_jit_assemble_apply", handle, h_ctx, ctx_bytes, nin, d_in, -1, nullptr))
    return rc;
  if (nelem <= 0) return 0;
  const int Q = c.en->Q;
  double mats[2 * 8 * 2];  // b200_k13_mats_t for this Q: interp1d [Q][2], then grad1d [Q][2]
  for (int i = 0; i < Q * 2; i++) {
    mats[i] = h_interp1d[i];
    mats[Q * 2 + i] = h_grad1d[i];
  }
  double *v;
  return launch_groups("b200_jit_assemble_apply", c, mats, nelem, [&](size_t e0, void **a) {
    v = d_values + e0 * 576;
    a[0] = &v;
  });
}

extern "C" int b200_jit_diag_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                                   const double *h_grad1d, const int *d_offsets, int nin, const double *const *d_in,
                                   double *d_diag, double *d_evec) {
  Call c;
  if (int rc = prologue(c, kDiag, "b200_jit_diag_apply", handle, h_ctx, ctx_bytes, nin, d_in, -1, nullptr)) return rc;
  if (nelem <= 0) return 0;
  const int P = c.en->P, Q = c.en->Q, P3 = P * P * P;
  double mats[3 * 8 * 8];  // b200_k14_mats_t for this (P, Q): B.B, B.D, D.D element-wise, each [Q][P]
  for (int i = 0; i < Q * P; i++) {
    mats[i] = h_interp1d[i] * h_interp1d[i];
    mats[Q * P + i] = h_interp1d[i] * h_grad1d[i];
    mats[2 * Q * P + i] = h_grad1d[i] * h_grad1d[i];
  }
  const int *off;
  double *ev;
  return launch_groups("b200_jit_diag_apply", c, mats, nelem, [&](size_t e0, void **a) {
    off = d_offsets + e0 * P3;
    ev = d_evec ? d_evec + e0 * 3 * P3 : nullptr;
    a[0] = &off, a[1] = &d_diag, a[2] = &ev;
  });
}
