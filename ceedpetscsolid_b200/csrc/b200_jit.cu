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
#include <dlfcn.h>
#include <nvrtc.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
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

// the K12 template (b200_jit_fused.cuh) as a string
const char *const kFusedTemplate =
#include "b200_jit_fused.inc"
    ;

// K12 blocks per SM asked of ptxas for the full-group kernel (__launch_bounds__ min blocks): 128 threads x 3 blocks
// leave 168 registers a thread.  Measured at P = Q = 5, C3 (profiles/jit_fused_ctas_ab.txt): the fastest setting at
// which port_HyperFSdF neither spills nor has a stack frame; 4 blocks (128 registers) ran 7 % faster with 112 bytes of
// spills.  B200_JIT_FUSED_CTAS overrides it (tuning runs).
const int kFusedCtas = 3;

// the K13 template (b200_jit_assemble.cuh) as a string
const char *const kAssembleTemplate =
#include "b200_jit_assemble.inc"
    ;

// K13 blocks per SM asked of ptxas for the full-group kernel, and whether the 9 unit-input calls of the user function
// are unrolled (NVCC may then share their input-independent part) or kept rolled.  Chosen by measurement at Q = 5,
// C3 (profiles/jit_assemble_ab.txt); B200_JIT_ASSEMBLE_CTAS and B200_JIT_ASSEMBLE_UNROLL override them (tuning runs).
const int kAssembleCtas = 2;
const int kAssembleUnroll = 0;
// most point tangents a K13 CTA holds in shared memory at once (81 doubles each)
const int kAssembleMaxChunk = 128;

struct Entry {
  std::string key;     // options + program text
  std::string kernel;  // b200_jit_<Name>, or b200_jit_fused_<Name> (K12: full element groups)
  std::vector<char> cubin;
  int nin = 0, nout = 0, in_size[B200_JIT_MAXF] = {}, out_size[B200_JIT_MAXF] = {};
  cudaLibrary_t lib = nullptr;
  cudaKernel_t fn = nullptr;
  // K12 only
  bool fused = false;
  int P = 0, Q = 0, ai = -1, ao = -1, lay[6] = {};  // lay: b200_apply_smem_layout {SY, SZ, SC, SE, EB, NT}
  size_t smem = 0;
  std::string kernel_tail;  // b200_jit_fused_tail_<Name>: the partial group at the end of a range
  cudaKernel_t fn_tail = nullptr;
  unsigned long long smem_set = 0;  // devices on which the dynamic shared-memory limit was raised
  // K13 only (P, Q, ai, ao, smem, kernel_tail and fn_tail as for K12; lay[4] = EB, lay[5] = threads)
  bool assemble = false;
};

std::mutex g_mu;
Nvrtc g_nv;
std::vector<Entry *> g_entries;
unsigned long long g_compiles = 0;

// the kernel parameters, laid out as the generated kernel declares them
struct alignas(16) JitCtx { unsigned char b[B200_JIT_MAX_CTX]; };
struct JitFields { const double *in[B200_JIT_MAXF]; double *out[B200_JIT_MAXF]; };

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

std::string generated_kernel(const char *name, int nin, const int *in_size, int nout, const int *out_size) {
  std::string k;
  char line[512];
  auto add = [&](const char *fmt, auto... a) {
    snprintf(line, sizeof line, fmt, a...);
    k += line;
  };
  k += "\n#line 1 \"b200_jit_kernel\"\n";
  add("struct alignas(16) b200_jit_ctx_t { unsigned char b[%d]; };\n", B200_JIT_MAX_CTX);
  add("struct b200_jit_fields_t { const double *in[%d]; double *out[%d]; };\n", B200_JIT_MAXF, B200_JIT_MAXF);
  add("extern \"C\" __global__ void __launch_bounds__(128) b200_jit_%s(const __grid_constant__ b200_jit_ctx_t ctx,\n"
      "    const __grid_constant__ b200_jit_fields_t f, const int nelem, const int nq) {\n", name);
  k += "  const long long total = (long long)nelem * nq;\n"
       "  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total;\n"
       "       t += (long long)gridDim.x * blockDim.x) {\n"
       "    const long long e = t / nq, q = t - e * nq;\n";
  for (int i = 0; i < nin; i++)
    add("    double in%d[%d];\n"
        "    { const double *p = f.in[%d] + e * %dLL * nq + q;\n"
        "#pragma unroll\n"
        "      for (int c = 0; c < %d; c++) in%d[c] = p[(long long)c * nq]; }\n",
        i, in_size[i], i, in_size[i], in_size[i], i);
  for (int i = 0; i < nout; i++) add("    double out%d[%d] = {};\n", i, out_size[i]);
  k += "    const double *ins[] = {";
  for (int i = 0; i < nin; i++) add("%sin%d", i ? ", " : "", i);
  k += "};\n    double *outs[] = {";
  for (int i = 0; i < nout; i++) add("%sout%d", i ? ", " : "", i);
  k += "};\n";
  add("    (void)%s((void *)ctx.b, 1, ins, outs);\n", name);
  for (int i = 0; i < nout; i++)
    add("    { double *p = f.out[%d] + e * %dLL * nq + q;\n"
        "#pragma unroll\n"
        "      for (int c = 0; c < %d; c++) p[(long long)c * nq] = out%d[c]; }\n",
        i, out_size[i], out_size[i], i);
  k += "  }\n}\n";
  return k;
}

int compile_locked(Entry &en, const char *src_name) {
  if (int rc = open_nvrtc()) return rc;
  const std::string &text = en.key;
  const size_t skip = text.find('\n') + 1;  // the key's first line holds the options
  nvrtcProgram prog;
  const char *hdr[] = {kCeedHeader, kCeedHeader, kMathHeader};
  const char *hdr_names[] = {"ceed.h", "ceed/ceed.h", "math.h"};
  nvrtcResult r = g_nv.create(&prog, text.c_str() + skip, src_name, 3, hdr, hdr_names);
  if (r != NVRTC_SUCCESS) {
    char msg[256];
    snprintf(msg, sizeof msg, "b200_jit: nvrtcCreateProgram: %s", g_nv.errstr(r));
    return b200::set_error_msg(msg);
  }
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

// text + generated kernel(s) -> entry; compiles unless the same program was compiled before in this process
int find_or_compile(Entry *proto, const char *src_name, int *handle) {
  std::lock_guard<std::mutex> lock(g_mu);
  for (size_t i = 0; i < g_entries.size(); i++)
    if (g_entries[i]->key == proto->key) {
      *handle = (int)i;
      delete proto;
      return 0;
    }
  if (int rc = compile_locked(*proto, src_name && src_name[0] ? src_name : "qfunction")) {
    delete proto;
    return rc;
  }
  g_entries.push_back(proto);
  *handle = (int)g_entries.size() - 1;
  return 0;
}

int check_fields(const char *fn, const char *name, int nin, const int *in_sizes, int nout, const int *out_sizes) {
  char msg[256];
  if (!is_identifier(name)) {
    snprintf(msg, sizeof msg, "%s: QFunction name \"%.128s\" is not a C identifier", fn, name);
    return b200::set_error_msg(msg);
  }
  if (nin < 0 || nout < 1 || nin > B200_JIT_MAXF || nout > B200_JIT_MAXF) {
    snprintf(msg, sizeof msg, "%s: need 0..8 input and 1..8 output fields", fn);
    return b200::set_error_msg(msg);
  }
  for (int i = 0; i < nin + nout; i++) {
    const int s = i < nin ? in_sizes[i] : out_sizes[i - nin];
    if (s < 1 || s > B200_JIT_MAX_FIELD) {
      snprintf(msg, sizeof msg, "%s: %s field %d of QFunction %.128s has %d components; a JIT QFunction "
               "field holds 1 to %d", fn, i < nin ? "input" : "output", i < nin ? i : i - nin, name, s, B200_JIT_MAX_FIELD);
      return b200::set_error_msg(msg);
    }
  }
  return 0;
}

std::string options_line() {
  std::string key;
  for (int i = 0; i < kNumOptions; i++) key += std::string(kOptions[i]) + " ";
  return key + "\n";
}

// K12: the prefix the template expects (constants, parameter structs, the point adapter), the template, the kernels
std::string generated_fused(const char *name, int nin, const int *in_size, int nout, const int *out_size, int ai, int ao,
                            int P, int Q, const int *lay, int ctas) {
  std::string k;
  char line[512];
  auto add = [&](const char *fmt, auto... a) {
    snprintf(line, sizeof line, fmt, a...);
    k += line;
  };
  k += "\n#line 1 \"b200_jit_fused_prefix\"\n";
  add("#define B200_K12_P %d\n#define B200_K12_Q %d\n", P, Q);
  add("#define B200_K12_SY %d\n#define B200_K12_SZ %d\n#define B200_K12_SC %d\n#define B200_K12_SE %d\n"
      "#define B200_K12_EB %d\n#define B200_K12_NT %d\n", lay[0], lay[1], lay[2], lay[3], lay[4], lay[5]);
  add("struct alignas(16) b200_jit_ctx_t { unsigned char b[%d]; };\n", B200_JIT_MAX_CTX);
  add("struct b200_k12_fields_t { const double *in[%d]; double *out[%d]; };\n", B200_JIT_MAXF, B200_JIT_MAXF);
  k += "__device__ __forceinline__ void b200_k12_point(const b200_jit_ctx_t &ctx, const b200_k12_fields_t &f,\n"
       "    const size_t grp, const size_t pos, const size_t cs, const double H[3][3], double W[3][3], const int padd) {\n";
  for (int i = 0; i < nin; i++) {
    add("  double in%d[%d];\n", i, in_size[i]);
    if (i == ai)
      add("#pragma unroll\n  for (int d = 0; d < 3; d++)\n#pragma unroll\n"
          "    for (int c = 0; c < 3; c++) in%d[d * 3 + c] = H[c][d];\n", i);
    else
      add("  { const double *p = f.in[%d] + grp * %d + pos;\n#pragma unroll\n"
          "    for (int c = 0; c < %d; c++) in%d[c] = __ldcs(p + c * cs); }\n", i, in_size[i], in_size[i], i);
  }
  for (int i = 0; i < nout; i++) add("  double out%d[%d] = {};\n", i, out_size[i]);
  k += "  const double *ins[] = {";
  for (int i = 0; i < nin; i++) add("%sin%d", i ? ", " : "", i);
  k += "};\n  double *outs[] = {";
  for (int i = 0; i < nout; i++) add("%sout%d", i ? ", " : "", i);
  k += "};\n";
  add("  (void)%s((void *)ctx.b, 1, ins, outs);\n", name);
  for (int i = 0; i < nout; i++) {
    if (i == ao)
      add("#pragma unroll\n  for (int kk = 0; kk < 3; kk++)\n#pragma unroll\n"
          "    for (int c = 0; c < 3; c++) W[c][kk] = out%d[kk * 3 + c];\n", i);
    else
      add("  { double *p = f.out[%d] + grp * %d + pos;\n"
          "    if (padd) {\n#pragma unroll\n      for (int c = 0; c < %d; c++) p[c * cs] += out%d[c];\n"
          "    } else {\n#pragma unroll\n      for (int c = 0; c < %d; c++) __stcs(p + c * cs, out%d[c]);\n    } }\n",
          i, out_size[i], out_size[i], i, out_size[i], i);
  }
  k += "}\n#line 1 \"b200_jit_fused.cuh\"\n";
  k += kFusedTemplate;
  k += "\n#line 1 \"b200_jit_fused_kernels\"\n";
  // the tail kernel runs as one CTA: occupancy is moot, so it gets every register it wants
  const char *variant[2] = {"", "tail_"};
  for (int v = 0; v < 2; v++)
    add("extern \"C\" __global__ void __launch_bounds__(%d, %d) b200_jit_fused_%s%s(\n"
        "    const __grid_constant__ b200_k12_mats_t m, const __grid_constant__ b200_jit_ctx_t ctx,\n"
        "    const __grid_constant__ b200_k12_fields_t f, const int nelem, const int *__restrict__ offsets,\n"
        "    const double *__restrict__ x, double *__restrict__ y, double *__restrict__ evec, const int padd) {\n"
        "  b200_k12_body<%s>(m, ctx, f, nelem, offsets, x, y, evec, padd);\n}\n",
        lay[5], v ? 1 : ctas, variant[v], name, v ? "false" : "true");
  return k;
}

// K13: the prefix b200_jit_assemble.cuh expects (constants, parameter structs, the point-tangent adapter), the template,
// the kernels
std::string generated_assemble(const char *name, int nin, const int *in_size, int nout, const int *out_size, int ai,
                               int ao, int Q, int EB, int NT, int CH, int ctas, int unroll) {
  std::string k;
  char line[512];
  auto add = [&](const char *fmt, auto... a) {
    snprintf(line, sizeof line, fmt, a...);
    k += line;
  };
  k += "\n#line 1 \"b200_jit_assemble_prefix\"\n";
  add("#define B200_K13_Q %d\n#define B200_K13_EB %d\n#define B200_K13_NT %d\n#define B200_K13_CH %d\n", Q, EB, NT, CH);
  add("struct alignas(16) b200_jit_ctx_t { unsigned char b[%d]; };\n", B200_JIT_MAX_CTX);
  add("struct b200_k13_fields_t { const double *in[%d]; };\n", B200_JIT_MAXF);
  k += "__device__ __forceinline__ void b200_k13_point(const b200_jit_ctx_t &ctx, const b200_k13_fields_t &f,\n"
       "    const size_t grp, const size_t pos, const size_t cs, double *__restrict__ d) {\n";
  for (int i = 0; i < nin; i++) {
    add("  double in%d[%d];\n", i, in_size[i]);
    if (i != ai)
      add("  { const double *p = f.in[%d] + grp * %d + pos;\n#pragma unroll\n"
          "    for (int c = 0; c < %d; c++) in%d[c] = __ldcs(p + c * cs); }\n", i, in_size[i], in_size[i], i);
  }
  k += unroll ? "#pragma unroll\n" : "#pragma unroll 1\n";
  k += "  for (int s = 0; s < 9; s++) {\n";
  add("#pragma unroll\n    for (int c = 0; c < 9; c++) in%d[c] = c == s ? 1.0 : 0.0;\n", ai);
  for (int i = 0; i < nout; i++) add("    double out%d[%d] = {};\n", i, out_size[i]);
  k += "    const double *ins[] = {";
  for (int i = 0; i < nin; i++) add("%sin%d", i ? ", " : "", i);
  k += "};\n    double *outs[] = {";
  for (int i = 0; i < nout; i++) add("%sout%d", i ? ", " : "", i);
  k += "};\n";
  add("    (void)%s((void *)ctx.b, 1, ins, outs);\n", name);
  add("#pragma unroll\n    for (int o = 0; o < 9; o++) d[s * 9 + o] = out%d[o];\n", ao);
  k += "  }\n}\n#line 1 \"b200_jit_assemble.cuh\"\n";
  k += kAssembleTemplate;
  k += "\n#line 1 \"b200_jit_assemble_kernels\"\n";
  // 384 threads (Q <= 3, EB = 16) leave at most 168 registers a thread whatever is asked: one block per SM, and the
  // tail kernel runs as one CTA
  const char *variant[2] = {"", "tail_"};
  for (int v = 0; v < 2; v++)
    add("extern \"C\" __global__ void __launch_bounds__(%d, %d) b200_jit_assemble_%s%s(\n"
        "    const __grid_constant__ b200_k13_mats_t m, const __grid_constant__ b200_jit_ctx_t ctx,\n"
        "    const __grid_constant__ b200_k13_fields_t f, const int nelem, double *__restrict__ values) {\n"
        "  b200_k13_body<%s>(m, ctx, f, nelem, values);\n}\n",
        NT, v || NT > 128 ? 1 : ctas, variant[v], name, v ? "false" : "true");
  return k;
}

}  // namespace

extern "C" int b200_jit_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                                int nout, const int *out_sizes, int *handle) {
  *handle = -1;
  if (!text || !name) return b200::set_error_msg("b200_jit_compile: NULL program text or name");
  if (int rc = check_fields("b200_jit_compile", name, nin, in_sizes, nout, out_sizes)) return rc;
  Entry *en = new Entry;
  en->key = options_line() + text + generated_kernel(name, nin, in_sizes, nout, out_sizes);
  en->kernel = std::string("b200_jit_") + name;
  en->nin = nin;
  en->nout = nout;
  for (int i = 0; i < nin; i++) en->in_size[i] = in_sizes[i];
  for (int i = 0; i < nout; i++) en->out_size[i] = out_sizes[i];
  return find_or_compile(en, src_name, handle);
}

extern "C" int b200_jit_fused_compile(const char *text, const char *src_name, const char *name, int nin,
                                      const int *in_sizes, int nout, const int *out_sizes, int active_in,
                                      int active_out, int P, int Q, int *handle) {
  *handle = -1;
  if (!text || !name) return b200::set_error_msg("b200_jit_fused_compile: NULL program text or name");
  if (int rc = check_fields("b200_jit_fused_compile", name, nin, in_sizes, nout, out_sizes)) return rc;
  if (active_in < 0 || active_in >= nin || active_out < 0 || active_out >= nout || in_sizes[active_in] != 9 ||
      out_sizes[active_out] != 9)
    return b200::set_error_msg("b200_jit_fused_compile: the active input and output must be fields of 9 components");
  int lay[6];
  if (b200_apply_smem_layout(P, Q, lay)) {
    char msg[160];
    snprintf(msg, sizeof msg, "b200_jit_fused_compile: (P, Q) = (%d, %d) has no fused lattice layout", P, Q);
    return b200::set_error_msg(msg);
  }
  const char *env = getenv("B200_JIT_FUSED_CTAS");  // read at every compile: part of the program text and its key
  const int ctas = env && atoi(env) > 0 ? atoi(env) : kFusedCtas;
  Entry *en = new Entry;
  en->key = options_line() + text + generated_fused(name, nin, in_sizes, nout, out_sizes, active_in, active_out, P, Q, lay, ctas);
  en->kernel = std::string("b200_jit_fused_") + name;
  en->kernel_tail = std::string("b200_jit_fused_tail_") + name;
  en->nin = nin;
  en->nout = nout;
  for (int i = 0; i < nin; i++) en->in_size[i] = in_sizes[i];
  for (int i = 0; i < nout; i++) en->out_size[i] = out_sizes[i];
  en->fused = true;
  en->P = P;
  en->Q = Q;
  en->ai = active_in;
  en->ao = active_out;
  memcpy(en->lay, lay, sizeof lay);
  en->smem = sizeof(double) * (size_t)lay[4] * lay[3] + sizeof(int) * (size_t)lay[4] * P * P * P;
  return find_or_compile(en, src_name, handle);
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
  Entry *en;
  {
    std::lock_guard<std::mutex> lock(g_mu);
    if (handle < 0 || handle >= (int)g_entries.size()) return b200::set_error_msg("b200_jit_apply: bad handle");
    en = g_entries[handle];
    if (en->fused || en->assemble)
      return b200::set_error_msg("b200_jit_apply: the handle names a fused operator or assembly program");
    if (!en->lib) {
      B200_CHECK(cudaLibraryLoadData(&en->lib, en->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
      B200_CHECK(cudaLibraryGetKernel(&en->fn, en->lib, en->kernel.c_str()));
    }
  }
  if (nin != en->nin || nout != en->nout) return b200::set_error_msg("b200_jit_apply: field count differs from the compiled one");
  if (ctx_bytes > B200_JIT_MAX_CTX) {
    char msg[160];
    snprintf(msg, sizeof msg, "b200_jit_apply: context of %zu bytes; a JIT QFunction takes at most %d", ctx_bytes,
             B200_JIT_MAX_CTX);
    return b200::set_error_msg(msg);
  }
  if (ctx_bytes && !h_ctx) return b200::set_error_msg("b200_jit_apply: NULL context");
  JitCtx ctx;
  memset(&ctx, 0, sizeof ctx);
  if (ctx_bytes) memcpy(ctx.b, h_ctx, ctx_bytes);
  JitFields f;
  memset(&f, 0, sizeof f);
  for (int i = 0; i < nin; i++) f.in[i] = d_in[i];
  for (int i = 0; i < nout; i++) f.out[i] = d_out[i];
  const size_t total = (size_t)nelem * nq;
  if (!total) return 0;
  const int nt = 128;
  const size_t nb = (total + nt - 1) / nt, cap = 148 * 32;
  void *args[] = {&ctx, &f, &nelem, &nq};
  B200_CHECK(cudaLaunchKernel((const void *)en->fn, dim3((unsigned)(nb < cap ? nb : cap)), dim3(nt), args, 0,
                              b200::g_stream));
  B200_LAUNCH_CHECK("b200_jit_apply");
  return 0;
}

extern "C" int b200_jit_fused_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem, const double *h_interp1d,
                                    const double *h_grad1d, const int *d_offsets, const double *d_x, double *d_y,
                                    double *d_evec, int nin, const double *const *d_in, int nout, double *const *d_out,
                                    int passive_add) {
  Entry *en;
  int dev;
  B200_CHECK(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lock(g_mu);
    if (handle < 0 || handle >= (int)g_entries.size() || !g_entries[handle]->fused)
      return b200::set_error_msg("b200_jit_fused_apply: bad handle");
    en = g_entries[handle];
    if (!en->lib) {
      B200_CHECK(cudaLibraryLoadData(&en->lib, en->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
      B200_CHECK(cudaLibraryGetKernel(&en->fn, en->lib, en->kernel.c_str()));
      B200_CHECK(cudaLibraryGetKernel(&en->fn_tail, en->lib, en->kernel_tail.c_str()));
    }
    // no (P, Q) of the table needs more than 48 KB today; a larger layout raises the limit once per device
    if (en->smem > 48 * 1024 && dev >= 0 && dev < 64 && !(en->smem_set >> dev & 1)) {
      B200_CHECK(cudaKernelSetAttributeForDevice(en->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
      B200_CHECK(cudaKernelSetAttributeForDevice(en->fn_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
      en->smem_set |= 1ull << dev;
    }
  }
  if (nin != en->nin || nout != en->nout)
    return b200::set_error_msg("b200_jit_fused_apply: field count differs from the compiled one");
  if (ctx_bytes > B200_JIT_MAX_CTX) {
    char msg[160];
    snprintf(msg, sizeof msg, "b200_jit_fused_apply: context of %zu bytes; a JIT QFunction takes at most %d", ctx_bytes,
             B200_JIT_MAX_CTX);
    return b200::set_error_msg(msg);
  }
  if (ctx_bytes && !h_ctx) return b200::set_error_msg("b200_jit_fused_apply: NULL context");
  if (nelem <= 0) return 0;
  const int P = en->P, Q = en->Q, P3 = P * P * P, Q3 = Q * Q * Q, EB = en->lay[4], NT = en->lay[5];
  // B and Gc as the kernel parameter b200_k12_mats_t (sized for this (P, Q))
  double mats[8 * 8 + 8 * 8];
  for (int i = 0; i < Q * P; i++) mats[i] = h_interp1d[i];
  if (b200::collocated_grad_1d(P, Q, h_interp1d, h_grad1d, mats + Q * P))
    return b200::set_error_msg("basis: no collocated gradient with Gc*B = D (rank-deficient interp1d)");
  JitCtx ctx;
  memset(&ctx, 0, sizeof ctx);
  if (ctx_bytes) memcpy(ctx.b, h_ctx, ctx_bytes);
  JitFields f;
  memset(&f, 0, sizeof f);
  for (int i = 0; i < nin; i++) f.in[i] = i == en->ai ? nullptr : d_in[i];
  for (int i = 0; i < nout; i++) f.out[i] = i == en->ao ? nullptr : d_out[i];
  const int nfull = nelem / EB, ntail = nelem - nfull * EB;
  if (nfull) {
    int n = nfull * EB;
    void *args[] = {mats, &ctx, &f, &n, &d_offsets, &d_x, &d_y, &d_evec, &passive_add};
    B200_CHECK(cudaLaunchKernel((const void *)en->fn, dim3(nfull), dim3(NT), args, en->smem, b200::g_stream));
    B200_LAUNCH_CHECK("b200_jit_fused_apply");
  }
  if (ntail) {  // the partial group at the end: the same stages with a run-time group extent, one CTA
    const size_t e0 = (size_t)nfull * EB;
    JitFields ft = f;
    for (int i = 0; i < nin; i++)
      if (ft.in[i]) ft.in[i] += e0 * en->in_size[i] * Q3;
    for (int i = 0; i < nout; i++)
      if (ft.out[i]) ft.out[i] += e0 * en->out_size[i] * Q3;
    const int *off = d_offsets + e0 * P3;
    double *ev = d_evec ? d_evec + e0 * 3 * P3 : nullptr;
    int n = ntail;
    void *args[] = {mats, &ctx, &ft, &n, &off, &d_x, &d_y, &ev, &passive_add};
    B200_CHECK(cudaLaunchKernel((const void *)en->fn_tail, dim3(1), dim3(NT), args, en->smem, b200::g_stream));
    B200_LAUNCH_CHECK("b200_jit_fused_apply(tail)");
  }
  return 0;
}

extern "C" int b200_jit_assemble_compile(const char *text, const char *src_name, const char *name, int nin,
                                         const int *in_sizes, int nout, const int *out_sizes, int active_in,
                                         int active_out, int P, int Q, int *handle) {
  *handle = -1;
  if (!text || !name) return b200::set_error_msg("b200_jit_assemble_compile: NULL program text or name");
  if (int rc = check_fields("b200_jit_assemble_compile", name, nin, in_sizes, nout, out_sizes)) return rc;
  if (active_in < 0 || active_in >= nin || active_out < 0 || active_out >= nout || in_sizes[active_in] != 9 ||
      out_sizes[active_out] != 9)
    return b200::set_error_msg("b200_jit_assemble_compile: the active input and output must be fields of 9 components");
  char msg[160];
  if (P != 2) {
    snprintf(msg, sizeof msg, "b200_jit_assemble_compile: element matrices are assembled on trilinear (P = 2) levels "
             "only, not P = %d", P);
    return b200::set_error_msg(msg);
  }
  if (!b200_fused_supported(P, Q)) {
    snprintf(msg, sizeof msg, "b200_jit_assemble_compile: (P, Q) = (%d, %d) is not instantiated", P, Q);
    return b200::set_error_msg(msg);
  }
  const char *env = getenv("B200_JIT_ASSEMBLE_CTAS");  // read at every compile: part of the program text and its key
  const int ctas = env && atoi(env) > 0 ? atoi(env) : kAssembleCtas;
  env = getenv("B200_JIT_ASSEMBLE_UNROLL");
  const int unroll = env && env[0] ? atoi(env) != 0 : kAssembleUnroll;
  const int EB = b200::elems_per_block(Q), NT = 24 * EB, CH = NT < kAssembleMaxChunk ? NT : kAssembleMaxChunk;
  Entry *en = new Entry;
  en->key = options_line() + text +
            generated_assemble(name, nin, in_sizes, nout, out_sizes, active_in, active_out, Q, EB, NT, CH, ctas, unroll);
  en->kernel = std::string("b200_jit_assemble_") + name;
  en->kernel_tail = std::string("b200_jit_assemble_tail_") + name;
  en->nin = nin;
  en->nout = nout;
  for (int i = 0; i < nin; i++) en->in_size[i] = in_sizes[i];
  for (int i = 0; i < nout; i++) en->out_size[i] = out_sizes[i];
  en->assemble = true;
  en->P = P;
  en->Q = Q;
  en->ai = active_in;
  en->ao = active_out;
  en->lay[4] = EB;
  en->lay[5] = NT;
  en->smem = sizeof(double) * 81 * (size_t)CH;
  return find_or_compile(en, src_name, handle);
}

extern "C" int b200_jit_assemble_apply(int handle, const void *h_ctx, size_t ctx_bytes, int nelem,
                                       const double *h_interp1d, const double *h_grad1d, int nin,
                                       const double *const *d_in, double *d_values) {
  Entry *en;
  int dev;
  B200_CHECK(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lock(g_mu);
    if (handle < 0 || handle >= (int)g_entries.size() || !g_entries[handle]->assemble)
      return b200::set_error_msg("b200_jit_assemble_apply: bad handle");
    en = g_entries[handle];
    if (!en->lib) {
      B200_CHECK(cudaLibraryLoadData(&en->lib, en->cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0));
      B200_CHECK(cudaLibraryGetKernel(&en->fn, en->lib, en->kernel.c_str()));
      B200_CHECK(cudaLibraryGetKernel(&en->fn_tail, en->lib, en->kernel_tail.c_str()));
    }
    // the point tangents of a chunk take 62 to 83 KB: the limit is raised once per device
    if (en->smem > 48 * 1024 && dev >= 0 && dev < 64 && !(en->smem_set >> dev & 1)) {
      B200_CHECK(cudaKernelSetAttributeForDevice(en->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
      B200_CHECK(cudaKernelSetAttributeForDevice(en->fn_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)en->smem, dev));
      en->smem_set |= 1ull << dev;
    }
  }
  if (nin != en->nin) return b200::set_error_msg("b200_jit_assemble_apply: field count differs from the compiled one");
  if (ctx_bytes > B200_JIT_MAX_CTX) {
    char msg[160];
    snprintf(msg, sizeof msg, "b200_jit_assemble_apply: context of %zu bytes; a JIT QFunction takes at most %d",
             ctx_bytes, B200_JIT_MAX_CTX);
    return b200::set_error_msg(msg);
  }
  if (ctx_bytes && !h_ctx) return b200::set_error_msg("b200_jit_assemble_apply: NULL context");
  if (nelem <= 0) return 0;
  const int Q = en->Q, Q3 = Q * Q * Q, EB = en->lay[4], NT = en->lay[5];
  double mats[2 * 8 * 2];  // b200_k13_mats_t for this Q: interp1d [Q][2], then grad1d [Q][2]
  for (int i = 0; i < Q * 2; i++) {
    mats[i] = h_interp1d[i];
    mats[Q * 2 + i] = h_grad1d[i];
  }
  JitCtx ctx;
  memset(&ctx, 0, sizeof ctx);
  if (ctx_bytes) memcpy(ctx.b, h_ctx, ctx_bytes);
  const double *fin[B200_JIT_MAXF] = {};
  for (int i = 0; i < nin; i++) fin[i] = i == en->ai ? nullptr : d_in[i];
  const int nfull = nelem / EB, ntail = nelem - nfull * EB;
  if (nfull) {
    int n = nfull * EB;
    void *args[] = {mats, &ctx, fin, &n, &d_values};
    B200_CHECK(cudaLaunchKernel((const void *)en->fn, dim3(nfull), dim3(NT), args, en->smem, b200::g_stream));
    B200_LAUNCH_CHECK("b200_jit_assemble_apply");
  }
  if (ntail) {  // the partial group at the end: a run-time group extent, one CTA
    const size_t e0 = (size_t)nfull * EB;
    const double *ft[B200_JIT_MAXF] = {};
    for (int i = 0; i < nin; i++)
      if (fin[i]) ft[i] = fin[i] + e0 * en->in_size[i] * Q3;
    double *v = d_values + e0 * 576;
    int n = ntail;
    void *args[] = {mats, &ctx, ft, &n, &v};
    B200_CHECK(cudaLaunchKernel((const void *)en->fn_tail, dim3(1), dim3(NT), args, en->smem, b200::g_stream));
    B200_LAUNCH_CHECK("b200_jit_assemble_apply(tail)");
  }
  return 0;
}
