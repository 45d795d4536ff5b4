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
#include <dlfcn.h>
#include <nvrtc.h>
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

struct Entry {
  std::string key;     // options + program text
  std::string kernel;  // b200_jit_<Name>
  std::vector<char> cubin;
  int nin = 0, nout = 0, in_size[B200_JIT_MAXF] = {}, out_size[B200_JIT_MAXF] = {};
  cudaLibrary_t lib = nullptr;
  cudaKernel_t fn = nullptr;
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

}  // namespace

extern "C" int b200_jit_compile(const char *text, const char *src_name, const char *name, int nin, const int *in_sizes,
                                int nout, const int *out_sizes, int *handle) {
  *handle = -1;
  if (!text || !name) return b200::set_error_msg("b200_jit_compile: NULL program text or name");
  if (!is_identifier(name)) {
    char msg[256];
    snprintf(msg, sizeof msg, "b200_jit_compile: QFunction name \"%.128s\" is not a C identifier", name);
    return b200::set_error_msg(msg);
  }
  if (nin < 0 || nout < 1 || nin > B200_JIT_MAXF || nout > B200_JIT_MAXF)
    return b200::set_error_msg("b200_jit_compile: need 0..8 input and 1..8 output fields");
  for (int i = 0; i < nin + nout; i++) {
    const int s = i < nin ? in_sizes[i] : out_sizes[i - nin];
    if (s < 1 || s > B200_JIT_MAX_FIELD) {
      char msg[256];
      snprintf(msg, sizeof msg, "b200_jit_compile: %s field %d of QFunction %.128s has %d components; a JIT QFunction "
               "field holds 1 to %d", i < nin ? "input" : "output", i < nin ? i : i - nin, name, s, B200_JIT_MAX_FIELD);
      return b200::set_error_msg(msg);
    }
  }
  std::string key;
  for (int i = 0; i < kNumOptions; i++) key += std::string(kOptions[i]) + " ";
  key += "\n";
  key += text;
  key += generated_kernel(name, nin, in_sizes, nout, out_sizes);
  std::lock_guard<std::mutex> lock(g_mu);
  for (size_t i = 0; i < g_entries.size(); i++)
    if (g_entries[i]->key == key) {
      *handle = (int)i;
      return 0;
    }
  Entry *en = new Entry;
  en->key = std::move(key);
  en->kernel = std::string("b200_jit_") + name;
  en->nin = nin;
  en->nout = nout;
  for (int i = 0; i < nin; i++) en->in_size[i] = in_sizes[i];
  for (int i = 0; i < nout; i++) en->out_size[i] = out_sizes[i];
  if (int rc = compile_locked(*en, src_name && src_name[0] ? src_name : "qfunction")) {
    delete en;
    return rc;
  }
  g_entries.push_back(en);
  *handle = (int)g_entries.size() - 1;
  return 0;
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
