// eval_check, specialised per circuit: the PolyExtStep program is turned into straight-line CUDA C++ and compiled for
// sm_100a with NVRTC the first time a circuit is seen (SURVEY.md 8a-a12).
//
// The reference gets its `poly_fp` the same way, only ahead of time: risc0-circuit-rv32im-sys compiles a generated
// C++/CUDA function of ~10^5 lines with nvcc at crate build time (un-vendored; call site
// /root/reference/crates/guest-prover-r0/src/prover.rs:90).  Here the constraint system arrives as data (circuit.hpp), so
// the specialisation happens at `zkb_prover_new` / first `zkb_eval_check`:
//   * every Fp temporary and every mix accumulator is an SSA value in registers (the interpreter in k_eval_check.cu
//     spends ~65 instructions of decode / shared-memory traffic per PolyExtStep; the compiled form spends 1-5);
//   * taps are read straight from the column-major LDE matrices, one coalesced 128-byte line per warp and tap;
//   * per-proof values (globals, powers of poly_mix, the four (3x)^n - 1 inverses) are kernel DATA, so one cubin serves
//     every segment of the circuit; cubins are cached in memory per ctx and on disk (ZKB_CACHE_DIR, default
//     /tmp/zkb200-cache) keyed by a hash of the generated source.
// libnvrtc / libcuda are dlopen'ed, not linked: when they are absent the caller falls back to the device interpreter
// (still CUDA -- there is no CPU path).
#include "common.cuh"
#include "circuit.hpp"
#include <cuda.h>
#include <nvrtc.h>
#include <dlfcn.h>
#include <sys/stat.h>
#include <unistd.h>
#include <fcntl.h>
#include <functional>
#include <thread>
#include <nvJitLink.h>
#include <cerrno>
#include <fstream>
#include <sstream>
#include <mutex>
#include <set>

namespace zkb {

namespace {

struct Api {
  bool ok = false;        // NVRTC usable (compile)
  bool cu_ok = false;     // driver API usable (load + launch)
  std::string why, cu_why;
  decltype(&nvrtcCreateProgram) createProgram;
  decltype(&nvrtcCompileProgram) compileProgram;
  decltype(&nvrtcGetCUBINSize) getCUBINSize;
  decltype(&nvrtcGetCUBIN) getCUBIN;
  decltype(&nvrtcGetProgramLogSize) getLogSize;
  decltype(&nvrtcGetProgramLog) getLog;
  decltype(&nvrtcDestroyProgram) destroyProgram;
  decltype(&nvrtcVersion) version = nullptr;
  decltype(&nvrtcGetPTXSize) getPTXSize = nullptr;
  decltype(&nvrtcGetPTX) getPTX = nullptr;
  // nvJitLink (flat form of heavy circuits: NVRTC kernel PTX + hand-emitted unit PTX -> one cubin); entry points are versioned (__nvJitLinkCreate_12_x)
  bool jl_ok = false; std::string jl_why;
  nvJitLinkResult (*jlCreate)(nvJitLinkHandle*, uint32_t, const char**) = nullptr;
  nvJitLinkResult (*jlDestroy)(nvJitLinkHandle*) = nullptr;
  nvJitLinkResult (*jlAddData)(nvJitLinkHandle, nvJitLinkInputType, const void*, size_t, const char*) = nullptr;
  nvJitLinkResult (*jlComplete)(nvJitLinkHandle) = nullptr;
  nvJitLinkResult (*jlCubinSize)(nvJitLinkHandle, size_t*) = nullptr;
  nvJitLinkResult (*jlCubin)(nvJitLinkHandle, void*) = nullptr;
  nvJitLinkResult (*jlLogSize)(nvJitLinkHandle, size_t*) = nullptr;
  nvJitLinkResult (*jlLog)(nvJitLinkHandle, char*) = nullptr;
  nvJitLinkResult (*jlInfoSize)(nvJitLinkHandle, size_t*) = nullptr;
  nvJitLinkResult (*jlInfo)(nvJitLinkHandle, char*) = nullptr;
  CUresult (*moduleLoadData)(CUmodule*, const void*);
  CUresult (*moduleGetFunction)(CUfunction*, CUmodule, const char*);
  CUresult (*moduleUnload)(CUmodule);
  CUresult (*launchKernel)(CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void**, void**);
  CUresult (*getErrorString)(CUresult, const char**);
  CUresult (*moduleGetGlobal)(CUdeviceptr*, size_t*, CUmodule, const char*);
  CUresult (*memcpyHtoDAsync)(CUdeviceptr, const void*, size_t, CUstream);
  CUresult (*funcSetAttribute)(CUfunction, CUfunction_attribute, int);
};

Api& api() {
  static Api a;
  static std::once_flag once;
  std::call_once(once, [] {
    // The NEWEST loadable NVRTC wins, not the first one found: a process that imported torch already has torch's bundled libnvrtc
    // (12.8 here) mapped under the same SONAME, and its code for the compact eval_check form is 8 % slower than the toolkit's 12.9
    // (134 vs 124 ms on SYN-HEAVY, profiles/r2_y_nvrtc_version.txt) -- the same source ran at two speeds depending on import order.
    // Candidates by path are separate mappings (RTLD_LOCAL: no symbol interposition between two NVRTCs).  ZKB_NVRTC_LIB pins one.
    void* rt = nullptr; int rt_ver = -1; std::string rt_dir;
    {
      std::vector<std::string> cands;
      if (const char* pin = getenv("ZKB_NVRTC_LIB")) cands.push_back(pin);
      else {
        for (const char* var : {"CUDA_HOME", "CUDA_PATH"}) if (const char* h = getenv(var)) if (*h == '/') cands.push_back(std::string(h) + "/lib64/libnvrtc.so.12");
        cands.push_back("/usr/local/cuda/lib64/libnvrtc.so.12"); cands.push_back("libnvrtc.so.12"); cands.push_back("libnvrtc.so");
      }
      for (const std::string& name : cands) {
        void* h = dlopen(name.c_str(), RTLD_NOW | RTLD_LOCAL);
        if (!h) continue;
        int maj = 0, min = 0;
        auto ver = (decltype(&nvrtcVersion))dlsym(h, "nvrtcVersion");
        if (ver && ver(&maj, &min) == NVRTC_SUCCESS && maj * 100 + min > rt_ver) {
          rt = h; rt_ver = maj * 100 + min;
          Dl_info info; rt_dir.clear();
          if (dladdr((void*)ver, &info) && info.dli_fname) { std::string f = info.dli_fname; size_t sl = f.rfind('/'); if (sl != std::string::npos) rt_dir = f.substr(0, sl); }
        }
      }
    }
    if (!rt) { a.why = "libnvrtc.so.12 not loadable"; return; }
    if (getenv("ZKB_EC_VERBOSE")) fprintf(stderr, "zkb200: NVRTC %d.%d from %s\n", rt_ver / 100, rt_ver % 100, rt_dir.empty() ? "?" : rt_dir.c_str());
    bool all = true;
    auto sym = [&](void* lib, const char* n) { void* p = dlsym(lib, n); if (!p) { all = false; a.why = std::string("missing symbol ") + n; } return p; };
    a.createProgram = (decltype(a.createProgram))sym(rt, "nvrtcCreateProgram");
    a.compileProgram = (decltype(a.compileProgram))sym(rt, "nvrtcCompileProgram");
    a.getCUBINSize = (decltype(a.getCUBINSize))sym(rt, "nvrtcGetCUBINSize");
    a.getCUBIN = (decltype(a.getCUBIN))sym(rt, "nvrtcGetCUBIN");
    a.getLogSize = (decltype(a.getLogSize))sym(rt, "nvrtcGetProgramLogSize");
    a.getLog = (decltype(a.getLog))sym(rt, "nvrtcGetProgramLog");
    a.destroyProgram = (decltype(a.destroyProgram))sym(rt, "nvrtcDestroyProgram");
    a.version = (decltype(a.version))dlsym(rt, "nvrtcVersion");
    a.getPTXSize = (decltype(a.getPTXSize))dlsym(rt, "nvrtcGetPTXSize");
    a.getPTX = (decltype(a.getPTX))dlsym(rt, "nvrtcGetPTX");
    a.ok = all;
    {
      void* jl = nullptr;          // the nvJitLink that ships next to the chosen NVRTC first (same toolkit version: it must accept that NVRTC's PTX)
      std::vector<std::string> jcands;
      if (!rt_dir.empty()) jcands.push_back(rt_dir + "/libnvJitLink.so.12");
      jcands.push_back("libnvJitLink.so.12"); jcands.push_back("libnvJitLink.so"); jcands.push_back("/usr/local/cuda/lib64/libnvJitLink.so.12");
      for (const std::string& name : jcands) { jl = dlopen(name.c_str(), RTLD_NOW | RTLD_LOCAL); if (jl) break; }
      if (!jl) a.jl_why = "libnvJitLink.so.12 not loadable";
      else {
        auto vsym = [&](const char* base) -> void* {
          for (int minor = 9; minor >= 0; --minor) { std::string n = std::string("__") + base + "_12_" + std::to_string(minor); if (void* p = dlsym(jl, n.c_str())) return p; }
          return dlsym(jl, base);
        };
        a.jlCreate = (decltype(a.jlCreate))vsym("nvJitLinkCreate"); a.jlDestroy = (decltype(a.jlDestroy))vsym("nvJitLinkDestroy");
        a.jlAddData = (decltype(a.jlAddData))vsym("nvJitLinkAddData"); a.jlComplete = (decltype(a.jlComplete))vsym("nvJitLinkComplete");
        a.jlCubinSize = (decltype(a.jlCubinSize))vsym("nvJitLinkGetLinkedCubinSize"); a.jlCubin = (decltype(a.jlCubin))vsym("nvJitLinkGetLinkedCubin");
        a.jlLogSize = (decltype(a.jlLogSize))vsym("nvJitLinkGetErrorLogSize"); a.jlLog = (decltype(a.jlLog))vsym("nvJitLinkGetErrorLog");
        a.jlInfoSize = (decltype(a.jlInfoSize))vsym("nvJitLinkGetInfoLogSize"); a.jlInfo = (decltype(a.jlInfo))vsym("nvJitLinkGetInfoLog");
        a.jl_ok = a.jlCreate && a.jlDestroy && a.jlAddData && a.jlComplete && a.jlCubinSize && a.jlCubin && a.getPTXSize && a.getPTX;
        if (!a.jl_ok) a.jl_why = "nvJitLink / nvrtcGetPTX entry points missing";
      }
    }
    void* cu = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!cu) { a.cu_why = "libcuda.so.1 not loadable"; return; }
    all = true;
    a.moduleLoadData = (decltype(a.moduleLoadData))sym(cu, "cuModuleLoadData");
    a.moduleGetFunction = (decltype(a.moduleGetFunction))sym(cu, "cuModuleGetFunction");
    a.moduleUnload = (decltype(a.moduleUnload))sym(cu, "cuModuleUnload");
    a.launchKernel = (decltype(a.launchKernel))sym(cu, "cuLaunchKernel");
    a.getErrorString = (decltype(a.getErrorString))sym(cu, "cuGetErrorString");
    a.moduleGetGlobal = (decltype(a.moduleGetGlobal))sym(cu, "cuModuleGetGlobal_v2");
    a.memcpyHtoDAsync = (decltype(a.memcpyHtoDAsync))sym(cu, "cuMemcpyHtoDAsync_v2");
    a.funcSetAttribute = (decltype(a.funcSetAttribute))sym(cu, "cuFuncSetAttribute");
    a.cu_ok = all;
    if (!all) a.cu_why = a.why;
  });
  return a;
}

constexpr int JIT_BLOCK = 128;

const char* PREAMBLE = R"(
typedef unsigned int u32; typedef unsigned long long u64;
#define P 2013265921u
#define NB 1073741848u   /* Montgomery form of -11 (Fp4 = Fp[x]/(x^4+11)) */
// Two-input additions / subtractions are written min(a +- b, ONES) with ONES = 0xffffffff read from the constant bank (opaque
// to the compiler): ptxas emits ONE VIADDMNMX (ALU pipe) for it and cannot choose IMAD.IADD, which would land on the
// multiplier pipe this kernel is bound by (see poseidon2.cuh).  ZKB_EC_ALU_ADDS=0 restores plain additions.
__constant__ u32 zkb_ones = 0xffffffffu;
#if ZKB_ALU_ADDS
#define ADD2(a, b) min((a) + (b), zkb_ones)
#define SUB2(a, b) min((a) - (b), zkb_ones)
#else
#define ADD2(a, b) ((a) + (b))
#define SUB2(a, b) ((a) - (b))
#endif
__device__ __forceinline__ u32 red(u32 x) { return min(x, x - P); }
__device__ __forceinline__ u32 mul(u32 a, u32 b) { u64 t = (u64)a * b; u32 m = (u32)t * 0x88000001u; u32 r = SUB2((u32)(t >> 32), __umulhi(m, P)); return min(r, r + P); }
__device__ __forceinline__ u32 add(u32 a, u32 b) { return red(ADD2(a, b)); }
__device__ __forceinline__ u32 sub(u32 a, u32 b) { u32 d = SUB2(a, b); return min(d, d + P); }
// Lazy accumulation of sum_k pw_k * f_k (pw_k, f_k canonical): a 64-bit accumulator per Fp4 component takes one
// IMAD.WIDE per term; after every second term its high word is brought back below P (one VIADDMNMX), which keeps the
// accumulator below P * 2^32 + 2 P^2 < 2^64; a single Montgomery reduction at the end of the chain gives the canonical
// word.  An accumulator that continues from a canonical value m starts as m << 32 (= m * R).
__device__ __forceinline__ u64 wide(u32 f, u32 w) { return (u64)f * w; }
__device__ __forceinline__ u64 widem(u32 m, u32 f, u32 w) { return ((u64)m << 32) + (u64)f * w; }
__device__ __forceinline__ void wacc(u64& a, u32 f, u32 w) { a += (u64)f * w; }
__device__ __forceinline__ u64 fixhi(u64 a) { u32 hi = (u32)(a >> 32); hi = min(hi, hi - P); return ((u64)hi << 32) | (u32)a; }
__device__ __forceinline__ u32 fin(u64 a) { a = fixhi(a); u32 m = (u32)a * 0x88000001u; u32 r = SUB2((u32)(a >> 32), __umulhi(m, P)); return min(r, r + P); }
__device__ __forceinline__ void st(u32* p, u32 v) { *p = v; }
)";

// Fp4 arithmetic over a component type T (u32 here; the helpers are generic); the second operand of mul4 is a power of poly_mix
const char* PREAMBLE_F4 = R"(
template <class T> struct F4T { T a, b, c, d; };
typedef F4T<u32> F4;
template <class T> __device__ __forceinline__ F4T<T> mul4(F4T<T> x, F4 y) {
  F4T<T> r;
  r.a = add(mul(x.a, y.a), mul(add(add(mul(x.b, y.d), mul(x.c, y.c)), mul(x.d, y.b)), NB));
  r.b = add(add(mul(x.a, y.b), mul(x.b, y.a)), mul(add(mul(x.c, y.d), mul(x.d, y.c)), NB));
  r.c = add(add(add(mul(x.a, y.c), mul(x.b, y.b)), mul(x.c, y.a)), mul(mul(x.d, y.d), NB));
  r.d = add(add(add(mul(x.a, y.d), mul(x.b, y.c)), mul(x.c, y.b)), mul(x.d, y.a));
  return r;
}
__device__ __forceinline__ F4 tof4(uint4 w) { F4 r; r.a = w.x; r.b = w.y; r.c = w.z; r.d = w.w; return r; }
template <class T, class S> __device__ __forceinline__ F4T<T> scale4(F4T<T> x, S s) { F4T<T> r; r.a = mul(x.a, s); r.b = mul(x.b, s); r.c = mul(x.c, s); r.d = mul(x.d, s); return r; }
template <class T> __device__ __forceinline__ F4T<T> add4(F4T<T> x, F4T<T> y) { F4T<T> r; r.a = add(x.a, y.a); r.b = add(x.b, y.b); r.c = add(x.c, y.c); r.d = add(x.d, y.d); return r; }
)";


uint64_t fnv1a(const std::string& s) {
  uint64_t h = 1469598103934665603ull;
  for (unsigned char c : s) { h ^= c; h *= 1099511628211ull; }
  return h;
}

}  // namespace

struct EvalJitKernel {
  CUmodule mod = nullptr;
  CUfunction fn = nullptr;
  uint32_t n_powers = 1;
  int block = 128;                // threads per CTA (one domain point per thread)
  int points = 0;                 // domain points per CTA if != block (flat form)
  std::vector<uint32_t> term_power;    // flat form: the power table is laid out in term order
  size_t smem = 0;                // dynamic shared memory per CTA
  CUdeviceptr cdata = 0;        // __constant__ zkb_cd (per-proof powers + globals) when the circuit's data fits in 64 KB
  size_t cdata_bytes = 0;
};
struct AccumJitKernel { CUmodule mod = nullptr; std::vector<CUfunction> phases; };
struct EvalJitCache {
  std::map<uint64_t, EvalJitKernel> kernels;     // keyed by hash of the circuit blob content
  std::map<uint64_t, bool> failed;
  std::map<uint64_t, AccumJitKernel> accum;      // witness programs (CircuitHal::accumulate), one kernel per phase
};

static int min_blocks();
// Variants of the register form that were measured on B200 and removed again (SYN-280, 2^22 points; profiles/r1_l_ec_variants.txt):
// 2 / 4 rows per thread with 64 / 128-bit tap loads and the `back` tap taken from the neighbouring lane by shuffle: 2.6-5.0 ms (the
// 64-bit accumulators of 4 rows spill); per-thread row pointers + uniform column offsets: 2.7 ms; this form: 2.4-2.5 ms.
static uint32_t ec_batch() { const char* e = getenv("ZKB_EC_BATCH"); int v = e ? atoi(e) : 4; return (uint32_t)(v < 1 ? 1 : v > 4096 ? 4096 : v); }
static uint32_t ec_prefetch() { const char* e = getenv("ZKB_EC_PREFETCH"); int v = e ? atoi(e) : 1; return (uint32_t)(v < 0 ? 0 : v > 8 ? 8 : v); }
// Per-proof kernel data: [powers of poly_mix, 4 words each][mix globals][out globals].  It lives in the module's
// __constant__ bank when it fits (operands then come straight from the constant cache), else behind a pointer.
constexpr size_t CONST_WORDS_MAX = 15 * 1024;
static bool const_mode(const CircuitDef& c, uint32_t n_powers) { return 4 * (size_t)n_powers + c.mix_size + c.out_size <= CONST_WORDS_MAX; }

// Straight-line source for the circuit (one domain point per thread); gi.n_powers = number of poly_mix powers the kernel reads.
// Liveness and mix-power bookkeeping shared by the generators.
struct Analysis {
  std::vector<char> fp_used, mx_used;
  std::vector<uint32_t> fp_of, mx_of;             // step index -> fp / mix value id
  std::vector<uint32_t> eqz_uses, other_uses;     // how each live mix value is consumed: as the base of a following AndEqz (chainable), or otherwise
  std::vector<uint32_t> mx_pow;                   // power of poly_mix a mix value has reached
  uint32_t n_powers = 1;
};
static Analysis analyse(const CircuitDef& c) {
  Analysis A;
  const size_t n = c.steps.size();
  A.fp_used.assign(c.n_fp_vars, 0); A.mx_used.assign(c.n_mix_vars, 0);
  A.fp_of.assign(n, 0); A.mx_of.assign(n, 0);
  { uint32_t fi = 0, mi = 0; for (size_t i = 0; i < n; ++i) { if (c.steps[i].op <= PX_MUL) A.fp_of[i] = fi++; else A.mx_of[i] = mi++; } }
  A.mx_used[c.ret] = 1;
  for (size_t i = n; i-- > 0;) {      // liveness from the returned mix value backwards
    const StepDef& s = c.steps[i];
    switch (s.op) {
      case PX_ADD: case PX_SUB: case PX_MUL: if (A.fp_used[A.fp_of[i]]) A.fp_used[s.a] = A.fp_used[s.b] = 1; break;
      case PX_AND_EQZ: if (A.mx_used[A.mx_of[i]]) { A.mx_used[s.a] = 1; A.fp_used[s.b] = 1; } break;
      case PX_AND_COND: if (A.mx_used[A.mx_of[i]]) { A.mx_used[s.a] = A.mx_used[s.c] = 1; A.fp_used[s.b] = 1; } break;
      default: break;
    }
  }
  A.eqz_uses.assign(c.n_mix_vars, 0); A.other_uses.assign(c.n_mix_vars, 0); A.mx_pow.assign(c.n_mix_vars, 0);
  uint32_t mi = 0;
  for (size_t i = 0; i < n; ++i) {
    const StepDef& s = c.steps[i];
    if (s.op <= PX_MUL) continue;
    uint32_t id = mi++;
    if (s.op == PX_AND_EQZ) { A.mx_pow[id] = A.mx_pow[s.a] + 1; if (A.mx_used[id]) { ++A.eqz_uses[s.a]; A.n_powers = std::max(A.n_powers, A.mx_pow[s.a] + 1); } }
    else if (s.op == PX_AND_COND) { A.mx_pow[id] = A.mx_pow[s.a] + A.mx_pow[s.c]; if (A.mx_used[id]) { ++A.other_uses[s.a]; ++A.other_uses[s.c]; A.n_powers = std::max(A.n_powers, A.mx_pow[s.a] + 1); } }
  }
  ++A.other_uses[c.ret];
  return A;
}

// Shared-memory staged form (mode "staged"): a CTA owns SG_BLOCK (512) consecutive domain points.  The columns its constraints
// read are brought into shared memory by bulk asynchronous copies (cp.async.bulk, completion on an mbarrier) issued by one
// elected thread: columns read many times (the code group's constants) stay resident, the others stream through a ring of
// `stages` slots of `cps` columns, refilled `stages` blocks ahead of their use.  Taps then are LDS with an immediate offset
// (row - 4 back is the same column slot, a few words earlier: the slot holds `halo` rows in front of the tile), the loads
// in flight per SM are decoupled from the register file (ring bytes instead of registers), and no address arithmetic runs
// on the multiplier pipe.
// threads (= domain points) per staged CTA; ZKB_EC_BLOCK in {128, 256, 512, 1024}.  Measured (SYN-280, 2^22 points): 128: 2.25 ms, 256: 1.79 ms,
// 512: 1.60 ms, 1024: 1.70 ms -- longer contiguous copies per column (2 KB) use the HBM better, at the same 2048 threads per SM.
static int sg_block() { const char* e = getenv("ZKB_EC_BLOCK"); int v = e ? atoi(e) : 512; return v == 128 || v == 256 || v == 1024 ? v : 512; }
#define SG_BLOCK sg_block()
struct GenInfo {
  uint32_t n_powers = 1;
  int block = JIT_BLOCK;     // threads per CTA
  int points = 0;            // domain points per CTA when that differs from `block` (flat form: several warp groups per point)
  std::vector<uint32_t> term_power;   // flat form: entry t of the kernel's power table is poly_mix^term_power[t] (table in TERM order)
  size_t smem = 0;           // dynamic shared memory (staged form)
  bool staged = false;
};
static bool ec_staged() { const char* e = getenv("ZKB_EC_STAGED"); return !e || atoi(e) != 0; }
static uint32_t env_u32(const char* name, uint32_t def, uint32_t lo, uint32_t hi) { const char* e = getenv(name); long v = e ? atol(e) : (long)def; return (uint32_t)(v < (long)lo ? lo : v > (long)hi ? hi : v); }

const char* PREAMBLE_STAGED = R"(
__device__ __forceinline__ u32 saddr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u64* bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(saddr(bar)), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(saddr(bar)), "r"(bytes) : "memory"); }
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity) {
  u32 ok;
  do { asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(saddr(bar)), "r"(parity) : "memory"); } while (!ok);
}
__device__ __forceinline__ void bulk_g2s(u32* dst, const u32* src, u32 bytes, u64* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" :: "r"(saddr(dst)), "l"(src), "r"(bytes), "r"(saddr(bar)) : "memory");
}
// rows [c0 - HALO, c0 + BLOCK) of one column into a slot; the first tile wraps around the end of the domain
__device__ __forceinline__ void copy_col(u32* dst, const u32* col, u32 c0, u32 mask, u64* bar) {
  if (HALO == 0) bulk_g2s(dst, col + c0, BLOCK * 4u, bar);
  else if (c0 >= HALO) bulk_g2s(dst, col + (c0 - HALO), ROWP * 4u, bar);
  else { bulk_g2s(dst, col + ((c0 - HALO) & mask), HALO * 4u, bar); bulk_g2s(dst + HALO, col + c0, BLOCK * 4u, bar); }
}
)";

static std::string generate(const CircuitDef& c, GenInfo& gi, bool staged) {
  const size_t n = c.steps.size();
  const Analysis A = analyse(c);
  uint32_t& n_powers = gi.n_powers;
  gi.block = JIT_BLOCK; gi.smem = 0; gi.staged = false;
  const std::vector<char>&fp_used = A.fp_used, &mx_used = A.mx_used;
  const std::vector<uint32_t>&fp_of = A.fp_of, &eqz_uses = A.eqz_uses, &other_uses = A.other_uses, &mx_pow = A.mx_pow;
  n_powers = A.n_powers;
  const bool cm = const_mode(c, n_powers);
  const size_t gl_off = 4 * (size_t)n_powers;
  // ---- staged form: which columns are resident, which stream, and in which block / slot every tap is found ----------
  struct ColUse { uint32_t group, column, uses; };
  uint32_t halo = 0, n_res = 0, cps = 0, stages = 0, rowp = 0;
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> res_slot;               // resident (group, column) -> slot
  std::vector<std::vector<std::pair<uint32_t, uint32_t>>> blocks;           // streamed columns of every block, slot order
  std::vector<uint32_t> get_block(n, 0), get_slot(n, 0);
  if (staged) {
    std::map<std::pair<uint32_t, uint32_t>, uint32_t> uses;
    for (size_t i = 0; i < n; ++i) if (c.steps[i].op == PX_GET && fp_used[fp_of[i]]) {
      const TapDef& t = c.taps[c.steps[i].a];
      ++uses[{t.group, t.column}];
      halo = std::max(halo, 4 * t.back);
    }
    const uint32_t res_max = env_u32("ZKB_EC_RES", 32, 0, 64), res_min_uses = env_u32("ZKB_EC_RES_USES", 4, 2, 1u << 30);
    // measured on B200, SYN-280 (profiles/r1_o_ec_staged.txt), 256-point CTAs: 2 stages x 6 columns = 1.82 ms (28 KB per CTA: eight CTAs = 2048
    // threads per SM), 3 x 6: 1.89-1.96 ms; deeper or wider rings cost occupancy (6 x 8: 3.25 ms, 10 x 8: 4.35 ms); the register form takes
    // 2.4-2.5 ms.  With 512-point CTAs (the default): 2 x 6 = 1.60 ms, 2 x 4 = 1.65 ms, 2 x 8 = 1.86 ms, 3 x 6 = 1.99 ms.
    cps = env_u32("ZKB_EC_CPS", 6, 1, 32); stages = env_u32("ZKB_EC_STAGES", 2, 2, 16);
    std::vector<ColUse> cand;
    for (auto& kv : uses) if (kv.second >= res_min_uses) cand.push_back({kv.first.first, kv.first.second, kv.second});
    std::stable_sort(cand.begin(), cand.end(), [](const ColUse& x, const ColUse& y) { return x.uses > y.uses; });
    for (auto& cu : cand) { if (n_res >= res_max) break; res_slot[{cu.group, cu.column}] = n_res++; }
    rowp = SG_BLOCK + halo;
    std::map<std::pair<uint32_t, uint32_t>, uint32_t> cur;                  // streamed column -> slot in the block being formed
    blocks.emplace_back();
    for (size_t i = 0; i < n; ++i) if (c.steps[i].op == PX_GET && fp_used[fp_of[i]]) {
      const TapDef& t = c.taps[c.steps[i].a];
      std::pair<uint32_t, uint32_t> key{t.group, t.column};
      if (res_slot.count(key)) { get_block[i] = (uint32_t)blocks.size() - 1; continue; }
      auto it = cur.find(key);
      if (it == cur.end()) {
        if (cur.size() == cps) { blocks.emplace_back(); cur.clear(); }
        it = cur.emplace(key, (uint32_t)cur.size()).first;
        blocks.back().push_back(key);
      }
      get_block[i] = (uint32_t)blocks.size() - 1; get_slot[i] = it->second;
    }
    if (blocks.back().empty() && blocks.size() > 1) blocks.pop_back();
    stages = std::min<uint32_t>(stages, (uint32_t)std::max<size_t>(blocks.size(), 1));
    gi.smem = ((size_t)n_res + (size_t)stages * cps) * rowp * 4 + (stages + 1) * 8;
    if (halo > SG_BLOCK || gi.smem > 200 * 1024) return std::string();      // does not fit this form: the caller uses the register form
    gi.block = SG_BLOCK; gi.staged = true;
  }
  std::ostringstream o;
  o << "#define ZKB_ALU_ADDS " << (env_u32("ZKB_EC_ALU_ADDS", 1, 0, 1) ? 1 : 0) << "\n" << PREAMBLE;
  if (staged) o << "#define HALO " << halo << "u\n#define BLOCK " << SG_BLOCK << "u\n#define ROWP " << rowp << "u\n" << PREAMBLE_STAGED;
  o << "typedef u32 RV; typedef u64 ACC;\n#define W0(f, w) wide(f, w)\n#define WM(m, f, w) widem(m, f, w)\n#define LD(p) __ldg(p)\n";
  o << PREAMBLE_F4 << "typedef F4T<RV> MV;\n";
  if (cm) {
    o << "__constant__ u32 zkb_cd[" << std::max<size_t>(gl_off + c.mix_size + c.out_size, 4) << "];\n"
         "#define PW(k) make_uint4(zkb_cd[4 * (k)], zkb_cd[4 * (k) + 1], zkb_cd[4 * (k) + 2], zkb_cd[4 * (k) + 3])\n"
         "#define GL(i) zkb_cd[" << gl_off << " + (i)]\n";
  } else {
    o << "#define PW(k) __ldg(pw + (k))\n#define GL(i) __ldg(gl + (i))\n";
  }
  const int ctas_per_sm = staged ? (int)std::max<size_t>(1, std::min<size_t>(env_u32("ZKB_EC_MINBLOCKS", 8, 1, 16), (227 * 1024) / (gi.smem + 1024))) : min_blocks();
  o << "extern \"C\" __global__ void __launch_bounds__(" << gi.block << ", " << ctas_per_sm << ") zkb_ec(u32* __restrict__ check, const u32* __restrict__ g0, const u32* __restrict__ g1, "
       "const u32* __restrict__ g2, const uint4* __restrict__ pw, const u32* __restrict__ gl, uint4 invden, u32 mask) {\n"
       << (staged ? "  size_t dom; asm(\"add.u64 %0, %1, 1;\" : \"=l\"(dom) : \"l\"((u64)mask));     // opaque: see the note on uniform address arithmetic below\n"
                  : "  const size_t dom = (size_t)mask + 1;\n")
       << "  const u32 c = blockIdx.x * " << gi.block << "u + threadIdx.x;\n";
  // producer code of one block: expect the bytes, then one bulk copy per column (issued by thread 0 only)
  auto issue_block = [&](uint32_t b) {
    const uint32_t st = b % stages;
    o << "    mbar_expect_tx(full + " << st << ", " << blocks[b].size() * rowp * 4 << "u);\n";
    for (size_t k = 0; k < blocks[b].size(); ++k)
      o << "    copy_col(ring + " << ((size_t)st * cps + k) * rowp << "u, g" << blocks[b][k].first << " + (size_t)" << blocks[b][k].second << " * dom, c0, mask, full + " << st << ");\n";
  };
  uint32_t cur_block = 0;
  if (staged) {
    o << "  extern __shared__ __align__(128) u32 zkb_sm[];\n"
         "  u32* const ring = zkb_sm + " << (size_t)n_res * rowp << "u;\n"
         "  u64* const full = reinterpret_cast<u64*>(zkb_sm + " << ((size_t)n_res + (size_t)stages * cps) * rowp << "u);     // [stages] ring barriers + 1 for the resident columns\n"
         "  const u32 c0 = blockIdx.x * BLOCK;\n"
         "  const u32* const sp = zkb_sm + threadIdx.x + HALO;          // this thread's row inside every column slot\n"
         "  if (threadIdx.x == 0) {\n    for (u32 i = 0; i <= " << stages << "u; ++i) mbar_init(full + i, 1u);\n"
         "    asm volatile(\"fence.mbarrier_init.release.cluster;\" ::: \"memory\");\n  }\n  __syncthreads();\n"
         "  if (threadIdx.x == 0) {\n";
    if (n_res) {
      o << "    mbar_expect_tx(full + " << stages << ", " << (size_t)n_res * rowp * 4 << "u);\n";
      for (auto& kv : res_slot) o << "    copy_col(zkb_sm + " << (size_t)kv.second * rowp << "u, g" << kv.first.first << " + (size_t)" << kv.first.second << " * dom, c0, mask, full + " << stages << ");\n";
    }
    for (uint32_t b = 0; b < stages && b < blocks.size(); ++b) if (!blocks[b].empty()) issue_block(b);
    o << "  }\n";
    if (n_res) o << "  mbar_wait(full + " << stages << ", 0u);\n";
    if (!blocks[0].empty()) o << "  mbar_wait(full + 0, 0u);\n";
  }
  // moves the kernel from block `cur_block` to block b: everybody has finished reading the old slot before it is refilled
  auto advance_to = [&](uint32_t b) {
    while (cur_block < b) {
      if (cur_block + stages < blocks.size()) {
        o << "  __syncthreads();\n  if (threadIdx.x == 0) {\n    asm volatile(\"fence.proxy.async.shared::cta;\" ::: \"memory\");\n";
        issue_block(cur_block + stages);
        o << "  }\n";
      }
      ++cur_block;
      o << "  mbar_wait(full + " << cur_block % stages << ", " << ((cur_block / stages) & 1) << "u);\n";
    }
  };
  auto staged_get = [&](size_t i) {
    const TapDef& t = c.taps[c.steps[i].a];
    advance_to(get_block[i]);
    auto r = res_slot.find({t.group, t.column});
    std::ostringstream a;
    const long slot_words = r != res_slot.end() ? (long)r->second * rowp : (long)((size_t)n_res + (size_t)(get_block[i] % stages) * cps + get_slot[i]) * rowp;
    a << "sp[" << slot_words - 4 * (long)t.back << "]";
    return a.str();
  };
  auto tap_addr = [&](const TapDef& t) {
    std::ostringstream a;
    a << "g" << t.group << " + (size_t)" << t.column << " * dom + ((c - " << 4 * t.back << "u) & mask)";
    return a.str();
  };
  enum { ST_ZERO = 0, ST_CANON = 1, ST_ACC = 2 };
  std::vector<char> state(c.n_mix_vars, ST_ZERO);
  std::vector<uint32_t> acc_set(c.n_mix_vars, 0), acc_terms(c.n_mix_vars, 0);
  auto materialize = [&](uint32_t id) {      // accumulators of `id` -> canonical Fp4 m<id>
    uint32_t a = acc_set[id];
    o << "  MV m" << id << "; m" << id << ".a = fin(A" << a << "_0); m" << id << ".b = fin(A" << a << "_1); m" << id << ".c = fin(A" << a << "_2); m" << id << ".d = fin(A" << a << "_3);\n";
    state[id] = ST_CANON;
  };
  // Load scheduling.  The kernel is bound by global-load latency (ncu: 87 % long-scoreboard stalls when every tap is loaded
  // right before its use), so the tap loads of the next `batch` constraints are hoisted in front of the arithmetic of the
  // current ones (software pipelining, distance `prefetch` batches); a tap needed twice within the hoisted group is loaded once.
  const uint32_t batch = ec_batch(), prefetch = ec_prefetch();
  std::vector<uint32_t> get_batch(n, 0);
  uint32_t n_batches = 1;
  {
    uint32_t live_mix = 0, mj = 0;
    for (size_t i = 0; i < n; ++i) {
      const StepDef& s = c.steps[i];
      if (s.op <= PX_MUL) { get_batch[i] = live_mix / batch; continue; }
      uint32_t id = mj++;
      if (s.op != PX_TRUE && mx_used[id]) ++live_mix;
    }
    n_batches = live_mix / batch + 1;
  }
  std::vector<std::vector<size_t>> gets_of(n_batches + 1);
  if (!staged) for (size_t i = 0; i < n; ++i) if (c.steps[i].op == PX_GET && fp_used[fp_of[i]]) gets_of[std::min<uint32_t>(get_batch[i], n_batches)].push_back(i);
  std::vector<char> get_done(n, 0);
  auto hoist = [&](uint32_t b) {
    if (b >= gets_of.size()) return;
    std::map<uint32_t, uint32_t> seen;       // tap -> fp id, within this group
    for (size_t i : gets_of[b]) {
      const StepDef& s = c.steps[i];
      auto it = seen.find(s.a);
      if (it != seen.end()) { o << "  const RV f" << fp_of[i] << " = f" << it->second << ";\n"; }
      else { o << "  const RV f" << fp_of[i] << " = LD(" << tap_addr(c.taps[s.a]) << ");\n"; seen[s.a] = fp_of[i]; }
      get_done[i] = 1;
    }
  };
  uint32_t hoisted_upto = 0;                  // batches [0, hoisted_upto) have had their loads emitted
  auto hoist_until = [&](uint32_t b_end) { while (hoisted_upto < b_end && hoisted_upto < gets_of.size()) hoist(hoisted_upto++); };
  hoist_until(1 + prefetch);
  uint32_t live_seen = 0;
  uint32_t fi = 0, mi = 0;
  for (size_t i = 0; i < n; ++i) {
    const StepDef& s = c.steps[i];
    if (s.op <= PX_MUL) {
      uint32_t id = fi++;
      if (!fp_used[id]) continue;
      if (s.op == PX_GET && get_done[i]) continue;
      std::string get_expr;
      if (s.op == PX_GET) get_expr = staged ? staged_get(i) : "LD(" + tap_addr(c.taps[s.a]) + ")";      // (staged_get may first emit a block change)
      o << "  const auto f" << id << " = ";
      switch (s.op) {
        case PX_CONST: o << Fp::from(s.a).v << "u"; break;
        case PX_GET: o << get_expr; break;
        case PX_GET_GLOBAL: o << "GL(" << (s.a == 0 ? s.b : c.mix_size + s.b) << ")"; break;
        case PX_ADD: o << "add(f" << s.a << ", f" << s.b << ")"; break;
        case PX_SUB: o << "sub(f" << s.a << ", f" << s.b << ")"; break;
        case PX_MUL: o << "mul(f" << s.a << ", f" << s.b << ")"; break;
      }
      o << ";\n";
      continue;
    }
    uint32_t id = mi++;
    if (s.op == PX_TRUE) { state[id] = ST_ZERO; continue; }
    if (!mx_used[id]) continue;
    ++live_seen;
    if (live_seen % batch == 0) hoist_until(live_seen / batch + 1 + prefetch);      // entering the next batch: start the loads `prefetch` batches ahead
    if (s.op == PX_AND_EQZ) {
      const uint32_t base = s.a, k = mx_pow[base];
      uint32_t set, terms;
      if (state[base] == ST_ACC && eqz_uses[base] == 1 && other_uses[base] == 0) {          // continue the chain in place
        set = acc_set[base]; terms = acc_terms[base];
        o << "  { const uint4 w = PW(" << k << "); wacc(A" << set << "_0, f" << s.b << ", w.x); wacc(A" << set << "_1, f" << s.b << ", w.y); wacc(A" << set
          << "_2, f" << s.b << ", w.z); wacc(A" << set << "_3, f" << s.b << ", w.w); }\n";
        ++terms;
      } else {
        set = id;
        if (state[base] == ST_ACC) materialize(base);       // (cannot happen: multi-use values are materialised at definition)
        if (state[base] == ST_ZERO) {
          o << "  ACC A" << set << "_0, A" << set << "_1, A" << set << "_2, A" << set << "_3; { const uint4 w = PW(" << k << "); A" << set << "_0 = W0(f" << s.b
            << ", w.x); A" << set << "_1 = W0(f" << s.b << ", w.y); A" << set << "_2 = W0(f" << s.b << ", w.z); A" << set << "_3 = W0(f" << s.b << ", w.w); }\n";
        } else {
          o << "  ACC A" << set << "_0, A" << set << "_1, A" << set << "_2, A" << set << "_3; { const uint4 w = PW(" << k << "); A" << set << "_0 = WM(m" << base
            << ".a, f" << s.b << ", w.x); A" << set << "_1 = WM(m" << base << ".b, f" << s.b << ", w.y); A" << set << "_2 = WM(m" << base
            << ".c, f" << s.b << ", w.z); A" << set << "_3 = WM(m" << base << ".d, f" << s.b << ", w.w); }\n";
        }
        terms = 1;
      }
      if (terms == 2) {
        o << "  A" << set << "_0 = fixhi(A" << set << "_0); A" << set << "_1 = fixhi(A" << set << "_1); A" << set << "_2 = fixhi(A" << set << "_2); A" << set << "_3 = fixhi(A" << set << "_3);\n";
        terms = 0;
      }
      state[id] = ST_ACC; acc_set[id] = set; acc_terms[id] = terms;
      if (!(eqz_uses[id] == 1 && other_uses[id] == 0)) materialize(id);
      continue;
    }
    // PX_AND_COND: m_id = m_a + f_b * (m_c (x) poly_mix^pow(a)); operands are canonical (materialised at definition)
    if (state[s.c] == ST_ZERO) {           // inner chain is empty: nothing is added
      if (state[s.a] == ST_ZERO) state[id] = ST_ZERO;
      else { o << "  const MV m" << id << " = m" << s.a << ";\n"; state[id] = ST_CANON; }
      continue;
    }
    o << "  const MV m" << id << " = ";
    if (state[s.a] == ST_ZERO) o << "scale4(mul4(m" << s.c << ", tof4(PW(" << mx_pow[s.a] << "))), f" << s.b << ")";
    else o << "add4(m" << s.a << ", scale4(mul4(m" << s.c << ", tof4(PW(" << mx_pow[s.a] << "))), f" << s.b << "))";
    o << ";\n";
    state[id] = ST_CANON;
  }
  o << "  const u32 den = (c & 3u) == 0 ? invden.x : (c & 3u) == 1 ? invden.y : (c & 3u) == 2 ? invden.z : invden.w;\n";
  if (state[c.ret] == ST_ZERO) o << "  MV r; r.a = r.b = r.c = r.d = sub(den, den);\n";
  else o << "  const MV r = scale4(m" << c.ret << ", den);\n";
  o << "  st(check + c, r.a); st(check + dom + c, r.b); st(check + 2 * dom + c, r.c); st(check + 3 * dom + c, r.d);\n}\n";
  return o.str();
}

// ---- flat form: heavy circuits -------------------------------------------------------------------------------------------------
// rv32im's generated poly_fp has ~10^4 constraints that read the same few hundred columns from everywhere in the program: a
// streaming column ring would re-fetch every column hundreds of times, and one straight-line function of 10^5 steps keeps ~10^3 tap
// values live (spills) and takes ptxas tens of minutes.  For such programs the constraint tree is FLATTENED:
//     result.tot = sum over AndEqz terms of (product of the enclosing AndCond conditions) * poly_mix^(absolute power) * value
// (AndCond(x, c, y).tot = x.tot + c * x.mul * y.tot and x.mul = poly_mix^pow(x) with pow known statically, so every term's absolute
// power and condition list follow from one top-down walk).  Terms under the same condition list form a group: its values are
// accumulated unreduced in four 64-bit accumulators (one IMAD.WIDE per term and component), reduced once, multiplied by the
// condition product once.  No Fp4 x Fp4 product is left.
//   * a CTA owns FL_POINTS (128) consecutive domain points and brings EVERY tapped column (+ halo) into shared memory with one bulk
//     copy each (280 columns x 576 B = 161 KB): a tap is an LDS with an immediate offset wherever it is used, nothing stays live;
//   * the groups are cut into units of <= ZKB_EC_UNIT terms, each a __noinline__ device function (bounded compile time and register
//     pressure); FL_GROUPS (4) warp groups of 128 threads run disjoint subsets of the units on the same 128 points and add their partial
//     sums through shared memory (16 warps per SM although only one CTA fits).
static bool flat_wanted(const CircuitDef& c) {
  const char* e = getenv("ZKB_EC_FORM");
  if (e && (!strcmp(e, "flat") || !strcmp(e, "compact"))) return true;      // forced: "compact" = program as data, "flat" = PTX units
  if (e && *e) return false;
  size_t eqz = 0;
  for (const StepDef& s : c.steps) eqz += s.op == PX_AND_EQZ;
  return eqz >= env_u32("ZKB_EC_FLAT_MIN", 2000, 1, 1u << 30);
}
struct FlatTerm { uint32_t power, cl, value; };
// The flat form is generated as a small CUDA C++ kernel (tile load, warp-group dispatch, reduction: compiled by NVRTC with -rdc) plus
// the units as hand-emitted PTX functions, linked with nvJitLink.  Going through CUDA C++ for the units costs ~15 ms of NVVM
// front-end / optimiser time per constraint (6 minutes for SYN-HEAVY); as PTX only ptxas runs, on code that is already the wanted
// instruction sequence (mul.wide / mul.lo / mul.hi Montgomery products, mad.wide accumulation, min-pinned additions).
struct FlatProgram { std::string main_cu; std::vector<std::string> unit_ptx; int threads = 512; };
struct PtxEmit {
  std::ostringstream body;
  uint32_t nr = 8, nd = 4;         // %r0 = ones, %r1..%r4 = unit totals, %r5 = the warp group's named barrier; %rd0 = sp (shared), %rd1 = pw, %rd2 = gl
  std::string r() { return "%r" + std::to_string(nr++); }
  std::string rd() { return "%rd" + std::to_string(nd++); }
  std::string add(const std::string& a, const std::string& b) {
    std::string t = r(), u = r(), o = r();
    body << "  add.u32 " << t << ", " << a << ", " << b << "; min.u32 " << t << ", " << t << ", %r0; sub.u32 " << u << ", " << t << ", 2013265921; min.u32 " << o << ", " << t << ", " << u << ";\n";
    return o;
  }
  std::string sub(const std::string& a, const std::string& b) {
    std::string d = r(), e = r(), o = r();
    body << "  sub.u32 " << d << ", " << a << ", " << b << "; min.u32 " << d << ", " << d << ", %r0; add.u32 " << e << ", " << d << ", 2013265921; min.u32 " << o << ", " << d << ", " << e << ";\n";
    return o;
  }
  // Montgomery reduction of {lo, hi}: hi - hi(lo * P^-1 * P), canonical
  std::string redc(const std::string& lo, const std::string& hi) {
    std::string m = r(), u = r(), x = r(), y = r(), o = r();
    body << "  mul.lo.u32 " << m << ", " << lo << ", 0x88000001; mul.hi.u32 " << u << ", " << m << ", 2013265921; sub.u32 " << x << ", " << hi << ", " << u << "; min.u32 " << x << ", " << x
         << ", %r0; add.u32 " << y << ", " << x << ", 2013265921; min.u32 " << o << ", " << x << ", " << y << ";\n";
    return o;
  }
  std::string mul(const std::string& a, const std::string& b) {
    std::string t = rd(), lo = r(), hi = r();
    body << "  mul.wide.u32 " << t << ", " << a << ", " << b << "; mov.b64 {" << lo << ", " << hi << "}, " << t << ";\n";
    return redc(lo, hi);
  }
  void fixhi(const std::string& acc) {
    std::string lo = r(), hi = r(), h2 = r();
    body << "  mov.b64 {" << lo << ", " << hi << "}, " << acc << "; sub.u32 " << h2 << ", " << hi << ", 2013265921; min.u32 " << hi << ", " << hi << ", " << h2 << "; mov.b64 " << acc << ", {" << lo << ", " << hi << "};\n";
  }
  std::string fin(const std::string& acc) {
    std::string lo = r(), hi = r(), h2 = r();
    body << "  mov.b64 {" << lo << ", " << hi << "}, " << acc << "; sub.u32 " << h2 << ", " << hi << ", 2013265921; min.u32 " << hi << ", " << hi << ", " << h2 << ";\n";
    return redc(lo, hi);
  }
};
static bool generate_flat(const CircuitDef& c, GenInfo& gi, FlatProgram& prog) {
  const size_t n = c.steps.size();
  std::vector<size_t> fp_step(c.n_fp_vars), mx_step(c.n_mix_vars);
  { uint32_t fi = 0, mi = 0; for (size_t i = 0; i < n; ++i) { if (c.steps[i].op <= PX_MUL) fp_step[fi++] = i; else mx_step[mi++] = i; } }
  // static power of every mix value
  std::vector<uint32_t> mpow(c.n_mix_vars, 0);
  for (uint32_t m = 0; m < c.n_mix_vars; ++m) {
    const StepDef& s = c.steps[mx_step[m]];
    if (s.op == PX_AND_EQZ) mpow[m] = mpow[s.a] + 1; else if (s.op == PX_AND_COND) mpow[m] = mpow[s.a] + mpow[s.c];
  }
  // top-down walk from the result: (mix value, power offset, condition list)
  std::vector<std::vector<uint32_t>> cls(1);                 // interned condition lists; 0 = empty
  std::map<std::vector<uint32_t>, uint32_t> cl_id{{{}, 0u}};
  std::vector<FlatTerm> terms;
  struct Item { uint32_t m, off, cl; };
  std::vector<Item> stack{{c.ret, 0u, 0u}};
  while (!stack.empty()) {
    Item it = stack.back(); stack.pop_back();
    for (;;) {
      const StepDef& s = c.steps[mx_step[it.m]];
      if (s.op == PX_TRUE) break;
      if (s.op == PX_AND_EQZ) { terms.push_back({it.off + mpow[s.a], it.cl, s.b}); it.m = s.a; continue; }
      std::vector<uint32_t> inner = cls[it.cl]; inner.push_back(s.b);          // AndCond(x = s.a, cond = s.b, y = s.c)
      auto f = cl_id.find(inner);
      uint32_t id;
      if (f == cl_id.end()) { id = (uint32_t)cls.size(); cl_id.emplace(inner, id); cls.push_back(inner); } else id = f->second;
      stack.push_back({s.c, it.off + mpow[s.a], id});
      it.m = s.a;
    }
  }
  if (terms.empty()) return false;
  std::stable_sort(terms.begin(), terms.end(), [](const FlatTerm& x, const FlatTerm& y) { return x.cl != y.cl ? x.cl < y.cl : x.power < y.power; });
  // the kernel's power table is laid out in TERM order (entry t = poly_mix^terms[t].power), so that a unit's slice is contiguous
  // and can be staged in shared memory (below)
  gi.n_powers = (uint32_t)terms.size();
  gi.term_power.resize(terms.size());
  for (size_t t = 0; t < terms.size(); ++t) gi.term_power[t] = terms[t].power;
  // columns: every tapped column is resident
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> slot;
  uint32_t halo = 0;
  for (const TapDef& t : c.taps) { slot.emplace(std::make_pair(t.group, t.column), 0u); halo = std::max(halo, 4 * t.back); }
  { uint32_t k = 0; for (auto& kv : slot) kv.second = k++; }
  const uint32_t groups = env_u32("ZKB_EC_FLAT_GROUPS", 4, 1, 8);
  const uint32_t unit_terms = env_u32("ZKB_EC_UNIT", 256, 8, 512);
  // per warp group: the poly_mix powers of the unit it is running, staged in shared memory (one coalesced copy per unit instead of
  // one L2-latency load per term: the L1 holds the 161 KB tile, not the 330 KB table)
  const size_t pw_words = (size_t)groups * unit_terms * 4;
  uint32_t points = env_u32("ZKB_EC_FLAT_POINTS", 128, 32, 512);
  while (points > 32 && ((size_t)slot.size() * (points + halo) * 4 + (size_t)(groups - 1) * points * 16 + pw_words * 4 + 64 > 220 * 1024)) points >>= 1;
  const uint32_t rowp = points + halo;
  const size_t col_words = (size_t)slot.size() * rowp;
  gi.smem = col_words * 4 + (size_t)(groups - 1) * points * 16 + pw_words * 4 + 16;
  if (gi.smem > 220 * 1024 || (halo & 3)) return false;
  gi.block = (int)(points * groups); gi.points = (int)points; gi.staged = true;
  // units
  struct Unit { size_t lo, hi; };
  std::vector<Unit> units;
  for (size_t i = 0; i < terms.size();) {
    size_t j = i;
    while (j < terms.size() && j - i < unit_terms) {           // whole groups while they fit; a group longer than a unit is cut
      size_t g_end = j; while (g_end < terms.size() && terms[g_end].cl == terms[j].cl) ++g_end;
      if (g_end - i <= unit_terms || j == i) j = std::min(g_end, i + unit_terms); else break;
    }
    units.push_back({i, j}); i = j;
  }
  // ---- the units, as PTX -----------------------------------------------------------------------------------------------
  const uint32_t per_module = env_u32("ZKB_EC_FLAT_MODULE", 16, 1, 1u << 20);      // unit functions per PTX module (one ptxas run each)
  // The code of a heavy circuit (9 MB for SYN-HEAVY) streams through the instruction caches once per tile; ncu shows the kernel bound by
  // instruction fetch from L2 (1.14 instructions / clock / SM, 9 of 14 cycles per issued instruction "no instruction") when every warp
  // fetches its own copy.  A named barrier every `sync_terms` terms keeps the four warps of a group within a few KB of each other, so a
  // line fetched into the SM's 32 KB L1.5 instruction cache serves all of them.
  const uint32_t sync_terms = env_u32("ZKB_EC_FLAT_SYNC", 16, 0, 1u << 20);
  prog.unit_ptx.clear();
  std::ostringstream mod;
  auto begin_module = [&] { mod.str(std::string()); mod << ".version 8.6\n.target sm_100a\n.address_size 64\n\n"; };      // 8.6 = the first ISA with sm_100a: accepted by every nvJitLink 12.x that knows the target
  begin_module();
  for (size_t u = 0; u < units.size(); ++u) {
    PtxEmit e;
    // Get / Const / GetGlobal are loaded where they are used; arithmetic nodes become registers local to one group
    std::function<std::string(uint32_t, std::map<uint32_t, std::string>&)> operand = [&](uint32_t f, std::map<uint32_t, std::string>& local) -> std::string {
      auto it = local.find(f);
      if (it != local.end()) return it->second;
      const StepDef& s = c.steps[fp_step[f]];
      if (s.op == PX_CONST) { std::string x = e.r(); e.body << "  mov.u32 " << x << ", " << Fp::from(s.a).v << ";\n"; return x; }
      if (s.op == PX_GET) {
        const TapDef& t = c.taps[s.a];
        std::string x = e.r();
        e.body << "  ld.shared.u32 " << x << ", [%rd0+" << 4 * ((long)slot[{t.group, t.column}] * rowp - 4 * (long)t.back) << "];\n";
        return x;
      }
      if (s.op == PX_GET_GLOBAL) { std::string x = e.r(); e.body << "  ld.global.nc.u32 " << x << ", [%rd2+" << 4 * (s.a == 0 ? s.b : c.mix_size + s.b) << "];\n"; return x; }
      std::string x = operand(s.a, local), y = operand(s.b, local);
      std::string o = s.op == PX_ADD ? e.add(x, y) : s.op == PX_SUB ? e.sub(x, y) : e.mul(x, y);
      local[f] = o;
      return o;
    };
    for (size_t i = units[u].lo; i < units[u].hi;) {
      size_t j = i; while (j < units[u].hi && terms[j].cl == terms[i].cl) ++j;
      std::map<uint32_t, std::string> local;
      std::string A[4] = {e.rd(), e.rd(), e.rd(), e.rd()};
      for (size_t k = i; k < j; ++k) {
        std::string v = operand(terms[k].value, local);
        std::string w[4] = {e.r(), e.r(), e.r(), e.r()};
        e.body << "  ld.shared.v4.u32 {" << w[0] << ", " << w[1] << ", " << w[2] << ", " << w[3] << "}, [%r6+" << 16 * (k - units[u].lo) << "];\n";
        for (int q = 0; q < 4; ++q) {
          if (k == i) e.body << "  mul.wide.u32 " << A[q] << ", " << v << ", " << w[q] << ";\n";
          else e.body << "  mad.wide.u32 " << A[q] << ", " << v << ", " << w[q] << ", " << A[q] << ";\n";
        }
        if (((k - i) & 1) == 1 && k + 1 < j) for (int q = 0; q < 4; ++q) e.fixhi(A[q]);
        if (sync_terms && groups > 0 && (k - units[u].lo) % sync_terms == sync_terms - 1) e.body << "  bar.sync %r5, " << points << ";\n";
      }
      std::string leaf[4];
      for (int q = 0; q < 4; ++q) leaf[q] = e.fin(A[q]);
      const std::vector<uint32_t>& cl = cls[terms[i].cl];
      if (!cl.empty()) {
        std::string cp = operand(cl[0], local);
        for (size_t q = 1; q < cl.size(); ++q) cp = e.mul(cp, operand(cl[q], local));
        for (int q = 0; q < 4; ++q) leaf[q] = e.mul(leaf[q], cp);
      }
      for (int q = 0; q < 4; ++q) { std::string t = e.add("%r" + std::to_string(1 + q), leaf[q]); e.body << "  mov.u32 %r" << 1 + q << ", " << t << ";\n"; }
      i = j;
    }
    const std::string fn = "zkb_u" + std::to_string(u);
    // prologue: the group's threads copy this unit's slice of the (term-ordered) power table into the group's staging area
    std::ostringstream stage;
    {
      const size_t nt = units[u].hi - units[u].lo;
      stage << "  {\n  .reg .pred %pz;\n  .reg .b32 %zi, %za, %zw<4>;\n  .reg .b64 %zg;\n  bar.sync %r5, " << points << ";\n";       // everybody is done with the previous unit's slice
      for (size_t base = 0; base < nt; base += points) {
        stage << "  add.u32 %zi, %r7, " << base << ";\n  setp.lt.u32 %pz, %zi, " << nt << ";\n  mul.wide.u32 %zg, %zi, 16;\n  add.u64 %zg, %zg, %rd1;\n"
              << "  @%pz ld.global.nc.v4.u32 {%zw0, %zw1, %zw2, %zw3}, [%zg+" << 16 * units[u].lo << "];\n  shl.b32 %za, %zi, 4;\n  add.u32 %za, %za, %r6;\n"
              << "  @%pz st.shared.v4.u32 [%za], {%zw0, %zw1, %zw2, %zw3};\n";
      }
      stage << "  bar.sync %r5, " << points << ";\n  }\n";
    }
    mod << ".visible .func  (.param .align 16 .b8 func_retval0[16]) " << fn << "(\n  .param .b64 " << fn << "_param_0,\n  .param .b64 " << fn << "_param_1,\n  .param .b64 "
        << fn << "_param_2,\n  .param .b32 " << fn << "_param_3,\n  .param .b32 " << fn << "_param_4,\n  .param .b32 " << fn << "_param_5,\n  .param .b32 " << fn << "_param_6\n)\n{\n  .reg .b32 %r<" << e.nr << ">;\n  .reg .b64 %rd<" << e.nd << ">;\n"
        << "  ld.param.u64 %rd0, [" << fn << "_param_0]; cvta.to.shared.u64 %rd0, %rd0;\n  ld.param.u64 %rd1, [" << fn << "_param_1]; cvta.to.global.u64 %rd1, %rd1;\n"
        << "  ld.param.u64 %rd2, [" << fn << "_param_2]; cvta.to.global.u64 %rd2, %rd2;\n  ld.param.u32 %r0, [" << fn << "_param_3];\n  ld.param.u32 %r5, [" << fn << "_param_4];\n"
        << "  ld.param.u32 %r6, [" << fn << "_param_5];\n  ld.param.u32 %r7, [" << fn << "_param_6];\n"
        << "  mov.u32 %r1, 0; mov.u32 %r2, 0; mov.u32 %r3, 0; mov.u32 %r4, 0;\n" << stage.str() << e.body.str()
        << "  st.param.v4.b32 [func_retval0], {%r1, %r2, %r3, %r4};\n  ret;\n}\n\n";
    if ((u + 1) % per_module == 0 || u + 1 == units.size()) { prog.unit_ptx.push_back(mod.str()); begin_module(); }
  }
  // ---- the kernel, as CUDA C++ ---------------------------------------------------------------------------------------------
  std::ostringstream o;
  o << "#define ZKB_ALU_ADDS " << (env_u32("ZKB_EC_ALU_ADDS", 1, 0, 1) ? 1 : 0) << "\n" << PREAMBLE;
  o << "#define HALO " << halo << "u\n#define BLOCK " << points << "u\n#define ROWP " << rowp << "u\n" << PREAMBLE_STAGED;
  for (size_t u = 0; u < units.size(); ++u) o << "extern \"C\" __device__ uint4 zkb_u" << u << "(const u32* sp, const uint4* pw, const u32* gl, u32 ones, u32 bar, u32 pwsm, u32 pt);\n";
  o << "#define UNIT(k) { const uint4 q = zkb_u##k(sp, pw, gl, zkb_ones, grp + 1u, pwsm, pt); ra = add(ra, q.x); rb = add(rb, q.y); rc = add(rc, q.z); rd = add(rd, q.w); }\n";
  o << "extern \"C\" __global__ void __launch_bounds__(" << gi.block << ", 1) zkb_ec(u32* __restrict__ check, const u32* __restrict__ g0, const u32* __restrict__ g1, "
       "const u32* __restrict__ g2, const uint4* __restrict__ pw, const u32* __restrict__ gl, uint4 invden, u32 mask) {\n"
       "  size_t dom; asm(\"add.u64 %0, %1, 1;\" : \"=l\"(dom) : \"l\"((u64)mask));\n"
       "  extern __shared__ __align__(128) u32 zkb_sm[];\n"
       "  u32* const part = zkb_sm + " << col_words << "u;\n"
       "  u32* const pwst = part + " << (size_t)(groups - 1) * points * 4 << "u;          // per warp group: the running unit's poly_mix powers\n"
       "  u64* const full = reinterpret_cast<u64*>(pwst + " << pw_words << "u);\n"
       "  const u32 c0 = blockIdx.x * BLOCK, pt = threadIdx.x % BLOCK, grp = threadIdx.x / BLOCK;\n"
       "  const u32 pwsm = saddr(pwst + grp * " << (size_t)unit_terms * 4 << "u);\n"
       "  if (threadIdx.x == 0) { mbar_init(full, 1u); asm volatile(\"fence.mbarrier_init.release.cluster;\" ::: \"memory\"); }\n  __syncthreads();\n"
       "  if (threadIdx.x == 0) {\n    mbar_expect_tx(full, " << col_words * 4 << "u);\n";
  for (auto& kv : slot) o << "    copy_col(zkb_sm + " << (size_t)kv.second * rowp << "u, g" << kv.first.first << " + (size_t)" << kv.first.second << " * dom, c0, mask, full);\n";
  o << "  }\n  mbar_wait(full, 0u);\n  const u32* const sp = zkb_sm + pt + HALO;\n  u32 ra = 0u, rb = 0u, rc = 0u, rd = 0u;\n  switch (grp) {\n";
  for (uint32_t g = 0; g < groups; ++g) {
    o << "    case " << g << ":\n";
    for (size_t u = g; u < units.size(); u += groups) o << "      UNIT(" << u << ")\n";
    o << "      break;\n";
  }
  o << "  }\n";
  if (groups > 1) o << "  if (grp) { uint4* q = reinterpret_cast<uint4*>(part) + (grp - 1u) * BLOCK + pt; *q = make_uint4(ra, rb, rc, rd); }\n  __syncthreads();\n  if (grp) return;\n"
                       "  for (u32 g = 0; g < " << groups - 1 << "u; ++g) { const uint4 q = reinterpret_cast<const uint4*>(part)[g * BLOCK + pt]; ra = add(ra, q.x); rb = add(rb, q.y); rc = add(rc, q.z); rd = add(rd, q.w); }\n";
  o << "  const u32 c = c0 + pt;\n"
       "  const u32 den = (c & 3u) == 0 ? invden.x : (c & 3u) == 1 ? invden.y : (c & 3u) == 2 ? invden.z : invden.w;\n"
       "  st(check + c, mul(ra, den)); st(check + dom + c, mul(rb, den)); st(check + 2 * dom + c, mul(rc, den)); st(check + 3 * dom + c, mul(rd, den));\n}\n";
  prog.main_cu = o.str();
  prog.threads = gi.block;
  return true;
}
// ---- compact form: the flat form with the PROGRAM AS DATA ---------------------------------------------------------------------
// ncu on the PTX flat form (profiles/r2_f_heavy_ec_ncu.txt): 8.6 of 12.2 cycles per issued instruction are "no instruction" stalls --
// 9 MB of straight-line code pass through the instruction caches once per 128-point tile and each warp waits for every line; only
// 4 warps per scheduler fit next to the 161 KB tile, so the latency is not hidden.  But the 20 k terms of a real constraint system
// have very few SHAPES (SYN-HEAVY: a - (x + k y) with and without a global; rv32im: a few hundred patterns repeated per instruction
// class).  Here each distinct expression shape is compiled ONCE as a loop body and the terms become operand records
// (shared-memory offsets of the taps, constants, global indices) in a read-only table: the instruction stream is a few KB and stays
// in the L0 / L1.5 instruction caches; per unit a warp group stages its slice of the operand table and of the poly_mix powers in
// shared memory (uniform, broadcast loads).  Terms of a group are sorted by shape, so a group is a handful of runs.
//   record layout (uint4 granules): unit = [n_groups,0,0,0] groups...; group = [n_conds, n_runs, 0, 0] [cond tap offsets...]
//   runs...; run = [shape, count, 0, 0] terms...; term = ceil(leaves / 4) granules of operands in depth-first order.
// Applies when every AndCond condition is a plain tap and no expression has more than 16 leaves; otherwise the PTX flat form is used.
struct CompactShape { std::string expr; uint32_t leaves = 0; };
static bool generate_compact_ppt(const CircuitDef& c, GenInfo& gi, std::string& src, const uint32_t ppt) {
  const size_t n = c.steps.size();
  std::vector<size_t> fp_step(c.n_fp_vars), mx_step(c.n_mix_vars);
  { uint32_t fi = 0, mi = 0; for (size_t i = 0; i < n; ++i) { if (c.steps[i].op <= PX_MUL) fp_step[fi++] = i; else mx_step[mi++] = i; } }
  std::vector<uint32_t> mpow(c.n_mix_vars, 0);
  for (uint32_t m = 0; m < c.n_mix_vars; ++m) {
    const StepDef& s = c.steps[mx_step[m]];
    if (s.op == PX_AND_EQZ) mpow[m] = mpow[s.a] + 1; else if (s.op == PX_AND_COND) mpow[m] = mpow[s.a] + mpow[s.c];
  }
  std::vector<std::vector<uint32_t>> cls(1);
  std::map<std::vector<uint32_t>, uint32_t> cl_id{{{}, 0u}};
  struct Term { uint32_t power, cl, value, shape; std::vector<uint32_t> ops; };
  std::vector<Term> terms;
  struct Item { uint32_t m, off, cl; };
  std::vector<Item> stack{{c.ret, 0u, 0u}};
  while (!stack.empty()) {
    Item it = stack.back(); stack.pop_back();
    for (;;) {
      const StepDef& s = c.steps[mx_step[it.m]];
      if (s.op == PX_TRUE) break;
      if (s.op == PX_AND_EQZ) { terms.push_back({it.off + mpow[s.a], it.cl, s.b, 0, {}}); it.m = s.a; continue; }
      if (c.steps[fp_step[s.b]].op != PX_GET) return false;               // conditions must be plain taps
      std::vector<uint32_t> inner = cls[it.cl]; inner.push_back(s.b);
      auto f = cl_id.find(inner);
      uint32_t id;
      if (f == cl_id.end()) { id = (uint32_t)cls.size(); cl_id.emplace(inner, id); cls.push_back(inner); } else id = f->second;
      stack.push_back({s.c, it.off + mpow[s.a], id});
      it.m = s.a;
    }
  }
  if (terms.empty()) return false;
  // columns
  std::map<std::pair<uint32_t, uint32_t>, uint32_t> slot;
  uint32_t halo = 0;
  for (const TapDef& t : c.taps) { slot.emplace(std::make_pair(t.group, t.column), 0u); halo = std::max(halo, 4 * t.back); }
  { uint32_t k = 0; for (auto& kv : slot) kv.second = k++; }
  // points per thread: with 2, a thread evaluates rows pt and pt + T of the tile (T = threads per warp group): one operand record, one
  // power load and one tap-address addition serve two points (the second tap is the same LDS with an immediate offset), and there are
  // twice as many independent chains per warp.  The block keeps 512 threads as 8 groups of 64, with correspondingly smaller units.
  // Measured on SYN-HEAVY (profiles/r2_v_ec_ppt_sweep.txt): 135.4 ms with one point per thread (main loop of 8 terms), 123.6 ms with two
  // (pairs of terms); ZKB_EC_PPT=1 restores the former.
  const uint32_t groups = env_u32("ZKB_EC_FLAT_GROUPS", ppt == 2 ? 8 : 4, 1, 15);      // (named barriers 1..15)
  const uint32_t unit_terms = env_u32("ZKB_EC_UNIT", ppt == 2 ? 96 : 256, 8, 512);
  const uint32_t unit_vecs = env_u32("ZKB_EC_UNIT_VECS", ppt == 2 ? 240 : 640, 64, 4096);          // operand-table granules (16 B) a unit may use
  uint32_t points = env_u32("ZKB_EC_FLAT_POINTS", 128, 32, 512);
  const size_t stage_words = (size_t)groups * ((size_t)unit_terms + unit_vecs) * 4;
  while (points > 32 && ((size_t)slot.size() * (points + halo) * 4 + (size_t)(groups - 1) * points * 16 + stage_words * 4 + 64 > 220 * 1024)) points >>= 1;
  const uint32_t rowp = points + halo;
  const size_t col_words = (size_t)slot.size() * rowp;
  gi.smem = col_words * 4 + (size_t)(groups - 1) * points * 16 + stage_words * 4 + 16;
  if (gi.smem > 220 * 1024 || (halo & 3)) return false;
  // BYTE offset of a tap from the thread's row in column slot 0: the load is then one add + LDS (word offsets cost IMAD.IADD + LEA + LDS)
  auto tap_off = [&](const TapDef& t) { return (uint32_t)(int32_t)(4 * ((long)slot[{t.group, t.column}] * rowp - 4 * (long)t.back)); };
  // shapes
  std::map<std::string, uint32_t> shape_id;
  std::vector<CompactShape> shapes;
  bool too_big = false;
  std::function<std::string(uint32_t, std::vector<uint32_t>&)> walk = [&](uint32_t f, std::vector<uint32_t>& ops) -> std::string {
    const StepDef& s = c.steps[fp_step[f]];
    if (ops.size() > 16) { too_big = true; return "0u"; }
    const std::string leaf = "L(" + std::to_string(ops.size()) + ")";
    switch (s.op) {
      case PX_CONST: ops.push_back(Fp::from(s.a).v); return leaf;
      case PX_GET: ops.push_back(tap_off(c.taps[s.a])); return "TAP(" + leaf + ")";
      case PX_GET_GLOBAL: ops.push_back(s.a == 0 ? s.b : c.mix_size + s.b); return "GL(" + leaf + ")";
      default: break;
    }
    std::string x = walk(s.a, ops), y = walk(s.b, ops);
    return std::string(s.op == PX_ADD ? "add(" : s.op == PX_SUB ? "sub(" : "mul(") + x + ", " + y + ")";
  };
  for (Term& t : terms) {
    std::string e = walk(t.value, t.ops);
    if (too_big || t.ops.size() > 16) return false;
    auto f = shape_id.find(e);
    if (f == shape_id.end()) { f = shape_id.emplace(e, (uint32_t)shapes.size()).first; shapes.push_back({e, (uint32_t)t.ops.size()}); }
    t.shape = f->second;
  }
  if (shapes.size() > env_u32("ZKB_EC_MAX_SHAPES", 512, 1, 1u << 20)) return false;
  std::stable_sort(terms.begin(), terms.end(), [](const Term& x, const Term& y) { return x.cl != y.cl ? x.cl < y.cl : x.shape != y.shape ? x.shape < y.shape : x.power < y.power; });
  gi.n_powers = (uint32_t)terms.size();
  gi.term_power.resize(terms.size());
  for (size_t t = 0; t < terms.size(); ++t) gi.term_power[t] = terms[t].power;
  const uint32_t tpg = points / ppt;                       // threads per warp group
  if (tpg % 32) return false;
  gi.block = (int)(tpg * groups); gi.points = (int)points; gi.staged = true;
  // the operand table, unit by unit
  std::vector<uint32_t> prog;                              // granules of 4 words
  struct UnitRec { uint32_t off, vecs, term0, nterms; };
  std::vector<UnitRec> urecs;
  auto vecs_of = [&](uint32_t leaves) { return std::max<uint32_t>(1, (leaves + 3) / 4); };
  for (size_t i = 0; i < terms.size();) {
    UnitRec u{(uint32_t)(prog.size() / 4), 0, (uint32_t)i, 0};
    const size_t hdr = prog.size(); prog.insert(prog.end(), {0u, 0u, 0u, 0u});
    uint32_t n_groups = 0;
    while (i < terms.size()) {
      // one (possibly partial) group: as many of its terms as still fit the unit
      const std::vector<uint32_t>& cl = cls[terms[i].cl];
      const uint32_t ghdr_vecs = 1 + (uint32_t)((cl.size() + 3) / 4);
      size_t j = i; uint32_t used = (uint32_t)((prog.size() - hdr) / 4) + ghdr_vecs; uint32_t cur_shape = ~0u;
      while (j < terms.size() && terms[j].cl == terms[i].cl) {
        uint32_t need = vecs_of(shapes[terms[j].shape].leaves) + (terms[j].shape != cur_shape ? 1u : 0u);
        if (used + need > unit_vecs || (j - u.term0) >= unit_terms) break;
        used += need; cur_shape = terms[j].shape; ++j;
      }
      if (j == i) { if (n_groups == 0) return false; break; }          // (a single term larger than a unit cannot happen with the limits above)
      const size_t gh = prog.size();
      prog.insert(prog.end(), {(uint32_t)cl.size(), 0u, 0u, 0u});
      for (size_t q = 0; q < (cl.size() + 3) / 4 * 4; ++q) prog.push_back(q < cl.size() ? tap_off(c.taps[c.steps[fp_step[cl[q]]].a]) : 0u);
      uint32_t n_runs = 0;
      for (size_t k = i; k < j;) {
        size_t e = k; while (e < j && terms[e].shape == terms[k].shape) ++e;
        prog.insert(prog.end(), {terms[k].shape, (uint32_t)(e - k), 0u, 0u}); ++n_runs;
        for (size_t q = k; q < e; ++q) { const uint32_t v = vecs_of(shapes[terms[q].shape].leaves); for (uint32_t w = 0; w < 4 * v; ++w) prog.push_back(w < terms[q].ops.size() ? terms[q].ops[w] : 0u); }
        k = e;
      }
      prog[gh + 1] = n_runs;
      ++n_groups; i = j;
      if ((uint32_t)((prog.size() - hdr) / 4) + 3 > unit_vecs || (i - u.term0) >= unit_terms) break;
    }
    prog[hdr] = n_groups;
    u.vecs = (uint32_t)(prog.size() / 4) - u.off; u.nterms = (uint32_t)(i - u.term0);
    urecs.push_back(u);
  }
  // ---- source -----------------------------------------------------------------------------------------------------------------
  std::ostringstream o;
  o << "#define ZKB_ALU_ADDS " << (env_u32("ZKB_EC_ALU_ADDS", 1, 0, 1) ? 1 : 0) << "\n" << PREAMBLE;
  o << "#define HALO " << halo << "u\n#define BLOCK " << points << "u\n#define ROWP " << rowp << "u\n" << PREAMBLE_STAGED;
  o << "typedef u64 ACC;\n#define GL(i) __ldg(gl + (i))\n";
  // ZKB_EC_PURE_LOADS=1: record / power loads are plain (schedulable) asm; they cannot be hoisted over the staging barrier or merged
  // across units because their base addresses are OUTPUTS of the volatile barrier statement.  0 (default): volatile loads in program
  // order -- measured equal (profiles/r2_s_ec_compact_sweep.txt), and ptxas spends fewer IMAD.MOV on it.
  const bool pure_loads = env_u32("ZKB_EC_PURE_LOADS", 0, 0, 1) != 0;
  o << "#define LDR_VOL " << (pure_loads ? "" : "volatile") << "\n";
  // operand records, powers and taps are read through 32-bit shared-window addresses (no 64-bit pointer arithmetic: IMAD.X / IADD3.X);
  // the record / power loads are volatile because their staging area is rewritten per unit (a pure asm would be CSE'd across units);
  // a tap address is spb + offset as min(a + b, ONES): one ALU-pipe VIADDMNMX instead of an IMAD.IADD on the multiplier pipe
  o << "__device__ __forceinline__ u32 lds32(u32 a) { u32 v; asm(\"ld.shared.u32 %0, [%1];\" : \"=r\"(v) : \"r\"(a)); return v; }\n"
       "__device__ __forceinline__ u32 ldr32(u32 a) { u32 v; asm LDR_VOL(\"ld.shared.u32 %0, [%1];\" : \"=r\"(v) : \"r\"(a)); return v; }\n"
       "__device__ __forceinline__ uint4 ldr128(u32 a) { uint4 v; asm LDR_VOL(\"ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];\" : \"=r\"(v.x), \"=r\"(v.y), \"=r\"(v.z), \"=r\"(v.w) : \"r\"(a)); return v; }\n"
       "#define TAP(o) lds32(ADD2(spb, (o)))\n";
  if (ppt == 2) o << "__device__ __forceinline__ u32 lds32b(u32 a) { u32 v; asm(\"ld.shared.u32 %0, [%1+" << 4 * tpg << "];\" : \"=r\"(v) : \"r\"(a)); return v; }\n"
                     "#define TAPB(o) lds32b(ADD2(spb, (o)))\n";
  o << "#define FIX4 { A0 = fixhi(A0); A1 = fixhi(A1); A2 = fixhi(A2); A3 = fixhi(A3); " << (ppt == 2 ? "B0 = fixhi(B0); B1 = fixhi(B1); B2 = fixhi(B2); B3 = fixhi(B3); " : "") << "}\n";
  o << "#define L(i) ((i) < 4 ? (&a0.x)[(i)] : (i) < 8 ? (&a1.x)[(i) - 4] : (i) < 12 ? (&a2.x)[(i) - 8] : (&a3.x)[(i) - 12])\n";
  o << "__device__ const uint4 zkb_units[" << urecs.size() << "] = {";
  for (const UnitRec& u : urecs) o << "{" << u.off << "u," << u.vecs << "u," << u.term0 << "u," << u.nterms << "u},";
  o << "};\n__device__ const uint4 zkb_prog[" << prog.size() / 4 << "] = {\n";
  for (size_t q = 0; q < prog.size(); q += 4) o << "{" << prog[q] << "u," << prog[q + 1] << "u," << prog[q + 2] << "u," << prog[q + 3] << "u}," << ((q / 4) % 8 == 7 ? "\n" : "");
  o << "};\n";
  o << "extern \"C\" __global__ void __launch_bounds__(" << gi.block << ", 1) zkb_ec(u32* __restrict__ check, const u32* __restrict__ g0, const u32* __restrict__ g1, "
       "const u32* __restrict__ g2, const uint4* __restrict__ pw, const u32* __restrict__ gl, uint4 invden, u32 mask) {\n"
       "  size_t dom; asm(\"add.u64 %0, %1, 1;\" : \"=l\"(dom) : \"l\"((u64)mask));\n"
       "  extern __shared__ __align__(128) u32 zkb_sm[];\n"
       "  u32* const part = zkb_sm + " << col_words << "u;\n"
       "  uint4* const stage = reinterpret_cast<uint4*>(part + " << (size_t)(groups - 1) * points * 4 << "u);\n"
       "  u64* const full = reinterpret_cast<u64*>(part + " << (size_t)(groups - 1) * points * 4 + stage_words << "u);\n"
       "  const u32 c0 = blockIdx.x * BLOCK, pt = threadIdx.x % " << tpg << "u, grp = threadIdx.x / " << tpg << "u;\n"
       "  uint4* const dsm = stage + grp * " << (unit_terms + unit_vecs) << "u;      // this warp group's operand records ...\n"
       "  uint4* const wsm = dsm + " << unit_vecs << "u;                              // ... and poly_mix powers of the unit it is running\n"
       "  if (threadIdx.x == 0) { mbar_init(full, 1u); asm volatile(\"fence.mbarrier_init.release.cluster;\" ::: \"memory\"); }\n  __syncthreads();\n"
       "  if (threadIdx.x == 0) {\n    mbar_expect_tx(full, " << col_words * 4 << "u);\n";
  for (auto& kv : slot) o << "    copy_col(zkb_sm + " << (size_t)kv.second * rowp << "u, g" << kv.first.first << " + (size_t)" << kv.first.second << " * dom, c0, mask, full);\n";
  const bool two = ppt == 2;
  o << "  }\n  mbar_wait(full, 0u);\n  const u32 spb = saddr(zkb_sm + pt + HALO);          // shared-window byte address of this thread's row in column slot 0\n"
       "  u32 ra = 0u, rb = 0u, rc = 0u, rd = 0u;\n" << (two ? "  u32 sa = 0u, sb = 0u, sc = 0u, sd = 0u;          // the second point (row pt + T)\n" : "")
    << "  for (u32 u = grp; u < " << urecs.size() << "u; u += " << groups << "u) {\n"
       "    const uint4 ur = zkb_units[u];\n"
       "    asm volatile(\"bar.sync %0, " << tpg << ";\" :: \"r\"(grp + 1u) : \"memory\");          // the group is done with the previous unit's records\n"
       "    for (u32 i = pt; i < ur.y; i += " << tpg << "u) dsm[i] = zkb_prog[ur.x + i];\n"
       "    for (u32 i = pt; i < ur.w; i += " << tpg << "u) wsm[i] = __ldg(pw + ur.z + i);\n"
       "    u32 d, w;          // defined by the barrier statement: loads through them stay behind it\n"
       "    asm volatile(\"bar.sync %2, " << tpg << "; mov.u32 %0, %3; mov.u32 %1, %4;\" : \"=r\"(d), \"=r\"(w) : \"r\"(grp + 1u), \"r\"(saddr(dsm)), \"r\"(saddr(wsm)) : \"memory\");\n"
       "    const u32 n_groups = ldr32(d); d += 16u;\n"
       "    for (u32 g = 0; g < n_groups; ++g) {\n"
       "      const uint4 gh = ldr128(d); d += 16u;\n"
       "      const u32 n_conds = gh.x, n_runs = gh.y;\n"
       "      u32 cp = 0u" << (two ? ", cq = 0u" : "") << ";\n"
       "      for (u32 q = 0; q < n_conds; ++q) { const u32 co = ldr32(d + 4u * q); const u32 cv = TAP(co); cp = q ? mul(cp, cv) : cv;"
    << (two ? " const u32 cw = TAPB(co); cq = q ? mul(cq, cw) : cw;" : "") << " }\n"
       "      d += ((n_conds + 3u) >> 2) << 4;\n"
       "      ACC A0 = 0, A1 = 0, A2 = 0, A3 = 0" << (two ? ", B0 = 0, B1 = 0, B2 = 0, B3 = 0" : "") << ";\n"
       "      for (u32 r = 0; r < n_runs; ++r) {\n"
       "        const uint4 rh = ldr128(d); d += 16u;\n"
       "        const u32 shape = rh.x, count = rh.y;\n"
       "        switch (shape) {\n";
  const uint32_t unroll = env_u32("ZKB_EC_UNROLL", two ? 2 : 8, 2, 8) & ~1u;          // terms per trip of a shape's main loop (even)
  for (size_t sidx = 0; sidx < shapes.size(); ++sidx) {
    const uint32_t v = vecs_of(shapes[sidx].leaves);
    // one term: operands -> value -> four unreduced accumulations; terms are taken in PAIRS with one high-word fix per pair (the accumulators
    // tolerate two products between fixes), an odd last term gets its own -- no per-term parity test, no predicated fixes
    std::string expr_b = shapes[sidx].expr;
    for (size_t at = 0; (at = expr_b.find("TAP(", at)) != std::string::npos; at += 5) expr_b.replace(at, 4, "TAPB(");
    std::ostringstream term;
    term << "{ const uint4 a0 = ldr128(d)";
    for (uint32_t q = 1; q < 4; ++q) term << ", a" << q << " = " << (q < v ? "ldr128(d + " + std::to_string(16 * q) + "u)" : std::string("a0"));
    term << "; d += " << 16 * v << "u; const u32 v = " << shapes[sidx].expr << "; " << (two ? "const u32 vb = " + expr_b + "; " : "")
         << "const uint4 m = ldr128(w); w += 16u; wacc(A0, v, m.x); wacc(A1, v, m.y); wacc(A2, v, m.z); wacc(A3, v, m.w); "
         << (two ? "wacc(B0, vb, m.x); wacc(B1, vb, m.y); wacc(B2, vb, m.z); wacc(B3, vb, m.w); " : "") << "}";
    const std::string pair = "              " + term.str() + "\n              " + term.str() + "\n              FIX4\n";
    o << "          case " << sidx << ": {\n            u32 i = 0;\n";
    if (unroll > 2) { o << "            for (; i + " << unroll << "u <= count; i += " << unroll << "u) {\n"; for (uint32_t q = 0; q < unroll; q += 2) o << pair; o << "            }\n"; }
    o << "            for (; i + 2u <= count; i += 2u) {\n" << pair << "            }\n            if (i < count) {\n              " << term.str() << "\n              FIX4\n            }\n          } break;\n";
  }
  o << "        }\n      }\n"
       "      { const u32 la = fin(A0), lb = fin(A1), lc = fin(A2), ld = fin(A3);\n"
       "        if (n_conds) { ra = add(ra, mul(la, cp)); rb = add(rb, mul(lb, cp)); rc = add(rc, mul(lc, cp)); rd = add(rd, mul(ld, cp)); }\n"
       "        else { ra = add(ra, la); rb = add(rb, lb); rc = add(rc, lc); rd = add(rd, ld); } }\n";
  if (two) o << "      { const u32 la = fin(B0), lb = fin(B1), lc = fin(B2), ld = fin(B3);\n"
                "        if (n_conds) { sa = add(sa, mul(la, cq)); sb = add(sb, mul(lb, cq)); sc = add(sc, mul(lc, cq)); sd = add(sd, mul(ld, cq)); }\n"
                "        else { sa = add(sa, la); sb = add(sb, lb); sc = add(sc, lc); sd = add(sd, ld); } }\n";
  o << "    }\n  }\n";
  if (groups > 1) {
    o << "  if (grp) { uint4* q = reinterpret_cast<uint4*>(part) + (grp - 1u) * BLOCK + pt; *q = make_uint4(ra, rb, rc, rd); " << (two ? "q[" + std::to_string(tpg) + "] = make_uint4(sa, sb, sc, sd); " : "") << "}\n"
         "  __syncthreads();\n  if (grp) return;\n"
         "  for (u32 g = 0; g < " << groups - 1 << "u; ++g) { const uint4* qp = reinterpret_cast<const uint4*>(part) + g * BLOCK + pt; const uint4 q = *qp; ra = add(ra, q.x); rb = add(rb, q.y); rc = add(rc, q.z); rd = add(rd, q.w); "
      << (two ? "const uint4 q2 = qp[" + std::to_string(tpg) + "]; sa = add(sa, q2.x); sb = add(sb, q2.y); sc = add(sc, q2.z); sd = add(sd, q2.w); " : "") << "}\n";
  }
  o << "  const u32 c = c0 + pt;\n"
       "  const u32 den = (c & 3u) == 0 ? invden.x : (c & 3u) == 1 ? invden.y : (c & 3u) == 2 ? invden.z : invden.w;          // (T is a multiple of 4: the same for both points)\n"
       "  st(check + c, mul(ra, den)); st(check + dom + c, mul(rb, den)); st(check + 2 * dom + c, mul(rc, den)); st(check + 3 * dom + c, mul(rd, den));\n";
  if (two) o << "  { const u32 c2 = c + " << tpg << "u; st(check + c2, mul(sa, den)); st(check + dom + c2, mul(sb, den)); st(check + 2 * dom + c2, mul(sc, den)); st(check + 3 * dom + c2, mul(sd, den)); }\n";
  o << "}\n";
  src = o.str();
  return true;
}
static bool generate_compact(const CircuitDef& c, GenInfo& gi, std::string& src) {
  const uint32_t ppt = env_u32("ZKB_EC_PPT", 2, 1, 2);
  if (ppt == 2) {
    GenInfo g2 = gi; std::string s2;
    if (generate_compact_ppt(c, g2, s2, 2)) { gi = g2; src.swap(s2); return true; }          // (a tile narrower than 64 points leaves less than a warp per group)
  }
  return generate_compact_ppt(c, gi, src, 1);
}
static bool compact_wanted() { const char* e = getenv("ZKB_EC_FORM"); return !(e && !strcmp(e, "flat")); }      // ZKB_EC_FORM=flat forces the PTX flat form

static std::string flat_text(const FlatProgram& p) { std::string t = p.main_cu; for (const std::string& u : p.unit_ptx) { t += "\n//----\n"; t += u; } return t; }

// ---- on-disk cubin cache -------------------------------------------------------------------------------------------------
// A cubin found on disk is code that will run inside the prover's CUDA context, next to the private witness, so the cache
// follows the rules of any per-user code cache (ADVICE r1):
//   * directory: ZKB_CACHE_DIR, else `_jitcache/` next to libzkb200.so when this user can write it (cubins compiled at build time
//     ship with the library), else $XDG_CACHE_HOME/zkb200 or ~/.cache/zkb200 created 0700.  Never a shared /tmp path; with no
//     usable directory the cache is memory-only.
//   * a directory or file is trusted only if it is owned by this uid (or root) and not writable by group / others;
//   * every file carries a header (magic, key = fnv1a64(source), a second hash over source + options + NVRTC version, payload size,
//     payload checksum), so stale or torn files are cache misses, not load errors;
//   * files are written to a mkstemp() name and renamed; compilation is serialised on a process-wide mutex (bench.py runs three
//     prover threads per process); a cubin that fails to LOAD is deleted and recompiled once.
static const char* const NVRTC_OPTS[] = {"--gpu-architecture=sm_100a", "--std=c++17", "-lineinfo", "--restrict"};
static bool trusted(const struct stat& st) { return (st.st_uid == geteuid() || st.st_uid == 0) && (st.st_mode & (S_IWGRP | S_IWOTH)) == 0; }
static bool usable_dir(const std::string& d, bool create) {
  if (create && mkdir(d.c_str(), 0700) != 0 && errno != EEXIST) return false;
  struct stat st;
  if (lstat(d.c_str(), &st) != 0 || !S_ISDIR(st.st_mode)) return false;
  return trusted(st);
}
static std::string cache_dir() {
  const char* e = getenv("ZKB_CACHE_DIR");
  if (e && *e) return usable_dir(e, true) ? std::string(e) : std::string();
  Dl_info info;
  if (dladdr((void*)&cache_dir, &info) && info.dli_fname) {
    std::string so = info.dli_fname;
    size_t slash = so.rfind('/');
    if (slash != std::string::npos) {
      std::string d = so.substr(0, slash) + "/_jitcache";
      if (usable_dir(d, access(so.substr(0, slash).c_str(), W_OK) == 0)) return d;     // read-only installs still use the shipped cubins
    }
  }
  std::string base;
  const char* x = getenv("XDG_CACHE_HOME"); const char* h = getenv("HOME");
  if (x && *x == '/') base = x; else if (h && *h == '/') { base = std::string(h) + "/.cache"; mkdir(base.c_str(), 0700); }
  if (base.empty()) return std::string();
  std::string d = base + "/zkb200";
  return usable_dir(d, true) ? d : std::string();
}
static int min_blocks() { const char* e = getenv("ZKB_EC_MINBLOCKS"); int v = e ? atoi(e) : 8; return v < 1 ? 1 : v > 16 ? 16 : v; }

struct CubinHeader { uint32_t magic; uint32_t version; uint64_t key; uint64_t key2; uint64_t size; uint64_t sum; };
static constexpr uint32_t CUBIN_MAGIC = 0x4a424b5au;      // "ZKBJ"
static uint64_t fnv1a_bytes(const char* p, size_t n, uint64_t h = 1469598103934665603ull) { for (size_t i = 0; i < n; ++i) { h ^= (unsigned char)p[i]; h *= 1099511628211ull; } return h; }
static uint64_t second_key(const std::string& src) {
  int maj = 0, min = 0; if (api().version) api().version(&maj, &min);
  std::string salt = "zkb200-jit-v2|nvrtc " + std::to_string(maj) + "." + std::to_string(min);
  for (const char* o : NVRTC_OPTS) { salt += '|'; salt += o; }
  if (const char* extra = getenv("ZKB_EC_NVRTC_EXTRA")) { salt += '|'; salt += extra; }
  uint64_t h = fnv1a_bytes(salt.data(), salt.size(), 0x9e3779b97f4a7c15ull);
  return fnv1a_bytes(src.data(), src.size(), h) ^ (uint64_t)src.size();
}
static std::string cubin_path(const std::string& dir, uint64_t key) {
  char name[64]; snprintf(name, sizeof name, "/ec_%016llx_sm100a.zkbj", (unsigned long long)key);
  return dir + name;
}
static bool cache_read(const std::string& path, uint64_t key, uint64_t key2, std::vector<char>& cubin) {
  int fd = open(path.c_str(), O_RDONLY | O_NOFOLLOW | O_CLOEXEC);
  if (fd < 0) return false;
  struct stat st; CubinHeader h;
  bool ok = fstat(fd, &st) == 0 && S_ISREG(st.st_mode) && trusted(st) && (size_t)st.st_size > sizeof h && read(fd, &h, sizeof h) == (ssize_t)sizeof h &&
            h.magic == CUBIN_MAGIC && h.version == 2 && h.key == key && h.key2 == key2 && h.size == (uint64_t)st.st_size - sizeof h;
  if (ok) {
    cubin.resize((size_t)h.size);
    size_t got = 0;
    while (got < cubin.size()) { ssize_t r = read(fd, cubin.data() + got, cubin.size() - got); if (r <= 0) break; got += (size_t)r; }
    ok = got == cubin.size() && fnv1a_bytes(cubin.data(), cubin.size()) == h.sum;
  }
  close(fd);
  if (!ok) cubin.clear();
  return ok;
}
static void cache_write(const std::string& dir, const std::string& path, uint64_t key, uint64_t key2, const std::vector<char>& cubin) {
  std::string tmpl = dir + "/.ec_tmp_XXXXXX";
  std::vector<char> tmp(tmpl.begin(), tmpl.end()); tmp.push_back('\0');
  int fd = mkstemp(tmp.data());          // unique per call (threads, processes, ranks), created 0600
  if (fd < 0) return;
  CubinHeader h{CUBIN_MAGIC, 2, key, key2, (uint64_t)cubin.size(), fnv1a_bytes(cubin.data(), cubin.size())};
  bool ok = write(fd, &h, sizeof h) == (ssize_t)sizeof h && write(fd, cubin.data(), cubin.size()) == (ssize_t)cubin.size();
  ok = (fchmod(fd, 0644) == 0) && ok;
  close(fd);
  if (!ok || rename(tmp.data(), path.c_str()) != 0) unlink(tmp.data());
}

static std::mutex g_compile_mutex;
static bool compile(const std::string& src, std::vector<char>& cubin, std::string& why, bool ignore_disk = false) {
  std::lock_guard<std::mutex> lock(g_compile_mutex);
  Api& a = api();
  const uint64_t key = fnv1a(src), key2 = second_key(src);
  const std::string dir = cache_dir();
  const std::string path = dir.empty() ? std::string() : cubin_path(dir, key);
  if (!path.empty()) {
    if (ignore_disk) unlink(path.c_str());
    else if (cache_read(path, key, key2, cubin)) return true;
  }
  nvrtcProgram prog;
  if (a.createProgram(&prog, src.c_str(), "zkb_eval_check.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) { why = "nvrtcCreateProgram failed"; return false; }
  std::vector<const char*> opts(NVRTC_OPTS, NVRTC_OPTS + sizeof NVRTC_OPTS / sizeof NVRTC_OPTS[0]);
  const char* extra = getenv("ZKB_EC_NVRTC_EXTRA");      // experiments only (e.g. --ptxas-options=-O1); part of the cache key through second_key()
  if (extra && *extra) opts.push_back(extra);
  nvrtcResult r = a.compileProgram(prog, (int)opts.size(), opts.data());
  if (r != NVRTC_SUCCESS) {
    size_t ls = 0; a.getLogSize(prog, &ls);
    std::string log(ls, '\0'); if (ls) a.getLog(prog, &log[0]);
    why = "nvrtc compile failed: " + log.substr(0, 600);
    a.destroyProgram(&prog);
    return false;
  }
  size_t sz = 0; a.getCUBINSize(prog, &sz);
  cubin.resize(sz); a.getCUBIN(prog, cubin.data());
  a.destroyProgram(&prog);
  if (!path.empty()) cache_write(dir, path, key, key2, cubin);
  return true;
}

// Flat form: NVRTC (-rdc) turns the kernel into PTX, nvJitLink compiles it together with the unit PTX modules into one cubin.
static bool compile_flat(const FlatProgram& prog, std::vector<char>& cubin, std::string& why, bool ignore_disk = false) {
  std::lock_guard<std::mutex> lock(g_compile_mutex);
  Api& a = api();
  if (!a.jl_ok) { why = a.jl_why.empty() ? "nvJitLink unavailable" : a.jl_why; return false; }
  const std::string text = flat_text(prog);
  const uint64_t key = fnv1a(text), key2 = second_key(text) ^ 0x666c6174ull;
  const std::string dir = cache_dir();
  const std::string path = dir.empty() ? std::string() : cubin_path(dir, key);
  if (!path.empty()) {
    if (ignore_disk) unlink(path.c_str());
    else if (cache_read(path, key, key2, cubin)) return true;
  }
  nvrtcProgram np;
  if (a.createProgram(&np, prog.main_cu.c_str(), "zkb_eval_check_flat.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) { why = "nvrtcCreateProgram failed"; return false; }
  const char* opts[] = {"--gpu-architecture=compute_100a", "--std=c++17", "-lineinfo", "--restrict", "-rdc=true"};
  nvrtcResult r = a.compileProgram(np, 5, opts);
  if (r != NVRTC_SUCCESS) {
    size_t ls = 0; a.getLogSize(np, &ls);
    std::string log(ls, '\0'); if (ls) a.getLog(np, &log[0]);
    why = "nvrtc compile (flat kernel) failed: " + log.substr(0, 600);
    a.destroyProgram(&np);
    return false;
  }
  size_t psz = 0; a.getPTXSize(np, &psz);
  std::string main_ptx(psz, '\0'); a.getPTX(np, &main_ptx[0]);
  a.destroyProgram(&np);
  // NVRTC and nvJitLink may come from different CUDA 12.x installs in one process (torch brings its own): an nvJitLink older than
  // NVRTC rejects the newer `.version`.  The kernel uses nothing beyond ISA 8.6 (the first with sm_100a), so declare that.
  { size_t v = main_ptx.find(".version "); if (v != std::string::npos) { size_t e = main_ptx.find('\n', v); main_ptx.replace(v, e - v, ".version 8.6"); } }
  nvJitLinkHandle h;
  // the units are separate functions: ptxas must be told the register budget the kernel's launch bounds imply
  const std::string maxreg = "-maxrregcount=" + std::to_string(std::min(255, (65536 / std::max(prog.threads, 32)) & ~7));
  // --split-compile=0: ptxas compiles the functions of a module on all host threads (2.2 x faster here with 8 threads)
  // (no -lineinfo: it embeds the 27 MB of unit PTX in the cubin as .nv_debug_ptx_txt sections)
  std::vector<const char*> lopts = {"-arch=sm_100a", maxreg.c_str(), "-Xptxas=--split-compile=0"};
  const char* jl_extra = getenv("ZKB_EC_JL_EXTRA");
  if (jl_extra && *jl_extra) lopts.push_back(jl_extra);
  const bool verbose = getenv("ZKB_EC_VERBOSE") != nullptr;       // ptxas -v (registers, spills, stack) of every unit to stderr
  if (verbose) { lopts.push_back("-verbose"); lopts.push_back("-Xptxas=-v"); }
  if (a.jlCreate(&h, (uint32_t)lopts.size(), lopts.data()) != NVJITLINK_SUCCESS) { why = "nvJitLinkCreate failed"; return false; }
  auto fail = [&](const char* what) {
    size_t ls = 0; std::string log;
    if (a.jlLogSize && a.jlLog && a.jlLogSize(h, &ls) == NVJITLINK_SUCCESS && ls) { log.resize(ls); a.jlLog(h, &log[0]); }
    why = std::string("nvJitLink ") + what + " failed: " + log.substr(0, 800);
    a.jlDestroy(&h);
    return false;
  };
  if (a.jlAddData(h, NVJITLINK_INPUT_PTX, main_ptx.c_str(), main_ptx.size(), "zkb_ec_kernel") != NVJITLINK_SUCCESS) return fail("add(kernel)");
  for (size_t i = 0; i < prog.unit_ptx.size(); ++i)
    if (a.jlAddData(h, NVJITLINK_INPUT_PTX, prog.unit_ptx[i].c_str(), prog.unit_ptx[i].size() + 1, ("zkb_units_" + std::to_string(i)).c_str()) != NVJITLINK_SUCCESS) return fail("add(units)");
  if (a.jlComplete(h) != NVJITLINK_SUCCESS) return fail("link");
  if (verbose && a.jlInfoSize && a.jlInfo) {
    size_t ls = 0;
    if (a.jlInfoSize(h, &ls) == NVJITLINK_SUCCESS && ls) { std::string log(ls, '\0'); a.jlInfo(h, &log[0]); fprintf(stderr, "%s\n", log.c_str()); }
  }
  size_t sz = 0;
  if (a.jlCubinSize(h, &sz) != NVJITLINK_SUCCESS) return fail("cubin size");
  cubin.resize(sz);
  if (a.jlCubin(h, cubin.data()) != NVJITLINK_SUCCESS) return fail("cubin");
  a.jlDestroy(&h);
  if (!path.empty()) cache_write(dir, path, key, key2, cubin);
  return true;
}

void eval_jit_free(zkb_ctx* ctx) {
  if (!ctx->jit) return;
  EvalJitCache* cache = (EvalJitCache*)ctx->jit;
  for (auto& kv : cache->kernels) if (kv.second.mod) api().moduleUnload(kv.second.mod);
  for (auto& kv : cache->accum) if (kv.second.mod) api().moduleUnload(kv.second.mod);
  delete cache;
  ctx->jit = nullptr;
}

// ---- CircuitHal::accumulate as data: the circuit blob's witness program, one straight-line kernel per phase --------------------
// (the counterpart of the reference's generated step_compute_accum; PrefixProduct phases are run by the caller in between)
struct AccumPhase { size_t lo, hi; };
static std::vector<AccumPhase> accum_phases(const CircuitDef& c) {
  std::vector<AccumPhase> ph;
  size_t lo = 0;
  for (size_t i = 0; i <= c.wsteps.size(); ++i)
    if (i == c.wsteps.size() || c.wsteps[i].op == WX_BARRIER || c.wsteps[i].op == WX_PREFIX_PRODUCT) { ph.push_back({lo, i}); lo = i + 1; }
  return ph;
}
std::string accumulate_jit_source(const CircuitDef& c) {
  std::ostringstream o;
  o << "#define ZKB_ALU_ADDS 1\n" << PREAMBLE;
  const std::vector<AccumPhase> ph = accum_phases(c);
  uint32_t val = 0;
  for (size_t k = 0; k < ph.size(); ++k) {
    o << "extern \"C\" __global__ void __launch_bounds__(256) zkb_acc_" << k << "(u32* __restrict__ accum, const u32* __restrict__ code, const u32* __restrict__ data, const u32* __restrict__ gl, u32 n) {\n"
         "  const u32 i = blockIdx.x * 256u + threadIdx.x;\n  if (i >= n) return;\n";
    for (size_t q = ph[k].lo; q < ph[k].hi; ++q) {
      const StepDef& s = c.wsteps[q];
      switch (s.op) {
        case WX_CONST: o << "  const u32 w" << val++ << " = " << Fp::from(s.a).v << "u;\n"; break;
        case WX_GET: {
          // a phase never reads an accum column it writes (checked by the parser): plain loads for accum, the read-only path for code / data
          std::ostringstream idx; idx << "(size_t)" << s.b << " * n + ((i - " << s.c << "u) & (n - 1u))";
          if (s.a == GROUP_ACCUM) o << "  const u32 w" << val++ << " = accum[" << idx.str() << "];\n";
          else o << "  const u32 w" << val++ << " = __ldg(" << (s.a == GROUP_CODE ? "code" : "data") << " + " << idx.str() << ");\n";
          break;
        }
        case WX_GET_GLOBAL: o << "  const u32 w" << val++ << " = __ldg(gl + " << (s.a == 0 ? s.b : c.mix_size + s.b) << ");\n"; break;
        case WX_ADD: o << "  const u32 w" << val++ << " = add(w" << s.a << ", w" << s.b << ");\n"; break;
        case WX_SUB: o << "  const u32 w" << val++ << " = sub(w" << s.a << ", w" << s.b << ");\n"; break;
        case WX_MUL: o << "  const u32 w" << val++ << " = mul(w" << s.a << ", w" << s.b << ");\n"; break;
        case WX_SET:
          if (s.c == WX_ALWAYS) o << "  accum[(size_t)" << s.a << " * n + i] = w" << s.b << ";\n";
          else o << "  if (w" << s.c << " != 0u) accum[(size_t)" << s.a << " * n + i] = w" << s.b << ";\n";
          break;
        default: break;
      }
    }
    o << "}\n";
  }
  return o.str();
}
// Launches phase `k` kernels; returns false (with why) when the JIT toolchain is unavailable.
bool accumulate_jit(zkb_ctx* ctx, const CircuitDef& c, size_t phase, uint32_t* d_accum, const uint32_t* d_code, const uint32_t* d_data, const uint32_t* d_gl, uint32_t n, std::string& why) {
  Api& a = api();
  if (!a.ok) { why = a.why; return false; }
  if (!a.cu_ok) { why = a.cu_why; return false; }
  if (!ctx->jit) ctx->jit = new EvalJitCache();
  EvalJitCache* cache = (EvalJitCache*)ctx->jit;
  const std::string src = accumulate_jit_source(c);
  const uint64_t key = fnv1a(src);
  auto it = cache->accum.find(key);
  if (it == cache->accum.end()) {
    if (cache->failed.count(key)) { why = "previous JIT attempt failed"; return false; }
    std::vector<char> cubin;
    if (!compile(src, cubin, why)) { cache->failed[key] = true; return false; }
    ZKB_CUDA(cudaFree(0));
    AccumJitKernel k;
    CUresult r = a.moduleLoadData(&k.mod, cubin.data());
    if (r != CUDA_SUCCESS) { cubin.clear(); if (!compile(src, cubin, why, true)) { cache->failed[key] = true; return false; } r = a.moduleLoadData(&k.mod, cubin.data()); }
    const size_t n_ph = accum_phases(c).size();
    for (size_t q = 0; q < n_ph && r == CUDA_SUCCESS; ++q) { CUfunction f = nullptr; r = a.moduleGetFunction(&f, k.mod, ("zkb_acc_" + std::to_string(q)).c_str()); k.phases.push_back(f); }
    if (r != CUDA_SUCCESS) { const char* es = nullptr; a.getErrorString(r, &es); why = std::string("accumulate JIT load: ") + (es ? es : "?"); cache->failed[key] = true; return false; }
    it = cache->accum.emplace(key, k).first;
  }
  ZKB_REQUIRE(phase < it->second.phases.size(), "accumulate: phase out of range");
  void* args[] = {&d_accum, &d_code, &d_data, &d_gl, &n};
  CUresult r = a.launchKernel(it->second.phases[phase], (n + 255u) / 256u, 1, 1, 256, 1, 1, 0, (CUstream)ctx->stream, args, nullptr);
  if (r != CUDA_SUCCESS) { const char* es = nullptr; a.getErrorString(r, &es); throw Error(std::string("zkb200: accumulate JIT launch failed: ") + (es ? es : "?")); }
  launched(ctx);
  return true;
}

// The generated source (for tests / inspection) -- no device needed.
std::string eval_jit_source(const CircuitDef& c) {
  GenInfo gi;
  if (flat_wanted(c)) {
    std::string cs;
    if (compact_wanted() && generate_compact(c, gi, cs)) return cs;
    FlatProgram fp; if (generate_flat(c, gi, fp)) return flat_text(fp);
  }
  if (ec_staged()) { std::string src = generate(c, gi, true); if (!src.empty()) return src; }
  return generate(c, gi, false);
}
// Compiles the source with NVRTC without loading it (CPU-only check that the generator emits valid CUDA).
bool eval_jit_compile_only(const CircuitDef& c, std::string& why) {
  Api& a = api();
  if (!a.ok) { why = a.why; return false; }
  std::vector<char> cubin; GenInfo gi;
  if (!c.wsteps.empty() && !compile(accumulate_jit_source(c), cubin, why)) return false;      // the witness program's phase kernels
  // heavy circuits: the flat form only (the straight-line forms of a 10^5-step program take ptxas tens of minutes and spill)
  if (flat_wanted(c)) {
    std::string cs;
    if (compact_wanted() && generate_compact(c, gi, cs)) return compile(cs, cubin, why);
    FlatProgram fp; if (generate_flat(c, gi, fp)) return compile_flat(fp, cubin, why);
  }
  // every form a proof may use: the staged kernel, and the register form used for tiny domains / unaligned sub-buffers
  if (ec_staged()) { std::string src = generate(c, gi, true); if (!src.empty() && !compile(src, cubin, why)) return false; }
  return compile(generate(c, gi, false), cubin, why);
}

static const EvalJitKernel* get_kernel(zkb_ctx* ctx, const CircuitDef& c, bool staged, std::string& why, bool flat = false) {
  Api& a = api();
  if (!a.ok) { why = a.why; return nullptr; }
  if (!a.cu_ok) { why = a.cu_why; return nullptr; }
  if (!ctx->jit) ctx->jit = new EvalJitCache();
  EvalJitCache* cache = (EvalJitCache*)ctx->jit;
  GenInfo gi;
  FlatProgram fprog;
  std::string src;
  bool ptx_flat = false;      // the PTX flat form goes through nvJitLink; everything else is one NVRTC program
  if (flat) {
    if (!(compact_wanted() && generate_compact(c, gi, src))) { src.clear(); if (generate_flat(c, gi, fprog)) { src = flat_text(fprog); ptx_flat = true; } }
  } else src = generate(c, gi, staged);
  if (src.empty()) { why = flat ? "circuit does not fit the flat form" : "circuit does not fit the staged form"; return nullptr; }
  const uint32_t np = gi.n_powers;
  uint64_t key = fnv1a(src);
  auto it = cache->kernels.find(key);
  if (it != cache->kernels.end()) return &it->second;
  if (cache->failed.count(key)) { why = "previous JIT attempt failed"; return nullptr; }
  std::vector<char> cubin;
  EvalJitKernel k; k.n_powers = np; k.block = gi.block; k.smem = gi.smem; k.points = gi.points ? gi.points : gi.block; k.term_power = gi.term_power;
  if (!(ptx_flat ? compile_flat(fprog, cubin, why) : compile(src, cubin, why))) { cache->failed[key] = true; return nullptr; }
  ZKB_CUDA(cudaFree(0));     // make sure the primary context is current for the driver API
  CUresult r = a.moduleLoadData(&k.mod, cubin.data());
  if (r != CUDA_SUCCESS) {      // a cached cubin that does not load (other driver, damaged file) is a cache miss: drop it, recompile once
    cubin.clear();
    if (!(ptx_flat ? compile_flat(fprog, cubin, why, /*ignore_disk=*/true) : compile(src, cubin, why, /*ignore_disk=*/true))) { cache->failed[key] = true; return nullptr; }
    r = a.moduleLoadData(&k.mod, cubin.data());
  }
  if (r == CUDA_SUCCESS) r = a.moduleGetFunction(&k.fn, k.mod, "zkb_ec");
  if (r == CUDA_SUCCESS && k.smem > 48 * 1024) r = a.funcSetAttribute(k.fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int)k.smem);
  if (r != CUDA_SUCCESS) { const char* s = nullptr; a.getErrorString(r, &s); why = std::string("cuModuleLoadData: ") + (s ? s : "?"); cache->failed[key] = true; return nullptr; }
  if (!flat && const_mode(c, np)) {
    r = a.moduleGetGlobal(&k.cdata, &k.cdata_bytes, k.mod, "zkb_cd");
    if (r != CUDA_SUCCESS) { const char* s = nullptr; a.getErrorString(r, &s); why = std::string("cuModuleGetGlobal(zkb_cd): ") + (s ? s : "?"); cache->failed[key] = true; return nullptr; }
  }
  return &(cache->kernels[key] = k);
}

// Returns false (with `why`) when the JIT path is unavailable; the caller then uses the interpreter.
bool eval_check_jit(zkb_ctx* ctx, uint32_t* d_check, const CircuitDef& c, const uint32_t* const d_groups[3], const uint32_t* mix_g, const uint32_t* out_g,
                    const Fp4& poly_mix, int po2, std::string& why) {
  const size_t n = (size_t)1 << po2, domain = n * INV_RATE;
  if (domain < (size_t)JIT_BLOCK) { why = "domain smaller than one block"; return false; }
  bool aligned = ((uintptr_t)d_check & 15) == 0;
  for (int g = 0; g < 3; ++g) if ((uintptr_t)d_groups[g] & 15) aligned = false;
  const EvalJitKernel* k = nullptr;
  if (flat_wanted(c)) {      // heavy circuit: flat form or nothing (the interpreter is the fallback, not a ten-minute compile)
    // the flat / compact forms stage columns with 16-byte copies; an unaligned sub-buffer view goes to the interpreter
    if (!aligned) { why = "heavy circuit on a buffer that is not 16-byte aligned"; return false; }
    k = get_kernel(ctx, c, false, why, true);
    if (k && domain < (size_t)k->points) { why = "domain smaller than one flat tile"; return false; }
    if (!k) return false;
  }
  if (!k && ec_staged() && aligned && domain >= (size_t)SG_BLOCK) {       // bulk copies need 16-byte aligned columns (pool allocations are; a caller's sub-buffer view may not be)
    std::string why_staged;
    k = get_kernel(ctx, c, true, why_staged);
  }
  if (!k) k = get_kernel(ctx, c, false, why);
  if (!k) return false;
  // per-proof data: [powers of poly_mix (4 words each)] [mix globals] [out globals]
  std::vector<uint32_t> h(4 * (size_t)k->n_powers + c.mix_size + c.out_size + 4);
  Fp4 cur = Fp4::one();
  if (k->term_power.empty()) {
    for (uint32_t i = 0; i < k->n_powers; ++i) { cur.store(&h[4 * i]); cur *= poly_mix; }
  } else {      // flat form: powers gathered into term order
    uint32_t maxp = 0;
    for (uint32_t pw_ : k->term_power) maxp = std::max(maxp, pw_);
    std::vector<Fp4> pows(maxp + 1);
    for (uint32_t i = 0; i <= maxp; ++i) { pows[i] = cur; cur *= poly_mix; }
    for (size_t t = 0; t < k->term_power.size(); ++t) pows[k->term_power[t]].store(&h[4 * t]);
  }
  uint32_t* gl = h.data() + 4 * (size_t)k->n_powers;
  for (uint32_t i = 0; i < c.mix_size; ++i) gl[i] = mix_g[i];
  for (uint32_t i = 0; i < c.out_size; ++i) gl[c.mix_size + i] = out_g[i];
  uint32_t* d_data = nullptr;
  const size_t data_words = 4 * (size_t)k->n_powers + c.mix_size + c.out_size;
  if (k->cdata) {
    ZKB_REQUIRE(data_words * 4 <= k->cdata_bytes, "eval_check JIT: constant bank smaller than the per-proof data");
    CUresult cr = api().memcpyHtoDAsync(k->cdata, h.data(), data_words * 4, (CUstream)ctx->stream);    // pageable source: staged before the call returns
    if (cr != CUDA_SUCCESS) { const char* s = nullptr; api().getErrorString(cr, &s); throw Error(std::string("zkb200: eval_check JIT constant upload failed: ") + (s ? s : "?")); }
  } else {
    pool_alloc(ctx, &d_data, h.size() * 4);
    ZKB_CUDA(cudaMemcpyAsync(d_data, h.data(), h.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
  }
  Fp w4 = pow(Fp::from(137), (uint64_t)1 << (MAX_ROU_PO2 - 2));
  Fp three_n = pow(Fp::from(3), n);
  uint4 invden; uint32_t* idp = &invden.x;
  Fp wr = Fp::one();
  for (int r = 0; r < 4; ++r) { idp[r] = inv(three_n * wr - Fp::one()).v; wr *= w4; }
  const uint32_t* g0 = d_groups[0]; const uint32_t* g1 = d_groups[1]; const uint32_t* g2 = d_groups[2];
  const uint4* pw = (const uint4*)d_data; const uint32_t* d_gl = d_data + 4 * (size_t)k->n_powers;
  uint32_t mask = (uint32_t)(domain - 1);
  void* args[] = {&d_check, &g0, &g1, &g2, &pw, &d_gl, &invden, &mask};
  CUresult r = api().launchKernel(k->fn, (unsigned)(domain / (size_t)(k->points ? k->points : k->block)), 1, 1, (unsigned)k->block, 1, 1, (unsigned)k->smem, (CUstream)ctx->stream, args, nullptr);
  if (r != CUDA_SUCCESS) { const char* s = nullptr; api().getErrorString(r, &s); throw Error(std::string("zkb200: eval_check JIT launch failed: ") + (s ? s : "?")); }
  launched(ctx);
  if (d_data) pool_free(ctx, d_data);
  return true;
}

}  // namespace zkb
