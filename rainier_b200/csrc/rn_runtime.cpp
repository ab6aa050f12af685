// rn_runtime.cpp -- librainier_cuda.so: the C ABI of include/rainier_cuda.h.
//
// rn_model   : parses the RIR, owns the device copy of the data columns and the NVRTC-compiled modules
//              (one per emit configuration); replaces Compiler.compileTargets + ir.CompiledFunction.
// rn_sampler : owns per-chain device state and drives the fused kernels; replaces Driver.sample for a whole
//              batch of chains (rainier-sampler/.../sampler/Driver.scala:7-119).
// No CPU fallback: anything that needs to execute fails with RN_E_CUDA when there is no driver/device.
#include <dlfcn.h>
#if defined(__x86_64__)
#include <emmintrin.h>
#endif
#include <nvrtc.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <cctype>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <tuple>
#include <vector>

#include "../../include/rainier_cuda.h"
#include "rn_args.h"
#include "rn_cuda_api.hpp"
#include "rn_emit.hpp"
#include "rn_inline.hpp"
#include "rn_graph.hpp"

using namespace rn;
using namespace rn::cu;

// ---------------------------------------------------------------------------------------------------------
// driver loader
// ---------------------------------------------------------------------------------------------------------
namespace rn {
namespace cu {
const Api* api(std::string* why) {
  static Api a;
  static bool tried = false, ok = false;
  static std::string err;
  static std::mutex mu;
  std::lock_guard<std::mutex> lk(mu);
  if (!tried) {
    tried = true;
    void* h = dlopen("libcuda.so.1", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libcuda.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      err = std::string("cannot load the CUDA driver (libcuda.so.1): ") + dlerror();
    } else {
      ok = true;
#define RN_SYM(field, name)                                       \
  a.field = (decltype(a.field))dlsym(h, name);                    \
  if (!a.field) {                                                 \
    ok = false;                                                   \
    err = std::string("CUDA driver lacks symbol ") + name;        \
  }
      RN_SYM(cuInit, "cuInit")
      RN_SYM(cuDeviceGet, "cuDeviceGet")
      RN_SYM(cuDeviceGetCount, "cuDeviceGetCount")
      RN_SYM(cuDeviceGetAttribute, "cuDeviceGetAttribute")
      RN_SYM(cuDevicePrimaryCtxRetain, "cuDevicePrimaryCtxRetain")
      RN_SYM(cuDevicePrimaryCtxRelease, "cuDevicePrimaryCtxRelease_v2")
      RN_SYM(cuCtxSetCurrent, "cuCtxSetCurrent")
      RN_SYM(cuCtxGetCurrent, "cuCtxGetCurrent")
      RN_SYM(cuModuleLoadData, "cuModuleLoadData")
      RN_SYM(cuModuleUnload, "cuModuleUnload")
      RN_SYM(cuModuleGetFunction, "cuModuleGetFunction")
      RN_SYM(cuMemAlloc, "cuMemAlloc_v2")
      RN_SYM(cuMemFree, "cuMemFree_v2")
      RN_SYM(cuMemAllocHost, "cuMemAllocHost_v2")
      RN_SYM(cuMemFreeHost, "cuMemFreeHost")
      RN_SYM(cuMemHostRegister, "cuMemHostRegister_v2")
      RN_SYM(cuMemHostUnregister, "cuMemHostUnregister")
      RN_SYM(cuPointerGetAttribute, "cuPointerGetAttribute")
      a.cuPointerGetAttributes = (decltype(a.cuPointerGetAttributes))dlsym(h, "cuPointerGetAttributes");  // optional
      a.cuCtxGetDevice = (decltype(a.cuCtxGetDevice))dlsym(h, "cuCtxGetDevice");        // optional (NUMA placement)
      a.cuDeviceGetPCIBusId = (decltype(a.cuDeviceGetPCIBusId))dlsym(h, "cuDeviceGetPCIBusId");
      RN_SYM(cuMemcpyHtoD, "cuMemcpyHtoD_v2")
      RN_SYM(cuMemcpyDtoH, "cuMemcpyDtoH_v2")
      RN_SYM(cuMemcpyHtoDAsync, "cuMemcpyHtoDAsync_v2")
      RN_SYM(cuMemcpyDtoHAsync, "cuMemcpyDtoHAsync_v2")
      RN_SYM(cuMemcpy2DAsync, "cuMemcpy2DAsync_v2")
      RN_SYM(cuMemsetD8Async, "cuMemsetD8Async")
      RN_SYM(cuStreamCreate, "cuStreamCreate")
      RN_SYM(cuStreamDestroy, "cuStreamDestroy_v2")
      RN_SYM(cuStreamSynchronize, "cuStreamSynchronize")
      RN_SYM(cuStreamWaitEvent, "cuStreamWaitEvent")
      RN_SYM(cuEventCreate, "cuEventCreate")
      RN_SYM(cuEventDestroy, "cuEventDestroy_v2")
      RN_SYM(cuEventRecord, "cuEventRecord")
      RN_SYM(cuEventSynchronize, "cuEventSynchronize")
      RN_SYM(cuEventElapsedTime, "cuEventElapsedTime")
      RN_SYM(cuLaunchKernel, "cuLaunchKernel")
      RN_SYM(cuFuncGetAttribute, "cuFuncGetAttribute")
      RN_SYM(cuFuncSetAttribute, "cuFuncSetAttribute")
      RN_SYM(cuGetErrorString, "cuGetErrorString")
#undef RN_SYM
      if (ok) {
        CUresult r = a.cuInit(0);
        if (r != 0) {
          ok = false;
          const char* s = nullptr;
          a.cuGetErrorString(r, &s);
          err = std::string("cuInit failed: ") + (s ? s : "?");
        }
      }
    }
  }
  if (!ok) {
    if (why) *why = err;
    return nullptr;
  }
  return &a;
}
}  // namespace cu
}  // namespace rn

// ---------------------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------------------
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
static int cufail(const Api* A, CUresult r, const char* what) {
  const char* s = nullptr;
  if (A) A->cuGetErrorString(r, &s);
  return fail(RN_E_CUDA, std::string(what) + ": " + (s ? s : "CUDA error ") + " (" + std::to_string(r) + ")");
}
#define CU(call)                                  \
  do {                                            \
    CUresult _r = (call);                         \
    if (_r != 0) return cufail(A, _r, #call);     \
  } while (0)

// ---------------------------------------------------------------------------------------------------------
// model
// ---------------------------------------------------------------------------------------------------------
struct KernelKey {
  bool adjoint, fast, ehmc;
  int mass_max, backend;
  int block = 0;  // thread-per-chain: CTA size the module was compiled for (RN_BLOCK_DIM), 0 = any (emit / density-only uses)
  bool operator<(const KernelKey& o) const {
    return std::tie(adjoint, fast, ehmc, mass_max, backend, block) < std::tie(o.adjoint, o.fast, o.ehmc, o.mass_max, o.backend, o.block);
  }
};
// CTA size of the thread-per-chain kernels: 128 threads when there are chains to fill the chip twice over; a few thousand chains
// (cfg 2 / cfg 4: 4096-8192) are spread over all 148 SMs with smaller CTAs instead of packing 64 SMs and idling the rest.
// The sampler's module is COMPILED for this size (slot offsets of the per-thread shared-memory state become immediates:
// 2.469 -> 2.446 ms per launch at the headline size, profiles/r2_sweep_iter_v7_keep_state_block_dim.jsonl).
static unsigned tpc_block_for(size_t chains) {
  unsigned block = 128u;
  while (block > 32u && chains < (size_t)block * 148 * 2) block >>= 1;
  if (const char* e = getenv("RN_BLOCK")) block = std::max(32u, std::min(128u, (unsigned)atoi(e) & ~31u));
  return block;
}
struct Kernel {
  std::string source;
  std::vector<char> cubin;
  CUmodule mod = nullptr;
  CUfunction k_init = nullptr, k_iter = nullptr, k_warmup = nullptr, k_density = nullptr, k_transpose = nullptr, k_pool_reduce = nullptr,
             k_pool_apply = nullptr, k_diag_chain = nullptr, k_diag_reduce = nullptr;
  const Program* prog = nullptr;
  int backend = 0;            // 0 thread per chain, 1 warp per chain
  unsigned tpc_block = 0;     // backend 0: the CTA size this module was compiled for (0: reads blockDim.x)
  int wpc_smem_doubles = 0;   // per-warp dynamic shared memory (backend 1)
  int warps_per_cta = 4;      // backend 1: CHAINS per CTA (each owned by wpc_k warps)
  int wpc_k = 1;
  int tma_stages = 0;         // CTA-shared data-tile pipeline (backend 1): stages, doubles per stage
  int tile_doubles = 0;
  bool mma = false;           // backend 1: chain-batched DMMA path compiled in (tile_doubles = its shared doubles)
  int mma_chains = 8;         //            chains per CTA on that path (8 or 16)
  // backend 0: bytes of dynamic shared memory per THREAD (rn_sampler.cuh: momentum, diagonal mass, EHMC snapshot momentum,
  // Stats counters live there instead of in registers) -- must mirror RN_TS_DOUBLES / RN_TS_INTS
  unsigned tpc_smem_per_thread = 0;
  unsigned smem_bytes() const {  // dynamic shared memory of one CTA: per-warp slices | 128B pad | stages | mbarriers
    size_t d = (size_t)warps_per_cta * wpc_smem_doubles;
    if (tma_stages > 0) d = ((d + 15) & ~(size_t)15) + (size_t)tma_stages * tile_doubles + (size_t)(mma ? 8 : tma_stages);
    return (unsigned)(d * 8);
  }
};

struct rn_model {
  // Handles derived from one model (samplers, rn_sample, rn_optimize, diagnostics) share its caches: compiled kernels, the
  // spare arena / stream, the sample and diagnostics scratch pools.  Every entry point that touches them takes this lock,
  // so distinct handles of one model may be used from distinct threads (they serialise where they share state).
  std::recursive_mutex mu;
  std::vector<uint8_t> rir;
  uint32_t n_params = 0, n_inputs = 0;
  bool rir_has_gradient = false;
  int device = -1;
  CUcontext ctx = nullptr;
  CUdeviceptr d_data = 0;
  std::vector<uint64_t> target_base;  // per target: element offset of its tile-major block in the data buffer
  std::vector<int> target_pitch;      // per target: doubles between the columns of a tile (32, or 36 where the DMMA path may run)
  int inlined_targets = 0;            // streamed targets folded into data-free polynomials at create (rn_inline.hpp)
  int64_t inlined_monomials = 0, inlined_rows = 0;
  uint64_t data_doubles = 0;
  std::map<std::pair<bool, bool>, std::unique_ptr<Program>> programs;  // (adjoint, fast)
  std::map<KernelKey, std::unique_ptr<Kernel>> kernels;
  CUdeviceptr pool[2] = {0, 0};  // grow-only scratch reused by rn_sample calls (cuMemAlloc/cuMemFree of GBs is slow)
  // one spare set of sampler resources handed from a destroyed sampler to the next one: rn_sample creates and destroys a
  // sampler per call, and cuMemAlloc / cuMemFree / cuStreamCreate are synchronising driver calls
  CUdeviceptr diag_scratch = 0;  // grow-only scratch of rn_sampler_diagnostics
  size_t diag_bytes = 0;
  CUdeviceptr spare_arena = 0;
  size_t spare_arena_bytes = 0;
  CUstream spare_stream = nullptr;
  size_t pool_bytes[2] = {0, 0};
  // rn_optimize: one module per (adjoint, fast, history) -- cubin, module, rn_k_lbfgs
  struct OptKernel {
    std::string source;
    std::vector<char> cubin;
    CUmodule mod = nullptr;
    CUfunction k_lbfgs = nullptr;
    int backend = 0;           // 0 one thread per start, 1 one warp per start
    int smem_doubles = 0;      // backend 1: shared-memory slice of one start
    int starts_per_cta = 1;    // backend 1
    int wpc_k = 1;             // backend 1: warps per start
  };
  std::map<std::tuple<bool, bool, int, int>, std::unique_ptr<OptKernel>> opt_kernels;
};

static int make_current(const Api* A, rn_model* m) {
  CU(A->cuCtxSetCurrent(m->ctx));
  return RN_OK;
}

static int get_program(rn_model* m, bool adjoint, bool fast, const Program** out) {
  if (!m->rir_has_gradient) adjoint = true;
  auto key = std::make_pair(adjoint, fast);
  auto it = m->programs.find(key);
  if (it == m->programs.end()) {
    std::unique_ptr<Program> P(new Program());
    std::string e = build_program(m->rir.data(), m->rir.size(), adjoint, fast, *P);
    if (!e.empty()) return fail(RN_E_INVALID, e);
    it = m->programs.emplace(key, std::move(P)).first;
  }
  *out = it->second.get();
  return RN_OK;
}

static KernelKey key_for(const rn_model* m, const rn_config* cfg) {
  KernelKey k;
  const int gm = cfg ? cfg->gradient_mode : RN_GRAD_AUTO;
  k.adjoint = (gm == RN_GRAD_ADJOINT) || !m->rir_has_gradient;
  k.fast = cfg && cfg->math_mode == RN_MATH_FAST;
  k.ehmc = cfg && cfg->sampler == RN_SAMPLER_EHMC;
  k.mass_max = 0;
  if (cfg) {
    if (cfg->mass_tuner == RN_MASS_DIAGONAL) k.mass_max = 1;
    if (cfg->mass_tuner == RN_MASS_DENSE) k.mass_max = 2;
    if (cfg->mass_tuner == RN_MASS_STATIC) k.mass_max = cfg->static_matrix == RN_MATRIX_DENSE ? 2 : (cfg->static_matrix == RN_MATRIX_DIAGONAL ? 1 : 0);
  }
  // kernel shape: warp per chain when rows are streamed (or the state cannot live in registers)
  int want = cfg ? cfg->backend : RN_BACKEND_AUTO;
  if (const char* e = getenv("RN_BACKEND")) want = atoi(e);
  if (want == RN_BACKEND_AUTO) {
    uint64_t row_work = 0;  // node evaluations per gradient spent in streamed rows
    auto it = m->programs.begin();
    if (it != m->programs.end())
      for (const TargetInfo& T : it->second->targets)
        if (T.streamed()) row_work += T.n_rows * (uint64_t)(T.row_fwd.size() + T.row_bwd.size() + 1);
    want = (row_work >= 16384 || m->n_params > 48) ? RN_BACKEND_WARP : RN_BACKEND_THREAD;
    if (k.mass_max == 2) want = RN_BACKEND_THREAD;  // AUTO keeps dense mass on the thread-per-chain kernels (the shape measured on
                                                    // the GPU); the warp-per-chain kernels take it when asked for explicitly
  }
  k.backend = want == RN_BACKEND_WARP ? 1 : 0;
  return k;
}

extern "C" const char* rn_version(void);
// emit + NVRTC (no device needed)
// source_only: just emit (rn_emit_source, the analogue of rainier-decompile) -- no NVRTC run, nothing cached
static int get_kernel(rn_model* m, const rn_config* cfg, Kernel** out, std::string* source_only = nullptr, size_t chains_hint = 0) {
  KernelKey key = key_for(m, cfg);
  if (key.backend == 0 && chains_hint > 0) key.block = (int)tpc_block_for(chains_hint);
  auto it = m->kernels.find(key);
  if (it != m->kernels.end()) {
    if (source_only)
      *source_only = it->second->source;
    else
      *out = it->second.get();
    return RN_OK;
  }
  const Program* P = nullptr;
  int rc = get_program(m, key.adjoint, key.fast, &P);
  if (rc) return rc;
  std::unique_ptr<Kernel> K(new Kernel());
  K->prog = P;
  EmitOptions eo;
  eo.backend = key.backend;
  eo.fast_math = key.fast;
  eo.mass_max = key.mass_max;
  eo.enable_ehmc = key.ehmc;
  eo.target_base = m->target_base;
  eo.target_pitch = m->target_pitch;
  if (eo.backend == 1 && P->symbolic && P->n_params > 96)
    return fail(RN_E_UNSUPPORTED, "warp-per-chain with a symbolic gradient keeps n+1 accumulators in registers; use RN_GRAD_ADJOINT for n > 96");
  K->backend = eo.backend;
  K->tpc_block = (unsigned)key.block;
  if (eo.backend == 0) {  // rn_sampler.cuh: RN_TS_DOUBLES * 8 + RN_TS_INTS * 4
    const unsigned n = P->n_params;
    const unsigned doubles = (n + 1) + (key.mass_max >= 1 ? n : 0) + (key.ehmc ? n : 0) + 5 + 4;
    K->tpc_smem_per_thread = doubles * 8 + 10 * 4;
    if ((size_t)K->tpc_smem_per_thread * 32 > 227 * 1024 - 1024)
      return fail(RN_E_UNSUPPORTED, "thread-per-chain shape: the chain's shared-memory state does not fit; use RN_BACKEND_WARP");
  }
  if (eo.backend == 1) {
    const size_t cap = 227 * 1024 - 128;  // opt-in dynamic shared memory per CTA on sm_100 (232448 B; the sampler kernels have no static
                                         // shared memory and the 1 KB the system reserves per CTA is outside that figure)
    int wmax = 8;
    if (const char* e = getenv("RN_WPC_WARPS")) wmax = std::max(1, std::min(32, atoi(e)));
    // warps per chain: one, unless the chain's shared-memory state is so large that fewer than 16 chains fit an SM
    {
      const WpcSizes z1 = wpc_sizes(*P, eo);
      const size_t pc = (size_t)z1.per_warp_doubles * 8;
      if (pc > cap) return fail(RN_E_UNSUPPORTED, "model state does not fit one chain's shared memory slice");
      const size_t fit = std::max<size_t>(1, (cap - std::min<size_t>(cap / 4, 2 * (size_t)z1.tile_doubles * 8)) / pc);
      int k = 1;
      while (k < 8 && fit * (size_t)k < 16) k *= 2;  // aim at 16 warps per SM (cfg 5: K=1/2/4 -> 4.4e4 / 8.9e4 / 1.23e5 steps*chains/s)
      if (const char* e = getenv("RN_WPC_K")) k = std::max(1, std::min(8, atoi(e)));
      if (k != 1 && k != 2 && k != 4 && k != 8) k = 1;
      eo.wpc_k = K->wpc_k = k;
    }
    if (eo.wpc_k > 1) wmax = std::min(wmax, 14);  // named barriers 2..15, one per chain slot
    const WpcSizes z = wpc_sizes(*P, eo);
    K->wpc_smem_doubles = z.per_warp_doubles;
    K->tile_doubles = z.tile_doubles;
    const size_t per_warp = (size_t)z.per_warp_doubles * 8, tile = (size_t)z.tile_doubles * 8;
    if (per_warp > cap) return fail(RN_E_UNSUPPORTED, "model state does not fit one chain's shared memory slice");
    // data-tile stages: two (prefetch overlaps compute) when at least 4 chains still fit beside them, else one, else off
    int stages = 0;
    if (tile > 0) {
      if (2 * tile + std::min<size_t>(4, wmax) * per_warp + 256 <= cap)
        stages = 2;
      else if (tile + std::min<size_t>(2, wmax) * per_warp + 256 <= cap)
        stages = 1;
    }
    if (const char* e = getenv("RN_TMA")) {
      const int want_stages = atoi(e);
      if (want_stages == 0 || (size_t)want_stages * tile + per_warp + 256 <= cap) stages = tile > 0 ? want_stages : 0;
    }
    K->tma_stages = stages;
    const size_t left = cap - (size_t)stages * tile - (stages ? 256 : 0);
    K->warps_per_cta = (int)std::max<size_t>(1, std::min<size_t>((size_t)wmax, left / std::max<size_t>(per_warp, 1)));
    eo.tma_stages = stages;
    // chain-batched fp64 tensor-core path (rn_emit.cpp: Emitter::mma_block): HMC (every chain of a CTA evaluates the density
    // equally often), not the dense-mass code, one warp per chain, 8 chains per CTA, and every streamed target eligible
    bool want_mma = !key.ehmc && key.mass_max < 2 && eo.wpc_k == 1 && z.mma_ok && !P->symbolic;
    if (const char* e = getenv("RN_MMA")) want_mma = want_mma && atoi(e) != 0;
    if (want_mma) {
      // 16 chains per CTA when they fit (two chain groups whose warps pair up on a dot's column block: twice the warps per
      // SM -- the path is latency-bound at 8 -- for the same staged bytes), else 8
      int want_chains = 16;
      if (const char* e = getenv("RN_MMA_CHAINS")) want_chains = atoi(e) >= 16 ? 16 : 8;
      for (int nc = want_chains; nc >= 8 && !K->mma; nc -= 8) {
        EmitOptions em = eo;
        em.mma = true;
        em.mma_chains = nc;
        em.tma_stages = 1;
        const WpcSizes zm = wpc_sizes(*P, em);
        const size_t need = (size_t)nc * (size_t)zm.per_warp_doubles * 8 + 128 + (size_t)zm.mma_shared_doubles * 8 + 64;
        if (zm.mma_ok && need <= cap) {
          eo = em;
          K->mma = true;
          K->mma_chains = nc;
          K->wpc_smem_doubles = zm.per_warp_doubles;
          K->tile_doubles = zm.mma_shared_doubles;
          K->tma_stages = 1;
          K->warps_per_cta = nc;
        }
      }
    }
  }
  if (eo.backend == 1) {  // registers per thread the CTA leaves (see the cap below): fewer components in flight when it is tight
    const int warps = K->warps_per_cta * K->wpc_k;
    const int regs = warps * 32 * 255 > 65536 ? ((65536 / warps) / 512) * 512 / 32 : 255;
    // (with the branch-free row functions the components in flight share ONE basic block and ptxas overlaps them completely:
    // two at 128 registers -- cfg 5: 2.46e5 against 2.41e5 with four, profiles/r2_bench_row_libm_ab_v1.txt; the DMMA kernels
    // keep CUDA's libm and four)
    eo.interleave = regs <= 128 ? (wpc_sizes(*P, eo).row_functions ? 2 : 4) : 8;
    if (const char* e = getenv("RN_INTERLEAVE")) eo.interleave = std::max(1, atoi(e));
  }
  K->source = emit_source(*P, eo);
  if (source_only) {
    *source_only = std::move(K->source);
    return RN_OK;
  }

  std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo"};
  opts.push_back(key.fast ? "--fmad=true" : "--fmad=false");
  const std::string block_def = "-DRN_BLOCK_DIM=" + std::to_string(key.block);
  if (key.block > 0) opts.push_back(block_def.c_str());
  std::string maxreg;
  {
    // registers/thread: the fused iteration kernel is latency-bound on dependent fp64 chains, so occupancy matters
    // more than a few spills (profiles/r1_ncu_rn_k_iter_funnel_*: 240 regs -> 8 warps/SM, fp64 pipe 30% busy)
    int cap = (P->n_params <= 16 && eo.backend == 0) ? 128 : 0;
    if (eo.backend == 1) {  // the CTA (chains x warps per chain) must fit the 64K-register file
      const int warps = K->warps_per_cta * K->wpc_k;  // registers are allocated per warp in units of 512
      if (warps * 32 * 255 > 65536) cap = std::min(255, ((65536 / warps) / 512) * 512 / 32);
    }
    if (const char* e = getenv("RN_MAXRREGCOUNT")) cap = atoi(e);
    if (cap > 0) {
      maxreg = "--maxrregcount=" + std::to_string(cap);
      opts.push_back(maxreg.c_str());
    }
  }
  // optional on-disk cubin cache (NVRTC + ptxas of a large emitted model can take a minute): RN_KERNEL_CACHE=<dir>
  std::string cache_path;
  if (const char* dir = getenv("RN_KERNEL_CACHE")) {
    uint64_t h = 1469598103934665603ull;
    auto mix = [&](const std::string& t) {
      for (unsigned char ch : t) {
        h ^= ch;
        h *= 1099511628211ull;
      }
    };
    mix(K->source);
    for (const char* o : opts) mix(o);
    mix(rn_version());
    char name[64];
    snprintf(name, sizeof(name), "/%016llx.cubin", (unsigned long long)h);
    cache_path = std::string(dir) + name;
    if (FILE* f = fopen(cache_path.c_str(), "rb")) {
      fseek(f, 0, SEEK_END);
      long sz = ftell(f);
      fseek(f, 0, SEEK_SET);
      K->cubin.resize((size_t)sz);
      size_t got = fread(K->cubin.data(), 1, (size_t)sz, f);
      fclose(f);
      if (got == (size_t)sz && sz > 4) {
        *out = K.get();
        m->kernels.emplace(key, std::move(K));
        return RN_OK;
      }
      K->cubin.clear();
    }
  }
  nvrtcProgram prog;
  if (nvrtcCreateProgram(&prog, K->source.c_str(), "rainier_model.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS)
    return fail(RN_E_COMPILE, "nvrtcCreateProgram failed");
  nvrtcResult r = nvrtcCompileProgram(prog, (int)opts.size(), opts.data());
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    nvrtcGetProgramLogSize(prog, &n);
    std::string log(n, '\0');
    nvrtcGetProgramLog(prog, &log[0]);
    nvrtcDestroyProgram(&prog);
    if (const char* dump = getenv("RN_DUMP_FAILED_SOURCE")) {
      FILE* f = fopen(dump, "w");
      if (f) {
        fputs(K->source.c_str(), f);
        fclose(f);
      }
    }
    return fail(RN_E_COMPILE, std::string("NVRTC: ") + nvrtcGetErrorString(r) + "\n" + log);
  }
  size_t n = 0;
  nvrtcGetCUBINSize(prog, &n);
  K->cubin.resize(n);
  nvrtcGetCUBIN(prog, K->cubin.data());
  nvrtcDestroyProgram(&prog);
  if (!cache_path.empty()) {
    std::string tmp = cache_path + ".tmp" + std::to_string((long long)getpid());
    if (FILE* f = fopen(tmp.c_str(), "wb")) {
      fwrite(K->cubin.data(), 1, K->cubin.size(), f);
      fclose(f);
      rename(tmp.c_str(), cache_path.c_str());
    }
  }
  *out = K.get();
  m->kernels.emplace(key, std::move(K));
  return RN_OK;
}

static int load_kernel(const Api* A, rn_model* m, Kernel* K) {
  if (K->mod) return RN_OK;
  int rc = make_current(A, m);
  if (rc) return rc;
  CU(A->cuModuleLoadData(&K->mod, K->cubin.data()));
  CU(A->cuModuleGetFunction(&K->k_init, K->mod, "rn_k_init"));
  CU(A->cuModuleGetFunction(&K->k_iter, K->mod, "rn_k_iter"));
  if (K->backend == 0)  // thread per chain: the warmup phase is its own entry point (the sampling kernel carries no adaptation)
    CU(A->cuModuleGetFunction(&K->k_warmup, K->mod, "rn_k_warmup"));
  else
    K->k_warmup = K->k_iter;
  CU(A->cuModuleGetFunction(&K->k_density, K->mod, "rn_k_density"));
  CU(A->cuModuleGetFunction(&K->k_transpose, K->mod, "rn_k_transpose"));
  CU(A->cuModuleGetFunction(&K->k_pool_reduce, K->mod, "rn_k_pool_reduce"));
  CU(A->cuModuleGetFunction(&K->k_pool_apply, K->mod, "rn_k_pool_apply"));
  CU(A->cuModuleGetFunction(&K->k_diag_chain, K->mod, "rn_k_diag_chain"));
  CU(A->cuModuleGetFunction(&K->k_diag_reduce, K->mod, "rn_k_diag_reduce"));
  if (K->backend == 1) {
    const int bytes = (int)K->smem_bytes();
    for (CUfunction f : {K->k_init, K->k_iter, K->k_density})
      CU(A->cuFuncSetAttribute(f, 8 /*CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES*/, bytes));
  } else {
    for (CUfunction f : {K->k_init, K->k_iter, K->k_warmup}) {
      if (K->tpc_smem_per_thread * 128u > 48u * 1024u)
        CU(A->cuFuncSetAttribute(f, 8 /*CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES*/, (int)(K->tpc_smem_per_thread * 128u)));
      // the chains' cold state lives in shared memory: ask for the largest carve-out, or the driver's default split
      // (seen on B200: room for 5 CTAs of 25 KB) caps the occupancy below what the registers allow
      CU(A->cuFuncSetAttribute(f, 9 /*CU_FUNC_ATTRIBUTE_PREFERRED_SHARED_MEMORY_CARVEOUT*/, 100));
    }
  }
  return RN_OK;
}

// ---------------------------------------------------------------------------------------------------------
// Device layout of the observation columns: per streamed target a TILE-MAJOR block [tile][column][32 rows], tiles of
// 32 consecutive rows (the last one zero-padded), every block 128-byte aligned.  One tile is one contiguous chunk of
// n_cols*256 bytes: the warp-per-chain kernels fetch it with a single cp.async.bulk (TMA) into shared memory, and a
// plain load of (column j, row r) is base + (r>>5)*n_cols*32 + j*32 + (r&31) -- still 256-byte coalesced across a warp.
// (The reference keeps one JVM array per column, ir/DataFunction.scala:13-30, and gathers per row.)
// ---------------------------------------------------------------------------------------------------------
static uint64_t data_layout(const Program& P, std::vector<uint64_t>& target_base, std::vector<int>& target_pitch) {
  uint64_t off = 0;
  target_base.assign(P.targets.size(), 0);
  target_pitch = default_pitches(P);
  if (getenv("RN_PITCH32")) target_pitch.assign(P.targets.size(), 32);
  for (size_t t = 0; t < P.targets.size(); t++) {
    const TargetInfo& T = P.targets[t];
    if (!T.streamed()) continue;
    target_base[t] = off;
    const uint64_t tiles = (T.n_rows + 31) / 32;
    off += tiles * (uint64_t)T.n_cols * (uint64_t)target_pitch[t];
    off = (off + 15) & ~15ull;
  }
  return off;
}
static void pack_columns(const Program& P, const std::vector<uint64_t>& target_base, const std::vector<int>& target_pitch,
                         const double* const* cols, double* image) {
  for (size_t t = 0; t < P.targets.size(); t++) {
    const TargetInfo& T = P.targets[t];
    if (!T.streamed()) continue;
    const uint64_t pitch = (uint64_t)target_pitch[t], td = (uint64_t)T.n_cols * pitch;
    for (uint32_t j = 0; j < T.n_cols; j++) {
      const double* src = cols[T.first_input - P.n_params + j];
      double* dst = image + target_base[t] + (uint64_t)j * pitch;
      for (uint64_t r = 0; r < T.n_rows; r++) dst[(r >> 5) * td + (r & 31)] = src[r];
    }
  }
}

// One primary-context retain per device that is never released: process-wide resources (the pinned staging ring of the
// drain, rn_host_alloc buffers, the worker pool) must outlive any single model handle.  Without it, destroying the last
// model drops the primary context's refcount to zero, the driver frees the pinned ring with the context, and the next
// rn_sample copies through dangling pointers.
static int host_ctx(const Api* A, int device) {
  static std::mutex mu;
  static std::map<int, CUcontext> ctxs;  // one primary-context retain per device for the life of the process
  std::lock_guard<std::mutex> lk(mu);
  auto it = ctxs.find(device);
  if (it == ctxs.end()) {
    CUdevice dev;
    CUcontext ctx = nullptr;
    CU(A->cuDeviceGet(&dev, device));
    CU(A->cuDevicePrimaryCtxRetain(&ctx, dev));
    it = ctxs.emplace(device, ctx).first;
  }
  CU(A->cuCtxSetCurrent(it->second));
  return RN_OK;
}

extern "C" {

const char* rn_last_error(void) { return g_err.c_str(); }
const char* rn_version(void) { return "rainier_b200 0.1 (sm_100a, NVRTC)"; }

void rn_config_default(rn_config* c) {  // DefaultConfig, sampler/Sampler.scala:17-27
  std::memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(*c);
  c->iterations = 1000;
  c->warmup_iterations = 1000;
  c->stats_window = 100;
  c->sampler = RN_SAMPLER_EHMC;
  c->n_steps = 1;
  c->max_steps = 1024;
  c->min_steps = 1;
  c->buf_size = 100;
  c->p_count = 0.1;
  c->step_size_tuner = RN_STEP_DUAL_AVG;
  c->delta = 0.8;
  c->static_step_size = 1.0;
  c->mass_tuner = RN_MASS_DIAGONAL;
  c->initial_window_size = 50;
  c->window_expansion = 1.5;
  c->skip_first = 50;
  c->skip_last = 50;
}

// sizes of the ABI structs, for the binding's self-check
void rn_abi_sizes(int32_t out[4]) {
  out[0] = (int32_t)sizeof(rn_config);
  out[1] = (int32_t)sizeof(rn_chain_stats);
  out[2] = (int32_t)sizeof(rn_rng_state);
  out[3] = (int32_t)sizeof(RnArgs);
}

static int device_inline(rn_model* streamed, const InlinePlan& plan, std::vector<uint8_t>& new_rir);

static int model_create_impl(const void* rir, size_t len, const double* const* cols, const int64_t* col_rows, int n_cols,
                             int device, rn_model** out) {
  if (!rir || !out) return fail(RN_E_INVALID, "null argument");
  std::unique_ptr<rn_model> m(new rn_model());
  m->rir.assign((const uint8_t*)rir, (const uint8_t*)rir + len);
  if (len < sizeof(rir_header)) return fail(RN_E_INVALID, "RIR: truncated header");
  rir_header h;
  std::memcpy(&h, rir, sizeof(h));
  m->n_params = h.n_params;
  m->n_inputs = h.n_inputs;
  m->rir_has_gradient = (h.flags & RIR_FLAG_GRADIENT) != 0;
  if ((int)(h.n_inputs - h.n_params) != n_cols) return fail(RN_E_INVALID, "column count does not match the RIR's inputs");
  // validates the container (and caches the default program)
  const Program* P = nullptr;
  int rc = get_program(m.get(), !m->rir_has_gradient, false, &P);
  if (rc) return rc;
  for (const TargetInfo& T : P->targets)
    for (uint32_t j = 0; j < T.n_cols; j++)
      if (T.n_rows > 0 && (uint64_t)col_rows[T.first_input - h.n_params + j] != T.n_rows)  // (n_rows == 0: inlined, columns unread)
        return fail(RN_E_INVALID, "column length does not match its target's row count");
  m->data_doubles = data_layout(*P, m->target_base, m->target_pitch);
  m->device = device;
  if (device >= 0) {
    std::string why;
    const Api* A = api(&why);
    if (!A) return fail(RN_E_CUDA, why);
    CUdevice dev;
    rc = host_ctx(A, device);  // process-lifetime retain (see host_ctx)
    if (rc) return rc;
    CU(A->cuDeviceGet(&dev, device));
    CU(A->cuDevicePrimaryCtxRetain(&m->ctx, dev));
    CU(A->cuCtxSetCurrent(m->ctx));
    if (m->data_doubles > 0) {
      std::vector<double> image(m->data_doubles, 0.0);
      pack_columns(*P, m->target_base, m->target_pitch, cols, image.data());
      CU(A->cuMemAlloc(&m->d_data, m->data_doubles * 8));
      CU(A->cuMemcpyHtoD(m->d_data, image.data(), m->data_doubles * 8));
    }
  }
  *out = m.release();
  return RN_OK;
}

// Model creation = the streamed container as sent, then device-side inlining of its separable targets (rn_inline.hpp): the
// column-only monomials are summed over the rows ON THE DEVICE (data already in place), the target becomes a data-free
// polynomial, and the model is rebuilt from the rewritten container.  RN_INLINE=0 keeps every target streamed.
int rn_model_create(const void* rir, size_t len, const double* const* cols, const int64_t* col_rows, int n_cols,
                    int device, rn_model** out) {
  rn_model* m = nullptr;
  int rc = model_create_impl(rir, len, cols, col_rows, n_cols, device, &m);
  if (rc) return rc;
  const char* e = getenv("RN_INLINE");
  if (device >= 0 && !(e && atoi(e) == 0)) {
    InlinePlan plan;
    if (plan_inline(rir, len, plan).empty() && !plan.inl.empty()) {
      std::vector<uint8_t> nr;
      rc = device_inline(m, plan, nr);
      rn_model* m2 = nullptr;
      if (rc == RN_OK) rc = model_create_impl(nr.data(), nr.size(), cols, col_rows, n_cols, device, &m2);
      if (rc) {
        const std::string keep = rn_last_error();
        rn_model_destroy(m);
        return fail(rc, keep);
      }
      m2->inlined_targets = (int)plan.inl.size();
      for (const InlineTarget& I : plan.inl) {
        m2->inlined_monomials += (int64_t)I.monos.size();
        m2->inlined_rows += (int64_t)plan.targets[I.target].t.n_rows;
      }
      rn_model_destroy(m);
      m = m2;
    }
  }
  *out = m;
  return RN_OK;
}
// the two host halves of the inlining for tooling and tests (no device): which targets are separable and the function-flavour
// program of target k's monomials; the rewritten container for given row sums
int rn_inline_plan(const void* rir, size_t len, int k, int* n_targets, int* target_index, int64_t* n_monomials, void* fn_rir, size_t cap,
                   size_t* needed) {
  InlinePlan plan;
  const std::string e = plan_inline(rir, len, plan);
  if (!e.empty()) return fail(RN_E_INVALID, e);
  if (n_targets) *n_targets = (int)plan.inl.size();
  if (k < 0 || k >= (int)plan.inl.size()) return RN_OK;
  if (target_index) *target_index = plan.inl[k].target;
  if (n_monomials) *n_monomials = (int64_t)plan.inl[k].monos.size();
  const std::vector<uint8_t> f = inline_function_rir(plan, (size_t)k);
  if (needed) *needed = f.size();
  if (fn_rir && cap >= f.size()) std::memcpy(fn_rir, f.data(), f.size());
  return RN_OK;
}
int rn_inline_apply(const void* rir, size_t len, const double* sums /* all targets' monomials, concatenated */, size_t n_sums, void* out,
                    size_t cap, size_t* needed) {
  InlinePlan plan;
  const std::string e = plan_inline(rir, len, plan);
  if (!e.empty()) return fail(RN_E_INVALID, e);
  std::vector<std::vector<double>> s(plan.inl.size());
  size_t pos = 0;
  for (size_t k = 0; k < plan.inl.size(); k++) {
    if (pos + plan.inl[k].monos.size() > n_sums) return fail(RN_E_INVALID, "too few sums");
    s[k].assign(sums + pos, sums + pos + plan.inl[k].monos.size());
    pos += plan.inl[k].monos.size();
  }
  const std::vector<uint8_t> nr = apply_inline(plan, s);
  if (needed) *needed = nr.size();
  if (out && cap >= nr.size()) std::memcpy(out, nr.data(), nr.size());
  return RN_OK;
}
// what create folded: streamed targets inlined, monomials summed, rows no longer streamed per gradient
int rn_model_inlined(const rn_model* m, int64_t* monomials, int64_t* rows) {
  if (!m) return 0;
  if (monomials) *monomials = m->inlined_monomials;
  if (rows) *rows = m->inlined_rows;
  return m->inlined_targets;
}

// test/debug: the packed image of the data buffer exactly as rn_model_create uploads it (host emulation of the emitted
// source needs the same layout)
int rn_model_pack_columns(const rn_model* m, const double* const* cols, double* image, size_t cap_doubles, size_t* needed) {
  if (!m) return fail(RN_E_INVALID, "null model");
  if (needed) *needed = (size_t)m->data_doubles;
  if (!image) return RN_OK;
  if (cap_doubles < m->data_doubles) return fail(RN_E_INVALID, "buffer too small");
  auto it = m->programs.begin();
  if (it == m->programs.end()) return fail(RN_E_INVALID, "model has no program");
  std::memset(image, 0, (size_t)m->data_doubles * 8);
  pack_columns(*it->second, m->target_base, m->target_pitch, cols, image);
  return RN_OK;
}

int rn_model_nvars(const rn_model* m) { return m ? (int)m->n_params : RN_E_INVALID; }

void rn_model_destroy(rn_model* m) {
  if (!m) return;
  std::string why;
  const Api* A = m->device >= 0 ? api(&why) : nullptr;
  if (A && m->ctx) {
    A->cuCtxSetCurrent(m->ctx);
    for (auto& kv : m->kernels)
      if (kv.second->mod) A->cuModuleUnload(kv.second->mod);
    for (auto& kv : m->opt_kernels)
      if (kv.second->mod) A->cuModuleUnload(kv.second->mod);
    if (m->d_data) A->cuMemFree(m->d_data);
    for (auto p : m->pool)
      if (p) A->cuMemFree(p);
    if (m->spare_arena) A->cuMemFree(m->spare_arena);
    if (m->diag_scratch) A->cuMemFree(m->diag_scratch);
    if (m->spare_stream) A->cuStreamDestroy(m->spare_stream);
    CUdevice dev;
    if (A->cuDeviceGet(&dev, m->device) == 0) A->cuDevicePrimaryCtxRelease(dev);
  }
  delete m;
}

int rn_emit_source(rn_model* m, const rn_config* cfg, char* buf, size_t cap, size_t* needed) {
  if (!m) return fail(RN_E_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  std::string src;
  int rc = get_kernel(m, cfg, nullptr, &src);
  if (rc) return rc;
  if (needed) *needed = src.size() + 1;
  if (buf && cap) {
    size_t n = std::min(cap - 1, src.size());
    std::memcpy(buf, src.data(), n);
    buf[n] = 0;
  }
  return RN_OK;
}

int rn_emit_cubin(rn_model* m, const rn_config* cfg, void* buf, size_t cap, size_t* needed) {
  if (!m) return fail(RN_E_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  Kernel* K = nullptr;
  int rc = get_kernel(m, cfg, &K);
  if (rc) return rc;
  if (needed) *needed = K->cubin.size();
  if (buf && cap) std::memcpy(buf, K->cubin.data(), std::min(cap, K->cubin.size()));
  return RN_OK;
}

// static op counts of one gradient evaluation: out = [flops_invariant, special_invariant, sum over streamed
// targets of rows*flops_row, sum of rows*special_row]
int rn_model_op_counts(rn_model* m, const rn_config* cfg, double out[4]) {
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  KernelKey key = key_for(m, cfg);
  const Program* P = nullptr;
  int rc = get_program(m, key.adjoint, key.fast, &P);
  if (rc) return rc;
  out[0] = P->counts.flops_inv;
  out[1] = P->counts.special_inv;
  out[2] = out[3] = 0;
  for (size_t t = 0; t < P->targets.size(); t++) {
    out[2] += P->counts.flops_row[t] * (double)P->targets[t].n_rows;
    out[3] += P->counts.special_row[t] * (double)P->targets[t].n_rows;
  }
  return RN_OK;
}

// dense structure of the streamed row bodies (DotInfo, rn_graph.hpp): out = [dot products per gradient evaluation summed
// over rows, their multiply-adds per gradient (forward only), longest dot, number of distinct dots in the emitted code]
int rn_model_dot_structure(rn_model* m, const rn_config* cfg, double out[4]) {
  if (!m || !out) return fail(RN_E_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  KernelKey key = key_for(m, cfg);
  const Program* P = nullptr;
  int rc = get_program(m, key.adjoint, key.fast, &P);
  if (rc) return rc;
  out[0] = out[1] = out[2] = out[3] = 0;
  for (const TargetInfo& T : P->targets)
    for (const DotInfo& d : T.dots) {
      out[0] += (double)T.n_rows;
      out[1] += (double)T.n_rows * (double)d.params.size();
      out[2] = std::max(out[2], (double)d.params.size());
      out[3] += 1;
    }
  return RN_OK;
}

// separability of the streamed targets (SeparableInfo, rn_graph.hpp): out = [streamed targets, separable among them, atoms
// (row sums a device-side inliner would have to reduce), rows no longer streamed per gradient evaluation]
int rn_model_separable_structure(rn_model* m, double out[4]) {
  if (!m || !out) return fail(RN_E_INVALID, "null argument");
  const Program* P = nullptr;
  int rc = get_program(m, true, false, &P);  // the primal outputs decide (adjoint-mode program: one output per target)
  if (rc) return rc;
  const SeparableInfo s = analyze_separable(*P);
  out[0] = s.streamed_targets;
  out[1] = s.separable_targets;
  out[2] = (double)s.atoms;
  out[3] = (double)s.rows_removed;
  return RN_OK;
}

int rn_density_batch(rn_model* m, const double* q, int chains, double* out) {
  if (!m || !q || !out || chains <= 0) return fail(RN_E_INVALID, "bad argument");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  if (m->device < 0) return fail(RN_E_CUDA, "model was created without a device (no CPU fallback)");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  Kernel* K = nullptr;
  int rc = get_kernel(m, nullptr, &K);
  if (rc) return rc;
  rc = load_kernel(A, m, K);
  if (rc) return rc;
  const int n = (int)m->n_params;
  std::vector<double> qt((size_t)n * chains), ot((size_t)(n + 1) * chains);
  for (int c = 0; c < chains; c++)
    for (int i = 0; i < n; i++) qt[(size_t)i * chains + c] = q[(size_t)c * n + i];
  CUdeviceptr dq = 0, dout = 0, derr = 0;
  struct Free {  // released on every exit path
    const Api* A;
    CUdeviceptr *a, *b, *c;
    ~Free() {
      for (CUdeviceptr* p : {a, b, c})
        if (*p) A->cuMemFree(*p);
    }
  } guard{A, &dq, &dout, &derr};
  rc = make_current(A, m);
  if (rc) return rc;
  CU(A->cuMemAlloc(&dq, qt.size() * 8 + 8));
  CU(A->cuMemAlloc(&dout, ot.size() * 8));
  CU(A->cuMemAlloc(&derr, 4));
  CU(A->cuMemsetD8Async(derr, 0, 4, nullptr));
  CU(A->cuMemcpyHtoD(dq, qt.data(), qt.size() * 8));
  CUdeviceptr ddata = m->d_data;
  int ch = chains;
  void* params[] = {&dq, &dout, &ddata, &derr, &ch};
  if (K->backend == 1) {
    const unsigned w = (unsigned)K->warps_per_cta;
    CU(A->cuLaunchKernel(K->k_density, (unsigned)((chains + w - 1) / w), 1, 1, w * 32 * (unsigned)K->wpc_k, 1, 1,
                         K->smem_bytes(), nullptr, params, nullptr));
  } else {
    CU(A->cuLaunchKernel(K->k_density, (unsigned)((chains + 127) / 128), 1, 1, 128, 1, 1, 0, nullptr, params, nullptr));
  }
  CU(A->cuMemcpyDtoH(ot.data(), dout, ot.size() * 8));
  int err = 0;
  CU(A->cuMemcpyDtoH(&err, derr, 4));
  for (int c = 0; c < chains; c++)
    for (int i = 0; i <= n; i++) out[(size_t)c * (n + 1) + i] = ot[(size_t)i * chains + c];
  if (err & 1) return fail(RN_E_LOOKUP, "lookup index out of range");
  return RN_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// communicator: NCCL loaded with dlopen (torch-bundled or system libnccl.so.2); only the warmup-phase all-reduce
// of pooled mass-matrix statistics uses it -- the sampling path has no collective.
// ---------------------------------------------------------------------------------------------------------
namespace {
struct NcclId {
  char b[128];
};
typedef int (*nccl_init_fn)(void**, int, NcclId, int);
struct Nccl {
  int (*GetUniqueId)(NcclId*) = nullptr;
  nccl_init_fn CommInitRank = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, void*) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
const Nccl* nccl(std::string* why) {
  static Nccl n;
  static bool tried = false, ok = false;
  static std::string err;
  if (!tried) {
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) {
      err = std::string("cannot load libnccl.so.2: ") + dlerror();
    } else {
      n.GetUniqueId = (int (*)(NcclId*))dlsym(h, "ncclGetUniqueId");
      n.CommInitRank = (nccl_init_fn)dlsym(h, "ncclCommInitRank");
      n.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, void*))dlsym(h, "ncclAllReduce");
      n.CommDestroy = (int (*)(void*))dlsym(h, "ncclCommDestroy");
      n.GetErrorString = (const char* (*)(int))dlsym(h, "ncclGetErrorString");
      ok = n.GetUniqueId && n.CommInitRank && n.AllReduce && n.CommDestroy;
      if (!ok) err = "libnccl lacks a required symbol";
    }
  }
  if (!ok) {
    if (why) *why = err;
    return nullptr;
  }
  return &n;
}
}  // namespace

struct rn_comm {
  void* comm = nullptr;
  int rank = 0, world = 1, device = 0;
  CUcontext ctx = nullptr;
};

// ---------------------------------------------------------------------------------------------------------
// sampler
// ---------------------------------------------------------------------------------------------------------
struct rn_sampler {
  rn_model* m = nullptr;
  rn_config cfg;
  int chains = 0;
  Kernel* K = nullptr;
  CUstream stream = nullptr;
  CUdeviceptr arena = 0;
  size_t arena_bytes = 0, arena_alloc = 0;
  size_t stats_off = 0, stats_bytes = 0;  // the block that `new Stats` zeroes
  RnArgs args;                            // device pointers + uniform config
  bool initialized = false;
  int warm_done = 0;
  bool stats_reset_for_sampling = false;
  // host mirror of WindowedMassMatrixTuner's counters (identical for every chain)
  int win_size = 0, win_i = 0, win_j = 0, est_samples = 0, mass_kind = 0;
  int64_t launches = 0;
  CUdeviceptr d_trace = 0;  // optional test instrumentation, [warmup+iterations][4][chains]
  size_t trace_iters = 0, trace_pos = 0;
  rn_comm* comm = nullptr;
  CUdeviceptr d_pool = 0;  // [2n+1] pooled window statistics (RN_ADAPT_POOLED)
  // device time of the sampling phase (Stats.gradientTimes / iterationTimes, Stats.scala:8-9): events bracket every
  // batch of phase-1 launches; closed spans are summed when the stats are read
  CUevent ev_run[2] = {nullptr, nullptr};
  bool ev_open = false;
  // the warmup-phase all-reduce (RN_ADAPT_POOLED over rn_comm): calls issued, and event pairs around them (device time)
  int64_t allreduce_calls = 0;
  std::vector<std::pair<CUevent, CUevent>> allreduce_events;
  double sampling_ms = 0.0;
  int64_t sampling_iterations = 0;
};

namespace {

struct Arena {
  size_t off = 0;
  size_t take(size_t bytes) {
    size_t o = off;
    off += (bytes + 255) & ~(size_t)255;
    return o;
  }
};

int launch(const Api* A, rn_sampler* s, CUfunction f, int count = -1) {
  void* params[] = {&s->args};
  const size_t chains = count < 0 ? (size_t)s->chains : (size_t)count;
  if (s->K->backend == 1) {
    const unsigned w = (unsigned)s->K->warps_per_cta;
    const unsigned grid = (unsigned)((chains + w - 1) / w);
    CU(A->cuLaunchKernel(f, grid, 1, 1, w * 32 * (unsigned)s->K->wpc_k, 1, 1, s->K->smem_bytes(), s->stream, params, nullptr));
    s->launches++;
    return RN_OK;
  }
  const unsigned block = s->K->tpc_block ? s->K->tpc_block : tpc_block_for(chains);  // (the module may be compiled for its CTA size)
  const unsigned grid = (unsigned)((chains + block - 1) / block);
  CU(A->cuLaunchKernel(f, grid, 1, 1, block, 1, 1, s->K->tpc_smem_per_thread * block, s->stream, params, nullptr));
  s->launches++;
  return RN_OK;
}

// DenseMassMatrix.choleskyUpperTriangular, sampler/MassMatrix.scala:76-117 (host side, for StaticMassMatrix)
std::vector<double> cholesky_upper(const double* matrix, int n) {
  auto tri = [](int k) { return (k * (k + 1)) / 2; };
  std::vector<double> lower(tri(n), 0.0), upper(tri(n), 0.0);
  int l = 0;
  for (int i = 0; i < n; i++)
    for (int k = 0; k <= i; k++) {
      double sum = 0.0;
      for (int j = 0; j < k; j++) sum += lower[tri(i) + j] * lower[tri(k) + j];
      double x = matrix[i * n + k] - sum;
      lower[l++] = (i == k) ? std::sqrt(x) : (1.0 / lower[tri(k + 1) - 1] * x);
    }
  l = 0;
  for (int i = 0; i < n; i++)
    for (int k = 0; k < n - i; k++) upper[l++] = lower[tri(k + i) + i];
  return upper;
}

// mirrors the device-side WindowedMassMatrixTuner.update; returns the length of the window that closed on the LAST
// of these iterations (0 if none closed there)
int advance_window(rn_sampler* s, int iters) {
  const rn_config& c = s->cfg;
  if (c.mass_tuner != RN_MASS_DIAGONAL && c.mass_tuner != RN_MASS_DENSE) return 0;
  int closed = 0;
  for (int k = 0; k < iters; k++) {
    closed = 0;
    s->win_j += 1;
    if (s->win_j < c.skip_first || (c.warmup_iterations - s->win_j) < c.skip_last) continue;
    s->win_i += 1;
    s->est_samples += 1;
    if (s->win_i == s->win_size) {
      closed = s->win_size;
      s->win_i = 0;
      double w = s->win_size * c.window_expansion;
      s->win_size = (w >= 2147483647.0) ? 2147483647 : (int)w;
      s->mass_kind = c.mass_tuner == RN_MASS_DIAGONAL ? RN_MATRIX_DIAGONAL : RN_MATRIX_DENSE;
    }
  }
  return closed;
}
// number of iterations from now up to and including the next window end (or `limit` if none within it)
int iterations_to_window_end(const rn_sampler* s, int limit) {
  const rn_config& c = s->cfg;
  int j = s->win_j, i = s->win_i;
  for (int k = 1; k <= limit; k++) {
    j += 1;
    if (j < c.skip_first || (c.warmup_iterations - j) < c.skip_last) continue;
    i += 1;
    if (i == s->win_size) return k;
  }
  return limit;
}

int check_config(const rn_model* m, const rn_config* c, int chains) {
  if (!c) return fail(RN_E_INVALID, "null config");
  if (c->struct_size != (int32_t)sizeof(rn_config)) return fail(RN_E_INVALID, "rn_config.struct_size mismatch");
  if (chains <= 0) return fail(RN_E_INVALID, "chains must be positive");
  if (c->iterations < 0 || c->warmup_iterations < 0 || c->stats_window <= 0) return fail(RN_E_INVALID, "bad iteration counts");
  if (c->sampler == RN_SAMPLER_HMC) {
    if (c->n_steps < 0) return fail(RN_E_INVALID, "n_steps < 0");
  } else if (c->sampler == RN_SAMPLER_EHMC) {
    if (c->max_steps < 1 || c->min_steps < 1 || c->buf_size < 1) return fail(RN_E_INVALID, "bad EHMC parameters");
  } else {
    return fail(RN_E_UNSUPPORTED, "only the built-in HMCSampler / EHMCSampler can be lowered to the GPU");
  }
  if (c->step_size_tuner != RN_STEP_DUAL_AVG && c->step_size_tuner != RN_STEP_STATIC)
    return fail(RN_E_UNSUPPORTED, "unknown step size tuner");
  if (c->mass_tuner < RN_MASS_IDENTITY || c->mass_tuner > RN_MASS_STATIC) return fail(RN_E_UNSUPPORTED, "unknown mass matrix tuner");
  if (c->mass_tuner == RN_MASS_STATIC && c->static_matrix != RN_MATRIX_IDENTITY && !c->static_matrix_elements)
    return fail(RN_E_INVALID, "static mass matrix without elements");
  if (c->mass_tuner == RN_MASS_DENSE || (c->mass_tuner == RN_MASS_STATIC && c->static_matrix == RN_MATRIX_DENSE)) {
    // thread per chain: the Cholesky scratch is thread-local; warp per chain: matrix, factor and estimator live in the
    // chain's global-memory state (n^2 doubles each)
    const bool warp = c->backend == RN_BACKEND_WARP;
    if (!warp && m->n_params > 64)
      return fail(RN_E_UNSUPPORTED, "dense mass matrix on the thread-per-chain kernels is supported for n <= 64 (use RN_BACKEND_WARP)");
    if (warp && m->n_params > 512) return fail(RN_E_UNSUPPORTED, "dense mass matrix supported for n <= 512");
  }
  if (c->adaptation == RN_ADAPT_POOLED && c->mass_tuner != RN_MASS_DIAGONAL)
    return fail(RN_E_UNSUPPORTED, "pooled adaptation is implemented for the diagonal mass-matrix tuner");
  return RN_OK;
}

}  // namespace

extern "C" {

int rn_sampler_create(rn_model* m, const rn_config* cfg, const int64_t* seeds, int chains, rn_sampler** out) {
  if (!m || !out) return fail(RN_E_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  int rc = check_config(m, cfg, chains);
  if (rc) return rc;
  if (!seeds && !cfg->rng_states) return fail(RN_E_INVALID, "need seeds or rng_states");
  if (m->device < 0) return fail(RN_E_CUDA, "model was created without a device (no CPU fallback)");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  struct Destroy {
    void operator()(rn_sampler* p) const { rn_sampler_destroy(p); }  // frees stream / arena / pools on a failed create
  };
  std::unique_ptr<rn_sampler, Destroy> s(new rn_sampler());
  s->m = m;
  s->cfg = *cfg;
  s->chains = chains;
  rc = get_kernel(m, cfg, &s->K, nullptr, (size_t)chains);
  if (rc) return rc;
  rc = load_kernel(A, m, s->K);
  if (rc) return rc;
  if (m->spare_stream) {
    s->stream = m->spare_stream;
    m->spare_stream = nullptr;
  } else {
    CU(A->cuStreamCreate(&s->stream, 1 /*CU_STREAM_NON_BLOCKING*/));
  }

  const size_t C = (size_t)chains, n = m->n_params, W = (size_t)cfg->stats_window;
  const bool dense = s->K && (key_for(m, cfg).mass_max == 2);
  const bool diag = key_for(m, cfg).mass_max >= 1;
  const bool ehmc = cfg->sampler == RN_SAMPLER_EHMC;
  Arena ar;
  const size_t o_params = ar.take((2 * n + 1) * C * 8), o_grad = ar.take(n * C * 8), o_seed = ar.take(C * 8),
               o_nng = ar.take(C * 8), o_have = ar.take(C * 4), o_da = ar.take(5 * C * 8), o_dait = ar.take(C * 4),
               o_mass = ar.take((dense ? n * n : (diag ? n : 0)) * C * 8 + 8),
               o_chol = ar.take((dense ? n * (n + 1) / 2 : 0) * C * 8 + 8), o_emean = ar.take((diag ? n : 0) * C * 8 + 8),
               o_eraw = ar.take((diag ? n : 0) * C * 8 + 8), o_ecov = ar.take((dense ? n * n : 0) * C * 8 + 8),
               o_ring = ar.take((ehmc ? (size_t)cfg->buf_size : 0) * C * 8 + 8), o_ri = ar.take(C * 4), o_rf = ar.take(C * 4),
               o_err = ar.take(C * 4);
  s->stats_off = ar.off;
  const size_t o_sg = ar.take(C * 8), o_ss = ar.take(C * 8), o_si = ar.take(C * 4), o_sa = ar.take(C * 4),
               o_se = ar.take(3 * C * 8), o_sen = ar.take(C * 4), o_sr = ar.take(3 * W * C * 8), o_sri = ar.take(3 * C * 4),
               o_srf = ar.take(3 * C * 4);
  s->stats_bytes = ar.off - s->stats_off;
  s->arena_bytes = ar.off;
  const size_t pool_off = (s->arena_bytes + 255) & ~(size_t)255, need = pool_off + (2 * n + 1) * 8;
  if (m->spare_arena && m->spare_arena_bytes >= need) {
    s->arena = m->spare_arena;
    s->arena_alloc = m->spare_arena_bytes;
    m->spare_arena = 0;
    m->spare_arena_bytes = 0;
  } else {
    CU(A->cuMemAlloc(&s->arena, need));
    s->arena_alloc = need;
  }
  s->d_pool = s->arena + pool_off;  // [2n+1] pooled window statistics live behind the chain state
  CU(A->cuMemsetD8Async(s->arena, 0, s->arena_bytes, s->stream));

  RnArgs& a = s->args;
  std::memset(&a, 0, sizeof(a));
  auto P = [&](size_t o) { return (void*)(uintptr_t)(s->arena + o); };
  a.chains = chains;
  a.params = (double*)P(o_params);
  a.grad = (double*)P(o_grad);
  a.rng_seed = (rn_i64*)P(o_seed);
  a.rng_nng = (double*)P(o_nng);
  a.rng_have = (int*)P(o_have);
  a.da = (double*)P(o_da);
  a.da_iter = (int*)P(o_dait);
  a.mass = (double*)P(o_mass);
  a.chol = (double*)P(o_chol);
  a.est_mean = (double*)P(o_emean);
  a.est_raw = (double*)P(o_eraw);
  a.est_cov = (double*)P(o_ecov);
  a.ring = (double*)P(o_ring);
  a.ring_i = (int*)P(o_ri);
  a.ring_full = (int*)P(o_rf);
  a.st_err = (int*)P(o_err);
  a.st_grads = (rn_i64*)P(o_sg);
  a.st_steps = (rn_i64*)P(o_ss);
  a.st_iters = (int*)P(o_si);
  a.st_accepted = (int*)P(o_sa);
  a.st_energy = (double*)P(o_se);
  a.st_energy_n = (int*)P(o_sen);
  a.st_rings = (double*)P(o_sr);
  a.st_ring_i = (int*)P(o_sri);
  a.st_ring_full = (int*)P(o_srf);
  a.data = (const double*)(uintptr_t)m->d_data;
  a.sampler = cfg->sampler;
  a.n_steps = cfg->n_steps;
  a.max_steps = cfg->max_steps;
  a.min_steps = cfg->min_steps;
  a.buf_size = cfg->buf_size;
  a.step_tuner = cfg->step_size_tuner;
  a.p_count = cfg->p_count;
  a.delta = cfg->delta;
  a.static_step = cfg->static_step_size;
  a.mass_tuner = cfg->mass_tuner;
  a.total_warmup = cfg->warmup_iterations;
  a.skip_first = cfg->skip_first;
  a.skip_last = cfg->skip_last;
  a.win_expansion = cfg->window_expansion;
  a.stats_window = cfg->stats_window;
  s->win_size = cfg->initial_window_size;

  // RNG state: ScalaRNG(seed) = new java.util.Random(seed): scrambled seed (sampler/RNG.scala:20-26)
  std::vector<int64_t> seed48(C);
  std::vector<double> nng(C, 0.0);
  std::vector<int32_t> have(C, 0);
  for (size_t c = 0; c < C; c++) {
    if (cfg->rng_states) {
      seed48[c] = cfg->rng_states[c].seed48;
      nng[c] = cfg->rng_states[c].next_gaussian;
      have[c] = cfg->rng_states[c].have_next;
    } else {
      seed48[c] = (seeds[c] ^ 0x5DEECE66DLL) & ((1LL << 48) - 1);
    }
  }
  CU(A->cuMemcpyHtoDAsync(s->arena + o_seed, seed48.data(), C * 8, s->stream));
  CU(A->cuMemcpyHtoDAsync(s->arena + o_nng, nng.data(), C * 8, s->stream));
  CU(A->cuMemcpyHtoDAsync(s->arena + o_have, have.data(), C * 4, s->stream));
  // StaticMassMatrix: replicate the shared matrix to every chain (and factor it once, on the host)
  if (cfg->mass_tuner == RN_MASS_STATIC && cfg->static_matrix != RN_MATRIX_IDENTITY) {
    const size_t ne = cfg->static_matrix == RN_MATRIX_DENSE ? n * n : n;
    std::vector<double> rep(ne * C);
    for (size_t e = 0; e < ne; e++) {
      if (cfg->static_matrix_elements[e] == 0.0)
        return fail(RN_E_INVALID, "requirement failed: mass matrix contains 0.0 (MassMatrix.scala:8,16)");
      for (size_t c = 0; c < C; c++) rep[e * C + c] = cfg->static_matrix_elements[e];
    }
    CU(A->cuMemcpyHtoDAsync(s->arena + o_mass, rep.data(), rep.size() * 8, s->stream));
    if (cfg->static_matrix == RN_MATRIX_DENSE) {
      std::vector<double> up = cholesky_upper(cfg->static_matrix_elements, (int)n);
      std::vector<double> repu(up.size() * C);
      for (size_t e = 0; e < up.size(); e++)
        for (size_t c = 0; c < C; c++) repu[e * C + c] = up[e];
      CU(A->cuMemcpyHtoDAsync(s->arena + o_chol, repu.data(), repu.size() * 8, s->stream));
    }
    CU(A->cuStreamSynchronize(s->stream));
  }
  CU(A->cuStreamSynchronize(s->stream));
  *out = s.release();
  return RN_OK;
}

// test instrumentation: per-iteration trace [warmup+iterations][4][chains] kept on the device
int rn_sampler_enable_trace(rn_sampler* s) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  s->trace_iters = (size_t)s->cfg.warmup_iterations + (size_t)s->cfg.iterations;
  CU(A->cuMemAlloc(&s->d_trace, std::max<size_t>(1, s->trace_iters) * 4 * (size_t)s->chains * 8));
  return RN_OK;
}
int rn_sampler_read_trace(rn_sampler* s, double* out /*[chains][iters][4]*/) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  CU(A->cuStreamSynchronize(s->stream));
  const size_t C = (size_t)s->chains, I = s->trace_pos;
  std::vector<double> tmp(I * 4 * C);
  CU(A->cuMemcpyDtoH(tmp.data(), s->d_trace, tmp.size() * 8));
  for (size_t c = 0; c < C; c++)
    for (size_t i = 0; i < I; i++)
      for (size_t k = 0; k < 4; k++) out[(c * s->trace_iters + i) * 4 + k] = tmp[(i * 4 + k) * C + c];
  return RN_OK;
}

static int pool_window(const Api* A, rn_sampler* s, int window_len) {
  const size_t n = s->m->n_params;
  CU(A->cuMemsetD8Async(s->d_pool, 0, (2 * n + 1) * 8, s->stream));
  std::string why;
  const Nccl* N = nullptr;
  if (s->comm && s->comm->world > 1) {
    N = nccl(&why);
    if (!N) return fail(RN_E_NCCL, why);
  }
  // two passes (pooled mean, then Chan's combination of the chains' M2 around it), each a deterministic reduction over this
  // GPU's chains followed by one small all-reduce over the ranks
  for (int pass = 0; pass < 2; pass++) {
    CUdeviceptr pool = s->d_pool;
    int wl = window_len, ps = pass;
    void* params[] = {&s->args, &pool, &wl, &ps};
    CU(A->cuLaunchKernel(s->K->k_pool_reduce, (unsigned)n, 1, 1, 256, 1, 1, 0, s->stream, params, nullptr));
    s->launches++;
    if (N) {
      CUevent e0 = nullptr, e1 = nullptr;
      if (s->allreduce_events.size() < 256) {
        CU(A->cuEventCreate(&e0, 0));
        CU(A->cuEventCreate(&e1, 0));
        CU(A->cuEventRecord(e0, s->stream));
      }
      const CUdeviceptr buf = pass ? s->d_pool + (1 + n) * 8 : s->d_pool;
      const size_t count = pass ? n : n + 1;
      int r = N->AllReduce((const void*)(uintptr_t)buf, (void*)(uintptr_t)buf, count, 8 /*ncclFloat64*/, 0 /*ncclSum*/, s->comm->comm,
                           (void*)s->stream);
      if (e1) {
        A->cuEventRecord(e1, s->stream);
        s->allreduce_events.push_back({e0, e1});
      }
      if (r != 0) return fail(RN_E_NCCL, std::string("ncclAllReduce: ") + (N->GetErrorString ? N->GetErrorString(r) : "?"));
      s->allreduce_calls++;
    }
  }
  {
    CUdeviceptr pool = s->d_pool;
    int wl = window_len;
    void* params[] = {&s->args, &pool, &wl};
    CU(A->cuLaunchKernel(s->K->k_pool_apply, (unsigned)((s->chains + 127) / 128), 1, 1, 128, 1, 1, 0, s->stream, params, nullptr));
    s->launches++;
  }
  return RN_OK;
}

static int run_phase(const Api* A, rn_sampler* s, int phase, int iterations, double* d_samples, int chain_begin = 0,
                     int chain_end = -1) {
  if (chain_end < 0) chain_end = s->chains;
  const int per_launch = s->cfg.launch_iterations > 0 ? s->cfg.launch_iterations : 1000;
  const bool pooled = phase == 0 && s->cfg.adaptation == RN_ADAPT_POOLED && s->cfg.mass_tuner == RN_MASS_DIAGONAL;
  int done = 0;
  if (phase == 1 && iterations > 0) {
    if (!s->ev_run[0]) {
      CU(A->cuEventCreate(&s->ev_run[0], 0));
      CU(A->cuEventCreate(&s->ev_run[1], 0));
    }
    if (!s->ev_open) {
      CU(A->cuEventRecord(s->ev_run[0], s->stream));
      s->ev_open = true;
    }
    if (chain_begin == 0) s->sampling_iterations += iterations;  // rn_sample's chain blocks repeat the same iterations
  }
  while (done < iterations) {
    int k = std::min(per_launch, iterations - done);
    if (pooled) k = iterations_to_window_end(s, k);  // launches end exactly at window ends
    RnArgs& a = s->args;
    a.phase = phase;
    a.n_iter = k;
    a.adaptation = s->cfg.adaptation == RN_ADAPT_POOLED ? 1 : 0;
    a.tma = s->K->tma_stages > 0 ? 1 : 0;
    // the DMMA path wants full CTAs (8 or 16 chains): the whole groups of a batch run it, a ragged tail (and a batch that
    // does not start on a group boundary) runs the per-warp path of the same kernel in a second launch
    int tail_begin = chain_end;
    if (s->K->mma) {
      const int nc = s->K->mma_chains;
      if (chain_begin % nc != 0)
        a.tma = 0;
      else
        tail_begin = chain_begin + ((chain_end - chain_begin) / nc) * nc;
      if (tail_begin == chain_begin) a.tma = 0, tail_begin = chain_end;
    }
    a.chain_begin = chain_begin;
    a.chain_end = tail_begin;
    a.mass_kind = s->mass_kind;
    a.win_size = s->win_size;
    a.win_i = s->win_i;
    a.win_j = s->win_j;
    a.est_samples = s->est_samples;
    a.samples = (phase == 1 && d_samples) ? d_samples + (size_t)done * s->m->n_params * (size_t)s->chains : nullptr;
    a.trace = s->d_trace ? (double*)(uintptr_t)(s->d_trace + s->trace_pos * 4 * (size_t)s->chains * 8) : nullptr;
    int rc = launch(A, s, phase == 0 ? s->K->k_warmup : s->K->k_iter, tail_begin - chain_begin);
    if (rc) return rc;
    if (tail_begin < chain_end) {
      a.tma = 0;
      a.chain_begin = tail_begin;
      a.chain_end = chain_end;
      rc = launch(A, s, phase == 0 ? s->K->k_warmup : s->K->k_iter, chain_end - tail_begin);
      if (rc) return rc;
    }
    if (phase == 0) {
      const int closed = advance_window(s, k);
      if (pooled && closed > 0) {
        rc = pool_window(A, s, closed);
        if (rc) return rc;
      }
    }
    if (s->d_trace) s->trace_pos += (size_t)k;
    done += k;
  }
  if (phase == 1 && iterations > 0) CU(A->cuEventRecord(s->ev_run[1], s->stream));
  return RN_OK;
}

int rn_sampler_warmup(rn_sampler* s, int iterations) {
  if (!s) return fail(RN_E_INVALID, "null sampler");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  if (!s->initialized) {
    s->args.mass_kind = 0;
    int rc = launch(A, s, s->K->k_init);  // LeapFrog.initialize + tuner initialisation
    if (rc) return rc;
    s->initialized = true;
    if (s->cfg.mass_tuner == RN_MASS_STATIC) s->mass_kind = s->cfg.static_matrix;  // StaticMassMatrix.initialize
  }
  const int left = s->cfg.warmup_iterations - s->warm_done;
  const int k = (iterations < 0 || iterations > left) ? left : iterations;
  int rc = run_phase(A, s, 0, k, nullptr);
  if (rc) return rc;
  s->warm_done += k;
  return RN_OK;
}

int rn_sampler_run(rn_sampler* s, int iterations, double* d_samples) {
  if (!s) return fail(RN_E_INVALID, "null sampler");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  if (!s->initialized) {
    int rc = rn_sampler_warmup(s, 0);
    if (rc) return rc;
  }
  if (!s->stats_reset_for_sampling) {  // lf.resetStats(), Driver.scala:31
    CU(A->cuMemsetD8Async(s->arena + s->stats_off, 0, s->stats_bytes, s->stream));
    s->stats_reset_for_sampling = true;
  }
  return run_phase(A, s, 1, iterations, d_samples);
}

namespace {
// fold the open event span of the sampling phase into sampling_ms (the stream must be idle)
int close_sampling_span(const Api* A, rn_sampler* s) {
  if (!s->ev_open) return RN_OK;
  float ms = 0.f;
  CU(A->cuEventElapsedTime(&ms, s->ev_run[0], s->ev_run[1]));
  s->sampling_ms += (double)ms;
  s->ev_open = false;
  return RN_OK;
}
}  // namespace

int rn_sampler_sync(rn_sampler* s) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  CU(A->cuStreamSynchronize(s->stream));
  return RN_OK;
}

void* rn_sampler_stream(rn_sampler* s) { return s ? (void*)s->stream : nullptr; }
int64_t rn_sampler_launches(const rn_sampler* s) { return s ? s->launches : 0; }

int rn_sampler_positions(rn_sampler* s, double* q) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  CU(A->cuStreamSynchronize(s->stream));
  const size_t C = (size_t)s->chains, n = s->m->n_params;
  std::vector<double> tmp(n * C);
  CU(A->cuMemcpyDtoH(tmp.data(), (CUdeviceptr)(uintptr_t)s->args.params + n * C * 8, n * C * 8));
  for (size_t c = 0; c < C; c++)
    for (size_t i = 0; i < n; i++) q[c * n + i] = tmp[i * C + c];
  return RN_OK;
}

int rn_sampler_stats(rn_sampler* s, rn_chain_stats* stats, double* mass, double* stats_rings) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  CU(A->cuStreamSynchronize(s->stream));
  {
    int rc = close_sampling_span(A, s);
    if (rc) return rc;
  }
  const size_t C = (size_t)s->chains, n = s->m->n_params, W = (size_t)s->cfg.stats_window;
  const RnArgs& a = s->args;
  auto D = [](const void* p) { return (CUdeviceptr)(uintptr_t)p; };
  std::vector<int32_t> err(C);
  CU(A->cuMemcpyDtoH(err.data(), D(a.st_err), C * 4));
  int any_err = 0;
  for (size_t c = 0; c < C; c++) any_err |= err[c];
  if (stats) {
    std::vector<int64_t> sg(C), ss(C), seed(C);
    std::vector<int32_t> si(C), sa(C), sen(C), sri(3 * C), srf(3 * C), have(C);
    std::vector<double> se(3 * C), da(5 * C), rings(3 * W * C), nng(C);
    CU(A->cuMemcpyDtoH(sg.data(), D(a.st_grads), C * 8));
    CU(A->cuMemcpyDtoH(ss.data(), D(a.st_steps), C * 8));
    CU(A->cuMemcpyDtoH(si.data(), D(a.st_iters), C * 4));
    CU(A->cuMemcpyDtoH(sa.data(), D(a.st_accepted), C * 4));
    CU(A->cuMemcpyDtoH(sen.data(), D(a.st_energy_n), C * 4));
    CU(A->cuMemcpyDtoH(sri.data(), D(a.st_ring_i), 3 * C * 4));
    CU(A->cuMemcpyDtoH(srf.data(), D(a.st_ring_full), 3 * C * 4));
    CU(A->cuMemcpyDtoH(se.data(), D(a.st_energy), 3 * C * 8));
    CU(A->cuMemcpyDtoH(da.data(), D(a.da), 5 * C * 8));
    CU(A->cuMemcpyDtoH(rings.data(), D(a.st_rings), 3 * W * C * 8));
    CU(A->cuMemcpyDtoH(seed.data(), D(a.rng_seed), C * 8));
    CU(A->cuMemcpyDtoH(nng.data(), D(a.rng_nng), C * 8));
    CU(A->cuMemcpyDtoH(have.data(), D(a.rng_have), C * 4));
    for (size_t c = 0; c < C; c++) {
      rn_chain_stats& o = stats[c];
      std::memset(&o, 0, sizeof(o));
      o.gradient_evaluations = sg[c];
      o.leapfrog_steps = ss[c];
      o.iterations = si[c];
      o.accepted = sa[c];
      o.error_flags = err[c];
      // stepSizeTuner.stepSize: exp(logStepSizeBar) for DualAvg (DualAvg.scala:23-25)
      o.step_size = s->cfg.step_size_tuner == RN_STEP_DUAL_AVG ? std::exp(da[2 * C + c]) : s->cfg.static_step_size;
      o.energy_mean = se[0 * C + c];
      o.energy_raw = se[1 * C + c];
      o.energy_transitions2 = se[2 * C + c];
      o.energy_samples = sen[c];
      double means[3];
      for (int r = 0; r < 3; r++) {
        o.ring_pos[r] = sri[r * C + c];
        o.ring_full[r] = srf[r * C + c];
        double sum = 0.0;  // RingBuffer.mean, Stats.scala:47-58
        for (size_t j = 0; j < W; j++) sum += rings[((size_t)r * W + j) * C + c];
        means[r] = o.ring_full[r] ? sum / (double)W : sum / (double)o.ring_pos[r];
        if (stats_rings)
          for (size_t j = 0; j < W; j++) stats_rings[(c * 3 + r) * W + j] = rings[((size_t)r * W + j) * C + c];
      }
      o.step_sizes_mean = means[0];
      o.acceptance_rates_mean = means[1];
      o.grads_per_iteration_mean = means[2];
      // Stats.gradientTimes / iterationTimes (Stats.scala:8-9, LeapFrog.scala:57,77,196-198) hold per-call nanoseconds of
      // ONE chain on a JVM thread; here all chains advance together, so the means are device time of the sampling
      // launches / count: per iteration of the batch, and per gradient evaluation of this chain
      const double ns = s->sampling_ms * 1e6;
      o.iteration_time_ns_mean = s->sampling_iterations > 0 ? ns / (double)s->sampling_iterations : 0.0;
      o.gradient_time_ns_mean = sg[c] > 0 ? ns / (double)sg[c] : 0.0;
      o.rng.seed48 = seed[c];
      o.rng.next_gaussian = nng[c];
      o.rng.have_next = have[c];
    }
  }
  if (mass) {
    const bool dense = s->cfg.mass_tuner == RN_MASS_DENSE || (s->cfg.mass_tuner == RN_MASS_STATIC && s->cfg.static_matrix == RN_MATRIX_DENSE);
    const size_t ne = dense ? n * n : n;
    if (s->mass_kind == RN_MATRIX_IDENTITY) {
      for (size_t c = 0; c < C; c++)
        for (size_t e = 0; e < ne; e++) mass[c * ne + e] = dense ? ((e / n == e % n) ? 1.0 : 0.0) : 1.0;
    } else {
      std::vector<double> tmp(ne * C);
      CU(A->cuMemcpyDtoH(tmp.data(), D(a.mass), ne * C * 8));
      for (size_t c = 0; c < C; c++)
        for (size_t e = 0; e < ne; e++) mass[c * ne + e] = tmp[e * C + c];
    }
  }
  if (any_err & 1) return fail(RN_E_LOOKUP, "lookup index out of range on at least one chain");
  if (any_err & 2) return fail(RN_E_INVALID, "requirement failed: adapted mass matrix contains 0.0 (MassMatrix.scala:8,16)");
  return RN_OK;
}

// Trace.diagnostics (core/Trace.scala:11-21,49-121) over a device-resident sample block: per-chain sums and the
// cross-chain reductions on the device (rn_diag.cuh), the scalar epilogue here.  layout 0: [iterations][n][chains] (what
// rn_sampler_run writes), 1: [chains][iterations][n] (the caller-facing order).  out: host [n][2] = rHat, ess.
int rn_sampler_diagnostics(rn_sampler* s, const double* d_samples, int iterations, int layout, double* out) {
  if (!s || !d_samples || !out) return fail(RN_E_INVALID, "null argument");
  std::lock_guard<std::recursive_mutex> model_lock_(s->m->mu);
  if (s->chains < 2) return fail(RN_E_INVALID, "requirement failed: diagnostics requires multiple chains (Trace.scala:12)");
  if (iterations < 2) return fail(RN_E_INVALID, "diagnostics needs at least 2 iterations");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  const int n = (int)s->m->n_params, C = s->chains, I = iterations;
  const int L = std::min(100, I - 1);  // lags whose variogram has a non-empty sum; lag == I gives 0/0 (see epilogue)
  const size_t nC = (size_t)n * C, nblk = ((size_t)C + 127) / 128;
  const size_t n_q = 2 + (size_t)L;            // quantities reduced over chains: mean, variance, variogram(1..L)
  const size_t n_sums = (n_q + 1) * n;         // + squared deviations of the chain means
  // scratch: [mean per chain | per-block partials | sums | shift]
  const size_t need = (nC + n_q * n * nblk + n_sums + n) * 8;
  if (s->m->diag_bytes < need) {
    if (s->m->diag_scratch) A->cuMemFree(s->m->diag_scratch);
    s->m->diag_scratch = 0;
    s->m->diag_bytes = 0;
    CU(A->cuMemAlloc(&s->m->diag_scratch, need));
    s->m->diag_bytes = need;
  }
  CUdeviceptr d_mean = s->m->diag_scratch, d_part = d_mean + nC * 8, d_sums = d_part + n_q * n * nblk * 8, d_shift = d_sums + n_sums * 8;
  {
    CUdeviceptr src = (CUdeviceptr)(uintptr_t)d_samples;
    long long st, si, sc;
    if (layout == 0) {
      st = (long long)n * C, si = C, sc = 1;
    } else {
      st = n, si = 1, sc = (long long)I * n;
    }
    int I_ = I, n_ = n, C_ = C, L_ = L;
    const size_t smem = (size_t)I * 128 * 8;
    int use_smem = smem <= (size_t)200 * 1024 ? 1 : 0;
    if (use_smem) CU(A->cuFuncSetAttribute(s->K->k_diag_chain, 8 /*MAX_DYNAMIC_SHARED_SIZE_BYTES*/, (int)smem));
    void* params[] = {&src, &st, &si, &sc, &I_, &n_, &C_, &L_, &use_smem, &d_mean, &d_part};
    CU(A->cuLaunchKernel(s->K->k_diag_chain, (unsigned)nblk, (unsigned)n, 1, 128, 1, 1, use_smem ? (unsigned)smem : 0, s->stream, params,
                         nullptr));
    s->launches++;
  }
  auto reduce = [&](CUdeviceptr in, size_t rows, size_t cols, CUdeviceptr shift, CUdeviceptr outp) -> int {
    int C_ = (int)cols;
    void* params[] = {&in, &C_, &shift, &outp};
    CU(A->cuLaunchKernel(s->K->k_diag_reduce, (unsigned)rows, 1, 1, 256, 1, 1, 0, s->stream, params, nullptr));
    s->launches++;
    return RN_OK;
  };
  int rc = reduce(d_part, n_q * n, nblk, 0, d_sums);  // sums[q * n + i]
  if (rc) return rc;
  std::vector<double> sums(n_sums);
  CU(A->cuStreamSynchronize(s->stream));
  CU(A->cuMemcpyDtoH(sums.data(), d_sums, (size_t)n * 8));
  const double m = (double)C, nn = (double)I;
  std::vector<double> meanMean(n);
  for (int i = 0; i < n; i++) meanMean[i] = sums[i] / m;  // means.sum / m, Trace.scala:73
  CU(A->cuMemcpyHtoD(d_shift, meanMean.data(), (size_t)n * 8));
  rc = reduce(d_mean, n, (size_t)C, d_shift, d_sums + n_q * n * 8);
  if (rc) return rc;
  CU(A->cuStreamSynchronize(s->stream));
  CU(A->cuMemcpyDtoH(sums.data(), d_sums, n_sums * 8));
  for (int i = 0; i < n; i++) {
    const double b = (nn / (m - 1)) * sums[(2 + (size_t)L) * n + i];  // Trace.scala:75-77
    const double w = sums[n + i] / m;                                  // :88
    const double v = (nn - 1) / nn * w + b / nn;                       // :90-92
    const double rHat = std::sqrt(v / w);
    double acc = 0.0;
    for (int lag = 1;; lag++) {  // Trace.autocorrelation, :97-109 (tail recursion as a loop)
      double vt;
      if (lag <= L)
        vt = sums[(2 + (size_t)(lag - 1)) * n + i] / m;
      else if (lag == I)
        vt = std::nan("");  // variogram: 0.0 / 0
      else
        vt = -0.0;          // lag > trace.size: empty sum over a negative count
      const double pt = 1.0 - (vt / (2.0 * v));
      if (pt > 0.0 && lag < 100)
        acc += pt;
      else
        break;
    }
    out[2 * i] = rHat;
    out[2 * i + 1] = nn * m / (1 + (2 * acc));  // :60
  }
  return RN_OK;
}

// number of ncclAllReduce calls of the pooled warmup so far and their summed device time (stream must be idle: syncs)
int rn_sampler_comm_stats(rn_sampler* s, int64_t* calls, double* total_us) {
  if (!s) return fail(RN_E_INVALID, "null sampler");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  CU(A->cuCtxSetCurrent(s->m->ctx));
  CU(A->cuStreamSynchronize(s->stream));
  double us = 0.0;
  for (auto& pr : s->allreduce_events) {
    float ms = 0.f;
    CU(A->cuEventElapsedTime(&ms, pr.first, pr.second));
    us += (double)ms * 1e3;
  }
  if (calls) *calls = s->allreduce_calls;
  if (total_us) *total_us = us;
  return RN_OK;
}

int rn_sampler_set_comm(rn_sampler* s, rn_comm* comm) {
  s->comm = comm;
  return RN_OK;
}

void rn_sampler_destroy(rn_sampler* s) {
  if (!s) return;
  std::unique_lock<std::recursive_mutex> model_lock_(s->m->mu);
  std::string why;
  const Api* A = api(&why);
  if (A) {
    A->cuCtxSetCurrent(s->m->ctx);
    if (s->stream) {
      A->cuStreamSynchronize(s->stream);
      if (!s->m->spare_stream)
        s->m->spare_stream = s->stream;
      else
        A->cuStreamDestroy(s->stream);
    }
    if (s->arena) {
      if (s->arena_alloc > s->m->spare_arena_bytes) {  // keep the larger one as the model's spare
        if (s->m->spare_arena) A->cuMemFree(s->m->spare_arena);
        s->m->spare_arena = s->arena;
        s->m->spare_arena_bytes = s->arena_alloc;
      } else {
        A->cuMemFree(s->arena);
      }
    }
    if (s->d_trace) A->cuMemFree(s->d_trace);
    for (CUevent e : s->ev_run)
      if (e) A->cuEventDestroy(e);
    for (auto& pr : s->allreduce_events) {
      A->cuEventDestroy(pr.first);
      A->cuEventDestroy(pr.second);
    }
  }
  delete s;
}

// ---------------------------------------------------------------------------------------------------------
// rn_sample: Model.sample lowered to one call.  Host buffers in and out.
//
// Samples are produced chain-fastest ([iteration][n][chain], coalesced stores), re-laid on the device into the
// caller's [chain][iteration][n] order, and drained to the (pageable) caller buffer through a ring of pinned
// staging buffers: slice k's PCIe copy overlaps the host-side memcpy of slice k-1 (worker threads).
// ---------------------------------------------------------------------------------------------------------
}  // extern "C"

namespace {

// Page-locked host memory should live on the socket the GPU hangs off: a D2H copy into the far socket crosses the
// inter-socket link (measured on the B200 box: 57 vs 38 GB/s).  The driver allocates pinned pages in the calling
// thread's context, so a temporary MPOL_PREFERRED policy around cuMemAllocHost places them.  Best effort: any failure
// (single-socket box, no sysfs, seccomp) leaves the default policy.
int gpu_numa_node(const Api* A) {
  CUdevice dev;
  if (!A->cuCtxGetDevice || A->cuCtxGetDevice(&dev) != 0) return -1;
  char bus[32] = {0};
  if (!A->cuDeviceGetPCIBusId || A->cuDeviceGetPCIBusId(bus, (int)sizeof(bus), dev) != 0) return -1;
  for (char* p = bus; *p; p++) *p = (char)tolower(*p);
  std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
  FILE* f = fopen(path.c_str(), "r");
  if (!f) return -1;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}
struct NumaScope {
  bool set = false;
  explicit NumaScope(int node) {
    if (node < 0 || node >= 1024 || getenv("RN_NO_NUMA")) {
      if (getenv("RN_TIMING")) fprintf(stderr, "[rn numa] gpu node %d: default placement\n", node);
      return;
    }
    unsigned long mask[16] = {0};
    mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
    set = syscall(SYS_set_mempolicy, 1 /*MPOL_PREFERRED*/, mask, 1024ul + 1) == 0;
    if (getenv("RN_TIMING")) fprintf(stderr, "[rn numa] gpu node %d: set_mempolicy %s\n", node, set ? "ok" : "refused");
  }
  ~NumaScope() {
    if (set) syscall(SYS_set_mempolicy, 0 /*MPOL_DEFAULT*/, nullptr, 0ul);
  }
};

struct PinnedRing {  // process-wide, grown on demand, never freed (pinning is expensive)
  static constexpr int R = 6;
  void* buf[R] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  size_t bytes = 0;
  std::mutex mu;
};
PinnedRing g_ring;

// pinned staging slice -> caller's pageable pages with non-temporal stores: a plain memcpy of a 2 MB stripe stays below
// glibc's non-temporal threshold, so every destination line is first read (RFO) -- with the DMA engine writing the ring
// at PCIe rate at the same time that extra read stream is what saturates the socket's memory bandwidth
void copy_streaming(char* dst, const char* src, size_t n) {
#if defined(__x86_64__) && defined(__SSE2__)
  size_t head = (16 - ((uintptr_t)dst & 15)) & 15;
  if (head > n) head = n;
  if (head) std::memcpy(dst, src, head);
  dst += head, src += head, n -= head;
  size_t body = n & ~(size_t)63;
  for (size_t i = 0; i < body; i += 64) {
    const __m128i a = _mm_loadu_si128((const __m128i*)(src + i)), b = _mm_loadu_si128((const __m128i*)(src + i + 16)),
                  c = _mm_loadu_si128((const __m128i*)(src + i + 32)), d = _mm_loadu_si128((const __m128i*)(src + i + 48));
    _mm_stream_si128((__m128i*)(dst + i), a);
    _mm_stream_si128((__m128i*)(dst + i + 16), b);
    _mm_stream_si128((__m128i*)(dst + i + 32), c);
    _mm_stream_si128((__m128i*)(dst + i + 48), d);
  }
  _mm_sfence();
  if (n > body) std::memcpy(dst + body, src + body, n - body);
#else
  std::memcpy(dst, src, n);
#endif
}

class Workers {  // persistent job pool for the pinned->pageable memcpy of the drain
 public:
  explicit Workers(int n) {
    for (int i = 0; i < n; i++) th_.emplace_back([this] { loop(); });
  }
  ~Workers() {
    {
      std::lock_guard<std::mutex> lk(mu_);
      stop_ = true;
    }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  int size() const { return (int)th_.size(); }
  void submit(int group, std::function<void()> f) {
    {
      std::lock_guard<std::mutex> lk(mu_);
      pending_[group]++;
      q_.push_back({group, std::move(f)});
    }
    cv_.notify_one();
  }
  void wait(int group) {
    std::unique_lock<std::mutex> lk(mu_);
    done_.wait(lk, [&] { return pending_[group] == 0; });
  }

 private:
  void loop() {
    for (;;) {
      std::pair<int, std::function<void()>> job;
      {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
        if (q_.empty()) return;
        job = std::move(q_.front());
        q_.pop_front();
      }
      job.second();
      {
        std::lock_guard<std::mutex> lk(mu_);
        pending_[job.first]--;
      }
      done_.notify_all();
    }
  }
  std::vector<std::thread> th_;
  std::deque<std::pair<int, std::function<void()>>> q_;
  std::map<int, int> pending_;
  std::mutex mu_;
  std::condition_variable cv_, done_;
  bool stop_ = false;
};

Workers& drain_workers() {  // created on first use, lives for the process (thread start-up is not free per call)
  static Workers* w = [] {
    int t = (int)std::thread::hardware_concurrency() / 4;
    if (const char* e = getenv("LOCAL_WORLD_SIZE"))  // one process per GPU (torchrun): share the host's cores
      t /= std::max(1, atoi(e));
    if (const char* e = getenv("RN_DRAIN_THREADS")) t = atoi(e);
    return new Workers(std::max(2, std::min(t, 16)));
  }();
  return *w;
}

// true when [p, p+bytes) is page-locked memory the driver knows (rn_host_alloc, rn_host_register, cudaHostAlloc,
// cudaHostRegister by the caller): the DMA engine can then write the caller's buffer directly
bool host_is_pinned(const Api* A, const void* p, size_t bytes) {
  if (!p || !bytes || !A->cuPointerGetAttributes) return false;
  // cuPointerGetAttributes (plural) reports memory type 0 for plain pageable memory instead of failing, so probing a
  // caller's malloc'ed buffer does not raise a driver error (compute-sanitizer would count one per call)
  auto type_of = [&](const void* q) -> unsigned {
    unsigned mt = 0;
    int attr = 2 /*CU_POINTER_ATTRIBUTE_MEMORY_TYPE*/;
    void* data = &mt;
    if (A->cuPointerGetAttributes(1, &attr, &data, (CUdeviceptr)(uintptr_t)q) != 0) return 0;
    return mt;
  };
  return type_of(p) == CU_MEMORYTYPE_HOST && type_of((const char*)p + bytes - 1) == CU_MEMORYTYPE_HOST;
}

// device -> caller's host buffer.  Page-locked destination: one DMA, no staging.  Pageable destination: a ring of
// pinned staging slices; slice k's PCIe copy overlaps the fan-out memcpy of slices < k into the caller's pages.
int drain_to_host(const Api* A, CUstream copy, CUdeviceptr src, double* dst, size_t bytes, bool sync) {
  if (host_is_pinned(A, dst, bytes) && !getenv("RN_DRAIN_FORCE_STAGED")) {
    CU(A->cuMemcpyDtoHAsync(dst, src, bytes, copy));
    if (sync) CU(A->cuStreamSynchronize(copy));
    return RN_OK;
  }
  const size_t slice = (size_t)32 << 20;
  {
    std::lock_guard<std::mutex> lk(g_ring.mu);
    if (g_ring.bytes < slice) {
      NumaScope numa(gpu_numa_node(A));  // staging buffers on the GPU's socket
      for (int r = 0; r < PinnedRing::R; r++) {
        if (g_ring.buf[r]) continue;  // (kept from an earlier, partly failed attempt)
        const CUresult a = A->cuMemAllocHost(&g_ring.buf[r], slice);
        if (a != 0) {
          g_ring.buf[r] = nullptr;
          return cufail(A, a, "drain: cuMemAllocHost");  // the slots allocated so far stay in g_ring and are reused next time
        }
      }
      g_ring.bytes = slice;
    }
  }
  std::lock_guard<std::mutex> lk(g_ring.mu);  // one drain at a time per process
  Workers& pool = drain_workers();
  const int T = pool.size();
  constexpr int R = PinnedRing::R;
  CUevent ev[R] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  for (int r = 0; r < R; r++) {
    const CUresult e = A->cuEventCreate(&ev[r], 2);
    if (e != 0) {
      for (int q = 0; q < r; q++) A->cuEventDestroy(ev[q]);
      return cufail(A, e, "drain: cuEventCreate");
    }
  }
  const size_t n_slices = (bytes + slice - 1) / slice;
  // Each worker owns one stripe of every slice: it waits until slice k has landed in the ring (`ready`), copies its
  // stripe into the caller's pages and counts itself in done[k]; the DMA of slices k+1.. runs meanwhile.
  std::atomic<size_t> ready{0};
  std::vector<std::atomic<int>> done(n_slices);
  for (auto& d : done) d.store(0);
  std::atomic<bool> abort{false};
  for (int t = 0; t < T; t++) {
    pool.submit(0, [&, t] {
      for (size_t k = 0; k < n_slices; k++) {
        while (ready.load(std::memory_order_acquire) <= k) {
          if (abort.load()) return;
          std::this_thread::yield();
        }
        const size_t off = k * slice, len = std::min(slice, bytes - off);
        const size_t part = ((len / (size_t)T) + 4095) & ~(size_t)4095;
        const size_t o = (size_t)t * part;
        if (o < len) copy_streaming((char*)dst + off + o, (const char*)g_ring.buf[k % R] + o, std::min(part, len - o));
        done[k].fetch_add(1, std::memory_order_release);
      }
    });
  }
  auto fail_out = [&](int rc) {
    abort.store(true);
    pool.wait(0);
    for (int r = 0; r < R; r++) A->cuEventDestroy(ev[r]);
    return rc;
  };
  const size_t ahead = R - 1;
  size_t issued = 0, landed = 0;
  while (landed < n_slices) {
    while (issued < n_slices && issued < landed + ahead) {
      if (issued >= (size_t)R)  // the slot's previous slice must be fully copied out
        while (done[issued - R].load(std::memory_order_acquire) < T) std::this_thread::yield();
      const size_t off = issued * slice, len = std::min(slice, bytes - off);
      CUresult r1 = A->cuMemcpyDtoHAsync(g_ring.buf[issued % R], src + off, len, copy);
      if (r1 == 0) r1 = A->cuEventRecord(ev[issued % R], copy);
      if (r1 != 0) return fail_out(cufail(A, r1, "drain: cuMemcpyDtoHAsync"));
      issued++;
    }
    CUresult r2 = A->cuEventSynchronize(ev[landed % R]);
    if (r2 != 0) return fail_out(cufail(A, r2, "drain: cuEventSynchronize"));
    ready.store(++landed, std::memory_order_release);
  }
  pool.wait(0);
  for (int r = 0; r < R; r++) A->cuEventDestroy(ev[r]);
  (void)sync;
  return RN_OK;
}

}  // namespace

extern "C" {

int rn_sample(rn_model* m, const rn_config* cfg, const int64_t* seeds, int chains, double* samples, double* mass,
              rn_chain_stats* stats) {
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  const bool timing = getenv("RN_TIMING") != nullptr;
  auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  double t0 = now();
  auto lap = [&](const char* what) {
    if (!timing) return;
    double t1 = now();
    fprintf(stderr, "[rn_sample] %-18s %8.2f ms\n", what, (t1 - t0) * 1e3);
    t0 = t1;
  };
  rn_sampler* s = nullptr;
  int rc = rn_sampler_create(m, cfg, seeds, chains, &s);
  if (rc) return rc;
  lap("sampler_create");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  struct Guard {
    rn_sampler* s;
    const Api* A;
    CUdeviceptr b[2] = {0, 0};
    CUstream copy = nullptr;
    CUevent done = nullptr;
    bool timing = false;
    ~Guard() {
      auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
      const double t0 = now();
      if (done) A->cuEventDestroy(done);
      if (copy) A->cuStreamDestroy(copy);
      rn_sampler_destroy(s);
      if (timing) fprintf(stderr, "[rn_sample] %-18s %8.2f ms\n", "teardown", (now() - t0) * 1e3);
    }
  } g{s, A};
  g.timing = timing;
  rc = rn_sampler_warmup(s, -1);
  if (rc) return rc;
  if (timing) rn_sampler_sync(s);
  lap("warmup");
  const size_t C = (size_t)chains, n = m->n_params, I = (size_t)cfg->iterations;
  rc = rn_sampler_run(s, 0, nullptr);  // lf.resetStats() after warmup even when no iteration follows (Driver.scala:31)
  if (rc) return rc;
  if (I > 0 && !samples && cfg->diagnostics) {
    // summaries only: the samples stay on the device ([iterations][n][chains], as the kernels write them) and
    // Trace.diagnostics is reduced there
    const size_t want = I * n * C * 8;
    if (m->pool_bytes[0] < want) {
      if (m->pool[0]) A->cuMemFree(m->pool[0]);
      m->pool[0] = 0;
      m->pool_bytes[0] = 0;
      CU(A->cuMemAlloc(&m->pool[0], want));
      m->pool_bytes[0] = want;
    }
    rc = rn_sampler_run(s, (int)I, (double*)(uintptr_t)m->pool[0]);
    if (rc) return rc;
    rc = rn_sampler_diagnostics(s, (const double*)(uintptr_t)m->pool[0], (int)I, 0, cfg->diagnostics);
    if (rc) return rc;
  } else if (I > 0 && samples) {
    const size_t total = C * I * n * 8;
    // the whole [C][I][n] result stays on the device while it is produced; runs larger than the cap are cut into
    // passes over the iteration axis (each pass drained with a strided copy)
    size_t cap = (size_t)32 << 30;
    if (const char* e = getenv("RN_SAMPLE_DEVICE_CAP_MB")) cap = (size_t)atoll(e) << 20;
    const size_t pass_iters = std::max<size_t>(1, std::min<size_t>(I, cap / std::max<size_t>(1, C * n * 8)));
    size_t chunk = std::max<size_t>(1, std::min<size_t>(pass_iters, ((size_t)1 << 30) / (n * C * 8 + 1)));
    if (cfg->launch_iterations > 0) chunk = std::min<size_t>(chunk, (size_t)cfg->launch_iterations);
    const size_t want[2] = {chunk * n * C * 8 /* [chunk][n][C] scratch */, pass_iters * n * C * 8 /* [C][pass_iters][n] */};
    for (int k = 0; k < 2; k++) {
      if (m->pool_bytes[k] < want[k]) {
        if (m->pool[k]) A->cuMemFree(m->pool[k]);
        m->pool[k] = 0;
        m->pool_bytes[k] = 0;
        CU(A->cuMemAlloc(&m->pool[k], want[k]));
        m->pool_bytes[k] = want[k];
      }
      g.b[k] = m->pool[k];
    }
    CU(A->cuStreamCreate(&g.copy, 1));
    CU(A->cuEventCreate(&g.done, 2));
    auto transpose = [&](CUdeviceptr src, CUdeviceptr dst, size_t k, size_t cols, size_t pi, size_t done) -> int {
      int rows = (int)(k * n), ncols = (int)cols;
      long long src_ld = (long long)C, ld = (long long)(pi * n), off = (long long)(done * n);
      void* params[] = {&src, &dst, &rows, &ncols, &src_ld, &ld, &off};
      CU(A->cuLaunchKernel(s->K->k_transpose, (unsigned)((ncols + 31) / 32), (unsigned)((rows + 31) / 32), 1, 32, 8, 1, 0, s->stream,
                           params, nullptr));
      s->launches++;
      return RN_OK;
    };
    if (pass_iters == I) {
      // Everything fits on the device.  The chains are cut into blocks: block b runs all its iterations and is
      // re-laid into the caller's [chain][iteration][n] order, then its (contiguous) slab starts crossing PCIe while
      // block b+1 computes -- the copy, not the kernel, is the long pole of this call.
      rc = rn_sampler_run(s, 0, nullptr);  // initialize + lf.resetStats() (Driver.scala:31), no iterations
      if (rc) return rc;
      size_t blocks = std::min<size_t>(8, C / 32768);
      if (total < ((size_t)64 << 20)) blocks = 1;
      if (const char* e = getenv("RN_SAMPLE_BLOCKS")) blocks = (size_t)atoll(e);
      blocks = std::max<size_t>(1, std::min(blocks, C));
      // geometric ramp (1/16, 1/16, 1/8, 1/4, 1/2 of the chains for >= 4 blocks): the first slab reaches the copy
      // engine after a fraction of a millisecond, later blocks keep the SMs full
      std::vector<std::pair<size_t, size_t>> ranges;
      if (blocks >= 4 && C >= 16 * 1024) {
        const size_t unit = ((C / 16) + 1023) & ~(size_t)1023;
        const size_t mult[5] = {1, 1, 2, 4, 8};
        size_t c0 = 0;
        for (int k = 0; k < 5 && c0 < C; k++) {
          const size_t c1 = (k == 4) ? C : std::min(C, c0 + mult[k] * unit);
          ranges.push_back({c0, c1});
          c0 = c1;
        }
      } else {
        const size_t per = (((C + blocks - 1) / blocks) + 1023) & ~(size_t)1023;
        for (size_t c0 = 0; c0 < C; c0 += per) ranges.push_back({c0, std::min(C, c0 + per)});
      }
      std::vector<CUevent> evs(ranges.size(), nullptr);
      struct EvGuard {
        const Api* A;
        std::vector<CUevent>& e;
        ~EvGuard() {
          for (CUevent x : e)
            if (x) A->cuEventDestroy(x);
        }
      } evg{A, evs};
      for (size_t bi = 0; bi < ranges.size(); bi++) {
        const size_t c0 = ranges[bi].first, c1 = ranges[bi].second;
        for (size_t done = 0; done < I;) {
          const size_t k = std::min(chunk, I - done);
          rc = run_phase(A, s, 1, (int)k, (double*)(uintptr_t)g.b[0], (int)c0, (int)c1);
          if (rc) return rc;
          rc = transpose(g.b[0] + c0 * 8, g.b[1] + c0 * I * n * 8, k, c1 - c0, I, done);
          if (rc) return rc;
          done += k;
        }
        CU(A->cuEventCreate(&evs[bi], 2));
        CU(A->cuEventRecord(evs[bi], s->stream));
      }
      if (timing) {
        rn_sampler_sync(s);
        lap("kernels");
      }
      for (size_t bi = 0; bi < ranges.size(); bi++) {
        const size_t c0 = ranges[bi].first, c1 = ranges[bi].second;
        CU(A->cuStreamWaitEvent(g.copy, evs[bi], 0));
        rc = drain_to_host(A, g.copy, g.b[1] + c0 * I * n * 8, samples + c0 * I * n, (c1 - c0) * I * n * 8,
                           /*sync=*/bi + 1 == ranges.size());
        if (rc) return rc;
      }
      if (cfg->diagnostics) {  // the [chain][iteration][n] block is still resident
        rc = rn_sampler_diagnostics(s, (const double*)(uintptr_t)g.b[1], (int)I, 1, cfg->diagnostics);
        if (rc) return rc;
      }
    } else {
      if (cfg->diagnostics) return fail(RN_E_UNSUPPORTED, "diagnostics need the whole sample block on the device (raise RN_SAMPLE_DEVICE_CAP_MB)");
      for (size_t p0 = 0; p0 < I; p0 += pass_iters) {  // strided passes over the iteration axis
        const size_t pi = std::min(pass_iters, I - p0);
        for (size_t done = 0; done < pi;) {
          const size_t k = std::min(chunk, pi - done);
          rc = rn_sampler_run(s, (int)k, (double*)(uintptr_t)g.b[0]);
          if (rc) return rc;
          rc = transpose(g.b[0], g.b[1], k, C, pi, done);
          if (rc) return rc;
          done += k;
        }
        CU(A->cuEventRecord(g.done, s->stream));
        CU(A->cuStreamWaitEvent(g.copy, g.done, 0));
        CUDA_MEMCPY2D cp;  // rows of pi*n doubles into a pitch of I*n
        std::memset(&cp, 0, sizeof(cp));
        cp.srcMemoryType = CU_MEMORYTYPE_DEVICE;
        cp.srcDevice = g.b[1];
        cp.srcPitch = pi * n * 8;
        cp.dstMemoryType = CU_MEMORYTYPE_HOST;
        cp.dstHost = samples + p0 * n;
        cp.dstPitch = I * n * 8;
        cp.WidthInBytes = pi * n * 8;
        cp.Height = C;
        CU(A->cuMemcpy2DAsync(&cp, g.copy));
        CU(A->cuStreamSynchronize(g.copy));
      }
    }
  } else if (I > 0) {
    rc = rn_sampler_run(s, (int)I, nullptr);
    if (rc) return rc;
  }
  lap("drain");
  rc = rn_sampler_stats(s, stats, mass, cfg->stats_rings);
  lap("stats");
  return rc;
}

// ---------------------------------------------------------------------------------------------------------
// page-locked host buffers for the caller (the JVM side wraps them as direct ByteBuffers): rn_sample DMAs straight
// into such a buffer instead of staging through the pinned ring
// ---------------------------------------------------------------------------------------------------------
int rn_host_alloc(int device, size_t bytes, void** out) {
  if (!out || !bytes) return fail(RN_E_INVALID, "bad argument");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = host_ctx(A, device);
  if (rc) return rc;
  NumaScope numa(gpu_numa_node(A));
  CU(A->cuMemAllocHost(out, bytes));
  return RN_OK;
}
int rn_host_free(int device, void* p) {
  if (!p) return RN_OK;
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = host_ctx(A, device);
  if (rc) return rc;
  CU(A->cuMemFreeHost(p));
  return RN_OK;
}
int rn_host_register(int device, void* p, size_t bytes) {
  if (!p || !bytes) return fail(RN_E_INVALID, "bad argument");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = host_ctx(A, device);
  if (rc) return rc;
  CU(A->cuMemHostRegister(p, bytes, 1 /*CU_MEMHOSTREGISTER_PORTABLE*/));
  return RN_OK;
}
int rn_host_unregister(int device, void* p) {
  if (!p) return RN_OK;
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = host_ctx(A, device);
  if (rc) return rc;
  CU(A->cuMemHostUnregister(p));
  return RN_OK;
}

// ---------------------------------------------------------------------------------------------------------
// communicator (NCCL); the unique id is exchanged by the caller (e.g. torch.distributed broadcast of 128 bytes)
// ---------------------------------------------------------------------------------------------------------
int rn_comm_unique_id(char id[128]) {
  std::string why;
  const Nccl* N = nccl(&why);
  if (!N) return fail(RN_E_NCCL, why);
  NcclId u;
  int r = N->GetUniqueId(&u);
  if (r != 0) return fail(RN_E_NCCL, "ncclGetUniqueId failed");
  std::memcpy(id, u.b, 128);
  return RN_OK;
}
int rn_comm_create(const char id[128], int rank, int world, int device, rn_comm** out) {
  std::string why;
  const Nccl* N = nccl(&why);
  if (!N) return fail(RN_E_NCCL, why);
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  std::unique_ptr<rn_comm> c(new rn_comm());
  c->rank = rank;
  c->world = world;
  c->device = device;
  CUdevice dev;
  CU(A->cuDeviceGet(&dev, device));
  CU(A->cuDevicePrimaryCtxRetain(&c->ctx, dev));
  CU(A->cuCtxSetCurrent(c->ctx));
  NcclId u;
  std::memcpy(u.b, id, 128);
  int r = N->CommInitRank(&c->comm, world, u, rank);
  if (r != 0) return fail(RN_E_NCCL, std::string("ncclCommInitRank: ") + (N->GetErrorString ? N->GetErrorString(r) : "?"));
  *out = c.release();
  return RN_OK;
}
void rn_comm_destroy(rn_comm* c) {
  if (!c) return;
  std::string why;
  const Nccl* N = nccl(&why);
  if (N && c->comm) N->CommDestroy(c->comm);
  const Api* A = api(&why);
  if (A && c->ctx) {
    CUdevice dev;
    if (A->cuDeviceGet(&dev, c->device) == 0) A->cuDevicePrimaryCtxRelease(dev);
  }
  delete c;
}
}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// rn_function: the OTHER compile seam -- Compiler.compile(inputs, outputs): ir.CompiledFunction
// (rainier-compute/.../compute/Compiler.scala:22-30) -- batched over posterior draws.  Generator.prepare
// (rainier-core/.../core/Generator.scala:59-94) compiles a generator's "requirements" with it and Trace.predict
// (core/Trace.scala:34-41) evaluates them once per draw through CompiledFunction.output; here one launch of rn_k_eval
// (rn_function.cuh) evaluates all m requirements of all draws, reading the draws where rn_sampler_run left them.
// ---------------------------------------------------------------------------------------------------------
struct rn_function {
  std::vector<uint8_t> rir;
  Program prog;
  bool fast = false;
  int device = -1;
  CUcontext ctx = nullptr;
  std::string source;
  std::vector<char> cubin;
  CUmodule mod = nullptr;
  CUfunction k_eval = nullptr, k_reduce = nullptr;
  CUstream stream = nullptr;
  CUstream stream2 = nullptr;  // second staging slot of rn_function_eval (host buffers)
  CUdeviceptr d_err = 0;
  CUdeviceptr scratch = 0;  // grow-only staging of rn_function_eval (host buffers)
  size_t scratch_bytes = 0;
  int sm_count = 148;
  int64_t launches = 0;
};

// NVRTC: source -> sm_100a cubin (the function and optimizer flavours; get_kernel keeps its own copy with the cubin cache)
static int nvrtc_to_cubin(const std::string& source, const char* name, bool fast, std::vector<char>& cubin) {
  std::vector<const char*> opts = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo"};
  opts.push_back(fast ? "--fmad=true" : "--fmad=false");
  nvrtcProgram prog;
  if (nvrtcCreateProgram(&prog, source.c_str(), name, 0, nullptr, nullptr) != NVRTC_SUCCESS)
    return fail(RN_E_COMPILE, "nvrtcCreateProgram failed");
  nvrtcResult r = nvrtcCompileProgram(prog, (int)opts.size(), opts.data());
  if (r != NVRTC_SUCCESS) {
    size_t n = 0;
    nvrtcGetProgramLogSize(prog, &n);
    std::string log(n, '\0');
    nvrtcGetProgramLog(prog, &log[0]);
    nvrtcDestroyProgram(&prog);
    return fail(RN_E_COMPILE, std::string("NVRTC: ") + nvrtcGetErrorString(r) + "\n" + log);
  }
  size_t n = 0;
  nvrtcGetCUBINSize(prog, &n);
  cubin.resize(n);
  nvrtcGetCUBIN(prog, cubin.data());
  nvrtcDestroyProgram(&prog);
  return RN_OK;
}

static int function_compile(rn_function* f) {
  if (!f->cubin.empty()) return RN_OK;
  return nvrtc_to_cubin(f->source, "rainier_function.cu", f->fast, f->cubin);
}

static int function_load(const Api* A, rn_function* f) {
  CU(A->cuCtxSetCurrent(f->ctx));
  if (f->mod) return RN_OK;
  int rc = function_compile(f);
  if (rc) return rc;
  CU(A->cuModuleLoadData(&f->mod, f->cubin.data()));
  CU(A->cuModuleGetFunction(&f->k_eval, f->mod, "rn_k_eval"));
  CU(A->cuModuleGetFunction(&f->k_reduce, f->mod, "rn_k_reduce_rows"));
  CU(A->cuStreamCreate(&f->stream, 1 /*CU_STREAM_NON_BLOCKING*/));
  CU(A->cuMemAlloc(&f->d_err, 8));
  CU(A->cuMemsetD8Async(f->d_err, 0, 8, f->stream));
  CU(A->cuStreamSynchronize(f->stream));  // evaluations may be enqueued on a caller's stream
  CUdevice dev;
  int sms = 0;
  if (A->cuDeviceGet(&dev, f->device) == 0 && A->cuDeviceGetAttribute(&sms, 16 /*MULTIPROCESSOR_COUNT*/, dev) == 0 && sms > 0)
    f->sm_count = sms;
  return RN_OK;
}

// one launch; grid = a multiple of the SM count (grid-stride loop), 128 threads per CTA
static int function_launch(const Api* A, rn_function* f, const RnEvalArgs& args, CUstream st) {
  RnEvalArgs a = args;
  a.err = (int*)(uintptr_t)f->d_err;
  const long long ctas_needed = (a.count + 127) / 128;
  const long long cap = (long long)f->sm_count * 16;
  const unsigned grid = (unsigned)std::max<long long>(1, std::min(ctas_needed, cap));
  void* params[] = {&a};
  CU(A->cuLaunchKernel(f->k_eval, grid, 1, 1, 128, 1, 1, 0, st, params, nullptr));
  f->launches++;
  return RN_OK;
}

// the row sums of an inlinable target's column-only monomials, on the device (rn_inline.hpp step 2): rn_k_eval over the
// target's tile-major block in place (one thread per row; values written [monomial][row]) and rn_k_reduce_rows (one block
// per monomial, fixed order), in chunks of rows
static int device_inline(rn_model* M, const InlinePlan& plan, std::vector<uint8_t>& new_rir) {
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  std::vector<std::vector<double>> sums(plan.inl.size());
  for (size_t k = 0; k < plan.inl.size(); k++) {
    const InlineTarget& I = plan.inl[k];
    const rir_target& T = plan.targets[I.target].t;
    const size_t m = I.monos.size();
    sums[k].assign(m, 0.0);
    if (m == 0) continue;
    const std::vector<uint8_t> frir = inline_function_rir(plan, k);
    rn_function* f = nullptr;
    int rc = rn_function_create(frir.data(), frir.size(), M->device, RN_MATH_PARITY, &f);
    if (rc) return rc;
    struct Done {
      rn_function* f;
      const Api* A;
      CUdeviceptr a = 0, b = 0;
      ~Done() {
        if (a) A->cuMemFree(a);
        if (b) A->cuMemFree(b);
        rn_function_destroy(f);
      }
    } g{f, A};
    rc = function_load(A, f);
    if (rc) return rc;
    const long long pitch = M->target_pitch[I.target], ncols = T.n_cols, rows = (long long)T.n_rows;
    const long long chunk = std::min<long long>((rows + 31) / 32 * 32, std::max<long long>(32, (((long long)64 << 20) / (long long)(m * 8)) / 32 * 32));
    CU(A->cuMemAlloc(&g.a, (size_t)chunk * m * 8));
    CU(A->cuMemAlloc(&g.b, m * 8));
    CU(A->cuMemsetD8Async(g.b, 0, m * 8, f->stream));
    for (long long r0 = 0; r0 < rows; r0 += chunk) {
      const long long cnt = std::min(chunk, rows - r0);
      RnEvalArgs a;
      std::memset(&a, 0, sizeof(a));
      a.x = (const double*)(uintptr_t)(M->d_data + (M->target_base[I.target] + (uint64_t)(r0 / 32) * (uint64_t)(ncols * pitch)) * 8);
      a.out = (double*)(uintptr_t)g.a;
      a.count = cnt;
      a.in_inner = 32, a.in_outer = ncols * pitch, a.in_pstride = 1, a.in_estride = pitch;  // row p of the tile-major block
      a.out_inner = cnt, a.out_outer = 0, a.out_pstride = 1, a.out_estride = cnt;           // [monomial][row]
      rc = function_launch(A, f, a, f->stream);
      if (rc) return rc;
      long long cn = cnt;
      int mi = (int)m;
      CUdeviceptr vals = g.a, sm = g.b;
      void* params[] = {&vals, &cn, &mi, &sm};
      CU(A->cuLaunchKernel(f->k_reduce, (unsigned)m, 1, 1, 256, 1, 1, 0, f->stream, params, nullptr));
      f->launches++;
    }
    rc = rn_function_sync(f);
    if (rc) return rc;
    CU(A->cuMemcpyDtoH(sums[k].data(), g.b, m * 8));
  }
  new_rir = apply_inline(plan, sums);
  return RN_OK;
}

extern "C" {

int rn_function_create(const void* rir, size_t len, int device, int math_mode, rn_function** out) {
  if (!rir || !out) return fail(RN_E_INVALID, "null argument");
  std::unique_ptr<rn_function> f(new rn_function());
  f->rir.assign((const uint8_t*)rir, (const uint8_t*)rir + len);
  std::string e = build_function(rir, len, f->prog);
  if (!e.empty()) return fail(RN_E_INVALID, e);
  f->fast = math_mode == RN_MATH_FAST;
  EmitOptions eo;
  eo.fast_math = f->fast;
  f->source = emit_function_source(f->prog, eo);
  f->device = device;
  if (device >= 0) {
    std::string why;
    const Api* A = api(&why);
    if (!A) return fail(RN_E_CUDA, why);
    int rc = host_ctx(A, device);
    if (rc) return rc;
    CUdevice dev;
    CU(A->cuDeviceGet(&dev, device));
    CU(A->cuDevicePrimaryCtxRetain(&f->ctx, dev));
  }
  *out = f.release();
  return RN_OK;
}

int rn_function_ninputs(const rn_function* f) { return f ? (int)f->prog.n_params : RN_E_INVALID; }
int rn_function_noutputs(const rn_function* f) { return f ? (int)f->prog.fn_outputs.size() : RN_E_INVALID; }
int64_t rn_function_launches(const rn_function* f) { return f ? f->launches : 0; }
void* rn_function_stream(rn_function* f) { return f ? (void*)f->stream : nullptr; }

int rn_function_emit_source(rn_function* f, char* buf, size_t cap, size_t* needed) {
  if (!f) return fail(RN_E_INVALID, "null function");
  if (needed) *needed = f->source.size() + 1;
  if (buf && cap) {
    size_t n = std::min(cap - 1, f->source.size());
    std::memcpy(buf, f->source.data(), n);
    buf[n] = 0;
  }
  return RN_OK;
}

int rn_function_emit_cubin(rn_function* f, void* buf, size_t cap, size_t* needed) {
  if (!f) return fail(RN_E_INVALID, "null function");
  int rc = function_compile(f);
  if (rc) return rc;
  if (needed) *needed = f->cubin.size();
  if (buf && cap) std::memcpy(buf, f->cubin.data(), std::min(cap, f->cubin.size()));
  return RN_OK;
}

// op counts of one point: out = [fp64 flops, transcendental calls]
int rn_function_op_counts(const rn_function* f, double out[2]) {
  if (!f || !out) return fail(RN_E_INVALID, "null argument");
  out[0] = f->prog.counts.flops_inv;
  out[1] = f->prog.counts.special_inv;
  return RN_OK;
}

int rn_function_eval_device(rn_function* f, const double* d_x, int layout, int64_t iterations, int64_t chains, double* d_out,
                            void* stream) {
  if (!f || !d_out || iterations < 0 || chains < 0) return fail(RN_E_INVALID, "bad argument");
  if (f->device < 0) return fail(RN_E_CUDA, "function was created without a device (no CPU fallback)");
  const long long n = (long long)f->prog.n_params, m = (long long)f->prog.fn_outputs.size();
  if (!d_x && n > 0) return fail(RN_E_INVALID, "null input");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = function_load(A, f);
  if (rc) return rc;
  const long long count = (long long)iterations * (long long)chains;
  if (count == 0) return RN_OK;
  RnEvalArgs a;
  std::memset(&a, 0, sizeof(a));
  a.x = d_x;
  a.out = d_out;
  a.count = count;
  if (layout == RN_LAYOUT_SAMPLER) {
    // in [iteration][n][chain] (rn_sampler_run) -> out [chain][iteration][m] (Trace.predict's order: chains.flatMap(_.map(fn)))
    a.in_inner = chains, a.in_outer = n * chains, a.in_pstride = 1, a.in_estride = chains;
    a.out_inner = chains, a.out_outer = m, a.out_pstride = (long long)iterations * m, a.out_estride = 1;
  } else if (layout == RN_LAYOUT_ROWS) {
    // in [count][n] -> out [count][m]
    a.in_inner = count, a.in_outer = 0, a.in_pstride = n, a.in_estride = 1;
    a.out_inner = count, a.out_outer = 0, a.out_pstride = m, a.out_estride = 1;
  } else {
    return fail(RN_E_INVALID, "unknown layout");
  }
  return function_launch(A, f, a, stream ? (CUstream)stream : f->stream);
}

int rn_function_sync(rn_function* f) {
  if (!f) return fail(RN_E_INVALID, "null function");
  if (f->device < 0) return fail(RN_E_CUDA, "function was created without a device (no CPU fallback)");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  if (!f->mod) return RN_OK;
  CU(A->cuCtxSetCurrent(f->ctx));
  CU(A->cuStreamSynchronize(f->stream));
  int err = 0;
  CU(A->cuMemcpyDtoH(&err, f->d_err, 4));
  if (err) {
    CU(A->cuMemsetD8Async(f->d_err, 0, 8, f->stream));
    CU(A->cuStreamSynchronize(f->stream));
    if (err & 1) return fail(RN_E_LOOKUP, "lookup index out of range");
  }
  return RN_OK;
}

int rn_function_eval(rn_function* f, const double* x, int64_t count, double* out) {
  if (!f || !out || count < 0) return fail(RN_E_INVALID, "bad argument");
  if (f->device < 0) return fail(RN_E_CUDA, "function was created without a device (no CPU fallback)");
  const size_t n = f->prog.n_params, m = f->prog.fn_outputs.size();
  if (!x && n > 0 && count > 0) return fail(RN_E_INVALID, "null input");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  int rc = function_load(A, f);
  if (rc) return rc;
  if (count == 0) return RN_OK;
  // Two staging slots, each with its own stream: chunk i is copied in, evaluated and copied out on stream i&1, so the
  // host->device copy of one chunk overlaps the device->host copy of the previous one (PCIe is full duplex) and the
  // kernel hides under both.  In-order streams make slot reuse safe without events.  [chunk][n] in, [chunk][m] out.
  const size_t per_point = (n + m) * 8;
  const int64_t chunk_max = std::max<int64_t>(1, (int64_t)((size_t)32 << 20) / (int64_t)per_point);
  const int64_t chunk = std::min<int64_t>(count, chunk_max);
  const size_t x_bytes = ((size_t)chunk * n * 8 + 255) & ~(size_t)255, slot_bytes = x_bytes + (((size_t)chunk * m * 8 + 255) & ~(size_t)255);
  const int slots = count > chunk ? 2 : 1;
  const size_t need = slot_bytes * (size_t)slots;
  if (f->scratch_bytes < need) {
    if (f->scratch) A->cuMemFree(f->scratch);
    f->scratch = 0;
    f->scratch_bytes = 0;
    CU(A->cuMemAlloc(&f->scratch, need));
    f->scratch_bytes = need;
  }
  if (slots == 2 && !f->stream2) CU(A->cuStreamCreate(&f->stream2, 1 /*CU_STREAM_NON_BLOCKING*/));
  int64_t i = 0;
  for (int64_t p0 = 0; p0 < count; p0 += chunk, i++) {
    const int64_t c = std::min<int64_t>(chunk, count - p0);
    const CUstream st = (i & 1) ? f->stream2 : f->stream;
    const CUdeviceptr d_x = f->scratch + (size_t)(i & 1) * slot_bytes, d_out = d_x + x_bytes;
    if (n > 0) CU(A->cuMemcpyHtoDAsync(d_x, x + (size_t)p0 * n, (size_t)c * n * 8, st));
    rc = rn_function_eval_device(f, (const double*)(uintptr_t)d_x, RN_LAYOUT_ROWS, 1, c, (double*)(uintptr_t)d_out, (void*)st);
    if (rc) return rc;
    CU(A->cuMemcpyDtoHAsync(out + (size_t)p0 * m, d_out, (size_t)c * m * 8, st));
  }
  if (f->stream2) CU(A->cuStreamSynchronize(f->stream2));
  return rn_function_sync(f);
}

void rn_function_destroy(rn_function* f) {
  if (!f) return;
  std::string why;
  const Api* A = f->device >= 0 ? api(&why) : nullptr;
  if (A && f->ctx) {
    A->cuCtxSetCurrent(f->ctx);
    if (f->stream) {
      A->cuStreamSynchronize(f->stream);
      A->cuStreamDestroy(f->stream);
    }
    if (f->stream2) {
      A->cuStreamSynchronize(f->stream2);
      A->cuStreamDestroy(f->stream2);
    }
    if (f->mod) A->cuModuleUnload(f->mod);
    if (f->d_err) A->cuMemFree(f->d_err);
    if (f->scratch) A->cuMemFree(f->scratch);
    CUdevice dev;
    if (A->cuDeviceGet(&dev, f->device) == 0) A->cuDevicePrimaryCtxRelease(dev);
  }
  delete f;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// rn_optimize: Optimizer.lbfgs (rainier-sampler/.../optimizer/Optimizer.scala:6-24) for a batch of starts, fused into
// one kernel (rn_optimizer.cuh).  Model.optimize (rainier-core/.../core/Model.scala:26-30) = start 0 of a batch whose
// x0 is NULL.
// ---------------------------------------------------------------------------------------------------------
static int get_opt_kernel(rn_model* m, const rn_optimize_config* oc, rn_model::OptKernel** out) {
  const bool fast = oc && oc->math_mode == RN_MATH_FAST;
  const int gm = oc ? oc->gradient_mode : RN_GRAD_AUTO;
  const bool adjoint = (gm == RN_GRAD_ADJOINT) || !m->rir_has_gradient;
  const int history = oc && oc->history > 0 ? oc->history : 5;
  if (history > 64) return fail(RN_E_INVALID, "L-BFGS history too long");
  // shape: like the samplers -- a warp per start when rows are streamed in earnest or the state is large
  int want = oc ? oc->backend : RN_BACKEND_AUTO;
  if (const char* e = getenv("RN_BACKEND")) want = atoi(e);
  if (want == RN_BACKEND_AUTO) want = key_for(m, nullptr).backend == 1 ? RN_BACKEND_WARP : RN_BACKEND_THREAD;
  const int backend = want == RN_BACKEND_WARP ? 1 : 0;
  auto key = std::make_tuple(adjoint, fast, history, backend);
  auto it = m->opt_kernels.find(key);
  if (it != m->opt_kernels.end()) {
    *out = it->second.get();
    return RN_OK;
  }
  const Program* P = nullptr;
  int rc = get_program(m, adjoint, fast, &P);
  if (rc) return rc;
  std::unique_ptr<rn_model::OptKernel> K(new rn_model::OptKernel());
  K->backend = backend;
  EmitOptions eo;
  eo.backend = backend;
  eo.fast_math = fast;
  eo.target_base = m->target_base;
  eo.target_pitch = m->target_pitch;
  const uint64_t lb_w = (uint64_t)P->n_params * (2 * (uint64_t)history + 1) + 2 * (uint64_t)history;
  if (backend == 0) {
    // the whole optimisation state of a start is thread-local: x, g, diag and the 2m-vector history
    if ((uint64_t)P->n_params * (2 * (uint64_t)history + 4) > 4096)
      return fail(RN_E_UNSUPPORTED, "rn_optimize (thread per start) keeps n*(2m+4) doubles per start in thread-local memory; use RN_BACKEND_WARP");
  } else {
    if (P->symbolic && P->n_params > 96)
      return fail(RN_E_UNSUPPORTED, "warp-per-start with a symbolic gradient keeps n+1 accumulators in registers; use RN_GRAD_ADJOINT for n > 96");
    eo.tma_stages = 0;
    eo.enable_ehmc = false;
    const uint64_t cap = (227 * 1024 - 2048) / 8;
    // warps per start: one, unless the start's shared-memory state is so large that fewer than 16 starts fit an SM (same
    // rule as the samplers, rn_runtime.cpp:get_kernel)
    int k = 1;
    {
      eo.wpc_k = 1;
      const uint64_t one = 4ull * P->n_params + (uint64_t)wpc_sizes(*P, eo).scratch_doubles + lb_w + 1;
      if (one > cap) return fail(RN_E_UNSUPPORTED, "rn_optimize: the L-BFGS history of one start does not fit shared memory");
      const uint64_t fit = std::max<uint64_t>(1, cap / one);
      while (k < 8 && fit * (uint64_t)k < 16) k *= 2;
      if (const char* e = getenv("RN_WPC_K")) k = std::max(1, std::min(8, atoi(e)));
      if (k != 1 && k != 2 && k != 4 && k != 8) k = 1;
    }
    eo.wpc_k = k;
    const WpcSizes z = wpc_sizes(*P, eo);  // RN_OPT_SMEM_DOUBLES (rn_optimizer.cuh): 4n (x, gradient, g, diag) + history + density scratch + k
    const uint64_t per_start = 4ull * P->n_params + (uint64_t)z.scratch_doubles + lb_w + (uint64_t)k;
    if (per_start > cap) return fail(RN_E_UNSUPPORTED, "rn_optimize: the L-BFGS history of one start does not fit shared memory");
    K->wpc_k = k;
    K->smem_doubles = (int)per_start;
    eo.expect_slice_doubles = (int)per_start;
    // at most 256 threads per CTA (255 registers each fit the register file); named barriers 2..15 when K > 1
    K->starts_per_cta = (int)std::max<uint64_t>(1, std::min<uint64_t>((uint64_t)(8 / k), cap / per_start));
  }
  K->source = emit_optimizer_source(*P, eo, history);
  rc = nvrtc_to_cubin(K->source, "rainier_optimizer.cu", fast, K->cubin);
  if (rc) return rc;
  *out = K.get();
  m->opt_kernels.emplace(key, std::move(K));
  return RN_OK;
}

extern "C" {

void rn_optimize_config_default(rn_optimize_config* c) {  // Optimizer.scala:12-13
  std::memset(c, 0, sizeof(*c));
  c->struct_size = (int32_t)sizeof(*c);
  c->history = 5;
  c->eps = 0.1;
  c->max_evaluations = 10000;
  c->math_mode = RN_MATH_PARITY;
  c->gradient_mode = RN_GRAD_AUTO;
  c->backend = RN_BACKEND_AUTO;
}

int rn_optimize_emit_source(rn_model* m, const rn_optimize_config* oc, char* buf, size_t cap, size_t* needed) {
  if (!m) return fail(RN_E_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  rn_model::OptKernel* K = nullptr;
  int rc = get_opt_kernel(m, oc, &K);
  if (rc) return rc;
  if (needed) *needed = K->source.size() + 1;
  if (buf && cap) {
    size_t n = std::min(cap - 1, K->source.size());
    std::memcpy(buf, K->source.data(), n);
    buf[n] = 0;
  }
  return RN_OK;
}

int rn_optimize_emit_cubin(rn_model* m, const rn_optimize_config* oc, void* buf, size_t cap, size_t* needed) {
  if (!m) return fail(RN_E_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  rn_model::OptKernel* K = nullptr;
  int rc = get_opt_kernel(m, oc, &K);
  if (rc) return rc;
  if (needed) *needed = K->cubin.size();
  if (buf && cap) std::memcpy(buf, K->cubin.data(), std::min(cap, K->cubin.size()));
  return RN_OK;
}

int rn_optimize(rn_model* m, const rn_optimize_config* oc, const double* x0, int starts, double* x, double* f, int32_t* info,
                int32_t* evaluations) {
  if (!m || !x || starts <= 0) return fail(RN_E_INVALID, "bad argument");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  if (m->device < 0) return fail(RN_E_CUDA, "model was created without a device (no CPU fallback)");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  rn_model::OptKernel* K = nullptr;
  int rc = get_opt_kernel(m, oc, &K);
  if (rc) return rc;
  rc = make_current(A, m);
  if (rc) return rc;
  if (!K->mod) {
    CU(A->cuModuleLoadData(&K->mod, K->cubin.data()));
    CU(A->cuModuleGetFunction(&K->k_lbfgs, K->mod, "rn_k_lbfgs"));
    if (K->backend == 1)
      CU(A->cuFuncSetAttribute(K->k_lbfgs, 8 /*MAX_DYNAMIC_SHARED_SIZE_BYTES*/, K->starts_per_cta * K->smem_doubles * 8));
  }
  const size_t n = m->n_params, S = (size_t)starts;
  // one allocation: x0 | x | f | info | evals
  const size_t off_x = n * S * 8, off_f = 2 * n * S * 8, off_info = off_f + S * 8, off_ev = off_info + S * 4;
  const size_t total = off_ev + S * 4;
  CUdeviceptr d = 0;
  struct Free {
    const Api* A;
    CUdeviceptr* p;
    ~Free() {
      if (*p) A->cuMemFree(*p);
    }
  } guard{A, &d};
  CU(A->cuMemAlloc(&d, total + 16));
  std::vector<double> t(n * S);
  if (x0) {
    for (size_t c = 0; c < S; c++)
      for (size_t i = 0; i < n; i++) t[i * S + c] = x0[c * n + i];
    CU(A->cuMemcpyHtoD(d, t.data(), n * S * 8));
  }
  RnOptArgs a;
  std::memset(&a, 0, sizeof(a));
  a.x0 = x0 ? (const double*)(uintptr_t)d : nullptr;
  a.x = (double*)(uintptr_t)(d + off_x);
  a.f = (double*)(uintptr_t)(d + off_f);
  a.info = (int*)(uintptr_t)(d + off_info);
  a.evals = (int*)(uintptr_t)(d + off_ev);
  a.data = (const double*)(uintptr_t)m->d_data;
  a.eps = oc ? oc->eps : 0.1;
  a.starts = starts;
  a.max_evals = oc && oc->max_evaluations > 0 ? oc->max_evaluations : 10000;
  void* params[] = {&a};
  if (K->backend == 1) {
    const unsigned spc = (unsigned)K->starts_per_cta;
    CU(A->cuLaunchKernel(K->k_lbfgs, (unsigned)((S + spc - 1) / spc), 1, 1, spc * 32 * (unsigned)K->wpc_k, 1, 1,
                         spc * (unsigned)K->smem_doubles * 8, nullptr, params, nullptr));
  } else {
    // small CTAs spread few starts over all SMs; starts diverge (different trajectory lengths), so warps are the unit
    const unsigned block = starts >= 148 * 128 ? 128 : 32;
    CU(A->cuLaunchKernel(K->k_lbfgs, (unsigned)((S + block - 1) / block), 1, 1, block, 1, 1, 0, nullptr, params, nullptr));
  }
  CU(A->cuMemcpyDtoH(t.data(), d + off_x, n * S * 8));
  for (size_t c = 0; c < S; c++)
    for (size_t i = 0; i < n; i++) x[c * n + i] = t[i * S + c];
  if (f) CU(A->cuMemcpyDtoH(f, d + off_f, S * 8));
  std::vector<int32_t> inf(S);
  CU(A->cuMemcpyDtoH(inf.data(), d + off_info, S * 4));
  if (info) std::memcpy(info, inf.data(), S * 4);
  if (evaluations) CU(A->cuMemcpyDtoH(evaluations, d + off_ev, S * 4));
  for (size_t c = 0; c < S; c++)
    if (inf[c] & 4) return fail(RN_E_LOOKUP, "lookup index out of range");
  return RN_OK;
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------------
// rn_sample_predict: `Model.sample(t, config)` (rainier-core/.../core/Model.scala:56-63) = model.sample(config).predict(gen)
// in one call.  The draws never leave the device: the chains are sampled into a resident [iterations][n][chains] block,
// rn_k_eval turns it into the generator's requirement values in Trace.predict's order, and only those
// chains*iterations*m doubles cross PCIe (m/n of what rn_sample ships; a single predicted Real of the funnel: 10x less).
// Built from the staged entry points (rn_sampler_*, rn_function_eval_device); rn_sample itself is untouched.
// ---------------------------------------------------------------------------------------------------------
extern "C" int rn_sample_predict(rn_model* m, const rn_config* cfg, rn_function* f, const int64_t* seeds, int chains,
                                 double* predictions, double* mass, rn_chain_stats* stats) {
  if (!m) return fail(RN_E_INVALID, "null model");
  std::lock_guard<std::recursive_mutex> model_lock_(m->mu);
  if (!m || !cfg || !f || chains <= 0 || cfg->iterations < 0) return fail(RN_E_INVALID, "bad argument");
  if (!predictions && cfg->iterations > 0) return fail(RN_E_INVALID, "null predictions buffer");
  if (m->device < 0 || f->device < 0) return fail(RN_E_CUDA, "model/function was created without a device (no CPU fallback)");
  if (m->device != f->device) return fail(RN_E_INVALID, "model and function live on different devices");
  if (f->prog.n_params != m->n_params) return fail(RN_E_INVALID, "the function's inputs are not the model's parameters");
  std::string why;
  const Api* A = api(&why);
  if (!A) return fail(RN_E_CUDA, why);
  rn_sampler* s = nullptr;
  int rc = rn_sampler_create(m, cfg, seeds, chains, &s);
  if (rc) return rc;
  struct Guard {
    rn_sampler* s;
    ~Guard() { rn_sampler_destroy(s); }
  } g{s};
  rc = rn_sampler_warmup(s, -1);
  if (rc) return rc;
  rc = rn_sampler_run(s, 0, nullptr);  // lf.resetStats() after warmup even when no iteration follows (Driver.scala:31)
  if (rc) return rc;
  const size_t C = (size_t)chains, n = m->n_params, I = (size_t)cfg->iterations, mo = f->prog.fn_outputs.size();
  if (I > 0) {
    const size_t want[2] = {I * n * C * 8 /* draws [I][n][C] */, C * I * mo * 8 /* predictions [C][I][m] */};
    for (int k = 0; k < 2; k++)
      if (m->pool_bytes[k] < want[k]) {
        if (m->pool[k]) A->cuMemFree(m->pool[k]);
        m->pool[k] = 0;
        m->pool_bytes[k] = 0;
        CU(A->cuMemAlloc(&m->pool[k], want[k]));
        m->pool_bytes[k] = want[k];
      }
    rc = rn_sampler_run(s, (int)I, (double*)(uintptr_t)m->pool[0]);
    if (rc) return rc;
    rc = function_load(A, f);  // same primary context as the model's
    if (rc) return rc;
    // on the sampler's stream: ordered after the last rn_k_iter launch, no event needed
    rc = rn_function_eval_device(f, (const double*)(uintptr_t)m->pool[0], RN_LAYOUT_SAMPLER, (int64_t)I, (int64_t)C,
                                 (double*)(uintptr_t)m->pool[1], (void*)s->stream);
    if (rc) return rc;
    rc = drain_to_host(A, s->stream, m->pool[1], predictions, want[1], /*sync=*/true);
    if (rc) return rc;
    if (cfg->diagnostics) {
      rc = rn_sampler_diagnostics(s, (const double*)(uintptr_t)m->pool[0], (int)I, 0, cfg->diagnostics);
      if (rc) return rc;
    }
    rc = rn_function_sync(f);  // lookup errors of the evaluation
    if (rc) return rc;
  }
  return rn_sampler_stats(s, stats, mass, cfg->stats_rings);
}
