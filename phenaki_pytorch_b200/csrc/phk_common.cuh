// Shared device/host helpers for libphk (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <float.h>
#include <utility>
#include "../../include/phk.h"
#include <cstdlib>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libphk is written for sm_100a (B200) only"
#endif

namespace phk {

void set_error(const char* msg);
void count_launch(int n = 1);
// patchify_tma.cu: TMA-gathered patchify + LayerNorm; returns 0 when launched, 1 when the shape is not eligible
int patchify_ln_tma_launch(const float* video, int B, int C, int F, int H, int W, int f0, int nt, int pt, int p1, int p2,
                           const float* ln_g, const float* ln_b, void* out, int out_bf16, cudaStream_t st);

#define PHK_REQUIRE(cond, code, msg) \
  do { if (!(cond)) { ::phk::set_error(msg); return (code); } } while (0)

// returns cudaError after a launch (sticky errors surface here without a sync)
#define PHK_LAUNCH_CHECK() \
  do { ::phk::count_launch(); cudaError_t e__ = cudaGetLastError(); if (e__ != cudaSuccess) return (int)e__; } while (0)

#define PHK_CUDA(call) \
  do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return (int)e__; } while (0)

#define PHK_TRY(call) \
  do { int r__ = (call); if (r__ != 0) return r__; } while (0)

static inline cudaStream_t to_stream(phk_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

constexpr int kNumSMs = 148;

// One-time per-DEVICE kernel configuration (cudaFuncSetAttribute is a per-device setting; a process may drive several
// devices): `mask` is a call-site static, bit d = "done on device d".
static inline bool device_configured(const unsigned long long* mask) {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= 64) return false;
  return (__atomic_load_n(mask, __ATOMIC_RELAXED) >> d) & 1ull;
}
static inline void mark_configured(unsigned long long* mask) {
  int d = 0;
  if (cudaGetDevice(&d) == cudaSuccess && d >= 0 && d < 64) __atomic_fetch_or(mask, 1ull << d, __ATOMIC_RELAXED);
}

// Optional per-kernel-family timing with CUDA events on the launching stream (bench.py roofline /
// share-of-step numbers).  Off by default: zero overhead beyond one relaxed load per entry point.
enum Family { FAM_PATCHIFY = 0, FAM_LAYERNORM, FAM_GEMM_F32, FAM_GEMM_BF16, FAM_ATTENTION, FAM_PEG, FAM_GEGLU,
              FAM_LFQ, FAM_EMBED, FAM_CPB, FAM_SAMPLE, FAM_TOPK, FAM_CRITIC, FAM_CFG, FAM_COUNT };
struct Prof {
  Prof(int fam, phk_stream_t s, double work = 0.0);
  ~Prof();
  int fam; cudaStream_t st; cudaEvent_t e0; bool on; double work;
};

// Programmatic dependent launch (PDL): every kernel of the library is launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, triggers its dependents immediately and waits for its
// predecessors right before its first global-memory access.  The next kernel's launch latency, block scheduling and
// prologue (barrier init, tensor-map prefetch, TMEM allocation) then overlap the tail of the running kernel.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_prologue() { pdl_trigger(); pdl_wait(); }

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                     Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  // PHK_PDL=0 (A/B measurements): plain stream order -- the kernels' griddepcontrol instructions are then no-ops
  static const bool pdl = [] { const char* e = std::getenv("PHK_PDL"); return !(e && e[0] == '0'); }();
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = pdl ? 1 : 0;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// Plain stream-ordered launch (no programmatic dependent launch: for kernels that do not call pdl_prologue()).
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                       Args&&... args) {
  kernel<<<grid, block, smem, st>>>(static_cast<KArgs>(args)...);
  return cudaGetLastError();
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// Block-wide sum for blockDim.x <= 1024 (multiple of 32). `red` is >= 32 floats of smem.
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();  // protect `red` from a previous use
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float t = (lane < nw) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;
}

__device__ __forceinline__ float gelu_erf(float x) {
  // F.gelu default (approximate='none'): 0.5 * x * (1 + erf(x / sqrt(2)))
  return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}

// ---- in-kernel sampling noise (statistical mode of the demasking loop: phk_sample_tokens without injected draws, the
// fused logits head).  Counter-based: Philox4x32 keyed by the torch CUDA seed, counter = noise offset + (token, v / 4).
// 7 rounds: the smallest count the Random123 authors report as passing BigCrush (10 is their safety-margin default); the
// generator sits in the logits head's epilogue, which is instruction-bound (ncu, profiles/), at 4 IMAD + 2 LOP3 per round.
constexpr int kNoiseRounds = 7;
template <int ROUNDS>
__device__ __forceinline__ void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                                           uint32_t* out) {
#pragma unroll
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
__device__ __forceinline__ float fast_lg2(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ float fast_ex2(float x) {
  float r;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
// Gumbel(0, 1) draw -log(-log(u)) (phenaki_pytorch.py:83-86) from 32 random bits: u = (2 k + 1) / 2^24 for the top 23 bits k
// -- strictly inside (0, 1), so the reference's 1e-10 guards are not needed -- built from the bits directly (no int->float
// conversion), both logarithms in base 2 on the MUFU unit: g = -ln2 * log2(-log2(u)) - ln(ln 2).
__device__ __forceinline__ float gumbel_from_bits(uint32_t r) {
  const float u = __uint_as_float(0x3f800000u | (r >> 9)) - 0.99999994f;  // [1, 2) - (1 - 2^-24): exact
  // e = -log2(u) > 0.  The approximate logarithm's error near 1 (absolute, 2^-22 on [0.5, 2]) is as large as e itself
  // for the largest u, which decide the argmax; above 1 - 2^-7 e comes from the exact complement w = 1 - u instead:
  // -ln(1 - w) = w (1 + w/2 + w^2/3 + ...), the two terms kept err by < w^2/3 < 2^-15.5 relative.
  const float w = 1.0f - u;
  const float e = u > 0.9921875f ? w * fmaf(w, 0.72134752f, 1.44269504f) : -fast_lg2(u);
  return fmaf(-0.69314718f, fast_lg2(e), 0.36651292f);
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}

// inference drivers bracket their GEMM calls with this: the W operands are weights that no kernel of the stream rewrites,
// so the tcgen05 GEMM may request their first tiles before its programmatic-dependent-launch wait (gemm_tcgen05.cu)
void gemm_static_weights(bool on);
struct StaticWeightsScope {
  StaticWeightsScope() { gemm_static_weights(true); }
  ~StaticWeightsScope() { gemm_static_weights(false); }
};

}  // namespace phk
