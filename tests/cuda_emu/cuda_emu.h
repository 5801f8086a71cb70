// TEST INFRASTRUCTURE: a single-threaded CPU executor for plain (non tensor-core) CUDA kernels, so that the build
// container -- which has nvcc but no GPU -- can RUN the kernels of csrc/train.cu and check them against the reference
// gradients before any GPU time is spent (tests/test_train_emulated_cpu.py).
//
// Every CUDA thread of a block is a ucontext fiber; blocks run one after another.  __syncthreads() and the warp
// shuffles are barriers between fibers (round-robin scheduler), so the lock-step semantics the kernels rely on
// (warp_sum, block_sum, shared-memory staging) are reproduced exactly; atomics are plain read-modify-writes.
// `__shared__` variables become function-local statics (one block is resident at a time).
// Only what csrc/train.cu uses is provided.
#pragma once
#include <ucontext.h>
#include <cfloat>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <algorithm>
#include <tuple>
#include <utility>
#include <vector>
#include "../../include/phk.h"

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct float2 { float x, y; };
static inline float2 make_float2(float a, float b) { return float2{a, b}; }
struct alignas(16) float4 { float x, y, z, w; };
static inline float4 make_float4(float a, float b, float c, float d) { return float4{a, b, c, d}; }
struct alignas(8) uint2 { unsigned x, y; };
static inline uint2 make_uint2(unsigned a, unsigned b) { return uint2{a, b}; }
struct alignas(16) uint4 { unsigned x, y, z, w; };
static inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return uint4{a, b, c, d}; }
struct __nv_bfloat16 { uint16_t bits; };
static inline __nv_bfloat16 __float2bfloat16_rn(float f) {  // round to nearest even, like the device intrinsic
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return __nv_bfloat16{(uint16_t)((u >> 16) | 0x40)};
  u += 0x7fffu + ((u >> 16) & 1u);
  return __nv_bfloat16{(uint16_t)(u >> 16)};
}
static inline float __bfloat162float(__nv_bfloat16 h) {
  const uint32_t u = (uint32_t)h.bits << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
struct __nv_bfloat162 { __nv_bfloat16 x, y; };
static inline float2 __bfloat1622float2(__nv_bfloat162 v) { return float2{__bfloat162float(v.x), __bfloat162float(v.y)}; }
static inline __nv_bfloat162 __floats2bfloat162_rn(float a, float b) {
  return __nv_bfloat162{__float2bfloat16_rn(a), __float2bfloat16_rn(b)};
}
typedef void* cudaStream_t;
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaMemcpyDeviceToDevice = 3, cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
template <typename K> static inline cudaError_t cudaFuncSetAttribute(K, int, int) { return 0; }
// ---- host-side runtime calls of the drivers (api.cu): one in-order "stream", so events and waits are no-ops, copies are
// memcpy, and stream capture reports failure (the drivers then keep launching eagerly, as with PHK_GRAPH=0)
typedef void* cudaEvent_t;
typedef void* cudaGraph_t;
typedef void* cudaGraphExec_t;
enum { cudaMemcpyHostToDevice = 1, cudaMemcpyDeviceToHost = 2, cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2,
       cudaStreamCaptureModeThreadLocal = 1, cudaErrorStreamCaptureUnsupported = 900, cudaErrorInvalidValue = 1 };
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = nullptr; return 0; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = nullptr; return 0; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return 0; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return 0; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return 0; }
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = nullptr; return 0; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return 0; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
cudaError_t cudaStreamBeginCapture(cudaStream_t, int);
cudaError_t cudaStreamEndCapture(cudaStream_t, cudaGraph_t* g);
cudaError_t cudaGraphInstantiate(cudaGraphExec_t* e, cudaGraph_t g, unsigned long long);
cudaError_t cudaGraphLaunch(cudaGraphExec_t e, cudaStream_t);
cudaError_t cudaGraphDestroy(cudaGraph_t g);
cudaError_t cudaGraphExecDestroy(cudaGraphExec_t e);
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }

namespace emu {
struct Group { int alive = 0, count = 0; unsigned gen = 0; };
struct State {
  dim3 t_idx, b_idx, b_dim, g_dim;
  void* dyn_smem = nullptr;
};
extern State S;
void yield();
void barrier(Group& g);
Group& block_group();
Group& warp_group();
float* warp_xchg();
void launch(dim3 grid, dim3 block, size_t smem, const std::function<void()>& body);
// one stream-ordered operation: executed now, or -- between cudaStreamBeginCapture / EndCapture -- recorded as a node of
// the graph under construction (arguments by value: exactly what a captured CUDA graph bakes in)
void submit(std::function<void()> op);
void set_schedule_seed(uint64_t seed);
}  // namespace emu

#define threadIdx (::emu::S.t_idx)
#define blockIdx (::emu::S.b_idx)
#define blockDim (::emu::S.b_dim)
#define gridDim (::emu::S.g_dim)

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
#define __launch_bounds__(...)
#define __align__(n) __attribute__((aligned(n)))
#define __shared__ static
#define PHK_CUDA_EMU_ACTIVE 1

static inline void __syncthreads() { ::emu::barrier(::emu::block_group()); }
template <typename T>
static inline T __shfl_xor_sync(unsigned, T v, int lane_mask) {  // any 32-bit type travels as raw bits
  static_assert(sizeof(T) == 4, "cuda_emu: 32-bit shuffles only");
  float* x = ::emu::warp_xchg();
  const int lane = (int)(threadIdx.x & 31);
  memcpy(&x[lane], &v, 4);
  ::emu::barrier(::emu::warp_group());
  T r;
  memcpy(&r, &x[lane ^ lane_mask], 4);
  ::emu::barrier(::emu::warp_group());
  return r;
}
static inline void __syncwarp(unsigned = 0xffffffffu) { ::emu::barrier(::emu::warp_group()); }
static inline float atomicAdd(float* p, float v) { const float o = *p; *p = o + v; return o; }
static inline float rsqrtf(float x) { return 1.0f / sqrtf(x); }
template <typename T> static inline T __ldg(const T* p) { return *p; }
// round-to-nearest single operations (the kernels use them to forbid FMA contraction; build with -ffp-contract=off)
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline float __fdividef(float a, float b) { return a / b; }
#define __expf(x) expf(x)
#define __logf(x) logf(x)
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((uint64_t)a * b) >> 32); }
using std::max;
using std::min;
static inline cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t) {
  ::emu::submit([=]() { memset(p, v, n); });
  return 0;
}
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, int, cudaStream_t) {
  ::emu::submit([=]() { memmove(d, s, n); });
  return 0;
}
static inline cudaError_t cudaMemcpy2DAsync(void* d, size_t dpitch, const void* s, size_t spitch, size_t width, size_t height,
                                            int, cudaStream_t) {
  ::emu::submit([=]() {
    for (size_t r = 0; r < height; ++r) memmove((char*)d + r * dpitch, (const char*)s + r * spitch, width);
  });
  return 0;
}
static inline cudaError_t cudaGetLastError() { return 0; }

namespace phk {
void set_error(const char* msg);
void count_launch(int n = 1);
#define PHK_REQUIRE(cond, code, msg) \
  do { if (!(cond)) { ::phk::set_error(msg); return (code); } } while (0)
#define PHK_LAUNCH_CHECK() do { ::phk::count_launch(); } while (0)
#define PHK_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return (int)e__; } while (0)
#define PHK_TRY(call) do { int r__ = (call); if (r__ != 0) return r__; } while (0)
static inline cudaStream_t to_stream(phk_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }
constexpr int kNumSMs = 148;
enum Family { FAM_PATCHIFY = 0, FAM_LAYERNORM, FAM_GEMM_F32, FAM_GEMM_BF16, FAM_ATTENTION, FAM_PEG, FAM_GEGLU,
              FAM_LFQ, FAM_EMBED, FAM_CPB, FAM_SAMPLE, FAM_TOPK, FAM_CRITIC, FAM_CFG, FAM_COUNT };
struct Prof {  // defined in api.cu (per-family event timing; the events are no-ops here)
  Prof(int fam, phk_stream_t s, double work = 0.0);
  ~Prof();
  int fam; cudaStream_t st; cudaEvent_t e0; bool on; double work;
};
static inline void pdl_trigger() {}
static inline void pdl_wait() {}
static inline void pdl_prologue() {}
int patchify_ln_tma_launch(const float*, int, int, int, int, int, int, int, int, int, int, const float*, const float*, void*,
                           int, cudaStream_t);
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t,
                                     Args&&... args) {
  auto params = std::make_tuple(static_cast<KArgs>(args)...);  // kernel parameters are copied at launch (or capture) time
  ::emu::submit([=]() { ::emu::launch(grid, block, smem, [&]() { std::apply(kernel, params); }); });
  return 0;
}
template <typename... KArgs, typename... Args>
static inline cudaError_t launch_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t,
                                       Args&&... args) {
  auto params = std::make_tuple(static_cast<KArgs>(args)...);
  ::emu::submit([=]() { ::emu::launch(grid, block, smem, [&]() { std::apply(kernel, params); }); });
  return 0;
}
__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  return (uint32_t)__float2bfloat16_rn(lo).bits | ((uint32_t)__float2bfloat16_rn(hi).bits << 16);
}

// same definitions as csrc/phk_common.cuh
static inline float __uint_as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline uint32_t __float_as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
constexpr int kNoiseRounds = 7;
template <int ROUNDS>
static inline void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t* out) {
  for (int r = 0; r < ROUNDS; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
static inline float fast_lg2(float x) { return log2f(x); }
static inline float fast_ex2(float x) { return exp2f(x); }
static inline float gumbel_from_bits(uint32_t r) {
  const float u = __uint_as_float(0x3f800000u | (r >> 9)) - 0.99999994f;
  const float w = 1.0f - u;
  const float e = u > 0.9921875f ? w * fmaf(w, 0.72134752f, 1.44269504f) : -fast_lg2(u);
  return fmaf(-0.69314718f, fast_lg2(e), 0.36651292f);
}

// One-time per-DEVICE kernel configuration (cudaFuncSetAttribute is a per-device setting; a process may drive several
// devices): `mask` is a call-site static, bit d = "done on device d".
static inline bool device_configured(const unsigned long long* mask) {
  int d = 0;
  if (cudaGetDevice(&d) != 0 || d < 0 || d >= 64) return false;
  return (__atomic_load_n(mask, __ATOMIC_RELAXED) >> d) & 1ull;
}
static inline void mark_configured(unsigned long long* mask) {
  int d = 0;
  if (cudaGetDevice(&d) == 0 && d >= 0 && d < 64) __atomic_fetch_or(mask, 1ull << d, __ATOMIC_RELAXED);
}
__device__ __forceinline__ float warp_sum(float v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float block_sum(float v, float* red) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  float t = (lane < nw) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;
}
struct StaticWeightsScope {};  // the GPU GEMM's weight prefetch hint (phk_common.cuh): nothing to do on the CPU executor
}  // namespace phk
