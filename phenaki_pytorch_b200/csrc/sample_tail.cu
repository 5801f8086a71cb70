// Tail of one demasking iteration restricted to the tokens that are still masked (phenaki_pytorch.py:495-509, 547-550).
//
// The reference computes logits for every position and then keeps the prediction only where the mask is set
// (`ids = where(mask, pred, ids)`, :509) and scores `where(mask, 1 - p, -1e4)` (:547-550).  Rows do not interact after
// the last attention, so the final LayerNorm, the guidance combination and the 2 x tokens x V x dim logits head -- a
// quarter of the step -- are only needed for the masked rows.  Their number is known on the host without a sync: the
// cosine schedule re-masks exactly k_s tokens per sequence (phk_topk_mask), 576, 574, ... 50 of 576 over 18 steps, i.e.
// 31 % fewer 128-token head tiles over a whole sample.
//
//   mask_compact      index[b*k]   <- positions of the masked tokens of each sequence, in order
//   ln_cfg_gather     emb[b*k, D]  <- norm_out(x_null) + s * (norm_out(x_cond) - norm_out(x_null)) of those rows (bf16)
//   phk_head_sample   on b*k rows  (tcgen05 GEMM + gumbel argmax + confidence, head_sample.cu; logits never stored)
//   scatter           ids / pred / score of the masked rows; score = -1e4 and ids untouched elsewhere
//
// Plain kernels (no tensor cores): they also run under tests/cuda_emu.
#include "phk_common.cuh"

namespace phk {
namespace {

// One CTA per sequence; thread t owns the contiguous positions [t*per, (t+1)*per): count, block-wide exclusive scan of
// the counts, then write.  Exactly k entries are produced per sequence: surplus masked positions are dropped and a
// shortfall is padded with -1 (neither happens when the mask comes from phk_topk_mask with the same k).
__global__ void __launch_bounds__(256) mask_compact_kernel(const uint8_t* __restrict__ mask, int n, int k,
                                                           int* __restrict__ index) {
  pdl_prologue();
  __shared__ int s_cnt[256];
  const int bi = blockIdx.x, t = threadIdx.x;
  const int per = (n + 255) / 256;
  const int p0 = t * per, p1 = (p0 + per < n) ? p0 + per : n;
  const uint8_t* mrow = mask + (int64_t)bi * n;
  int c = 0;
  for (int p = p0; p < p1; ++p) c += mrow[p] ? 1 : 0;
  s_cnt[t] = c;
  __syncthreads();
  for (int off = 1; off < 256; off <<= 1) {  // inclusive Hillis-Steele scan
    const int v = (t >= off) ? s_cnt[t - off] : 0;
    __syncthreads();
    s_cnt[t] += v;
    __syncthreads();
  }
  int pos = s_cnt[t] - c;  // exclusive prefix
  const int total = s_cnt[255];
  int* out = index + (int64_t)bi * k;
  for (int p = p0; p < p1; ++p)
    if (mrow[p]) { if (pos < k) out[pos] = bi * n + p; ++pos; }
  for (int j = total + t; j < k; j += 256) out[j] = -1;
}

// norm_out of both halves + guidance for the gathered rows; same arithmetic and summation order as ln_cfg_kernel
// (head_sample.cu), so a row's embedding is bit-identical whether it is computed here or there
template <int VEC>
__global__ void __launch_bounds__(256) ln_cfg_gather_kernel(const float* __restrict__ xc, const float* __restrict__ xn,
                                                            const float* __restrict__ g, const float* __restrict__ b,
                                                            float scale, const int* __restrict__ index,
                                                            __nv_bfloat16* __restrict__ out, int64_t rows, int dim,
                                                            int seq_n, int src_stride, int src_off) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= rows) return;
  // index = sequence * seq_n + position among the sampled tokens; the residual stream may carry a prime prefix:
  // its row is sequence * src_stride + src_off + position (phenaki_pytorch.py:493, 503-504)
  const int idx = index[row];
  const int src = idx < 0 ? -1 : (idx / seq_n) * src_stride + src_off + idx % seq_n;
  float4 o[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) o[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (src >= 0) {
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const float4* xr = reinterpret_cast<const float4*>((pass ? xn : xc) + (int64_t)src * dim);
      float4 v[VEC];
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < VEC; ++j) { v[j] = xr[lane + 32 * j]; s += (v[j].x + v[j].y) + (v[j].z + v[j].w); }
      const float mean = warp_sum(s) / (float)dim;
      float q = 0.f;
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float a = v[j].x - mean, bb = v[j].y - mean, c = v[j].z - mean, d = v[j].w - mean;
        q += (a * a + bb * bb) + (c * c + d * d);
      }
      const float rstd = rsqrtf(warp_sum(q) / (float)dim + 1e-5f);
      const float w = pass ? (1.0f - scale) : scale;  // null + s*(cond - null) = s*cond + (1-s)*null
#pragma unroll
      for (int j = 0; j < VEC; ++j) {
        const float4 gg = reinterpret_cast<const float4*>(g)[lane + 32 * j], bb = reinterpret_cast<const float4*>(b)[lane + 32 * j];
        o[j].x += w * ((v[j].x - mean) * rstd * gg.x + bb.x);
        o[j].y += w * ((v[j].y - mean) * rstd * gg.y + bb.y);
        o[j].z += w * ((v[j].z - mean) * rstd * gg.z + bb.z);
        o[j].w += w * ((v[j].w - mean) * rstd * gg.w + bb.w);
      }
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j)
    reinterpret_cast<uint2*>(out + row * dim)[lane + 32 * j] = make_uint2(pack_bf16x2(o[j].x, o[j].y), pack_bf16x2(o[j].z, o[j].w));
}

// every position: score = -1e4 (:549), pred = the current id (only masked positions carry a prediction)
__global__ void tail_init_kernel(const int64_t* __restrict__ ids, int64_t* __restrict__ pred_out,
                                 float* __restrict__ score_out, int64_t tokens) {
  pdl_prologue();
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < tokens; i += (int64_t)gridDim.x * blockDim.x) {
    if (score_out) score_out[i] = -1e4f;
    if (pred_out) pred_out[i] = ids[i];
  }
}

// masked positions: ids = pred (:509), score = 1 - p[pred] (:547-548)
__global__ void tail_scatter_kernel(const int* __restrict__ index, const int64_t* __restrict__ pred_c,
                                    const float* __restrict__ score_c, int64_t* __restrict__ ids,
                                    int64_t* __restrict__ pred_out, float* __restrict__ score_out, int64_t rows) {
  pdl_prologue();
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < rows; r += (int64_t)gridDim.x * blockDim.x) {
    const int t = index[r];
    if (t < 0) continue;
    ids[t] = pred_c[r];
    if (pred_out) pred_out[t] = pred_c[r];
    if (score_out) score_out[t] = score_c[r];
  }
}

// rng_state[1] += stride: the noise counters one iteration consumed (device-resident key of a replayed graph)
__global__ void rng_advance_kernel(unsigned long long* rng_state, unsigned long long stride) {
  pdl_prologue();
  if (blockIdx.x == 0 && threadIdx.x == 0) rng_state[1] += stride;
}

// phk_noise_probe: thread q owns counter offset + q, i.e. the four words i = 4q .. 4q+3
__global__ void noise_probe_kernel(const uint32_t* __restrict__ bits_in, uint64_t seed, uint64_t offset, int64_t n,
                                   uint32_t* __restrict__ bits_out, float* __restrict__ gumbel_out) {
  pdl_prologue();
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q * 4 < n; q += (int64_t)gridDim.x * blockDim.x) {
    uint32_t r[4];
    if (!bits_in) {
      const uint64_t ctr = offset + (uint64_t)q;
      philox4x32<kNoiseRounds>((uint32_t)ctr, (uint32_t)(ctr >> 32), 0u, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    }
    for (int j = 0; j < 4 && q * 4 + j < n; ++j) {
      const uint32_t w = bits_in ? bits_in[q * 4 + j] : r[j];
      bits_out[q * 4 + j] = w;
      gumbel_out[q * 4 + j] = gumbel_from_bits(w);
    }
  }
}

struct TailBufs { int* index; __nv_bfloat16* emb; uint8_t* ones; int64_t* ids_c; int64_t* pred_c; float* score_c; char* head; int64_t head_bytes; };

int64_t align256(int64_t v) { return (v + 255) & ~int64_t(255); }

int64_t carve(char* base, int64_t rows, int dim, TailBufs* t) {
  int64_t off = 0;
  auto take = [&](int64_t bytes) { char* p = base ? base + off : nullptr; off += align256(bytes); return p; };
  char* a = take(rows * 4);
  char* e = take(rows * (int64_t)dim * 2);
  char* o = take(rows);
  char* i = take(rows * 8);
  char* p = take(rows * 8);
  char* s = take(rows * 4);
  const int64_t hb = phk_head_sample_scratch_bytes((int32_t)rows);
  char* h = take(hb);
  if (t) *t = TailBufs{(int*)a, (__nv_bfloat16*)e, (uint8_t*)o, (int64_t*)i, (int64_t*)p, (float*)s, h, hb};
  return off + 256;
}

}  // namespace
}  // namespace phk

using namespace phk;

extern "C" int64_t phk_sample_tail_scratch_bytes(int32_t b, int32_t k, int32_t dim) {
  if (b <= 0 || k <= 0 || dim <= 0) return -1;
  return carve(nullptr, (int64_t)b * k, dim, nullptr);
}

extern "C" int phk_sample_tail_rows(const float* x_cond, const float* x_null, const float* gamma, const float* beta,
                                    float cond_scale, const void* head_w, int64_t ldw, const float* head_b, int32_t b,
                                    int32_t n, int32_t k, int32_t V, int32_t dim, float temperature, uint64_t seed,
                                    uint64_t offset, const uint64_t* rng_state, const uint8_t* mask, int64_t* ids,
                                    int64_t* pred_out, float* score_out, int32_t src_stride, int32_t src_off,
                                    void* scratch, int64_t scratch_bytes, phk_stream_t s) {
  PHK_REQUIRE(src_stride >= n && src_off >= 0 && src_off + n <= src_stride, PHK_E_ARG, "phk_sample_tail: bad source row map");
  PHK_REQUIRE(x_cond && x_null && gamma && beta && head_w && mask && ids && scratch, PHK_E_ARG, "phk_sample_tail: null pointer");
  PHK_REQUIRE(b > 0 && n > 0 && k > 0 && k <= n && V > 0, PHK_E_ARG, "phk_sample_tail: bad size");
  PHK_REQUIRE(dim % 128 == 0 && dim <= 1024, PHK_E_UNSUPPORTED, "phk_sample_tail: dim must be a multiple of 128, <= 1024");
  PHK_REQUIRE((int64_t)b * n < (1LL << 31), PHK_E_UNSUPPORTED, "phk_sample_tail: more than 2^31 tokens");
  PHK_REQUIRE(scratch_bytes >= phk_sample_tail_scratch_bytes(b, k, dim), PHK_E_WORKSPACE, "phk_sample_tail: scratch too small");
  cudaStream_t st = to_stream(s);
  const int64_t rows = (int64_t)b * k, tokens = (int64_t)b * n;
  TailBufs t;
  char* base = (char*)(((uintptr_t)scratch + 255) & ~(uintptr_t)255);
  carve(base, rows, dim, &t);
  PHK_CUDA(launch_pdl(mask_compact_kernel, dim3((unsigned)b), dim3(256), (size_t)0, st, mask, n, k, t.index));
  PHK_LAUNCH_CHECK();
  const dim3 grid((unsigned)((rows + 7) / 8)), block(256);
  switch (dim / 128) {
    case 1: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<1>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 2: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<2>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 3: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<3>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 4: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<4>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 5: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<5>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 6: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<6>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    case 7: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<7>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
    default: PHK_CUDA(launch_pdl(ln_cfg_gather_kernel<8>, grid, block, (size_t)0, st, x_cond, x_null, gamma, beta, cond_scale, t.index, t.emb, rows, dim, (int)n, (int)src_stride, (int)src_off)); break;
  }
  PHK_LAUNCH_CHECK();
  PHK_CUDA(cudaMemsetAsync(t.ones, 1, rows, st));
  PHK_TRY(phk_head_sample_rng(t.emb, dim, rows, head_w, ldw, head_b, (int32_t)rows, V, dim, temperature, seed, offset,
                              rng_state, t.ones, t.ids_c, t.pred_c, t.score_c, t.head, t.head_bytes, s));
  const unsigned g1 = (unsigned)((tokens + 255) / 256 < 1184 ? (tokens + 255) / 256 : 1184);
  PHK_CUDA(launch_pdl(tail_init_kernel, dim3(g1), dim3(256), (size_t)0, st, (const int64_t*)ids, pred_out, score_out, tokens));
  PHK_LAUNCH_CHECK();
  const unsigned g2 = (unsigned)((rows + 255) / 256 < 1184 ? (rows + 255) / 256 : 1184);
  PHK_CUDA(launch_pdl(tail_scatter_kernel, dim3(g2), dim3(256), (size_t)0, st, (const int*)t.index, (const int64_t*)t.pred_c,
                      (const float*)t.score_c, ids, pred_out, score_out, rows));
  PHK_LAUNCH_CHECK();
  return 0;
}

extern "C" int phk_sample_tail(const float* x_cond, const float* x_null, const float* gamma, const float* beta,
                               float cond_scale, const void* head_w, int64_t ldw, const float* head_b, int32_t b,
                               int32_t n, int32_t k, int32_t V, int32_t dim, float temperature, uint64_t seed,
                               uint64_t offset, const uint64_t* rng_state, const uint8_t* mask, int64_t* ids,
                               int64_t* pred_out, float* score_out, void* scratch, int64_t scratch_bytes,
                               phk_stream_t s) {
  return phk_sample_tail_rows(x_cond, x_null, gamma, beta, cond_scale, head_w, ldw, head_b, b, n, k, V, dim, temperature, seed,
                              offset, rng_state, mask, ids, pred_out, score_out, n, 0, scratch, scratch_bytes, s);
}

extern "C" int phk_rng_advance(uint64_t* rng_state, uint64_t stride, phk_stream_t s) {
  PHK_REQUIRE(rng_state, PHK_E_ARG, "phk_rng_advance: null pointer");
  PHK_CUDA(launch_pdl(rng_advance_kernel, dim3(1), dim3(32), (size_t)0, to_stream(s),
                      reinterpret_cast<unsigned long long*>(rng_state), (unsigned long long)stride));
  PHK_LAUNCH_CHECK();
  return 0;
}

extern "C" int phk_noise_probe(const uint32_t* bits_in, uint64_t seed, uint64_t offset, int64_t n, uint32_t* bits_out,
                               float* gumbel_out, phk_stream_t s) {
  PHK_REQUIRE(bits_out && gumbel_out, PHK_E_ARG, "phk_noise_probe: null pointer");
  PHK_REQUIRE(n >= 0, PHK_E_ARG, "phk_noise_probe: bad size");
  if (n == 0) return 0;
  const int64_t threads = (n + 3) / 4;
  const unsigned grid = (unsigned)((threads + 255) / 256 < 4736 ? (threads + 255) / 256 : 4736);
  PHK_CUDA(launch_pdl(noise_probe_kernel, dim3(grid), dim3(256), (size_t)0, to_stream(s), bits_in, seed, offset, n, bits_out,
                      gumbel_out));
  PHK_LAUNCH_CHECK();
  return 0;
}
