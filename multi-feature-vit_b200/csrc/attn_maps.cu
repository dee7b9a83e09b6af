// Explain pass of the encoder: per-head attention probabilities recomputed from the 16-bit qkv the forward stored, their
// mean over heads, and CLS attention rollout over a stack of such means (include/mfvit.h, DESIGN.md 3.9).
//
// The fused attention forward never writes P (it lives in TMEM / registers), so the maps are recomputed here, from the
// same stored q and k the forward read, with a plain two-pass softmax per row: no tensor cores and no reuse of the
// forward's lse (which follows the lazy-rescale convention of attn_tc.cu).
//   attn_probs_kernel  : one CTA per (32-query tile, image), 8 warps of 4 query rows each, looping over the heads.  K_h
//                        is staged in shared memory as 16-bit pairs (row stride D/2 + 1 words: lane j reads row j
//                        without bank conflicts), q_h as fp32.  Lane `lane` owns keys j = lane + 32 t of its rows, so
//                        the same thread accumulates the same head_mean element for every head (fixed order h = 0..H-1,
//                        no atomics).
//   attn_rollout_kernel: one CTA per image; v <- v (A_l + I) / 2 from block L-1 down to 0, each thread owning columns
//                        and summing over the rows i = 0..S-1 in order.
#include "common.cuh"
#include "mfvit_internal.h"

namespace mfv {

constexpr int AM_THREADS = 256;
constexpr int AM_WARPS = AM_THREADS / 32;
constexpr int AM_QT = 32;                       // query rows per CTA
constexpr int AM_ROWS = AM_QT / AM_WARPS;       // query rows per warp
constexpr int AM_MAX_S = 608;                   // keys per row held in registers: 19 per lane
constexpr int AM_KT = AM_MAX_S / 32;
constexpr int RO_THREADS = 256;
constexpr int RO_MAX_S = 1024;
constexpr int RO_COLS = RO_MAX_S / RO_THREADS;  // columns per thread

template <int D>
__host__ __device__ constexpr size_t am_smem_bytes(int S, bool mean) {
  return (size_t)S * (D / 2 + 1) * 4 + (size_t)AM_QT * D * 4 + (mean ? (size_t)AM_QT * S * 4 : 0);
}

template <int D, bool F16>
__global__ void __launch_bounds__(AM_THREADS, 1)
attn_probs_kernel(const uint16_t* __restrict__ qkv, float* __restrict__ probs, float* __restrict__ head_mean, int S,
                  int H, float scale) {
  constexpr int W = D / 2;       // 32-bit words of one head row
  constexpr int KS = W + 1;      // padded shared-memory row stride (words)
  extern __shared__ __align__(16) uint32_t am_smem[];
  uint32_t* Ks = am_smem;                                   // [S][KS]
  float* Qs = reinterpret_cast<float*>(Ks + (size_t)S * KS); // [AM_QT][D]
  float* acc = Qs + AM_QT * D;                              // [AM_QT][S] (head_mean only)
  const int tile = blockIdx.x, nb = blockIdx.y;
  const int i0 = tile * AM_QT;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const size_t row_words = (size_t)3 * H * W;               // one token's q, k, v of all heads
  const uint32_t* base = reinterpret_cast<const uint32_t*>(qkv) + (size_t)nb * S * row_words;

  for (int h = 0; h < H; ++h) {
    __syncthreads();  // the previous head's K / q are no longer read
    for (int idx = threadIdx.x; idx < S * W; idx += AM_THREADS) {
      const int j = idx / W, w = idx - j * W;
      Ks[j * KS + w] = __ldg(base + (size_t)j * row_words + (size_t)(H + h) * W + w);
    }
    for (int idx = threadIdx.x; idx < AM_QT * W; idx += AM_THREADS) {
      const int r = idx / W, w = idx - r * W;
      const int i = i0 + r;
      float2 v = make_float2(0.f, 0.f);
      if (i < S) {
        const uint32_t u = __ldg(base + (size_t)i * row_words + (size_t)h * W + w);
        v = F16 ? unpack_f16(u) : unpack_bf16(u);
      }
      Qs[r * D + 2 * w] = v.x;
      Qs[r * D + 2 * w + 1] = v.y;
    }
    __syncthreads();
    for (int rr = 0; rr < AM_ROWS; ++rr) {
      const int r = warp + rr * AM_WARPS;
      const int i = i0 + r;
      if (i >= S) break;  // warp-uniform
      float q[D];
#pragma unroll
      for (int d = 0; d < D; ++d) q[d] = Qs[r * D + d];
      float s[AM_KT];
      float m = -INFINITY;
#pragma unroll
      for (int t = 0; t < AM_KT; ++t) {
        const int j = lane + 32 * t;
        s[t] = -INFINITY;
        if (j < S) {
          // q . k as one fp32 FMA chain over d of exact 16-bit products, then the scale
          float a = 0.f;
          const uint32_t* kr = Ks + j * KS;
#pragma unroll
          for (int w = 0; w < W; ++w) {
            const float2 k2 = F16 ? unpack_f16(kr[w]) : unpack_bf16(kr[w]);
            a = fmaf(q[2 * w], k2.x, a);
            a = fmaf(q[2 * w + 1], k2.y, a);
          }
          s[t] = scale * a;
          m = fmaxf(m, s[t]);
        }
      }
      m = warp_max(m);
      float l = 0.f;
#pragma unroll
      for (int t = 0; t < AM_KT; ++t) {
        s[t] = (lane + 32 * t < S) ? __expf(s[t] - m) : 0.f;
        l += s[t];
      }
      l = warp_sum(l);
      float* prow = probs ? probs + (((size_t)nb * H + h) * S + i) * S : nullptr;
#pragma unroll
      for (int t = 0; t < AM_KT; ++t) {
        const int j = lane + 32 * t;
        if (j < S) {
          const float p = __fdiv_rn(s[t], l);
          if (prow) prow[j] = p;
          if (head_mean) acc[r * S + j] = (h == 0) ? p : acc[r * S + j] + p;
        }
      }
    }
  }
  if (head_mean) {
    // every acc element is read back by the thread that wrote it: no barrier needed
    for (int rr = 0; rr < AM_ROWS; ++rr) {
      const int r = warp + rr * AM_WARPS;
      const int i = i0 + r;
      if (i >= S) break;
      float* mrow = head_mean + ((size_t)nb * S + i) * S;
      for (int j = lane; j < S; j += 32) mrow[j] = __fdiv_rn(acc[r * S + j], (float)H);
    }
  }
}

__global__ void __launch_bounds__(RO_THREADS)
attn_rollout_kernel(const float* __restrict__ head_mean, float* __restrict__ out, int L, int NB, int S) {
  __shared__ float v[2][RO_MAX_S];
  const int nb = blockIdx.x;
  for (int j = threadIdx.x; j < S; j += RO_THREADS) v[0][j] = (j == 0) ? 1.f : 0.f;
  __syncthreads();
  int cur = 0;
  for (int l = L - 1; l >= 0; --l) {
    const float* A = head_mean + ((size_t)l * NB + nb) * S * S;
    float a[RO_COLS];
#pragma unroll
    for (int c = 0; c < RO_COLS; ++c) a[c] = 0.f;
#pragma unroll 4
    for (int i = 0; i < S; ++i) {
      const float vi = v[cur][i];
      const float* row = A + (size_t)i * S;
#pragma unroll
      for (int c = 0; c < RO_COLS; ++c) {
        const int j = threadIdx.x + c * RO_THREADS;
        if (j < S) a[c] = fmaf(vi, __ldg(row + j), a[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < RO_COLS; ++c) {
      const int j = threadIdx.x + c * RO_THREADS;
      if (j < S) v[cur ^ 1][j] = 0.5f * (a[c] + v[cur][j]);  // (v A + v) / 2: the halving is exact
    }
    cur ^= 1;
    __syncthreads();
  }
  for (int j = threadIdx.x; j < S; j += RO_THREADS) out[(size_t)nb * S + j] = v[cur][j];
}

template <int D, bool F16>
static int launch_probs(const void* qkv, float* probs, float* head_mean, int64_t NB, int64_t S, int64_t H, float scale,
                        cudaStream_t st) {
  static bool attr = false;
  if (!attr) {  // opt in once for the largest shape
    MFV_CUDA_CHECK(cudaFuncSetAttribute(attn_probs_kernel<D, F16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)am_smem_bytes<D>(AM_MAX_S, true)));
    attr = true;
  }
  const dim3 grid((unsigned)((S + AM_QT - 1) / AM_QT), (unsigned)NB);
  attn_probs_kernel<D, F16><<<grid, AM_THREADS, am_smem_bytes<D>((int)S, head_mean != nullptr), st>>>(
      static_cast<const uint16_t*>(qkv), probs, head_mean, (int)S, (int)H, scale);
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}

}  // namespace mfv

extern "C" int mfv_attn_probs(const void* qkv, int qkv_is_f16, float* probs, float* head_mean, int64_t NB, int64_t S,
                              int64_t H, int64_t D, float scale, void* stream) {
  using namespace mfv;
  if (!qkv || NB <= 0 || NB > 65535 || S < 1 || S > 577 || H <= 0 || (D != 32 && D != 64)) return MFV_ERR_SHAPE;
  if (reinterpret_cast<uintptr_t>(qkv) & 3) return MFV_ERR_ALIGN;
  if (!probs && !head_mean) return MFV_OK;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (D == 64)
    return qkv_is_f16 ? launch_probs<64, true>(qkv, probs, head_mean, NB, S, H, scale, st)
                      : launch_probs<64, false>(qkv, probs, head_mean, NB, S, H, scale, st);
  return qkv_is_f16 ? launch_probs<32, true>(qkv, probs, head_mean, NB, S, H, scale, st)
                    : launch_probs<32, false>(qkv, probs, head_mean, NB, S, H, scale, st);
}

extern "C" int mfv_attn_rollout(const float* head_mean, float* out, int64_t L, int64_t NB, int64_t S, void* stream) {
  using namespace mfv;
  if (!head_mean || !out || L <= 0 || NB <= 0 || NB > 2147483647LL || S < 1 || S > RO_MAX_S) return MFV_ERR_SHAPE;
  attn_rollout_kernel<<<(unsigned)NB, RO_THREADS, 0, reinterpret_cast<cudaStream_t>(stream)>>>(head_mean, out, (int)L,
                                                                                               (int)NB, (int)S);
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}
