// Multi-tensor LARS step (moco/optimizer.py:10-43) over a device-resident table of tensors (include/mfvit.h).
//
// Every tensor is cut into chunks of MFV_LARS_CHUNK elements and every chunk is one CTA of 256 threads, so the 16.8 M
// element projector matrix (512 chunks) and a 384-element LayerNorm vector (1 chunk) spread over the SMs alike.
//   lars_norms_kernel : trust tensors only - fp32 partial sums of p^2 and dp^2 (dp = g + wd*p) of the chunk, written to
//                       workspace[2 * chunk + {0, 1}].
//   lars_update_kernel: each CTA re-sums its tensor's partials (a few hundred floats from L2), forms the trust ratio q
//                       and updates mu, p and the 16-bit shadows of its chunk.
// Reduction order (fixed, so two runs are bit-identical): within a chunk each thread keeps four lane sums over its
// 32 float4 (a serial run of 32 FMAs), then lanes -> warp butterfly -> 8 warps in a tree; across chunks each thread
// sums ceil(chunks / 256) partials serially, then the same warp / CTA tree.  Depth 32 + 10 + ceil(chunks / 256) + 8
// roundings: relative error of a norm^2 <= ~60 u32 for the largest tensor here.  No floating-point atomics.
#include "common.cuh"
#include "mfvit_internal.h"

namespace mfv {

constexpr int kLarsThreads = 256;
static_assert(MFV_LARS_CHUNK % (4 * kLarsThreads) == 0, "a chunk is a whole number of float4 per thread");

// Index of the record that owns chunk c: the number of records with chunk0 <= c, minus one (chunk0 ascending).  One
// pass of parallel loads over the table instead of a dependent binary search.
__device__ __forceinline__ int lars_find(const mfv_lars_tensor* __restrict__ table, int n_tensors, long long c) {
  int cnt = 0;
  for (int base = 0; base < n_tensors; base += kLarsThreads) {
    const int i = base + (int)threadIdx.x;
    cnt += __syncthreads_count(i < n_tensors && __ldg(&table[i].chunk0) <= c);
  }
  return cnt - 1;
}

// Sum of (a, b) over the CTA in a fixed order; the result is returned to every thread.
__device__ __forceinline__ float2 block_sum2(float a, float b, float2* red) {
  a = warp_sum(a);
  b = warp_sum(b);
  const int warp = threadIdx.x >> 5;
  if ((threadIdx.x & 31) == 0) red[warp] = make_float2(a, b);
  __syncthreads();
  const float2 w0 = red[0], w1 = red[1], w2 = red[2], w3 = red[3], w4 = red[4], w5 = red[5], w6 = red[6], w7 = red[7];
  __syncthreads();  // red is reused by the caller's next reduction
  return make_float2(((w0.x + w1.x) + (w2.x + w3.x)) + ((w4.x + w5.x) + (w6.x + w7.x)),
                     ((w0.y + w1.y) + (w2.y + w3.y)) + ((w4.y + w5.y) + (w6.y + w7.y)));
}

__global__ void __launch_bounds__(kLarsThreads)
lars_norms_kernel(const mfv_lars_tensor* __restrict__ table, int n_tensors, float* __restrict__ ws, float wd) {
  __shared__ float2 red[kLarsThreads / 32];
  const long long c = blockIdx.x;
  const int t = lars_find(table, n_tensors, c);
  if (!__ldg(&table[t].trust)) return;  // CTA-uniform
  const float* __restrict__ p = table[t].p;
  const float* __restrict__ g = table[t].g;
  const long long n = (long long)table[t].n;
  const long long lo = (c - (long long)table[t].chunk0) * MFV_LARS_CHUNK;
  const long long hi = min(lo + (long long)MFV_LARS_CHUNK, n);
  float4 sp = make_float4(0.f, 0.f, 0.f, 0.f), sd = sp;
  const long long lo4 = lo >> 2, hi4 = hi >> 2;
#pragma unroll 4
  for (long long i = lo4 + threadIdx.x; i < hi4; i += kLarsThreads) {
    const float4 pv = __ldg(reinterpret_cast<const float4*>(p) + i);
    const float4 gv = __ldg(reinterpret_cast<const float4*>(g) + i);
    const float dx = fmaf(wd, pv.x, gv.x), dy = fmaf(wd, pv.y, gv.y), dz = fmaf(wd, pv.z, gv.z),
                dw = fmaf(wd, pv.w, gv.w);
    sp.x = fmaf(pv.x, pv.x, sp.x); sp.y = fmaf(pv.y, pv.y, sp.y); sp.z = fmaf(pv.z, pv.z, sp.z); sp.w = fmaf(pv.w, pv.w, sp.w);
    sd.x = fmaf(dx, dx, sd.x); sd.y = fmaf(dy, dy, sd.y); sd.z = fmaf(dz, dz, sd.z); sd.w = fmaf(dw, dw, sd.w);
  }
  const long long tail = (hi4 << 2) + threadIdx.x;  // the last 1-3 elements of a tensor whose n is not a multiple of 4
  if (tail < hi) {
    const float pv = p[tail], dv = fmaf(wd, pv, g[tail]);
    sp.x = fmaf(pv, pv, sp.x);
    sd.x = fmaf(dv, dv, sd.x);
  }
  const float2 s = block_sum2((sp.x + sp.y) + (sp.z + sp.w), (sd.x + sd.y) + (sd.z + sd.w), red);
  if (threadIdx.x == 0) reinterpret_cast<float2*>(ws)[c] = s;
}

__device__ __forceinline__ uint2 bf16x4(float a, float b, float c, float d) {
  return make_uint2(pack_bf16(a, b), pack_bf16(c, d));
}
__device__ __forceinline__ uint2 f16x4(float a, float b, float c, float d) {
  return make_uint2(pack_f16(a, b), pack_f16(c, d));
}

__global__ void __launch_bounds__(kLarsThreads)
lars_update_kernel(const mfv_lars_tensor* __restrict__ table, int n_tensors, const float* __restrict__ ws,
                   float* __restrict__ q_out, const float* __restrict__ lr_dev, float mom, float wd, float eta) {
  __shared__ float2 red[kLarsThreads / 32];
  const long long c = blockIdx.x;
  const int t = lars_find(table, n_tensors, c);
  const mfv_lars_tensor rec = table[t];
  const bool trust = rec.trust != 0;
  float q = 1.f;
  if (trust) {  // CTA-uniform: the per-tensor finish, repeated identically by every chunk of the tensor
    const long long nch = (rec.n + MFV_LARS_CHUNK - 1) / MFV_LARS_CHUNK;
    float a = 0.f, b = 0.f;
    for (long long k = threadIdx.x; k < nch; k += kLarsThreads) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(ws) + rec.chunk0 + k);
      a += v.x;
      b += v.y;
    }
    const float2 s = block_sum2(a, b, red);
    const float pn = sqrtf(s.x), un = sqrtf(s.y);
    q = (pn > 0.f && un > 0.f) ? __fdiv_rn(eta * pn, un) : 1.f;
  }
  if (q_out != nullptr && c == rec.chunk0 && threadIdx.x == 0) q_out[t] = q;
  const float lr = __ldg(lr_dev);
  const float wdt = trust ? wd : 0.f;  // fmaf(0, p, g) == g exactly: one code path for both kinds of tensor
  float* __restrict__ p = rec.p;
  const float* __restrict__ g = rec.g;
  float* __restrict__ mu = rec.mu;
  __nv_bfloat16* __restrict__ sb = reinterpret_cast<__nv_bfloat16*>(rec.shadow_bf16);
  __half* __restrict__ sh = reinterpret_cast<__half*>(rec.shadow_f16);
  const long long lo = (c - (long long)rec.chunk0) * MFV_LARS_CHUNK;
  const long long hi = min(lo + (long long)MFV_LARS_CHUNK, (long long)rec.n);
  const long long lo4 = lo >> 2, hi4 = hi >> 2;
#pragma unroll 2
  for (long long i = lo4 + threadIdx.x; i < hi4; i += kLarsThreads) {
    float4 pv = reinterpret_cast<const float4*>(p)[i];
    const float4 gv = __ldg(reinterpret_cast<const float4*>(g) + i);
    float4 mv = reinterpret_cast<const float4*>(mu)[i];
    mv.x = fmaf(mom, mv.x, fmaf(wdt, pv.x, gv.x) * q);
    mv.y = fmaf(mom, mv.y, fmaf(wdt, pv.y, gv.y) * q);
    mv.z = fmaf(mom, mv.z, fmaf(wdt, pv.z, gv.z) * q);
    mv.w = fmaf(mom, mv.w, fmaf(wdt, pv.w, gv.w) * q);
    pv.x = fmaf(-lr, mv.x, pv.x);
    pv.y = fmaf(-lr, mv.y, pv.y);
    pv.z = fmaf(-lr, mv.z, pv.z);
    pv.w = fmaf(-lr, mv.w, pv.w);
    reinterpret_cast<float4*>(mu)[i] = mv;
    reinterpret_cast<float4*>(p)[i] = pv;
    if (sb) reinterpret_cast<uint2*>(sb)[i] = bf16x4(pv.x, pv.y, pv.z, pv.w);
    if (sh) reinterpret_cast<uint2*>(sh)[i] = f16x4(pv.x, pv.y, pv.z, pv.w);
  }
  const long long tail = (hi4 << 2) + threadIdx.x;
  if (tail < hi) {
    const float m = fmaf(mom, mu[tail], fmaf(wdt, p[tail], g[tail]) * q);
    const float np_ = fmaf(-lr, m, p[tail]);
    mu[tail] = m;
    p[tail] = np_;
    if (sb) sb[tail] = __float2bfloat16_rn(np_);
    if (sh) sh[tail] = __float2half_rn(np_);
  }
}

}  // namespace mfv

using namespace mfv;

extern "C" size_t mfv_lars_workspace_bytes(int64_t n_chunks) {
  return n_chunks > 0 ? (size_t)n_chunks * 2 * sizeof(float) : 0;
}

extern "C" int mfv_lars_step_dev(const mfv_lars_tensor* table_dev, int64_t n_tensors, int64_t n_chunks,
                                 float* workspace, float* q_out, const float* lr_dev, float momentum,
                                 float weight_decay, float trust_coefficient, void* stream) {
  if (n_tensors <= 0 || n_chunks <= 0) return MFV_OK;
  if (n_chunks < n_tensors || n_tensors > (1LL << 30) || n_chunks > 0x7fffffffLL) return MFV_ERR_SHAPE;
  if (!table_dev || !workspace || !lr_dev) return MFV_ERR_ARG;
  if ((reinterpret_cast<uintptr_t>(table_dev) | reinterpret_cast<uintptr_t>(workspace)) & 7) return MFV_ERR_ALIGN;
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  lars_norms_kernel<<<(unsigned)n_chunks, kLarsThreads, 0, st>>>(table_dev, (int)n_tensors, workspace, weight_decay);
  MFV_LAUNCH_CHECK();
  lars_update_kernel<<<(unsigned)n_chunks, kLarsThreads, 0, st>>>(table_dev, (int)n_tensors, workspace, q_out, lr_dev,
                                                                  momentum, weight_decay, trust_coefficient);
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}
