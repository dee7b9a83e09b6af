// CLS-query cross-attention fusion of MF-ViT CA, forward and backward (SURVEY K7/K8, section 3.2).
//
// Reference semantics (FUS:35-65,126-157 + MOD:15-21,108-137), per sample b and direction d (d=0: the CXR CLS token
// queries the ENH patches; d=1: the ENH CLS token queries the CXR patches), with a = query branch, o = other branch:
//     rows r_0 = tok[a][b][0],  r_j = tok[o][b][j] (j >= 1);   xh_j = LN1_{eps 1e-5}(r_j)
//     q = Wq xh_0;  s_{h,j} = scale * q_h . (Wk xh_j)_h;  p_h = softmax_j s_h;  o_h = sum_j p_{h,j} (Wv xh_j)_h
//     c = r_0 + Wp o + bp;  e = r_0 + LN2_{eps 1e-6}(c);  fused_d = Wh e + bh;  x_d = Wvh r_0 + bvh
//     fused = fused_0 + fused_1
// Only one query row exists, so the K/V projections are folded to the query side:
//     t_h = Wk_h^T q_h  ->  s_{h,j} = scale * t_h . xh_j ;   u_h = sum_j p_{h,j} xh_j  ->  o_h = Wv_h u_h
// i.e. no [S,C]x[C,C] GEMM at all: one streaming pass over the 197 LN'd rows with a per-warp online softmax.
// Forward: ONE kernel, one CTA per (b, d), the two directions of a sample form a 2-CTA cluster and the d=1 CTA hands
// its partial logits to the d=0 CTA through distributed shared memory.  Backward: one kernel per (b, d) that
// recomputes the forward, back-propagates to every token row, and leaves the per-sample factors of the weight
// gradients in scratch; a second small kernel contracts them over the batch (deterministic, no atomics).
#include <cooperative_groups.h>
#include "common.cuh"
#include "mfvit_internal.h"

namespace cg = cooperative_groups;

namespace mfv {

constexpr int FUS_THREADS = 384;
constexpr int FUS_WARPS = FUS_THREADS / 32;
constexpr int MAX_HEADS = 4;
constexpr int MAX_NC = 8;

// per-(b,d) scratch record written by the backward main kernel, read by the weight-gradient kernel (floats)
//   [dq C][xh0 C][q C][dt heads*C][do C][u heads*C][dy C][o C][dz C][chat C][e C][f0 C][dg1 C][db1 C]
__host__ __device__ inline size_t fus_rec_floats(int C, int heads) { return (size_t)C * (12 + 2 * heads); }

template <int CPL>
__device__ __forceinline__ int col_of(int i, int lane) { return (i >> 2) * 128 + lane * 4 + (i & 3); }

template <int CPL>
__device__ __forceinline__ void load_row(float (&v)[CPL], const float* row, int lane) {
#pragma unroll
  for (int i = 0; i < CPL / 4; ++i) {
    const float4 t = reinterpret_cast<const float4*>(row)[i * 32 + lane];
    v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
  }
}
template <int CPL>
__device__ __forceinline__ void store_row(const float (&v)[CPL], float* row, int lane) {
#pragma unroll
  for (int i = 0; i < CPL / 4; ++i)
    reinterpret_cast<float4*>(row)[i * 32 + lane] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
}
template <int CPL>
__device__ __forceinline__ float dot_row(const float (&v)[CPL], const float* vec, int lane) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < CPL / 4; ++i) {
    const float4 t = reinterpret_cast<const float4*>(vec)[i * 32 + lane];
    s += v[4 * i] * t.x + v[4 * i + 1] * t.y + v[4 * i + 2] * t.z + v[4 * i + 3] * t.w;
  }
  return warp_sum(s);
}
// in-register LayerNorm statistics + normalisation (n = (v-mean)*rstd)
template <int CPL>
__device__ __forceinline__ void ln_stats(const float (&v)[CPL], float (&n)[CPL], float eps, float& rstd) {
  constexpr float invC = 1.0f / (CPL * 32);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) s += v[i];
  const float mean = warp_sum(s) * invC;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) { n[i] = v[i] - mean; ss += n[i] * n[i]; }
  rstd = rsqrtf(warp_sum(ss) * invC + eps);
#pragma unroll
  for (int i = 0; i < CPL; ++i) n[i] *= rstd;
}
// out[i] = W[i] . vec (+ bias[i]) for all rows i < C: one warp per output row, vec in shared memory
template <int CPL>
__device__ __forceinline__ void matvec_rows(const float* __restrict__ W, const float* vec, const float* bias,
                                            float* out, int warp, int lane) {
  constexpr int C = CPL * 32;
  // four weight rows per iteration: their loads are all in flight before the first reduction (one CTA streams six
  // 590 KB matrices out of L2 per sample, so the loop is load-latency bound)
  for (int i0 = warp; i0 < C; i0 += 4 * FUS_WARPS) {
    float w[4][CPL];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) load_row<CPL>(w[r], W + (size_t)i * C, lane);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) {
        const float s = dot_row<CPL>(w[r], vec, lane);
        if (lane == 0) out[i] = s + (bias ? bias[i] : 0.f);
      }
    }
  }
}

struct FusPtrs {  // one direction's parameters
  const float *ln1_w, *ln1_b, *wq, *wk, *wv, *proj_w, *proj_b, *ln2_w, *ln2_b, *head_w, *head_b, *vhead_w, *vhead_b;
};
__device__ __forceinline__ FusPtrs pick(const mfv_fusion_params& p, int d) {
  FusPtrs f;
  f.ln1_w = p.ln1_w[d]; f.ln1_b = p.ln1_b[d]; f.wq = p.wq[d]; f.wk = p.wk[d]; f.wv = p.wv[d];
  f.proj_w = p.proj_w[d]; f.proj_b = p.proj_b[d]; f.ln2_w = p.ln2_w[d]; f.ln2_b = p.ln2_b[d];
  f.head_w = p.head_w[d]; f.head_b = p.head_b[d]; f.vhead_w = p.vhead_w[d]; f.vhead_b = p.vhead_b[d];
  return f;
}

// Shared-memory vectors of the forward core (all length C unless noted)
struct FusSmem {
  float *g1, *b1, *f0, *n0, *xh0, *q, *t /*heads*C*/, *u /*heads*C*/, *o, *c, *chat, *e;
  float *merge;   // [FUS_WARPS][merge_slots(heads)][C] per-warp partials
  float *stat;    // [FUS_WARPS][heads][2] (m, l) ; then [heads] lse at stat_lse
  float *lse;     // [heads]
  float *misc;    // [8]: rho0, rhoc, ...
};
// per-warp slots of the merge buffer: one per head in the forward; the backward kernel also parks its two LN1
// weight-gradient partials (dg1, db1) there, so there are at least two even with one head
__host__ __device__ constexpr int merge_slots(int heads) { return heads < 2 ? 2 : heads; }
template <int CPL>
__device__ __forceinline__ FusSmem carve(float* base, int heads) {
  constexpr int C = CPL * 32;
  FusSmem s;
  float* p = base;
  s.g1 = p; p += C; s.b1 = p; p += C; s.f0 = p; p += C; s.n0 = p; p += C; s.xh0 = p; p += C; s.q = p; p += C;
  s.t = p; p += heads * C; s.u = p; p += heads * C; s.o = p; p += C; s.c = p; p += C; s.chat = p; p += C;
  s.e = p; p += C;
  s.merge = p; p += FUS_WARPS * merge_slots(heads) * C;
  s.stat = p; p += FUS_WARPS * MAX_HEADS * 2;
  s.lse = p; p += MAX_HEADS;
  s.misc = p; p += 8;
  return s;
}
template <int CPL>
__host__ __device__ constexpr size_t fus_smem_floats(int heads) {
  return (size_t)(CPL * 32) * (10 + 2 * heads) + (size_t)FUS_WARPS * merge_slots(heads) * (CPL * 32) + FUS_WARPS * MAX_HEADS * 2 +
         MAX_HEADS + 8;
}

// Forward core.  On return (after the trailing __syncthreads) smem holds f0,n0,xh0,q,t,lse,u,o,c,chat,e and
// misc[0] = rstd of row 0 (LN1), misc[1] = rstd of c (LN2).
template <int CPL>
__device__ void fusion_forward_core(const FusSmem& sm, const FusPtrs& P, const float* __restrict__ cls_row,
                                    const float* __restrict__ other_rows /* tok[o][b], row 0 unused */, int S,
                                    int heads, float scale) {
  constexpr int C = CPL * 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int hd = C / heads;
  for (int c = tid; c < C; c += FUS_THREADS) {
    sm.g1[c] = P.ln1_w[c];
    sm.b1[c] = P.ln1_b[c];
    sm.f0[c] = cls_row[c];
  }
  __syncthreads();
  if (warp == 0) {  // LN1 of the CLS row
    float v[CPL], n[CPL];
    load_row<CPL>(v, sm.f0, lane);
    float rstd;
    ln_stats<CPL>(v, n, 1e-5f, rstd);
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      sm.n0[c] = n[i];
      sm.xh0[c] = n[i] * sm.g1[c] + sm.b1[c];
    }
    if (lane == 0) sm.misc[0] = rstd;
  }
  __syncthreads();
  matvec_rows<CPL>(P.wq, sm.xh0, nullptr, sm.q, warp, lane);  // q = Wq xh0
  __syncthreads();
  // t[h][c] = sum_{i in head h} Wk[i][c] q[i]   (thread per column, coalesced over c)
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      const float* wk = P.wk + (size_t)(h * hd) * C + c;
#pragma unroll 16
      for (int i = 0; i < hd; ++i) acc += __ldg(wk + (size_t)i * C) * sm.q[h * hd + i];
      sm.t[h * C + c] = acc;
    }
  }
  __syncthreads();
  // streaming pass over the S rows: per-warp online softmax for each head, weighted sum of xh
  {
    float m[MAX_HEADS], l[MAX_HEADS], uacc[MAX_HEADS][CPL];
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h) {
      m[h] = -INFINITY; l[h] = 0.f;
#pragma unroll
      for (int i = 0; i < CPL; ++i) uacc[h][i] = 0.f;
    }
    float vn[CPL];  // next row of this warp, requested one iteration ahead (the pass is load-latency bound)
    if (warp < S) load_row<CPL>(vn, warp == 0 ? sm.f0 : other_rows + (size_t)warp * C, lane);
    for (int j = warp; j < S; j += FUS_WARPS) {
      float v[CPL], xh[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) v[i] = vn[i];
      if (j + FUS_WARPS < S) load_row<CPL>(vn, other_rows + (size_t)(j + FUS_WARPS) * C, lane);
      float rstd;
      ln_stats<CPL>(v, xh, 1e-5f, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = col_of<CPL>(i, lane);
        xh[i] = xh[i] * sm.g1[c] + sm.b1[c];
      }
#pragma unroll
      for (int h = 0; h < MAX_HEADS; ++h) {
        if (h < heads) {
          const float s = scale * dot_row<CPL>(xh, sm.t + h * C, lane);
          const float mn = fmaxf(m[h], s);
          const float a = __expf(m[h] - mn), p = __expf(s - mn);
          l[h] = l[h] * a + p;
#pragma unroll
          for (int i = 0; i < CPL; ++i) uacc[h][i] = uacc[h][i] * a + p * xh[i];
          m[h] = mn;
        }
      }
    }
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h) {
      if (h < heads) {
        store_row<CPL>(uacc[h], sm.merge + ((size_t)warp * heads + h) * C, lane);
        if (lane == 0) { sm.stat[(warp * MAX_HEADS + h) * 2] = m[h]; sm.stat[(warp * MAX_HEADS + h) * 2 + 1] = l[h]; }
      }
    }
  }
  __syncthreads();
  if (tid < heads) {  // global (m, l) per head -> lse
    float mm = -INFINITY;
    for (int w = 0; w < FUS_WARPS; ++w) mm = fmaxf(mm, sm.stat[(w * MAX_HEADS + tid) * 2]);
    float ll = 0.f;
    for (int w = 0; w < FUS_WARPS; ++w) {
      const float mw = sm.stat[(w * MAX_HEADS + tid) * 2];
      ll += (mw == -INFINITY) ? 0.f : sm.stat[(w * MAX_HEADS + tid) * 2 + 1] * __expf(mw - mm);
    }
    sm.lse[tid] = mm + __logf(ll);
  }
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      for (int w = 0; w < FUS_WARPS; ++w) {
        const float mw = sm.stat[(w * MAX_HEADS + h) * 2];
        if (mw != -INFINITY) acc += sm.merge[((size_t)w * heads + h) * C + c] * __expf(mw - sm.lse[h]);
      }
      sm.u[h * C + c] = acc;  // = sum_j softmax_j * xh_j
    }
  }
  __syncthreads();
  // o[i] = Wv[i] . u_{head(i)}
  for (int i0 = warp; i0 < C; i0 += 4 * FUS_WARPS) {
    float w[4][CPL];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) load_row<CPL>(w[r], P.wv + (size_t)i * C, lane);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) {
        const float s = dot_row<CPL>(w[r], sm.u + (i / hd) * C, lane);
        if (lane == 0) sm.o[i] = s;
      }
    }
  }
  __syncthreads();
  matvec_rows<CPL>(P.proj_w, sm.o, P.proj_b, sm.c, warp, lane);  // y = Wp o + bp (into c)
  __syncthreads();
  if (warp == 0) {  // c = f0 + y ; LN2 ; e = f0 + LN2(c)
    float v[CPL], n[CPL];
    load_row<CPL>(v, sm.c, lane);
#pragma unroll
    for (int i = 0; i < CPL; ++i) v[i] += sm.f0[col_of<CPL>(i, lane)];
    float rstd;
    ln_stats<CPL>(v, n, 1e-6f, rstd);
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      sm.c[c] = v[i];
      sm.chat[c] = n[i];
      sm.e[c] = sm.f0[c] + n[i] * __ldg(P.ln2_w + c) + __ldg(P.ln2_b + c);
    }
    if (lane == 0) sm.misc[1] = rstd;
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------ forward kernel
template <int CPL>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(FUS_THREADS, 1)
fusion_fwd_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, float* __restrict__ out_fused,
                  float* __restrict__ out_x, int B, int S, int heads, int NC, float scale) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  __shared__ float partial[MAX_NC];       // this CTA's fused logits
  __shared__ float peer_partial[MAX_NC];  // written by the d=1 CTA of the cluster (DSMEM)
  cg::cluster_group cluster = cg::this_cluster();
  const int d = blockIdx.x, b = blockIdx.y;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const FusSmem sm = carve<CPL>(fsm, heads);
  const FusPtrs P = pick(prm, d);
  const int a = d, o = 1 - d;
  const float* cls_row = tok + ((size_t)a * B + b) * S * C;
  const float* other = tok + ((size_t)o * B + b) * S * C;
  fusion_forward_core<CPL>(sm, P, cls_row, other, S, heads, scale);
  // heads: fused_d[n] = Wh[n].e + bh[n] ; x_d[n] = Wvh[n].f0 + bvh[n]
  for (int n = warp; n < 2 * NC; n += FUS_WARPS) {
    const bool is_x = n >= NC;
    const int nn = is_x ? n - NC : n;
    const float* W = is_x ? P.vhead_w : P.head_w;
    const float* bias = is_x ? P.vhead_b : P.head_b;
    if (W) {
      float w[CPL];
      load_row<CPL>(w, W + (size_t)nn * C, lane);
      const float s = dot_row<CPL>(w, is_x ? sm.f0 : sm.e, lane) + (bias ? bias[nn] : 0.f);
      if (lane == 0) {
        if (is_x) out_x[((size_t)d * B + b) * NC + nn] = s;
        else partial[nn] = s;
      }
    }
  }
  __syncthreads();
  if (d == 1 && threadIdx.x < NC) {
    float* remote = cluster.map_shared_rank(peer_partial, 0);
    remote[threadIdx.x] = partial[threadIdx.x];
  }
  cluster.sync();
  if (d == 0 && threadIdx.x < NC) out_fused[(size_t)b * NC + threadIdx.x] = partial[threadIdx.x] + peer_partial[threadIdx.x];
}

// ------------------------------------------------------------------------------------------------ backward kernel
template <int CPL>
__global__ void __launch_bounds__(FUS_THREADS, 1)
fusion_bwd_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, const float* __restrict__ d_fused,
                  const float* __restrict__ d_x, float* __restrict__ dtok, float* __restrict__ scratch, int B, int S,
                  int heads, int NC, float scale) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  const int d = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int hd = C / heads;
  const FusSmem sm = carve<CPL>(fsm, heads);
  // extra backward vectors after the forward block
  float* bw = fsm + fus_smem_floats<CPL>(heads);
  float* s_de = bw;            // dE = dz
  float* s_df0 = s_de + C;     // gradient accumulator of the raw CLS row
  float* s_dy = s_df0 + C;     // = dc
  float* s_do = s_dy + C;
  float* s_du = s_do + C;      // heads*C
  float* s_dt = s_du + heads * C;  // heads*C
  float* s_dq = s_dt + heads * C;
  float* s_dxh0 = s_dq + C;
  float* s_D = s_dxh0 + C;     // [heads] du_h . u_h
  float* s_dl = s_D + MAX_HEADS;  // [2*MAX_NC] upstream logits grads
  const FusPtrs P = pick(prm, d);
  const int a = d, o = 1 - d;
  const float* cls_row = tok + ((size_t)a * B + b) * S * C;
  const float* other = tok + ((size_t)o * B + b) * S * C;
  float* rec = scratch + ((size_t)b * 2 + d) * fus_rec_floats(C, heads);
  float* r_dq = rec; float* r_xh0 = r_dq + C; float* r_q = r_xh0 + C; float* r_dt = r_q + C;
  float* r_do = r_dt + heads * C; float* r_u = r_do + C; float* r_dy = r_u + heads * C; float* r_o = r_dy + C;
  float* r_dz = r_o + C; float* r_chat = r_dz + C; float* r_e = r_chat + C; float* r_f0 = r_e + C;
  float* r_dg1 = r_f0 + C; float* r_db1 = r_dg1 + C;

  fusion_forward_core<CPL>(sm, P, cls_row, other, S, heads, scale);

  if (tid < NC) {
    s_dl[tid] = d_fused[(size_t)b * NC + tid];
    s_dl[MAX_NC + tid] = (d_x && P.vhead_w) ? d_x[((size_t)d * B + b) * NC + tid] : 0.f;
  }
  __syncthreads();
  // de = Wh^T dfused ; df0 = de + Wvh^T dx
  for (int c = tid; c < C; c += FUS_THREADS) {
    float de = 0.f, dv = 0.f;
    for (int n = 0; n < NC; ++n) {
      de += __ldg(P.head_w + (size_t)n * C + c) * s_dl[n];
      if (P.vhead_w) dv += __ldg(P.vhead_w + (size_t)n * C + c) * s_dl[MAX_NC + n];
    }
    s_de[c] = de;
    s_df0[c] = de + dv;
  }
  __syncthreads();
  if (warp == 0) {  // LN2 backward: dc = rstd * (g - mean(g) - chat*mean(g*chat)), g = dz * gamma2
    float g[CPL], ch[CPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      ch[i] = sm.chat[c];
      g[i] = s_de[c] * __ldg(P.ln2_w + c);
      s1 += g[i];
      s2 += g[i] * ch[i];
    }
    constexpr float invC = 1.0f / C;
    const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
    const float rstd = sm.misc[1];
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      const float dc = rstd * (g[i] - c1 - ch[i] * c2);
      s_dy[c] = dc;
      s_df0[c] += dc;
    }
  }
  __syncthreads();
  // do = Wp^T dy   (thread per column k: sum_i Wp[i][k] dy[i])
  for (int k = tid; k < C; k += FUS_THREADS) {
    float acc = 0.f;
#pragma unroll 16
    for (int i = 0; i < C; ++i) acc += __ldg(P.proj_w + (size_t)i * C + k) * s_dy[i];
    s_do[k] = acc;
  }
  __syncthreads();
  // du_h[c] = sum_{i in h} Wv[i][c] do[i]
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      const float* wv = P.wv + (size_t)(h * hd) * C + c;
#pragma unroll 16
      for (int i = 0; i < hd; ++i) acc += __ldg(wv + (size_t)i * C) * s_do[h * hd + i];
      s_du[h * C + c] = acc;
    }
  }
  __syncthreads();
  if (warp < heads) {  // D_h = du_h . u_h
    float v[CPL];
    load_row<CPL>(v, s_du + warp * C, lane);
    const float dd = dot_row<CPL>(v, sm.u + warp * C, lane);
    if (lane == 0) s_D[warp] = dd;
  }
  __syncthreads();
  // second streaming pass: probabilities from lse, gradients of every row
  float dg1[CPL], db1[CPL];
  {
    float dtacc[MAX_HEADS][CPL];
#pragma unroll
    for (int i = 0; i < CPL; ++i) dg1[i] = db1[i] = 0.f;
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h)
#pragma unroll
      for (int i = 0; i < CPL; ++i) dtacc[h][i] = 0.f;
    float* drows = dtok + ((size_t)o * B + b) * S * C;
    float vn[CPL];  // next row, requested one iteration ahead
    if (warp < S) load_row<CPL>(vn, warp == 0 ? sm.f0 : other + (size_t)warp * C, lane);
    for (int j = warp; j < S; j += FUS_WARPS) {
      float v[CPL], n[CPL], xh[CPL], dxh[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) v[i] = vn[i];
      if (j + FUS_WARPS < S) load_row<CPL>(vn, other + (size_t)(j + FUS_WARPS) * C, lane);
      float rstd;
      ln_stats<CPL>(v, n, 1e-5f, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = col_of<CPL>(i, lane);
        xh[i] = n[i] * sm.g1[c] + sm.b1[c];
        dxh[i] = 0.f;
      }
#pragma unroll
      for (int h = 0; h < MAX_HEADS; ++h) {
        if (h < heads) {
          const float s = scale * dot_row<CPL>(xh, sm.t + h * C, lane);
          const float p = __expf(s - sm.lse[h]);
          const float dp = dot_row<CPL>(xh, s_du + h * C, lane);
          const float ds = p * (dp - s_D[h]);
          const float dss = ds * scale;
#pragma unroll
          for (int i = 0; i < CPL; ++i) {
            const int c = col_of<CPL>(i, lane);
            dtacc[h][i] += dss * xh[i];
            dxh[i] += p * s_du[h * C + c] + dss * sm.t[h * C + c];
          }
        }
      }
      if (j == 0) {
        // row 0 still needs the query-path gradient: stash, finish after dq is known
#pragma unroll
        for (int i = 0; i < CPL; ++i) s_dxh0[col_of<CPL>(i, lane)] = dxh[i];
      } else {
        float s1 = 0.f, s2 = 0.f, g[CPL];
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = col_of<CPL>(i, lane);
          dg1[i] += dxh[i] * n[i];
          db1[i] += dxh[i];
          g[i] = dxh[i] * sm.g1[c];
          s1 += g[i];
          s2 += g[i] * n[i];
        }
        constexpr float invC = 1.0f / C;
        const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
#pragma unroll
        for (int i = 0; i < CPL; ++i) g[i] = rstd * (g[i] - c1 - n[i] * c2);
        store_row<CPL>(g, drows + (size_t)j * C, lane);
      }
    }
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h)
      if (h < heads) store_row<CPL>(dtacc[h], sm.merge + ((size_t)warp * heads + h) * C, lane);
  }
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      for (int w = 0; w < FUS_WARPS; ++w) acc += sm.merge[((size_t)w * heads + h) * C + c];
      s_dt[h * C + c] = acc;
    }
  }
  __syncthreads();
  // dq[i] = Wk[i] . dt_{head(i)}
  for (int i0 = warp; i0 < C; i0 += 4 * FUS_WARPS) {
    float w[4][CPL];
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) load_row<CPL>(w[r], P.wk + (size_t)i * C, lane);
    }
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const int i = i0 + r * FUS_WARPS;
      if (i < C) {
        const float s = dot_row<CPL>(w[r], s_dt + (i / hd) * C, lane);
        if (lane == 0) s_dq[i] = s;
      }
    }
  }
  __syncthreads();
  // dxh0 += Wq^T dq
  for (int c = tid; c < C; c += FUS_THREADS) {
    float acc = 0.f;
#pragma unroll 16
    for (int i = 0; i < C; ++i) acc += __ldg(P.wq + (size_t)i * C + c) * s_dq[i];
    s_dxh0[c] += acc;
  }
  __syncthreads();
  // per-warp LN1 gamma/beta partials -> merge buffer (2 slots per warp)
  store_row<CPL>(dg1, sm.merge + ((size_t)warp * 2) * C, lane);
  store_row<CPL>(db1, sm.merge + ((size_t)warp * 2 + 1) * C, lane);
  __syncthreads();
  if (warp == 0) {  // LN1 backward of row 0, total CLS-row gradient
    float g[CPL], n[CPL], dxh[CPL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      n[i] = sm.n0[c];
      dxh[i] = s_dxh0[c];
      g[i] = dxh[i] * sm.g1[c];
      s1 += g[i];
      s2 += g[i] * n[i];
    }
    constexpr float invC = 1.0f / C;
    const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
    const float rstd = sm.misc[0];
    float* drow0 = dtok + ((size_t)a * B + b) * S * C;
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      drow0[c] = s_df0[c] + rstd * (g[i] - c1 - n[i] * c2);
    }
  }
  // scratch record for the batched weight-gradient contraction
  for (int c = tid; c < C; c += FUS_THREADS) {
    r_dq[c] = s_dq[c]; r_xh0[c] = sm.xh0[c]; r_q[c] = sm.q[c]; r_do[c] = s_do[c]; r_dy[c] = s_dy[c];
    r_o[c] = sm.o[c]; r_dz[c] = s_de[c]; r_chat[c] = sm.chat[c]; r_e[c] = sm.e[c]; r_f0[c] = sm.f0[c];
    for (int h = 0; h < heads; ++h) { r_dt[h * C + c] = s_dt[h * C + c]; r_u[h * C + c] = sm.u[h * C + c]; }
    float ag = s_dxh0[c] * sm.n0[c], ab = s_dxh0[c];  // row 0 contribution to dgamma1/dbeta1
    for (int w = 0; w < FUS_WARPS; ++w) {
      ag += sm.merge[((size_t)w * 2) * C + c];
      ab += sm.merge[((size_t)w * 2 + 1) * C + c];
    }
    r_dg1[c] = ag;
    r_db1[c] = ab;
  }
}

// Weight gradients: contraction of the per-sample records over the batch.  grid = (C/4, 5, 2):
//   y = 0: dWq[i][c] += sum_b dq[i] xh0[c]      y = 1: dWk[i][c] += sum_b q[i] dt_{h(i)}[c]
//   y = 2: dWv[i][c] += sum_b do[i] u_{h(i)}[c]  y = 3: dWp[i][c] += sum_b dy[i] o[c]
//   y = 4: vectors (ln1, ln2, proj bias, heads) - blockIdx.x == 0 only
template <int CPL>
__global__ void __launch_bounds__(FUS_THREADS)
fusion_wgrad_kernel(const float* __restrict__ scratch, const float* __restrict__ d_fused, const float* __restrict__ d_x,
                    const mfv_fusion_grads g, int B, int heads, int NC) {
  constexpr int C = CPL * 32;
  const int d = blockIdx.z, which = blockIdx.y;
  const int hd = C / heads;
  const size_t recf = fus_rec_floats(C, heads);
  const float* base = scratch + (size_t)d * recf;  // record of (b=0, d); stride 2*recf per sample
  const size_t bs = 2 * recf;
  const size_t off_dq = 0, off_xh0 = C, off_q = 2 * C, off_dt = 3 * C, off_do = off_dt + (size_t)heads * C,
               off_u = off_do + C, off_dy = off_u + (size_t)heads * C, off_o = off_dy + C, off_dz = off_o + C,
               off_chat = off_dz + C, off_e = off_chat + C, off_f0 = off_e + C, off_dg1 = off_f0 + C,
               off_db1 = off_dg1 + C;
  if (which < 4) {
    float* out = which == 0 ? g.wq[d] : which == 1 ? g.wk[d] : which == 2 ? g.wv[d] : g.proj_w[d];
    if (!out) return;
    const size_t offL = which == 0 ? off_dq : which == 1 ? off_q : which == 2 ? off_do : off_dy;
    const int i0 = blockIdx.x * 4;
    for (int c = threadIdx.x; c < C; c += FUS_THREADS) {
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 8
      for (int b = 0; b < B; ++b) {
        const float* rb = base + (size_t)b * bs;
#pragma unroll
        for (int r = 0; r < 4; ++r) {
          const int i = i0 + r;
          size_t offR;
          if (which == 0) offR = off_xh0;
          else if (which == 1) offR = off_dt + (size_t)(i / hd) * C;
          else if (which == 2) offR = off_u + (size_t)(i / hd) * C;
          else offR = off_o;
          acc[r] += rb[offL + i] * rb[offR + c];
        }
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) out[(size_t)(i0 + r) * C + c] += acc[r];
    }
  } else if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < C; c += FUS_THREADS) {
      float a_g1 = 0.f, a_b1 = 0.f, a_g2 = 0.f, a_b2 = 0.f, a_pb = 0.f;
      float hw[MAX_NC], vw[MAX_NC];
#pragma unroll
      for (int n = 0; n < MAX_NC; ++n) hw[n] = vw[n] = 0.f;
      for (int b = 0; b < B; ++b) {
        const float* rb = base + (size_t)b * bs;
        a_g1 += rb[off_dg1 + c];
        a_b1 += rb[off_db1 + c];
        const float dz = rb[off_dz + c];
        a_g2 += dz * rb[off_chat + c];
        a_b2 += dz;
        a_pb += rb[off_dy + c];
        const float e = rb[off_e + c], f0 = rb[off_f0 + c];
        for (int n = 0; n < NC; ++n) {
          hw[n] += d_fused[(size_t)b * NC + n] * e;
          if (d_x) vw[n] += d_x[((size_t)d * B + b) * NC + n] * f0;
        }
      }
      if (g.ln1_w[d]) g.ln1_w[d][c] += a_g1;
      if (g.ln1_b[d]) g.ln1_b[d][c] += a_b1;
      if (g.ln2_w[d]) g.ln2_w[d][c] += a_g2;
      if (g.ln2_b[d]) g.ln2_b[d][c] += a_b2;
      if (g.proj_b[d]) g.proj_b[d][c] += a_pb;
      for (int n = 0; n < NC; ++n) {
        if (g.head_w[d]) g.head_w[d][(size_t)n * C + c] += hw[n];
        if (g.vhead_w[d]) g.vhead_w[d][(size_t)n * C + c] += vw[n];
      }
    }
    if ((int)threadIdx.x < NC) {
      float hb = 0.f, vb = 0.f;
      for (int b = 0; b < B; ++b) {
        hb += d_fused[(size_t)b * NC + threadIdx.x];
        if (d_x) vb += d_x[((size_t)d * B + b) * NC + threadIdx.x];
      }
      if (g.head_b[d]) g.head_b[d][threadIdx.x] += hb;
      if (g.vhead_b[d]) g.vhead_b[d][threadIdx.x] += vb;
    }
  }
}


// =====================================================================================================================
// Batched path (round 2).  The single-kernel forward / backward above give every (sample, direction) CTA its own pass
// over six 590 KB weight matrices: 64 CTAs x 2.4 MB of L2 reads behind a chain of dependent mat-vecs (78 us forward,
// 146 us backward at 32 pairs).  Here the mat-vecs of ALL samples of a direction are one small batched product each -
// every weight matrix is read once per launch - and only the per-sample work (LayerNorms, the streaming softmax pass
// over the 197 rows, the heads) stays per instance:
//   forward : ln0 -> Q = Xh0 Wq^T -> T_h = Wk_h^T q_h -> streaming pass (u, lse) -> O = Wv u -> Y = Wp o + bp -> LN2 + heads
//   backward: heads/LN2 -> dO = Wp^T dY -> dU_h = Wv_h^T dO_h -> streaming pass (d rows, dT) -> dQ = Wk dT
//             -> dXh0 += Wq^T dQ -> LN1 backward of the CLS row + the records the weight-gradient kernel contracts
// Per-instance state lives in the caller's `saved` buffer: [records B*2*recf][forward state 2B*FWD][backward temps 2B*BWT].
// Instance index r = b * 2 + d (the order of the records).
__host__ __device__ inline size_t fus2_fwd_floats(int C, int heads) { return (size_t)C * (8 + 2 * heads) + 16; }
__host__ __device__ inline size_t fus2_bwt_floats(int C, int heads) { return (size_t)C * (2 + heads) + 16; }
struct Fus2Off {  // offsets (floats) inside one instance's forward-state block
  size_t f0, n0, xh0, q, t, u, o, y, chat, e, misc;  // misc: [0] rstd0, [1] rstd2, [4..8) lse
  __host__ __device__ Fus2Off(int C, int heads) {
    f0 = 0; n0 = C; xh0 = 2 * (size_t)C; q = 3 * (size_t)C; t = 4 * (size_t)C; u = t + (size_t)heads * C;
    o = u + (size_t)heads * C; y = o + C; chat = y + C; e = chat + C; misc = e + C;
  }
};
struct Fus2Rec {  // offsets inside one record (layout of fus_rec_floats, read by fusion_wgrad_kernel)
  size_t dq, xh0, q, dt, d_o, u, dy, o, dz, chat, e, f0, dg1, db1;
  __host__ __device__ Fus2Rec(int C, int heads) {
    dq = 0; xh0 = C; q = 2 * (size_t)C; dt = 3 * (size_t)C; d_o = dt + (size_t)heads * C; u = d_o + C;
    dy = u + (size_t)heads * C; o = dy + C; dz = o + C; chat = dz + C; e = chat + C; f0 = e + C; dg1 = f0 + C;
    db1 = dg1 + C;
  }
};
struct Fus2Bwt {  // backward temporaries per instance
  size_t du, dxh0, df0, misc;
  __host__ __device__ Fus2Bwt(int C, int heads) { du = 0; dxh0 = (size_t)heads * C; df0 = dxh0 + C; misc = df0 + C; }
};

// LN1 of the CLS row of every instance: one warp per instance.
template <int CPL>
__global__ void __launch_bounds__(128)
fus2_ln0_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, float* __restrict__ fwd, size_t fstride,
                int B, int S, int heads) {
  constexpr int C = CPL * 32;
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (r >= 2 * B) return;
  const int b = r >> 1, d = r & 1;
  const Fus2Off O(C, heads);
  float* st = fwd + (size_t)r * fstride;
  const float* row = tok + ((size_t)d * B + b) * S * C;
  float v[CPL], n[CPL];
  load_row<CPL>(v, row, lane);
  float rstd;
  ln_stats<CPL>(v, n, 1e-5f, rstd);
  float xh[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = col_of<CPL>(i, lane);
    xh[i] = n[i] * __ldg(prm.ln1_w[d] + c) + __ldg(prm.ln1_b[d] + c);
  }
  store_row<CPL>(v, st + O.f0, lane);
  store_row<CPL>(n, st + O.n0, lane);
  store_row<CPL>(xh, st + O.xh0, lane);
  if (lane == 0) st[O.misc] = rstd;
}

// out[r][i] = W_d[i] . vec[r][sel(i)] (+ bias_d[i]) for the instances r = b*2+d of direction d = blockIdx.y, 32 instances
// per blockIdx.z.  The 32 vectors are staged in shared memory with every load in flight at once (the stage is latency-
// bound: a dependent chain of L2 reads is what made the first version slower than the single-kernel path); one warp per
// weight row, held in registers.  nsel = 1, or heads (the vector of the head the 8 output rows of the block belong to:
// o = Wv u_h, dq = Wk dt_h; hd is a multiple of 8).
constexpr int FUS2_RB = 32;  // instances per rowdot CTA
constexpr int FUS2_CB = 16;  // instances per coldot CTA
template <int CPL>
__global__ void __launch_bounds__(256)
fus2_rowdot_kernel(const float* __restrict__ W0, const float* __restrict__ W1, const float* __restrict__ bias0,
                   const float* __restrict__ bias1, const float* __restrict__ in, size_t in_stride,
                   float* __restrict__ out, size_t out_stride, int B, int nsel, int hd) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];  // [FUS2_RB][C]
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int d = blockIdx.y;
  const int b_base = blockIdx.z * FUS2_RB;
  const int i = blockIdx.x * 8 + warp;
  const float* W = d ? W1 : W0;
  const float* bias = d ? bias1 : bias0;
  const size_t sel = nsel > 1 ? (size_t)((blockIdx.x * 8) / hd) * C : 0;
  for (int idx = threadIdx.x; idx < FUS2_RB * (C / 4); idx += 256) {
    const int k = idx / (C / 4), c4 = idx - k * (C / 4);
    const int b = min(b_base + k, B - 1);
    reinterpret_cast<float4*>(fsm)[idx] = reinterpret_cast<const float4*>(in + (size_t)(b * 2 + d) * in_stride + sel)[c4];
  }
  float w[CPL];
  load_row<CPL>(w, W + (size_t)i * C, lane);
  const float bi = bias ? __ldg(bias + i) : 0.f;
  __syncthreads();
  float mine = 0.f;  // lane k keeps the result of instance k
#pragma unroll 4
  for (int k = 0; k < FUS2_RB; ++k) {
    const float s = dot_row<CPL>(w, fsm + (size_t)k * C, lane);
    if (lane == k) mine = s;
  }
  const int b = b_base + lane;
  if (b < B) out[(size_t)(b * 2 + d) * out_stride + i] = mine + bi;
}

// out[r][s][c] (+)= sum_{i in segment s} W_d[i][c] * vec[r][i]   (W^T products: t_h = Wk_h^T q_h, do = Wp^T dy, du_h = Wv_h^T
// do_h, dxh0 += Wq^T dq).  grid (C/32, 2, ceil(B/16)): a CTA owns 32 columns for 16 instances.  Both the W[:, 32 columns]
// slice (48 KB) and the 16 instance vectors (24 KB) are staged in shared memory with all loads in flight at once;
// thread = (column, 2 instances).
template <int CPL>
__global__ void __launch_bounds__(256)
fus2_coldot_kernel(const float* __restrict__ W0, const float* __restrict__ W1, const float* __restrict__ in,
                   size_t in_stride, float* __restrict__ out, size_t out_stride, int B, int segs, int accumulate) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  float* ws = fsm;                 // [C][32]
  float* vec = fsm + C * 32;       // [FUS2_CB][C]
  griddep_wait();
  griddep_launch();
  const int d = blockIdx.y;
  const int b_base = blockIdx.z * FUS2_CB;
  const float* W = (d ? W1 : W0) + blockIdx.x * 32;
  for (int idx = threadIdx.x; idx < C * 8; idx += 256) {  // 8 float4 per weight row slice
    const int i = idx >> 3, c4 = idx & 7;
    reinterpret_cast<float4*>(ws)[idx] = __ldg(reinterpret_cast<const float4*>(W + (size_t)i * C) + c4);
  }
  for (int idx = threadIdx.x; idx < FUS2_CB * (C / 4); idx += 256) {
    const int k = idx / (C / 4), c4 = idx - k * (C / 4);
    const int b = min(b_base + k, B - 1);
    reinterpret_cast<float4*>(vec)[idx] = reinterpret_cast<const float4*>(in + (size_t)(b * 2 + d) * in_stride)[c4];
  }
  __syncthreads();
  const int cl = threadIdx.x & 31;
  const int c = blockIdx.x * 32 + cl;
  const int k0 = (threadIdx.x >> 5) * 2;  // this thread's two instances: k0, k0 + 1
  const int seg_len = C / segs;
  for (int s = 0; s < segs; ++s) {
    float a0 = 0.f, a1 = 0.f;
    const float* wp = ws + (size_t)(s * seg_len) * 32 + cl;
    const float* v0 = vec + (size_t)k0 * C + s * seg_len;
    const float* v1 = v0 + C;
#pragma unroll 8
    for (int i = 0; i < seg_len; ++i) {
      const float w = wp[i * 32];
      a0 = fmaf(w, v0[i], a0);
      a1 = fmaf(w, v1[i], a1);
    }
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int b = b_base + k0 + k;
      if (b < B) {
        float* o = out + (size_t)(b * 2 + d) * out_stride + (size_t)s * C + c;
        const float a = k ? a1 : a0;
        *o = accumulate ? *o + a : a;
      }
    }
  }
}

// Streaming pass of the forward for one instance: online softmax per head over the S LayerNorm'd rows -> u, lse.
template <int CPL>
__global__ void __launch_bounds__(FUS_THREADS, 1)
fus2_stream_fwd_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, float* __restrict__ fwd, size_t fstride,
                       int B, int S, int heads, float scale) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  griddep_wait();
  griddep_launch();
  const int d = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Fus2Off O(C, heads);
  float* st = fwd + (size_t)(b * 2 + d) * fstride;
  float* s_g1 = fsm; float* s_b1 = s_g1 + C; float* s_f0 = s_b1 + C; float* s_t = s_f0 + C;
  float* s_merge = s_t + heads * C;                           // [FUS_WARPS][heads][C]
  float* s_stat = s_merge + (size_t)FUS_WARPS * heads * C;     // [FUS_WARPS][MAX_HEADS][2]
  float* s_lse = s_stat + FUS_WARPS * MAX_HEADS * 2;
  const float* other = tok + ((size_t)(1 - d) * B + b) * S * C;
  for (int c = tid; c < C; c += FUS_THREADS) {
    s_g1[c] = prm.ln1_w[d][c];
    s_b1[c] = prm.ln1_b[d][c];
    s_f0[c] = st[O.f0 + c];
    for (int h = 0; h < heads; ++h) s_t[h * C + c] = st[O.t + (size_t)h * C + c];
  }
  __syncthreads();
  {
    float m[MAX_HEADS], l[MAX_HEADS], uacc[MAX_HEADS][CPL];
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h) {
      m[h] = -INFINITY; l[h] = 0.f;
#pragma unroll
      for (int i = 0; i < CPL; ++i) uacc[h][i] = 0.f;
    }
    float vn[CPL];
    if (warp < S) load_row<CPL>(vn, warp == 0 ? s_f0 : other + (size_t)warp * C, lane);
    for (int j = warp; j < S; j += FUS_WARPS) {
      float v[CPL], xh[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) v[i] = vn[i];
      if (j + FUS_WARPS < S) load_row<CPL>(vn, other + (size_t)(j + FUS_WARPS) * C, lane);
      float rstd;
      ln_stats<CPL>(v, xh, 1e-5f, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = col_of<CPL>(i, lane);
        xh[i] = xh[i] * s_g1[c] + s_b1[c];
      }
#pragma unroll
      for (int h = 0; h < MAX_HEADS; ++h) {
        if (h < heads) {
          const float s = scale * dot_row<CPL>(xh, s_t + h * C, lane);
          const float mn = fmaxf(m[h], s);
          const float a = __expf(m[h] - mn), p = __expf(s - mn);
          l[h] = l[h] * a + p;
#pragma unroll
          for (int i = 0; i < CPL; ++i) uacc[h][i] = uacc[h][i] * a + p * xh[i];
          m[h] = mn;
        }
      }
    }
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h) {
      if (h < heads) {
        store_row<CPL>(uacc[h], s_merge + ((size_t)warp * heads + h) * C, lane);
        if (lane == 0) { s_stat[(warp * MAX_HEADS + h) * 2] = m[h]; s_stat[(warp * MAX_HEADS + h) * 2 + 1] = l[h]; }
      }
    }
  }
  __syncthreads();
  if (tid < heads) {
    float mm = -INFINITY;
    for (int w = 0; w < FUS_WARPS; ++w) mm = fmaxf(mm, s_stat[(w * MAX_HEADS + tid) * 2]);
    float ll = 0.f;
    for (int w = 0; w < FUS_WARPS; ++w) {
      const float mw = s_stat[(w * MAX_HEADS + tid) * 2];
      ll += (mw == -INFINITY) ? 0.f : s_stat[(w * MAX_HEADS + tid) * 2 + 1] * __expf(mw - mm);
    }
    s_lse[tid] = mm + __logf(ll);
    st[O.misc + 4 + tid] = s_lse[tid];
  }
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      for (int w = 0; w < FUS_WARPS; ++w) {
        const float mw = s_stat[(w * MAX_HEADS + h) * 2];
        if (mw != -INFINITY) acc += s_merge[((size_t)w * heads + h) * C + c] * __expf(mw - s_lse[h]);
      }
      st[O.u + (size_t)h * C + c] = acc;
    }
  }
}

// c = f0 + y ; LN2 ; e = f0 + LN2(c) ; logits.  One CTA per sample, warp d = direction d; fused = fused_0 + fused_1.
template <int CPL>
__global__ void __launch_bounds__(64)
fus2_ln2_heads_kernel(const mfv_fusion_params prm, float* __restrict__ fwd, size_t fstride, float* __restrict__ out_fused,
                      float* __restrict__ out_x, int B, int heads, int NC) {
  constexpr int C = CPL * 32;
  __shared__ float part[2][MAX_NC];
  griddep_wait();
  griddep_launch();
  const int b = blockIdx.x, d = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Fus2Off O(C, heads);
  float* st = fwd + (size_t)(b * 2 + d) * fstride;
  float f0[CPL], v[CPL], n[CPL], e[CPL];
  load_row<CPL>(f0, st + O.f0, lane);
  load_row<CPL>(v, st + O.y, lane);
#pragma unroll
  for (int i = 0; i < CPL; ++i) v[i] += f0[i];
  float rstd;
  ln_stats<CPL>(v, n, 1e-6f, rstd);
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = col_of<CPL>(i, lane);
    e[i] = f0[i] + n[i] * __ldg(prm.ln2_w[d] + c) + __ldg(prm.ln2_b[d] + c);
  }
  store_row<CPL>(n, st + O.chat, lane);
  store_row<CPL>(e, st + O.e, lane);
  if (lane == 0) st[O.misc + 1] = rstd;
  for (int n_ = 0; n_ < NC; ++n_) {
    const float s = dot_row<CPL>(e, prm.head_w[d] + (size_t)n_ * C, lane) + (prm.head_b[d] ? prm.head_b[d][n_] : 0.f);
    if (lane == 0) part[d][n_] = s;
    if (prm.vhead_w[d]) {
      const float x = dot_row<CPL>(f0, prm.vhead_w[d] + (size_t)n_ * C, lane) + (prm.vhead_b[d] ? prm.vhead_b[d][n_] : 0.f);
      if (lane == 0) out_x[((size_t)d * B + b) * NC + n_] = x;
    }
  }
  __syncthreads();
  if (threadIdx.x < NC) out_fused[(size_t)b * NC + threadIdx.x] = part[0][threadIdx.x] + part[1][threadIdx.x];
}

// Backward of the heads and LN2 for one instance (one warp): dz = Wh^T dfused, df0 = dz + Wvh^T dx, dy = LN2'(dz), df0 += dy.
template <int CPL>
__global__ void __launch_bounds__(128)
fus2_bwd_heads_kernel(const mfv_fusion_params prm, const float* __restrict__ d_fused, const float* __restrict__ d_x,
                      const float* __restrict__ fwd, size_t fstride, float* __restrict__ rec, size_t rstride,
                      float* __restrict__ bwt, size_t bstride, int B, int heads, int NC) {
  constexpr int C = CPL * 32;
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (r >= 2 * B) return;
  const int b = r >> 1, d = r & 1;
  const Fus2Off O(C, heads);
  const Fus2Rec R(C, heads);
  const Fus2Bwt T(C, heads);
  const float* st = fwd + (size_t)r * fstride;
  float* rc = rec + (size_t)r * rstride;
  float* bt = bwt + (size_t)r * bstride;
  float de[CPL], df0[CPL], ch[CPL], g[CPL];
  load_row<CPL>(ch, st + O.chat, lane);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = col_of<CPL>(i, lane);
    float a = 0.f, v = 0.f;
    for (int n = 0; n < NC; ++n) {
      a += __ldg(prm.head_w[d] + (size_t)n * C + c) * d_fused[(size_t)b * NC + n];
      if (d_x && prm.vhead_w[d]) v += __ldg(prm.vhead_w[d] + (size_t)n * C + c) * d_x[((size_t)d * B + b) * NC + n];
    }
    de[i] = a;
    df0[i] = a + v;
    g[i] = a * __ldg(prm.ln2_w[d] + c);
    s1 += g[i];
    s2 += g[i] * ch[i];
  }
  constexpr float invC = 1.0f / C;
  const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
  const float rstd = st[O.misc + 1];
  float dy[CPL];
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    dy[i] = rstd * (g[i] - c1 - ch[i] * c2);
    df0[i] += dy[i];
  }
  store_row<CPL>(de, rc + R.dz, lane);
  store_row<CPL>(dy, rc + R.dy, lane);
  store_row<CPL>(df0, bt + T.df0, lane);
}

// Streaming pass of the backward for one instance: gradients of every row of the other branch, dt, the CLS-row stash.
template <int CPL>
__global__ void __launch_bounds__(FUS_THREADS, 1)
fus2_stream_bwd_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, const float* __restrict__ fwd,
                       size_t fstride, float* __restrict__ rec, size_t rstride, float* __restrict__ bwt, size_t bstride,
                       float* __restrict__ dtok, int B, int S, int heads, float scale) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  griddep_wait();
  griddep_launch();
  const int d = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int r = b * 2 + d;
  const Fus2Off O(C, heads);
  const Fus2Rec R(C, heads);
  const Fus2Bwt T(C, heads);
  const float* st = fwd + (size_t)r * fstride;
  float* rc = rec + (size_t)r * rstride;
  float* bt = bwt + (size_t)r * bstride;
  float* s_g1 = fsm; float* s_b1 = s_g1 + C; float* s_f0 = s_b1 + C; float* s_t = s_f0 + C;
  float* s_du = s_t + heads * C;
  float* s_merge = s_du + heads * C;                         // [FUS_WARPS][max(heads, 2)][C]
  float* s_lse = s_merge + (size_t)FUS_WARPS * MAX_HEADS * C;
  float* s_D = s_lse + MAX_HEADS;
  const float* other = tok + ((size_t)(1 - d) * B + b) * S * C;
  for (int c = tid; c < C; c += FUS_THREADS) {
    s_g1[c] = prm.ln1_w[d][c];
    s_b1[c] = prm.ln1_b[d][c];
    s_f0[c] = st[O.f0 + c];
    for (int h = 0; h < heads; ++h) {
      s_t[h * C + c] = st[O.t + (size_t)h * C + c];
      s_du[h * C + c] = bt[T.du + (size_t)h * C + c];
    }
  }
  if (tid < heads) s_lse[tid] = st[O.misc + 4 + tid];
  __syncthreads();
  if (warp < heads) {  // D_h = du_h . u_h
    float v[CPL];
    load_row<CPL>(v, s_du + warp * C, lane);
    const float dd = dot_row<CPL>(v, st + O.u + (size_t)warp * C, lane);
    if (lane == 0) s_D[warp] = dd;
  }
  __syncthreads();
  float dg1[CPL], db1[CPL];
  {
    float dtacc[MAX_HEADS][CPL];
#pragma unroll
    for (int i = 0; i < CPL; ++i) dg1[i] = db1[i] = 0.f;
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h)
#pragma unroll
      for (int i = 0; i < CPL; ++i) dtacc[h][i] = 0.f;
    float* drows = dtok + ((size_t)(1 - d) * B + b) * S * C;
    float vn[CPL];
    if (warp < S) load_row<CPL>(vn, warp == 0 ? s_f0 : other + (size_t)warp * C, lane);
    for (int j = warp; j < S; j += FUS_WARPS) {
      float v[CPL], n[CPL], xh[CPL], dxh[CPL];
#pragma unroll
      for (int i = 0; i < CPL; ++i) v[i] = vn[i];
      if (j + FUS_WARPS < S) load_row<CPL>(vn, other + (size_t)(j + FUS_WARPS) * C, lane);
      float rstd;
      ln_stats<CPL>(v, n, 1e-5f, rstd);
#pragma unroll
      for (int i = 0; i < CPL; ++i) {
        const int c = col_of<CPL>(i, lane);
        xh[i] = n[i] * s_g1[c] + s_b1[c];
        dxh[i] = 0.f;
      }
#pragma unroll
      for (int h = 0; h < MAX_HEADS; ++h) {
        if (h < heads) {
          const float s = scale * dot_row<CPL>(xh, s_t + h * C, lane);
          const float p = __expf(s - s_lse[h]);
          const float dp = dot_row<CPL>(xh, s_du + h * C, lane);
          const float dss = p * (dp - s_D[h]) * scale;
#pragma unroll
          for (int i = 0; i < CPL; ++i) {
            const int c = col_of<CPL>(i, lane);
            dtacc[h][i] += dss * xh[i];
            dxh[i] += p * s_du[h * C + c] + dss * s_t[h * C + c];
          }
        }
      }
      if (j == 0) {
        store_row<CPL>(dxh, bt + T.dxh0, lane);  // the CLS row still needs the query-path gradient (Wq^T dq)
      } else {
        float s1 = 0.f, s2 = 0.f, g[CPL];
#pragma unroll
        for (int i = 0; i < CPL; ++i) {
          const int c = col_of<CPL>(i, lane);
          dg1[i] += dxh[i] * n[i];
          db1[i] += dxh[i];
          g[i] = dxh[i] * s_g1[c];
          s1 += g[i];
          s2 += g[i] * n[i];
        }
        constexpr float invC = 1.0f / C;
        const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
#pragma unroll
        for (int i = 0; i < CPL; ++i) g[i] = rstd * (g[i] - c1 - n[i] * c2);
        store_row<CPL>(g, drows + (size_t)j * C, lane);
      }
    }
#pragma unroll
    for (int h = 0; h < MAX_HEADS; ++h)
      if (h < heads) store_row<CPL>(dtacc[h], s_merge + ((size_t)warp * MAX_HEADS + h) * C, lane);
  }
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      for (int w = 0; w < FUS_WARPS; ++w) acc += s_merge[((size_t)w * MAX_HEADS + h) * C + c];
      rc[R.dt + (size_t)h * C + c] = acc;
    }
  }
  __syncthreads();
  store_row<CPL>(dg1, s_merge + ((size_t)warp * MAX_HEADS) * C, lane);
  store_row<CPL>(db1, s_merge + ((size_t)warp * MAX_HEADS + 1) * C, lane);
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {  // rows j >= 1; the CLS row's share is added by fus2_bwd_row0_kernel
    float ag = 0.f, ab = 0.f;
    for (int w = 0; w < FUS_WARPS; ++w) {
      ag += s_merge[((size_t)w * MAX_HEADS) * C + c];
      ab += s_merge[((size_t)w * MAX_HEADS + 1) * C + c];
    }
    rc[R.dg1 + c] = ag;
    rc[R.db1 + c] = ab;
  }
}

// LN1 backward of the CLS row (now that dxh0 is complete) -> its dtok row; completes the record for the weight gradients.
template <int CPL>
__global__ void __launch_bounds__(128)
fus2_bwd_row0_kernel(const mfv_fusion_params prm, const float* __restrict__ fwd, size_t fstride, float* __restrict__ rec,
                     size_t rstride, const float* __restrict__ bwt, size_t bstride, float* __restrict__ dtok, int B, int S,
                     int heads) {
  constexpr int C = CPL * 32;
  griddep_wait();
  griddep_launch();
  const int lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (r >= 2 * B) return;
  const int b = r >> 1, d = r & 1;
  const Fus2Off O(C, heads);
  const Fus2Rec R(C, heads);
  const Fus2Bwt T(C, heads);
  const float* st = fwd + (size_t)r * fstride;
  float* rc = rec + (size_t)r * rstride;
  const float* bt = bwt + (size_t)r * bstride;
  float n[CPL], dxh[CPL], g[CPL], df0[CPL], dg1[CPL], db1[CPL];
  load_row<CPL>(n, st + O.n0, lane);
  load_row<CPL>(dxh, bt + T.dxh0, lane);
  load_row<CPL>(df0, bt + T.df0, lane);
  load_row<CPL>(dg1, rc + R.dg1, lane);
  load_row<CPL>(db1, rc + R.db1, lane);
  float s1 = 0.f, s2 = 0.f;
#pragma unroll
  for (int i = 0; i < CPL; ++i) {
    const int c = col_of<CPL>(i, lane);
    g[i] = dxh[i] * __ldg(prm.ln1_w[d] + c);
    s1 += g[i];
    s2 += g[i] * n[i];
    dg1[i] += dxh[i] * n[i];
    db1[i] += dxh[i];
  }
  constexpr float invC = 1.0f / C;
  const float c1 = warp_sum(s1) * invC, c2 = warp_sum(s2) * invC;
  const float rstd = st[O.misc];
#pragma unroll
  for (int i = 0; i < CPL; ++i) g[i] = df0[i] + rstd * (g[i] - c1 - n[i] * c2);
  store_row<CPL>(g, dtok + ((size_t)d * B + b) * S * C, lane);
  store_row<CPL>(dg1, rc + R.dg1, lane);
  store_row<CPL>(db1, rc + R.db1, lane);
  // forward vectors the weight-gradient contraction reads
  float v[CPL];
  load_row<CPL>(v, st + O.xh0, lane); store_row<CPL>(v, rc + R.xh0, lane);
  load_row<CPL>(v, st + O.q, lane); store_row<CPL>(v, rc + R.q, lane);
  load_row<CPL>(v, st + O.o, lane); store_row<CPL>(v, rc + R.o, lane);
  load_row<CPL>(v, st + O.chat, lane); store_row<CPL>(v, rc + R.chat, lane);
  load_row<CPL>(v, st + O.e, lane); store_row<CPL>(v, rc + R.e, lane);
  load_row<CPL>(v, st + O.f0, lane); store_row<CPL>(v, rc + R.f0, lane);
  for (int h = 0; h < heads; ++h) {
    load_row<CPL>(v, st + O.u + (size_t)h * C, lane);
    store_row<CPL>(v, rc + R.u + (size_t)h * C, lane);
  }
}

// ------------------------------------------------------------------------------------------------ attention maps
// probs[b][d][h][j] = softmax_j(scale t_h . xh_j) of instance (b, d): the same LN1 / q / t / score steps as the forward
// core, the scores kept in shared memory, then a two-pass softmax per head (one warp per head).  Explain pass only.
__host__ __device__ constexpr size_t fus_attn_smem_floats(int C, int heads, int S) {
  return (size_t)C * (5 + heads) + (size_t)heads * S;
}
template <int CPL>
__global__ void __launch_bounds__(FUS_THREADS, 1)
fusion_attn_kernel(const float* __restrict__ tok, const mfv_fusion_params prm, float* __restrict__ probs, int B, int S,
                   int heads, float scale) {
  constexpr int C = CPL * 32;
  extern __shared__ __align__(16) float fsm[];
  float* g1 = fsm;
  float* b1 = g1 + C;
  float* f0 = b1 + C;
  float* xh0 = f0 + C;
  float* q = xh0 + C;
  float* t = q + C;           // [heads][C]
  float* s = t + heads * C;   // [heads][S]
  const int d = blockIdx.x, b = blockIdx.y;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int hd = C / heads;
  const FusPtrs P = pick(prm, d);
  const float* cls_row = tok + ((size_t)d * B + b) * S * C;
  const float* other = tok + ((size_t)(1 - d) * B + b) * S * C;
  for (int c = tid; c < C; c += FUS_THREADS) {
    g1[c] = P.ln1_w[c];
    b1[c] = P.ln1_b[c];
    f0[c] = cls_row[c];
  }
  __syncthreads();
  if (warp == 0) {
    float v[CPL], n[CPL];
    load_row<CPL>(v, f0, lane);
    float rstd;
    ln_stats<CPL>(v, n, 1e-5f, rstd);
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      xh0[c] = n[i] * g1[c] + b1[c];
    }
  }
  __syncthreads();
  matvec_rows<CPL>(P.wq, xh0, nullptr, q, warp, lane);
  __syncthreads();
  for (int c = tid; c < C; c += FUS_THREADS) {
    for (int h = 0; h < heads; ++h) {
      float acc = 0.f;
      const float* wk = P.wk + (size_t)(h * hd) * C + c;
#pragma unroll 16
      for (int i = 0; i < hd; ++i) acc += __ldg(wk + (size_t)i * C) * q[h * hd + i];
      t[h * C + c] = acc;
    }
  }
  __syncthreads();
  for (int j = warp; j < S; j += FUS_WARPS) {  // key 0: the query's own CLS row; keys 1..S-1: the other branch's patches
    float v[CPL], xh[CPL];
    load_row<CPL>(v, j == 0 ? f0 : other + (size_t)j * C, lane);
    float rstd;
    ln_stats<CPL>(v, xh, 1e-5f, rstd);
#pragma unroll
    for (int i = 0; i < CPL; ++i) {
      const int c = col_of<CPL>(i, lane);
      xh[i] = xh[i] * g1[c] + b1[c];
    }
    for (int h = 0; h < heads; ++h) {
      const float sc = scale * dot_row<CPL>(xh, t + h * C, lane);
      if (lane == 0) s[h * S + j] = sc;
    }
  }
  __syncthreads();
  if (warp < heads) {
    float* sh = s + warp * S;
    float m = -INFINITY;
    for (int j = lane; j < S; j += 32) m = fmaxf(m, sh[j]);
    m = warp_max(m);
    float l = 0.f;
    for (int j = lane; j < S; j += 32) {
      const float e = __expf(sh[j] - m);
      sh[j] = e;
      l += e;
    }
    l = warp_sum(l);
    float* out = probs + (((size_t)b * 2 + d) * heads + warp) * S;
    for (int j = lane; j < S; j += 32) out[j] = __fdiv_rn(sh[j], l);
  }
}

}  // namespace mfv

extern "C" size_t mfv_fusion_saved_floats(int64_t B, int64_t S, int64_t C, int64_t heads) {
  (void)S;
  return (size_t)B * 2 * (mfv::fus_rec_floats((int)C, (int)heads) + mfv::fus2_fwd_floats((int)C, (int)heads) +
                          mfv::fus2_bwt_floats((int)C, (int)heads));
}

namespace mfv {
// Which forward the state inside a `saved` buffer belongs to (host-side bookkeeping: the executor entry points are
// driven from one host thread).  mfv_fusion_bwd reuses the state only when it is called with the same buffer, tokens
// and shape as the most recent batched forward; otherwise it recomputes the forward into the buffer first.
struct Fus2Last { const float* tok; const float* saved; long long B, S, heads; };
static Fus2Last g_fus2_last = {nullptr, nullptr, 0, 0, 0};

struct Fus2Ws {
  float *rec, *fwd, *bwt;
  size_t rstride, fstride, bstride;
  Fus2Ws(float* saved, long long B, int C, int heads) {
    rstride = fus_rec_floats(C, heads);
    fstride = fus2_fwd_floats(C, heads);
    bstride = fus2_bwt_floats(C, heads);
    rec = saved;
    fwd = rec + (size_t)B * 2 * rstride;
    bwt = fwd + (size_t)B * 2 * fstride;
  }
};

static bool batched_fusion_enabled() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("MFVIT_FUSION_BATCHED");
    v = (e && e[0] == '0') ? 0 : 1;
  }
  return v == 1;
}

constexpr size_t FUS2_ROW_SMEM = (size_t)FUS2_RB * 384 * sizeof(float);
constexpr size_t FUS2_COL_SMEM = ((size_t)384 * 32 + (size_t)FUS2_CB * 384) * sizeof(float);

static int fus2_set_attrs() {  // opt-in dynamic shared memory of the batched kernels, once per process
  static bool done = false;
  if (done) return MFV_OK;
  MFV_CUDA_CHECK(cudaFuncSetAttribute(fus2_stream_fwd_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
  MFV_CUDA_CHECK(cudaFuncSetAttribute(fus2_stream_bwd_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 120 * 1024));
  MFV_CUDA_CHECK(cudaFuncSetAttribute(fus2_rowdot_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUS2_ROW_SMEM));
  MFV_CUDA_CHECK(cudaFuncSetAttribute(fus2_coldot_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FUS2_COL_SMEM));
  done = true;
  return MFV_OK;
}
#define RC_ATTRS()                \
  do {                            \
    int _rc = fus2_set_attrs();   \
    if (_rc) return _rc;          \
  } while (0)

static int fus2_forward(const float* tok, const mfv_fusion_params* p, float* out_fused, float* out_x, float* saved,
                        long long B, long long S, int heads, int NC, cudaStream_t st) {
  constexpr int CPL = 12, C = 384;
  const Fus2Ws ws(saved, B, C, heads);
  const Fus2Off O(C, heads);
  const int hd = C / heads;
  const float scale = 1.0f / sqrtf((float)hd);
  const unsigned inst_blocks = (unsigned)((2 * B + 3) / 4);
  const size_t smem_s = ((size_t)C * (3 + heads) + (size_t)FUS_WARPS * heads * C + FUS_WARPS * MAX_HEADS * 2 + MAX_HEADS) *
                        sizeof(float);
  RC_ATTRS();
  const unsigned rz = (unsigned)((B + FUS2_RB - 1) / FUS2_RB), cz = (unsigned)((B + FUS2_CB - 1) / FUS2_CB);
  MFV_CUDA_CHECK(launch_pdl(fus2_ln0_kernel<CPL>, dim3(inst_blocks), dim3(128), 0, st, tok, *p, ws.fwd, ws.fstride, (int)B,
                            (int)S, heads));
  MFV_LAUNCH_CHECK();
  // q = Wq xh0
  MFV_CUDA_CHECK(launch_pdl(fus2_rowdot_kernel<CPL>, dim3(C / 8, 2, rz), dim3(256), FUS2_ROW_SMEM, st, p->wq[0], p->wq[1],
                            (const float*)nullptr, (const float*)nullptr, (const float*)(ws.fwd + O.xh0), ws.fstride,
                            ws.fwd + O.q, ws.fstride, (int)B, 1, hd));
  MFV_LAUNCH_CHECK();
  // t_h = Wk_h^T q_h
  MFV_CUDA_CHECK(launch_pdl(fus2_coldot_kernel<CPL>, dim3(C / 32, 2, cz), dim3(256), FUS2_COL_SMEM, st, p->wk[0],
                            p->wk[1], (const float*)(ws.fwd + O.q), ws.fstride, ws.fwd + O.t, ws.fstride, (int)B, heads, 0));
  MFV_LAUNCH_CHECK();
  MFV_CUDA_CHECK(launch_pdl(fus2_stream_fwd_kernel<CPL>, dim3(2, (unsigned)B), dim3(FUS_THREADS), smem_s, st, tok, *p, ws.fwd,
                            ws.fstride, (int)B, (int)S, heads, scale));
  MFV_LAUNCH_CHECK();
  // o = Wv u_h
  MFV_CUDA_CHECK(launch_pdl(fus2_rowdot_kernel<CPL>, dim3(C / 8, 2, rz), dim3(256), FUS2_ROW_SMEM, st, p->wv[0], p->wv[1],
                            (const float*)nullptr, (const float*)nullptr, (const float*)(ws.fwd + O.u), ws.fstride,
                            ws.fwd + O.o, ws.fstride, (int)B, heads, hd));
  MFV_LAUNCH_CHECK();
  // y = Wp o + bp
  MFV_CUDA_CHECK(launch_pdl(fus2_rowdot_kernel<CPL>, dim3(C / 8, 2, rz), dim3(256), FUS2_ROW_SMEM, st, p->proj_w[0], p->proj_w[1], p->proj_b[0],
                            p->proj_b[1], (const float*)(ws.fwd + O.o), ws.fstride, ws.fwd + O.y, ws.fstride, (int)B, 1, hd));
  MFV_LAUNCH_CHECK();
  MFV_CUDA_CHECK(launch_pdl(fus2_ln2_heads_kernel<CPL>, dim3((unsigned)B), dim3(64), 0, st, *p, ws.fwd, ws.fstride, out_fused,
                            out_x, (int)B, heads, NC));
  MFV_LAUNCH_CHECK();
  g_fus2_last = {tok, saved, B, S, heads};
  return MFV_OK;
}

static int fus2_backward_main(const float* tok, const mfv_fusion_params* p, float* saved, const float* d_fused,
                              const float* d_x, float* dtok, long long B, long long S, int heads, int NC, cudaStream_t st) {
  constexpr int CPL = 12, C = 384;
  const Fus2Ws ws(saved, B, C, heads);
  const Fus2Rec R(C, heads);
  const Fus2Bwt T(C, heads);
  const int hd = C / heads;
  const float scale = 1.0f / sqrtf((float)hd);
  const unsigned inst_blocks = (unsigned)((2 * B + 3) / 4);
  const unsigned bz = (unsigned)((B + FUS2_CB - 1) / FUS2_CB), rz = (unsigned)((B + FUS2_RB - 1) / FUS2_RB);
  const size_t smem_s = ((size_t)C * (3 + 2 * heads) + (size_t)FUS_WARPS * MAX_HEADS * C + 2 * MAX_HEADS) * sizeof(float);
  RC_ATTRS();
  MFV_CUDA_CHECK(launch_pdl(fus2_bwd_heads_kernel<CPL>, dim3(inst_blocks), dim3(128), 0, st, *p, d_fused, d_x,
                            (const float*)ws.fwd, ws.fstride, ws.rec, ws.rstride, ws.bwt, ws.bstride, (int)B, heads, NC));
  MFV_LAUNCH_CHECK();
  // do = Wp^T dy
  MFV_CUDA_CHECK(launch_pdl(fus2_coldot_kernel<CPL>, dim3(C / 32, 2, bz), dim3(256), FUS2_COL_SMEM, st, p->proj_w[0], p->proj_w[1],
                            (const float*)(ws.rec + R.dy), ws.rstride, ws.rec + R.d_o, ws.rstride, (int)B, 1, 0));
  MFV_LAUNCH_CHECK();
  // du_h = Wv_h^T do_h
  MFV_CUDA_CHECK(launch_pdl(fus2_coldot_kernel<CPL>, dim3(C / 32, 2, bz), dim3(256), FUS2_COL_SMEM, st, p->wv[0], p->wv[1],
                            (const float*)(ws.rec + R.d_o), ws.rstride, ws.bwt + T.du, ws.bstride, (int)B, heads, 0));
  MFV_LAUNCH_CHECK();
  MFV_CUDA_CHECK(launch_pdl(fus2_stream_bwd_kernel<CPL>, dim3(2, (unsigned)B), dim3(FUS_THREADS), smem_s, st, tok, *p,
                            (const float*)ws.fwd, ws.fstride, ws.rec, ws.rstride, ws.bwt, ws.bstride, dtok, (int)B, (int)S,
                            heads, scale));
  MFV_LAUNCH_CHECK();
  // dq = Wk dt_h
  MFV_CUDA_CHECK(launch_pdl(fus2_rowdot_kernel<CPL>, dim3(C / 8, 2, rz), dim3(256), FUS2_ROW_SMEM, st, p->wk[0], p->wk[1],
                            (const float*)nullptr, (const float*)nullptr, (const float*)(ws.rec + R.dt), ws.rstride,
                            ws.rec + R.dq, ws.rstride, (int)B, heads, hd));
  MFV_LAUNCH_CHECK();
  // dxh0 += Wq^T dq
  MFV_CUDA_CHECK(launch_pdl(fus2_coldot_kernel<CPL>, dim3(C / 32, 2, bz), dim3(256), FUS2_COL_SMEM, st, p->wq[0], p->wq[1],
                            (const float*)(ws.rec + R.dq), ws.rstride, ws.bwt + T.dxh0, ws.bstride, (int)B, 1, 1));
  MFV_LAUNCH_CHECK();
  MFV_CUDA_CHECK(launch_pdl(fus2_bwd_row0_kernel<CPL>, dim3(inst_blocks), dim3(128), 0, st, *p, (const float*)ws.fwd, ws.fstride,
                            ws.rec, ws.rstride, (const float*)ws.bwt, ws.bstride, dtok, (int)B, (int)S, heads));
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}
}  // namespace mfv

extern "C" int mfv_fusion_fwd(const float* tok, const mfv_fusion_params* p, float* out_fused, float* out_x,
                              float* saved, int64_t B, int64_t S, int64_t C, int64_t heads, int64_t NC, void* stream) {
  using namespace mfv;
  if (!p || B <= 0 || S < 2 || heads <= 0 || heads > MAX_HEADS || NC <= 0 || NC > MAX_NC) return MFV_ERR_SHAPE;
  if (C != 384 || C % heads) return MFV_ERR_SHAPE;
  if (B > 65535) return MFV_ERR_SHAPE;
  if (saved && batched_fusion_enabled())  // batched path: every weight matrix read once per launch, state kept for the backward
    return fus2_forward(tok, p, out_fused, out_x, saved, B, S, (int)heads, (int)NC, reinterpret_cast<cudaStream_t>(stream));
  const size_t smem = fus_smem_floats<12>((int)heads) * sizeof(float);
  static bool attr = false;
  if (!attr) {  // opt in once for the largest head count, so a later call with more heads still launches
    MFV_CUDA_CHECK(cudaFuncSetAttribute(fusion_fwd_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)(fus_smem_floats<12>(MAX_HEADS) * sizeof(float))));
    attr = true;
  }
  const float scale = 1.0f / sqrtf((float)(C / heads));
  fusion_fwd_kernel<12><<<dim3(2, (unsigned)B), FUS_THREADS, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      tok, *p, out_fused, out_x, (int)B, (int)S, (int)heads, (int)NC, scale);
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}

namespace mfv {
static bool g_fusion_wgrad_pending = false;  // a deferred weight-gradient contraction is in flight on the side stream
static SideStream* g_fusion_ss = nullptr;

static int fusion_bwd_impl(const float* tok, const mfv_fusion_params* p, const float* saved, const float* d_fused,
                           const float* d_x, float* dtok, const mfv_fusion_grads* g, int64_t B, int64_t S, int64_t C,
                           int64_t heads, int64_t NC, void* stream, bool defer) {
  if (!p || !g || !saved || B <= 0 || S < 2 || heads <= 0 || heads > MAX_HEADS || NC <= 0 || NC > MAX_NC)
    return MFV_ERR_SHAPE;
  if (C != 384 || C % heads) return MFV_ERR_SHAPE;
  if (B > 65535) return MFV_ERR_SHAPE;
  float* scratch = const_cast<float*>(saved);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  // A deferred contraction still in flight reads its records and accumulates into the gradients: everything this
  // backward writes (records, and the gradients when it is not deferred) must wait for it.
  if (g_fusion_wgrad_pending) MFV_CUDA_CHECK(cudaStreamWaitEvent(st, g_fusion_ss->fusion_done, 0));
  // Without the backbone heads there is no x and so no gradient for their parameters, whatever d_x holds.
  mfv_fusion_grads gg = *g;
  for (int d = 0; d < 2; ++d)
    if (!p->vhead_w[d]) gg.vhead_w[d] = gg.vhead_b[d] = nullptr;
  if (batched_fusion_enabled()) {
    const bool have_fwd = g_fus2_last.tok == tok && g_fus2_last.saved == saved && g_fus2_last.B == B &&
                          g_fus2_last.S == S && g_fus2_last.heads == heads;
    if (!have_fwd) {  // the forward ran without this buffer (or something ran in between): rebuild its state here
      float* tmp_out = scratch;  // logits are not needed: park them in the record area, which the backward overwrites
      int rc = fus2_forward(tok, p, tmp_out, tmp_out + B * NC, scratch, B, S, (int)heads, (int)NC, st);
      if (rc) return rc;
    }
    g_fus2_last.tok = nullptr;  // consumed: a later backward on the same buffer must not trust it blindly
    int rc = fus2_backward_main(tok, p, scratch, d_fused, d_x, dtok, B, S, (int)heads, (int)NC, st);
    if (rc) return rc;
  } else {
    auto smem_for = [&](int h) {
      return (fus_smem_floats<12>(h) + (size_t)C * (6 + 2 * h) + MAX_HEADS + 2 * MAX_NC) * sizeof(float);
    };
    const size_t smem = smem_for((int)heads);
    static bool attr = false;
    if (!attr) {  // opt in once for the largest head count, so a later call with more heads still launches
      MFV_CUDA_CHECK(cudaFuncSetAttribute(fusion_bwd_kernel<12>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)smem_for(MAX_HEADS)));
      attr = true;
    }
    const float scale = 1.0f / sqrtf((float)(C / heads));
    fusion_bwd_kernel<12><<<dim3(2, (unsigned)B), FUS_THREADS, smem, st>>>(tok, *p, d_fused, d_x, dtok, scratch, (int)B,
                                                                            (int)S, (int)heads, (int)NC, scale);
    MFV_LAUNCH_CHECK();
  }
  // The contraction of the per-sample records into the parameter gradients feeds only the optimizer: deferred, it runs
  // on the side stream beside the encoder backward that consumes dtok.
  SideStream* ss = defer ? side_stream() : nullptr;
  cudaStream_t sw = st;
  if (ss) {
    MFV_CUDA_CHECK(cudaEventRecord(ss->fusion_fork, st));
    MFV_CUDA_CHECK(cudaStreamWaitEvent(ss->stream, ss->fusion_fork, 0));
    sw = ss->stream;
  }
  fusion_wgrad_kernel<12><<<dim3((unsigned)(C / 4), 5, 2), FUS_THREADS, 0, sw>>>(scratch, d_fused, d_x, gg, (int)B,
                                                                                 (int)heads, (int)NC);
  MFV_LAUNCH_CHECK();
  if (ss) {
    MFV_CUDA_CHECK(cudaEventRecord(ss->fusion_done, sw));
    g_fusion_wgrad_pending = true;
    g_fusion_ss = ss;
  }
  return MFV_OK;
}
}  // namespace mfv

extern "C" int mfv_fusion_bwd(const float* tok, const mfv_fusion_params* p, const float* saved, const float* d_fused,
                              const float* d_x, float* dtok, const mfv_fusion_grads* g, int64_t B, int64_t S, int64_t C,
                              int64_t heads, int64_t NC, void* stream) {
  return mfv::fusion_bwd_impl(tok, p, saved, d_fused, d_x, dtok, g, B, S, C, heads, NC, stream, false);
}

extern "C" int mfv_fusion_bwd_deferred(const float* tok, const mfv_fusion_params* p, const float* saved,
                                       const float* d_fused, const float* d_x, float* dtok, const mfv_fusion_grads* g,
                                       int64_t B, int64_t S, int64_t C, int64_t heads, int64_t NC, void* stream) {
  return mfv::fusion_bwd_impl(tok, p, saved, d_fused, d_x, dtok, g, B, S, C, heads, NC, stream, true);
}

extern "C" int mfv_fusion_bwd_join(void* stream) {
  using namespace mfv;
  if (!g_fusion_wgrad_pending) return MFV_OK;
  MFV_CUDA_CHECK(cudaStreamWaitEvent(reinterpret_cast<cudaStream_t>(stream), g_fusion_ss->fusion_done, 0));
  g_fusion_wgrad_pending = false;
  return MFV_OK;
}

extern "C" int mfv_fusion_attn(const float* tok, const mfv_fusion_params* p, float* probs, int64_t B, int64_t S,
                               int64_t C, int64_t heads, void* stream) {
  using namespace mfv;
  if (!p || !tok || !probs || B <= 0 || B > 65535 || S < 2 || S > 2048 || heads <= 0 || heads > MAX_HEADS)
    return MFV_ERR_SHAPE;
  if (C != 384 || C % heads) return MFV_ERR_SHAPE;
  const size_t smem = fus_attn_smem_floats((int)C, (int)heads, (int)S) * sizeof(float);  // < 48 KB for S <= 2048
  const float scale = 1.0f / sqrtf((float)(C / heads));
  fusion_attn_kernel<12><<<dim3(2, (unsigned)B), FUS_THREADS, smem, reinterpret_cast<cudaStream_t>(stream)>>>(
      tok, *p, probs, (int)B, (int)S, (int)heads, scale);
  MFV_LAUNCH_CHECK();
  return MFV_OK;
}
