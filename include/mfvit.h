/* mfvit.h - C ABI of libmfvit.so: hand-written sm_100a kernels for the MF-ViT CA training hot path.
 *
 * The reference (endiqq/Multi-Feature-ViT) has no FFI of its own: its hot path is PyTorch library calls made from
 * Python nn.Modules.  This header is the boundary a maintainer binds *below* that module surface; each entry point
 * names the reference call-site(s) it replaces (paths relative to the reference tree; MAIN_CA / MAIN_PRE / FUS / MOD /
 * BLD are the aliases defined in SURVEY.md).  See INTEGRATION.md for the ctypes binding.
 *
 * Conventions
 *   - every function returns 0 on success, a negative MFV_ERR_* for rejected arguments (shape / alignment / arch), or a
 *     positive cudaError_t.  There is no CPU fallback and no alternate backend: on a non-sm_100 device mfv_init fails.
 *   - all pointers are device pointers owned by the caller (PyTorch tensors); the library allocates nothing
 *     persistent, never synchronises the stream and is safe under CUDA-graph capture.
 *   - `stream` is a cudaStream_t passed as void*.
 *   - bf16 = __nv_bfloat16 storage, f32 = float.  "G" is the group count: the two MF-ViT branches (CXR, enhanced) are
 *     processed by one launch with per-group weights (G = 2), a single ViT uses G = 1.
 */
#ifndef MFVIT_H_
#define MFVIT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MFV_ABI_VERSION 1

/* ---- runtime ------------------------------------------------------------------------------------------------- */
int mfv_abi_version(void);
/* Binds the library to `device`; checks compute capability 10.x, resolves cuTensorMapEncodeTiled.  One device per
 * process: a second call with a different device returns MFV_ERR_ARG (side stream, events and opt-in shared-memory
 * attributes are process-wide state).                                                                             */
int mfv_init(int device);
const char* mfv_strerror(int code);
/* "file:line: expression" of the last CUDA runtime failure returned to this thread ("" if none); debugging aid. */
const char* mfv_last_error_where(void);
/* Runtime switches (A/B measurements, tests).  Each key starts from its environment variable, read on first use; the
 * value in brackets is the default when that variable is unset.  Returns MFV_ERR_ARG for an unknown key.
 *   "pdl"              programmatic dependent launch                          [1]  MFVIT_PDL=0 switches it off
 *   "side_stream"      weight gradients on a second stream                    [1]  MFVIT_SIDE_STREAM=0
 *   "legacy_attention" mma.sync attention kernels instead of tcgen05          [0]  MFVIT_ATTN=legacy
 *   "rows96"           192-row pair tiles for the forward N = 384 GEMMs       [0]  MFVIT_ROWS96=<digit>
 *   "fuse_ln"          LayerNorm inside the proj / fc2 epilogues              [1]  MFVIT_FUSE_LN=0
 *   "dx32"             fp32 residual-gradient stream in the backward          [0]  MFVIT_DX32=1
 *   "patch_tma"        im2col-free patch-embedding GEMM (TMA from the images) [1]  MFVIT_PATCH_TMA=0
 *   "reserve_sms"      SMs left free for concurrent collectives               [0]  MFVIT_RESERVE_SMS=<n>
 *   "gemm_mc"          B-operand multicast between CTA pairs                  [0]  MFVIT_GEMM_MC=1
 *   "streamk"          stream-K bit mask of GEMM families (allocates; not
 *                      inside a stream capture)                               [0]  MFVIT_STREAMK=<mask>
 *   "streamk_min_kb"   fewest k-blocks per stream-K range                     [12] MFVIT_STREAMK_MINKB=<n>   */
int mfv_set_option(const char* key, int value);
int mfv_num_sms(void);
/* Number of kernels this library has launched so far in the process (bench.py reports the per-step delta). */
uint64_t mfv_launch_count(void);
/* Optional device-side timing of mfv_vit_forward/backward per kernel class (CUDA events on the launching stream).
 * mfv_prof_read synchronises the device, ACCUMULATES elapsed ms / launch counts per label into the arrays and resets. */
int mfv_prof_enable(int on);
int mfv_prof_num_labels(void);
const char* mfv_prof_label_name(int label);
int mfv_prof_read(float* ms_per_label, int* count_per_label, int nlabels);

/* ---- GEMM (tcgen05 / TMEM / TMA) ----------------------------------------------------------------------------------
 * C[g][m][n] = epilogue( sum_k A[g][m][k] * B[g][n][k] ), bf16 operands, fp32 accumulation in TMEM.
 * Replaces: timm Block qkv/proj/fc1/fc2 nn.Linear forward + autograd backward (absent vits.py; same math restated at
 * MOD:45-63 and MOD:23-34), the cuBLASLt calls behind them, and the bias/GELU/residual ATen kernels (SURVEY K3,K5,K6).
 * Operand (m,k) of A lives at A + g*a_gstride + (a_mn_major ? k*lda + m : m*lda + k); likewise B with (n,k).        */
enum {
  MFV_EPI_BF16 = 0,       /* C(bf16)  = acc + bias                                           (qkv, dgrad)        */
  MFV_EPI_GELU = 1,       /* C(bf16)  = u = acc + bias ; C2(bf16) = gelu_erf(u)             (fc1)                */
  MFV_EPI_RESID_F32 = 2,  /* C(f32)   = acc + bias + aux(f32)                               (proj, fc2)          */
  MFV_EPI_DGELU = 3,      /* C(bf16)  = acc * gelu_erf'(aux(bf16) = u)                      (fc2 dgrad)          */
  MFV_EPI_F32 = 4,        /* C(f32)   = acc + bias                                                               */
  MFV_EPI_ATOMIC_F32 = 5, /* C(f32)  += acc  (red.global.add; split-K weight gradients)                          */
  MFV_EPI_RESID_LN = 6    /* C(f32) = x = acc + bias + aux(f32) ; C2 = LayerNorm(x) (16-bit or f32), C3 = optional bf16
                           * copy, ln_mean / ln_rstd = the row statistics.  N == 384 only: the 256 x 384 pair tile owns whole
                           * rows, so proj / fc2 also emit the operand of the NEXT Linear (SURVEY K2: LayerNorm fused into
                           * the producing epilogue; the standalone LayerNorm launch and its fp32 re-read disappear)      */
};
typedef struct {
  const void* A;
  const void* B;
  void* C;
  void* C2;         /* MFV_EPI_GELU: gelu(u) (required).  MFV_EPI_DGELU: optional bf16 gelu(aux) recomputed for the fc2 wgrad */
  void* C3;         /* MFV_EPI_GELU only: optional bf16 copy of C2 (kept for the backward GEMMs when C2 is fp16) */
  const void* bias; /* f32 [G][N] or NULL */
  const void* aux;
  int64_t M, N, K, G;
  int64_t lda, ldb, ldc;                 /* elements */
  int64_t a_gstride, b_gstride, c_gstride; /* elements between groups */
  int64_t aux_ld, aux_gstride, bias_gstride;
  int32_t a_mn_major, b_mn_major; /* 0: reduction dim contiguous (K-major), 1: M/N dim contiguous */
  int32_t epilogue;
  int32_t splits;  /* split-K factor (only with MFV_EPI_ATOMIC_F32) */
  int32_t block_n; /* 0 = auto, else 64/128/256 */
  int32_t dtype_flags; /* bit0: A is fp16, bit1: B is fp16, bit2: 16-bit outputs are fp16 (default bf16 everywhere).
                          Bits 8..20 are measurement aids (tests/gpu_*probe*.py, gpu_epi_prof.py) and must be 0 in a real
                          call: 8 accumulators released unread, 9 bulk stores skipped, 10..11 stream-K probes, 12..15 operand
                          ring depth, 16..19 UMMA / operand-load probes, 20 per-warp phase clocks into row_sum */
  int32_t cta_group;   /* 0 = auto, 1 = 128-row tiles, 2 = CTA pairs (tcgen05 cta_group::2, 256-row tiles) */
  int32_t rows_per_cta; /* 384-wide pair tiles with K-major A only: 0 = default (128), or 96 = 192-row pair tiles
                         * (more, smaller tiles: fills the SMs better for M ~ 6-12 k; opt-in, see gemm.cu)           */
  /* MFV_EPI_ATOMIC_F32 with 384-wide pair tiles (N == 384) only: f32 [G][M] (group stride bias_gstride), += the row
   * sums of A over the reduction dimension, i.e. the bias gradient of a weight-gradient GEMM (A = dY read MN-major),
   * computed by one extra N=16 UMMA per k-step against a tile of ones.  NULL = off.                                */
  float* row_sum;
  /* MFV_EPI_RESID_LN only: gamma / beta f32 [G][N] (group stride bias_gstride); mean / rstd f32 [G][M] outputs (group
   * stride M) saved for the backward; eps; ln_out_f32 = 1: C2 is f32 [G][M][N] (the final norm writes the tokens). */
  const float* ln_gamma;
  const float* ln_beta;
  float* ln_mean;
  float* ln_rstd;
  float ln_eps;
  int32_t ln_out_f32;
} mfv_gemm_args;
int mfv_gemm(const mfv_gemm_args* args, void* stream);
/* Two split-K weight-gradient GEMMs (MFV_EPI_ATOMIC_F32, N % 384 == 0, M > 128; same K, G, splits, majorness, formats,
 * bias_gstride) as ONE grid of 256 x 384 pair tiles: the four weight gradients of a transformer block (autograd of the
 * four nn.Linear, absent timm Block) take two launches instead of four.                                              */
int mfv_gemm_wgrad_pair(const mfv_gemm_args* a, const mfv_gemm_args* b, void* stream);

/* ---- LayerNorm ------------------------------------------------------------------------------------------------------
 * Replaces nn.LayerNorm(384, eps=1e-6) x25 per branch in the absent timm ViT, PreNorm's LayerNorm (MOD:15-21).
 * x f32 [G][rows][C] -> y16 (16-bit GEMM operand: bf16, or fp16 when y16_is_f16; optional extra bf16 copy for the
 * backward GEMMs) and/or y32 f32; mean/rstd f32 [G][rows] saved for backward.
 * gamma/beta f32 [G][C] (group stride gb_gstride elements).                                                          */
int mfv_layernorm_fwd(const float* x, const float* gamma, const float* beta, void* y16, int y16_is_f16,
                      void* y_bf16_copy, float* y_f32, float* mean, float* rstd, int64_t G, int64_t rows, int64_t C,
                      int64_t gb_gstride, float eps, void* stream);
/* dx = dres (optional residual-path gradient: f32 `dres` or bf16 `dres_bf16`, not both) + LN'(dy); dy is bf16
 * (dy_bf16) or f32 (dy_f32).  Writes dx as f32 (dx_f32, optional) and / or as the bf16 copy that feeds the next
 * dgrad / wgrad GEMMs (dx_bf16, optional).
 * dgamma/dbeta f32 [G][C] are ACCUMULATED (+=) with red.global.add; dx_colsum (optional, f32 [G][C], +=) receives the
 * column sums of dx, i.e. the bias gradient of the Linear whose output was added into x (proj / fc2), for free.                                                   */
int mfv_layernorm_bwd(const void* dy_bf16, const float* dy_f32, const float* dres, const void* dres_bf16, const float* x, const float* mean,
                      const float* rstd, const float* gamma, float* dx_f32, void* dx_bf16, float* dgamma, float* dbeta,
                      float* dx_colsum, int64_t G, int64_t rows, int64_t C, int64_t gb_gstride, void* stream);

/* ---- fused softmax self-attention -----------------------------------------------------------------------------------
 * Replaces timm Attention: q@k^T*scale -> softmax -> @v and the transpose copies around it (SURVEY K4; same math
 * MOD:52-64).  qkv bf16 [NB][S][3][H][D] (the qkv GEMM's natural output), o bf16 [NB][S][H][D], lse f32 [NB][H][S].
 * o may be written as fp16 (o_is_f16; proj GEMM operand of the fp16-forward mode) with an optional bf16 copy.
 * D in {32, 64}; any S >= 1 (197 @224^2, 577 @384^2).                                                                 */
int mfv_attn_fwd(const void* qkv, int qkv_is_f16, void* o, int o_is_f16, void* o_bf16_copy, float* lse, int64_t NB,
                 int64_t S, int64_t H, int64_t D, float scale, void* stream);
/* dqkv bf16 [NB][S][3][H][D]; delta f32 [NB][H][S] is scratch (rowsum(dO*O)); o and d_o are bf16.  When the forward
 * kept qkv in fp16 (qkv_is_f16) the tiles are converted to bf16 in shared memory: the backward always runs in bf16.                                        */
int mfv_attn_bwd(const void* qkv, int qkv_is_f16, const void* o, const void* d_o, const float* lse, float* delta,
                 void* dqkv, int64_t NB, int64_t S, int64_t H, int64_t D, float scale, void* stream);
/* Same, with a workspace: f32 [NB][S][H*D] (mfv_attn_bwd_workspace_bytes).  With it, sequences longer than 224 tokens
 * (D == 64) also run on tcgen05: one CTA per (image, head, 128-key block), dK / dV accumulated in TMEM over the query
 * tiles, the key blocks' shares of dQ summed in the workspace by fp32 TMA reduce-adds and converted at the end.      */
size_t mfv_attn_bwd_workspace_bytes(int64_t NB, int64_t S, int64_t H, int64_t D);
int mfv_attn_bwd_ws(const void* qkv, int qkv_is_f16, const void* o, const void* d_o, const float* lse, float* delta,
                    void* dqkv, float* workspace, int64_t NB, int64_t S, int64_t H, int64_t D, float scale,
                    void* stream);

/* ---- patch embedding -----------------------------------------------------------------------------------------------
 * Replaces timm PatchEmbed Conv2d(3,C,k=16,s=16)+flatten+transpose, cls-token concat and pos-embed add
 * (commented restatement FUS:197-221, crossvit.py:130-146; SURVEY K1).
 * mfv_patchify: img f32 [G][B][3][HW][HW] -> patches bf16 [G][B*np][768] (k = c*256 + i*16 + j), np = (HW/16)^2.
 * The GEMM itself is mfv_gemm; mfv_embed_finish writes tokens x f32 [G][B][np+1][C]:
 *   row 0 = cls + pos[0], row 1+p = acc[p] + bias + pos[1+p].                                                         */
int mfv_patchify(const float* img, void* patches, int patches_is_f16, void* patches_bf16_copy, int64_t GB, int64_t HW,
                 void* stream);
/* The same three steps as ONE im2col-free GEMM (default forward path, C == 384): the A operand is fetched by TMA from the
 * NCHW fp32 images through a 5-D tensor map (j, i, patch column, patch row, channel x image) as dense [patch][64 k] fp32
 * tiles, rounded to the 16-bit operand format in shared memory by the epilogue warps (no patch matrix in HBM), and
 * multiplied on tcgen05 with the 16-bit weight shadow w16 [G][C][768] (fp16 when w_is_f16, else bf16); the epilogue adds
 * bias + position embedding and writes x f32 [G][B][np+1][C] including the class-token row.  img0 / img1: the images of
 * group 0 / 1 (img1 unused for G == 1); bias / cls / pos inside the groups' parameter blocks (p_gstride elements apart). */
/* Test aid: the raw shared-memory image (8192 floats) of ONE 5-D TMA box of mfv_patch_embed_tma's image map. */
int mfv_debug_patch_tma_probe(const float* img, float* out8192, int64_t B, int64_t HW, int64_t kb, int64_t ph0, int64_t cb,
                              void* stream);
int mfv_patch_embed_tma(const float* img0, const float* img1, const void* w16, int w_is_f16, const float* bias,
                        const float* cls, const float* pos, float* x, int64_t G, int64_t B, int64_t HW, int64_t C,
                        int64_t p_gstride, void* stream);
int mfv_embed_finish(const float* acc, const float* bias, const float* cls, const float* pos, float* x, int64_t G,
                     int64_t B, int64_t np, int64_t C, int64_t p_gstride, void* stream);
/* backward of the above: dacc bf16 [G][B*np][C] (for the conv weight gradient GEMM), dbias/dcls accumulated.
 * (pos_embed is a fixed sin-cos table, requires_grad=False.)                                                          */
int mfv_embed_finish_bwd(const float* dx, void* dacc_bf16, float* dbias, float* dcls, int64_t G, int64_t B, int64_t np,
                         int64_t C, int64_t p_gstride, void* stream);

/* ---- column sums (bias gradients) ----------------------------------------------------------------------------------
 * out f32 [G][C] += sum over rows of x bf16 [G][rows][C]                                                              */
int mfv_colsum_bf16(const void* x, float* out, int64_t G, int64_t rows, int64_t C, int64_t out_gstride, void* stream);

/* ---- CLS-query cross-attention fusion (single kernel forward, single kernel backward) ---------------------------------
 * Replaces Fus_CrossViT.forward after the backbones (FUS:137-157), MultiScaleTransformerEncoder.forward (FUS:35-65),
 * PreNorm (MOD:15-21), CrossAttention (MOD:123-137), both mlp heads and both backbone heads (SURVEY K7, K8).
 * tok f32 [2][B][S][C] final-normed tokens of (cxr, enh).  Parameter block layout: see mfv_fusion_params.           */
typedef struct {
  /* index d = 0: the CXR-CLS query (cross_attn_layers.0.0 + LayerNorm .3, mlp_head_cxr, vit_cxr.head)
   * index d = 1: the ENH-CLS query (cross_attn_layers.0.2 + LayerNorm .1, mlp_head_enh, vit_enh.head)              */
  const float* ln1_w[2]; const float* ln1_b[2];     /* PreNorm LayerNorm, eps 1e-5 */
  const float* wq[2]; const float* wk[2]; const float* wv[2]; /* [C][C], no bias */
  const float* proj_w[2]; const float* proj_b[2];
  const float* ln2_w[2]; const float* ln2_b[2];     /* post LayerNorm, eps 1e-6 */
  const float* head_w[2]; const float* head_b[2];   /* mlp_head_{cxr,enh}: [NC][C] */
  const float* vhead_w[2]; const float* vhead_b[2]; /* backbone heads: [NC][C] (may be NULL -> x_* not computed) */
} mfv_fusion_params;
typedef struct {
  float* ln1_w[2]; float* ln1_b[2];
  float* wq[2]; float* wk[2]; float* wv[2];
  float* proj_w[2]; float* proj_b[2];
  float* ln2_w[2]; float* ln2_b[2];
  float* head_w[2]; float* head_b[2];
  float* vhead_w[2]; float* vhead_b[2];
} mfv_fusion_grads;
/* out_fused / out_x f32: fused [B][NC], x [2][B][NC]; `saved` f32 scratch of mfv_fusion_saved_floats(B,S,C,heads). */
size_t mfv_fusion_saved_floats(int64_t B, int64_t S, int64_t C, int64_t heads);
int mfv_fusion_fwd(const float* tok, const mfv_fusion_params* p, float* out_fused, float* out_x, float* saved,
                   int64_t B, int64_t S, int64_t C, int64_t heads, int64_t NC, void* stream);
/* dtok f32 [2][B][S][C] is OVERWRITTEN (all rows); parameter gradients are accumulated (+=).                          */
int mfv_fusion_bwd(const float* tok, const mfv_fusion_params* p, const float* saved, const float* d_fused,
                   const float* d_x, float* dtok, const mfv_fusion_grads* g, int64_t B, int64_t S, int64_t C,
                   int64_t heads, int64_t NC, void* stream);
/* Same, but only dtok is complete in `stream` order on return: the contraction of the per-sample records into the
 * parameter gradients (it feeds the optimizer only) runs on the library's side stream, beside the encoder backward.
 * `saved`, d_fused, d_x and the gradient buffers must stay untouched until mfv_fusion_bwd_join(stream), which orders
 * `stream` after that contraction (a no-op when nothing is pending or the side stream is disabled).                  */
int mfv_fusion_bwd_deferred(const float* tok, const mfv_fusion_params* p, const float* saved, const float* d_fused,
                            const float* d_x, float* dtok, const mfv_fusion_grads* g, int64_t B, int64_t S, int64_t C,
                            int64_t heads, int64_t NC, void* stream);
int mfv_fusion_bwd_join(void* stream);

/* ---- small-N linear (classification heads, N <= 32) ------------------------------------------------------------------
 * Replaces `head = nn.Linear(384, 3)` (MAIN_CA:309-310, MAIN_LPFT:288) applied to the CLS row.
 * x f32 rows with stride ldx; y f32 [rows][N].                                                                        */
int mfv_linear_small_fwd(const float* x, int64_t ldx, const float* w, const float* b, float* y, int64_t rows,
                         int64_t C, int64_t N, void* stream);
int mfv_linear_small_bwd(const float* x, int64_t ldx, const float* w, const float* dy, float* dx, int64_t lddx,
                         float* dw, float* db, int64_t rows, int64_t C, int64_t N, void* stream);

/* ---- softmax cross-entropy on small class counts -------------------------------------------------------------------
 * Replaces nn.CrossEntropyLoss on `output_fus+output_cxr+output_enh` (MAIN_CA:868-873).  logits = a + b + c (b, c
 * optional), mean reduction.  loss f32 [1]; dlogits f32 [rows][NC] = (softmax - onehot)/rows.                         */
int mfv_ce_small(const float* a, const float* b, const float* c, const int64_t* target, float* loss, float* dlogits,
                 int64_t rows, int64_t NC, void* stream);

/* ---- MoCo: momentum (EMA) update -----------------------------------------------------------------------------------
 * Replaces MoCo._momentum_update_key_encoder (BLD:83-89): k = k*m + q*(1.-m), bit-exact with the 3-op eager sequence
 * (two roundings of the products, one of the sum: no FMA contraction).  m and one_minus_m are the separately
 * rounded fp32 values of the Python doubles m and (1.-m).  Chunk table: n_chunks x {k ptr, q ptr, count}.             */
typedef struct {
  float* k;
  const float* q;
  int64_t n;
} mfv_ema_chunk;
int mfv_ema_update(const mfv_ema_chunk* chunks_dev, int64_t n_chunks, int64_t max_chunk_elems, float m,
                   float one_minus_m, void* stream);

/* ---- MoCo: InfoNCE logits (v2 loss) ---------------------------------------------------------------------------------
 * Replaces BLD:165,175 (F.normalize), BLD:183-191 (l_pos, l_neg = q @ queue, cat, /T) and MAIN_PRE:535 (CE, label 0).
 * q_raw, k_raw f32 [N][D] un-normalised; queue f32 [D][K] (column j = key j).  Outputs: qn, kn f32 [N][D] normalised,
 * logits f32 [N][1+K], lse f32 [N*(1+2*K/64)] (first N: log-sum-exp of each logits row, for the fused CE; the rest is
 * per-tile scratch), loss f32 [1] (mean CE).                                                                          */
int mfv_infonce_fwd(const float* q_raw, const float* k_raw, const float* queue, float* qn, float* kn, float* logits,
                    float* lse, float* loss, int64_t N, int64_t D, int64_t K, float T, void* stream);
/* d(q_raw) f32 [N][D] from the mean-CE loss (scaled by gscale), through /T, the logits and F.normalize.
 * dlogits_ext (optional, f32 [N][1+K]) lets autograd pass an arbitrary upstream gradient instead of the fused CE.
 * queue_override (optional, f32 [D][ov_n]): the pre-enqueue contents of queue columns [ov_start, ov_start+ov_n), so the
 * backward sees the queue the forward saw without the reference's 64 MiB queue.clone() (BLD:185).                     */
int mfv_infonce_bwd(const float* q_raw, const float* qn, const float* kn, const float* queue, const float* logits,
                    const float* lse, const float* dlogits_ext, const float* queue_override, int64_t ov_start,
                    int64_t ov_n, float gscale, float* dq_raw, int64_t N, int64_t D, int64_t K, float T, void* stream);
/* Tensor-core InfoNCE (same reference lines): l_neg = (qn / T) @ queue on the tcgen05 GEMM with fp16 operands (qn / T
 * and an fp16 shadow of the queue; entries in [-1, 1], logits within ~5e-4 of the fp32 kernels at T = 0.2) and fp32
 * accumulation, written straight into `logits`.  Buffers (caller-owned):
 *   queue16 fp16 [D][K]: shadow of queue, kept current with mfv_queue16_update (whole queue once, then the enqueued columns)
 *   logits  f32 [N][ld], ld = K + 8 (16-byte aligned l_neg block): column 7 = l_pos/T, columns 8.. = l_neg/T; the
 *           tensor given to the loss is the strided view logits[:, 7:]
 *   qs16    fp16 [N][D] scratch;  lse f32 [N * (1 + 2 * K / 1024)] (lse first, then per-chunk partials);  loss f32 [1]
 * Backward: dl16 fp16 [N][K] scratch (scaled gradient operand of the split-K GEMM dqn = dlogits @ queue^T), scal f32 [4]
 * scratch; queue_override / ov_start / ov_n as in mfv_infonce_bwd (pre-enqueue columns, exact fp32 contribution).
 * D == 256, K % 1024 == 0.                                                                                               */
int mfv_infonce_tc_fwd(const float* q_raw, const float* k_raw, const void* queue16, float* qn, float* kn, void* qs16,
                       float* logits, int64_t ld_logits, float* lse, float* loss, int64_t N, int64_t D, int64_t K,
                       float T, void* stream);
int mfv_infonce_tc_bwd(const float* q_raw, const float* qn, const float* kn, const void* queue16, const float* logits,
                       int64_t ld_logits, const float* lse, const float* dlogits_ext, const float* queue_override,
                       int64_t ov_start, int64_t ov_n, float gscale, void* dl16, float* scal, float* dq_raw, int64_t N,
                       int64_t D, int64_t K, float T, void* stream);
/* queue16[:, col0:col0+ncols] = fp16(queue[:, col0:col0+ncols])                                                         */
int mfv_queue16_update(const float* queue, void* queue16, int64_t D, int64_t K, int64_t col0, int64_t ncols,
                       void* stream);
/* queue[:, ptr:ptr+n] = keys^T  (BLD:102); keys f32 [n][D] (already all-gathered, rank-major).                        */
int mfv_enqueue_keys(const float* keys, float* queue, int64_t n, int64_t D, int64_t K, int64_t ptr, void* stream);

/* ---- whole-encoder orchestration (native runtime) ------------------------------------------------------------------
 * Enqueues every kernel of the ViT-S/16 encoder forward / backward for G branches in one call (no per-kernel Python
 * round trips; capture-safe).  Replaces VisionTransformer.forward_features of the absent vits.py (timm): patch embed ->
 * +cls -> +pos -> depth x Block -> norm, and its autograd backward.  All buffers are caller-owned.
 * Parameter addressing: tensor t of group g lives at master + g*P + off_t (f32), shadow + g*P + off_t (bf16 copy) and
 * shadow16 + g*P + off_t (fp16 copy).                                                                                   */
typedef struct {
  int64_t G, B, S, C, H, depth, hidden, img, np;
  int64_t P;
  const float* master;
  const void* shadow;   /* bf16 [G][P] */
  const void* shadow16; /* fp16 [G][P] (fwd_f16 mode) */
  float* grad; /* f32 [G][P], accumulated into (caller zeroes) */
  int64_t off_cls, off_pos, off_pe_w, off_pe_b, off_norm_w, off_norm_b, off_block0, block_stride;
  int64_t r_ln1_w, r_ln1_b, r_qkv_w, r_qkv_b, r_proj_w, r_proj_b, r_ln2_w, r_ln2_b, r_fc1_w, r_fc1_b, r_fc2_w, r_fc2_b;
  const float* images[2]; /* per group: f32 [B][3][img][img] */
  void* patches;          /* bf16 [G][B*np][768] */
  float* acc;             /* f32  [G][B*np][C] */
  float* x;               /* f32  [nslot_x][G][M][C]  residual stream: slot 0 = embed out, 2l+1 = mid of block l, 2l+2 = out */
  void* xn;               /* bf16 [nslot][G][M][C]    LayerNorm outputs: slot 2l = norm1, 2l+1 = norm2 */
  float* stats;           /* f32  [nslot_x][2][G][M]  mean, rstd of the LN applied to x slot i */
  void* qkv;              /* bf16 [nblk][G][M][3C] */
  void* attn_o;           /* bf16 [nblk][G][M][C] */
  float* lse;             /* f32  [nblk][G*B][H][S] */
  void* u;                /* bf16 [nblk][G][M][hidden] pre-GELU */
  void* gact;             /* bf16 [nblk][G][M][hidden] GELU out */
  float* tokens;          /* f32  [G][M][C] final-normed tokens (features3D) */
  int32_t save_for_backward; /* 1: one slot per block (training); 0: slots are reused (inference / momentum encoder) */
  int32_t stop_grad_conv1;
  /* fwd_f16 = 1: forward GEMM operands (patches, xn, attn_o, gact, weights) are IEEE fp16 (8x finer than bf16; keeps the
   * logits within 2e-3 of the fp32 reference); the backward stays bf16 and reads the *_bf copies written alongside
   * (only when save_for_backward).  fwd_f16 = 0: everything bf16, the *_bf pointers are unused.                        */
  int32_t fwd_f16;
  int32_t gact_bf_per_block; /* 1: gact_bf holds one slot per block, written by the fc1 epilogue of the forward; 0: one slot,
                                recomputed per block by the fc2-dgrad epilogue of the backward (was a reserved field) */
  void* patches_bf; void* xn_bf; void* attn_o_bf; /* same slot layout as patches / xn / attn_o */
  void* gact_bf; /* bf16 gelu(u) for the fc2 weight gradient: [G][M][hidden] x (gact_bf_per_block ? depth : 1) slots */
  /* backward only */
  const float* dtokens;   /* f32 [G][M][C] */
  float* dx[2];           /* f32 [G][M][C] ping-pong */
  void* dx16[2];          /* bf16 copies */
  void* dhid;             /* bf16 [G][M][hidden] */
  void* dxn;              /* bf16 [G][M][C] */
  void* d_o;              /* bf16 [G][M][C] */
  void* dqkv;             /* bf16 [G][M][3C] */
  float* delta;           /* f32 [G*B][H][S] */
  void* dacc;             /* bf16 [G][B*np][C] */
  float* attn_ws;         /* f32 [G*B][S][C] (or NULL): fp32 dQ accumulator of the long-sequence attention backward */
} mfv_vit_plan;
int mfv_vit_forward(const mfv_vit_plan* plan, void* stream);
int mfv_vit_backward(const mfv_vit_plan* plan, void* stream);
/* The backward in segments: blocks block_hi .. block_lo (inclusive, descending).  MFV_BWD_HEAD adds the final-norm
 * backward in front (first segment), MFV_BWD_TAIL the embedding part behind (last segment).  When a call returns, the
 * gradients of its blocks are complete in stream order, so a data-parallel caller can start the all-reduce of that
 * slice of the flat gradient buffer while the next segment runs.  (The fc2 bias gradient of block l-1 is produced by
 * block l's LayerNorm backward, i.e. earlier than its own segment - never later.)                                    */
#define MFV_BWD_HEAD 1
#define MFV_BWD_TAIL 2
int mfv_vit_backward_range(const mfv_vit_plan* plan, void* stream, int block_hi, int block_lo, int flags);

/* ---- elementwise / optimiser ------------------------------------------------------------------------------------------
 * f32 master -> 16-bit shadow weights for the GEMM operands: bf16 (backward) and/or fp16 (forward); either may be NULL. */
int mfv_cast_shadow(const float* src, void* dst_bf16, void* dst_f16, int64_t n, void* stream);
/* bf16 -> f32: the data-parallel trainer all-reduces the weight gradients as bf16 (half the NVLink volume of the DDP
 * fp32 all-reduce, MAIN_PRE:312) and widens the averaged result back into the fp32 buffer the optimizer reads.        */
int mfv_cast_bf16_f32(const void* src_bf16, float* dst, int64_t n, void* stream);
int mfv_fill_f32(float* dst, float value, int64_t n, void* stream);
/* torch.optim.SGD semantics (MAIN_CA:449): g += wd*p ; buf = mom*buf + g (buf = g on first step) ; p -= lr*buf.
 * Optionally refreshes the bf16 shadow in the same pass.                                                              */
int mfv_sgd_step(float* p, const float* g, float* buf, void* shadow_bf16, void* shadow_f16, int64_t n, float lr,
                 float momentum, float weight_decay, int first_step, void* stream);
/* torch.optim.Adam / AdamW semantics (MAIN_CA:457, MAIN_PRE:339); step is 1-based.                                    */
int mfv_adam_step(float* p, const float* g, float* exp_avg, float* exp_avg_sq, void* shadow_bf16, void* shadow_f16,
                  int64_t n, float lr, float beta1, float beta2, float eps, float weight_decay, int decoupled_wd,
                  int64_t step, void* stream);
/* The same two steps with the per-step scalars read from DEVICE memory, so a step captured in a CUDA graph follows the
 * learning-rate schedule (adjust_learning_rate, MAIN_CA:1043-1055 / MAIN_PRE:608-619) and Adam's bias correction
 * without being re-captured: lr_dev f32 [1]; step_dev i64 [1] = 1-based count of this update (the caller increments it
 * on the same stream before the call).                                                                               */
int mfv_sgd_step_dev(float* p, const float* g, float* buf, void* shadow_bf16, void* shadow_f16, int64_t n,
                     const float* lr_dev, float momentum, float weight_decay, int first_step, void* stream);
int mfv_adam_step_dev(float* p, const float* g, float* exp_avg, float* exp_avg_sq, void* shadow_bf16, void* shadow_f16,
                      int64_t n, const float* lr_dev, float beta1, float beta2, float eps, float weight_decay,
                      int decoupled_wd, const int64_t* step_dev, void* stream);

/* ---- LARS (MoCo-v3 optimizer) -------------------------------------------------------------------------------------
 * Replaces moco/optimizer.py:10-43 (LARS.step over every parameter with a gradient), built at MAIN_PRE:334-345 and
 * stepped at MAIN_PRE:547.  Per tensor, with eta = trust_coefficient:
 *   trust (ndim > 1): dp = g + wd*p ; q = (||p|| > 0 && ||dp|| > 0) ? eta*||p||/||dp|| : 1 ; dp *= q
 *   else            : dp = g                          (no weight decay, no trust ratio)
 *   mu = momentum*mu + dp ; p -= lr*mu                 (mu starts at zero; the 16-bit shadows are rewritten from p)
 * Frozen tensors are simply not in the table.  The table lives in device memory and is built once by the caller: one
 * record per tensor, every tensor split into chunks of MFV_LARS_CHUNK elements, chunk0 = the sum of
 * ceil(n / MFV_LARS_CHUNK) over the records before it (ascending), n_chunks = the total.  p, g, mu 16-byte aligned,
 * shadows 8-byte aligned (any n).  Two launches: the first writes per-chunk fp32 partial sums of p^2 and
 * dp^2 of the trust tensors into `workspace` (mfv_lars_workspace_bytes); in the second every chunk sums its tensor's partials in a fixed tree,
 * forms q (also stored in q_out f32 [n_tensors] when not NULL; 1 for the other tensors) and updates mu, p and the
 * shadows.  No atomics: bit-identical results for the same table and state.  lr_dev f32 [1] (the schedule, read on the
 * device, so a captured step follows it).                                                                            */
#define MFV_LARS_CHUNK 32768
typedef struct {
  float* p;
  const float* g;
  float* mu;
  void* shadow_bf16; /* NULL or bf16 [n] */
  void* shadow_f16;  /* NULL or fp16 [n] */
  int64_t n;
  int64_t chunk0;
  int32_t trust;     /* 1: ndim > 1 */
  int32_t reserved;
} mfv_lars_tensor;
size_t mfv_lars_workspace_bytes(int64_t n_chunks);
int mfv_lars_step_dev(const mfv_lars_tensor* table_dev, int64_t n_tensors, int64_t n_chunks, float* workspace,
                      float* q_out, const float* lr_dev, float momentum, float weight_decay, float trust_coefficient,
                      void* stream);

/* ---- paired input pipeline, device side (SURVEY 8(f) row 3) -----------------------------------------------------------
 * Replaces the per-sample torchvision transform of the training loaders (image_transform.py:50-84 composed at
 * MAIN_CA:524-531, applied at loader.py:127-129): RandomHorizontalFlip -> RandomRotation (nearest, Pillow's 16.16
 * fixed-point inverse map) -> RandomCrop / CenterCrop -> ToTensor -> Normalize, bit-identical to the eager sequence.
 * src uint8 [B][Hs][Ws][3] (the decoded + resized image), out f32 [B][3][crop][crop]; crop % 4 == 0.
 * params int32 [B][MFV_AUG_PARAMS] on the device: {flip, rotate, a0, a1, a2, a3, a4, a5, top, left, 0, 0}; with rotate != 0
 * the source pixel of rotated (x, y) is ((a2 + y*a1 + x*a0) >> 16, (a5 + y*a4 + x*a3) >> 16), outside the image -> 0.
 * mean3 / std3: f32 [3] on the device.                                                                                */
#define MFV_AUG_PARAMS 12
int mfv_augment_u8(const void* src_u8, const int32_t* params, const float* mean3, const float* std3, float* out,
                   int64_t B, int64_t Hs, int64_t Ws, int64_t crop, void* stream);

/* ---- epoch metrics kept on the device (SURVEY 8(f) row 2) -------------------------------------------------------------
 * Replaces the per-iteration `.item()` / `.cpu()` reads of MAIN_CA:884-899: logits = a + b + c (b, c optional),
 * loss_sum f64 [1] += loss[0] * rows, counters i64 [3] = {rows seen, argmax == target, rows dropped for capacity};
 * row i of this call goes to slot counters[0] + i of vals f32 [capacity][NC], preds / gts i32 [capacity].  The host
 * reads the buffers once per epoch (ROC AUC needs all scores) and zeroes loss_sum / counters.                          */
int mfv_epoch_metrics(const float* a, const float* b, const float* c, const int64_t* target, const float* loss,
                      int64_t rows, int64_t NC, double* loss_sum, int64_t* counters, int64_t capacity, float* vals,
                      int32_t* preds, int32_t* gts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MFVIT_H_ */
