"""Tensor-level wrappers over the C ABI (one function per mfv_* entry point).  PyTorch is used for device memory and
streams only; every computation below runs in libmfvit.so.  Inputs must be CUDA tensors - there is no CPU path."""
import ctypes as C

import torch

from . import _lib
from ._lib import (EPI_ATOMIC_F32, EPI_BF16, EPI_DGELU, EPI_F32, EPI_GELU, EPI_RESID_F32, EPI_RESID_LN, LARS_CHUNK,
                   EmaChunk, FusionGrads, FusionParams, GemmArgs, LarsTensor, MfvError, check)


def _lib_for(t):
    if not t.is_cuda:
        raise MfvError("mfvit ops need CUDA tensors (sm_100a); got a %s tensor - there is no CPU fallback" % t.device)
    return _lib.init(t.device.index if t.device.index is not None else torch.cuda.current_device())


def _p(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def gemm(A, B, Cout, *, M, N, K, G=1, lda, ldb, ldc, a_gstride=0, b_gstride=0, c_gstride=0, bias=None,
         bias_gstride=0, aux=None, aux_ld=0, aux_gstride=0, C2=None, C3=None, a_mn=False, b_mn=False, epilogue=EPI_BF16,
         splits=1, block_n=0, dtype_flags=0, cta_group=0, row_sum=None, rows_per_cta=0, ln=None):
    """ln (MFV_EPI_RESID_LN): dict(gamma, beta, mean, rstd, eps, out_f32)."""
    lib = _lib_for(A)
    a = GemmArgs()
    if ln is not None:
        a.ln_gamma, a.ln_beta = ln["gamma"].data_ptr(), ln["beta"].data_ptr()
        a.ln_mean, a.ln_rstd = ln["mean"].data_ptr(), ln["rstd"].data_ptr()
        a.ln_eps, a.ln_out_f32 = float(ln["eps"]), int(bool(ln.get("out_f32", False)))
    a.A, a.B, a.C, a.C2, a.bias, a.aux = (A.data_ptr(), B.data_ptr(), Cout.data_ptr(),
                                           C2.data_ptr() if C2 is not None else None,
                                           bias.data_ptr() if bias is not None else None,
                                           aux.data_ptr() if aux is not None else None)
    a.C3 = C3.data_ptr() if C3 is not None else None
    a.M, a.N, a.K, a.G = M, N, K, G
    a.lda, a.ldb, a.ldc = lda, ldb, ldc
    a.a_gstride, a.b_gstride, a.c_gstride = a_gstride, b_gstride, c_gstride
    a.aux_ld, a.aux_gstride, a.bias_gstride = aux_ld, aux_gstride, bias_gstride
    a.a_mn_major, a.b_mn_major, a.epilogue, a.splits, a.block_n = int(a_mn), int(b_mn), epilogue, splits, block_n
    a.dtype_flags = dtype_flags
    a.cta_group = cta_group
    a.rows_per_cta = rows_per_cta
    a.row_sum = row_sum.data_ptr() if row_sum is not None else None
    check(lib.mfv_gemm(C.byref(a), _stream()), "mfv_gemm")
    return Cout


def linear_fwd(x16, w16, bias=None, epilogue=EPI_BF16, out=None, out2=None, aux=None, block_n=0, dtype_flags=0,
               out3=None, cta_group=0, rows_per_cta=0):
    """x16 [G,M,K] bf16, w16 [G,N,K] bf16, bias [G,N] f32."""
    G, M, K = x16.shape
    N = w16.shape[1]
    if out is None:
        out = torch.empty(G, M, N, device=x16.device,
                          dtype=torch.float32 if epilogue in (EPI_RESID_F32, EPI_F32) else torch.bfloat16)
    return gemm(x16, w16, out, M=M, N=N, K=K, G=G, lda=K, ldb=K, ldc=N, a_gstride=M * K, b_gstride=N * K,
                c_gstride=M * N, bias=bias, bias_gstride=N, aux=aux, aux_ld=N, aux_gstride=M * N, C2=out2, C3=out3,
                epilogue=epilogue, block_n=block_n, dtype_flags=dtype_flags, cta_group=cta_group, rows_per_cta=rows_per_cta)


def linear_fwd_ln(x16, w16, bias, resid, gamma, beta, eps=1e-6, out_f32=False, f16=False, bf16_copy=False,
                  rows_per_cta=0):
    """x_new = resid + x16 @ w16^T + bias and LayerNorm(x_new) from the same epilogue (MFV_EPI_RESID_LN, N == 384).
    Returns (x_new f32, y (16-bit, or f32 with out_f32), y_bf16_copy | None, mean, rstd)."""
    G, M, K = x16.shape
    N = w16.shape[1]
    dev = x16.device
    x_new = torch.empty(G, M, N, device=dev, dtype=torch.float32)
    y = torch.empty(G, M, N, device=dev, dtype=torch.float32 if out_f32 else (torch.float16 if f16 else torch.bfloat16))
    ycopy = torch.empty(G, M, N, device=dev, dtype=torch.bfloat16) if bf16_copy else None
    mean = torch.empty(G, M, device=dev, dtype=torch.float32)
    rstd = torch.empty_like(mean)
    flags = (3 if x16.dtype == torch.float16 else 0) | (4 if f16 else 0)
    gemm(x16, w16, x_new, M=M, N=N, K=K, G=G, lda=K, ldb=K, ldc=N, a_gstride=M * K, b_gstride=N * K, c_gstride=M * N,
         bias=bias, bias_gstride=N, aux=resid, aux_ld=N, aux_gstride=M * N, C2=y, C3=ycopy, epilogue=EPI_RESID_LN,
         dtype_flags=flags, rows_per_cta=rows_per_cta,
         ln=dict(gamma=gamma, beta=beta, mean=mean, rstd=rstd, eps=eps, out_f32=out_f32))
    return x_new, y, ycopy, mean, rstd


def linear_dgrad(dy16, w16, epilogue=EPI_BF16, aux=None, out=None, block_n=0, cta_group=0, out2=None, rows_per_cta=0):
    """dy16 [G,M,N] bf16, w16 [G,N,K] bf16 -> dx [G,M,K]."""
    G, M, N = dy16.shape
    K = w16.shape[2]
    if out is None:
        out = torch.empty(G, M, K, device=dy16.device, dtype=torch.float32 if epilogue == EPI_F32 else torch.bfloat16)
    return gemm(dy16, w16, out, M=M, N=K, K=N, G=G, lda=N, ldb=K, ldc=K, a_gstride=M * N, b_gstride=N * K,
                c_gstride=M * K, aux=aux, aux_ld=K, aux_gstride=M * K, b_mn=True, epilogue=epilogue, block_n=block_n,
                cta_group=cta_group, C2=out2, rows_per_cta=rows_per_cta)


def linear_wgrad(dy16, x16, dw, splits=8, block_n=0, cta_group=0, db=None):
    """dw [G,N,K] f32 += dy16[G,M,N]^T x16[G,M,K]; db [G,N] f32 += colsum(dy16) (384-wide pair tiles only)."""
    G, M, N = dy16.shape
    K = x16.shape[2]
    return gemm(dy16, x16, dw, M=N, N=K, K=M, G=G, lda=N, ldb=K, ldc=K, a_gstride=M * N, b_gstride=M * K,
                c_gstride=N * K, a_mn=True, b_mn=True, epilogue=EPI_ATOMIC_F32, splits=splits, block_n=block_n,
                cta_group=cta_group, row_sum=db, bias_gstride=N if db is not None else 0)


def linear_wgrad_pair(dy0, x0, dw0, db0, dy1, x1, dw1, db1, splits=4):
    """Two weight gradients in one launch (mfv_gemm_wgrad_pair): dw_i [G,N_i,K_i] += dy_i^T x_i, db_i += colsum(dy_i)."""
    lib = _lib_for(dy0)
    args = []
    for dy, x, dw, db in ((dy0, x0, dw0, db0), (dy1, x1, dw1, db1)):
        G, M, N = dy.shape
        K = x.shape[2]
        a = GemmArgs()
        a.A, a.B, a.C = dy.data_ptr(), x.data_ptr(), dw.data_ptr()
        a.M, a.N, a.K, a.G = N, K, M, G
        a.lda, a.ldb, a.ldc = N, K, K
        a.a_gstride, a.b_gstride, a.c_gstride = M * N, M * K, N * K
        a.a_mn_major, a.b_mn_major, a.epilogue, a.splits = 1, 1, EPI_ATOMIC_F32, splits
        a.bias_gstride = N if db is not None else 0
        a.row_sum = db.data_ptr() if db is not None else None
        args.append(a)
    if args[0].bias_gstride != args[1].bias_gstride:  # one stride for both bias outputs: the caller packs them alike
        raise MfvError("linear_wgrad_pair: both bias gradients must use the same group stride")
    check(lib.mfv_gemm_wgrad_pair(C.byref(args[0]), C.byref(args[1]), _stream()), "mfv_gemm_wgrad_pair")


def layernorm_fwd(x, gamma, beta, eps, want_bf16=True, want_f32=False, f16=False, bf16_copy=False):
    G, rows, Cd = x.shape
    lib = _lib_for(x)
    y16 = torch.empty_like(x, dtype=torch.float16 if f16 else torch.bfloat16) if want_bf16 else None
    ycopy = torch.empty_like(x, dtype=torch.bfloat16) if bf16_copy else None
    y32 = torch.empty_like(x) if want_f32 else None
    mean = torch.empty(G, rows, device=x.device, dtype=torch.float32)
    rstd = torch.empty_like(mean)
    check(lib.mfv_layernorm_fwd(_p(x), _p(gamma), _p(beta), _p(y16), int(f16), _p(ycopy), _p(y32), _p(mean), _p(rstd),
                                G, rows, Cd, gamma.stride(0) if gamma.dim() > 1 else 0, eps, _stream()),
          "mfv_layernorm_fwd")
    if bf16_copy:
        return y16, y32, mean, rstd, ycopy
    return y16, y32, mean, rstd


def layernorm_bwd(dy, x, mean, rstd, gamma, dres=None, dgamma=None, dbeta=None, want_bf16=True, dx_colsum=None,
                  want_f32=True):
    """dres: f32 or bf16 residual-path gradient (or None)."""
    G, rows, Cd = x.shape
    lib = _lib_for(x)
    dx = torch.empty_like(x) if want_f32 else None
    dx16 = torch.empty_like(x, dtype=torch.bfloat16) if want_bf16 else None
    dy16 = dy if dy.dtype == torch.bfloat16 else None
    dy32 = dy if dy.dtype == torch.float32 else None
    dres32 = dres if dres is not None and dres.dtype == torch.float32 else None
    dres16 = dres if dres is not None and dres.dtype == torch.bfloat16 else None
    check(lib.mfv_layernorm_bwd(_p(dy16), _p(dy32), _p(dres32), _p(dres16), _p(x), _p(mean), _p(rstd), _p(gamma), _p(dx), _p(dx16),
                                _p(dgamma), _p(dbeta), _p(dx_colsum), G, rows, Cd,
                                gamma.stride(0) if gamma.dim() > 1 else 0,
                                _stream()), "mfv_layernorm_bwd")
    return dx, dx16


def attn_fwd(qkv, H, f16=False, bf16_copy=False):
    """qkv bf16 [NB,S,3,H,D] -> o (bf16 | fp16) [NB,S,H,D], lse f32 [NB,H,S] (+ optional bf16 copy of o)."""
    NB, S, three, Hh, D = qkv.shape
    assert three == 3 and Hh == H
    lib = _lib_for(qkv)
    o = torch.empty(NB, S, H, D, device=qkv.device, dtype=torch.float16 if f16 else torch.bfloat16)
    ocopy = torch.empty(NB, S, H, D, device=qkv.device, dtype=torch.bfloat16) if bf16_copy else None
    lse = torch.empty(NB, H, S, device=qkv.device, dtype=torch.float32)
    check(lib.mfv_attn_fwd(_p(qkv), int(qkv.dtype == torch.float16), _p(o), int(f16), _p(ocopy), _p(lse), NB, S, H, D, float(D) ** -0.5, _stream()),
          "mfv_attn_fwd")
    if bf16_copy:
        return o, lse, ocopy
    return o, lse


def attn_bwd(qkv, o, d_o, lse):
    NB, S, _, H, D = qkv.shape
    lib = _lib_for(qkv)
    dqkv = torch.empty_like(qkv, dtype=torch.bfloat16)
    delta = torch.empty_like(lse)
    nws = lib.mfv_attn_bwd_workspace_bytes(NB, S, H, D)
    ws = torch.empty(nws // 4, device=qkv.device, dtype=torch.float32) if nws else None
    check(lib.mfv_attn_bwd_ws(_p(qkv), int(qkv.dtype == torch.float16), _p(o), _p(d_o), _p(lse), _p(delta), _p(dqkv),
                              _p(ws), NB, S, H, D, float(D) ** -0.5, _stream()), "mfv_attn_bwd_ws")
    return dqkv


def colsum_bf16(x, out):
    G, rows, Cd = x.shape
    check(_lib_for(x).mfv_colsum_bf16(_p(x), _p(out), G, rows, Cd, out.stride(0) if out.dim() > 1 else 0, _stream()),
          "mfv_colsum_bf16")
    return out


def cast_bf16(src, dst=None):
    if dst is None:
        dst = torch.empty_like(src, dtype=torch.bfloat16)
    check(_lib_for(src).mfv_cast_shadow(_p(src), _p(dst), None, src.numel(), _stream()), "mfv_cast_shadow")
    return dst


def cast_shadow(src, dst_bf16=None, dst_f16=None):
    """One pass over the fp32 master writing the bf16 and/or fp16 GEMM-operand copies."""
    check(_lib_for(src).mfv_cast_shadow(_p(src), _p(dst_bf16), _p(dst_f16), src.numel(), _stream()), "mfv_cast_shadow")


def patch_embed_tma(imgs, w, bias, cls, pos, f16=True):
    """imgs: list of G f32 [B,3,HW,HW]; w f32 [G,C,768] (rounded here to the 16-bit operand format), bias / cls f32 [G,C],
    pos f32 [G,S,C] -> x f32 [G,B,S,C].  The G parameter sets must sit at one stride inside a common buffer (as the
    engine's flat master / shadow do): here they are packed into one."""
    G, B, HW = len(imgs), imgs[0].shape[0], imgs[0].shape[-1]
    Cd, S = w.shape[1], pos.shape[1]
    n = [Cd * 768, Cd, Cd, S * Cd]
    P = (sum(n) + 7) // 8 * 8
    flat = torch.zeros(G, P, device=w.device, dtype=torch.float32)
    offs, o = [], 0
    for k in n:
        offs.append(o)
        o += k
    for g in range(G):
        for t, off, k in zip((w[g], bias[g], cls[g], pos[g]), offs, n):
            flat[g, off:off + k] = t.reshape(-1)
    flat16 = flat.to(torch.float16 if f16 else torch.bfloat16)
    x = torch.empty(G, B, S, Cd, device=w.device, dtype=torch.float32)
    im = [t.contiguous() for t in imgs]
    check(_lib_for(w).mfv_patch_embed_tma(_p(im[0]), _p(im[1]) if G > 1 else None, _p(flat16[0, offs[0]:]), int(f16),
                                          _p(flat[0, offs[1]:]), _p(flat[0, offs[2]:]), _p(flat[0, offs[3]:]), _p(x), G, B,
                                          HW, Cd, P, _stream()), "mfv_patch_embed_tma")
    return x


def cast_bf16_f32_(src_bf16, dst_f32):
    check(_lib_for(src_bf16).mfv_cast_bf16_f32(_p(src_bf16), _p(dst_f32), src_bf16.numel(), _stream()), "mfv_cast_bf16_f32")
    return dst_f32


def fill_(t, value=0.0):
    check(_lib_for(t).mfv_fill_f32(_p(t), float(value), t.numel(), _stream()), "mfv_fill_f32")
    return t


def ema_update_(chunks_dev, n_chunks, max_elems, m):
    """chunks_dev: uint8 CUDA tensor holding n_chunks mfv_ema_chunk records.  k = k*m + q*(1.-m), bit-exact with the
    eager reference: m and (1.-m) are rounded to fp32 separately, exactly as torch does for Python-scalar operands."""
    check(_lib_for(chunks_dev).mfv_ema_update(_p(chunks_dev), n_chunks, max_elems, float(m), float(1.0 - m),
                                              _stream()), "mfv_ema_update")


def make_ema_chunks(pairs, device):
    """pairs: list of (k_tensor, q_tensor) fp32 contiguous.  Adjacent-in-memory tensors are merged into one chunk."""
    merged = []
    for k, q in pairs:
        n = k.numel()
        if merged:
            pk, pq, pn = merged[-1]
            if pk + 4 * pn == k.data_ptr() and pq + 4 * pn == q.data_ptr():
                merged[-1] = (pk, pq, pn + n)
                continue
        merged.append((k.data_ptr(), q.data_ptr(), n))
    arr = (EmaChunk * len(merged))()
    for i, (pk, pq, n) in enumerate(merged):
        arr[i].k, arr[i].q, arr[i].n = pk, pq, n
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    return host.to(device), len(merged), max(n for _, _, n in merged)


def fusion_param_struct(tensors, cls=FusionParams):
    """tensors: dict name -> (t_dir0, t_dir1) with None allowed."""
    s = cls()
    for name, pair in tensors.items():
        arr = getattr(s, name)
        for d in range(2):
            arr[d] = pair[d].data_ptr() if pair[d] is not None else None
    return s


def fusion_fwd(tok, params, B, S, Cd, heads, NC, saved=None):
    """saved (fusion_scratch): runs the batched stage kernels and keeps the forward state there for fusion_bwd; without
    it the single-kernel forward runs and a later backward recomputes what it needs."""
    lib = _lib_for(tok)
    fused = torch.empty(B, NC, device=tok.device, dtype=torch.float32)
    x = torch.empty(2, B, NC, device=tok.device, dtype=torch.float32)
    check(lib.mfv_fusion_fwd(_p(tok), C.byref(params), _p(fused), _p(x), _p(saved), B, S, Cd, heads, NC, _stream()),
          "mfv_fusion_fwd")
    return fused, x


def fusion_scratch(tok, B, S, Cd, heads):
    n = _lib_for(tok).mfv_fusion_saved_floats(B, S, Cd, heads)
    return torch.empty(n, device=tok.device, dtype=torch.float32)


def fusion_bwd(tok, params, grads, d_fused, d_x, B, S, Cd, heads, NC, dtok=None, scratch=None, defer=False):
    """defer=True: only dtok is ordered on the current stream; the parameter gradients are finished by
    fusion_bwd_join(), and `scratch`, d_fused, d_x must be kept alive and untouched until then."""
    lib = _lib_for(tok)
    if scratch is None:
        if defer:
            raise MfvError("a deferred fusion backward needs a caller-owned scratch buffer")
        scratch = fusion_scratch(tok, B, S, Cd, heads)
    if dtok is None:
        dtok = torch.empty_like(tok)
    fn = lib.mfv_fusion_bwd_deferred if defer else lib.mfv_fusion_bwd
    check(fn(_p(tok), C.byref(params), _p(scratch), _p(d_fused), _p(d_x), _p(dtok), C.byref(grads), B, S, Cd, heads, NC,
             _stream()), "mfv_fusion_bwd")
    return dtok


def fusion_bwd_join(device=None):
    lib = _lib.init(torch.cuda.current_device() if device is None or device.index is None else device.index)
    check(lib.mfv_fusion_bwd_join(_stream()), "mfv_fusion_bwd_join")


def linear_small_fwd(x, ldx, w, b, rows):
    N, Cd = w.shape
    y = torch.empty(rows, N, device=x.device, dtype=torch.float32)
    check(_lib_for(x).mfv_linear_small_fwd(_p(x), ldx, _p(w), _p(b), _p(y), rows, Cd, N, _stream()),
          "mfv_linear_small_fwd")
    return y


def linear_small_bwd(x, ldx, w, dy, dx, lddx, dw, db, rows):
    N, Cd = w.shape
    check(_lib_for(x).mfv_linear_small_bwd(_p(x), ldx, _p(w), _p(dy), _p(dx), lddx, _p(dw), _p(db), rows, Cd, N,
                                           _stream()), "mfv_linear_small_bwd")


def _check_labels(target, rows, device, what):
    """The kernels read `target` as int64 [rows]: anything else would be reinterpreted silently (the reference casts
    with target.long(), MAIN_CA:859)."""
    if target.dtype != torch.int64 or tuple(target.shape) != (rows,) or not target.is_contiguous() \
            or target.device != device:
        raise MfvError("%s wants a contiguous int64 label tensor of shape [%d] on %s, got %s %s on %s"
                       % (what, rows, device, target.dtype, tuple(target.shape), target.device))


def ce_small(a, b, c, target, want_grad=True):
    rows, NC = a.shape
    if NC > 32:
        raise MfvError("ce_small handles at most 32 classes")
    _check_labels(target, rows, a.device, "ce_small")
    loss = torch.empty(1, device=a.device, dtype=torch.float32)
    dl = torch.empty_like(a) if want_grad else None
    check(_lib_for(a).mfv_ce_small(_p(a), _p(b), _p(c), _p(target), _p(loss), _p(dl), rows, NC, _stream()),
          "mfv_ce_small")
    return loss, dl


def augment_u8(src_u8, params, mean3, std3, crop, out=None):
    """src uint8 [B][Hs][Ws][3], params int32 [B][12] (mfvit.data.pack_params) -> normalised f32 [B][3][crop][crop]."""
    B, Hs, Ws, ch = src_u8.shape
    if ch != 3 or src_u8.dtype != torch.uint8 or not src_u8.is_contiguous():
        raise MfvError("augment_u8 wants a contiguous uint8 [B][H][W][3] batch")
    if params.dtype != torch.int32 or tuple(params.shape) != (B, 12) or not params.is_contiguous():
        raise MfvError("augment_u8 wants int32 [B][12] parameters")
    if out is None:
        out = torch.empty(B, 3, crop, crop, device=src_u8.device, dtype=torch.float32)
    check(_lib_for(src_u8).mfv_augment_u8(_p(src_u8), _p(params), _p(mean3), _p(std3), _p(out), B, Hs, Ws, crop,
                                          _stream()), "mfv_augment_u8")
    return out


def epoch_metrics_(a, b, c, target, loss, loss_sum, counters, vals, preds, gts):
    rows, NC = a.shape
    _check_labels(target, rows, a.device, "epoch_metrics_")
    check(_lib_for(a).mfv_epoch_metrics(_p(a), _p(b), _p(c), _p(target), _p(loss), rows, NC, _p(loss_sum),
                                        _p(counters), vals.shape[0], _p(vals), _p(preds), _p(gts), _stream()),
          "mfv_epoch_metrics")


def infonce_fwd(q_raw, k_raw, queue, T):
    N, D = q_raw.shape
    K = queue.shape[1]
    dev = q_raw.device
    qn = torch.empty_like(q_raw)
    kn = torch.empty_like(k_raw)
    logits = torch.empty(N, K + 1, device=dev, dtype=torch.float32)
    lse = torch.empty(N * (1 + 2 * (K // 64)), device=dev, dtype=torch.float32)
    loss = torch.empty(1, device=dev, dtype=torch.float32)
    check(_lib_for(q_raw).mfv_infonce_fwd(_p(q_raw), _p(k_raw), _p(queue), _p(qn), _p(kn), _p(logits), _p(lse),
                                          _p(loss), N, D, K, float(T), _stream()), "mfv_infonce_fwd")
    return qn, kn, logits, lse, loss


def infonce_bwd(q_raw, qn, kn, queue, logits, lse, T, dlogits=None, gscale=1.0, override=None, ov_start=0):
    N, D = q_raw.shape
    K = queue.shape[1]
    dq = torch.empty_like(q_raw)
    ov_n = 0 if override is None else override.shape[1]
    check(_lib_for(q_raw).mfv_infonce_bwd(_p(q_raw), _p(qn), _p(kn), _p(queue), _p(logits), _p(lse), _p(dlogits),
                                          _p(override), int(ov_start), int(ov_n), float(gscale), _p(dq), N, D, K,
                                          float(T), _stream()), "mfv_infonce_bwd")
    return dq


def queue16_update_(queue, queue16, col0=0, ncols=None):
    """queue16[:, col0:col0+ncols] = fp16(queue[...]): the fp16 shadow the tensor-core InfoNCE reads."""
    D, K = queue.shape
    ncols = K - col0 if ncols is None else ncols
    check(_lib_for(queue).mfv_queue16_update(_p(queue), _p(queue16), D, K, int(col0), int(ncols), _stream()),
          "mfv_queue16_update")
    return queue16


def infonce_tc_fwd(q_raw, k_raw, queue16, T):
    """Tensor-core InfoNCE forward.  Returns (qn, kn, logits_buf [N, K+8], lse, loss); logits = logits_buf[:, 7:]."""
    N, D = q_raw.shape
    K = queue16.shape[1]
    dev = q_raw.device
    qn, kn = torch.empty_like(q_raw), torch.empty_like(k_raw)
    qs16 = torch.empty(N, D, device=dev, dtype=torch.float16)
    buf = torch.empty(N, K + 8, device=dev, dtype=torch.float32)
    lse = torch.empty(N * (1 + 2 * (K // 1024)), device=dev, dtype=torch.float32)
    loss = torch.empty(1, device=dev, dtype=torch.float32)
    check(_lib_for(q_raw).mfv_infonce_tc_fwd(_p(q_raw), _p(k_raw), _p(queue16), _p(qn), _p(kn), _p(qs16), _p(buf), K + 8,
                                             _p(lse), _p(loss), N, D, K, float(T), _stream()), "mfv_infonce_tc_fwd")
    return qn, kn, buf, lse, loss


def infonce_tc_bwd(q_raw, qn, kn, queue16, buf, lse, T, dlogits_buf=None, gscale=1.0, override=None, ov_start=0):
    """dq_raw of the tensor-core path; dlogits_buf (optional) has the [N, K+8] layout of the logits buffer."""
    N, D = q_raw.shape
    K = queue16.shape[1]
    dev = q_raw.device
    dq = torch.empty_like(q_raw)
    dl16 = torch.empty(N, K, device=dev, dtype=torch.float16)
    scal = torch.empty(4, device=dev, dtype=torch.float32)
    ov_n = 0 if override is None else override.shape[1]
    check(_lib_for(q_raw).mfv_infonce_tc_bwd(_p(q_raw), _p(qn), _p(kn), _p(queue16), _p(buf), K + 8, _p(lse),
                                             _p(dlogits_buf), _p(override), int(ov_start), int(ov_n), float(gscale),
                                             _p(dl16), _p(scal), _p(dq), N, D, K, float(T), _stream()),
          "mfv_infonce_tc_bwd")
    return dq


def enqueue_keys_(keys, queue, ptr):
    n, D = keys.shape
    K = queue.shape[1]
    check(_lib_for(keys).mfv_enqueue_keys(_p(keys), _p(queue), n, D, K, int(ptr), _stream()), "mfv_enqueue_keys")


def sgd_step_(p, g, buf, shadow, lr, momentum, weight_decay, first_step, shadow16=None):
    check(_lib_for(p).mfv_sgd_step(_p(p), _p(g), _p(buf), _p(shadow), _p(shadow16), p.numel(), float(lr), float(momentum),
                                   float(weight_decay), int(bool(first_step)), _stream()), "mfv_sgd_step")


def sgd_step_dev_(p, g, buf, shadow, lr_dev, momentum, weight_decay, first_step, shadow16=None):
    """SGD step with the learning rate read from the 1-element device tensor lr_dev (graph-replay safe schedules)."""
    check(_lib_for(p).mfv_sgd_step_dev(_p(p), _p(g), _p(buf), _p(shadow), _p(shadow16), p.numel(), _p(lr_dev),
                                       float(momentum), float(weight_decay), int(bool(first_step)), _stream()),
          "mfv_sgd_step_dev")


def adam_step_dev_(p, g, m1, m2, shadow, lr_dev, betas, eps, weight_decay, decoupled, step_dev, shadow16=None):
    """Adam / AdamW step with lr and the 1-based step count read from device tensors (f32 [1], i64 [1])."""
    check(_lib_for(p).mfv_adam_step_dev(_p(p), _p(g), _p(m1), _p(m2), _p(shadow), _p(shadow16), p.numel(), _p(lr_dev),
                                        float(betas[0]), float(betas[1]), float(eps), float(weight_decay),
                                        int(bool(decoupled)), _p(step_dev), _stream()), "mfv_adam_step_dev")


def make_lars_table(records, device):
    """records: list of (p, g, mu, shadow_bf16 | None, shadow_f16 | None, trust) with p, g, mu contiguous fp32 CUDA
    tensors of one size (16-byte aligned) and the shadows bf16 / fp16 of that size (8-byte aligned); trust = the
    tensor is a matrix (ndim > 1).  Returns (table_dev uint8, n_tensors, n_chunks).  The table holds raw pointers: the
    caller keeps every tensor alive (and in place) for as long as it steps with the table."""
    arr = (LarsTensor * len(records))()
    chunk = 0
    for i, (p, g, mu, sb, sh, trust) in enumerate(records):
        n = p.numel()
        for t, what in ((p, "p"), (g, "g"), (mu, "mu")):
            _lib_for(t)
            if t.dtype != torch.float32 or t.numel() != n or not t.is_contiguous() or t.device != p.device:
                raise MfvError("make_lars_table: record %d: %s must be a contiguous fp32 tensor of %d elements on %s"
                               % (i, what, n, p.device))
            if t.data_ptr() & 15:
                raise MfvError("make_lars_table: record %d: %s is not 16-byte aligned" % (i, what))
        for t, dt, what in ((sb, torch.bfloat16, "shadow_bf16"), (sh, torch.float16, "shadow_f16")):
            if t is None:
                continue
            _lib_for(t)
            if t.dtype != dt or t.numel() != n or not t.is_contiguous() or t.device != p.device:
                raise MfvError("make_lars_table: record %d: %s must be a contiguous %s tensor of %d elements on %s"
                               % (i, what, dt, n, p.device))
            if t.data_ptr() & 7:
                raise MfvError("make_lars_table: record %d: %s is not 8-byte aligned" % (i, what))
        if n == 0:
            raise MfvError("make_lars_table: record %d is empty" % i)
        r = arr[i]
        r.p, r.g, r.mu = p.data_ptr(), g.data_ptr(), mu.data_ptr()
        r.shadow_bf16 = sb.data_ptr() if sb is not None else None
        r.shadow_f16 = sh.data_ptr() if sh is not None else None
        r.n, r.chunk0, r.trust = n, chunk, int(bool(trust))
        chunk += (n + LARS_CHUNK - 1) // LARS_CHUNK
    host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8)
    return host.to(device), len(records), chunk


def lars_workspace(n_chunks, device):
    n = _lib.load().mfv_lars_workspace_bytes(int(n_chunks))
    return torch.empty(max(n // 4, 2), device=device, dtype=torch.float32)


def lars_step_dev_(table_dev, n_tensors, n_chunks, workspace, lr_dev, momentum, weight_decay, trust_coefficient,
                   q_out=None):
    """LARS step (moco/optimizer.py:10-43) over every tensor of a make_lars_table() table, learning rate read from the
    device tensor lr_dev f32 [1]; q_out (optional) f32 [n_tensors] receives the trust ratio of each tensor (1 for
    vectors and for matrices with a zero norm)."""
    lib = _lib_for(table_dev)
    if workspace.numel() * 4 < lib.mfv_lars_workspace_bytes(int(n_chunks)) or workspace.dtype != torch.float32:
        raise MfvError("lars_step_dev_: the workspace holds fewer than the %d chunks' partial sums" % n_chunks)
    if q_out is not None and (q_out.dtype != torch.float32 or q_out.numel() < n_tensors or not q_out.is_contiguous()):
        raise MfvError("lars_step_dev_: q_out must be a contiguous fp32 tensor of at least %d elements" % n_tensors)
    check(lib.mfv_lars_step_dev(_p(table_dev), int(n_tensors), int(n_chunks), _p(workspace), _p(q_out), _p(lr_dev),
                                float(momentum), float(weight_decay), float(trust_coefficient), _stream()),
          "mfv_lars_step_dev")


def adam_step_(p, g, m1, m2, shadow, lr, betas, eps, weight_decay, decoupled, step, shadow16=None):
    check(_lib_for(p).mfv_adam_step(_p(p), _p(g), _p(m1), _p(m2), _p(shadow), _p(shadow16), p.numel(), float(lr), float(betas[0]),
                                    float(betas[1]), float(eps), float(weight_decay), int(bool(decoupled)), int(step),
                                    _stream()), "mfv_adam_step")
