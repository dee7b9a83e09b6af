"""Where the model looked, in plain PyTorch: the definition the GPU explain pass (mfvit.explain) is checked against.

  * vit_attention: per-block, per-head attention probabilities of an oracle/vit_ref.py encoder, computed by replaying
    its own modules block by block (the softmax of Attention.forward, MOD:52-64, restated without touching vit_ref).
  * rollout: CLS attention rollout (Abnar & Zuidema 2020) of head-averaged maps, A'_l = (A_l + I) / 2,
    out = e_0^T A'_{L-1} ... A'_0, as the row-vector chain v <- v A'_l from the last block down to the first.
  * cross_attention: the CrossAttention probabilities of an oracle/fusion_ref.py fusion on given final-normed tokens,
    from its own PreNorm / wq / wk modules, with the keys the forward builds (torch.cat((cal_q, x_other)), FUS:58,61).
"""
import torch


def block_attention(attn, x):
    """softmax(q k^T * scale) of a vit_ref Attention on its input x [B, S, C] (the output of norm1) -> [B, H, S, S]."""
    B, N, C = x.shape
    qkv = attn.qkv(x).reshape(B, N, 3, attn.num_heads, C // attn.num_heads).permute(2, 0, 3, 1, 4)
    q, k = qkv[0], qkv[1]
    return ((q @ k.transpose(-2, -1)) * attn.scale).softmax(dim=-1)


def vit_attention(vit, images):
    """vit_ref.VisionTransformerMoCo on images [B, 3, H, W] -> (tokens [B, S, C] as features3D returns them,
    probs [B, depth, H, S, S]).  Rows are query tokens, columns keys; token 0 is CLS, tokens 1.. the patches in
    row-major grid order."""
    x = vit.patch_embed(images)
    x = torch.cat((vit.cls_token.expand(x.shape[0], -1, -1), x), dim=1) + vit.pos_embed
    maps = []
    for blk in vit.blocks:
        maps.append(block_attention(blk.attn, blk.norm1(x)))
        x = blk(x)
    return vit.norm(x), torch.stack(maps, dim=1)


def rollout(means):
    """CLS attention rollout of head-averaged maps means [B, L, S, S] (block l at index l) -> [B, S]."""
    B, L, S, _ = means.shape
    eye = torch.eye(S, dtype=means.dtype, device=means.device)
    v = torch.zeros(B, 1, S, dtype=means.dtype, device=means.device)
    v[:, 0, 0] = 1
    for l in reversed(range(L)):
        v = v @ ((means[:, l] + eye) / 2)
    return v[:, 0]


def cross_probs(ca, x):
    """Attention of the CLS query of a fusion_ref CrossAttention on its (PreNorm'd) input x [B, S, C] -> [B, heads, S]."""
    B, N, C = x.shape
    h = ca.num_heads
    q = ca.wq(x[:, 0:1]).reshape(B, 1, h, C // h).permute(0, 2, 1, 3)
    k = ca.wk(x).reshape(B, N, h, C // h).permute(0, 2, 1, 3)
    return ((q @ k.transpose(-2, -1)) * ca.scale).softmax(dim=-1)[:, :, 0]


def cross_attention(fus, tok_cxr, tok_enh):
    """fusion_ref.Fus_CrossViT on final-normed tokens [B, S, C] of both branches -> [B, 2, heads, S]: direction 0 is
    the CXR CLS querying the ENH patches (cross_attn_layers.0.0), direction 1 the ENH CLS querying the CXR patches
    (cross_attn_layers.0.2); key 0 is the query's own CLS row."""
    layers = fus.multi_scale_transformers[0].cross_attn_layers[0]
    out = []
    for pre, own, other in ((layers[0], tok_cxr, tok_enh), (layers[2], tok_enh, tok_cxr)):
        x = pre.norm(torch.cat((own[:, 0:1], other[:, 1:]), dim=1))
        out.append(cross_probs(pre.fn, x))
    return torch.stack(out, dim=1)
