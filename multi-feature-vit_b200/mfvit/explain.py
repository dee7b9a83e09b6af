"""Explain pass: where the model looked.  Per-head attention maps and CLS attention rollout of the encoder, and the
cross-attention maps of the fusion, computed on the GPU from buffers the ordinary forward already writes.

The fused attention never stores its probabilities, and an evaluation forward (save=False) keeps one activation slot
for all blocks.  So this runs one SAVING forward (every block keeps its qkv slot), recomputes the softmax of the
requested blocks from those 16-bit q / k with mfv_attn_probs, and hands the workspace back before returning.  Nothing on
the training or evaluation path changes: no new engine mode, no new workspace field (DESIGN.md 3.9)."""
import operator

import torch

from . import ops
from ._lib import MfvError
from .functions import FUSION_FIELDS


def _check_blocks(blocks, depth):
    out = []
    for b in blocks:
        try:
            i = operator.index(b)
        except TypeError:
            raise MfvError("block indices must be integers, got %r" % (b,)) from None
        if not 0 <= i < depth:
            raise MfvError("block index %d is outside [0, %d)" % (i, depth))
        out.append(i)
    return out


def encoder_attention(engine, images, blocks, rollout):
    """One saving forward of `engine` (G branches) on `images` (list of G CUDA tensors [B,3,H,W]), then the explain
    kernels on its stored qkv.  Returns (tokens f32 [G,B,S,C], maps f32 [G,B,len(blocks),H,S,S] or None when `blocks`
    is empty, rollout f32 [G,B,S] or None).  `maps` is a view of one [len(blocks),G*B,H,S,S] buffer (no copy)."""
    lay = engine.layout
    blocks = _check_blocks(blocks, lay.depth)
    with torch.no_grad():
        tokens, lease = engine.forward(list(images), save=True)
    try:
        ws = lease.ws
        G, B, S, H, L = engine.G, ws.B, lay.S, lay.H, lay.depth
        D, NB = lay.C // H, engine.G * ws.B
        dev = tokens.device
        # the qkv slots hold fp16 bits in the fp16-forward mode (the buffer is typed bf16)
        qkv = ws.qkv.view(torch.float16 if engine.fwd_f16 else torch.bfloat16).view(L, NB, S, 3, H, D)
        maps = torch.empty(len(blocks), NB, H, S, S, device=dev, dtype=torch.float32) if blocks else None
        means = torch.empty(L, NB, S, S, device=dev, dtype=torch.float32) if rollout else None
        for l in range(L):
            ks = [k for k, b in enumerate(blocks) if b == l]
            first = maps[ks[0]] if ks else None
            if first is not None or means is not None:
                ops.attn_probs(qkv[l], first, means[l] if means is not None else None)
            for k in ks[1:]:  # a block requested twice
                ops.attn_probs(qkv[l], maps[k])
        roll = ops.attn_rollout(means).view(G, B, S) if rollout else None
    finally:
        lease.release()
    if maps is not None:
        maps = maps.view(len(blocks), G, B, H, S, S).permute(1, 2, 0, 3, 4, 5)
    return tokens, maps, roll


def fusion_attention(tok, params, heads):
    """Cross-attention probabilities f32 [B,2,heads,S] of the fusion on final-normed tokens tok f32 [2,B,S,C];
    `params` are the 26 fusion tensors in FUSION_FIELDS x direction order (Fus_CrossViT._fusion_params)."""
    ps = [None if p is None else p.detach().contiguous() for p in params]
    struct = ops.fusion_param_struct({n: (ps[2 * i], ps[2 * i + 1]) for i, n in enumerate(FUSION_FIELDS)})
    return ops.fusion_attn(tok.contiguous(), struct, heads)
