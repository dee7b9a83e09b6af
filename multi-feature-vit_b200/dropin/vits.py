"""Drop-in for the reference's absent `vits.py` (facebookresearch/moco-v3 VisionTransformerMoCo over timm's
VisionTransformer): same constructor names, attributes and state-dict keys (SURVEY.md 3.5 / 8(b)), but the arithmetic
runs in libmfvit.so on sm_100a.  Call sites served: MAIN_LPFT:44,276; MAIN_PRE:39,274; BLD:28-30,217-222.

The nn.Module tree below only *holds parameters* (so state_dict(), named_parameters(), head replacement, freezing and
optimisers behave exactly as with timm); `features3D` / `forward` hand the whole encoder to mfvit.engine.  There is no
eager / CPU path: calling forward on a CPU tensor raises.
"""
import math
from functools import reduce
from operator import mul

import _path  # noqa: F401
import torch
import torch.nn as nn
from mfvit import MfvError, explain
from mfvit.engine import encode, engine_for
from mfvit.functions import HeadFn

__all__ = ["vit_small", "vit_base", "vit_small_ori", "vit_base_ori", "vit_conv_small", "vit_conv_base",
           "VisionTransformerMoCo"]


def _no_eager(self, *a, **k):
    raise MfvError("%s has no eager forward: the encoder runs as fused sm_100a kernels through "
                   "VisionTransformerMoCo.features3D/forward" % type(self).__name__)


class PatchEmbed(nn.Module):
    def __init__(self, img_size=224, patch_size=16, in_chans=3, embed_dim=384):
        super().__init__()
        self.img_size = (img_size, img_size)
        self.patch_size = (patch_size, patch_size)
        self.grid_size = (img_size // patch_size, img_size // patch_size)
        self.num_patches = self.grid_size[0] * self.grid_size[1]
        self.proj = nn.Conv2d(in_chans, embed_dim, kernel_size=patch_size, stride=patch_size)

    forward = _no_eager


class Attention(nn.Module):
    def __init__(self, dim, num_heads, qkv_bias=True):
        super().__init__()
        self.num_heads = num_heads
        self.scale = (dim // num_heads) ** -0.5
        self.qkv = nn.Linear(dim, dim * 3, bias=qkv_bias)
        self.proj = nn.Linear(dim, dim)

    forward = _no_eager


class Mlp(nn.Module):
    def __init__(self, dim, hidden):
        super().__init__()
        self.fc1 = nn.Linear(dim, hidden)
        self.act = nn.GELU()
        self.fc2 = nn.Linear(hidden, dim)

    forward = _no_eager


class Block(nn.Module):
    def __init__(self, dim, num_heads, mlp_ratio, eps):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim, eps=eps)
        self.attn = Attention(dim, num_heads)
        self.norm2 = nn.LayerNorm(dim, eps=eps)
        self.mlp = Mlp(dim, int(dim * mlp_ratio))

    forward = _no_eager


def _sincos_pos_embed(grid_h, grid_w, embed_dim, temperature=10000.0):
    gw = torch.arange(grid_w, dtype=torch.float32)
    gh = torch.arange(grid_h, dtype=torch.float32)
    gw, gh = torch.meshgrid(gw, gh, indexing="ij")
    pos_dim = embed_dim // 4
    omega = 1.0 / (temperature ** (torch.arange(pos_dim, dtype=torch.float32) / pos_dim))
    out_w = torch.einsum("m,d->md", [gw.flatten(), omega])
    out_h = torch.einsum("m,d->md", [gh.flatten(), omega])
    pos = torch.cat([torch.sin(out_w), torch.cos(out_w), torch.sin(out_h), torch.cos(out_h)], dim=1)[None]
    return torch.cat([torch.zeros(1, 1, embed_dim), pos], dim=1)


class VisionTransformerMoCo(nn.Module):
    """ViT with fixed 2-D sin-cos position embedding and MoCo-v3 initialisation; timm-0.4 style attributes."""

    def __init__(self, img_size=224, patch_size=16, in_chans=3, num_classes=1000, embed_dim=384, depth=12, num_heads=6,
                 mlp_ratio=4.0, qkv_bias=True, stop_grad_conv1=False, norm_eps=1e-6, **unused):
        super().__init__()
        if in_chans != 3 or not qkv_bias or norm_eps != 1e-6:
            raise MfvError("mfvit encoder supports in_chans=3, qkv_bias=True, LayerNorm eps=1e-6")
        self.img_size, self.patch_size = img_size, patch_size
        self.num_classes = num_classes
        self.embed_dim = self.num_features = embed_dim
        self.depth, self.num_heads = depth, num_heads
        self.hidden_dim = int(embed_dim * mlp_ratio)
        self.num_tokens = 1
        self.patch_embed = PatchEmbed(img_size, patch_size, in_chans, embed_dim)
        self.cls_token = nn.Parameter(torch.zeros(1, 1, embed_dim))
        self.pos_embed = nn.Parameter(torch.zeros(1, self.patch_embed.num_patches + 1, embed_dim))
        self.blocks = nn.Sequential(*[Block(embed_dim, num_heads, mlp_ratio, norm_eps) for _ in range(depth)])
        self.norm = nn.LayerNorm(embed_dim, eps=norm_eps)
        self.head = nn.Linear(embed_dim, num_classes) if num_classes > 0 else nn.Identity()
        # --- MoCo-v3 initialisation (same order of RNG consumption as upstream vits.py)
        self.pos_embed = nn.Parameter(_sincos_pos_embed(*self.patch_embed.grid_size, embed_dim))
        self.pos_embed.requires_grad = False
        for name, m in self.named_modules():
            if isinstance(m, nn.Linear):
                if "qkv" in name:
                    val = math.sqrt(6.0 / float(m.weight.shape[0] // 3 + m.weight.shape[1]))
                    nn.init.uniform_(m.weight, -val, val)
                else:
                    nn.init.xavier_uniform_(m.weight)
                nn.init.zeros_(m.bias)
        nn.init.normal_(self.cls_token, std=1e-6)
        val = math.sqrt(6.0 / float(3 * reduce(mul, self.patch_embed.patch_size, 1) + embed_dim))
        nn.init.uniform_(self.patch_embed.proj.weight, -val, val)
        nn.init.zeros_(self.patch_embed.proj.bias)
        if stop_grad_conv1:
            self.patch_embed.proj.weight.requires_grad = False
            self.patch_embed.proj.bias.requires_grad = False

    # ------------------------------------------------------------------------------------------------ hot path
    def features3D(self, x):
        """All tokens after the final LayerNorm: [B, N+1, C] (FUS:128)."""
        return encode(engine_for(self), [x])[0]

    def forward_features(self, x):
        return self.features3D(x)[:, 0]

    def apply_head(self, tok):
        """head(tok[:, 0]) with whatever `self.head` currently is (MAIN_CA:309 re-assigns it, BLD:218-222 swaps in an MLP)."""
        head = self.head
        if isinstance(head, nn.Linear) and head.out_features <= 32 and tok.is_cuda:
            return HeadFn.apply(tok, head.weight, head.bias)
        return head(tok[:, 0])

    def forward(self, x):
        return self.apply_head(self.features3D(x))

    # ------------------------------------------------------------------------------------------------ explain pass
    def attention_maps(self, x, blocks=None):
        """Per-head attention probabilities f32 [B, len(blocks), H, S, S] of the given blocks (None: all of them), i.e.
        what a hook on each Attention's softmax would record; row i is query token i (0 = CLS), patches in row-major
        grid order.  Detached; works with or without grad mode."""
        blocks = range(self.depth) if blocks is None else list(blocks)
        _, maps, _ = explain.encoder_attention(engine_for(self), [x], blocks, rollout=False)
        if maps is None:
            S = self.patch_embed.num_patches + 1
            return torch.empty(x.shape[0], 0, self.num_heads, S, S, device=x.device)
        return maps[0]

    def attention_rollout(self, x):
        """CLS attention rollout f32 [B, S] over all blocks (head-averaged maps, identity added, Abnar & Zuidema
        2020): entry 0 is the CLS token, entries 1.. the patches in row-major grid order.  Detached."""
        _, _, roll = explain.encoder_attention(engine_for(self), [x], (), rollout=True)
        return roll[0]


def vit_small(**kwargs):
    # north_star: 197 tokens, head_dim 64 -> 6 heads (SURVEY fact 8); pass num_heads=12 for upstream MoCo-v3 checkpoints
    kwargs.setdefault("num_heads", 6)
    return VisionTransformerMoCo(patch_size=16, embed_dim=384, depth=12, mlp_ratio=4, **kwargs)


def vit_base(**kwargs):
    kwargs.setdefault("num_heads", 12)
    return VisionTransformerMoCo(patch_size=16, embed_dim=768, depth=12, mlp_ratio=4, **kwargs)


def vit_small_ori(**kwargs):
    kwargs.setdefault("num_heads", 12)  # upstream MoCo-v3 vit_small: 12 heads of 32
    return vit_small(**kwargs)


def vit_base_ori(**kwargs):
    return vit_base(**kwargs)


def vit_conv_small(**kwargs):
    raise NotImplementedError("vit_conv_small (ConvStem) is outside the MF-ViT CA hot path (SURVEY 8(b))")


def vit_conv_base(**kwargs):
    raise NotImplementedError("vit_conv_base (ConvStem) is outside the MF-ViT CA hot path (SURVEY 8(b))")
