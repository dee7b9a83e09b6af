"""Drop-in for the reference fusion model (FUS): MultiScaleTransformerEncoder FUS:12-65 and Fus_CrossViT FUS:72-157.

Same constructor signature, module tree and 22 state-dict keys as the reference; the backbones are held as bound
`features3D` methods, NOT as sub-modules, exactly like FUS:80,83 (so parameters()/state_dict() exclude them, SURVEY
fact 4).  forward(vit_cxr, vit_enh, img_cxr, img_enh) returns (fused, x_cxr, x_enh) like FUS:157, computed as:
   one grouped pass of both ViT-S/16 encoders (mfv_vit_forward, G=2)  -> tokens [2,B,197,384]
   one fused CLS cross-attention + heads kernel (mfv_fusion_fwd)      -> fused, x_cxr, x_enh
The reference evaluates each backbone twice (FUS:128,131 / 133,135); with all drop rates 0 both evaluations are the
same function, so each backbone runs once here (SURVEY fact 5)."""
import os
import sys
from collections import namedtuple

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import _path  # noqa: E402,F401
import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
from mfvit import MfvError, explain  # noqa: E402
from mfvit.engine import encode, engine_for  # noqa: E402
from mfvit.functions import FusionFn  # noqa: E402
from model.module import Attention, CrossAttention, FeedForward, PreNorm  # noqa: E402,F401
from torch.nn.init import trunc_normal_  # noqa: E402  (timm.models.layers.trunc_normal_ in the reference, FUS:9)


# Fus_CrossViT.explain: the three outputs of forward plus where both backbones and the fusion looked
Explanation = namedtuple("Explanation", "fused x_cxr x_enh rollout cross maps")


class MultiScaleTransformerEncoder(nn.Module):
    def __init__(self, small_dim=384, large_dim=384, cross_attn_depth=1, cross_attn_heads=3, dropout=0.):
        super().__init__()
        if cross_attn_depth != 1 or dropout:
            raise MfvError("fused fusion kernel supports cross_attn_depth=1, dropout=0 (the reference's configuration)")
        self.cross_attn_layers = nn.ModuleList([])
        for _ in range(cross_attn_depth):
            self.cross_attn_layers.append(nn.ModuleList([
                PreNorm(large_dim, CrossAttention(large_dim, num_heads=cross_attn_heads, attn_drop=dropout)),
                nn.LayerNorm(large_dim, eps=1e-6),
                PreNorm(small_dim, CrossAttention(small_dim, num_heads=cross_attn_heads, attn_drop=dropout)),
                nn.LayerNorm(small_dim, eps=1e-6),
            ]))

    def forward(self, xs, xl):
        raise MfvError("MultiScaleTransformerEncoder is evaluated inside Fus_CrossViT.forward by the fused kernel; "
                       "only the CLS rows it produces are ever consumed (FUS:144-145)")


class Fus_CrossViT(nn.Module):
    def __init__(self, model_vit_cxr, model_vit_enh, num_classes=3, small_dim=384, large_dim=384, cross_attn_depth=1,
                 multi_scale_enc_depth=1, heads=3, dropout=0., pool='cls'):
        super().__init__()
        if multi_scale_enc_depth != 1 or pool != 'cls' or small_dim != large_dim:
            raise MfvError("fused fusion kernel supports multi_scale_enc_depth=1, pool='cls', equal dims")
        self.vit_features_cxr = model_vit_cxr.features3D
        self.vit_features_enh = model_vit_enh.features3D
        self.multi_scale_transformers = nn.ModuleList([])
        for _ in range(multi_scale_enc_depth):
            self.multi_scale_transformers.append(MultiScaleTransformerEncoder(
                small_dim=small_dim, large_dim=large_dim, cross_attn_depth=cross_attn_depth, cross_attn_heads=heads,
                dropout=dropout))
        self.pool = pool
        self.num_classes = num_classes
        self.heads = heads
        self.mlp_head_cxr = nn.Sequential(nn.Linear(small_dim, num_classes))
        self.mlp_head_enh = nn.Sequential(nn.Linear(large_dim, num_classes))
        self.apply(self._init_weights)

    def _init_weights(self, m):  # FUS:117-124
        if isinstance(m, nn.Linear):
            trunc_normal_(m.weight, std=.02)
            if isinstance(m, nn.Linear) and m.bias is not None:
                nn.init.constant_(m.bias, 0)
        elif isinstance(m, nn.LayerNorm):
            nn.init.constant_(m.bias, 0)
            nn.init.constant_(m.weight, 1.0)

    def _fusion_params(self, vit_cxr, vit_enh):
        L = self.multi_scale_transformers[0].cross_attn_layers[0]
        # direction 0: CXR CLS queries ENH patches  = cross_attn_s (index 0) + n_s (index 3) + mlp_head_cxr (FUS:58-63)
        # direction 1: ENH CLS queries CXR patches  = cross_attn_l (index 2) + n_l (index 1) + mlp_head_enh (FUS:50-55)
        pre, post = (L[0], L[2]), (L[3], L[1])
        head = (self.mlp_head_cxr[0], self.mlp_head_enh[0])
        vh = []
        for v in (vit_cxr, vit_enh):
            h = getattr(v, "head", None)
            vh.append(h if isinstance(h, nn.Linear) and h.out_features == self.num_classes else None)
        fields = [
            [m.norm.weight for m in pre], [m.norm.bias for m in pre],
            [m.fn.wq.weight for m in pre], [m.fn.wk.weight for m in pre], [m.fn.wv.weight for m in pre],
            [m.fn.proj.weight for m in pre], [m.fn.proj.bias for m in pre],
            [m.weight for m in post], [m.bias for m in post],
            [m.weight for m in head], [m.bias for m in head],
            [None if h is None else h.weight for h in vh], [None if h is None else h.bias for h in vh],
        ]
        return [t for pair in fields for t in pair], vh

    def fuse_tokens(self, tok, vit_cxr=None, vit_enh=None):
        """tok f32 [2,B,S,C] (cxr, enh) -> (fused, x_cxr, x_enh)."""
        params, vh = self._fusion_params(vit_cxr, vit_enh)
        fused, x = FusionFn.apply(tok, self.heads, *params)
        outs = []
        for g, (v, h) in enumerate(zip((vit_cxr, vit_enh), vh)):
            if h is not None:
                outs.append(x[g])
            elif v is not None:
                outs.append(v.apply_head(tok[g]) if hasattr(v, "apply_head") else v.head(tok[g][:, 0]))
            else:
                outs.append(None)
        return fused, outs[0], outs[1]

    def _check_backbones(self, vit_cxr, vit_enh, what):
        if getattr(self.vit_features_cxr, "__self__", None) is not vit_cxr or \
                getattr(self.vit_features_enh, "__self__", None) is not vit_enh:
            raise MfvError("Fus_CrossViT.%s expects the same backbone modules it was constructed with "
                           "(MAIN_CA:393,862)" % what)

    def forward(self, vit_cxr, vit_enh, img_cxr, img_enh):
        self._check_backbones(vit_cxr, vit_enh, "forward")
        tok = encode(engine_for(vit_cxr, vit_enh), [img_cxr, img_enh])
        return self.fuse_tokens(tok, vit_cxr, vit_enh)

    def explain(self, vit_cxr, vit_enh, img_cxr, img_enh, blocks=()):
        """forward's outputs and where the model looked, from one saving pass of the grouped encoder that forward uses
        (a branch's own single-branch engine would re-point its Parameters away from the buffer a trainer steps).
        Returns Explanation(fused, x_cxr, x_enh, rollout f32 [2, B, S] (cxr, enh), cross f32 [B, 2, heads, S],
        maps f32 [2, B, len(blocks), H, S, S] or None when `blocks` is empty).  cross[:, 0] is the CXR CLS querying
        the ENH patches, cross[:, 1] the reverse; key 0 is the query's own CLS row.  Everything is detached."""
        self._check_backbones(vit_cxr, vit_enh, "explain")
        with torch.no_grad():
            tok, maps, roll = explain.encoder_attention(engine_for(vit_cxr, vit_enh), [img_cxr, img_enh], blocks,
                                                        rollout=True)
            fused, x_cxr, x_enh = self.fuse_tokens(tok, vit_cxr, vit_enh)
            cross = explain.fusion_attention(tok, self._fusion_params(vit_cxr, vit_enh)[0], self.heads)
        return Explanation(fused, x_cxr, x_enh, roll, cross, maps)
