"""oracle/attention_ref.py (no GPU): the replayed maps are the softmax the oracle modules compute inside their own forward,
the rollout is the product it is defined as, and the mistakes an explain pass is likely to make are caught."""
import contextlib

import pytest
import torch

from oracle import attention_ref as A
from oracle import fusion_ref, vit_ref


@contextlib.contextmanager
def capture_softmax():
    """Records the output of every Tensor.softmax call made inside the block."""
    seen = []
    orig = torch.Tensor.softmax

    def rec(self, *a, **k):
        out = orig(self, *a, **k)
        seen.append(out.detach().clone())
        return out
    torch.Tensor.softmax = rec
    try:
        yield seen
    finally:
        torch.Tensor.softmax = orig


def _same(a, b):
    return a.shape == b.shape and torch.allclose(a, b, rtol=1e-6, atol=1e-7)


def _small_vit(heads, seed=0):
    torch.manual_seed(seed)
    return vit_ref.VisionTransformerMoCo(img_size=64, embed_dim=96, depth=3, num_heads=heads, num_classes=3).double()


def _fusion(heads, seed=0, B=3, S=17, C=384):
    torch.manual_seed(seed)
    vc, ve = _small_vit(3, seed), _small_vit(3, seed + 1)
    fus = fusion_ref.Fus_CrossViT(vc, ve, heads=heads).double()
    with torch.no_grad():
        for p in fus.parameters():
            if p.dim() == 1:
                p.add_(torch.randn_like(p) * 0.05)
    g = torch.Generator().manual_seed(seed + 7)
    tc = torch.randn(B, S, C, generator=g, dtype=torch.float64)
    te = torch.randn(B, S, C, generator=g, dtype=torch.float64)
    return fus, tc, te


# ------------------------------------------------------------------------------------------------ replay = forward
@pytest.mark.parametrize("heads", [1, 2, 3, 4, 6, 12])
def test_vit_replay_equals_the_softmax_of_the_forward(heads):
    vit = _small_vit(heads)
    x = torch.randn(2, 3, 64, 64, dtype=torch.float64)
    with torch.no_grad(), capture_softmax() as seen:
        tok_fwd = vit.features3D(x)
    with torch.no_grad():
        tok, maps = A.vit_attention(vit, x)
    assert len(seen) == 3 and maps.shape == (2, 3, heads, 17, 17)
    assert torch.equal(tok, tok_fwd)
    for l in range(3):
        assert _same(maps[:, l], seen[l]), l
    # mutation: a transposed map (keys as rows) is not what the forward computed
    assert not _same(maps[:, 1].transpose(-1, -2), seen[1])


@pytest.mark.parametrize("heads", [1, 2, 3, 4])
def test_fusion_replay_equals_the_softmax_of_the_forward(heads):
    fus, tc, te = _fusion(heads, seed=heads)
    with torch.no_grad(), capture_softmax() as seen:
        fus.fuse(tc, te)
    with torch.no_grad():
        cross = A.cross_attention(fus, tc, te)
    # MultiScaleTransformerEncoder.forward runs cross_attn_l (ENH CLS query, direction 1) first, then cross_attn_s
    assert len(seen) == 2 and cross.shape == (3, 2, heads, 17)
    assert _same(cross[:, 1], seen[0][:, :, 0]) and _same(cross[:, 0], seen[1][:, :, 0])
    assert torch.allclose(cross.sum(-1), torch.ones((), dtype=torch.float64))
    # mutation: key 0 taken from the other branch's CLS row instead of the query's own
    layers = fus.multi_scale_transformers[0].cross_attn_layers[0]
    with torch.no_grad():
        wrong = A.cross_probs(layers[0].fn, layers[0].norm(te))
    assert not _same(wrong, seen[1][:, :, 0])
    # mutation: the directions swapped
    assert not _same(cross[:, 0], seen[0][:, :, 0])


# ------------------------------------------------------------------------------------------------------ rollout
HAND_A1 = [[0.5, 0.5, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]]
HAND_A0 = [[0.0, 0.5, 0.5], [0.0, 0.0, 1.0], [1.0, 0.0, 0.0]]
# e0 (A1 + I)/2 = [3/4, 1/4, 0];  [3/4, 1/4, 0] (A0 + I)/2 = [3/8, 5/16, 5/16]
HAND_OUT = [0.375, 0.3125, 0.3125]


def _hand():
    return torch.tensor([[HAND_A0, HAND_A1]], dtype=torch.float64)  # [B=1, L=2, 3, 3]


def test_rollout_matches_the_hand_worked_example():
    out = A.rollout(_hand())
    assert out.tolist() == [HAND_OUT]
    assert out.sum().item() == 1.0


def _naive(means):
    B, L, S, _ = means.shape
    eye = torch.eye(S, dtype=torch.float64)
    R = eye.expand(B, S, S)
    for l in range(L):
        R = ((means[:, l] + eye) / 2) @ R       # R = A'_l ... A'_0
    return R[:, 0]


def _random_means(B=4, L=12, S=10, H=3, seed=0):
    g = torch.Generator().manual_seed(seed)
    probs = torch.softmax(torch.randn(B, L, H, S, S, generator=g, dtype=torch.float64) * 2, -1)
    return probs


def test_rollout_equals_the_full_matrix_product():
    means = _random_means().mean(2)
    out = A.rollout(means)
    assert torch.allclose(out, _naive(means), rtol=0, atol=1e-14)
    assert torch.allclose(out.sum(-1), torch.ones((), dtype=torch.float64), atol=1e-14)


def test_rollout_mutations_fail():
    hand = _hand()
    want = torch.tensor([HAND_OUT], dtype=torch.float64)
    eye = torch.eye(3, dtype=torch.float64)
    # identity not added
    v = torch.tensor([[1.0, 0, 0]], dtype=torch.float64)
    for l in (1, 0):
        v = v @ hand[0, l]
    assert not torch.allclose(v, want)
    # product order reversed: block 0 applied first
    v = torch.tensor([[1.0, 0, 0]], dtype=torch.float64)
    for l in (0, 1):
        v = v @ ((hand[0, l] + eye) / 2)
    assert not torch.allclose(v, want)
    # a transposed map
    assert not torch.allclose(A.rollout(hand.transpose(-1, -2)), want)
    # heads summed instead of averaged
    probs = _random_means(B=2, L=4, S=6, H=3, seed=1)
    good = A.rollout(probs.mean(2))
    assert not torch.allclose(A.rollout(probs.sum(2)), good)
    assert torch.allclose(good.sum(-1), torch.ones((), dtype=torch.float64))
