"""CPU: the LARS restatement (oracle/lars_ref.py, moco/optimizer.py:10-43) against float64 values worked out by hand for
every branch, and the argument checks of the pretrainer / op that need no GPU."""
import importlib
import math
from functools import partial
from types import SimpleNamespace

import pytest
import torch

from oracle import lars_ref

LR, WD, MOM, ETA = 0.1, 0.5, 0.9, 0.001


def _t(rows):
    return torch.tensor(rows, dtype=torch.float64)


def _step(p, g, mu):
    return lars_ref.lars_update_(p, g, mu, LR, WD, MOM, ETA)


def test_vector_gets_momentum_only():
    p, g, mu = _t([1.0, -2.0]), _t([0.5, 0.25]), torch.zeros(2, dtype=torch.float64)
    q = _step(p, g, mu)
    assert float(q) == 1.0
    assert mu.tolist() == [0.5, 0.25]                                  # no weight decay, no trust ratio
    assert p.tolist() == [1.0 - 0.1 * 0.5, -2.0 - 0.1 * 0.25]


def test_zero_weight_matrix_uses_q_one():
    p, g, mu = torch.zeros(2, 2, dtype=torch.float64), _t([[3.0, 0.0], [0.0, 4.0]]), torch.zeros(2, 2, dtype=torch.float64)
    q = _step(p, g, mu)
    assert float(q) == 1.0                                             # ||p|| = 0
    assert mu.tolist() == [[3.0, 0.0], [0.0, 4.0]]                     # dp = g + 0.5 * 0
    assert p.tolist() == [[-0.1 * 3.0, 0.0], [0.0, -0.1 * 4.0]]


def test_matrix_with_zero_decayed_update_uses_q_one():
    p, g, mu = _t([[2.0, -4.0]]), _t([[-1.0, 2.0]]), torch.zeros(1, 2, dtype=torch.float64)
    q = _step(p, g, mu)                                                # dp = g + 0.5 p = 0 exactly
    assert float(q) == 1.0
    assert mu.tolist() == [[0.0, 0.0]] and p.tolist() == [[2.0, -4.0]]


def test_first_and_second_step_of_a_matrix():
    p, g, mu = _t([[3.0, 4.0]]), _t([[1.5, -2.0]]), torch.zeros(1, 2, dtype=torch.float64)
    # step 1: dp = [1.5 + 1.5, -2 + 2] = [3, 0]; ||p|| = 5, ||dp|| = 3, q = 0.001 * 5 / 3; mu = q dp = [0.005, 0]
    q1 = _step(p, g, mu)
    assert math.isclose(float(q1), 0.001 * 5.0 / 3.0, rel_tol=1e-15)
    assert math.isclose(mu[0, 0].item(), 0.005, rel_tol=1e-14) and mu[0, 1].item() == 0.0
    assert math.isclose(p[0, 0].item(), 3.0 - 0.1 * 0.005, rel_tol=1e-15) and p[0, 1].item() == 4.0
    # step 2: p = [2.9995, 4], dp = [1.5 + 0.5 * 2.9995, 0] = [2.99975, 0]; q dp = [0.001 ||p||, 0];
    # mu = 0.9 * 0.005 + 0.001 * sqrt(2.9995^2 + 16)  (momentum carries the first step)
    q2 = _step(p, g, mu)
    pn = math.sqrt(2.9995 ** 2 + 16.0)
    assert math.isclose(float(q2), 0.001 * pn / 2.99975, rel_tol=1e-13)
    mu_want = 0.9 * 0.005 + 0.001 * pn
    assert math.isclose(mu[0, 0].item(), mu_want, rel_tol=1e-13) and mu[0, 1].item() == 0.0
    assert math.isclose(p[0, 0].item(), 2.9995 - 0.1 * mu_want, rel_tol=1e-14) and p[0, 1].item() == 4.0


def test_cls_token_shape_gets_the_trust_ratio():
    p, g, mu = _t([[[0.0, 3.0, 4.0]]]), _t([[[0.0, 1.0, 0.0]]]), torch.zeros(1, 1, 3, dtype=torch.float64)
    q = _step(p, g, mu)                                                # (1, 1, C): ndim 3 > 1
    dp = [0.0, 1.0 + 1.5, 2.0]
    want_q = 0.001 * 5.0 / math.sqrt(dp[1] ** 2 + dp[2] ** 2)
    assert math.isclose(float(q), want_q, rel_tol=1e-15)
    assert all(math.isclose(a, want_q * b, rel_tol=1e-14, abs_tol=0.0) for a, b in zip(mu.flatten().tolist(), dp))


def test_optimizer_skips_frozen_tensors_and_keeps_state():
    w = torch.nn.Parameter(_t([[3.0, 4.0]]))
    b = torch.nn.Parameter(_t([1.0]))
    frozen = torch.nn.Parameter(_t([[7.0, 8.0]]), requires_grad=False)
    opt = lars_ref.LARS([w, b, frozen], lr=LR, weight_decay=WD, momentum=MOM, trust_coefficient=ETA)
    w.grad, b.grad = _t([[1.5, -2.0]]), _t([2.0])
    opt.step()
    opt.step()
    assert frozen.tolist() == [[7.0, 8.0]] and frozen not in opt.state  # no grad: untouched, no momentum buffer
    assert math.isclose(opt.state[b]["mu"].item(), 0.9 * 2.0 + 2.0, rel_tol=1e-15)
    assert math.isclose(b.item(), 1.0 - 0.1 * 2.0 - 0.1 * 3.8, rel_tol=1e-15)
    pn = math.sqrt(2.9995 ** 2 + 16.0)                                 # same matrix as the two-step test
    assert math.isclose(float(opt.state[w]["q"]), 0.001 * pn / 2.99975, rel_tol=1e-13)


def test_pretrainer_rejects_unknown_optimizer_and_op_rejects_cpu_tensors():
    import vits
    from mfvit import MfvError, ops
    from mfvit.pretrain import MoCoPretrainer
    bm = importlib.import_module("moco.builder_vit_mocov3structure_mocov2loss")
    moco = bm.MoCo_ViT(partial(vits.vit_small, stop_grad_conv1=True), SimpleNamespace(arch="vit_small"), 256, 4096, 0.2)
    with pytest.raises(MfvError, match="'adamw', 'adam' or 'lars'"):
        MoCoPretrainer(moco, lr=1e-3, optimizer="sgd")
    for opt in ("adamw", "adam", "lars"):
        assert MoCoPretrainer(moco, lr=1e-3, optimizer=opt, fast_syncbn=False).optimizer == opt
    x = torch.zeros(8)
    with pytest.raises(MfvError, match="CUDA"):
        ops.make_lars_table([(x, x, x, None, None, False)], torch.device("cpu"))
