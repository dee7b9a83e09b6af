"""The reference's OWN training loop executed over the drop-in (VERDICT r1 item 9, SURVEY 8(b) "scripts run unmodified").

MFVIT_REFERENCE names an unmodified checkout of the reference tree (the repository does not contain one; without it
these tests skip).  tools/overlay.py lays dropin/ over a copy of its moco_pretraining/moco/
directory exactly as INTEGRATION.md section 2 tells a maintainer to; the MAIN_CA script is then imported AS A MODULE -
every one of its imports (`vits_returnftrs`, `model.crossvit_..._sum`, `moco.loader`, `training_tools`, `aihc_utils`,
`config`) resolving inside that deployed tree - and its `train()` (MAIN_CA:793-926) is called twice with the same
synthetic loaders: once over the oracle modules (plain PyTorch fp32) and once over the drop-in (libmfvit.so kernels).
"""
import importlib.util
import os
import sys
import types

import pytest
import torch
import torch.nn as nn

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import e2e_common as E  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REFERENCE = os.environ.get("MFVIT_REFERENCE", "")
needs_reference = pytest.mark.skipif(not (REFERENCE and os.path.isdir(REFERENCE)),
                                     reason="set MFVIT_REFERENCE to a checkout of endiqq/Multi-Feature-ViT")
MAIN_CA = ("main_vit_covid_test_val_single_img_type_5draws_rev_v2loss_v3structure_crossvit_2vits_2additionaloutputs_"
           "trainval_sum.py")


MAIN_LPFT = "main_vit_covid_test_val_single_img_type_5draws_rev_v2loss_v3structure_vitsmall.py"


def _import_reference_script(tmp_path, script=MAIN_CA):
    sys.path.insert(0, os.path.join(ROOT, "multi-feature-vit_b200", "tools"))
    import overlay
    import_root = overlay.make_overlay(REFERENCE, str(tmp_path / "deploy"))
    for n in ("matplotlib", "matplotlib.pyplot"):  # imported by the script, never used by train(); absent in this image
        sys.modules.setdefault(n, types.ModuleType(n))
    # the deployed tree must win over the in-repo dropin/ directory for every module the script imports
    saved_path, saved_mods = list(sys.path), dict(sys.modules)
    for name in list(sys.modules):
        if name.split(".")[0] in ("vits", "vits_returnftrs", "model", "moco", "_path"):
            del sys.modules[name]
    sys.path.insert(0, import_root)
    try:
        spec = importlib.util.spec_from_file_location("reference_" + script[:-3], os.path.join(str(tmp_path / "deploy"), script))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        assert os.path.realpath(mod.vits.__file__).startswith(os.path.realpath(import_root))
        if hasattr(mod, "Fus_CrossViT"):
            assert os.path.realpath(mod.Fus_CrossViT.__init__.__code__.co_filename).startswith(os.path.realpath(import_root))
        return mod
    finally:
        sys.path[:] = saved_path
        for name in list(sys.modules):
            if name.split(".")[0] in ("vits", "vits_returnftrs", "model", "moco", "_path") and name not in saved_mods:
                sys.modules.pop(name)
        sys.modules.update({k: v for k, v in saved_mods.items()
                            if k.split(".")[0] in ("vits", "vits_returnftrs", "model", "moco", "_path")})


class _Writer:
    def __init__(self):
        self.rows = []

    def add_scalar(self, tag, value, step):
        self.rows.append((tag, float(value), step))


def _loaders(n_batches, B):
    """What MAIN_CA:573-578,664-669 hand to train(): per phase, a loader of ((view1, view2), target) per image type."""
    cxr, enh = {}, {}
    for pi, phase in enumerate(("train", "val")):
        cxr[phase], enh[phase] = [], []
        for i in range(n_batches):
            c, e, t = E.synthetic_pair(B, 224, rank=10 * pi + i)
            cxr[phase].append(((c, c), t.int()))  # the script casts with target.long() (MAIN_CA:859)
            enh[phase].append(((e, e), t.int()))
    return cxr, enh


@pytest.mark.gpu
@needs_reference
def test_reference_train_function_runs_unmodified_over_the_dropin(tmp_path):
    ref_main = _import_reference_script(tmp_path)
    torch.backends.cuda.matmul.allow_tf32 = False
    n_batches, B = 2, 8
    results = {}
    for which in ("oracle", "dropin"):
        (fus, cxr, enh), _ = E.build_mfvit_pair(seed=31)
        if which == "dropin":  # built the way the deployed script builds them (MAIN_CA:289-316,393), same weights
            mine = []
            for r in (cxr, enh):
                v = ref_main.vits.__dict__["vit_small"]()
                v.head = nn.Linear(v.head.in_features, 3)
                v.load_state_dict(r.state_dict(), strict=True)
                mine.append(v.cuda())
            f = ref_main.Fus_CrossViT(mine[0], mine[1])
            f.load_state_dict(fus.state_dict(), strict=True)
            fus, cxr, enh = f.cuda(), mine[0], mine[1]
            for obj in (fus, cxr):  # really the deployed tree's classes, not the in-repo dropin/ directory
                assert str(tmp_path / "deploy") in type(obj).__init__.__code__.co_filename
        optimizer = torch.optim.SGD(fus.parameters(), 0.01, momentum=0.9, weight_decay=0.0)  # MAIN_CA:435-449
        args = types.SimpleNamespace(semi_supervised=True)
        loaders, loaders_enh = _loaders(n_batches, B)
        num_imgs = {"train": n_batches * B, "val": n_batches * B}
        writer = _Writer()
        out = ref_main.train(loaders, loaders_enh, fus, cxr, enh, nn.CrossEntropyLoss().cuda(), optimizer, 0, args,
                             num_imgs, writer)
        epoch_loss, epoch_auc, epoch_acc = out[0], out[1], out[2]
        results[which] = (float(epoch_loss), float(epoch_auc), float(epoch_acc), dict((t, v) for t, v, _ in writer.rows),
                          {n: p.detach().clone() for n, p in fus.named_parameters()},
                          cxr.blocks[0].attn.qkv.weight.grad.detach().clone())
    (l0, a0, c0, w0, p0, g0), (l1, a1, c1, w1, p1, g1) = results["oracle"], results["dropin"]
    assert abs(l0 - l1) <= 2e-3, (l0, l1)                       # val loss of the epoch (MAIN_CA:907)
    assert abs(w0["train/loss"] - w1["train/loss"]) <= 2e-3
    assert abs(c0 - c1) <= 1.0 / (n_batches * B) + 1e-9 and abs(a0 - a1) <= 0.05
    for n in p0:                                                # the optimizer stepped the fusion's tensors identically
        assert (p0[n] - p1[n]).abs().max().item() <= 2e-4, n
    assert E.cos(g0, g1) >= 0.999                               # backbones received gradients (never stepped, fact 4)


@pytest.mark.gpu
@needs_reference
@pytest.mark.parametrize("semi_supervised", [False, True])
def test_reference_lpft_train_and_test_functions_over_the_dropin(tmp_path, semi_supervised):
    """MAIN_LPFT's own train() (:647-763) and test() (:765-826), imported from the deployed tree, over the oracle ViT and
    over the drop-in `vits.vit_small` - linear probe (everything but the head frozen, MAIN_LPFT:283-286) and
    --semi-supervised fine-tuning - and the sync-free ViTClassifierTrainer / run_phase on the same batches."""
    from mfvit.data import EpochMetrics
    from mfvit.finetune import ViTClassifierTrainer, run_phase
    ref_main = _import_reference_script(tmp_path, MAIN_LPFT)
    torch.backends.cuda.matmul.allow_tf32 = False
    n_batches, B = 2, 8
    loaders = {ph: [((c, c), t.int()) for c, _, t in (E.synthetic_pair(B, 224, rank=20 * pi + i) for i in range(n_batches))]
               for pi, ph in enumerate(("train", "val"))}
    num_imgs = {"train": n_batches * B, "val": n_batches * B}
    args = types.SimpleNamespace(semi_supervised=semi_supervised)

    def freeze(m):  # MAIN_LPFT:283-286
        if not semi_supervised:
            for name, p in m.named_parameters():
                if name not in ("head.weight", "head.bias"):
                    p.requires_grad = False
        return m

    def make_dropin(ref):
        v = ref_main.vits.__dict__["vit_small"]()                       # MAIN_LPFT:276
        v.head = nn.Linear(v.head.in_features, 3)                       # MAIN_LPFT:288
        v.load_state_dict(ref.state_dict(), strict=True)
        assert str(tmp_path / "deploy") in type(v).__init__.__code__.co_filename
        return freeze(v.cuda())

    results = {}
    for which in ("oracle", "dropin"):
        ref, _ = E.build_vit_pair(seed=33)
        model = freeze(ref) if which == "oracle" else make_dropin(ref)
        params = [p for p in model.parameters() if p.requires_grad]    # MAIN_LPFT:380-392
        assert semi_supervised or len(params) == 2
        opt = torch.optim.SGD(params, 0.05, momentum=0.9, weight_decay=0.0)
        writer = _Writer()
        out = ref_main.train(loaders, model, nn.CrossEntropyLoss().cuda(), opt, 0, args, num_imgs, writer)
        t_loss, t_auc, t_acc = ref_main.test(loaders["val"], model, nn.CrossEntropyLoss().cuda(), opt, 0, num_imgs["val"])
        results[which] = (float(out[0]), dict((t, v) for t, v, _ in writer.rows), float(t_loss), float(t_acc),
                          model.head.weight.detach().clone(), model.blocks[5].mlp.fc1.weight.detach().clone())
    (l0, w0, tl0, ta0, h0, f0), (l1, w1, tl1, ta1, h1, f1) = results["oracle"], results["dropin"]
    assert abs(l0 - l1) <= 2e-3 and abs(w0["train/loss"] - w1["train/loss"]) <= 2e-3 and abs(tl0 - tl1) <= 2e-3
    assert abs(ta0 - ta1) <= 1.0 / (n_batches * B) + 1e-9
    assert (h0 - h1).abs().max().item() <= 2e-4
    assert E.cos(f0, f1) >= 0.999999 and (semi_supervised or torch.equal(f1, E.build_vit_pair(seed=33)[0].blocks[5].mlp.fc1.weight))
    # the sync-free trainer on the same batches: same epoch numbers as the reference loop over the oracle
    ref, _ = E.build_vit_pair(seed=33)
    mine = make_dropin(ref)
    metrics = EpochMetrics(capacity=n_batches * B, num_classes=3, device="cuda")
    tr = ViTClassifierTrainer(mine, lr=0.05, momentum=0.9, metrics=metrics)
    dev = lambda phase: [(c.cuda(), t.cuda()) for (c, _), t in loaders[phase]]  # noqa: E731
    tl, _, _ = run_phase("train", tr, dev("train"), metrics, num_imgs["train"])
    vl, _, vacc = run_phase("val", tr, dev("val"), metrics, num_imgs["val"])
    assert abs(tl - w0["train/loss"]) <= 2e-3 and abs(vl - l0) <= 2e-3 and abs(vacc - ta0) <= 1.0 / (n_batches * B) + 1e-9
    assert (mine.head.weight - h0).abs().max().item() <= 2e-4
