"""Generates tests/golden/*.pt by running the REAL reference modules on seeded inputs.

    MFVIT_REFERENCE=/path/to/Multi-Feature-ViT python oracle/gen_golden.py

Fixtures are kept small (reduced width / tiny ViT) so they can be committed; the restatement in oracle/ is
width-agnostic, so pinning it at width 96 pins the code that the CUDA parity tests use at width 384."""
import os
import sys
from functools import partial
from types import SimpleNamespace

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_loader  # noqa: E402
from oracle.vit_ref import VisionTransformerMoCo  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


class TokenStub(torch.nn.Module):
    """Backbone stand-in: 'images' are already token tensors; forward = head(tokens[:, 0]) like the absent ViT."""

    def __init__(self, dim, nc):
        super().__init__()
        self.head = torch.nn.Linear(dim, nc)

    def features3D(self, x):
        return x

    def forward(self, x):
        return self.head(x[:, 0])


def gen_fusion():
    _, fus_py, _ = ref_loader.load_reference()
    torch.manual_seed(1234)
    dim, B, S, NC = 96, 3, 10, 3
    v_c, v_e = TokenStub(dim, NC), TokenStub(dim, NC)
    model = fus_py.Fus_CrossViT(v_c, v_e, small_dim=dim, large_dim=dim)
    with torch.no_grad():  # make LayerNorm affine / biases non-trivial
        for p in model.parameters():
            p.add_(torch.randn_like(p) * 0.05)
    t_c = torch.randn(B, S, dim, requires_grad=True)
    t_e = torch.randn(B, S, dim, requires_grad=True)
    fused, x_c, x_e = model(v_c, v_e, t_c, t_e)
    target = torch.tensor([0, 2, 1])
    loss = torch.nn.functional.cross_entropy(fused + x_c + x_e, target)
    loss.backward()
    torch.save({
        "dim": dim, "heads": 3, "state_dict": {k: v.clone() for k, v in model.state_dict().items()},
        "head_c": {k: v.clone() for k, v in v_c.state_dict().items()},
        "head_e": {k: v.clone() for k, v in v_e.state_dict().items()},
        "t_c": t_c.detach(), "t_e": t_e.detach(), "target": target,
        "fused": fused.detach(), "x_c": x_c.detach(), "x_e": x_e.detach(), "loss": loss.detach(),
        "d_t_c": t_c.grad, "d_t_e": t_e.grad,
        "grads": {k: p.grad.clone() for k, p in model.named_parameters()},
        "n_params": sum(p.numel() for p in model.parameters()),
    }, os.path.join(OUT, "fusion_ref.pt"))
    # key inventory at the real width (SURVEY 8(b): 22 keys, 1 185 798 parameters)
    full = fus_py.Fus_CrossViT(TokenStub(384, 3), TokenStub(384, 3))
    torch.save({"keys": {k: tuple(v.shape) for k, v in full.state_dict().items()},
                "n_params": sum(p.numel() for p in full.parameters())}, os.path.join(OUT, "fusion_keys.pt"))


def gen_moco():
    _, _, bld_py = ref_loader.load_reference()
    import torch.distributed as dist
    if not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29533")
        dist.init_process_group("gloo", rank=0, world_size=1)
    torch.Tensor.cuda = lambda self, *a, **k: self  # BLD:121,194 hard-code .cuda()
    torch.manual_seed(4321)
    factory = partial(VisionTransformerMoCo, img_size=32, patch_size=16, embed_dim=64, depth=2, num_heads=2)
    dim, mlp_dim, T, B = 32, 48, 0.2, 8
    model = bld_py.MoCo_ViT(factory, SimpleNamespace(arch="vit_tiny"), dim, mlp_dim, T)
    queue0 = model.queue.clone()
    with torch.no_grad():  # make base != momentum so the EMA is non-trivial
        for p in model.base_encoder.parameters():
            p.add_(torch.randn_like(p) * 0.01)
    im_q, im_k = torch.randn(B, 3, 32, 32), torch.randn(B, 3, 32, 32)
    m = 0.99
    pk_before = [p.detach().clone() for p in model.momentum_encoder.parameters()]
    pq = [p.detach().clone() for p in model.base_encoder.parameters()]
    model.train()
    # capture raw predictor outputs through hooks
    raw = []
    h = model.predictor.register_forward_hook(lambda mod, i, o: raw.append(o.detach().clone()))
    idx_rec = []
    orig_unshuffle = model._batch_unshuffle_ddp
    model._batch_unshuffle_ddp = lambda x, idx: (idx_rec.append(idx.clone()), orig_unshuffle(x, idx))[1]
    logits, labels = model(im_q, im_k, m)
    h.remove()
    raw[1] = raw[1][idx_rec[0]]  # keys were computed in shuffled order (BLD:172); store them in sample order
    loss = torch.nn.functional.cross_entropy(logits, labels)
    pk_after = [p.detach().clone() for p in model.momentum_encoder.parameters()]
    torch.save({
        "dim": dim, "T": T, "m": m, "K": model.K, "seed": 4321,
        "queue_checksum": (float(queue0.double().sum()), float(queue0.double().abs().sum())),
        "queue_cols": queue0[:, ::4096].clone(),  # 16 sampled columns
        "q_raw": raw[0], "k_raw": raw[1],
        "logits_head": logits[:, :65].detach().clone(), "logits_sampled": logits[:, 1::4096].detach().clone(),
        "lse": torch.logsumexp(logits.detach(), dim=1), "loss": loss.detach(), "labels": labels,
        "queue_ptr_after": model.queue_ptr.clone(), "enqueued": model.queue[:, :B].clone(),
        "ema_before": pk_before[:6], "ema_q": pq[:6], "ema_after": pk_after[:6],
        "n_base": sum(p.numel() for p in model.base_encoder.parameters()),
    }, os.path.join(OUT, "moco_ref.pt"))
    # parameter inventory at the real width (SURVEY a11/a12)
    from oracle.vit_ref import vit_small
    full = bld_py.MoCo_ViT(partial(vit_small, stop_grad_conv1=True), SimpleNamespace(arch="vit_small"), 256, 4096, 0.2)
    torch.save({"n_base": sum(p.numel() for p in full.base_encoder.parameters()),
                "n_pred": sum(p.numel() for p in full.predictor.parameters()),
                "keys": sorted(full.state_dict().keys())}, os.path.join(OUT, "moco_keys.pt"))


def gen_augment():
    """The reference's own transform lists (image_transform.get_transform_type, image_transform.py:50-84) composed as
    MAIN_CA:524-531 does, run on seeded uint8 images with torch's global RNG seeded per case."""
    import importlib.util

    import numpy as np
    import torchvision.transforms as T
    from PIL import Image
    spec = importlib.util.spec_from_file_location(
        "ref_image_transform", os.path.join(ref_loader.REF_ROOT, "aihc_utils", "image_transform.py"))
    it = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(it)
    rng = np.random.default_rng(99)
    cases = []
    for i, (h, w, crop, rotate, img_type) in enumerate([
            (64, 64, 64, False, "data"), (64, 64, 64, True, "Train_Mix"), (72, 80, 64, True, "data"),
            (80, 72, 48, 5, "Train_Mix"), (64, 64, 48, 30, "CheXpert_Enh"), (96, 96, 64, True, "CheXpert-v1.0-small")]):
        img = rng.integers(0, 256, size=(h, w, 3), dtype=np.uint8)
        # the stored image is already resized: Resize(shorter side) in front of the list returns it unchanged
        args = SimpleNamespace(maintain_ratio=True, img_size=min(h, w), rotate=rotate, crop=crop)
        out = {}
        for training in (True, False):
            tf = T.Compose(it.get_transform_type(args, training=training, img_type=img_type))
            seed = 700 + i
            torch.manual_seed(seed)
            out["train" if training else "eval"] = tf(Image.fromarray(img)).clone()
        cases.append({"img": torch.from_numpy(img), "crop": crop, "rotate": rotate, "img_type": img_type, "seed": seed,
                      "train": out["train"], "eval": out["eval"]})
    torch.save(cases, os.path.join(OUT, "augment_ref.pt"))


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    gen_fusion()
    gen_moco()
    gen_augment()
    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))
