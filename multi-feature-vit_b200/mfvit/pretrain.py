"""Sync-free MoCo-v3-structure / v2-loss pretraining step (MAIN_PRE:500-548, SURVEY 8(a) row a15 and 8(f) row 1).

    model = MoCo_ViT(partial(vits.vit_small, stop_grad_conv1=True), args, dim, mlp_dim, T)      # MAIN_PRE:273-275
    model = torch.nn.SyncBatchNorm.convert_sync_batchnorm(model).cuda()                          # MAIN_PRE:297
    ddp   = torch.nn.parallel.DistributedDataParallel(model, device_ids=[gpu])                   # MAIN_PRE:312
    pre = MoCoPretrainer(ddp, lr=base_lr(args.lr, args.batch_size), weight_decay=args.weight_decay,
                         epochs=args.epochs, warmup_epochs=args.warmup_epochs, moco_m=args.moco_m)
    loss = pre.step(im_q, im_k, epoch + i / iters_per_epoch)       # device tensor; no host sync

What changes against the reference's loop body:
  * the three `loss.item()` host syncs per iteration (MAIN_PRE:537-542) are gone: the running loss accumulates on the
    device (`pre.epoch_loss()` reads it once per epoch);
  * `GradScaler` is not needed: the encoder backward runs with bf16 operands (fp32 range) and the projector / predictor
    run under bf16 autocast, so nothing can underflow the way fp16 gradients do (SURVEY 8(f) row 1);
  * `torch.optim.AdamW` over ~170 tensors becomes the fused flat-buffer AdamW (mfv_adam_step_dev): one launch for the
    encoder's flat master (which also rewrites the 16-bit GEMM shadows, so the next forward skips the cast pass) and one
    for the packed projector + predictor parameters; the learning rate and step count live on the device.  The other
    two optimizers MAIN_PRE:334-345 offers run the same way: optimizer='adam' (torch.optim.Adam, L2 weight decay) and
    optimizer='lars' (moco/optimizer.py, the script's argparse default, MAIN_PRE:131): two launches of mfv_lars_step_dev
    over a table of every trainable tensor - the per-tensor trust ratios are formed on the device;
  * the cosine learning rate with warm-up and the cosine momentum (MAIN_PRE:608-629) come from mfvit.schedules.
DistributedDataParallel keeps doing the gradient all-reduce (bucketed NCCL, overlapped with the backward) and
SyncBatchNorm the global statistics, exactly as MAIN_PRE:297,312 set them up.
"""
import torch
import torch.nn.functional as F

from . import ops, schedules
from ._lib import MfvError
from .engine import engine_for
from .trainer import FlatParams


class MoCoPretrainer:
    def __init__(self, model, lr, weight_decay=0.1, betas=(0.9, 0.999), eps=1e-8, epochs=100, warmup_epochs=0,
                 moco_m=0.99, moco_m_cos=True, cos=True, schedule=(), autocast_dtype=torch.bfloat16, fast_syncbn=True,
                 optimizer="adamw", momentum=0.9, trust_coefficient=0.001):
        """optimizer: "adamw" (torch.optim.AdamW, MAIN_PRE:339; betas, eps), "adam" (torch.optim.Adam with L2 weight
        decay; betas, eps) or "lars" (moco/optimizer.py LARS: momentum, trust_coefficient; matrices get weight decay and
        the trust ratio, vectors momentum only).  weight_decay applies to all three."""
        if optimizer not in ("adamw", "adam", "lars"):
            raise MfvError("optimizer must be 'adamw', 'adam' or 'lars', not %r" % (optimizer,))
        self.optimizer, self.momentum, self.trust_coefficient = optimizer, float(momentum), float(trust_coefficient)
        # nn.SyncBatchNorm (MAIN_PRE:297) -> the lean implementation sharing its tensors (mfvit/syncbn.py): same numbers,
        # one collective per call, a tenth of the host time; fast_syncbn=False keeps the stock modules
        self.swapped_syncbn = 0
        if fast_syncbn:
            from .syncbn import swap_sync_batchnorm
            self.swapped_syncbn = swap_sync_batchnorm(model)
        self.wrapped = model
        self.moco = model.module if hasattr(model, "module") else model
        self.lr, self.wd, self.betas, self.eps = float(lr), float(weight_decay), tuple(betas), float(eps)
        self.epochs, self.warmup_epochs, self.cos, self.schedule = epochs, warmup_epochs, cos, tuple(schedule)
        self.moco_m, self.moco_m_cos = moco_m, moco_m_cos
        self.autocast_dtype = autocast_dtype
        self.engine = engine_for(self.moco.base_encoder)
        self._ready = False
        self._gather = False
        self.steps = 0

    # -- lazily bind to the device of the first batch
    def _prepare(self, device):
        if self._ready:
            return
        eng, moco = self.engine, self.moco
        if not eng.is_adopted() or eng.device != device:
            eng.adopt(device)
        enc_ids = {id(p) for p in eng.params_flat()}
        # everything the optimizer owns besides the encoder's flat buffer: projector (base_encoder.head) + predictor
        rest = [p for p in moco.parameters() if p.requires_grad and id(p) not in enc_ids]
        self._small = FlatParams(rest, device)
        for p, gv in zip(rest, self._small.gviews):
            p.grad = gv  # autograd (and DDP's bucket copy-back) accumulate in place into the packed gradient buffer
        z = torch.zeros_like
        if self.optimizer == "lars":
            self._mu_e, self._mu_s = z(eng.master), z(self._small.master)
            self._lars_tables = {}
            self._lars_ws = self.lars_q = None
        else:
            self._m1_e, self._m2_e = z(eng.master), z(eng.master)
            self._m1_s, self._m2_s = z(self._small.master), z(self._small.master)
        self._lr_dev = torch.full((1,), self.lr, device=device, dtype=torch.float32)
        self._step_dev = torch.zeros(1, device=device, dtype=torch.int64)
        self._loss_sum = torch.zeros(1, device=device, dtype=torch.float64)
        self._n_seen = 0
        # contiguous trainable runs of the encoder layout (pos_embed is a fixed table; stop_grad_conv1 freezes the conv)
        lay = eng.layout
        runs, run = [], None
        for (name, shape, off), (_, p) in zip(lay.entries, eng._params[0]):
            if p.requires_grad:
                if run is not None and run[1] >= off - 8:
                    run[1] = off + p.numel()
                else:
                    if run is not None:
                        runs.append(run)
                    run = [off, off + p.numel()]
            elif run is not None:
                runs.append(run)
                run = None
        if run is not None:
            runs.append(run)
        self._runs = [(lo, min((hi + 3) // 4 * 4, lay.P)) for lo, hi in runs]
        self._shadow_complete = False
        self._ready = True

    def set_lr(self, lr):
        self._lr_dev.fill_(float(lr))

    def lr_at(self, epoch):
        return schedules.pretrain_lr(epoch, self.lr, self.epochs, self.warmup_epochs, self.cos, self.schedule)

    def momentum_at(self, epoch):
        return schedules.moco_momentum(epoch, self.epochs, self.moco_m) if self.moco_m_cos else self.moco_m

    def step(self, im_q, im_k, epoch):
        """One iteration of MAIN_PRE:510-548 at fractional epoch `epoch` (= epoch + i / iters_per_epoch)."""
        device = im_q.device
        if device.type != "cuda":
            raise MfvError("MoCoPretrainer runs only on CUDA sm_100a devices (no CPU fallback)")
        self._prepare(device)
        eng = self.engine
        self.set_lr(self.lr_at(epoch))                                  # MAIN_PRE:512-520
        m = self.momentum_at(epoch)                                     # MAIN_PRE:523-524
        ops.fill_(self._small.grad, 0.0)                                # optimizer.zero_grad() for the packed tensors
        for _, p in eng._params[0]:
            p.grad = None                                               # the encoder gradient buffer is re-zeroed by its backward
        with torch.autocast("cuda", dtype=self.autocast_dtype):         # MAIN_PRE:533 (fp16 + GradScaler there)
            logits, labels = self.wrapped(im_q, im_k, m)
            loss = F.cross_entropy(logits.float(), labels)              # MAIN_PRE:535
        loss.backward()                                                 # DDP all-reduces bucket by bucket
        grad = self._flat_encoder_grad()
        lars = self.optimizer == "lars"
        decoupled = self.optimizer == "adamw"
        if lars:                                                        # MAIN_PRE:547: LARS, encoder + projector + predictor
            table, n_tensors, n_chunks = self._lars_table(grad)
            ops.lars_step_dev_(table, n_tensors, n_chunks, self._lars_ws, self._lr_dev, self.momentum, self.wd,
                               self.trust_coefficient, q_out=self.lars_q)
        else:
            self._step_dev.add_(1)
            for lo, hi in self._runs:                                   # MAIN_PRE:547: AdamW, fused over the flat buffers
                sl = slice(lo, hi)
                ops.adam_step_dev_(eng.master[0, sl], grad[0, sl], self._m1_e[0, sl], self._m2_e[0, sl],
                                   eng.shadow[0, sl], self._lr_dev, self.betas, self.eps, self.wd, decoupled,
                                   self._step_dev, shadow16=eng.shadow16[0, sl] if eng.fwd_f16 else None)
        if not self._shadow_complete:
            eng.cast_shadow()
            self._shadow_complete = True
        eng.mark_shadow_fresh()
        sm = self._small
        if not lars:
            ops.adam_step_dev_(sm.master, sm.grad, self._m1_s, self._m2_s, None, self._lr_dev, self.betas, self.eps,
                               self.wd, decoupled, self._step_dev)
        self._loss_sum += loss.detach().double() * im_q.shape[0]        # MAIN_PRE:537 without the .item()
        self._n_seen += im_q.shape[0]
        self.steps += 1
        return loss.detach()

    def _lars_table(self, grad):
        """The LARS tensor table for this gradient buffer (the engine alternates between two) and shadow format: one
        record per trainable tensor of the encoder layout - frozen tensors (pos_embed, the conv under stop_grad_conv1)
        and the alignment gaps between tensors are never touched - then one per projector / predictor tensor.  Built
        once per buffer; self.lars_params lists the Parameters in table order, self.lars_q their trust ratios of the
        last step (1 for vectors)."""
        eng = self.engine
        key = (grad.data_ptr(), eng.fwd_f16)
        tab = self._lars_tables.get(key)
        if tab is not None:
            return tab
        lay, sm = eng.layout, self._small
        recs, params = [], []
        for (name, shape, off), (_, p) in zip(lay.entries, eng._params[0]):
            if p.requires_grad:
                sl = slice(off, off + p.numel())
                recs.append((eng.master[0, sl], grad[0, sl], self._mu_e[0, sl], eng.shadow[0, sl],
                             eng.shadow16[0, sl] if eng.fwd_f16 else None, len(shape) > 1))
                params.append(p)
        base = sm.master.data_ptr()
        for p, v, gv in zip(sm.params, sm.views, sm.gviews):
            off = (v.data_ptr() - base) // 4
            recs.append((v.view(-1), gv.view(-1), self._mu_s[off:off + v.numel()], None, None, v.dim() > 1))
            params.append(p)
        tab = ops.make_lars_table(recs, grad.device)
        if self._lars_ws is None:
            self._lars_ws = ops.lars_workspace(tab[2], grad.device)
            self.lars_q = torch.ones(tab[1], device=grad.device, dtype=torch.float32)
        if len(self._lars_tables) >= 4:  # gradient buffers replaced over time: keep the table cache small
            self._lars_tables.clear()
        self._lars_tables[key] = tab
        self.lars_params = params
        return tab

    def _flat_encoder_grad(self):
        """The engine's flat gradient buffer of this backward.  autograd normally adopts the views the encoder backward
        returns as the .grad tensors (so DDP's averaged result lands in the flat buffer by itself); if some build of
        torch copies them instead, the averaged .grad tensors are gathered back - correct either way."""
        eng = self.engine
        grad = eng.grads[eng.grad_idx]
        lay, base = eng.layout, grad.data_ptr()
        if self.steps < 2 or self._gather:
            self._gather = any(p.requires_grad and (p.grad is None or p.grad.data_ptr() != base + 4 * lay.offset[n])
                               for n, p in eng._params[0])
        if self._gather:
            for n, p in eng._params[0]:
                if p.requires_grad and p.grad is not None:
                    off = lay.offset[n]
                    grad[0, off:off + p.numel()].view(p.shape).copy_(p.grad)
        return grad

    def epoch_loss(self, reset=True):
        """running_loss / num_imgs of MAIN_PRE:551 - the one host read of the epoch."""
        out = float(self._loss_sum) / max(self._n_seen, 1)
        if reset:
            self._loss_sum.zero_()
            self._n_seen = 0
        return out
