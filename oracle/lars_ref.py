"""Restatement of the MoCo-v3 LARS optimizer (moco/optimizer.py:10-43, built at MAIN_PRE:334-345), pure PyTorch.

For each parameter p with a gradient (lr, weight_decay, momentum, trust_coefficient eta):
    dp = p.grad
    if p.ndim > 1:                     # matrices only: no decay and no trust ratio for biases / norm weights
        dp = dp + weight_decay * p
        q = eta * ||p|| / ||dp||  if ||p|| > 0 and ||dp|| > 0  else 1
        dp = dp * q
    mu = momentum * mu + dp            # mu starts at zero
    p  = p - lr * mu
Works in the dtype of the tensors it is given (fp32 as the reference runs it, fp64 as the tests' reference) on any
device.  Parameters without a gradient (frozen ones) are skipped entirely."""
import torch


@torch.no_grad()
def lars_update_(p, grad, mu, lr, weight_decay, momentum=0.9, trust_coefficient=0.001):
    """One LARS update of one tensor, in place on p and mu.  Returns the trust ratio q (a 0-dim tensor; 1 for ndim <= 1)."""
    dp = grad
    q = torch.ones((), dtype=p.dtype, device=p.device)
    if p.ndim > 1:
        dp = dp.add(p, alpha=weight_decay)
        param_norm = torch.norm(p)
        update_norm = torch.norm(dp)
        one = torch.ones_like(param_norm)
        q = torch.where(param_norm > 0.,
                        torch.where(update_norm > 0, (trust_coefficient * param_norm / update_norm), one), one)
        dp = dp.mul(q)
    mu.mul_(momentum).add_(dp)
    p.add_(mu, alpha=-lr)
    return q


class LARS(torch.optim.Optimizer):
    """LARS without rate scaling or weight decay for parameters with ndim <= 1 (moco/optimizer.py:10-43).  The trust
    ratio of the last step is kept in state[p]["q"] for the tests."""

    def __init__(self, params, lr=0, weight_decay=0, momentum=0.9, trust_coefficient=0.001):
        defaults = dict(lr=lr, weight_decay=weight_decay, momentum=momentum, trust_coefficient=trust_coefficient)
        super().__init__(params, defaults)

    @torch.no_grad()
    def step(self, closure=None):
        for g in self.param_groups:
            for p in g["params"]:
                if p.grad is None:
                    continue
                state = self.state[p]
                if "mu" not in state:
                    state["mu"] = torch.zeros_like(p)
                state["q"] = lars_update_(p, p.grad, state["mu"], g["lr"], g["weight_decay"], g["momentum"],
                                          g["trust_coefficient"])
