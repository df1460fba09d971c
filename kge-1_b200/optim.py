"""Optimizers with torch.optim semantics (kge/util/optimizer.py:10-17 -> getattr(torch.optim, name)) whose
parameter updates run in the kgeb200 kernels.  They are torch.optim.Optimizer subclasses so that the
reference's zero_grad / step / state_dict / param_groups / lr-scheduler uses (train.py:267,278,314,375,388;
optimizer.py:36-38) keep working; state keys follow torch ("sum"/"step", "exp_avg"/"exp_avg_sq")."""
from __future__ import annotations

import torch

from . import lib


def adagrad_clr(lr: float, lr_decay: float, step: float) -> float:
    """Effective learning rate of Adagrad step `step` (1-based, the value of state["step"] after its increment), as
    torch.optim.Adagrad computes it: lr / (1 + (step - 1) * lr_decay).  Adagrad.step and the captured steps of
    trainer.py share this one formula."""
    return lr / (1 + (step - 1) * lr_decay)


def group_of(optimizer: torch.optim.Optimizer, param: torch.Tensor) -> dict:
    """The parameter group of `optimizer` that holds `param` (by identity; ValueError if none does)."""
    for group in optimizer.param_groups:
        if any(p is param for p in group["params"]):
            return group
    raise ValueError("the tensor is not a parameter of any group of the optimizer")


class Adagrad(torch.optim.Optimizer):
    """torch.optim.Adagrad: g += wd*w; sum += g*g; w -= lr/(1+(step-1)*lr_decay) * g / (sqrt(sum) + eps).
    Dense gradients update every element; sparse (COO) gradients update the touched rows only."""

    def __init__(self, params, lr=1e-2, lr_decay=0.0, weight_decay=0.0, initial_accumulator_value=0.0, eps=1e-10):
        defaults = dict(lr=lr, lr_decay=lr_decay, weight_decay=weight_decay,
                        initial_accumulator_value=initial_accumulator_value, eps=eps)
        super().__init__(params, defaults)
        for group in self.param_groups:
            for p in group["params"]:
                st = self.state[p]
                st["step"] = torch.tensor(0.0)
                st["sum"] = torch.full_like(p, initial_accumulator_value, memory_format=torch.preserve_format)

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        for group in self.param_groups:
            for p in group["params"]:
                if p.grad is None:
                    continue
                st = self.state[p]
                st["step"] += 1
                clr = adagrad_clr(group["lr"], group["lr_decay"], st["step"].item())
                g = p.grad
                if g.is_sparse:
                    if group["weight_decay"] != 0:
                        raise RuntimeError("weight_decay option is not compatible with sparse gradients")
                    g = g.coalesce()
                    ids, rows = g.indices()[0].contiguous(), g.values().contiguous()
                    cnt = torch.tensor([ids.numel()], dtype=torch.int64, device=p.device)
                    lib.call("kgeb_adagrad_rows", lib.f32(p.data, "param"), lib.f32(st["sum"], "state"), ids.data_ptr(),
                             lib.f32(rows, "grad rows"), cnt.data_ptr(), ids.numel(), p.shape[1], clr, group["eps"],
                             lib.stream_ptr(p))
                else:
                    lib.call("kgeb_adagrad_dense", lib.f32(p.data, "param"), lib.f32(st["sum"], "state"),
                             lib.f32(g.contiguous(), "grad"), None, p.numel(), clr, group["eps"],
                             group["weight_decay"], None, lib.stream_ptr(p))
                torch.autograd.graph.increment_version(p)  # the kernel wrote through the raw pointer
        return loss


class Adam(torch.optim.Optimizer):
    """torch.optim.Adam (amsgrad=False, dense gradients)."""

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0):
        super().__init__(params, dict(lr=lr, betas=betas, eps=eps, weight_decay=weight_decay))

    @torch.no_grad()
    def step(self, closure=None):
        loss = closure() if closure is not None else None
        for group in self.param_groups:
            b1, b2 = group["betas"]
            for p in group["params"]:
                if p.grad is None:
                    continue
                if p.grad.is_sparse:
                    raise RuntimeError("Adam does not support sparse gradients, please consider SparseAdam instead")
                st = self.state[p]
                if len(st) == 0:
                    st["step"] = torch.tensor(0.0)
                    st["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                    st["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
                st["step"] += 1
                t = st["step"].item()
                lib.call("kgeb_adam_dense", lib.f32(p.data, "param"), lib.f32(st["exp_avg"]), lib.f32(st["exp_avg_sq"]),
                         lib.f32(p.grad.contiguous(), "grad"), p.numel(), group["lr"], b1, b2, group["eps"],
                         group["weight_decay"], 1 - b1 ** t, 1 - b2 ** t, lib.stream_ptr(p))
                torch.autograd.graph.increment_version(p)
        return loss


def create(name: str, params, **kw) -> torch.optim.Optimizer:
    """KgeOptimizer.create (optimizer.py:10-17): kernels for Adagrad / Adam, ValueError otherwise."""
    if name == "Adagrad":
        return Adagrad(params, **kw)
    if name == "Adam":
        return Adam(params, **kw)
    raise ValueError(f"train.optimizer={name}: built optimizers are Adagrad and Adam")
