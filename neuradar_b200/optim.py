"""Fused Adam / AdamW for the hot path's parameters (SURVEY.md 8f next-2).

The reference trains hash grids with `torch.optim.Adam(lr=1e-2, eps=1e-15)` and the field MLPs with
`torch.optim.AdamW(lr=1e-2, eps=1e-15, weight_decay=1e-7)` (nerfstudio/configs/method_configs.py:393-400), built by
`OptimizerConfig.setup` as `_target(params, lr=..., eps=..., weight_decay=...)` (engine/optimizers.py:47-52) and
stepped through `GradScaler.step` (engine/optimizers.py:159-165).  `FusedAdam` / `FusedAdamW` take the same
constructor arguments, so they drop in as `_target`; each parameter group lives in one flat fp32 buffer (parameters,
gradients and both moments) and a step is ONE kernel per group (csrc/optimizer.cu), with the GradScaler division, the
data-parallel average and zero_grad folded in.  No CPU path.
"""
from __future__ import annotations

from typing import Dict, Iterable, List, Optional

import torch
from torch import Tensor

from . import _lib
from ._lib import AdamCfg, ptr, stream_ptr
from .dist import GradArena, padded_numel

import ctypes as C


class _FlatGroup:
    """Parameters of one group re-homed into one flat buffer `p`, with Adam's moments `m` and `v` at the same offsets.
    The gradients are a GradArena over the same parameters in the same order: `g` is its flat buffer."""

    def __init__(self, params: List[torch.nn.Parameter], direct_scatter: bool = False, early=None):
        if not all(p.is_cuda for p in params):
            raise ValueError("FusedAdam expects fp32 CUDA parameters on one device (there is no CPU path)")
        # p before g: their placement shows in the field backward's gradient flush (B200, config 2 with the optimizer:
        # nrb_field_fused_bwd 0.84 ms with g allocated first, 0.82 ms this way)
        self.numel = sum(padded_numel(p.numel()) for p in params)
        self.p = torch.zeros((self.numel,), device=params[0].device, dtype=torch.float32)
        self.arena = GradArena(params, direct_scatter=direct_scatter, early=early)
        self.params, self.offsets, self.g = self.arena.params, self.arena.offsets, self.arena.flat
        self.m = torch.zeros_like(self.p)
        self.v = torch.ones_like(self.p)  # padding lanes keep v = 1 so that eps = 0 cannot make them 0 / 0
        self.skipped = torch.zeros((1,), device=self.g.device, dtype=torch.float32)  # steps GradScaler skipped (found_inf)
        for p, off in zip(self.params, self.offsets):
            self.v[off : off + p.numel()].zero_()
            view = self.p[off : off + p.numel()].view_as(p)
            view.copy_(p.data)
            p.data = view


class FusedAdam(torch.optim.Optimizer):
    """torch.optim.Adam(params, lr, betas, eps, weight_decay) semantics, one CUDA kernel per parameter group."""

    _decoupled = False
    _step_supports_amp_scaling = True  # GradScaler hands us grad_scale / found_inf instead of unscaling itself

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                 direct_scatter: bool = False, early=None):
        if lr < 0 or eps < 0 or not 0 <= betas[0] < 1 or not 0 <= betas[1] < 1 or weight_decay < 0:
            raise ValueError("invalid Adam hyper-parameters")
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay))
        self._flat: List[_FlatGroup] = []
        for group in self.param_groups:
            ps = [p for p in group["params"] if p.requires_grad]
            self._flat.append(_FlatGroup(ps, direct_scatter, early))
            group["step"] = 0
        if any(f.arena.peer is None for f in self._flat):  # all groups take one route, so one multiplier serves them all
            for f in self._flat:
                if f.arena.peer is not None:
                    f.arena.reducer.use_nccl()
        # GradScaler.step sets (and deletes) self.grad_scale / self.found_inf around step(); they must not pre-exist

    # ---- the flat views (data parallelism reduces `flat_grads()` with one collective per group)
    def flat_grads(self) -> List[Tensor]:
        return [f.g for f in self._flat]

    def flat_params(self) -> List[Tensor]:
        return [f.p for f in self._flat]

    def zero_grad(self, set_to_none: bool = False) -> None:  # gradients stay views of the flat buffer
        for f in self._flat:
            f.arena.zero()

    def all_reduce_grads(self, group=None) -> float:
        """Sum gradients over the ranks of the default process group; returns the multiplier for step(grad_mult=...):
        1 / world_size after NCCL, 1 after the peer-memory kernel (which averages in place)."""
        mults = {f.arena.reduce(group) for f in self._flat}  # (the `early` gradients may already be in flight)
        assert len(mults) == 1, f"parameter groups reduced by different routes: multipliers {mults}"
        return mults.pop()

    def check_finite(self, found_inf: Optional[Tensor] = None) -> Tensor:
        """Device flag (1.0 if any gradient is inf / nan), like GradScaler's per-optimizer found_inf."""
        dev = self._flat[0].p.device
        flag = found_inf if found_inf is not None else torch.zeros((1,), device=dev, dtype=torch.float32)
        for f in self._flat:
            _lib.call("nrb_grad_check", ptr(f.g), f.numel, ptr(flag), stream_ptr())
        return flag

    @torch.no_grad()
    def step(self, closure=None, grad_mult: float = 1.0, zero_grad: bool = False):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        scale, found = getattr(self, "grad_scale", None), getattr(self, "found_inf", None)
        for group, f in zip(self.param_groups, self._flat):
            for p, off in zip(f.params, f.offsets):
                if p.data_ptr() != f.p.data_ptr() + 4 * off:  # model.to() / .float() / p.data = ... detached it
                    view = f.p[off : off + p.numel()].view_as(p)
                    view.copy_(p.data)
                    p.data = view
            f.arena.relink()  # someone replaced .grad (e.g. zero_grad(set_to_none=True))
            group["step"] += 1
            cfg = AdamCfg(float(group["lr"]), float(group["betas"][0]), float(group["betas"][1]), float(group["eps"]),
                          float(group["weight_decay"]), int(self._decoupled), int(group["step"]), float(grad_mult),
                          int(zero_grad))
            _lib.call("nrb_adam_step", ptr(f.p), ptr(f.g), ptr(f.m), ptr(f.v), f.numel, C.byref(cfg),
                      ptr(scale.float()) if scale is not None else None, ptr(found.float()) if found is not None else None,
                      ptr(f.skipped) if found is not None else None, stream_ptr())
        return loss

    # ---- torch.optim.Adam-shaped state (checkpoints written by the reference's trainer load into this and back)
    def state_dict(self) -> Dict:
        state, idx = {}, 0
        groups = []
        for group, f in zip(self.param_groups, self._flat):
            ids = []
            where = {id(p): off for p, off in zip(f.params, f.offsets)}
            for p in group["params"]:  # torch numbers EVERY parameter of the group, trainable or not
                off = where.get(id(p))
                if off is not None:
                    n = p.numel()
                    state[idx] = {"step": torch.tensor(float(group["step"])) - f.skipped.cpu()[0],
                                  "exp_avg": f.m[off : off + n].view_as(p).clone(),
                                  "exp_avg_sq": f.v[off : off + n].view_as(p).clone()}
                ids.append(idx)
                idx += 1
            groups.append({**{k: v for k, v in group.items() if k != "params"}, "params": ids})
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd: Dict) -> None:
        idx = 0
        for group, f, saved in zip(self.param_groups, self._flat, sd["param_groups"]):
            for k, v in saved.items():
                if k != "params":
                    group[k] = v
            where = {id(p): off for p, off in zip(f.params, f.offsets)}
            for p in group["params"]:
                off = where.get(id(p))
                st = sd["state"].get(idx)
                if st is not None and off is not None:
                    n = p.numel()
                    f.m[off : off + n].view_as(p).copy_(st["exp_avg"])
                    f.v[off : off + n].view_as(p).copy_(st["exp_avg_sq"])
                    group["step"] = int(st["step"])
                    f.skipped.zero_()
                idx += 1


class FusedAdamW(FusedAdam):
    """torch.optim.AdamW semantics (decoupled weight decay: p *= 1 - lr * weight_decay before the update)."""

    _decoupled = True

    def __init__(self, params, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2,
                 direct_scatter: bool = False, early=None):
        super().__init__(params, lr=lr, betas=betas, eps=eps, weight_decay=weight_decay, direct_scatter=direct_scatter,
                         early=early)
