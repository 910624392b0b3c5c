"""Oracle training step: a functional fp32 restatement of train_one_epoch's body.

TEST INFRASTRUCTURE — see ``oracle/__init__.py``.  Mirrors
/root/reference/main_esvit.py:507-590 (lr/wd set, teacher fwd, student fwd, loss,
backward, per-tensor clip, cancel last-layer grads, AdamW, teacher EMA) for one
process; DDP averaging / center all-reduce are the identity at world_size 1 and are
modelled by an optional ``all_reduce`` hook for the gloo tests.
"""
from __future__ import annotations

import math
import time
from typing import Callable, Dict, List, Optional, Tuple

import torch

from . import losses as L
from . import swin as S

Tensor = torch.Tensor


def param_names(sd: Dict[str, Tensor]) -> List[str]:
    """state_dict keys that are nn.Parameters in the reference (buffers excluded:
    relative_position_index is the only buffer of Swin + DINOHead)."""
    return [k for k in sd if not k.endswith("relative_position_index")]


class OracleStep:
    def __init__(self, state_dict: Dict[str, Tensor], spec: S.SwinSpec, ncrops: int, out_dim: int,
                 teacher_temp: float = 0.04, student_temp: float = 0.1, center_momentum: float = 0.9,
                 lr: float = 5e-4, weight_decay: float = 0.04, clip_grad: float = 3.0,
                 freeze_last_layer: int = 1, momentum_teacher: float = 0.996,
                 norm_last_layer: bool = True, device: str = "cpu"):
        self.spec, self.ncrops, self.out_dim = spec, ncrops, out_dim
        self.teacher_temp, self.student_temp, self.center_momentum = teacher_temp, student_temp, center_momentum
        self.clip_grad, self.freeze_last_layer, self.m = clip_grad, freeze_last_layer, momentum_teacher
        self.lr, self.wd = lr, weight_decay
        self.names = param_names(state_dict)
        # teacher.load_state_dict(student.state_dict()) — main_esvit.py:379
        self.student = {k: v.detach().clone().to(device) for k, v in state_dict.items()}
        self.teacher = {k: v.detach().clone().to(device) for k, v in state_dict.items()}
        for k in self.names:
            frozen = norm_last_layer and k.endswith("last_layer.weight_g")
            self.student[k].requires_grad_(not frozen)
        # utils.get_params_groups (utils.py:672-683)
        reg = [self.student[k] for k in self.names if self.student[k].requires_grad
               and not (k.endswith(".bias") or self.student[k].dim() == 1)]
        noreg = [self.student[k] for k in self.names if self.student[k].requires_grad
                 and (k.endswith(".bias") or self.student[k].dim() == 1)]
        self.opt = torch.optim.AdamW([{"params": reg}, {"params": noreg, "weight_decay": 0.0}])
        self.center = torch.zeros(1, out_dim, device=device)
        self.center_grid = torch.zeros(1, out_dim, device=device)
        self.last_indices = None

    def step(self, crops: List[Tensor], epoch: int = 0, all_reduce: Optional[Callable] = None,
             world_size: int = 1, keep_grads: bool = False) -> float:
        for i, g in enumerate(self.opt.param_groups):  # main_esvit.py:507-510
            g["lr"] = self.lr
            if i == 0:
                g["weight_decay"] = self.wd
        with torch.no_grad():
            t_out = S.multicrop_forward(crops[:2], self.teacher, self.spec)
        s_out = S.multicrop_forward(crops, self.student, self.spec)
        if self.spec.use_dense_prediction:
            loss, self.last_indices = L.ddino_loss(s_out, t_out, self.center, self.center_grid, self.ncrops,
                                                   self.teacher_temp, self.student_temp, return_indices=True)
            with torch.no_grad():
                self.center = L.center_update(self.center, t_out[0], self.center_momentum, world_size, all_reduce)
                self.center_grid = L.center_update(self.center_grid, t_out[1], self.center_momentum,
                                                   world_size, all_reduce)
        else:
            loss = L.dino_loss(s_out, t_out, self.center, self.ncrops, self.teacher_temp, self.student_temp)
            with torch.no_grad():
                self.center = L.center_update(self.center, t_out, self.center_momentum, world_size, all_reduce)
        self.opt.zero_grad(set_to_none=True)
        loss.backward()
        params = [self.student[k] for k in self.names]
        if all_reduce is not None:  # DDP gradient AVG
            for p in params:
                if p.grad is not None:
                    all_reduce(p.grad)
                    p.grad.div_(world_size)
        if keep_grads:  # raw (pre-clip) gradients, for the parity tests
            self.grads_step = {k: self.student[k].grad.detach().clone() for k in self.names
                               if self.student[k].grad is not None}
            self.indices_step = self.last_indices
        if self.clip_grad:
            L.clip_gradients([p.grad for p in params], self.clip_grad)
        if epoch < self.freeze_last_layer:  # utils.cancel_gradients_last_layer (utils.py:118-123)
            for k in self.names:
                if "last_layer" in k:
                    self.student[k].grad = None
        self.opt.step()
        L.ema_update([self.teacher[k] for k in self.names], [self.student[k] for k in self.names], self.m)
        return float(loss.detach())


def synthetic_crops(batch: int, n_local: int, seed: int = 1234, global_size: int = 224, local_size: int = 96,
                    device: str = "cpu") -> List[Tensor]:
    """BASELINE.md §2.3: per-rank generator seed 1234+r, standard-normal fp32 crops."""
    g = torch.Generator().manual_seed(seed)
    crops = [torch.randn(batch, 3, global_size, global_size, generator=g) for _ in range(2)]
    crops += [torch.randn(batch, 3, local_size, local_size, generator=g) for _ in range(n_local)]
    return [c.to(device) for c in crops]


def synthetic_state_dict(layout: List[Tuple[str, Tuple[int, ...]]], seed: int) -> Dict[str, Tensor]:
    """Seeded fp32 weights for the (name, shape) layout of a reference state_dict, so that a fixture stores a seed and
    a layout instead of the weights.  Random (not zero / one) biases, LN affine and bias tables exercise every term;
    Linear / conv weights follow the reference's trunc_normal_(std=.02) scale; DINOHead's frozen weight_g is 1
    (models/vision_transformer.py DINOHead); relative_position_index is its closed form."""
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name, shape in layout:
        shape = tuple(shape)
        if name.endswith("relative_position_index"):
            sd[name] = S.rel_pos_index(math.isqrt(shape[0]))
        elif name.endswith("last_layer.weight_g"):
            sd[name] = torch.ones(shape)
        elif name.endswith(".bias"):
            sd[name] = torch.randn(shape, generator=g) * 0.05
        elif len(shape) == 1 and "norm" in name:
            sd[name] = 1 + torch.randn(shape, generator=g) * 0.1
        elif "relative_position_bias_table" in name:
            sd[name] = torch.randn(shape, generator=g) * 0.5
        else:
            sd[name] = torch.randn(shape, generator=g) * 0.02
    return sd


def sample_elements(t: Tensor, n: int = 512, seed: int = 0) -> Tensor:
    """A fixed, seeded choice of n elements of t (all of them, permuted, when t is smaller): what a fixture stores of a
    tensor too large to keep whole, and what a test takes of its own result to compare with it."""
    flat = t.detach().reshape(-1)
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(seed))[:n]
    return flat[idx.to(flat.device)]


def time_steps(stepper: OracleStep, crops: List[Tensor], steps: int, warmup: int) -> float:
    for _ in range(warmup):
        stepper.step(crops)
    t0 = time.perf_counter()
    for _ in range(steps):
        stepper.step(crops)
    return (time.perf_counter() - t0) / max(steps, 1)
