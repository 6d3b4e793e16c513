"""torch.optim.Adam / AdamW mirrors whose state lives next to the flat replica parameter buffers
(train.py:66,84). The step itself is fused into the update kernels (csrc/mlp.cu adam_kernel: the arithmetic of
torch's `_single_tensor_adam`, hyper-parameters kept in double like the Python floats they are).

`lr` and `weight_decay` also take one value per replica ([R] tensor or sequence): replica r then steps with its own values, bit for bit what
a run configured with those floats computes (the replica-batched hyperparameter search of sweep.py)."""
from __future__ import annotations

import ctypes as C
from typing import Iterable, Union

import torch
from torch import Tensor

from . import _lib

Hyper = Union[float, Tensor]


def per_replica(x, device, dtype=torch.float32):
  """None for a Python / numpy scalar (the scalar path), else the values as a contiguous 1-D device tensor of `dtype`. A tensor that already
  has that form is used as is: captured CUDA graphs bake its address in, so the caller keeps it alive and updates it in place."""
  if isinstance(x, (int, float)) or (not isinstance(x, Tensor) and getattr(x, 'ndim', 1) == 0): return None
  t = torch.as_tensor(x)
  return t.to(device=device, dtype=dtype).reshape(-1).contiguous()


class Adam:
  decoupled = False

  def __init__(self, params: Iterable[Tensor], lr: Hyper = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: Hyper = 0.0):
    params = list(params)
    assert len(params) == 1 and params[0].is_cuda, 'expects the single flat parameter tensor returned by module.parameters()'
    self.param = params[0]
    self.lr_r, self.weight_decay_r = per_replica(lr, self.param.device, torch.float64), per_replica(weight_decay, self.param.device, torch.float64)
    if (self.weight_decay_r is not None or weight_decay != 0) and not self.decoupled:
      raise NotImplementedError('coupled (L2) weight decay is not used by the reference (train.py:66)')
    self.lr, self.betas, self.eps, self.weight_decay = lr, betas, eps, weight_decay
    self.replica_floats = 0
    for t in (self.lr_r, self.weight_decay_r):
      if t is None: continue
      assert self.param.numel() % t.numel() == 0, f'{t.numel()} per-replica values do not divide the {self.param.numel()} parameters'
      assert self.replica_floats in (0, self.param.numel() // t.numel()), 'lr and weight_decay have different replica counts'
      self.replica_floats = self.param.numel() // t.numel()
    self.exp_avg, self.exp_avg_sq = torch.zeros_like(self.param), torch.zeros_like(self.param)
    self.step_count = torch.zeros(1, dtype=torch.int64, device=self.param.device)

  def c_struct(self) -> _lib.Adam:
    a = _lib.Adam()
    a.m, a.v, a.step = self.exp_avg.data_ptr(), self.exp_avg_sq.data_ptr(), self.step_count.data_ptr()
    scalar = lambda x, t: 0.0 if t is not None else x  # an array replaces the scalar in every kernel
    a.lr, a.beta1, a.beta2, a.eps, a.weight_decay = scalar(self.lr, self.lr_r), self.betas[0], self.betas[1], self.eps, scalar(self.weight_decay, self.weight_decay_r)
    a.lr_r, a.weight_decay_r, a.replica_floats = _lib.ptr(self.lr_r), _lib.ptr(self.weight_decay_r), self.replica_floats
    return a

  def zero_grad(self, set_to_none: bool = True):
    pass  # gradients never persist between fused updates (training.py:29,40,47 zero them every call)

  def step_with(self, grads: Tensor):
    """One optimiser step from an explicit flat gradient (tests / custom losses)."""
    a = self.c_struct()
    _lib.check(_lib.lib().il_adam_step(_lib.handle(), self.param.data_ptr(), grads.contiguous().data_ptr(), C.byref(a), self.param.numel(), _lib.stream()))

  def state_dict(self):
    return dict(exp_avg=self.exp_avg.clone(), exp_avg_sq=self.exp_avg_sq.clone(), step=int(self.step_count.item()))


class AdamW(Adam):
  decoupled = True

  def __init__(self, params, lr: Hyper = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: Hyper = 1e-2):
    super().__init__(params, lr, betas, eps, weight_decay)
