"""Host-side mirror of the reference's models.py surface (same names / arguments / behaviour) over the sm_100a
kernels. Every class takes an extra `replicas` axis (default 1 = the reference's shapes).

Cited lines are in the reference's models.py unless noted.
"""
from __future__ import annotations

import copy
import ctypes as C
from math import sqrt
from typing import Dict, List, Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from .memory import ReplayMemory, TransitionBatch
from .net import ReplicaMLP, ReplicaRNG, init_fcnn_params, _null_ctx
from .optim import per_replica


def _cfg_get(cfg, key, default=None):
  if hasattr(cfg, 'get'): return cfg.get(key, default)
  return getattr(cfg, key, default)


def _as_rns(x: Tensor, R: int, width: int, device) -> Tensor:
  """[n, w] (R == 1) or [R, n, w] -> contiguous [R, n, w] on the device."""
  x = torch.as_tensor(x, dtype=torch.float32).to(device)
  if x.dim() == 2:
    assert R == 1, f'expected a [R={R}, n, {width}] tensor'
    x = x.unsqueeze(0)
  assert x.dim() == 3 and x.size(0) == R and x.size(2) == width, f'bad shape {tuple(x.shape)}; expected [{R}, n, {width}]'
  return x.contiguous()


class _RNG:
  """Device noise source (Philox, il_fill_normal / il_fill_uniform) standing in for torch's global RNG draws."""

  def __init__(self, seed: int = 0, device=None):
    self.seed = seed
    self.counter = None
    self.device = device

  def _ctr(self, device):
    if self.counter is None: self.counter = torch.zeros(1, dtype=torch.int64, device=device)
    return self.counter

  def normal(self, shape, device, stream_id: int = 1, out: Optional[Tensor] = None) -> Tensor:
    out = torch.empty(shape, device=device, dtype=torch.float32) if out is None else out
    ctr = self._ctr(device)
    _lib.check(_lib.lib().il_fill_normal(_lib.handle(), out.data_ptr(), out.numel(), self.seed, stream_id, ctr.data_ptr(), _lib.stream()))
    _lib.check(_lib.lib().il_counter_add(_lib.handle(), ctr.data_ptr(), (out.numel() + 3) // 4, _lib.stream()))
    return out

  def uniform(self, shape, device, stream_id: int = 2, out: Optional[Tensor] = None) -> Tensor:
    out = torch.empty(shape, device=device, dtype=torch.float32) if out is None else out
    ctr = self._ctr(device)
    _lib.check(_lib.lib().il_fill_uniform(_lib.handle(), out.data_ptr(), out.numel(), self.seed, stream_id, ctr.data_ptr(), _lib.stream()))
    _lib.check(_lib.lib().il_counter_add(_lib.handle(), ctr.data_ptr(), (out.numel() + 3) // 4, _lib.stream()))
    return out


default_rng = _RNG(0)


def manual_seed(seed: int):
  """Seeds the device noise source used when noise is not injected."""
  default_rng.seed, default_rng.counter = seed, None


class _Module:
  """Minimal nn.Module-like surface (parameters / state_dict / train / eval) over flat replica buffers."""
  training = True

  def train(self, mode: bool = True):
    self.training = mode
    return self

  def eval(self):
    return self.train(False)

  def parameters(self) -> List[Tensor]:
    return [self.mlp.flat]

  def _state_items(self) -> List[Tuple[str, Tensor]]:
    raise NotImplementedError

  def state_dict(self) -> Dict[str, Tensor]:
    """Reference key names (SURVEY §5). R == 1: the reference's shapes; R > 1: a leading replica axis."""
    return {k: (v[0] if v.size(0) == 1 else v).detach().clone() for k, v in self._state_items()}

  def load_state_dict(self, sd: Dict[str, Tensor]):
    for k, v in self._state_items():
      src = torch.as_tensor(sd[k]).to(v.device, torch.float32)
      v.copy_(src.reshape(v.shape) if src.numel() == v.numel() else src.unsqueeze(0).expand_as(v))


class TanhNormalPolicy:
  """What `SoftActor.forward` returns (:90-94): the TransformedDistribution surface the reference uses —
  .sample() / .rsample() / .log_prob(a) / .base_dist.mean — evaluated by the fused actor-head kernel."""

  def __init__(self, actor: 'SoftActor', state: Tensor):
    self.actor, self.state = actor, state
    self._cached_action, self._cached_log_prob = None, None

  class _Base:
    def __init__(self, outer): self.outer = outer

    @property
    def mean(self) -> Tensor:
      o = self.outer
      return o.actor._squeeze(o.actor._run(o.state, want=('mean', ))['mean'])

    @property
    def stddev(self) -> Tensor:
      o = self.outer
      return o.actor._squeeze(o.actor._run(o.state, want=('log_std', ))['log_std'].exp())

  @property
  def base_dist(self): return TanhNormalPolicy._Base(self)

  def sample(self, eps: Optional[Tensor] = None) -> Tensor:
    a = self.actor
    if eps is None: eps = default_rng.normal((a.replicas, self.state.size(1), a.action_size), a.device)
    out = a._run(self.state, eps=eps, want=('action', 'log_prob'))
    self._cached_action, self._cached_log_prob = a._squeeze(out['action']), a._squeeze(out['log_prob'])  # TanhTransform(cache_size=1)
    return self._cached_action

  rsample = sample

  def log_prob(self, action: Tensor) -> Tensor:
    if action is self._cached_action: return self._cached_log_prob
    a = self.actor
    return a._squeeze(a._run(self.state, given=action, want=('log_prob', ))['log_prob'])


class SoftActor(_Module):
  """:84-102. `actor(state)` returns a TanhNormalPolicy; state is [n, S] (R == 1) or [R, n, S]."""

  ENSEMBLE = 5  # :105

  def __init__(self, state_size: int, action_size: int, model_cfg, replicas: int = 1, rng: Optional[ReplicaRNG] = None, device=None):
    # :88 — a policy with dropout is DRIL's "discriminator" (train.py:74); its density / BC update run on the dropout MLP program (csrc/dropout_nets.cu)
    self.input_dropout, self.dropout = float(_cfg_get(model_cfg, 'input_dropout', 0) or 0), float(_cfg_get(model_cfg, 'dropout', 0) or 0)
    self.training, self.q, self._drop_ws, self._drop_rng = True, None, None, None
    self.state_size, self.action_size, self.replicas = state_size, action_size, replicas
    self.log_std_dev_min, self.log_std_dev_max = -20, 2  # :87 (the kernel hard-codes the same clamp)
    dims = [state_size] + [model_cfg.hidden_size] * model_cfg.depth + [2 * action_size]
    self.mlp = ReplicaMLP(dims, model_cfg.activation, replicas, 1, device)
    self.device = self.mlp.device
    for r in range(replicas):
      with (rng.replica(r) if rng is not None else _null_ctx()):
        self.mlp.load_params(r, 0, init_fcnn_params(dims, model_cfg.activation))
    self._ws = None

  def _squeeze(self, t: Tensor) -> Tensor:
    return t[0] if self.replicas == 1 else t

  def _state_items(self):
    v = self.mlp.layer_views()[0]
    base, step = (1 if self.input_dropout > 0 else 0), (3 if self.dropout > 0 else 2)  # nn.Sequential indices: [Dropout], Linear, [Dropout], activation, ... (:51-61)
    return [(f'actor.{base + step * l}.{n}', v[2 * l + i]) for l in range(self.mlp.n_layers) for i, n in enumerate(('weight', 'bias'))]

  def _run(self, state: Tensor, eps: Optional[Tensor] = None, given: Optional[Tensor] = None, want=('action', )) -> Dict[str, Tensor]:
    R, A = self.replicas, self.action_size
    s = _as_rns(state, R, self.state_size, self.device)
    n = s.size(1)
    m = self.mlp.c_struct()
    need = _lib.lib().il_actor_workspace_bytes(C.byref(m), R, n)
    if self._ws is None or self._ws.numel() < need: self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
    out = {k: torch.empty((R, n, A) if k in ('action', 'mean', 'log_std') else (R, n), device=self.device) for k in want}
    eps_t = None if eps is None else _as_rns(eps, R, A, self.device)
    given_t = None if given is None else _as_rns(given, R, A, self.device)
    _lib.check(_lib.lib().il_actor_forward(_lib.handle(), C.byref(m), R, n, s.data_ptr(), s.stride(0), s.stride(1), _lib.ptr(eps_t), _lib.ptr(given_t), _lib.ptr(out.get('action')),
                                           _lib.ptr(out.get('log_prob')), _lib.ptr(out.get('mean')), _lib.ptr(out.get('log_std')), self._ws.data_ptr(), self._ws.numel(),
                                           _lib.stream()))
    return out

  @property
  def has_dropout(self) -> bool: return self.input_dropout > 0 or self.dropout > 0

  def forward(self, state: Tensor) -> TanhNormalPolicy:
    if self.has_dropout and self.training: raise NotImplementedError('sampling from a dropout policy in train mode is not used by the reference (DRIL only evaluates log_prob, models.py:104-120)')
    return TanhNormalPolicy(self, _as_rns(state, self.replicas, self.state_size, self.device))

  __call__ = forward

  # ---- dropout policy (DRIL) ----------------------------------------------------------------------------------------------------
  def draw_masks(self, n: int) -> List[Optional[Tensor]]:
    """[input mask [R, n, S] or None, one [R, n, H] mask per hidden layer or None]: Bernoulli(1 - p) / (1 - p) draws on the device (Philox), the analogue
    of nn.Dropout's draws from torch's global stream."""
    if self._drop_rng is None: self._drop_rng = _RNG(default_rng.seed + 977, self.device)
    rng, R, lib = self._drop_rng, self.replicas, _lib.lib()
    def draw(width, p):
      if p <= 0: return None
      out = torch.empty(R, n, width, device=self.device)
      ctr = rng._ctr(self.device)
      _lib.check(lib.il_fill_dropout_mask(_lib.handle(), out.data_ptr(), out.numel(), p, rng.seed, 31, ctr.data_ptr(), _lib.stream()))
      _lib.check(lib.il_counter_add(_lib.handle(), ctr.data_ptr(), (out.numel() + 3) // 4, _lib.stream()))
      return out
    return [draw(self.state_size, self.input_dropout)] + [draw(self.mlp.dims[l + 1], self.dropout) for l in range(self.mlp.n_layers - 1)]

  def _log_prob_dropout(self, state: Tensor, action: Tensor, repeat: int = 1, masks: Optional[List[Optional[Tensor]]] = None) -> Tensor:
    R, S, A = self.replicas, self.state_size, self.action_size
    s, a = _as_rns(state, R, S, self.device), _as_rns(action, R, A, self.device)
    n = s.size(1) * repeat
    if masks is None: masks = self.draw_masks(n)
    masks = [None if m is None else torch.as_tensor(m, dtype=torch.float32).to(self.device).reshape(R, n, -1).contiguous() for m in masks]
    m = self.mlp.c_struct()
    need = _lib.lib().il_actor_dropout_workspace_bytes(C.byref(m), R, n)
    if self._drop_ws is None or self._drop_ws.numel() < need: self._drop_ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
    out = torch.empty(R, n, device=self.device)
    _lib.check(_lib.lib().il_actor_log_prob_dropout(_lib.handle(), C.byref(m), R, n, repeat, s.data_ptr(), s.stride(0), s.stride(1), a.data_ptr(), _lib.ptr(masks[0]), _lib.mask_array(masks[1:]),
                                                    out.data_ptr(), self._drop_ws.data_ptr(), self._drop_ws.numel(), _lib.stream()))
    return out

  def _get_action_uncertainty(self, state: Tensor, action: Tensor, masks=None) -> Tensor:  # :104-107
    lp = self._log_prob_dropout(state, action, repeat=self.ENSEMBLE, masks=masks)
    R, B = self.replicas, lp.size(1) // self.ENSEMBLE
    var = torch.empty(R, B, device=self.device)
    _lib.check(_lib.lib().il_dril_reward(_lib.handle(), lp.data_ptr(), R, B, self.ENSEMBLE, None, 0, None, 0, 0, var.data_ptr(), _lib.stream()))
    return self._squeeze(var)

  def set_uncertainty_threshold(self, expert_state: Tensor, expert_action: Tensor, quantile_cutoff, masks=None):  # :110-111 (one-off set-up statistic)
    """quantile_cutoff: a float, or one cutoff per replica ([R]; each row's quantile is taken on the host side of the set-up, row by row)."""
    R = self.replicas
    es = torch.as_tensor(expert_state, dtype=torch.float32).to(self.device)
    ea = torch.as_tensor(expert_action, dtype=torch.float32).to(self.device)
    if es.dim() == 2: es, ea = es.unsqueeze(0).expand(R, -1, -1), ea.unsqueeze(0).expand(R, -1, -1)
    var = self._get_action_uncertainty(es, ea, masks=masks).reshape(R, -1)
    if isinstance(quantile_cutoff, (int, float)): self._q = torch.quantile(var, quantile_cutoff, dim=1).contiguous()
    else:
      cut = [float(c) for c in torch.as_tensor(quantile_cutoff).reshape(-1).tolist()]
      assert len(cut) == R, f'{len(cut)} quantile cutoffs for {R} replicas'
      self._q = torch.cat([torch.quantile(var[r:r + 1], cut[r], dim=1) for r in range(R)]).contiguous()
    self.q = float(self._q[0]) if R == 1 else self._q

  def predict_reward(self, state: Tensor, action: Tensor, masks=None, out: Optional[Tensor] = None) -> Tensor:  # :113-120
    lp = self._log_prob_dropout(state, action, repeat=self.ENSEMBLE, masks=masks)
    R, B = self.replicas, lp.size(1) // self.ENSEMBLE
    out = torch.empty(R, B, device=self.device) if out is None else out
    _lib.check(_lib.lib().il_dril_reward(_lib.handle(), lp.data_ptr(), R, B, self.ENSEMBLE, self._q.data_ptr(), 0, out.data_ptr(), out.stride(0), out.stride(1), None, _lib.stream()))
    return self._squeeze(out) if out.dim() == 2 and out.is_contiguous() else out

  def log_prob(self, state: Tensor, action: Tensor, masks=None) -> Tensor:  # :97-99
    if self.has_dropout and (self.training or masks is not None): return self._squeeze(self._log_prob_dropout(state, action, masks=masks))
    return self._squeeze(self._run(state, given=action, want=('log_prob', ))['log_prob'])

  def get_greedy_action(self, state: Tensor) -> Tensor:  # :101-102
    return self._squeeze(self._run(state, want=('action', ))['action'])


class TwinCritic(_Module):
  """:123-141; parameters of critic_1 then critic_2 per replica in one flat buffer (2R nets)."""

  def __init__(self, state_size: int, action_size: int, model_cfg, replicas: int = 1, rng: Optional[ReplicaRNG] = None, device=None):
    self.state_size, self.action_size, self.replicas = state_size, action_size, replicas
    dims = [state_size + action_size] + [model_cfg.hidden_size] * model_cfg.depth + [1]
    self.mlp = ReplicaMLP(dims, model_cfg.activation, replicas, 2, device)
    self.device = self.mlp.device
    for r in range(replicas):
      with (rng.replica(r) if rng is not None else _null_ctx()):
        self.mlp.load_params(r, 0, init_fcnn_params(dims, model_cfg.activation))  # critic_1 (:136)
        self.mlp.load_params(r, 1, init_fcnn_params(dims, model_cfg.activation))  # critic_2 (:137)
    self._ws = None

  def c_struct(self) -> _lib.Mlp:
    return self.mlp.c_struct()

  def _state_items(self):
    out = []
    for t in (0, 1):
      v = self.mlp.layer_views()[t]
      out += [(f'critic_{t + 1}.critic.{2 * l}.{n}', v[2 * l + i]) for l in range(self.mlp.n_layers) for i, n in enumerate(('weight', 'bias'))]
    return out

  def forward(self, state: Tensor, action: Tensor) -> Tuple[Tensor, Tensor]:
    R = self.replicas
    s, a = _as_rns(state, R, self.state_size, self.device), _as_rns(action, R, self.action_size, self.device)
    n = s.size(1)
    m = self.mlp.c_struct()
    need = _lib.lib().il_critic_workspace_bytes(C.byref(m), R, n)
    if self._ws is None or self._ws.numel() < need: self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
    q1, q2 = torch.empty(R, n, device=self.device), torch.empty(R, n, device=self.device)
    _lib.check(_lib.lib().il_critic_forward(_lib.handle(), C.byref(m), R, n, self.state_size, s.data_ptr(), s.stride(0), s.stride(1), a.data_ptr(), a.stride(0), a.stride(1),
                                            q1.data_ptr(), q2.data_ptr(), self._ws.data_ptr(), self._ws.numel(), _lib.stream()))
    return (q1[0], q2[0]) if R == 1 else (q1, q2)

  __call__ = forward


def create_target_network(network):
  """:72-76."""
  target = copy.copy(network)
  target.mlp = copy.copy(network.mlp)
  target.mlp.flat = network.mlp.flat.clone()
  target._ws = None
  return target


def update_target_network(network, target_network, polyak_factor: float):
  """:79-81."""
  t, o = target_network.mlp.flat, network.mlp.flat
  _lib.check(_lib.lib().il_polyak(_lib.handle(), t.data_ptr(), o.data_ptr(), t.numel(), polyak_factor, _lib.stream()))


def make_gail_input(state: Tensor, action: Tensor, next_state: Tensor, terminal: Tensor, actor: SoftActor, reward_shaping: bool, subtract_log_policy: bool) -> Dict[str, Tensor]:
  """:145-149."""
  inp = {'state': state, 'action': action}
  if reward_shaping: inp.update({'next_state': next_state, 'terminal': terminal})
  if subtract_log_policy: inp.update({'log_policy': actor.log_prob(state, action)})
  return inp


def _spectral_norm_init(weight: Tensor) -> Tuple[Tensor, Tensor]:
  """torch parametrizations.spectral_norm construction (_SpectralNorm.__init__): u, v ~ N(0, 1) from the global RNG,
  normalised, then 15 power iterations (sites :58,66,159)."""
  h, w = weight.shape
  nz = lambda x: x / x.norm().clamp_min(1e-12)
  u, v = nz(weight.new_empty(h).normal_(0, 1)), nz(weight.new_empty(w).normal_(0, 1))
  for _ in range(15):
    u = nz(torch.mv(weight, v))
    v = nz(torch.mv(weight.t(), u))
  return u, v


class GAILDiscriminator(_Module):
  """:152-180. Accelerated configuration: the depth-1 relu `g` network of conf/algorithm/GAIL.yaml (no reward
  shaping / log-policy subtraction), with or without spectral norm."""

  def __init__(self, state_size: int, action_size: int, imitation_cfg, discount, replicas: int = 1, rng: Optional[ReplicaRNG] = None, device=None):
    """discount: a float, or one value per replica ([R]) for the reward-shaping term of the general discriminator."""
    model_cfg = imitation_cfg.discriminator
    self.discount, self.state_only = discount, bool(imitation_cfg.state_only)
    self.discount_r = per_replica(discount, torch.device('cuda') if device is None else device)
    self.reward_shaping, self.subtract_log_policy, self.reward_function = bool(model_cfg.reward_shaping), bool(model_cfg.subtract_log_policy), model_cfg.reward_function
    self.state_size, self.action_size, self.replicas = state_size, action_size, replicas
    self.spectral_norm = bool(imitation_cfg.spectral_norm)
    # the default configuration (GAIL.yaml:10-17: one relu hidden layer, no shaping, no log-policy term) runs in the fused one-CTA-per-replica
    # kernel (csrc/gail.cu); every other configuration of models.py:157-175 runs as the replica-batched GEMM program of csrc/gail_general.cu
    self.general = self.reward_shaping or self.subtract_log_policy or model_cfg.depth != 1 or model_cfg.activation != 'relu'
    self._ws = None
    if self.general:
      self._init_general(model_cfg, rng, device)
      return
    d, H = (state_size if self.state_only else state_size + action_size), model_cfg.hidden_size
    dims = [d, H, 1]
    self.mlp = ReplicaMLP(dims, 'relu', replicas, 1, device)
    self.device = self.mlp.device
    self.u = torch.zeros(replicas, H + 1, device=self.device) if self.spectral_norm else None  # layer0 u [H], layer1 u [1]
    self.v = torch.zeros(replicas, d + H, device=self.device) if self.spectral_norm else None  # layer0 v [d], layer1 v [H]
    for r in range(replicas):
      with (rng.replica(r) if rng is not None else _null_ctx()):
        params, us, vs = [], [], []
        for l in range(2):  # _create_fcnn order (:52-59,:62-67): Linear, orthogonal_, zero bias, then spectral_norm
          layer = torch.nn.Linear(dims[l], dims[l + 1])
          torch.nn.init.orthogonal_(layer.weight, gain=torch.nn.init.calculate_gain('relu') if l == 0 else 1)
          torch.nn.init.constant_(layer.bias, 0)
          w = layer.weight.detach()
          if self.spectral_norm:
            u_, v_ = _spectral_norm_init(w)
            us.append(u_)
            vs.append(v_)
          params += [w, layer.bias.detach()]
        self.mlp.load_params(r, 0, params)
        if self.spectral_norm:
          self.u[r].copy_(torch.cat(us))
          self.v[r].copy_(torch.cat(vs))
    self.training = True

  # ---- general configuration (models.py:157-162): flat [R, g | h] parameter buffer, per-net spectral-norm vectors ----------------
  def _init_general(self, model_cfg, rng, device):
    R, S, A = self.replicas, self.state_size, self.action_size
    din, H, depth, act = (S if self.state_only else S + A), model_cfg.hidden_size, model_cfg.depth, model_cfg.activation
    self.activation = act
    self.g_dims = [din, 1] if self.reward_shaping else [din] + [H] * depth + [1]
    self.h_dims = ([S] + [H] * depth + [1]) if self.reward_shaping else None
    self.device = torch.device('cuda') if device is None else torch.device(device)
    g_total = _lib.py_mlp_offsets(self.g_dims)[2]
    h_total = _lib.py_mlp_offsets(self.h_dims)[2] if self.h_dims else 0
    self.flat = torch.zeros(R, g_total + h_total, device=self.device)
    self.g_mlp = ReplicaMLP(self.g_dims, act, R, 1, self.device)
    self.g_mlp.flat, self.g_mlp.stride = self.flat, g_total + h_total
    self.h_mlp = None
    if self.h_dims:
      self.h_mlp = ReplicaMLP(self.h_dims, act, R, 1, self.device)
      self.h_mlp.flat, self.h_mlp.stride = self.flat[:, g_total:], g_total + h_total
    self.mlp = self.g_mlp  # parameters() / generic helpers see the flat buffer through g
    sn = self.spectral_norm
    mk = lambda dims: (torch.zeros(R, sum(dims[1:]), device=self.device), torch.zeros(R, sum(dims[:-1]), device=self.device)) if sn else (None, None)
    self.g_u, self.g_v = mk(self.g_dims)
    self.h_u, self.h_v = mk(self.h_dims) if self.h_dims else (None, None)

    def fcnn(dims):  # _create_fcnn (:48-69): per layer Linear() draws, orthogonal_, zero bias, then the u / v draws of spectral_norm
      params, us, vs = [], [], []
      for l in range(len(dims) - 1):
        layer = torch.nn.Linear(dims[l], dims[l + 1])
        torch.nn.init.orthogonal_(layer.weight, gain=torch.nn.init.calculate_gain(act) if l < len(dims) - 2 else 1)
        torch.nn.init.constant_(layer.bias, 0)
        if sn:
          u_, v_ = _spectral_norm_init(layer.weight.detach())
          us.append(u_); vs.append(v_)
        params += [layer.weight.detach(), layer.bias.detach()]
      return params, us, vs

    for r in range(R):
      with (rng.replica(r) if rng is not None else _null_ctx()):
        if self.reward_shaping:  # :158-160: g is a plain nn.Linear (default init), then h
          lin = torch.nn.Linear(din, 1)
          gp, gu, gv = [lin.weight.detach(), lin.bias.detach()], [], []
          if sn:
            u_, v_ = _spectral_norm_init(gp[0])
            gu, gv = [u_], [v_]
          hp, hu, hv = fcnn(self.h_dims)
          self.h_mlp.load_params(r, 0, hp)
          if sn: self.h_u[r].copy_(torch.cat(hu)); self.h_v[r].copy_(torch.cat(hv))
        else:
          gp, gu, gv = fcnn(self.g_dims)
        self.g_mlp.load_params(r, 0, gp)
        if sn: self.g_u[r].copy_(torch.cat(gu)); self.g_v[r].copy_(torch.cat(gv))
    self.training = True

  def cx_struct(self) -> _lib.Gailx:
    d = _lib.Gailx()
    d.g = self.g_mlp.c_struct()
    if self.h_mlp is not None: d.h = self.h_mlp.c_struct()
    if self.spectral_norm:
      d.g_u, d.g_v, d.g_u_stride, d.g_v_stride = self.g_u.data_ptr(), self.g_v.data_ptr(), self.g_u.stride(0), self.g_v.stride(0)
      if self.h_mlp is not None: d.h_u, d.h_v, d.h_u_stride, d.h_v_stride = self.h_u.data_ptr(), self.h_v.data_ptr(), self.h_u.stride(0), self.h_v.stride(0)
    d.state_only, d.reward_function, d.subtract_log_policy, d.discount = int(self.state_only), _lib.REWARD[self.reward_function], int(self.subtract_log_policy), \
        0.0 if self.discount_r is not None else self.discount
    d.discount_r = _lib.ptr(self.discount_r)
    return d

  def _general_state_items(self):
    out = []
    for name, mlp, u, v, seq in (('g', self.g_mlp, self.g_u, self.g_v, not self.reward_shaping), ('h', self.h_mlp, self.h_u, self.h_v, True)):
      if mlp is None: continue
      views, uo, vo = mlp.layer_views()[0], 0, 0
      for l in range(mlp.n_layers):
        pre = f'{name}.{2 * l}' if seq else name  # nn.Sequential indices: Linear, activation, Linear, ... (no dropout modules: models.py:160,162)
        od, idim = mlp.dims[l + 1], mlp.dims[l]
        if self.spectral_norm:
          out += [(f'{pre}.bias', views[2 * l + 1]), (f'{pre}.parametrizations.weight.original', views[2 * l]), (f'{pre}.parametrizations.weight.0._u', u[:, uo:uo + od]),
                  (f'{pre}.parametrizations.weight.0._v', v[:, vo:vo + idim])]
        else:
          out += [(f'{pre}.weight', views[2 * l]), (f'{pre}.bias', views[2 * l + 1])]
        uo, vo = uo + od, vo + idim
    return out

  def _run_general(self, batch: TransitionBatch, reward_out: Optional[Tensor], want_logits: bool, log_policy: Optional[Tensor]) -> Dict[str, Tensor]:
    R, B = self.replicas, batch.B
    lib, d, b = _lib.lib(), self.cx_struct(), batch.c_struct()
    need = lib.il_gailx_reward_workspace_bytes(C.byref(d), R, B)
    if self._ws is None or self._ws.numel() < need: self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
    out = {'reward': torch.empty(R, B, device=self.device) if reward_out is None else reward_out}
    if want_logits: out['logits'] = torch.empty(R, B, device=self.device)
    if self.subtract_log_policy:
      assert log_policy is not None, 'subtract_log_policy needs log_policy (make_gail_input, models.py:148)'
      log_policy = torch.as_tensor(log_policy, dtype=torch.float32).to(self.device).reshape(R, B).contiguous()
    _lib.check(lib.il_gailx_reward(_lib.handle(), C.byref(d), R, C.byref(b), _lib.ptr(log_policy) if self.subtract_log_policy else None, out['reward'].data_ptr(), out['reward'].stride(0),
                                   out['reward'].stride(1), _lib.ptr(out.get('logits')), self._ws.data_ptr(), self._ws.numel(), _lib.stream()))
    return out

  def parameters(self) -> List[Tensor]:
    return [self.flat] if self.general else [self.mlp.flat]

  def c_struct(self) -> _lib.Gail:
    g = _lib.Gail()
    g.g = self.mlp.c_struct()
    if self.spectral_norm:
      g.u, g.v, g.u_stride, g.v_stride = self.u.data_ptr(), self.v.data_ptr(), self.u.stride(0), self.v.stride(0)
    g.state_only, g.reward_function = int(self.state_only), _lib.REWARD[self.reward_function]
    return g

  def _state_items(self):
    if self.general: return self._general_state_items()
    v = self.mlp.layer_views()[0]
    d, H = self.mlp.dims[0], self.mlp.dims[1]
    if not self.spectral_norm:
      return [(f'g.{2 * l}.{n}', v[2 * l + i]) for l in range(2) for i, n in enumerate(('weight', 'bias'))]
    return [('g.0.bias', v[1]), ('g.0.parametrizations.weight.original', v[0]), ('g.0.parametrizations.weight.0._u', self.u[:, :H]), ('g.0.parametrizations.weight.0._v', self.v[:, :d]),
            ('g.2.bias', v[3]), ('g.2.parametrizations.weight.original', v[2]), ('g.2.parametrizations.weight.0._u', self.u[:, H:H + 1]),
            ('g.2.parametrizations.weight.0._v', self.v[:, d:d + H])]

  def _batch_of(self, state: Tensor, action: Tensor, next_state=None, terminal=None) -> TransitionBatch:
    R = self.replicas
    s, a = _as_rns(state, R, self.state_size, self.device), _as_rns(action, R, self.action_size, self.device)
    off, row = _lib.py_row_layout(self.state_size, self.action_size)
    tb = TransitionBatch(torch.zeros(R, s.size(1), row, device=self.device), self.state_size, self.action_size, False)
    tb.rows[..., :self.state_size], tb.rows[..., self.state_size:self.state_size + self.action_size] = s, a
    if next_state is not None: tb.rows[..., off['next_states']:off['next_states'] + self.state_size] = _as_rns(next_state, R, self.state_size, self.device)
    if terminal is not None: tb.rows[..., off['terminals']] = torch.as_tensor(terminal, dtype=torch.float32).to(self.device).reshape(R, -1)
    return tb

  def _run(self, batch: TransitionBatch, reward_out: Optional[Tensor] = None, want_logits: bool = False, log_policy: Optional[Tensor] = None) -> Dict[str, Tensor]:
    if self.training and self.spectral_norm: raise RuntimeError('train-mode forward outside adversarial_imitation_update is not supported; call .eval() (train.py:147,180)')
    if self.general: return self._run_general(batch, reward_out, want_logits, log_policy)
    R, B = self.replicas, batch.B
    g, b = self.c_struct(), batch.c_struct()
    out = {}
    if reward_out is None: reward_out = torch.empty(R, B, device=self.device)
    out['reward'] = reward_out
    if want_logits: out['logits'] = torch.empty(R, B, device=self.device)
    _lib.check(_lib.lib().il_gail_reward(_lib.handle(), C.byref(g), R, C.byref(b), reward_out.data_ptr(), reward_out.stride(0), reward_out.stride(1), _lib.ptr(out.get('logits')),
                                         _lib.stream()))
    return out

  def forward(self, state: Tensor, action: Tensor, next_state=None, terminal=None, log_policy=None) -> Tensor:  # :172-175
    out = self._run(self._batch_of(state, action, next_state, terminal), want_logits=True, log_policy=log_policy)['logits']
    return out[0] if self.replicas == 1 else out

  __call__ = forward

  def predict_reward(self, state: Tensor, action: Tensor, next_state=None, terminal=None, log_policy=None) -> Tensor:  # :177-180
    out = self._run(self._batch_of(state, action, next_state, terminal), log_policy=log_policy)['reward']
    return out[0] if self.replicas == 1 else out

  def predict_reward_batch(self, batch: TransitionBatch, write_rewards: bool = True, actor: Optional['SoftActor'] = None) -> Tensor:
    """Fast path of train.py:194: rewards of a packed batch, written straight into its reward column. `actor` supplies the
    log-policy term of make_gail_input (models.py:148) when subtract_log_policy is set."""
    lp = actor._run(batch.rows[..., :batch.S], given=batch.rows[..., batch.S:batch.S + batch.A], want=('log_prob', ))['log_prob'] if self.subtract_log_policy else None
    if write_rewards:
      view = batch.rows[..., batch.off['rewards']]
      self._run(batch, reward_out=view, log_policy=lp)
      return view
    return self._run(batch, log_policy=lp)['reward']


class GMMILDiscriminator:
  """:183-201."""

  def __init__(self, state_size: int, action_size: int, imitation_cfg, replicas: int = 1, device=None):
    self.state_only, self.replicas = bool(imitation_cfg.state_only), replicas
    self.state_size, self.action_size = state_size, action_size
    self.device = torch.device('cuda') if device is None else torch.device(device)
    self.gamma = None  # [R, 2] once set (gamma_1, gamma_2 of :187)
    self._ws = None

  @property
  def gamma_1(self): return None if self.gamma is None else (float(self.gamma[0, 0]) if self.replicas == 1 else self.gamma[:, 0])

  @property
  def gamma_2(self): return None if self.gamma is None else (float(self.gamma[0, 1]) if self.replicas == 1 else self.gamma[:, 1])

  def _pack(self, state, action, weight) -> TransitionBatch:
    R = self.replicas
    s, a = _as_rns(state, R, self.state_size, self.device), _as_rns(action, R, self.action_size, self.device)
    off, row = _lib.py_row_layout(self.state_size, self.action_size)
    tb = TransitionBatch(torch.zeros(R, s.size(1), row, device=self.device), self.state_size, self.action_size, False)
    tb.rows[..., :self.state_size], tb.rows[..., self.state_size:self.state_size + self.action_size] = s, a
    tb.rows[..., off['weights']] = torch.as_tensor(weight, dtype=torch.float32).to(self.device).reshape(R, -1)
    return tb

  def predict_reward_batch(self, policy: TransitionBatch, expert: TransitionBatch, reward_out: Optional[Tensor] = None) -> Tensor:
    R, B = self.replicas, policy.B
    lib, h, p, e = _lib.lib(), _lib.handle(), policy.c_struct(), expert.c_struct()
    if self.gamma is None:  # :193-195: bandwidths from the first batch, then frozen
      need = lib.il_gmmil_workspace_bytes(R, B)
      ws = torch.empty(need, dtype=torch.uint8, device=self.device)
      self.gamma = torch.empty(R, 2, device=self.device)
      _lib.check(lib.il_gmmil_bandwidth(h, R, C.byref(p), C.byref(e), int(self.state_only), self.gamma.data_ptr(), ws.data_ptr(), need, _lib.stream()))
    if reward_out is None: reward_out = torch.empty(R, B, device=self.device)
    _lib.check(lib.il_gmmil_reward(h, R, C.byref(p), C.byref(e), int(self.state_only), self.gamma.data_ptr(), reward_out.data_ptr(), reward_out.stride(0), reward_out.stride(1),
                                   _lib.stream()))
    return reward_out

  def predict_reward(self, state, action, expert_state, expert_action, weight, expert_weight) -> Tensor:
    out = self.predict_reward_batch(self._pack(state, action, weight), self._pack(expert_state, expert_action, expert_weight))
    return out[0] if self.replicas == 1 else out


class PWILDiscriminator:
  """:216-249. The expert atoms are shared by all replicas; the remaining-weight vector is per replica."""

  def __init__(self, state_size: int, action_size: int, imitation_cfg, expert_memory: ReplayMemory, time_horizon: int, replicas: int = 1, device=None,
               reward_scale=None, reward_bandwidth_scale=None):
    """reward_scale / reward_bandwidth_scale override imitation_cfg's values with a float or one value per replica ([R])."""
    self.state_only, self.replicas = bool(imitation_cfg.state_only), replicas
    self.state_size, self.action_size, self.time_horizon = state_size, action_size, time_horizon
    self.expert_memory = expert_memory
    self.device = torch.device('cuda') if device is None else torch.device(device)
    atoms = self._get_expert_atoms().to(self.device)
    inv_scale, offset = atoms.std(dim=0, keepdim=True), -atoms.mean(dim=0, keepdim=True)  # :205-208 (one-off setup)
    inv_scale[inv_scale == 0] = 1
    self.data_scale, self.data_offset = (1 / inv_scale).contiguous(), offset.contiguous()
    self.atoms = (self.data_scale * (atoms + self.data_offset)).contiguous()  # :229
    self.reward_scale = imitation_cfg.reward_scale if reward_scale is None else reward_scale
    self.reward_bandwidth = self._bandwidth(imitation_cfg.reward_bandwidth_scale if reward_bandwidth_scale is None else reward_bandwidth_scale)
    self.reward_scale_r, self.reward_bandwidth_r = per_replica(self.reward_scale, self.device), per_replica(self.reward_bandwidth, self.device)
    for t in (self.reward_scale_r, self.reward_bandwidth_r): assert t is None or t.numel() == replicas, 'one PWIL reward scale / bandwidth per replica'
    self.expert_weights = torch.empty(replicas, self.atoms.size(0), device=self.device)
    self.reset()

  def _bandwidth(self, scale):
    if per_replica(scale, 'cpu') is not None: scale = per_replica(scale, 'cpu', torch.float64)  # the host expression below in double, replica by replica
    return scale * self.time_horizon / sqrt(self.state_size if self.state_only else self.state_size + self.action_size)  # :222

  def set_reward_hparams(self, reward_scale=None, reward_bandwidth_scale=None):
    """Rewrites the per-replica reward scale / bandwidth arrays in place (same expressions as the constructor); None leaves one as it is."""
    if reward_scale is not None: self.reward_scale_r.copy_(per_replica(reward_scale, self.device))
    if reward_bandwidth_scale is not None: self.reward_bandwidth_r.copy_(per_replica(self._bandwidth(reward_bandwidth_scale), self.device))

  def _get_expert_atoms(self) -> Tensor:  # :225-226
    s, a = self.expert_memory['states'], self.expert_memory['actions']
    return (s if self.state_only else torch.cat([s, a], dim=1)).clone()

  def c_struct(self) -> _lib.Pwil:
    p = _lib.Pwil()
    p.atoms, p.scale, p.offset, p.weights = self.atoms.data_ptr(), self.data_scale.data_ptr(), self.data_offset.data_ptr(), self.expert_weights.data_ptr()
    p.N, p.d, p.S, p.A = self.atoms.size(0), self.atoms.size(1), self.state_size, self.action_size
    p.state_only, p.time_horizon = int(self.state_only), self.time_horizon
    p.reward_scale = 0.0 if self.reward_scale_r is not None else self.reward_scale
    p.reward_bandwidth = 0.0 if self.reward_bandwidth_r is not None else self.reward_bandwidth
    p.reward_scale_r, p.reward_bandwidth_r = _lib.ptr(self.reward_scale_r), _lib.ptr(self.reward_bandwidth_r)
    return p

  def reset(self, mask: Optional[Tensor] = None):  # :228-230
    p = self.c_struct()
    _lib.check(_lib.lib().il_pwil_reset(_lib.handle(), C.byref(p), self.replicas, _lib.ptr(mask), _lib.stream()))

  def compute_reward_batch(self, state: Tensor, action: Tensor, out: Optional[Tensor] = None, active: Optional[Tensor] = None) -> Tensor:
    R = self.replicas
    s = torch.as_tensor(state, dtype=torch.float32).to(self.device).reshape(R, self.state_size).contiguous()
    a = torch.as_tensor(action, dtype=torch.float32).to(self.device).reshape(R, self.action_size).contiguous()
    if out is None: out = torch.empty(R, device=self.device)
    p = self.c_struct()
    _lib.check(_lib.lib().il_pwil_reward(_lib.handle(), C.byref(p), R, s.data_ptr(), a.data_ptr(), out.data_ptr(), _lib.ptr(active), _lib.stream()))
    return out

  def compute_reward(self, state: Tensor, action: Tensor):  # :232-249
    out = self.compute_reward_batch(state, action)
    return float(out[0]) if self.replicas == 1 else out


class REDDiscriminator(_Module):
  """:252-284 — predictor (with dropout) and frozen random target embedding networks (din -> hidden^depth -> din), one pair per replica."""

  def __init__(self, state_size: int, action_size: int, imitation_cfg, replicas: int = 1, rng: Optional[ReplicaRNG] = None, device=None):
    cfg = imitation_cfg.discriminator
    self.state_only, self.replicas = bool(imitation_cfg.state_only), replicas
    self.state_size, self.action_size = state_size, action_size
    din = state_size if self.state_only else state_size + action_size
    dims = [din] + [cfg.hidden_size] * cfg.depth + [din]
    self.input_dropout, self.dropout = float(_cfg_get(cfg, 'input_dropout', 0) or 0), float(_cfg_get(cfg, 'dropout', 0) or 0)
    self.predictor, self.target = ReplicaMLP(dims, cfg.activation, replicas, 1, device), ReplicaMLP(dims, cfg.activation, replicas, 1, device)
    self.mlp = self.predictor  # parameters(): only the predictor trains (:267-268; AdamW skips the frozen target, train.py:84)
    self.device = self.predictor.device
    for r in range(replicas):
      with (rng.replica(r) if rng is not None else _null_ctx()):
        self.predictor.load_params(r, 0, init_fcnn_params(dims, cfg.activation))  # :265
        self.target.load_params(r, 0, init_fcnn_params(dims, cfg.activation))     # :266
    s1 = _cfg_get(imitation_cfg, 'reward_bandwidth_scale', None)
    self.sigma = torch.full((replicas, ), float(s1) if s1 else 0.0, device=self.device)  # :269
    self._sigma_set = bool(s1)
    self.training, self._ws, self._rng = True, None, None

  @property
  def sigma_1(self): return None if not self._sigma_set else (float(self.sigma[0]) if self.replicas == 1 else self.sigma)

  def c_struct(self) -> _lib.Red:
    d = _lib.Red()
    d.predictor, d.target, d.sigma, d.state_only = self.predictor.c_struct(), self.target.c_struct(), self.sigma.data_ptr(), int(self.state_only)
    return d

  def _state_items(self):
    out = []
    for name, mlp in (('predictor', self.predictor), ('target', self.target)):
      v = mlp.layer_views()[0]
      step = 2 + (1 if (name == 'predictor' and self.dropout > 0) else 0)  # nn.Sequential indices: [Dropout], Linear, [Dropout], activation, ...
      base = 1 if (name == 'predictor' and self.input_dropout > 0) else 0
      out += [(f'{name}.embedding.{base + step * l}.{n}', v[2 * l + i]) for l in range(mlp.n_layers) for i, n in enumerate(('weight', 'bias'))]
    return out

  def workspace(self, B: int) -> Tensor:
    d = self.c_struct()
    need = _lib.lib().il_red_workspace_bytes(C.byref(d), self.replicas, B)
    if self._ws is None or self._ws.numel() < need: self._ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
    return self._ws

  def draw_masks(self, n: int) -> List[Optional[Tensor]]:
    if self._rng is None: self._rng = _RNG(default_rng.seed + 1979, self.device)
    rng, R, lib = self._rng, self.replicas, _lib.lib()
    def draw(width, p):
      if p <= 0: return None
      out = torch.empty(R, n, width, device=self.device)
      ctr = rng._ctr(self.device)
      _lib.check(lib.il_fill_dropout_mask(_lib.handle(), out.data_ptr(), out.numel(), p, rng.seed, 32, ctr.data_ptr(), _lib.stream()))
      _lib.check(lib.il_counter_add(_lib.handle(), ctr.data_ptr(), (out.numel() + 3) // 4, _lib.stream()))
      return out
    return [draw(self.predictor.dims[0], self.input_dropout)] + [draw(self.predictor.dims[l + 1], self.dropout) for l in range(self.predictor.n_layers - 1)]

  def _batch_of(self, state: Tensor, action: Tensor) -> TransitionBatch:
    R = self.replicas
    s, a = _as_rns(state, R, self.state_size, self.device), _as_rns(action, R, self.action_size, self.device)
    _, row = _lib.py_row_layout(self.state_size, self.action_size)
    tb = TransitionBatch(torch.zeros(R, s.size(1), row, device=self.device), self.state_size, self.action_size, False)
    tb.rows[..., :self.state_size], tb.rows[..., self.state_size:self.state_size + self.action_size] = s, a
    return tb

  def set_sigma_batch(self, batch: TransitionBatch, masks=None):  # :277-280
    if self._sigma_set: return
    if masks is None and self.training: masks = self.draw_masks(batch.B)
    masks = masks or [None] * self.predictor.n_layers
    d, b, ws = self.c_struct(), batch.c_struct(), self.workspace(batch.B)
    _lib.check(_lib.lib().il_red_sigma(_lib.handle(), C.byref(d), self.replicas, C.byref(b), _lib.ptr(masks[0]), _lib.mask_array(masks[1:]), ws.data_ptr(), ws.numel(), _lib.stream()))
    self._sigma_set = True

  def set_sigma(self, expert_state: Tensor, expert_action: Tensor, masks=None):
    es, ea = torch.as_tensor(expert_state, dtype=torch.float32).to(self.device), torch.as_tensor(expert_action, dtype=torch.float32).to(self.device)
    if es.dim() == 2 and self.replicas > 1: es, ea = es.unsqueeze(0).expand(self.replicas, -1, -1), ea.unsqueeze(0).expand(self.replicas, -1, -1)
    self.set_sigma_batch(self._batch_of(es, ea), masks)

  def predict_reward_batch(self, batch: TransitionBatch, reward_out: Optional[Tensor] = None) -> Tensor:  # :282-284 (eval mode, train.py:147)
    R, B = self.replicas, batch.B
    if reward_out is None: reward_out = torch.empty(R, B, device=self.device)
    d, b, ws = self.c_struct(), batch.c_struct(), self.workspace(B)
    _lib.check(_lib.lib().il_red_reward(_lib.handle(), C.byref(d), R, C.byref(b), reward_out.data_ptr(), reward_out.stride(0), reward_out.stride(1), ws.data_ptr(), ws.numel(), _lib.stream()))
    return reward_out

  def predict_reward(self, state: Tensor, action: Tensor) -> Tensor:
    out = self.predict_reward_batch(self._batch_of(state, action))
    return out[0] if self.replicas == 1 else out


def mix_expert_agent_transitions(transitions: TransitionBatch, expert_transitions: TransitionBatch):
  """:287-290 — first B // 2 rows of every field replaced by expert rows."""
  b, e = transitions.c_struct(), expert_transitions.c_struct()
  _lib.check(_lib.lib().il_mix_expert_rows(_lib.handle(), C.byref(b), C.byref(e), transitions.R, _lib.stream()))


class RewardRelabeller:
  """:293-318 — AdRIL (update_freq > 0) / SQIL (update_freq == 0): builds the training batch from expert and policy data and labels the
  rewards; one kernel, with the balanced-sampling alternation flag kept on the device so the call can live inside a captured CUDA graph."""

  def __init__(self, update_freq: int, balanced: bool, device=None):
    self.update_freq, self.balanced = int(update_freq), bool(balanced)
    self.device = torch.device('cuda') if device is None else torch.device(device)
    self._flag = torch.ones(1, dtype=torch.int32, device=self.device)  # sample_expert = True (:295)

  @property
  def sample_expert(self) -> bool: return bool(self._flag.item())

  def resample_and_relabel(self, transitions: TransitionBatch, expert_transitions: TransitionBatch, step, num_trajectories, num_expert_trajectories: int, step_offset: float = 0.0):
    """`step`: the loop step (int, or a device float tensor [R] + `step_offset`); `num_trajectories`: int or the device counters [R] of the replay memory."""
    R, dev = transitions.R, self.device
    step_t = step if torch.is_tensor(step) else torch.full((R, ), float(step), device=dev)
    nt = num_trajectories if torch.is_tensor(num_trajectories) else torch.full((R, ), int(num_trajectories), dtype=torch.int32, device=dev)
    b, e = transitions.c_struct(), expert_transitions.c_struct()
    _lib.check(_lib.lib().il_adril_relabel(_lib.handle(), C.byref(b), C.byref(e), R, int(self.balanced), self.update_freq, self._flag.data_ptr(), step_t.data_ptr(), float(step_offset),
                                           nt.data_ptr(), int(nt.numel() == 1), int(num_expert_trajectories), _lib.stream()))
