"""The training orchestrator (reference train.py:26-243) for R seed-sharded replicas on one GPU.

`Trainer.rollout()` is train.py:150-168 and `Trainer.update()` is train.py:171-203, each a fixed sequence of C-ABI
calls on one CUDA stream with every piece of per-step state (env state, replay ring indices, optimiser step
counts, RNG counters, the `step` counter) resident on the device — so both sequences are captured once as CUDA
graphs and replayed without host involvement. Replica r is a reference-equivalent run with seed `cfg.seed + r`.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
import time
from typing import Dict, List, Optional

import numpy as np
import torch
from torch import Tensor

from . import _lib, distributed, sweep
from .config import Config, load_config
from .environments import D4RLEnv, ENVS
from .evaluation import evaluate_agent
from .memory import ReplayMemory, TransitionBatch
from .models import GAILDiscriminator, GMMILDiscriminator, PWILDiscriminator, REDDiscriminator, RewardRelabeller, SoftActor, TwinCritic, _RNG, create_target_network
from .net import ReplicaRNG
from .optim import Adam, AdamW

ACCELERATED = ['AdRIL', 'BC', 'DRIL', 'SAC', 'GAIL', 'GMMIL', 'PWIL', 'RED']
MAX_SWEEP_REPLICAS = 4096  # replicas per AdamW launch with per-replica hyperparameters (ADAM_MAX_REPLICAS, csrc/mlp.cu)


def check_config(cfg: Config):
  """train.py:28-48."""
  assert cfg.algorithm in ['AdRIL', 'BC', 'DRIL', 'GAIL', 'GMMIL', 'PWIL', 'RED', 'SAC']
  assert cfg.env in ENVS
  cfg.memory.size = min(cfg.steps, cfg.memory.size)
  assert cfg.bc_pretraining.iterations >= 0
  assert cfg.imitation.trajectories >= 0
  assert cfg.imitation.subsample >= 1
  assert cfg.imitation.mix_expert_data in ['none', 'mixed_batch', 'prefill_memory']
  if cfg.algorithm == 'AdRIL':  # train.py:35-37
    assert cfg.imitation.mix_expert_data == 'mixed_batch'
    assert cfg.imitation.update_freq >= 0
  if cfg.algorithm == 'DRIL': assert 0 <= cfg.imitation.quantile_cutoff <= 1  # train.py:38-39
  if cfg.algorithm == 'GAIL':
    assert cfg.imitation.mix_expert_data != 'prefill_memory'
    assert cfg.imitation.discriminator.reward_function in ['AIRL', 'FAIRL', 'GAIL']
    assert cfg.imitation.grad_penalty >= 0
    assert cfg.imitation.entropy_bonus >= 0
    assert cfg.imitation.loss_function in ['BCE', 'Mixup', 'PUGAIL']
    if cfg.imitation.loss_function == 'Mixup': assert cfg.imitation.mixup_alpha > 0
    if cfg.imitation.loss_function == 'PUGAIL': assert 0 <= cfg.imitation.pos_class_prior <= 1 and cfg.imitation.nonnegative_margin >= 0
  assert cfg.logging.interval >= 0
  if cfg.algorithm not in ACCELERATED:
    raise NotImplementedError(f'algorithm={cfg.algorithm} is outside the accelerated hot path (BASELINE.json north_star; SURVEY §8f); supported: {ACCELERATED}')


class Trainer:
  def __init__(self, cfg: Config, replicas: Optional[int] = None, seed_offset: int = 0, fast_init: bool = False, device=None, hparams: Optional[Dict[str, Tensor]] = None,
               grad_penalty_any: Optional[bool] = None):
    """hparams: {key: [R] values} of per-replica hyperparameters (the keys of sweep.BATCHABLE); replica r trains with its own values and
    equals, bit for bit, a run configured with them. Without it every replica uses the config's values. They can be changed in place later
    (set_hparams). grad_penalty_any: whether any replica may ever have a positive imitation.grad_penalty (default: any initial value > 0);
    it decides at set-up whether the penalty noise is drawn and whether the general discriminator runs its penalty pass."""
    check_config(cfg)
    self.cfg = cfg
    self.R = R = int(cfg.get('replicas', 1) if replicas is None else replicas)
    self.device = dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
    self.hparams = self._check_hparams(hparams or {}, cfg, R, dev)
    hp = lambda key, default: self.hparams.get(key, default)  # float64 [R] (the optimisers keep lr / weight decay in double) or the config float
    self.lib, self.h = _lib.lib(), _lib.handle(dev.index)
    _lib.check(self.lib.il_set_gemm_mode(self.h, _lib.GEMM_MODE[cfg.get('gemm_mode', 'fp32')]))
    self.seed = seed = cfg.seed + seed_offset
    np.random.seed(seed)
    torch.manual_seed(seed)  # train.py:51-52
    self.algorithm = cfg.algorithm
    absorbing = bool(cfg.imitation.absorbing)
    # train.py:55-61
    self.env, self.eval_env = D4RLEnv(cfg.env, absorbing, load_data=True, replicas=R, device=dev), D4RLEnv(cfg.env, absorbing, replicas=R, device=dev)
    self.env.seed(seed)
    self.eval_env.seed(seed)
    self.normalization_max, self.normalization_min = self.env.env.ref_max_score, self.env.env.ref_min_score
    need_expert = self.algorithm != 'SAC' or cfg.bc_pretraining.iterations > 0 or cfg.imitation.bc_aux_loss
    self.expert_memory = self.env.get_dataset(trajectories=cfg.imitation.trajectories, subsample=cfg.imitation.subsample) if need_expert else None
    self.S, self.A = S, A = self.env.observation_space.shape[0], self.env.action_space.shape[0]
    derived = self._derived_hparams()
    # train.py:64-67 — replica r draws its initial weights from the stream of seed + r (fast_init: one stream, replicated)
    rng = None if (R == 1 or fast_init) else ReplicaRNG(seed, R)
    nrep = 1 if fast_init else R
    self.actor, self.critic = SoftActor(S, A, cfg.reinforcement.actor, replicas=nrep, rng=rng, device=dev), TwinCritic(S, A, cfg.reinforcement.critic, replicas=nrep, rng=rng, device=dev)
    self.discriminator = None
    self.discount, self.polyak = derived['discount'], derived['polyak']
    if self.algorithm == 'GAIL': self.discriminator = GAILDiscriminator(S, A, cfg.imitation, self.discount, replicas=nrep, rng=rng, device=dev)
    elif self.algorithm == 'DRIL': self.discriminator = SoftActor(S, A, cfg.imitation.discriminator, replicas=nrep, rng=rng, device=dev)  # train.py:74
    elif self.algorithm == 'RED': self.discriminator = REDDiscriminator(S, A, cfg.imitation, replicas=nrep, rng=rng, device=dev)  # train.py:82
    if fast_init and R > 1: self._replicate()
    self.log_alpha = torch.zeros(R, device=dev)
    self.target_critic = create_target_network(self.critic)
    self.entropy_target = derived['entropy_target']
    lr, wd = hp('training.learning_rate', cfg.training.learning_rate), hp('training.weight_decay', cfg.training.weight_decay)
    self.actor_optimiser, self.critic_optimiser = AdamW(self.actor.parameters(), lr=lr, weight_decay=wd), AdamW(self.critic.parameters(), lr=lr, weight_decay=wd)
    self.temperature_optimiser = Adam([self.log_alpha], lr=lr)
    need = R * int(cfg.memory.size) * _lib.py_row_layout(S, A)[1] * 4
    free = torch.cuda.mem_get_info(dev)[0]
    if need > 0.9 * free:
      raise MemoryError(f'replay rings need {need / 2**30:.1f} GiB ({R} replicas x memory.size {cfg.memory.size} rows x {_lib.py_row_layout(S, A)[1] * 4} B) but only {free / 2**30:.1f} GiB '
                        f'are free on {dev}; lower memory.size (train.py:30 caps it at `steps`) or `replicas`')
    self.memory = ReplayMemory(cfg.memory.size, S, A, absorbing, replicas=R, device=dev)
    self.memory.seed = seed
    # train.py:70-84
    if self.algorithm in ('DRIL', 'GAIL', 'RED'):
      self.discriminator_optimiser = AdamW(self.discriminator.parameters(), lr=hp('imitation.learning_rate', cfg.imitation.learning_rate),
                                           weight_decay=hp('imitation.weight_decay', cfg.imitation.weight_decay))  # train.py:83-84
    if self.algorithm == 'GAIL':
      self.discriminator.eval()  # train.py:147
    elif self.algorithm == 'AdRIL':
      self.discriminator = RewardRelabeller(cfg.imitation.update_freq, cfg.imitation.balanced, device=dev)  # train.py:72
      self._expert_trajectories = int(self.expert_memory.num_trajectories)  # constant: read once, outside any graph capture
    elif self.algorithm == 'GMMIL':
      self.discriminator = GMMILDiscriminator(S, A, cfg.imitation, replicas=R, device=dev)
    elif self.algorithm == 'PWIL':
      self.discriminator = PWILDiscriminator(S, A, cfg.imitation, self.expert_memory, self.env.max_episode_steps, replicas=R, device=dev,
                                             reward_scale=hp('imitation.reward_scale', None), reward_bandwidth_scale=hp('imitation.reward_bandwidth_scale', None))
    if self.expert_memory is not None: self.expert_memory.seed = seed + 7919
    if self.algorithm == 'PWIL' and cfg.imitation.mix_expert_data != 'none': self._pwil_relabel_expert()  # train.py:136-140
    if self.algorithm in ('GMMIL', 'PWIL') and cfg.imitation.mix_expert_data == 'prefill_memory': self.memory.transfer_transitions(self.expert_memory)  # train.py:141,143
    # ---- per-step device state -------------------------------------------------------------------------------
    B = self.B = cfg.training.batch_size
    f = lambda *shape: torch.zeros(*shape, device=dev)
    i32 = lambda *shape: torch.zeros(*shape, dtype=torch.int32, device=dev)
    self.state, self.next_state, self.action = f(R, S), f(R, S), f(R, A)
    self.env_reward, self.store_reward = f(R), f(R)
    self.done, self.timeout, self.terminal_f, self.timeout_f = i32(R), i32(R), f(R), f(R)
    self.step_f = torch.ones(R, device=dev)  # train.py:149: steps count from 1
    self.running_return, self.last_return, self.return_sum, self.episodes = f(R), f(R), f(R), i32(R)
    self.eps_act, self.u_reset = f(R, A), f(R, self.env.obs)
    self.idx_pol, self.idx_exp = i32(R, B), i32(R, B)
    self.u_pol, self.u_exp = f(R, B), f(R, B)  # host-drawn uniforms (device_rng: false)
    row = self.memory.row
    self.batch = TransitionBatch(f(R, B, row), S, A, absorbing)
    self.expert_batch = TransitionBatch(f(R, B, row), S, A, absorbing)
    self.eps_gp, self.eps_mix, self.eps_next, self.eps_new = f(R, B), f(R, B), f(R, B, A), f(R, B, A)
    self.sac_out = dict(log_probs=f(R, B), q_values=f(R, B), losses=f(R, 3))
    self.gail_losses = f(R, 2)
    self.rng = _RNG(seed, dev)
    self.grad_penalty, self.entropy_bonus = derived['grad_penalty'], derived['entropy_bonus']
    self.grad_penalty_any = None
    if 'imitation.grad_penalty' in self.hparams:  # set-up time, never in a capture
      positive = bool((self.hparams['imitation.grad_penalty'] > 0).any())
      if grad_penalty_any is False and positive: raise ValueError('grad_penalty_any=False but some replica starts with imitation.grad_penalty > 0')
      self.grad_penalty_any = positive if grad_penalty_any is None else bool(grad_penalty_any)
    self._src_of = None  # exploit(): the device replica map, allocated on first use and rewritten in place
    self.inject = False  # tests: True = all noise / index buffers are filled by the caller before each step
    self.dril_masks = None  # tests (inject): the dropout masks of this step's DRIL ensemble pass
    self.device_rng = bool(cfg.get('device_rng', True))
    self.actor_ws = torch.empty(self.lib.il_actor_workspace_bytes(C.byref(self.actor.mlp.c_struct()), R, 1), dtype=torch.uint8, device=dev)
    self._sac_args = None
    self.step = 0
    self.updates = 0
    self.graphs: Dict[str, torch.cuda.CUDAGraph] = {}
    self.graph_launches: Dict[str, int] = {}
    self.use_graphs = bool(cfg.get('cuda_graphs', True))
    self.metrics = dict(train_steps=[], train_returns=[], test_steps=[], test_returns=[], test_returns_normalized=[], update_steps=[], predicted_rewards=[], alphas=[],
                        entropies=[], Q_values=[])  # train.py:87
    self.score: List[float] = []
    self.env.batch.reset(self.env.reset_noise(R), self.state)  # train.py:146

  @staticmethod
  def _check_hparams(hparams, cfg: Config, R: int, dev) -> Dict[str, Tensor]:
    if hparams and R > MAX_SWEEP_REPLICAS:
      raise ValueError(f'per-replica hyperparameters support up to {MAX_SWEEP_REPLICAS} replicas per GPU (the per-replica AdamW kernels keep a table of every '
                       f'replica in shared memory); {R} requested: use more GPUs or fewer replicas')
    if cfg.algorithm == 'PWIL' and cfg.imitation.mix_expert_data != 'none' and {'imitation.reward_scale', 'imitation.reward_bandwidth_scale'} & set(hparams):
      raise ValueError('PWIL reward scale / bandwidth cannot vary per replica with imitation.mix_expert_data != none: the expert memory shared by all replicas '
                       'holds one relabelled reward per transition')
    out = {}
    for k, v in hparams.items():
      if k not in sweep.BATCHABLE: raise ValueError(f'hparams: {k} cannot vary per replica; batchable keys: {", ".join(sweep.BATCHABLE)}')
      t = torch.as_tensor(v, dtype=torch.float64).reshape(-1)
      if t.numel() != R: raise ValueError(f'hparams: {k} has {t.numel()} values for {R} replicas')
      host = t.cpu()
      if k == 'imitation.quantile_cutoff' and not bool(((host >= 0) & (host <= 1)).all()): raise ValueError('hparams: quantile_cutoff outside [0, 1]')
      if k in ('imitation.grad_penalty', 'imitation.entropy_bonus') and not bool((host >= 0).all()): raise ValueError(f'hparams: {k} must be >= 0')
      out[k] = t.to(dev).contiguous()
    return out

  def _derived_hparams(self) -> Dict[str, object]:
    """The float32 kernel arguments computed from self.hparams (a [R] device array for a per-replica key, else the config's scalar or None):
    the constructor creates them and set_hparams rewrites them in place, through this one function."""
    cfg, hps = self.cfg, self.hparams
    hp32 = lambda key, default: hps[key].float() if key in hps else default  # float scalars of the kernels, rounded like a Python float
    tt = hps.get('reinforcement.target_temperature', cfg.reinforcement.target_temperature)
    A = self.A
    return dict(discount=hp32('reinforcement.discount', cfg.reinforcement.discount), polyak=hp32('reinforcement.polyak_factor', cfg.reinforcement.polyak_factor),
                entropy_target=(tt * A).float() if isinstance(tt, Tensor) else tt * A,
                grad_penalty=hp32('imitation.grad_penalty', None), entropy_bonus=hp32('imitation.entropy_bonus', None))

  def set_hparams(self, values: Dict[str, object]):
    """Writes new [R] values of per-replica hyperparameters in place: self.hparams, every float32 array derived from them and the arrays the
    optimisers hold. Nothing is allocated that a kernel reads, so captured CUDA graphs keep running, now with the new values. Only keys the
    trainer was built with can change (a key set up as a scalar is baked into the graphs)."""
    new = self._check_hparams(values, self.cfg, self.R, self.device)
    fixed = [k for k in new if k not in self.hparams]
    if fixed: raise ValueError(f'set_hparams: {", ".join(fixed)} was not per-replica at construction (Trainer(hparams=...)); per-replica keys: {", ".join(self.hparams) or "none"}')
    if 'imitation.grad_penalty' in new and not self.grad_penalty_any and bool((new['imitation.grad_penalty'] > 0).any()):
      raise ValueError('set_hparams: a positive imitation.grad_penalty needs Trainer(grad_penalty_any=True): this trainer was set up without the penalty draws')
    for k, v in new.items(): self.hparams[k].copy_(v)
    for name, v in self._derived_hparams().items():
      cur = getattr(self, name)
      if isinstance(cur, Tensor): cur.copy_(v)
    if self.algorithm == 'PWIL': self.discriminator.set_reward_hparams(self.hparams.get('imitation.reward_scale'), self.hparams.get('imitation.reward_bandwidth_scale'))
    for name, (lr_key, wd_key) in (('actor_optimiser', ('training.learning_rate', 'training.weight_decay')), ('critic_optimiser', ('training.learning_rate', 'training.weight_decay')),
                                   ('temperature_optimiser', ('training.learning_rate', None)),
                                   ('discriminator_optimiser', ('imitation.learning_rate', 'imitation.weight_decay'))):
      opt = getattr(self, name, None)
      if opt is None: continue
      for arr, key in ((opt.lr_r, lr_key), (opt.weight_decay_r, wd_key)):
        if arr is not None and key in self.hparams and arr.data_ptr() != self.hparams[key].data_ptr(): arr.copy_(self.hparams[key])

  def replica_state(self) -> List[Tensor]:
    """Every tensor whose leading axis is the replica axis and that carries training state from one step to the next: network, target and
    optimiser state, log_alpha, the discriminator's learned and set-up state, the replay ring and its counters, the environments and the loop's
    episode bookkeeping. Excluded: values shared by all replicas (step counts, RNG counters, AdRIL's flag, the expert memory), workspaces,
    noise and index buffers and per-call outputs, which are rewritten before they are read."""
    out = [self.actor.mlp.flat, self.critic.mlp.flat, self.target_critic.mlp.flat, self.log_alpha]
    for name in ('actor_optimiser', 'critic_optimiser', 'temperature_optimiser', 'discriminator_optimiser'):
      opt = getattr(self, name, None)
      if opt is not None: out += [opt.exp_avg, opt.exp_avg_sq]
    d = self.discriminator
    if self.algorithm == 'GAIL':
      out += [d.flat, d.g_u, d.g_v, d.h_u, d.h_v] if d.general else [d.mlp.flat, d.u, d.v]
    elif self.algorithm == 'DRIL': out += [d.mlp.flat, d._q if d.q is not None else None]
    elif self.algorithm == 'RED': out += [d.predictor.flat, d.target.flat, d.sigma]
    elif self.algorithm == 'PWIL': out += [d.expert_weights]
    elif self.algorithm == 'GMMIL': out += [d.gamma]
    m = self.memory
    out += [m.rows, m._idx, m._full, m._num_trajectories, self.env.batch.x, self.env.batch.t]
    out += [self.state, self.step_f, self.running_return, self.last_return, self.return_sum, self.episodes]
    return [t for t in out if t is not None]

  def exploit(self, src_of):
    """Population-based training's exploit step: replica r becomes a copy of replica src_of[r] (a host [R] map, or {destination: source}) in
    every tensor of replica_state() and every per-replica hyperparameter, with one il_replica_copy launch. A source must be its own source.
    A destination keeps its seed and its position in the noise buffers, so afterwards it differs from its source only in the noise it draws."""
    R = self.R
    if isinstance(src_of, dict):
      m = np.arange(R)
      for dst, src in src_of.items(): m[int(dst)] = int(src)
    else: m = np.asarray(src_of).reshape(-1)
    if m.shape != (R, ) or not np.issubdtype(m.dtype, np.integer) or m.min() < 0 or m.max() >= R:
      raise ValueError(f'exploit: expected {R} replica indices in [0, {R}), got {src_of!r}')
    m = m.astype(np.int32)
    if not np.array_equal(m[m], m): raise ValueError(f'exploit: replicas {np.flatnonzero(m[m] != m).tolist()} copy from a replica that is itself overwritten')
    if self._src_of is None: self._src_of = torch.empty(R, dtype=torch.int32, device=self.device)
    self._src_of.copy_(torch.from_numpy(m))
    bufs = self.replica_state()
    for t in bufs: assert t.size(0) == R and t.is_contiguous() and t.element_size() == 4, 'replica_state(): contiguous 4-byte [R, ...] buffers'
    n = len(bufs)
    base = (C.c_void_p * n)(*[t.data_ptr() for t in bufs])
    stride = (C.c_int64 * n)(*[t.stride(0) * 4 for t in bufs])
    nbytes = (C.c_int64 * n)(*[t[0].numel() * 4 for t in bufs])
    _lib.check(self.lib.il_replica_copy(self.h, n, base, stride, nbytes, R, self._src_of.data_ptr(), _lib.stream()))
    if self.hparams: self.set_hparams({k: v.cpu()[torch.from_numpy(m).long()] for k, v in self.hparams.items()})

  def _pwil_relabel_expert(self):
    """train.py:136-140: the expert's own transitions get their greedy PWIL reward, walking the expert memory in order and
    restoring the atoms at every episode end. The expert memory is shared by all replicas and every replica would compute the
    same numbers, so one single-replica coupling state does the walk (one-off setup: one small launch per expert transition)."""
    em, d = self.expert_memory, self.discriminator
    one = PWILDiscriminator(self.S, self.A, self.cfg.imitation, em, self.env.max_episode_steps, replicas=1, device=self.device)
    ends = ((em.rows[0, :, em.off['terminals']] != 0) | (em.rows[0, :, em.off['timeouts']] != 0)).cpu().numpy()  # setup-time read of the episode boundaries
    states, actions, rewards = em.rows[0, :, em.off['states']:em.off['states'] + self.S], em.rows[0, :, em.off['actions']:em.off['actions'] + self.A], em.rows[0, :, em.off['rewards']]
    out = torch.empty(1, device=self.device)
    for i in range(em.size):
      one.compute_reward_batch(states[i:i + 1], actions[i:i + 1], out=out)
      rewards[i:i + 1].copy_(out)  # expert_memory.rewards[i] = ...
      if ends[i]: one.reset()
    # the reference walks the expert data with THE discriminator, so whatever atoms the last (unfinished) expert episode consumed
    # stay consumed when training starts: every replica inherits the walk's remaining-weight vector
    d.expert_weights.copy_(one.expert_weights.expand_as(d.expert_weights))

  def _replicate(self):
    """fast_init: every replica starts from replica 0's initial weights (throughput runs; replicas still diverge
    through their own env / noise streams)."""
    for mod in (self.actor, self.critic, self.discriminator):
      if mod is None: continue
      if getattr(mod, 'general', False):  # general GAIL discriminator: one flat [R, g | h] buffer with two net views
        g_total = mod.h_mlp.flat.storage_offset() - mod.flat.storage_offset() if mod.h_mlp is not None else 0
        mod.flat = mod.flat.expand(self.R, -1).contiguous()
        mod.g_mlp.flat, mod.g_mlp.replicas = mod.flat, self.R
        if mod.h_mlp is not None: mod.h_mlp.flat, mod.h_mlp.replicas = mod.flat[:, g_total:], self.R
        mod.replicas = self.R
        for n in ('g_u', 'g_v', 'h_u', 'h_v'):
          if getattr(mod, n, None) is not None: setattr(mod, n, getattr(mod, n).expand(self.R, -1).contiguous())
        continue
      mod.mlp.flat = mod.mlp.flat.expand(self.R, -1).contiguous()
      mod.mlp.replicas = self.R
      mod.replicas = self.R
      if isinstance(mod, REDDiscriminator):  # the frozen target network and the bandwidths as well
        mod.target.flat, mod.target.replicas = mod.target.flat.expand(self.R, -1).contiguous(), self.R
        mod.sigma = mod.sigma.expand(self.R).contiguous()
      if getattr(mod, 'u', None) is not None: mod.u, mod.v = mod.u.expand(self.R, -1).contiguous(), mod.v.expand(self.R, -1).contiguous()

  # ---- train.py:150-168 -------------------------------------------------------------------------------------------
  def rollout(self):
    lib, h, st, R = self.lib, self.h, _lib.stream(), self.R
    if not self.inject: self.rng.normal(None, self.device, stream_id=1, out=self.eps_act)
    m = self.actor.mlp.c_struct()
    _lib.check(lib.il_actor_forward(h, C.byref(m), R, 1, self.state.data_ptr(), self.S, self.S, self.eps_act.data_ptr(), None, self.action.data_ptr(), None, None, None,
                                    self.actor_ws.data_ptr(), self.actor_ws.numel(), st))  # train.py:152
    self.env.batch.step(self.action, self.next_state, self.env_reward, self.done, timeout=self.timeout, terminal_f=self.terminal_f, timeout_f=self.timeout_f)  # train.py:153
    reward = self.env_reward
    if self.algorithm == 'PWIL': reward = self.discriminator.compute_reward_batch(self.state, self.action, out=self.store_reward)  # train.py:156
    mem = self.memory.c_struct()
    _lib.check(lib.il_replay_append(h, C.byref(mem), R, self.step_f.data_ptr(), self.state.data_ptr(), self.action.data_ptr(), reward.data_ptr(), self.next_state.data_ptr(),
                                    self.terminal_f.data_ptr(), self.timeout_f.data_ptr(), None, int(self.memory.absorbing), st))  # train.py:157,162
    _lib.check(lib.il_rollout_bookkeep(h, R, self.env_reward.data_ptr(), self.done.data_ptr(), self.running_return.data_ptr(), self.last_return.data_ptr(),
                                       self.return_sum.data_ptr(), self.episodes.data_ptr(), self.step_f.data_ptr(), st))  # train.py:155,165-166
    if self.algorithm == 'PWIL': self.discriminator.reset(mask=self.done)  # train.py:163
    if not self.inject: self.rng.uniform(None, self.device, stream_id=2, out=self.u_reset)
    self.env.batch.reset(self.u_reset, self.state, mask=self.done, else_state=self.next_state)  # train.py:158,168

  # ---- train.py:171-203 -------------------------------------------------------------------------------------------
  def update(self):
    cfg, B = self.cfg, self.B
    uni = None if self.device_rng else (self.u_pol, self.u_exp)
    if not self.inject: self.memory.sample_indices_device(B, out=self.idx_pol, stream_id=3, uniform=None if uni is None else uni[0])
    self.memory.gather(self.idx_pol, out=self.batch)  # train.py:173
    if self.expert_memory is not None:
      if not self.inject: self.expert_memory.sample_indices_device(B, out=self.idx_exp, stream_id=4, uniform=None if uni is None else uni[1])
      self.expert_memory.gather(self.idx_exp, out=self.expert_batch)
    if self.algorithm == 'GAIL':
      from .training import adversarial_imitation_update
      gp_draw = self.grad_penalty_any if self.grad_penalty is not None else cfg.imitation.grad_penalty > 0
      if gp_draw and not self.inject: self.rng.uniform(None, self.device, stream_id=5, out=self.eps_gp)
      eps_mix = None
      if cfg.imitation.loss_function == 'Mixup':  # training.py:106: Beta(a, a) draws; a == 1 (all published configs) is U(0, 1)
        if float(cfg.imitation.mixup_alpha) != 1.0: raise NotImplementedError('mixup_alpha != 1 needs Beta draws; only mixup_alpha = 1 (the reference default) is on the graph-captured path')
        if not self.inject: self.rng.uniform(None, self.device, stream_id=8, out=self.eps_mix)
        eps_mix = self.eps_mix
      self.discriminator.train()  # train.py:178-180
      adversarial_imitation_update(self.actor, self.discriminator, self.batch, self.expert_batch, self.discriminator_optimiser, cfg.imitation, eps_gp=self.eps_gp,
                                   eps_mix=eps_mix, out_losses=self.gail_losses, grad_penalty=self.grad_penalty, entropy_bonus=self.entropy_bonus,
                                   grad_penalty_any=self.grad_penalty_any)
      self.discriminator.eval()
    if self.algorithm in ('GAIL', 'GMMIL'):
      if cfg.imitation.mix_expert_data == 'mixed_batch':
        from .models import mix_expert_agent_transitions
        mix_expert_agent_transitions(self.batch, self.expert_batch)  # train.py:183
      if self.algorithm == 'GAIL': self.discriminator.predict_reward_batch(self.batch, write_rewards=True, actor=self.actor)  # train.py:194
      else: self.discriminator.predict_reward_batch(self.batch, self.expert_batch, reward_out=self.batch.rows[..., self.batch.off['rewards']])  # train.py:196
    if self.algorithm in ('DRIL', 'RED'):  # train.py:183,190-191,196-197
      if cfg.imitation.mix_expert_data == 'mixed_batch':
        from .models import mix_expert_agent_transitions
        mix_expert_agent_transitions(self.batch, self.expert_batch)
      view = self.batch.rows[..., self.batch.off['rewards']]
      if self.algorithm == 'DRIL':
        masks = self.dril_masks if self.inject else None
        self.discriminator.predict_reward(self.batch.rows[..., :self.S], self.batch.rows[..., self.S:self.S + self.A], masks=masks, out=view)
      else: self.discriminator.predict_reward_batch(self.batch, reward_out=view)
    if self.algorithm == 'AdRIL':  # train.py:188-189; `step` of the reference = step_f - 1 here (the rollout has already advanced the counter)
      self.discriminator.resample_and_relabel(self.batch, self.expert_batch, self.step_f, self.memory._num_trajectories, self._expert_trajectories, step_offset=-1.0)
    from .training import sac_update
    if cfg.imitation.bc_aux_loss:  # train.py:201
      from .training import behavioural_cloning_update
      behavioural_cloning_update(self.actor, self.expert_batch, self.actor_optimiser)
    if not self.inject:
      self.rng.normal(None, self.device, stream_id=6, out=self.eps_next)
      self.rng.normal(None, self.device, stream_id=7, out=self.eps_new)
    sac_update(self.actor, self.critic, self.log_alpha, self.target_critic, self.batch, self.actor_optimiser, self.critic_optimiser, self.temperature_optimiser,
               self.discount, self.entropy_target, self.polyak, eps_next=self.eps_next, eps_new=self.eps_new, out=self.sac_out)  # train.py:203

  def bc_pretrain(self, iterations: Optional[int] = None) -> Tensor:
    """train.py:93-99: `iterations` behavioural-cloning steps on epoch-wise shuffled expert minibatches (drop_last), with a
    separate AdamW (bc_pretraining.learning_rate / weight_decay). Every replica draws its own permutations (host RNG, like
    the reference's DataLoader; the exact DataLoader stream is not reproduced). Returns the last per-replica loss."""
    from .training import behavioural_cloning_update
    cfg, B, n = self.cfg, self.B, self.expert_memory.size
    iterations = cfg.bc_pretraining.iterations if iterations is None else iterations
    opt = AdamW(self.actor.parameters(), lr=self.hparams.get('bc_pretraining.learning_rate', cfg.bc_pretraining.learning_rate),
                weight_decay=self.hparams.get('bc_pretraining.weight_decay', cfg.bc_pretraining.weight_decay))
    loss = torch.zeros(self.R, device=self.device)
    per_epoch = max(n // B, 1)
    perm = None
    for it in range(iterations):
      if it % per_epoch == 0: perm = torch.stack([torch.randperm(n) for _ in range(self.R)]).to(self.device, torch.int32)
      j = it % per_epoch
      idx = perm[:, j * B:(j + 1) * B] if n >= B else perm[:, torch.arange(B) % n]
      self.expert_memory.gather(idx.contiguous(), out=self.expert_batch)
      behavioural_cloning_update(self.actor, self.expert_batch, opt, out_loss=loss)
    return loss

  def pretrain_discriminator(self, iterations: Optional[int] = None, batches=None, masks=None, threshold_masks=None):
    """train.py:117-133 for DRIL / RED: `iterations` updates of the dropout policy ensemble (behavioural cloning) / the RED predictor (regression onto its random
    target) on epoch-wise shuffled expert minibatches (every replica draws its own permutations; `batches` injects the index rows instead), then the uncertainty
    threshold (all expert transitions) / the kernel bandwidth (first minibatch) is fixed, and the expert data optionally pre-fills the replay memory."""
    from .training import behavioural_cloning_update, target_estimation_update
    cfg, B, n, d = self.cfg, self.B, self.expert_memory.size, self.discriminator
    iterations = cfg.imitation.pretraining.iterations if iterations is None else iterations
    per_epoch, perm = max(n // B, 1), None
    for it in range(iterations):
      if batches is not None: idx = torch.as_tensor(batches[it], dtype=torch.int32).to(self.device).reshape(-1, B)
      else:
        if it % per_epoch == 0: perm = torch.stack([torch.randperm(n) for _ in range(self.R)]).to(self.device, torch.int32)
        j = it % per_epoch
        idx = perm[:, j * B:(j + 1) * B] if n >= B else perm[:, torch.arange(B) % n]
      self.expert_memory.gather(idx.contiguous(), out=self.expert_batch)
      m = None if masks is None else masks[it]
      if self.algorithm == 'DRIL': behavioural_cloning_update(d, self.expert_batch, self.discriminator_optimiser, masks=m)
      else: target_estimation_update(d, self.expert_batch, self.discriminator_optimiser, masks=m)
    em = self.expert_memory
    if self.algorithm == 'DRIL':
      d.set_uncertainty_threshold(em.rows[0, :, :self.S], em.rows[0, :, self.S:self.S + self.A], self.hparams.get('imitation.quantile_cutoff', cfg.imitation.quantile_cutoff),
                                  masks=threshold_masks)  # train.py:127
    else:
      first = torch.arange(B, dtype=torch.int32, device=self.device).unsqueeze(0).expand(self.R, -1).contiguous() % n
      self.expert_memory.gather(first, out=self.expert_batch)
      d.set_sigma_batch(self.expert_batch, masks=threshold_masks)  # train.py:129: estimated on one minibatch
      d.eval()  # train.py:147
    if cfg.imitation.mix_expert_data == 'prefill_memory': self.memory.transfer_transitions(self.expert_memory)  # train.py:133
    self._pretrained = True

  def _will_update(self, step: int) -> bool:
    return step >= self.cfg.training.start and step % self.cfg.training.interval == 0  # train.py:171

  def _run(self, name: str, fn):
    """Eager for the first calls (lazy allocations, GMMIL bandwidths), then captured as a CUDA graph and replayed."""
    if not self.use_graphs:
      fn()
      return
    g = self.graphs.get(name)
    if g is None:
      n = self.graph_launches.get(name + '#eager', 0)
      if n < 2:
        fn()
        self.graph_launches[name + '#eager'] = n + 1
        return
      torch.cuda.synchronize()
      before = _lib.launch_count()
      g = torch.cuda.CUDAGraph()
      with torch.cuda.graph(g):
        fn()
      self.graph_launches[name] = _lib.launch_count() - before  # kernels recorded into the graph (capture does not execute)
      self.graphs[name] = g
    g.replay()
    self.replayed_launches = getattr(self, 'replayed_launches', 0) + self.graph_launches[name]

  def train_step(self, host_uniform: bool = False):
    """One iteration of the loop at train.py:149: rollout, then (after `training.start`) one update."""
    self.step += 1
    if self._will_update(self.step):
      if not self.device_rng:  # host-drawn index uniforms (the reference draws its indices on the host: memory.py:54)
        if getattr(self, '_pin', None) is None:
          self._pin = [torch.empty(2, self.R, self.B, pin_memory=True) for _ in range(2)]  # double-buffered pinned staging
          self._pin_ev = [None, None]
          self._host_rng = np.random.default_rng(self.seed)  # per-rank stream: seed + first replica of this shard
        slot = self.step & 1
        if self._pin_ev[slot] is not None: self._pin_ev[slot].synchronize()  # the H2D copy that last used this buffer is done
        self._host_rng.random(out=self._pin[slot].numpy(), dtype=np.float32)
        self.u_pol.copy_(self._pin[slot][0], non_blocking=True)
        self.u_exp.copy_(self._pin[slot][1], non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        self._pin_ev[slot] = ev
      self._run('step+update', lambda: (self.rollout(), self.update()))
      self.updates += 1
    else:
      self._run('step', self.rollout)

  def total_launches(self) -> int:
    """Kernels launched by this library for this process (eager launches + kernels replayed through CUDA graphs)."""
    captured = sum(v for k, v in self.graph_launches.items() if not k.endswith('#eager'))
    return _lib.launch_count() - captured + getattr(self, 'replayed_launches', 0)

  def evaluate(self) -> Tensor:
    """train.py:213-219 for all replicas; returns [R, episodes]."""
    r = evaluate_agent(self.actor, self.eval_env, self.cfg.evaluation.episodes)
    return torch.as_tensor(r, device=self.device).reshape(self.R, -1) if self.R == 1 else r

  def log_aux(self):
    """train.py:205-210."""
    m = self.metrics
    m['update_steps'].append(self.step)
    m['predicted_rewards'].append(self.batch['rewards'].cpu().numpy())
    m['alphas'].append(self.log_alpha.exp().cpu().numpy())
    m['entropies'].append((-self.sac_out['log_probs']).cpu().numpy())
    m['Q_values'].append(self.sac_out['q_values'].cpu().numpy())

  def state_dicts(self) -> Dict[str, Dict[str, Tensor]]:
    """train.py:237: agent.pth contents."""
    return dict(actor=self.actor.state_dict(), critic=self.critic.state_dict(), log_alpha=self.log_alpha.detach().clone().cpu())


def train(cfg: Config, file_prefix: str = '') -> float:
  """train.py:26-243 (accelerated algorithms). Multi-GPU: launched one process per GPU (torch.distributed.run); the
  replica axis is split across ranks and evaluation returns are reduced over NCCL (distributed.py)."""
  rank, world = distributed.init('nccl')
  total = int(cfg.get('replicas', 1))
  lo, hi = distributed.shard(total, rank, world)
  keys, values = sweep.setup(cfg)  # hyperparameter search on the replica axis (sweep.space / sweep.trials)
  pbt = sweep.pbt_config(cfg, world)  # population-based training on top of it (sweep.pbt.*); None when off
  hparams, sweep_sums, pbt_records, initial_values = None, [], [], values
  if values is not None:
    hparams = sweep.shard(sweep.replica_hparams(keys, values, total), lo, hi)
    trials_here = sweep.trial_of(total, len(values))[lo:hi]
  trainer = Trainer(cfg, replicas=hi - lo, seed_offset=lo, hparams=hparams, grad_penalty_any=None if pbt is None else pbt['grad_penalty_any'])
  metrics, score = trainer.metrics, trainer.score

  def sweep_eval(normalized, step):
    nonlocal values
    if values is None: return
    sweep_sums.append(sweep.reduce_sums(sweep.trial_sums(normalized, trials_here, len(values))))
    if pbt is not None and len(sweep_sums) % pbt['interval'] == 0 and step + cfg.evaluation.interval <= cfg.steps:  # the final evaluation ranks, it does not exploit
      scores_now = sweep.latest_scores(sweep_sums, len(values))
      parents, values = sweep.pbt_step(pbt, keys, values, scores_now, len(pbt_records))
      trainer.exploit(sweep.replica_map(parents, total)[lo:hi] - lo)  # rank-local: every source of this rank's replicas lives on this rank
      trainer.set_hparams(sweep.shard(sweep.replica_hparams(keys, values, total), lo, hi))
      pbt_records.append(dict(step=step, parents=parents, values=values, scores=scores_now))

  def sweep_save():
    if values is None or rank != 0: return
    if pbt is None: sweep.write_results(file_prefix, keys, values, total // len(values), sweep.scores(sweep_sums, len(values)))
    else: sweep.write_results(file_prefix, keys, values, total // len(values), sweep.latest_scores(sweep_sums, len(values)), pbt=dict(initial=initial_values, records=pbt_records))
  start_time = time.time()
  if cfg.bc_pretraining.iterations > 0:  # train.py:93-112
    trainer.bc_pretrain()
    if cfg.algorithm == 'BC':
      returns = trainer.evaluate()
      mean, std, n = distributed.return_statistics(returns)
      normalized = (returns.cpu().numpy() - trainer.normalization_min) / (trainer.normalization_max - trainer.normalization_min)
      sweep_eval(normalized, 0)
      sweep_save()
      flat = total == 1
      metrics['test_steps'], metrics['test_returns'], metrics['test_returns_normalized'] = [0], [returns.cpu().numpy().reshape(-1).tolist() if flat else returns.cpu().numpy().tolist()], \
          [normalized.reshape(-1).tolist() if flat else normalized.tolist()]
      if rank == 0:
        print(f'BC: test return {mean:.3f} +- {std:.3f} over {n} episodes', flush=True)
        torch.save(dict(actor=trainer.actor.state_dict()), f'{file_prefix}agent.pth')  # train.py:108
        torch.save(metrics, f'{file_prefix}metrics.pth')
      return float(np.mean(normalized))
  if cfg.algorithm in ('DRIL', 'RED'): trainer.pretrain_discriminator()  # train.py:117-133
  for step in range(1, cfg.steps + 1):
    trainer.train_step()
    if cfg.logging.interval > 0 and step % cfg.logging.interval == 0 and trainer._will_update(step): trainer.log_aux()  # train.py:205: only inside the update branch
    if step % cfg.evaluation.interval == 0 and not cfg.check_time_usage:  # train.py:213
      returns = trainer.evaluate()
      mean, std, n = distributed.return_statistics(returns)
      normalized = (returns.cpu().numpy() - trainer.normalization_min) / (trainer.normalization_max - trainer.normalization_min)
      score.append(float((mean - trainer.normalization_min) / (trainer.normalization_max - trainer.normalization_min)))
      sweep_eval(normalized, step)
      metrics['test_steps'].append(step)
      flat = total == 1  # the reference's schema: one list of `episodes` floats per evaluation (train.py:214-219); R > 1 keeps [R][episodes]
      metrics['test_returns'].append(returns.cpu().numpy().reshape(-1).tolist() if flat else returns.cpu().numpy().tolist())
      metrics['test_returns_normalized'].append(normalized.reshape(-1).tolist() if flat else normalized.tolist())
      if rank == 0: print(f'step {step}: test return {mean:.3f} +- {std:.3f} over {n} episodes ({world} rank(s))', flush=True)
  if cfg.check_time_usage: metrics['training_time'] = time.time() - start_time  # train.py:229-230
  eps = trainer.episodes.cpu().numpy()
  metrics['train_returns'] = (trainer.return_sum.cpu().numpy() / np.maximum(eps, 1)).tolist()
  if cfg.save_trajectories:  # train.py:232-235: trajectories of the trained agent (every rank writes its own shard of the replica axis; rank 0 keeps the reference's file name)
    if cfg.render: raise NotImplementedError('render=true needs a PyBullet window (environments.py:52-53); the synthetic device env has none')
    _, trajectories = evaluate_agent(trainer.actor, trainer.eval_env, cfg.evaluation.episodes, return_trajectories=True)
    torch.save(trajectories, f'{file_prefix}trajectories.pth' if rank == 0 else f'{file_prefix}trajectories.rank{rank}.pth')
  if rank == 0:  # train.py:237-239
    torch.save(trainer.state_dicts(), f'{file_prefix}agent.pth')
    if cfg.algorithm in ('DRIL', 'GAIL', 'RED'): torch.save(trainer.discriminator.state_dict(), f'{file_prefix}discriminator.pth')  # train.py:238
    torch.save(metrics, f'{file_prefix}metrics.pth')
  sweep_save()
  return float(np.mean(score)) if score else float('nan')


def main(argv: Optional[List[str]] = None) -> float:
  """`python train.py algorithm=<ALG> env=<ENV> [key=value ...]` (train.py:21-23, 246)."""
  cfg = load_config(sys.argv[1:] if argv is None else argv)
  out_dir = os.path.join(cfg.get('output_dir', './outputs'), f'{cfg.algorithm}_{cfg.env}', time.strftime('%m-%d_%H-%M-%S'))  # conf/train_config.yaml:54-60
  os.makedirs(out_dir, exist_ok=True)
  try:
    return train(cfg, file_prefix=out_dir + os.sep)
  finally:
    distributed.shutdown()
