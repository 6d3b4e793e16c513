"""Host-side mirror of the reference's training.py (same function names and argument order); each call is one
C-ABI entry point that runs the whole update for all replicas on the current CUDA stream."""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple, Union

import torch
from torch import Tensor

from . import _lib
from .memory import TransitionBatch
from .models import GAILDiscriminator, SoftActor, TwinCritic, default_rng
from .optim import Adam, Hyper, per_replica

def _workspace(owner, key: str, nbytes: int, device) -> Tensor:
  """Scratch for one fused update, owned by the module that is updated (so two trainers never share it and a buffer whose
  address is baked into a captured CUDA graph is never freed behind the graph's back: a larger request allocates a new
  buffer and the old one stays alive in `owner._ws_retired`). Zero-initialised once: the 4 / 32-float alignment pads of
  the flat gradient buffers are never written by the kernels but are streamed by the AdamW pass."""
  cache = owner.__dict__.setdefault('_ws_cache', {})
  ws = cache.get(key)
  if ws is None or ws.numel() < nbytes:
    if ws is not None: owner.__dict__.setdefault('_ws_retired', []).append(ws)
    ws = torch.zeros(max(nbytes, 256), dtype=torch.uint8, device=device)
    cache[key] = ws
  return ws


def _hyper(owner, key: str, x: Hyper, R: int, device) -> Tuple[float, Optional[Tensor]]:
  """(scalar, per-replica array) of one float hyperparameter: a float keeps the scalar path; a [R] tensor or sequence becomes a float32 device
  array (kept alive on `owner` when it had to be converted, since a captured CUDA graph holds its address) and the scalar field is unused."""
  t = per_replica(x, device)
  if t is None: return float(x), None
  assert t.numel() == R, f'{key}: {t.numel()} per-replica values for {R} replicas'
  if t is not x: owner.__dict__.setdefault('_hp_keep', {})[key] = t
  return 0.0, t


def _as_batch(t: Union[TransitionBatch, Dict[str, Tensor]], device) -> Tuple[TransitionBatch, Optional[Tensor]]:
  if isinstance(t, TransitionBatch): return t, None
  tb = TransitionBatch.from_dict(t, device=device)
  absorbing = None
  if 'absorbing' in t and not tb.absorbing: absorbing = torch.as_tensor(t['absorbing'], dtype=torch.float32).to(device).reshape(tb.R, tb.B).contiguous()
  return tb, absorbing


def sac_update(actor: SoftActor, critic: TwinCritic, log_alpha: Tensor, target_critic: TwinCritic, transitions, actor_optimiser: Adam, critic_optimiser: Adam,
               temperature_optimiser: Adam, discount: Hyper, entropy_target: Hyper, polyak_factor: Hyper, eps_next: Optional[Tensor] = None, eps_new: Optional[Tensor] = None,
               out: Optional[Dict[str, Tensor]] = None) -> Tuple[Tensor, Tensor]:
  """training.py:14-54. `eps_next` / `eps_new` inject the two policy noise draws (:21, :35); when omitted they are
  drawn on the device. Returns (new_log_probs, min(values_1, values_2)) like the reference (:54). `discount`, `entropy_target` and
  `polyak_factor` each take a float or one value per replica ([R])."""
  R, device = actor.replicas, actor.device
  batch, absorbing = _as_batch(transitions, device)
  B, A = batch.B, actor.action_size
  assert batch.R == R and log_alpha.is_cuda and log_alpha.numel() == R
  if eps_next is None: eps_next = default_rng.normal((R, B, A), device, stream_id=11)
  if eps_new is None: eps_new = default_rng.normal((R, B, A), device, stream_id=12)
  eps_next = torch.as_tensor(eps_next, dtype=torch.float32).to(device).reshape(R, B, A).contiguous()
  eps_new = torch.as_tensor(eps_new, dtype=torch.float32).to(device).reshape(R, B, A).contiguous()
  out = {} if out is None else out
  for k, shape in (('log_probs', (R, B)), ('q_values', (R, B)), ('losses', (R, 3))):
    if k not in out: out[k] = torch.empty(shape, device=device)
  a = _lib.SacArgs()
  a.actor, a.critic, a.target = actor.mlp.c_struct(), critic.mlp.c_struct(), target_critic.mlp.c_struct()
  a.actor_opt, a.critic_opt, a.alpha_opt = actor_optimiser.c_struct(), critic_optimiser.c_struct(), temperature_optimiser.c_struct()
  a.log_alpha, a.batch = log_alpha.data_ptr(), batch.c_struct()
  a.absorbing, a.absorbing_from_state, a.R = _lib.ptr(absorbing), int(batch.absorbing and absorbing is None), R
  a.eps_next, a.eps_new = eps_next.data_ptr(), eps_new.data_ptr()
  (a.discount, disc_r), (a.entropy_target, ent_r), (a.polyak_factor, pol_r) = (_hyper(actor, k, x, R, device) for k, x in
                                                                              (('discount', discount), ('entropy_target', entropy_target), ('polyak_factor', polyak_factor)))
  a.discount_r, a.entropy_target_r, a.polyak_r = _lib.ptr(disc_r), _lib.ptr(ent_r), _lib.ptr(pol_r)
  a.out_log_probs, a.out_q_values, a.out_losses = out['log_probs'].data_ptr(), out['q_values'].data_ptr(), out['losses'].data_ptr()
  need = _lib.lib().il_sac_workspace_bytes(C.byref(a))
  ws = _workspace(actor, 'sac', need, device)
  a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
  _lib.check(_lib.lib().il_sac_update(_lib.handle(), C.byref(a), _lib.stream()))
  sq = (lambda t: t[0]) if R == 1 else (lambda t: t)
  return sq(out['log_probs']), sq(out['q_values'])


def adversarial_imitation_update(actor: SoftActor, discriminator: GAILDiscriminator, transitions, expert_transitions, discriminator_optimiser: Adam, imitation_cfg,
                                 eps_gp: Optional[Tensor] = None, eps_mix: Optional[Tensor] = None, out_losses: Optional[Tensor] = None,
                                 grad_penalty: Optional[Hyper] = None, entropy_bonus: Optional[Hyper] = None, grad_penalty_any: Optional[bool] = None):
  """training.py:85-134. `eps_gp` injects the U(0,1) draw of :118 and `eps_mix` the Beta draw of :106. `grad_penalty` / `entropy_bonus`
  override imitation_cfg's values with a float or one value per replica ([R]). With per-replica gradient penalties, whether any replica has
  one (the general discriminator runs the penalty pass for all replicas or none) is `grad_penalty_any`, a host decision: when omitted it is
  read from the values once per array, which cannot happen during CUDA-graph capture."""
  R, device = discriminator.replicas, discriminator.device
  pol, _ = _as_batch(transitions, device)
  exp, _ = _as_batch(expert_transitions, device)
  B = pol.B
  loss_function = imitation_cfg.loss_function
  gp, gp_r = _hyper(discriminator, 'grad_penalty', imitation_cfg.grad_penalty if grad_penalty is None else grad_penalty, R, device)
  eb, eb_r = _hyper(discriminator, 'entropy_bonus', imitation_cfg.entropy_bonus if entropy_bonus is None else entropy_bonus, R, device)
  if gp_r is not None:  # the scalar field carries the pass decision of the general discriminator
    if grad_penalty_any is None:
      cache = discriminator.__dict__.setdefault('_gp_any', {})
      key = (gp_r.data_ptr(), gp_r.numel())
      if key not in cache: cache[key] = bool((gp_r > 0).any())
      grad_penalty_any = cache[key]
    gp = 1.0 if grad_penalty_any else 0.0
  if (gp > 0 or gp_r is not None) and eps_gp is None: eps_gp = default_rng.uniform((R, B), device, stream_id=21)
  if loss_function == 'Mixup' and eps_mix is None:
    alpha = float(imitation_cfg.mixup_alpha)  # training.py:106
    if alpha == 1.0: eps_mix = default_rng.uniform((R, B), device, stream_id=22)  # Beta(1, 1) = U(0, 1): every published config uses mixup_alpha 1
    else: eps_mix = torch.distributions.Beta(torch.full((R, B), alpha, device=device), torch.full((R, B), alpha, device=device)).sample()
  as_dev = lambda t: None if t is None else torch.as_tensor(t, dtype=torch.float32).to(device).reshape(R, B).contiguous()
  eps_gp, eps_mix = as_dev(eps_gp), as_dev(eps_mix)
  if discriminator.general:
    return _general_adversarial_update(actor, discriminator, pol, exp, discriminator_optimiser, imitation_cfg, eps_gp, eps_mix, out_losses, (gp, gp_r, eb, eb_r))
  a = _lib.GailUpdateArgs()
  a.disc, a.opt, a.policy, a.expert = discriminator.c_struct(), discriminator_optimiser.c_struct(), pol.c_struct(), exp.c_struct()
  a.eps_gp, a.eps_mix, a.R, a.loss_function, a.training = _lib.ptr(eps_gp), _lib.ptr(eps_mix), R, _lib.LOSS[loss_function], int(discriminator.training)
  a.grad_penalty, a.entropy_bonus, a.grad_penalty_r, a.entropy_bonus_r = gp, eb, _lib.ptr(gp_r), _lib.ptr(eb_r)
  a.pos_class_prior, a.nonnegative_margin = float(imitation_cfg.pos_class_prior), float(imitation_cfg.nonnegative_margin)
  a.out_losses = _lib.ptr(out_losses)
  _lib.check(_lib.lib().il_gail_update(_lib.handle(), C.byref(a), _lib.stream()))


def _general_adversarial_update(actor, disc: GAILDiscriminator, pol: TransitionBatch, exp: TransitionBatch, opt: Adam, imitation_cfg, eps_gp, eps_mix, out_losses, hyper):
  """training.py:85-134 for the non-default discriminator configurations (reward shaping, subtract_log_policy, depth > 1, tanh / sigmoid):
  the log-policy inputs of make_gail_input (models.py:148, evaluated under no_grad) are computed first, then one il_gailx_update call."""
  R, B, device, lib = disc.replicas, pol.B, disc.device, _lib.lib()
  loss_function = imitation_cfg.loss_function
  logp = {}
  if disc.subtract_log_policy:
    lp = lambda tb: actor._run(tb.rows[..., :tb.S], given=tb.rows[..., tb.S:tb.S + tb.A], want=('log_prob', ))['log_prob']
    if loss_function == 'Mixup':  # make_gail_input on the mixed state / action (training.py:107-108)
      mix = TransitionBatch(torch.empty_like(pol.rows), pol.S, pol.A, pol.absorbing)
      e, p_, m = exp.c_struct(), pol.c_struct(), mix.c_struct()
      _lib.check(lib.il_gail_mix_batch(_lib.handle(), C.byref(e), C.byref(p_), eps_mix.data_ptr(), R, C.byref(m), _lib.stream()))
      logp['mix'] = lp(mix)
    else:
      logp['policy'], logp['expert'] = lp(pol), lp(exp)
  a = _lib.GailxUpdateArgs()
  a.disc, a.opt, a.params_floats, a.policy, a.expert = disc.cx_struct(), opt.c_struct(), disc.flat.numel(), pol.c_struct(), exp.c_struct()
  a.eps_gp, a.eps_mix = _lib.ptr(eps_gp), _lib.ptr(eps_mix)
  a.logp_policy, a.logp_expert, a.logp_mix = _lib.ptr(logp.get('policy')), _lib.ptr(logp.get('expert')), _lib.ptr(logp.get('mix'))
  a.R, a.loss_function, a.training = R, _lib.LOSS[loss_function], int(disc.training)
  gp, gp_r, eb, eb_r = hyper
  a.grad_penalty, a.entropy_bonus, a.grad_penalty_r, a.entropy_bonus_r = gp, eb, _lib.ptr(gp_r), _lib.ptr(eb_r)
  a.pos_class_prior, a.nonnegative_margin = float(imitation_cfg.pos_class_prior), float(imitation_cfg.nonnegative_margin)
  a.out_losses = _lib.ptr(out_losses)
  need = lib.il_gailx_workspace_bytes(C.byref(a))
  ws = _workspace(disc, 'gailx', need, device)
  a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
  _lib.check(lib.il_gailx_update(_lib.handle(), C.byref(a), _lib.stream()))


def behavioural_cloning_update(actor: SoftActor, expert_transition, actor_optimiser: Adam, out_loss: Optional[Tensor] = None, masks=None):
  """training.py:57-64: one maximum-likelihood step of the actor on expert (state, action, weight) rows. A policy with dropout in train mode (DRIL's
  ensemble, train.py:120) runs on the dropout program; `masks` injects its dropout draws ([input mask, hidden masks...], pre-scaled)."""
  R, device = actor.replicas, actor.device
  batch, _ = _as_batch(expert_transition, device)
  a = _lib.BcArgs()
  a.actor, a.opt, a.batch, a.R, a.out_loss = actor.mlp.c_struct(), actor_optimiser.c_struct(), batch.c_struct(), R, _lib.ptr(out_loss)
  if getattr(actor, 'has_dropout', False) and (actor.training or masks is not None):
    if masks is None: masks = actor.draw_masks(batch.B)
    masks = [None if m is None else torch.as_tensor(m, dtype=torch.float32).to(device).reshape(R, batch.B, -1).contiguous() for m in masks]
    need = _lib.lib().il_actor_dropout_workspace_bytes(C.byref(a.actor), R, batch.B)
    ws = _workspace(actor, 'bc_dropout', need, device)
    a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
    _lib.check(_lib.lib().il_bc_update_dropout(_lib.handle(), C.byref(a), _lib.ptr(masks[0]), _lib.mask_array(masks[1:]), _lib.stream()))
    return
  need = _lib.lib().il_bc_workspace_bytes(C.byref(a))
  ws = _workspace(actor, 'bc', need, device)
  a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
  _lib.check(_lib.lib().il_bc_update(_lib.handle(), C.byref(a), _lib.stream()))


def target_estimation_update(discriminator, expert_transition, discriminator_optimiser: Adam, out_loss: Optional[Tensor] = None, masks=None):
  """training.py:68-75: one regression step of RED's predictor onto its frozen random target on expert rows (dropout masks drawn on the device in train mode,
  or injected through `masks`)."""
  R, device = discriminator.replicas, discriminator.device
  batch, _ = _as_batch(expert_transition, device)
  if masks is None and discriminator.training and (discriminator.input_dropout > 0 or discriminator.dropout > 0): masks = discriminator.draw_masks(batch.B)
  masks = [None if m is None else torch.as_tensor(m, dtype=torch.float32).to(device).reshape(R, batch.B, -1).contiguous() for m in (masks or [None] * discriminator.predictor.n_layers)]
  a = _lib.RedUpdateArgs()
  a.disc, a.opt, a.batch, a.R = discriminator.c_struct(), discriminator_optimiser.c_struct(), batch.c_struct(), R
  a.mask_in = _lib.ptr(masks[0])
  for i, m in enumerate(masks[1:]): a.mask_hid[i] = _lib.ptr(m)
  a.out_loss = _lib.ptr(out_loss)
  ws = discriminator.workspace(batch.B)
  a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
  _lib.check(_lib.lib().il_red_update(_lib.handle(), C.byref(a), _lib.stream()))
