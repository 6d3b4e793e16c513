"""Replica-batched hyperparameter search: many trials of the continuous hyperparameters on the replica axis of one run.

`python train.py algorithm=GAIL env=hopper replicas=1024 sweep.space=space.yaml sweep.trials=256` samples 256 trials from a search space in
the reference's Ax layout (conf/hyperparameter_search_space/*.yaml of the reference: `params: {key: {type: range, bounds: [lo, hi],
log_scale: bool} | {type: choice, values: [...]}}`) and runs them as one program: replica r belongs to trial r // (replicas / trials) and keeps
seed `seed + r`, so each trial is scored over replicas / trials seeds. Only hyperparameters that change neither a shape nor the control flow
can differ between replicas (BATCHABLE); the kernels receive them as per-replica arrays. Sampling is uniform (log-uniform with log_scale)
from numpy.random.default_rng(sweep.seed), identical on every rank. The driver samples and ranks; it does not adapt (no Bayesian optimiser).
"""
from __future__ import annotations

import os
from typing import Dict, List, Sequence, Tuple

import numpy as np
import torch
import yaml

# key -> algorithms that read it (None: every algorithm)
BATCHABLE = {
  'training.learning_rate': None,
  'training.weight_decay': None,
  'reinforcement.discount': None,
  'reinforcement.target_temperature': None,
  'reinforcement.polyak_factor': None,
  'imitation.learning_rate': ('DRIL', 'GAIL', 'RED'),
  'imitation.weight_decay': ('DRIL', 'GAIL', 'RED'),
  'imitation.grad_penalty': ('GAIL', ),
  'imitation.entropy_bonus': ('GAIL', ),
  'imitation.reward_scale': ('PWIL', ),
  'imitation.reward_bandwidth_scale': ('PWIL', ),
  'imitation.quantile_cutoff': ('DRIL', ),
  'bc_pretraining.learning_rate': None,
  'bc_pretraining.weight_decay': None,
}


def load_space(path: str, algorithm: str = None) -> Dict[str, dict]:
  """Reads and validates a search space; rejects keys that cannot differ between replicas of one program."""
  with open(path) as f: doc = yaml.safe_load(f) or {}
  params = doc.get('params') if isinstance(doc, dict) else None
  if not isinstance(params, dict) or not params: raise ValueError(f'{path}: expected a non-empty `params:` mapping')
  bad = [k for k in params if k not in BATCHABLE]
  if bad:
    raise ValueError(f'{path}: {", ".join(bad)} cannot vary across the replicas of one run (they change shapes or control flow); '
                     f'batchable keys: {", ".join(BATCHABLE)}')
  if algorithm is not None:
    unused = [k for k in params if BATCHABLE[k] is not None and algorithm not in BATCHABLE[k]]
    if unused: raise ValueError(f'{path}: {", ".join(unused)} not used by algorithm={algorithm}')
  space = {}
  for k, p in params.items():
    kind = p.get('type') if isinstance(p, dict) else None
    if kind == 'range':
      lo, hi = (float(b) for b in p['bounds'])
      log = bool(p.get('log_scale', False))
      if not lo <= hi or (log and lo <= 0): raise ValueError(f'{path}: {k}: bad bounds [{lo}, {hi}]' + (' for log_scale' if log else ''))
      space[k] = dict(type='range', bounds=(lo, hi), log_scale=log)
    elif kind == 'choice':
      values = [float(v) for v in p.get('values') or []]
      if not values: raise ValueError(f'{path}: {k}: choice without values')
      space[k] = dict(type='choice', values=values)
    else:
      raise ValueError(f'{path}: {k}: type must be range or choice, got {kind!r}')
  return space


def sample(space: Dict[str, dict], trials: int, seed: int) -> Tuple[List[str], np.ndarray]:
  """(keys, values [trials, len(keys)] float64): per key in file order, `trials` uniform (log-uniform) draws or choices."""
  rng = np.random.default_rng(seed)
  keys, cols = list(space), []
  for k in keys:
    p = space[k]
    if p['type'] == 'range':
      lo, hi = p['bounds']
      if p['log_scale']: cols.append(np.exp(rng.uniform(np.log(lo), np.log(hi), size=trials)))
      else: cols.append(rng.uniform(lo, hi, size=trials))
    else:
      cols.append(np.asarray(p['values'], dtype=np.float64)[rng.integers(len(p['values']), size=trials)])
  values = np.stack(cols, axis=1) if cols else np.zeros((trials, 0))
  for j, k in enumerate(keys):  # uniform draws lie in [lo, hi); exp(log(.)) may round one ulp outside
    if space[k]['type'] == 'range': values[:, j] = np.clip(values[:, j], *space[k]['bounds'])
  return keys, values


def trial_of(replicas: int, trials: int) -> np.ndarray:
  """[replicas] trial index of every replica: contiguous blocks of replicas / trials seeds."""
  if trials < 1 or replicas % trials != 0: raise ValueError(f'replicas ({replicas}) must be a multiple of sweep.trials ({trials})')
  return np.arange(replicas) // (replicas // trials)


def replica_hparams(keys: Sequence[str], values: np.ndarray, replicas: int, device=None) -> Dict[str, torch.Tensor]:
  """{key: float64 [replicas]} for Trainer(hparams=...)."""
  t = trial_of(replicas, values.shape[0])
  return {k: torch.as_tensor(values[t, j], dtype=torch.float64, device=device) for j, k in enumerate(keys)}


def shard(hparams: Dict[str, torch.Tensor], lo: int, hi: int) -> Dict[str, torch.Tensor]:
  """The slice of every per-replica array owned by one rank (distributed.shard)."""
  return {k: v[lo:hi].contiguous() for k, v in hparams.items()}


def trial_sums(normalized: np.ndarray, trials_of_shard: np.ndarray, trials: int) -> np.ndarray:
  """[2, trials] float64: sum of the normalised returns [local replicas, episodes] of each trial, and their count."""
  n = np.asarray(normalized, dtype=np.float64).reshape(len(trials_of_shard), -1)
  return np.stack([np.bincount(trials_of_shard, weights=n.sum(axis=1), minlength=trials),
                   np.bincount(trials_of_shard, minlength=trials).astype(np.float64) * n.shape[1]])


def reduce_sums(sums: np.ndarray, device=None) -> np.ndarray:
  """Sums over all ranks (one host-side all-reduce per evaluation, outside any graph); identity in a single process."""
  import torch.distributed as dist
  if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1): return sums
  t = torch.as_tensor(sums, dtype=torch.float64, device='cuda' if dist.get_backend() == 'nccl' else 'cpu')
  dist.all_reduce(t, op=dist.ReduceOp.SUM)
  return t.cpu().numpy()


def scores(per_eval_sums: Sequence[np.ndarray], trials: int) -> np.ndarray:
  """[trials]: the mean over evaluations of each trial's mean normalised return (train()'s objective, per trial); NaN without evaluations."""
  if not per_eval_sums: return np.full(trials, np.nan)
  return np.mean([s[0] / np.maximum(s[1], 1) for s in per_eval_sums], axis=0)


def overlay(keys: Sequence[str], row: np.ndarray) -> str:
  """One trial as a global config overlay in the layout of conf/optimised_hyperparameters/."""
  tree: Dict[str, dict] = {}
  for k, v in zip(keys, row):
    node = tree
    parts = k.split('.')
    for p in parts[:-1]: node = node.setdefault(p, {})
    node[parts[-1]] = float(v)
  return '# @package _global_\n' + yaml.safe_dump(tree, default_flow_style=None, sort_keys=True)


def write_results(prefix: str, keys: Sequence[str], values: np.ndarray, seeds_per_trial: int, trial_scores: np.ndarray, top: int = 5) -> dict:
  """sweep.pth (schema below), sweep_best.yaml and a printed ranking; returns the sweep.pth contents."""
  order = [int(i) for i in np.argsort(np.where(np.isfinite(trial_scores), -trial_scores, np.inf), kind='stable')]  # unscored (NaN) trials last
  best = order[0]
  res = dict(trials=int(values.shape[0]), seeds_per_trial=int(seeds_per_trial), keys=list(keys), values=np.asarray(values, dtype=np.float64),
             scores=np.asarray(trial_scores, dtype=np.float64), best=best)
  torch.save(res, f'{prefix}sweep.pth')
  with open(f'{prefix}sweep_best.yaml', 'w') as f: f.write(overlay(keys, values[best]))
  print(f'sweep: {values.shape[0]} trials x {seeds_per_trial} seeds; top {min(top, len(order))}:', flush=True)
  for rank, i in enumerate(order[:top]):
    print(f'  #{rank + 1} trial {i}: score {trial_scores[i]:.4f}  ' + '  '.join(f'{k}={values[i, j]:.6g}' for j, k in enumerate(keys)), flush=True)
  return res


def setup(cfg) -> Tuple[List[str], np.ndarray]:
  """(keys, values [T, K]) of cfg.sweep, or ([], None) without `sweep.space`."""
  sw = cfg.get('sweep') or {}
  if not sw.get('space'): return [], None
  trials = int(sw.get('trials', 1))
  trial_of(int(cfg.get('replicas', 1)), trials)  # validates the replica count
  space = load_space(os.path.expanduser(str(sw['space'])), cfg.algorithm)
  return sample(space, trials, int(sw.get('seed', cfg.seed)))
