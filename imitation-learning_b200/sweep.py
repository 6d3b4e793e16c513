"""Replica-batched hyperparameter search: many trials of the continuous hyperparameters on the replica axis of one run.

`python train.py algorithm=GAIL env=hopper replicas=1024 sweep.space=space.yaml sweep.trials=256` samples 256 trials from a search space in
the reference's Ax layout (conf/hyperparameter_search_space/*.yaml of the reference: `params: {key: {type: range, bounds: [lo, hi],
log_scale: bool} | {type: choice, values: [...]}}`) and runs them as one program: replica r belongs to trial r // (replicas / trials) and keeps
seed `seed + r`, so each trial is scored over replicas / trials seeds. Only hyperparameters that change neither a shape nor the control flow
can differ between replicas (BATCHABLE); the kernels receive them as per-replica arrays. Sampling is uniform (log-uniform with log_scale)
from numpy.random.default_rng(sweep.seed), identical on every rank. The driver samples and ranks; without sweep.pbt it does not adapt (no
Bayesian optimiser).

Population-based training (`sweep.pbt.interval=k`): at every k-th evaluation the bottom `sweep.pbt.fraction` of the trials on each rank copy
the full training state of a uniformly chosen top trial of the same rank (seed j of the bottom block from seed j of the top block, one device
gather: Trainer.exploit), then perturb the copied values (explore): range keys move by +-`perturb` x (hi - lo) in their sampling coordinate
(log for log_scale) and are clipped to the bounds, choice keys move to a neighbouring value in the listed order, and with probability
`resample` a key is redrawn as `sample` draws it. Keys that only act before the training loop (PBT_FROZEN) are inherited and never perturbed.
Trials are scored by their mean normalised return at the latest evaluation. Every decision comes from numpy.random.default_rng([sweep.seed,
exploit index]) and the all-reduced scores, so every rank computes the same ones; no replica state crosses a rank.
"""
from __future__ import annotations

import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import yaml

from . import distributed

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


def _draw(p: dict, rng: np.random.Generator, size: int) -> np.ndarray:
  """`size` uniform (log-uniform) draws or choices of one key."""
  if p['type'] == 'range':
    lo, hi = p['bounds']
    x = np.exp(rng.uniform(np.log(lo), np.log(hi), size=size)) if p['log_scale'] else rng.uniform(lo, hi, size=size)
    return np.clip(x, lo, hi)  # uniform draws lie in [lo, hi); exp(log(.)) may round one ulp outside
  return np.asarray(p['values'], dtype=np.float64)[rng.integers(len(p['values']), size=size)]


def sample(space: Dict[str, dict], trials: int, seed: int) -> Tuple[List[str], np.ndarray]:
  """(keys, values [trials, len(keys)] float64): per key in file order, `trials` uniform (log-uniform) draws or choices."""
  rng = np.random.default_rng(seed)
  keys = list(space)
  cols = [_draw(space[k], rng, trials) for k in keys]
  return keys, (np.stack(cols, axis=1) if cols else np.zeros((trials, 0)))


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


def _ranking(trial_scores: np.ndarray) -> np.ndarray:
  """Trial indices from the best score down; unscored (NaN) trials last, ties in index order."""
  return np.argsort(np.where(np.isfinite(trial_scores), -trial_scores, np.inf), kind='stable')


def write_results(prefix: str, keys: Sequence[str], values: np.ndarray, seeds_per_trial: int, trial_scores: np.ndarray, top: int = 5,
                  pbt: Optional[dict] = None) -> dict:
  """sweep.pth (schema below), sweep_best.yaml and a printed ranking; returns the sweep.pth contents. With population-based training
  `values` are the trials' final values, `trial_scores` those of the final evaluation, and sweep.pth also holds `pbt`: dict(initial=[T, K]
  values, records=[one dict(step, parents [T], values [T, K] after exploring, scores [T]) per exploit])."""
  order = [int(i) for i in _ranking(trial_scores)]
  best = order[0]
  res = dict(trials=int(values.shape[0]), seeds_per_trial=int(seeds_per_trial), keys=list(keys), values=np.asarray(values, dtype=np.float64),
             scores=np.asarray(trial_scores, dtype=np.float64), best=best)
  if pbt is not None: res['pbt'] = pbt
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


# ---- population-based training ------------------------------------------------------------------------------------------------------------
PBT_FROZEN = ('bc_pretraining.learning_rate', 'bc_pretraining.weight_decay', 'imitation.quantile_cutoff')  # act only before the training loop


def populations(replicas: int, trials: int, world: int) -> List[np.ndarray]:
  """The trials of each rank (distributed.shard of the replica axis). A trial's seeds must live on one rank and every rank needs two trials."""
  trial_of(replicas, trials)
  per = replicas // trials
  pops = []
  for rank in range(world):
    lo, hi = distributed.shard(replicas, rank, world)
    if lo % per or hi % per:
      raise ValueError(f'sweep.pbt: rank {rank} holds replicas [{lo}, {hi}), which splits a trial of {per} seeds across ranks; choose replicas, '
                       f'sweep.trials and the GPU count so that every rank holds whole trials')
    if (hi - lo) // per < 2: raise ValueError(f'sweep.pbt: rank {rank} holds {(hi - lo) // per} trial(s); population-based training needs at least 2 per rank')
    pops.append(np.arange(lo // per, hi // per))
  return pops


def pbt_config(cfg, world: int = 1) -> Optional[dict]:
  """The validated sweep.pbt settings (with the search space, the per-rank populations and the seed), or None when sweep.pbt.interval is 0."""
  sw = cfg.get('sweep') or {}
  pb = sw.get('pbt') or {}
  interval = int(pb.get('interval', 0))
  if interval == 0: return None
  if interval < 0: raise ValueError(f'sweep.pbt.interval must be >= 0 (0 = off), got {interval}')
  if not sw.get('space'): raise ValueError('sweep.pbt needs a search space (sweep.space)')
  if cfg.algorithm == 'BC': raise ValueError('sweep.pbt: algorithm=BC has no training loop to adapt (behavioural cloning runs before it)')
  if cfg.get('check_time_usage', False): raise ValueError('sweep.pbt: check_time_usage=true runs no evaluations, so trials cannot be ranked')
  fraction, perturb, resample = float(pb.get('fraction', 0.25)), float(pb.get('perturb', 0.2)), float(pb.get('resample', 0.25))
  if not 0 < fraction <= 0.5: raise ValueError(f'sweep.pbt.fraction must lie in (0, 0.5], got {fraction}')
  if perturb < 0: raise ValueError(f'sweep.pbt.perturb must be >= 0, got {perturb}')
  if not 0 <= resample <= 1: raise ValueError(f'sweep.pbt.resample must lie in [0, 1], got {resample}')
  replicas, trials = int(cfg.get('replicas', 1)), int(sw.get('trials', 1))
  pops = populations(replicas, trials, world)
  space = load_space(os.path.expanduser(str(sw['space'])), cfg.algorithm)
  gp = space.get('imitation.grad_penalty')
  gp_any = None if gp is None else bool(gp['bounds'][1] > 0 if gp['type'] == 'range' else max(gp['values']) > 0)
  return dict(interval=interval, fraction=fraction, perturb=perturb, resample=resample, seed=int(sw.get('seed', cfg.seed)), space=space, populations=pops,
              grad_penalty_any=gp_any)


def pbt_select(scores: np.ndarray, pops: Sequence[np.ndarray], fraction: float, rng: np.random.Generator) -> np.ndarray:
  """parents [T]: in each population the floor(fraction x size) lowest-scored trials (NaN lowest) each copy a uniformly chosen trial of the
  as many highest-scored ones; every other trial is its own parent."""
  scores = np.asarray(scores, dtype=np.float64)
  parents = np.arange(len(scores))
  for pop in pops:
    k = int(np.floor(fraction * len(pop) + 1e-9))
    if k == 0: continue
    order = pop[_ranking(scores[pop])]
    parents[order[len(pop) - k:]] = order[:k][rng.integers(k, size=k)]
  return parents


def replica_map(parents: np.ndarray, replicas: int) -> np.ndarray:
  """[replicas] source replica of every replica: seed j of an exploited trial copies seed j of its parent; a source maps to itself."""
  per = replicas // len(parents)
  r = np.arange(replicas)
  return np.asarray(parents)[r // per] * per + r % per


def pbt_explore(space: Dict[str, dict], keys: Sequence[str], values: np.ndarray, parents: np.ndarray, perturb: float, resample: float,
                rng: np.random.Generator) -> np.ndarray:
  """[T, K]: the parents' values, perturbed on every exploited trial (module docstring); other trials keep theirs."""
  new = np.asarray(values, dtype=np.float64)[parents].copy()
  for t in np.flatnonzero(parents != np.arange(len(parents))):
    for j, k in enumerate(keys):
      if k in PBT_FROZEN: continue
      p = space[k]
      if rng.random() < resample:
        new[t, j] = _draw(p, rng, 1)[0]
        continue
      sign = 1.0 if rng.random() < 0.5 else -1.0
      if p['type'] == 'range':
        lo, hi = p['bounds']
        if p['log_scale']: new[t, j] = np.exp(np.log(new[t, j]) + sign * perturb * (np.log(hi) - np.log(lo)))
        else: new[t, j] = new[t, j] + sign * perturb * (hi - lo)
        new[t, j] = np.clip(new[t, j], lo, hi)
      else:
        vals = p['values']
        i = vals.index(new[t, j]) + int(sign)
        if not 0 <= i < len(vals): i -= 2 * int(sign)  # at an end of the list the only neighbour is inward
        new[t, j] = vals[min(max(i, 0), len(vals) - 1)]
  return new


def pbt_step(pbt: dict, keys: Sequence[str], values: np.ndarray, scores: np.ndarray, index: int) -> Tuple[np.ndarray, np.ndarray]:
  """Exploit number `index`: (parents [T], values [T, K] after exploring)."""
  rng = np.random.default_rng([pbt['seed'], index])
  parents = pbt_select(scores, pbt['populations'], pbt['fraction'], rng)
  return parents, pbt_explore(pbt['space'], keys, values, parents, pbt['perturb'], pbt['resample'], rng)


def latest_scores(per_eval_sums: Sequence[np.ndarray], trials: int) -> np.ndarray:
  """[trials]: each trial's mean normalised return at the latest evaluation; NaN without evaluations."""
  if not per_eval_sums: return np.full(trials, np.nan)
  s = per_eval_sums[-1]
  return s[0] / np.maximum(s[1], 1)


def lineage(res: dict, trial: int) -> List[Tuple[int, np.ndarray]]:
  """The hyperparameter schedule that produced `trial` in a PBT sweep.pth: [(first step, values [K])], starting at step 0 with the initial
  values of its earliest ancestor and adding one entry at every exploit that replaced its line, found by following `parents` back."""
  pbt = res['pbt']
  out, t = [], int(trial)
  for rec in reversed(pbt['records']):
    p = int(rec['parents'][t])
    if p != t: out.append((int(rec['step']), np.asarray(rec['values'][t], dtype=np.float64)))
    t = p
  out.append((0, np.asarray(pbt['initial'][t], dtype=np.float64)))
  return out[::-1]
