"""Cost of per-replica hyperparameters on the flagship workload: GAIL hopper, R = 1024, batch 256, tf32x3, CUDA graphs on.

Times, in one process and alternating, the uniform configuration (every replica on the config's scalars, the default step of bench.py) and
a 1024-trial sweep in which every GAIL and SAC batchable key differs per replica (the per-replica kernel variants). Prints one JSON line with
ms/step of both, the relative cost, and the card name and power limit it ran on.

  python scripts/sweep_bench.py [--steps 40] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

SPACE = {  # conf/hyperparameter_search_space/GAIL*.yaml of the reference, batchable lines (bounds of the same order)
  'training.learning_rate': (1e-5, 1e-3, True), 'training.weight_decay': (0.0, 1.0, False), 'reinforcement.discount': (0.95, 0.999, False),
  'reinforcement.target_temperature': (-2.0, 0.0, False), 'reinforcement.polyak_factor': (0.95, 0.999, False), 'imitation.learning_rate': (1e-5, 1e-3, True),
  'imitation.weight_decay': (0.0, 10.0, False), 'imitation.grad_penalty': (0.01, 10.0, True), 'imitation.entropy_bonus': (0.0, 1.0, False)}


def card():
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout.strip()
    return q.splitlines()[0]
  except Exception as e:  # noqa: BLE001
    return f'nvidia-smi unavailable ({e})'


def main():
  p = argparse.ArgumentParser()
  p.add_argument('--replicas', type=int, default=1024)
  p.add_argument('--batch-size', type=int, default=256)
  p.add_argument('--start', type=int, default=300)
  p.add_argument('--steps', type=int, default=40, help='timed steps per round and configuration')
  p.add_argument('--rounds', type=int, default=5)
  p.add_argument('--out', help='also append the JSON line to this file')
  a = p.parse_args()
  import numpy as np
  import torch
  from il_b200 import sweep
  from il_b200.config import load_config
  from il_b200.train import Trainer
  R = a.replicas
  total = a.start + 8 + 2 * a.rounds * a.steps + 64
  cfg = lambda: load_config(['algorithm=GAIL', 'env=hopper', f'steps={total}', f'training.start={a.start}', f'training.batch_size={a.batch_size}', 'imitation.trajectories=5',
                             f'replicas={R}', 'gemm_mode=tf32x3', f'memory.size={max(total * 2, 4096)}', 'seed=0'])
  rng = np.random.default_rng(0)
  keys = list(SPACE)
  values = np.stack([np.exp(rng.uniform(np.log(lo), np.log(hi), R)) if log else rng.uniform(lo, hi, R) for lo, hi, log in SPACE.values()], axis=1)
  trainers = dict(uniform=Trainer(cfg(), replicas=R, fast_init=True),
                  sweep=Trainer(cfg(), replicas=R, fast_init=True, hparams=sweep.replica_hparams(keys, values, R)))
  for tr in trainers.values():
    for _ in range(a.start + 7): tr.train_step()  # prefill, then warm-up updates incl. the CUDA-graph capture
  torch.cuda.synchronize()
  times = {k: [] for k in trainers}
  for _ in range(a.rounds):
    for name, tr in trainers.items():
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      torch.cuda.synchronize()
      e0.record()
      for _ in range(a.steps): tr.train_step()
      e1.record()
      torch.cuda.synchronize()
      times[name].append(e0.elapsed_time(e1) / a.steps)
  med = {k: float(np.median(v)) for k, v in times.items()}
  line = dict(workload=f'GAIL hopper R={R} B={a.batch_size} tf32x3 cuda_graphs', trials=R, keys=keys, rounds=a.rounds, steps_per_round=a.steps,
              ms_per_step_uniform=med['uniform'], ms_per_step_sweep=med['sweep'], sweep_over_uniform=med['sweep'] / med['uniform'],
              rounds_ms_uniform=times['uniform'], rounds_ms_sweep=times['sweep'], card=card())
  s = json.dumps(line)
  print(s, flush=True)
  if a.out:
    with open(a.out, 'a') as f: f.write(s + '\n')


if __name__ == '__main__':
  main()
