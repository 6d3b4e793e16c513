"""Cost of population-based training on the flagship workload: GAIL hopper, R = 1024, batch 256, tf32x3, CUDA graphs on, 20 000 ring rows.

In one process: (1) one exploit (Trainer.exploit: il_replica_copy over replica_state()) with 256 destination replicas, against a
device-to-device copy of the same total bytes (one cudaMemcpyAsync of a flat buffer), both timed with CUDA events over many repetitions;
(2) ms/step of a PBT-configured sweep trainer between exploits against the same sweep without PBT, alternated. Prints one JSON line with
the card name and power limit it ran on.

  python scripts/pbt_bench.py [--steps 40] [--rounds 5] [--out FILE]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))

from sweep_bench import SPACE, card  # noqa: E402


def main():
  p = argparse.ArgumentParser()
  p.add_argument('--replicas', type=int, default=1024)
  p.add_argument('--trials', type=int, default=256)
  p.add_argument('--batch-size', type=int, default=256)
  p.add_argument('--memory', type=int, default=20000)
  p.add_argument('--start', type=int, default=300)
  p.add_argument('--steps', type=int, default=40, help='timed steps per round and configuration')
  p.add_argument('--rounds', type=int, default=5)
  p.add_argument('--copies', type=int, default=50, help='timed exploits (and as many reference copies)')
  p.add_argument('--out', help='also append the JSON line to this file')
  a = p.parse_args()
  import numpy as np
  import torch
  from il_b200 import sweep
  from il_b200.config import load_config
  from il_b200.train import Trainer
  R, T = a.replicas, a.trials
  total = a.start + 8 + 2 * a.rounds * a.steps + 64
  cfg = lambda: load_config(['algorithm=GAIL', 'env=hopper', f'steps={max(total, a.memory)}', f'training.start={a.start}', f'training.batch_size={a.batch_size}',
                             'imitation.trajectories=5', f'replicas={R}', 'gemm_mode=tf32x3', f'memory.size={a.memory}', 'seed=0'])
  rng = np.random.default_rng(0)
  keys = list(SPACE)
  values = np.stack([np.exp(rng.uniform(np.log(lo), np.log(hi), T)) if log else rng.uniform(lo, hi, T) for lo, hi, log in SPACE.values()], axis=1)
  hp = lambda: sweep.replica_hparams(keys, values, R)
  trainers = dict(sweep=Trainer(cfg(), replicas=R, fast_init=True, hparams=hp()),
                  pbt=Trainer(cfg(), replicas=R, fast_init=True, hparams=hp(), grad_penalty_any=True))
  for tr in trainers.values():
    for _ in range(a.start + 7): tr.train_step()  # prefill, then warm-up updates incl. the CUDA-graph capture
  torch.cuda.synchronize()
  # (1) one exploit: the bottom quarter of the trials (256 replicas) copy a top trial
  tr = trainers['pbt']
  parents = np.arange(T)
  parents[T - T // 4:] = rng.integers(T // 4, size=T // 4)
  src = sweep.replica_map(parents, R)
  dst = int((src != np.arange(R)).sum())
  state = tr.replica_state()
  per_replica = sum(t[0].numel() * t.element_size() for t in state)
  moved = per_replica * dst
  flat_src, flat_dst = torch.empty(moved, dtype=torch.uint8, device='cuda'), torch.empty(moved, dtype=torch.uint8, device='cuda')
  def timed(fn, n):
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
  # the device part of an exploit (the state copy alone), then the whole call including the host-side map upload and set_hparams
  import ctypes as C
  from il_b200 import _lib
  n = len(state)
  base = (C.c_void_p * n)(*[t.data_ptr() for t in state])
  stride = (C.c_int64 * n)(*[t.stride(0) * 4 for t in state])
  nbytes = (C.c_int64 * n)(*[t[0].numel() * 4 for t in state])
  tr.exploit(src)
  dev_map = tr._src_of
  copy_only = lambda: _lib.check(tr.lib.il_replica_copy(tr.h, n, base, stride, nbytes, R, dev_map.data_ptr(), _lib.stream()))
  rounds_copy, rounds_d2d, rounds_exploit = [], [], []
  for _ in range(3):
    rounds_copy.append(timed(copy_only, a.copies))
    rounds_d2d.append(timed(lambda: flat_dst.copy_(flat_src), a.copies))
    rounds_exploit.append(timed(lambda: tr.exploit(src), max(a.copies // 5, 1)))
  # (2) step time between exploits, alternated
  times = {k: [] for k in trainers}
  for _ in range(a.rounds):
    for name, t in trainers.items(): times[name].append(timed(t.train_step, a.steps))
  med = lambda v: float(np.median(v))
  line = dict(workload=f'GAIL hopper R={R} B={a.batch_size} tf32x3 cuda_graphs memory.size={a.memory}', trials=T, destinations=dst, buffers=n,
              bytes_per_replica=per_replica, bytes_moved=moved, ms_replica_copy=med(rounds_copy), ms_d2d_same_bytes=med(rounds_d2d),
              copy_over_d2d=med(rounds_copy) / med(rounds_d2d), ms_exploit_call=med(rounds_exploit), rounds_ms_replica_copy=rounds_copy, rounds_ms_d2d=rounds_d2d,
              rounds_ms_exploit_call=rounds_exploit, ms_per_step_sweep=med(times['sweep']), ms_per_step_pbt=med(times['pbt']),
              pbt_over_sweep=med(times['pbt']) / med(times['sweep']), rounds_ms_sweep=times['sweep'], rounds_ms_pbt=times['pbt'], card=card())
  s = json.dumps(line)
  print(s, flush=True)
  if a.out:
    with open(a.out, 'a') as f: f.write(s + '\n')


if __name__ == '__main__':
  main()
