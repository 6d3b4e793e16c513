"""Benchmark of the hot path named by BASELINE.json: GAIL Hopper, 1024 replica-envs per GPU (weak scaling over the
replica axis), one full loop iteration per step = rollout (actor forward, env step, replay append) + replay gather x2
+ discriminator update + reward relabel + SAC update, for every replica. Prints ONE JSON line (see the task contract).

  python bench.py --gpus 1 --steps 20 --warmup 3                      # this arm (B200 kernels)
  python bench.py --impl reference --gpus 1 --steps 20 --warmup 3     # the reference's CPU path (oracle port loop)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P bench.py --gpus N ...
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path: sys.path.insert(0, ROOT)

METRIC, UNIT = 'env_steps_per_s', 'env-steps/s'


def parse():
  p = argparse.ArgumentParser()
  p.add_argument('--gpus', type=int, default=1)
  p.add_argument('--steps', type=int, default=100)
  p.add_argument('--warmup', type=int, default=3)
  p.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  p.add_argument('--algorithm', default='GAIL')
  p.add_argument('--env', default='hopper')
  p.add_argument('--replicas', type=int, default=1024, help='replica-envs per GPU')
  p.add_argument('--batch-size', type=int, default=256)
  p.add_argument('--start', type=int, default=300, help='update-free prefill steps before the timed region (training.start)')
  p.add_argument('--gemm-mode', default=os.environ.get('IL_GEMM_MODE', 'tf32x3'), choices=['fp32', 'tf32x3', 'tf32'],
                 help='arithmetic of the 256x256 layers: tf32x3 = 3xTF32 split on tcgen05 (fp32-level accuracy, parity-tested), fp32 = FFMA engine')
  p.add_argument('--total-replicas', type=int, default=1024, help='strong-scaling record: this many replica-envs split over the N ranks (SURVEY §8d config 2)')
  p.add_argument('--eval-episodes', type=int, default=30, help='eval record: greedy episodes per replica (conf/train_config.yaml:23)')
  p.add_argument('--no-strong', action='store_true')
  p.add_argument('--no-eval', action='store_true')
  p.add_argument('--no-e2e', action='store_true')
  p.add_argument('--no-cpu-baseline', action='store_true')
  p.add_argument('--ref-steps-per-step', type=int, default=10, help='reference arm: oracle loop iterations per bench step and worker')
  p.add_argument('--dump-outputs', metavar='DIR', help='after the timed steps, write what the last one computed (rank 0) to DIR/<name>.npy, float32, < 64 MB in all')
  return p.parse_args()


def workload(a):
  return dict(workload=f'{a.algorithm} {a.env}, {a.replicas} replica-envs per GPU (one reference-equivalent agent + env + replay each), batch {a.batch_size}, '
                       f'256x2 actor/critic, conf/algorithm/{a.algorithm}.yaml defaults',
              algorithm=a.algorithm, env=a.env, replicas_per_gpu=a.replicas, batch_size=a.batch_size, parallelism=f'replica-sharded x{a.gpus} (no data-path collective)',
              l2='working set per step (parameters + Adam state + activations, > 8 GB at 1024 replicas) exceeds the 126 MB L2; no flush needed')


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle port loop on the host cores
# ------------------------------------------------------------------------------------------------------------------
def usable_cores():
  """Host cores this process may actually use: affinity mask, capped by the cgroup CPU quota when one is set."""
  n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else (os.cpu_count() or 1)
  try:
    quota, period = open('/sys/fs/cgroup/cpu.max').read().split()
    if quota != 'max': n = max(1, min(n, int(float(quota) / float(period))))
  except Exception:
    pass
  return n


def cpu_reference(a, steps, warmup, procs=None):
  from oracle import loop
  procs = procs or usable_cores()
  per_worker = max(steps * a.ref_steps_per_step, 1)
  r = loop.measure_multiprocess(procs, a.algorithm, a.env, steps=per_worker, warmup=max(warmup, 1), batch_size=a.batch_size, prefill=a.start)
  return r, procs, per_worker


def run_reference(a):
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0: return
  import torch
  r, procs, per_worker = cpu_reference(a, a.steps, a.warmup)
  value = r['steps_per_s']
  line = dict(impl='reference', metric=METRIC, value=value, unit=UNIT, n_gpus=a.gpus, steps=a.steps, warmup=a.warmup, ms_per_step=1e3 * r['seconds'] / a.steps,
              higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32', data='synthetic', config=workload(a), grad_updates_per_s=value,
              cpu_baseline=dict(value=value, unit=UNIT, cores=procs, kind='port',
                                sample=f'{procs} independent single-thread processes (the reference scaling model, train_all.py:26) x {per_worker} loop iterations each of the oracle port '
                                       f'(oracle/loop.py) after {a.start} prefill steps; torch {torch.__version__} CPU'),
              e2e=dict(value=value, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0), gpu_launches=0)
  print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# clocks sampling
# ------------------------------------------------------------------------------------------------------------------
class Clocks:
  FIELDS = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

  def __init__(self, gpu_index):
    self.rows, self.proc, self.gpu, self.mark_idx = [], None, gpu_index, 0

  def start(self):
    try:
      self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.FIELDS}', '--format=csv,noheader,nounits', '-lms', '25', '-i', str(self.gpu)], stdout=subprocess.PIPE,
                                   stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._read, daemon=True).start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout: self.rows.append(line.strip())

  def mark(self):
    """Call at the start of the timed region: only samples taken after this point are reported."""
    self.mark_idx = len(self.rows)

  def stop(self):
    if self.proc is None: return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])
    end_idx = len(self.rows)
    time.sleep(0.05)
    self.proc.terminate()
    rows, note = self.rows[self.mark_idx:max(end_idx, self.mark_idx + 1)], None
    if not rows:  # timed region shorter than the sampling period: fall back to the samples taken under the same load just before it
      rows, note = self.rows[-8:], 'no sample landed inside the timed region; these are the last samples of the warm-up under the same load'
    out = self._summarise(rows)
    if note: out['note'] = note
    return out

  def _summarise(self, rows):
    sm, mx, reasons = [], [], set()
    for r in rows:
      f = [x.strip() for x in r.split(',')]
      if len(f) < 9: continue
      try:
        sm.append(float(f[1])); mx.append(float(f[2]))
      except ValueError:
        continue
      for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
        if v.lower().startswith('active'): reasons.add(name)
    sm.sort()
    return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=sorted(reasons), samples=len(sm))


# ------------------------------------------------------------------------------------------------------------------
# this arm
# ------------------------------------------------------------------------------------------------------------------
def run_b200(a):
  import torch
  import torch.distributed as dist
  import il_b200
  from il_b200 import _lib, distributed
  from il_b200.config import load_config
  from il_b200.train import Trainer
  rank, world = distributed.init('nccl')
  assert world == a.gpus, f'--gpus {a.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run for N > 1)'
  dev = torch.cuda.current_device()
  K, W, R = a.steps, max(a.warmup, 3), a.replicas
  total_steps = a.start + 2 * (W + K) + 64
  cfg = load_config([f'algorithm={a.algorithm}', f'env={a.env}', f'steps={total_steps}', f'training.start={a.start}', f'training.batch_size={a.batch_size}', 'imitation.trajectories=5',
                     f'replicas={R}', f'gemm_mode={a.gemm_mode}', f'memory.size={max(total_steps * 2, 4096)}', 'seed=0'])
  lo, hi = distributed.shard(R * world, rank, world)
  tr = Trainer(cfg, replicas=R, seed_offset=lo, fast_init=True)
  clocks = Clocks(dev)
  clocks.start()  # sampler runs from the prefill on; only samples after clocks.mark() (timed region) are reported
  for _ in range(a.start - 1): tr.train_step()  # update-free prefill (train.py:171), untimed setup
  for _ in range(W): tr.train_step()            # warm-up incl. CUDA-graph capture
  torch.cuda.synchronize()

  def timed(n, e2e=False, trainer=None):
    tr_ = tr if trainer is None else trainer
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # e2e: every step's results (losses, returns) are copied device -> pinned host memory and consumed one step later,
    # so the read-back of step i overlaps the kernels of step i+1 (the host never skips a step's results)
    outs = (tr_.sac_out['losses'], tr_.gail_losses, tr_.last_return)
    pinned = [[torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in outs] for _ in range(2)]
    done = [None, None]
    consumed = 0.0
    distributed.barrier(); torch.cuda.synchronize()
    launches0 = tr_.total_launches()
    ev0.record()
    for i in range(n):
      tr_.train_step()
      if e2e:
        slot = i & 1
        for dst, src in zip(pinned[slot], outs): dst.copy_(src, non_blocking=True)
        done[slot] = torch.cuda.Event(); done[slot].record()
        prev = done[slot ^ 1]
        if prev is not None:
          prev.synchronize()
          consumed += float(pinned[slot ^ 1][0][0, 0])  # host touches the previous step's results
    ev1.record()
    torch.cuda.synchronize(); distributed.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device='cuda')
    if world > 1: dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item()), tr_.total_launches() - launches0

  clocks.mark()
  ms, launches = timed(K)
  clk = clocks.stop()
  value = R * world * K / (ms / 1e3)
  if a.dump_outputs and rank == 0: dump_outputs(tr, a.dump_outputs)  # before the diagnostics below run further steps

  # ---- per-kernel roofline of the dominant kernel (the dense 256x256 grouped GEMMs), measured with CUDA events around
  # each launch on the launching stream during 2 extra eager steps
  roof = None
  try:
    roof = measure_dense_gemm(tr, a)
  except Exception as e:  # never lose the headline number to the diagnostic
    roof = dict(bound='hbm', achieved=None, peak=None, unit='GB/s', frac=None, traffic=None, error=str(e))

  # ---- end-to-end arm: indices' uniforms drawn by numpy on the host and copied H2D every step, results read back every step
  e2e = None
  if not a.no_e2e:
    tr.device_rng = False
    tr.graphs.clear()
    tr.graph_launches = {k: v for k, v in tr.graph_launches.items() if k.endswith('#eager')}
    for _ in range(W): tr.train_step()
    ms_e, _ = timed(K, e2e=True)
    e2e = dict(value=R * world * K / (ms_e / 1e3), unit=UNIT, h2d_bytes_per_step=2 * R * a.batch_size * 4, d2h_bytes_per_step=R * (3 + 2 + 1) * 4, ms_per_step=ms_e / K)

  # ---- evaluation record (SURVEY §8d: "eval excluded from the training rate and reported as eval-steps/s"): il_eval_rollout (device
  # while-loop graph) for episodes x replicas, then the fused return reduction (stats kernel + ncclAllReduce on the same stream)
  ev = None
  if not a.no_eval:
    try:
      ev = measure_eval(tr, a, world)
    except Exception as e:
      ev = dict(error=str(e))
  # ---- strong-scaling record: --total-replicas split over the ranks (at N = 1 it is the weak configuration when totals agree)
  strong = None
  if not a.no_strong:
    try:
      strong = measure_strong(a, world, rank, tr if (world == 1 and a.total_replicas == R) else None, value, ms / K, timed)
    except Exception as e:
      strong = dict(error=str(e))

  cpu = None
  if rank == 0 and world == 1 and not a.no_cpu_baseline:
    r, procs, per_worker = cpu_reference(a, steps=20, warmup=1)
    cpu = dict(value=r['steps_per_s'], unit=UNIT, cores=procs, kind='port',
               sample=f'{procs} single-thread processes x {per_worker} loop iterations of oracle/loop.py ({a.algorithm} {a.env}, batch {a.batch_size}) after {a.start} prefill steps')
  if rank == 0:
    line = dict(metric=METRIC, value=value, unit=UNIT, n_gpus=world, steps=K, warmup=W, ms_per_step=ms / K, higher_is_better=True, scaling='weak', vs_baseline=None, dtype='f32',
                data='synthetic', config=workload(a), grad_updates_per_s=value, clocks=clk, e2e=e2e, gpu_launches=launches, roofline=roof, cpu_baseline=cpu,
                gemm_mode=a.gemm_mode, eval=ev, strong=strong)
    print(json.dumps(line), flush=True)
  distributed.barrier()


DUMP_LIMIT = 1 << 21  # entries kept per array; at most four arrays (the parameter buffers) exceed it, so a dump stays well under 64 MB


def dump_outputs(tr, out_dir):
  """Writes what the last train_step computed, as its caller reads it, to <out_dir>/<name>.npy (float32): the SAC and
  discriminator results of the step, the relabelled rewards of its batch, the last episode returns, log_alpha and the
  parameter buffers ([replicas, P]) the step left behind. An array above DUMP_LIMIT entries keeps a fixed, seeded sample
  of its flattened entries, at the same positions for any build with the same shapes."""
  import numpy as np
  import torch
  torch.cuda.synchronize()
  arrays = dict(sac_log_probs=tr.sac_out['log_probs'], sac_q_values=tr.sac_out['q_values'], sac_losses=tr.sac_out['losses'], gail_losses=tr.gail_losses,
                batch_rewards=tr.batch['rewards'], last_return=tr.last_return, log_alpha=tr.log_alpha)
  for name, mod in (('actor', tr.actor), ('critic', tr.critic), ('target_critic', tr.target_critic), ('discriminator', tr.discriminator)):
    params = mod.parameters() if hasattr(mod, 'parameters') else []
    if params: arrays[f'{name}_params'] = torch.cat([p.reshape(-1) for p in params])
  os.makedirs(out_dir, exist_ok=True)
  for name, t in arrays.items():
    v = t.detach().float().cpu().numpy()
    if v.size > DUMP_LIMIT: v = v.reshape(-1)[np.sort(np.random.default_rng(v.size).choice(v.size, DUMP_LIMIT, replace=False))]
    np.save(os.path.join(out_dir, f'{name}.npy'), v)


def measure_eval(tr, a, world):
  """Times Trainer.evaluate() (evaluation.py:11-35 for every replica: il_eval_rollout) and the return reduction (il_return_allreduce)
  with CUDA events; max over ranks. Episodes end early in the synthetic env, so env steps are counted on the device."""
  import torch
  import torch.distributed as dist
  from il_b200 import distributed
  from il_b200.evaluation import evaluate_agent
  E = a.eval_episodes
  stats = {}
  evaluate_agent(tr.actor, tr.eval_env, E, out_stats=stats)  # warm-up: builds the device graph
  distributed.return_stats_device(torch.zeros(tr.R, E, device='cuda'))
  distributed.barrier(); torch.cuda.synchronize()
  e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
  e0.record()
  returns = evaluate_agent(tr.actor, tr.eval_env, E)
  e1.record()
  out = distributed.return_stats_device(returns if torch.is_tensor(returns) else torch.tensor(returns, device='cuda'))
  e2.record()
  torch.cuda.synchronize()
  evaluate_agent(tr.actor, tr.eval_env, E, out_stats=stats)  # same seeds are not replayed: counters of a like-for-like rollout
  t = torch.tensor([e0.elapsed_time(e1), e1.elapsed_time(e2), float(stats['env_steps']), float(stats['iterations'])], device='cuda', dtype=torch.float64)
  mx = t.clone()
  if world > 1:
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
  rollout_ms, reduce_ms, steps_total, iters = float(mx[0]), float(mx[1]), float(t[2]), float(mx[3])
  mean, std, n = distributed.stats_from_sums(out)
  return dict(metric='eval_steps_per_s', value=steps_total / (rollout_ms / 1e3), unit='env-steps/s', episodes_per_replica=E, replicas_per_gpu=tr.R, env_steps=int(steps_total),
              loop_iterations=int(iters), rollout_ms=rollout_ms, return_allreduce_us=reduce_ms * 1e3, mean_return=mean, std_return=std, episodes=n,
              how='il_eval_rollout: one CUDA graph with a device-side WHILE node (greedy actor forward + env step per iteration, no host sync); il_return_allreduce: '
                  'per-rank (sum, sum^2, n) kernel + ncclAllReduce on the same stream' + (' over the ranks' if world > 1 else ' (single rank: no collective)'))


def measure_strong(a, world, rank, reuse_trainer, weak_value, weak_ms, timed):
  """--total-replicas replica-envs split contiguously over the ranks (SURVEY §8d config 2, §8e): same K timed steps."""
  import torch
  from il_b200 import distributed
  from il_b200.config import load_config
  from il_b200.train import Trainer
  total = a.total_replicas
  lo, hi = distributed.shard(total, rank, world)
  if reuse_trainer is not None:
    return dict(total_replicas=total, replicas_per_gpu=hi - lo, value=weak_value, unit=UNIT, ms_per_step=weak_ms, note='N = 1: identical to the weak-scaling configuration above')
  K, W = a.steps, max(a.warmup, 3)
  total_steps = a.start + 2 * (W + K) + 64
  cfg = load_config([f'algorithm={a.algorithm}', f'env={a.env}', f'steps={total_steps}', f'training.start={a.start}', f'training.batch_size={a.batch_size}', 'imitation.trajectories=5',
                     f'replicas={hi - lo}', f'gemm_mode={a.gemm_mode}', f'memory.size={max(total_steps * 2, 4096)}', 'seed=0'])
  tr = Trainer(cfg, replicas=hi - lo, seed_offset=lo, fast_init=True)
  for _ in range(a.start - 1 + W): tr.train_step()
  torch.cuda.synchronize()
  ms, _ = timed(K, trainer=tr)
  out = dict(total_replicas=total, replicas_per_gpu=hi - lo, value=total * K / (ms / 1e3), unit=UNIT, ms_per_step=ms / K)
  del tr
  torch.cuda.empty_cache()
  return out


def measure_dense_gemm(tr, a):
  import ctypes as C
  import torch
  from il_b200 import _lib
  lib, h = _lib.lib(), tr.h
  if not hasattr(lib, 'il_profile_begin'): return None
  lib.il_profile_begin.argtypes, lib.il_profile_end.argtypes = [C.c_void_p], [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]
  saved = tr.use_graphs
  tr.use_graphs = False
  torch.cuda.synchronize()
  lib.il_profile_begin(h)
  for _ in range(2): tr.train_step()
  torch.cuda.synchronize()
  ms, flops, n = C.c_double(), C.c_double(), C.c_int64()
  lib.il_profile_end(h, C.byref(ms), C.byref(flops), C.byref(n))
  nbytes = C.c_double()
  lib.il_profile_bytes.argtypes = [C.c_void_p, C.POINTER(C.c_double)]
  lib.il_profile_bytes(h, C.byref(nbytes))
  tr.use_graphs = saved
  peaks = {}
  try:
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
  except Exception:
    pass
  bf16 = peaks.get('bf16_tflops_sustained')
  t_peak, t_src = (bf16, 'MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)') if bf16 else (1400.0, 'fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)')
  hbm = peaks.get('hbm_gbs')
  h_peak, h_src = (hbm, 'MEASURED_PEAKS.json hbm_gbs (copy bandwidth)') if hbm else (6500.0, 'fallback 6.5 TB/s (B200_PROFILING.md)')
  if not ms.value > 0: return dict(bound='hbm', achieved=None, peak=h_peak, unit='GB/s', frac=None, traffic=None)
  sec = ms.value * 1e-3
  tflops = flops.value / sec / 1e12
  gbs = nbytes.value / sec / 1e9
  traffic = None
  try:
    traffic = json.load(open(os.path.join(ROOT, 'profiles', 'dense_gemm_traffic.json'))).get('dram_bytes_per_launch')
  except Exception:
    pass
  # Which roof binds: fp32 operands in and out give 2*256^3 flops per 768 KB, i.e. the minimum HBM time of a launch
  # (bytes / peak bandwidth) is ~5x its minimum tensor time at the bf16 dense peak -> the kernel is HBM-bound.
  t_hbm, t_tensor = nbytes.value / (h_peak * 1e9), flops.value / (t_peak * 1e12)
  tensor = dict(achieved=tflops, peak=t_peak, unit='TFLOP/s', frac=tflops / t_peak, peak_source=t_src, arithmetic=a.gemm_mode,
                mma_tflops=tflops * (3 if a.gemm_mode == 'tf32x3' else 1),
                note='tf32x3 issues 3 tf32 MMAs per algorithmic product (fp32-level accuracy); dense tf32 peak is half the bf16 denominator, so the ceiling '
                     'of this arithmetic is peak/6 algorithmic TFLOP/s' if a.gemm_mode == 'tf32x3' else None)
  return dict(bound='hbm' if t_hbm >= t_tensor else 'tensor', kernel='tc_gemm_kernel: grouped dense-layer GEMM (256x256x256 per net, fwd(+head) / dX / dW) of the SAC update',
              achieved=gbs, peak=h_peak, unit='GB/s', frac=gbs / h_peak, traffic=traffic, launches=int(n.value), avg_launch_ms=ms.value / max(n.value, 1),
              algorithmic_bytes_per_launch=nbytes.value / max(n.value, 1), algorithmic_flops_per_launch=flops.value / max(n.value, 1), peak_source=h_src,
              min_time_ratio_hbm_over_tensor=t_hbm / t_tensor, tensor=tensor)


def main():
  a = parse()
  if a.impl == 'reference': run_reference(a)
  else:
    run_b200(a)
    from il_b200 import distributed
    distributed.shutdown()


if __name__ == '__main__':
  main()
