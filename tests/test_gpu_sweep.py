"""Per-replica hyperparameters on the B200: a replica of a sweep equals, bit for bit, a run configured with its values (AdamW entry points on
both kernel variants, and the whole graph-captured training loop of every algorithm that reads a batchable key), broadcast arrays equal the
scalar path, and the train.py CLI writes a complete sweep result."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# four value sets; every grad_penalty > 0 so every replica draws the same noise as its scalar run
SETS = [
  {'training.learning_rate': 3e-4, 'training.weight_decay': 0.0, 'reinforcement.discount': 0.99, 'reinforcement.target_temperature': -1.0,
   'reinforcement.polyak_factor': 0.995, 'imitation.learning_rate': 3e-4, 'imitation.weight_decay': 0.0, 'imitation.grad_penalty': 1.0, 'imitation.entropy_bonus': 0.0},
  {'training.learning_rate': 1e-3, 'training.weight_decay': 0.01, 'reinforcement.discount': 0.97, 'reinforcement.target_temperature': -0.5,
   'reinforcement.polyak_factor': 0.98, 'imitation.learning_rate': 1e-4, 'imitation.weight_decay': 8.5, 'imitation.grad_penalty': 0.28, 'imitation.entropy_bonus': 0.24},
  {'training.learning_rate': 5e-5, 'training.weight_decay': 1e-4, 'reinforcement.discount': 0.9, 'reinforcement.target_temperature': -2.0,
   'reinforcement.polyak_factor': 0.9, 'imitation.learning_rate': 2e-3, 'imitation.weight_decay': 0.1, 'imitation.grad_penalty': 5.0, 'imitation.entropy_bonus': 1e-3},
  {'training.learning_rate': 2.5e-4, 'training.weight_decay': 0.5, 'reinforcement.discount': 0.999, 'reinforcement.target_temperature': -0.81,
   'reinforcement.polyak_factor': 0.971, 'imitation.learning_rate': 2.8e-4, 'imitation.weight_decay': 0.0, 'imitation.grad_penalty': 0.5, 'imitation.entropy_bonus': 0.5},
]
EXTRA_KEYS = {'PWIL': {'imitation.reward_scale': [5.0, 1.0, 10.0, 0.5], 'imitation.reward_bandwidth_scale': [5.0, 2.0, 0.5, 9.0]},
              'DRIL': {'imitation.quantile_cutoff': [0.98, 0.5, 0.9, 0.2], 'bc_pretraining.learning_rate': [2.5e-4, 1e-3, 1e-4, 5e-4],
                       'bc_pretraining.weight_decay': [0.0, 0.01, 0.1, 0.0]}}
USED = {'SAC': (), 'PWIL': (), 'GAIL': ('imitation.learning_rate', 'imitation.weight_decay', 'imitation.grad_penalty', 'imitation.entropy_bonus'),
        'DRIL': ('imitation.learning_rate', 'imitation.weight_decay'), 'RED': ('imitation.learning_rate', 'imitation.weight_decay')}


def _sets(algorithm):
  keys = [k for k in SETS[0] if not k.startswith('imitation.') or k in USED[algorithm]]
  out = [{k: s[k] for k in keys} for s in SETS]
  for k, vals in EXTRA_KEYS.get(algorithm, {}).items():
    for s, v in zip(out, vals): s[k] = v
  return out


def _cfg(algorithm, extra, overrides=()):
  from il_b200.config import load_config
  return load_config([f'algorithm={algorithm}', 'env=hopper', 'steps=40', 'training.start=21', 'training.batch_size=32', 'imitation.trajectories=2',
                      'reinforcement.actor.hidden_size=64', 'reinforcement.critic.hidden_size=64', 'cuda_graphs=true', 'gemm_mode=tf32x3', 'replicas=4', 'seed=3',
                      'memory.size=64', *extra, *[f'{k}={v}' for k, v in overrides]])


def _run(tr):
  if tr.algorithm in ('DRIL', 'RED'): tr.pretrain_discriminator()
  if tr.cfg.bc_pretraining.iterations > 0: tr.bc_pretrain()
  for _ in range(tr.cfg.steps): tr.train_step()
  torch.cuda.synchronize()
  return tr


def _state(tr):
  """Every parameter / optimiser / output buffer of the trainer, replica-major."""
  out = dict(actor=tr.actor.mlp.flat, critic=tr.critic.mlp.flat, target=tr.target_critic.mlp.flat, log_alpha=tr.log_alpha.reshape(tr.R, 1),
             **{f'sac_{k}': v.reshape(tr.R, -1) for k, v in tr.sac_out.items()})
  for name in ('actor_optimiser', 'critic_optimiser', 'temperature_optimiser', 'discriminator_optimiser'):
    o = getattr(tr, name, None)
    if o is not None: out[name + '.m'], out[name + '.v'] = o.exp_avg.reshape(tr.R, -1), o.exp_avg_sq.reshape(tr.R, -1)
  d = tr.discriminator
  if tr.algorithm == 'GAIL':
    out['disc'] = (d.flat if d.general else d.mlp.flat).reshape(tr.R, -1)
    for n in ('u', 'v', 'g_u', 'g_v', 'h_u', 'h_v'):
      if getattr(d, n, None) is not None: out['disc.' + n] = getattr(d, n).reshape(tr.R, -1)
  elif tr.algorithm == 'DRIL': out['disc'], out['q'] = d.mlp.flat, d._q.reshape(tr.R, 1)
  elif tr.algorithm == 'RED': out['disc'] = d.predictor.flat
  elif tr.algorithm == 'PWIL': out['pwil'] = d.expert_weights
  out['rewards'] = tr.batch.rows[..., tr.batch.off['rewards']].reshape(tr.R, -1)
  return {k: v.detach().clone() for k, v in out.items()}


LOOPS = [('GAIL', ()), ('GAIL', ('imitation.discriminator.reward_shaping=true', 'imitation.discriminator.subtract_log_policy=true')), ('SAC', ()), ('PWIL', ()),
         ('DRIL', ('imitation.pretraining.iterations=5', 'bc_pretraining.iterations=3')), ('RED', ('imitation.pretraining.iterations=5', ))]


@pytest.mark.parametrize('algorithm,extra', LOOPS)
def test_sweep_loop_replica_equals_scalar_run(algorithm, extra):
  """40 graph-captured steps (20 updates), R = 4: replica k of the sweep trainer == replica k of a trainer configured with set k, bit for bit;
  and arrays that broadcast set 0 == the scalar trainer of set 0 on every replica."""
  from il_b200.train import Trainer
  sets = _sets(algorithm)
  keys = list(sets[0])
  sweep = _state(_run(Trainer(_cfg(algorithm, extra), hparams={k: torch.tensor([s[k] for s in sets], dtype=torch.float64) for k in keys})))
  bcast = _state(_run(Trainer(_cfg(algorithm, extra), hparams={k: torch.full((4, ), sets[0][k], dtype=torch.float64) for k in keys})))
  for k in range(4):
    ref = _state(_run(Trainer(_cfg(algorithm, extra, sets[k].items()))))
    for name, t in ref.items():
      assert torch.equal(sweep[name][k], t[k]), f'{algorithm} {extra}: replica {k} differs from its scalar run in {name}'
      if k == 0: assert torch.equal(bcast[name], t), f'{algorithm} {extra}: broadcast arrays differ from the scalar path in {name}'


@pytest.mark.parametrize('extra', [(), ('imitation.discriminator.reward_shaping=true', 'imitation.discriminator.subtract_log_policy=true')])
def test_mixed_zero_and_positive_grad_penalty(extra):
  """grad_penalty 0 on some replicas, > 0 on others, one update with every draw injected: positive replicas equal their scalar runs bit for
  bit. A zero replica equals the zero scalar run bit for bit on the fused discriminator (the penalty pass is chosen per replica) and to the
  single-call tolerance on the general one, except its spectral-norm vectors: the penalty pass runs for all replicas there, and its power
  iteration moves them."""
  from il_b200.train import Trainer
  gps = [0.0, 0.5, 0.0, 2.0]
  def one(tr):
    tr.inject = True
    rs = np.random.RandomState(7)
    for step in range(1, 23):
      tr.eps_act.copy_(torch.from_numpy(rs.standard_normal((4, tr.A)).astype(np.float32)))
      tr.u_reset.copy_(torch.from_numpy(rs.uniform(size=(4, tr.env.obs)).astype(np.float32)))
      if step >= 21:
        tr.idx_pol.copy_(torch.from_numpy(rs.randint(0, step - 2, size=(4, 32)).astype(np.int32)))
        tr.idx_exp.copy_(torch.from_numpy(rs.randint(0, tr.expert_memory.size - 1, size=(4, 32)).astype(np.int32)))
        for b in (tr.eps_gp, tr.eps_next, tr.eps_new): b.copy_(torch.from_numpy(rs.uniform(size=tuple(b.shape)).astype(np.float32)))
      tr.train_step()
    torch.cuda.synchronize()
    return _state(tr)
  base = ('steps=22', 'cuda_graphs=false', *extra)
  sweep = one(Trainer(_cfg('GAIL', base), hparams={'imitation.grad_penalty': torch.tensor(gps, dtype=torch.float64)}))
  general = bool(extra)
  for k, gp in enumerate(gps):
    ref = one(Trainer(_cfg('GAIL', base, [('imitation.grad_penalty', gp)])))
    for name, t in ref.items():
      if gp > 0 or not general: assert torch.equal(sweep[name][k], t[k]), f'replica {k} (gp {gp}) differs in {name}'
      elif name not in ('disc.g_u', 'disc.g_v', 'disc.h_u', 'disc.h_v'):  # the extra power iteration is the expected difference
        torch.testing.assert_close(sweep[name][k], t[k], rtol=2e-4, atol=2e-5, msg=f'replica {k} (gp 0) differs in {name}')


@pytest.mark.parametrize('polyak', [False, True])
@pytest.mark.parametrize('R,n_per', [(4, 70688), (4, 524288), (32, 70688)])
def test_adam_step_entry_points(polyak, R, n_per):
  """il_adam_step / il_adam_step_polyak: broadcast arrays == the scalar call, and replica k of a per-replica call == the scalar call with its
  set, on params, m, v and the target. R x n_per = 4 x 70688: plain kernel; 4 x 524288: TMA-staged kernel, tiles inside one replica;
  32 x 70688 (the actor stride, not a multiple of any tile): TMA-staged kernel with tiles that straddle replica boundaries."""
  import ctypes as C
  from il_b200 import _lib
  from il_b200.optim import AdamW
  g0 = torch.Generator(device='cuda').manual_seed(5)
  p0, t0 = torch.randn(R, n_per, device='cuda', generator=g0), torch.randn(R, n_per, device='cuda', generator=g0)
  grads = [torch.randn(R, n_per, device='cuda', generator=g0) for _ in range(3)]
  lrs, wds = [3e-4, 1e-3, 5e-5, 2.5e-4], [0.0, 0.01, 8.5, 0.5]
  def run(lr, wd):
    p, t = p0.clone(), t0.clone()
    opt = AdamW([p], lr=lr, weight_decay=wd)
    for g in grads:
      a = opt.c_struct()
      if polyak: _lib.check(_lib.lib().il_adam_step_polyak(_lib.handle(), p.data_ptr(), g.data_ptr(), C.byref(a), p.numel(), t.data_ptr(), 0.97, _lib.stream()))
      else: _lib.check(_lib.lib().il_adam_step(_lib.handle(), p.data_ptr(), g.data_ptr(), C.byref(a), p.numel(), _lib.stream()))
    torch.cuda.synchronize()
    return dict(p=p, m=opt.exp_avg, v=opt.exp_avg_sq, t=t)
  per = run(torch.tensor([lrs[r % 4] for r in range(R)], dtype=torch.float64), torch.tensor([wds[r % 4] for r in range(R)], dtype=torch.float64))
  bc = run(torch.full((R, ), lrs[1], dtype=torch.float64), torch.full((R, ), wds[1], dtype=torch.float64))
  for k in range(4):
    ref = run(lrs[k], wds[k])
    for name in ref:
      for r in range(k, R, 4): assert torch.equal(per[name][r], ref[name][r]), f'replica {r}: {name}'
      if k == 1: assert torch.equal(bc[name], ref[name]), f'broadcast: {name}'


class _Injected:
  """Noise source for the oracle loop that replays this step's pre-drawn arrays."""

  def __init__(self, seq): self.seq = seq
  def _pop(self, k): return self.seq[k].pop(0)
  def reset_u(self): return self._pop('reset_u')
  def act_eps(self, A): return self._pop('act_eps')
  def policy_indices(self, mem, n): return self._pop('idx_pol')
  def expert_indices(self, mem, n): return self._pop('idx_exp')
  def gp_eps(self, B): return self._pop('eps_gp')
  def sac_eps(self, B, A): return self._pop('eps_next'), self._pop('eps_new')


def test_sweep_matches_oracle_loop_per_replica():
  """Reference anchor: a 2-replica GAIL hopper sweep (learning rate, discount, polyak factor, target temperature, discriminator learning rate and
  gradient penalty all differ) against oracle/loop.OracleLoop run per replica with that replica's values, every noise draw and index injected
  on both sides, at the loop tolerances (state 2e-3, Q / reward 5e-3, actor 5e-4)."""
  from il_b200.train import Trainer
  from oracle import loop as oloop
  R, B, H, steps, start = 2, 32, 64, 50, 30
  vals = [dict(lr=3e-4, discount=0.97, polyak=0.99, tt=-0.5, ilr=3e-5, gp=1.0), dict(lr=1e-3, discount=0.9, polyak=0.95, tt=-1.5, ilr=3e-4, gp=0.3)]
  keys = {'training.learning_rate': 'lr', 'reinforcement.discount': 'discount', 'reinforcement.polyak_factor': 'polyak', 'reinforcement.target_temperature': 'tt',
          'imitation.learning_rate': 'ilr', 'imitation.grad_penalty': 'gp'}
  cfg = _cfg('GAIL', (f'steps={steps}', f'training.start={start}', 'cuda_graphs=false', 'gemm_mode=fp32', f'replicas={R}', 'memory.size=1000'))
  tr = Trainer(cfg, replicas=R, hparams={k: torch.tensor([v[n] for v in vals], dtype=torch.float64) for k, n in keys.items()})
  tr.inject = True
  rs = np.random.RandomState(123)
  S, A, obs = tr.S, tr.A, tr.env.obs
  expert_raw = tr.env.synthesize_raw_dataset(5)
  loops = []
  for r, v in enumerate(vals):
    d, Hd = S + A, tr.discriminator.mlp.dims[1]
    init = dict(actor=tr.actor.mlp.export_params(r, 0), twin=[tr.critic.mlp.export_params(r, 0), tr.critic.mlp.export_params(r, 1)], g=tr.discriminator.mlp.export_params(r, 0),
                sn=[(tr.discriminator.u[r, :Hd].cpu().clone(), tr.discriminator.v[r, :d].cpu().clone()),
                    (tr.discriminator.u[r, Hd:Hd + 1].cpu().clone(), tr.discriminator.v[r, d:d + Hd].cpu().clone())])
    loops.append(oloop.OracleLoop('GAIL', 'hopper', seed=3 + r, batch_size=B, start=start, memory_size=cfg.memory.size, hidden_size=H, trajectories=2, expert_raw=expert_raw,
                                  init=init, lr=v['lr'], discount=v['discount'], polyak=v['polyak'], target_temperature=v['tt'],
                                  imitation=dict(learning_rate=v['ilr'], grad_penalty=v['gp'])))
  Ne = tr.expert_memory.size
  u0 = rs.uniform(size=(R, obs)).astype(np.float32)
  tr.env.batch.reset(torch.from_numpy(u0).cuda(), tr.state)
  for r, lp in enumerate(loops): lp.state, lp.t = lp.env.reset(torch.from_numpy(u0[r])), 0
  err = {}
  for step in range(1, steps + 1):
    noise = dict(act_eps=rs.standard_normal((R, A)).astype(np.float32), reset_u=rs.uniform(size=(R, obs)).astype(np.float32), eps_gp=rs.uniform(size=(R, B)).astype(np.float32),
                 eps_next=rs.standard_normal((R, B, A)).astype(np.float32), eps_new=rs.standard_normal((R, B, A)).astype(np.float32))
    upd = step >= start
    if upd:
      noise['idx_pol'] = np.stack([rs.randint(0, max(lp.memory.idx - 1, 1), size=B) for lp in loops]).astype(np.int32)
      noise['idx_exp'] = rs.randint(0, Ne - 1, size=(R, B)).astype(np.int32)
    tr.eps_act.copy_(torch.from_numpy(noise['act_eps']))
    tr.u_reset.copy_(torch.from_numpy(noise['reset_u']))
    if upd:
      for name in ('idx_pol', 'idx_exp', 'eps_gp', 'eps_next', 'eps_new'): getattr(tr, name).copy_(torch.from_numpy(noise[name]))
    tr.train_step()
    for r, lp in enumerate(loops):
      seq = {k: [torch.from_numpy(np.asarray(v[r]))] for k, v in noise.items()}
      seq['act_eps'] = [torch.from_numpy(noise['act_eps'][r:r + 1])]
      lp.noise = _Injected(seq)
      lp.run_step()
      err['state'] = max(err.get('state', 0), float((tr.state[r].cpu() - lp.state[0]).abs().max()))
      if upd:
        err['q'] = max(err.get('q', 0), float((tr.sac_out['q_values'][r].cpu() - lp.last['sac']['q_values']).abs().max()))
        err['reward'] = max(err.get('reward', 0), float((tr.batch['rewards'][r].cpu() - lp.last['rewards']).abs().max()))
  for r, lp in enumerate(loops):
    for i, p in enumerate(lp.agent.actor): err['actor'] = max(err.get('actor', 0), float((tr.actor.mlp.layer_views()[0][i][r].cpu() - p.detach()).abs().max()))
  print('sweep vs oracle', err)
  assert err['state'] < 2e-3 and err['q'] < 5e-3 and err['reward'] < 5e-3 and err['actor'] < 5e-4, err


def test_cli_sweep(tmp_path):
  space = tmp_path / 'space.yaml'
  space.write_text('params:\n  training.learning_rate: {type: range, bounds: [1.0e-4, 1.0e-3], log_scale: true}\n'
                   '  reinforcement.discount: {type: range, bounds: [0.95, 0.99]}\n  imitation.grad_penalty: {type: choice, values: [0, 1]}\n')
  out = tmp_path / 'out'
  cmd = [sys.executable, 'train.py', 'algorithm=GAIL', 'env=hopper', 'replicas=8', 'sweep.trials=4', f'sweep.space={space}', 'steps=60', 'training.start=20',
         'evaluation.interval=30', 'evaluation.episodes=2', 'training.batch_size=32', 'imitation.trajectories=2', 'reinforcement.actor.hidden_size=32',
         'reinforcement.critic.hidden_size=32', 'memory.size=100', f'output_dir={out}']
  r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
  assert 'top 4' in r.stdout
  run_dir = next(p for p in out.rglob('sweep.pth')).parent
  res = torch.load(run_dir / 'sweep.pth', weights_only=False)
  assert set(res) == {'trials', 'seeds_per_trial', 'keys', 'values', 'scores', 'best'}
  assert res['trials'] == 4 and res['seeds_per_trial'] == 2 and res['values'].shape == (4, 3) and res['values'].dtype == np.float64
  lr, disc, gp = res['values'].T
  assert ((lr >= 1e-4) & (lr <= 1e-3)).all() and ((disc >= 0.95) & (disc <= 0.99)).all() and set(gp) <= {0.0, 1.0}
  assert np.isfinite(res['scores']).all() and res['best'] == int(np.argmax(res['scores']))
  from il_b200 import sweep
  hp = sweep.replica_hparams(res['keys'], res['values'], 8)
  assert all(torch.equal(v[0::2], v[1::2]) for v in hp.values())  # the two replicas of a trial share their values
  import yaml
  best = yaml.safe_load((run_dir / 'sweep_best.yaml').read_text())
  assert best['training']['learning_rate'] == lr[res['best']] and best['imitation']['grad_penalty'] == gp[res['best']]
