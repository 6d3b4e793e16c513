"""Population-based training on the B200: il_replica_copy against torch indexing (eagerly and replayed from a CUDA graph with a rewritten
map), clone completeness of Trainer.exploit for every accelerated loop (a destination equals its source bit for bit when fed the same
noise), completeness of Trainer.replica_state(), in-place Trainer.set_hparams (eager and mid-run under CUDA graphs), and the train.py CLI."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _copy(bufs, src_of):
  """il_replica_copy over [R, ...] tensors (possibly column slices: `bytes` < `stride`)."""
  from il_b200 import _lib
  n, R = len(bufs), bufs[0].size(0)
  base = (C.c_void_p * n)(*[t.data_ptr() for t in bufs])
  stride = (C.c_int64 * n)(*[t.stride(0) * t.element_size() for t in bufs])
  nbytes = (C.c_int64 * n)(*[t[0].numel() * t.element_size() for t in bufs])
  _lib.check(_lib.lib().il_replica_copy(_lib.handle(), n, base, stride, nbytes, R, src_of.data_ptr(), _lib.stream()))


def _random_buffers(rs, n, R):
  """n [R, ...] buffers: 16-byte aligned rows, 4-byte aligned rows (odd float counts), column slices whose length is not a multiple of 16 B,
  int32 counters and [R] scalars; one large buffer spans many work items."""
  out = []
  for i in range(n):
    kind = i % 5
    if kind == 0: out.append(torch.randn(R, int(rs.randint(1, 600)) * 4, device='cuda'))
    elif kind == 1: out.append(torch.randn(R, int(rs.randint(1, 3000)) | 1, device='cuda'))
    elif kind == 2: out.append(torch.randn(R, 70, device='cuda')[:, 1:1 + int(rs.randint(1, 69))])
    elif kind == 3: out.append(torch.randint(-2**31, 2**31 - 1, (R, ), dtype=torch.int32, device='cuda'))
    else: out.append(torch.randn(R, device='cuda'))
  if n > 1: out[1] = torch.randn(R, 40000 + 7, device='cuda')
  return out


def _reference(bufs, m):
  idx = torch.as_tensor(m, dtype=torch.long, device='cuda')
  return [t[idx].clone() for t in bufs]


@pytest.mark.parametrize('nbufs', [1, 2, 7, 64])
def test_replica_copy_matches_torch_indexing(nbufs):
  rs = np.random.RandomState(nbufs)
  R = 9
  bufs = _random_buffers(rs, nbufs, R)
  m = np.array([0, 1, 1, 3, 0, 5, 3, 7, 7], dtype=np.int32)  # identity entries 0, 1, 3, 5, 7; every source is its own source
  want = _reference(bufs, m)
  before = [t.clone() for t in bufs]
  _copy(bufs, torch.from_numpy(m).cuda())
  torch.cuda.synchronize()
  for t, w, b in zip(bufs, want, before):
    assert torch.equal(t, w)
    for r in np.flatnonzero(m == np.arange(R)): assert torch.equal(t[r], b[r])  # identity replicas untouched


def test_replica_copy_bytes_outside_rows_untouched():
  """Column slices: the bytes between `bytes` and `stride` of every row keep their values."""
  R = 6
  parent = torch.randn(R, 37, device='cuda')
  keep = parent.clone()
  m = np.array([0, 0, 2, 2, 4, 4], dtype=np.int32)
  _copy([parent[:, 3:30]], torch.from_numpy(m).cuda())
  torch.cuda.synchronize()
  assert torch.equal(parent[:, :3], keep[:, :3]) and torch.equal(parent[:, 30:], keep[:, 30:])
  assert torch.equal(parent[:, 3:30], keep[torch.as_tensor(m, dtype=torch.long, device='cuda'), 3:30])


def test_replica_copy_graph_replay_after_map_rewrite():
  rs = np.random.RandomState(3)
  R = 8
  bufs = _random_buffers(rs, 12, R)
  src = torch.arange(R, dtype=torch.int32, device='cuda')
  eager = [t.clone() for t in bufs]
  g = torch.cuda.CUDAGraph()
  s = torch.cuda.Stream()
  s.wait_stream(torch.cuda.current_stream())
  with torch.cuda.stream(s):
    _copy(bufs, src)  # warm-up outside the capture (identity map: nothing moves)
    with torch.cuda.graph(g, stream=s):
      _copy(bufs, src)
  torch.cuda.current_stream().wait_stream(s)
  torch.cuda.synchronize()
  for t, e in zip(bufs, eager): assert torch.equal(t, e)
  for m in ([2, 2, 2, 3, 4, 4, 6, 2], [0, 0, 0, 0, 7, 7, 7, 7]):
    m = np.asarray(m, dtype=np.int32)
    src.copy_(torch.from_numpy(m))
    _copy(eager, torch.from_numpy(m).cuda())
    g.replay()
    torch.cuda.synchronize()
    for t, e in zip(bufs, eager): assert torch.equal(t, e)


def test_replica_copy_rejects_bad_arguments():
  from il_b200 import _lib
  t = torch.randn(4, 8, device='cuda')
  src = torch.arange(4, dtype=torch.int32, device='cuda')
  one = lambda stride, nbytes, nb=1: _lib.lib().il_replica_copy(_lib.handle(), nb, (C.c_void_p * 1)(t.data_ptr()), (C.c_int64 * 1)(stride), (C.c_int64 * 1)(nbytes),
                                                                  4, src.data_ptr(), _lib.stream())
  assert one(32, 64) != 0 and 'stride' in _lib.last_error()
  assert one(32, 30) != 0 and 'aligned' in _lib.last_error()
  assert one(32, 32, 0) != 0 and one(32, 32, 65) != 0
  assert one(32, 32) == 0


# ---- Trainer -------------------------------------------------------------------------------------------------------------------------------
HSETS = [
  {'training.learning_rate': 3e-4, 'training.weight_decay': 0.0, 'reinforcement.discount': 0.99, 'reinforcement.target_temperature': -1.0,
   'reinforcement.polyak_factor': 0.995, 'imitation.learning_rate': 3e-4, 'imitation.weight_decay': 0.0, 'imitation.grad_penalty': 1.0, 'imitation.entropy_bonus': 0.0},
  {'training.learning_rate': 1e-3, 'training.weight_decay': 0.01, 'reinforcement.discount': 0.97, 'reinforcement.target_temperature': -0.5,
   'reinforcement.polyak_factor': 0.98, 'imitation.learning_rate': 1e-4, 'imitation.weight_decay': 8.5, 'imitation.grad_penalty': 0.28, 'imitation.entropy_bonus': 0.24},
  {'training.learning_rate': 5e-5, 'training.weight_decay': 1e-4, 'reinforcement.discount': 0.9, 'reinforcement.target_temperature': -2.0,
   'reinforcement.polyak_factor': 0.9, 'imitation.learning_rate': 2e-3, 'imitation.weight_decay': 0.1, 'imitation.grad_penalty': 5.0, 'imitation.entropy_bonus': 1e-3},
  {'training.learning_rate': 2.5e-4, 'training.weight_decay': 0.5, 'reinforcement.discount': 0.999, 'reinforcement.target_temperature': -0.81,
   'reinforcement.polyak_factor': 0.971, 'imitation.learning_rate': 2.8e-4, 'imitation.weight_decay': 0.0, 'imitation.grad_penalty': 0.5, 'imitation.entropy_bonus': 0.5},
  {'training.learning_rate': 7e-4, 'training.weight_decay': 0.2, 'reinforcement.discount': 0.95, 'reinforcement.target_temperature': -1.5,
   'reinforcement.polyak_factor': 0.99, 'imitation.learning_rate': 5e-5, 'imitation.weight_decay': 1.0, 'imitation.grad_penalty': 2.0, 'imitation.entropy_bonus': 0.1},
]
EXTRA = {'PWIL': {'imitation.reward_scale': [5.0, 1.0, 10.0, 0.5, 2.0], 'imitation.reward_bandwidth_scale': [5.0, 2.0, 0.5, 9.0, 1.0]},
         'DRIL': {'imitation.quantile_cutoff': [0.98, 0.5, 0.9, 0.2, 0.7]}}
USED = {'GAIL': ('imitation.learning_rate', 'imitation.weight_decay', 'imitation.grad_penalty', 'imitation.entropy_bonus'),
        'DRIL': ('imitation.learning_rate', 'imitation.weight_decay'), 'RED': ('imitation.learning_rate', 'imitation.weight_decay')}
GENERAL = ('imitation.discriminator.reward_shaping=true', 'imitation.discriminator.subtract_log_policy=true')
PRE = ('imitation.pretraining.iterations=3', )
LOOPS = [('GAIL', ()), ('GAIL', GENERAL), ('SAC', ()), ('PWIL', ()), ('GMMIL', ()), ('DRIL', PRE), ('RED', PRE), ('AdRIL', ())]
LOOP_IDS = ['GAIL-fused', 'GAIL-general', 'SAC', 'PWIL', 'GMMIL', 'DRIL', 'RED', 'AdRIL']


def _hparams(algorithm, R, shift=0):
  """{key: float64 [R]}: replica r takes value set (r + shift) % 5 of every key the algorithm reads."""
  keys = [k for k in HSETS[0] if not k.startswith('imitation.') or k in USED.get(algorithm, ())]
  out = {k: torch.tensor([HSETS[(r + shift) % 5][k] for r in range(R)], dtype=torch.float64) for k in keys}
  for k, vals in EXTRA.get(algorithm, {}).items(): out[k] = torch.tensor([vals[(r + shift) % 5] for r in range(R)], dtype=torch.float64)
  return out


def _cfg(algorithm, extra, R, steps, graphs=True):
  from il_b200.config import load_config
  return load_config([f'algorithm={algorithm}', 'env=hopper', f'steps={steps}', 'training.start=11', 'training.batch_size=32', 'imitation.trajectories=2',
                      'reinforcement.actor.hidden_size=64', 'reinforcement.critic.hidden_size=64', f'cuda_graphs={str(graphs).lower()}', 'gemm_mode=tf32x3',
                      f'replicas={R}', 'seed=3', 'memory.size=128', *extra])


def _trainer(algorithm, extra, R, steps, graphs=True, shift=0):
  from il_b200.train import Trainer
  tr = Trainer(_cfg(algorithm, extra, R, steps, graphs), hparams=_hparams(algorithm, R, shift))
  tr.inject = True
  if algorithm == 'DRIL':  # persistent injected dropout masks of the ensemble pass ([R, 5 B, width]); graphs hold their addresses
    d, n = tr.discriminator, 5 * tr.B
    tr.dril_masks = [None if p <= 0 else torch.ones(R, n, w, device='cuda') for w, p in
                     [(d.state_size, d.input_dropout)] + [(d.mlp.dims[l + 1], d.dropout) for l in range(d.mlp.n_layers - 1)]]
  if algorithm in ('DRIL', 'RED'): tr.pretrain_discriminator()
  return tr


def _feed(tr, rs, step, src):
  """Fill every injected noise / index buffer for the coming step; replica r gets the draws of replica src[r]."""
  R, B = tr.R, tr.B
  idx = torch.as_tensor(src, dtype=torch.long)
  put = lambda buf, x: buf.copy_(torch.from_numpy(x)[idx].to(buf.dtype))
  put(tr.eps_act, rs.standard_normal((R, tr.A)).astype(np.float32))
  put(tr.u_reset, rs.uniform(size=(R, tr.env.obs)).astype(np.float32))
  if tr._will_update(step):
    put(tr.idx_pol, rs.randint(0, max(min(step - 1, tr.memory.size) - 1, 1), size=(R, B)).astype(np.int32))
    if tr.expert_memory is not None: put(tr.idx_exp, rs.randint(0, tr.expert_memory.size - 1, size=(R, B)).astype(np.int32))
    for b in (tr.eps_gp, tr.eps_mix): put(b, rs.uniform(size=tuple(b.shape)).astype(np.float32))
    for b in (tr.eps_next, tr.eps_new): put(b, rs.standard_normal(tuple(b.shape)).astype(np.float32))
    for mk in tr.dril_masks or []:
      if mk is not None: put(mk, (rs.uniform(size=tuple(mk.shape)) > 0.1).astype(np.float32) / 0.9)


def _outputs(tr):
  return [tr.sac_out['log_probs'], tr.sac_out['q_values'], tr.sac_out['losses'], tr.batch.rows[..., tr.batch.off['rewards']].contiguous()]


@pytest.mark.parametrize('algorithm,extra', LOOPS, ids=LOOP_IDS)
def test_exploit_clones_replica_state(algorithm, extra):
  """R = 4, distinct hyperparameters, graphs on: after the capture, exploit({2: 0, 3: 1}), then 12 more graph-replayed steps with each
  destination fed its source's noise: every replica_state() tensor, the SAC outputs and the relabelled rewards of replica 2 equal replica 0
  and those of 3 equal 1, bit for bit; the graphs were neither re-captured nor extended."""
  R, steps = 4, 30
  tr = _trainer(algorithm, extra, R, steps)
  rs = np.random.RandomState(11)
  ident = np.arange(R)
  for step in range(1, 19):
    _feed(tr, rs, step, ident)
    tr.train_step()
  assert 'step+update' in tr.graphs
  graphs, launches = dict(tr.graphs), dict(tr.graph_launches)
  before = [t.clone() for t in tr.replica_state()]
  tr.exploit({2: 0, 3: 1})
  after = tr.replica_state()
  for b, a in zip(before, after):  # the copy itself: rows 0 and 1 unchanged, 2 and 3 now theirs
    assert torch.equal(a[:2], b[:2]) and torch.equal(a[2], b[0]) and torch.equal(a[3], b[1])
  for k, v in tr.hparams.items(): assert torch.equal(v[2], v[0]) and torch.equal(v[3], v[1]), k
  src = np.array([0, 1, 0, 1])
  for step in range(19, steps + 1):
    _feed(tr, rs, step, src)
    tr.train_step()
  torch.cuda.synchronize()
  assert tr.graphs == graphs and tr.graph_launches == launches
  for i, t in enumerate(tr.replica_state() + _outputs(tr)):
    assert torch.equal(t[2], t[0]) and torch.equal(t[3], t[1]), f'{algorithm} {extra}: buffer {i} {tuple(t.shape)} differs between a destination and its source'


def _walk(obj, path, seen, out, R):
  if id(obj) in seen: return
  seen.add(id(obj))
  if isinstance(obj, torch.Tensor):
    if obj.is_cuda and obj.dim() >= 1 and obj.size(0) == R: out.append((path, obj))
    return
  if isinstance(obj, dict): items = [(f'{path}[{k!r}]', v) for k, v in obj.items()]
  elif isinstance(obj, (list, tuple)): items = [(f'{path}[{i}]', v) for i, v in enumerate(obj)]
  elif hasattr(obj, '__dict__') and type(obj).__module__.startswith('il_b200'): items = [(f'{path}.{k}', v) for k, v in vars(obj).items()]
  else: return
  for p, v in items: _walk(v, p, seen, out, R)


# Per-replica CUDA tensors that are deliberately not in replica_state(), by attribute path suffix; each carries nothing from one step to the next.
EXCLUDED = {
  # per-call outputs of the rollout, written before they are read
  '.next_state', '.action', '.env_reward', '.store_reward', '.done', '.timeout', '.terminal_f', '.timeout_f',
  # noise and index buffers (the caller's or the device RNG's draws of this step)
  '.eps_act', '.u_reset', '.idx_pol', '.idx_exp', '.u_pol', '.u_exp', '.eps_gp', '.eps_mix', '.eps_next', '.eps_new', '.dril_masks[0]', '.dril_masks[1]',
  # per-call gathers and outputs of the update
  '.batch.rows', '.expert_batch.rows', ".sac_out['log_probs']", ".sac_out['q_values']", ".sac_out['losses']", '.gail_losses',
  # the evaluation environments and the single-call API buffers of D4RLEnv (not used by the training loop)
  '.eval_env.batch.x', '.eval_env.batch.t', '.eval_env._state', '.eval_env._reward', '.eval_env._done', '.env._state', '.env._reward', '.env._done',
  # the replica map of exploit() itself
  '._src_of',
}


def _hparam_arrays(tr):
  """Storages of the per-replica hyperparameter arrays: exploit() copies them through set_hparams, not through the state copy."""
  arrs = list(tr.hparams.values()) + [v for v in (tr.discount, tr.polyak, tr.entropy_target, tr.grad_penalty, tr.entropy_bonus) if isinstance(v, torch.Tensor)]
  for name in ('actor_optimiser', 'critic_optimiser', 'temperature_optimiser', 'discriminator_optimiser'):
    o = getattr(tr, name, None)
    if o is not None: arrs += [t for t in (o.lr_r, o.weight_decay_r) if t is not None]
  d = tr.discriminator
  for n in ('discount_r', 'reward_scale', 'reward_scale_r', 'reward_bandwidth_r', 'discount'):
    v = getattr(d, n, None)
    if isinstance(v, torch.Tensor): arrs.append(v)
  for owner in (tr.actor, d):
    arrs += list(getattr(owner, '__dict__', {}).get('_hp_keep', {}).values())
  return {t.untyped_storage().data_ptr() for t in arrs}


@pytest.mark.parametrize('algorithm,extra', LOOPS, ids=LOOP_IDS)
def test_replica_state_registry_is_complete(algorithm, extra):
  """R = 5 (no other dimension is 5): every CUDA tensor reachable from the trainer with a leading replica axis is registered, a per-replica
  hyperparameter array, or in EXCLUDED. A new per-replica buffer that is none of these fails here."""
  R = 5
  tr = _trainer(algorithm, extra, R, 16)
  rs = np.random.RandomState(0)
  for step in range(1, 17):
    _feed(tr, rs, step, np.arange(R))
    tr.train_step()
  found = []
  _walk(tr, 'trainer', set(), found, R)
  registered = {t.untyped_storage().data_ptr() for t in tr.replica_state()}
  hp = _hparam_arrays(tr)
  missing = [p for p, t in found if t.untyped_storage().data_ptr() not in registered | hp and not any(p.endswith(e) for e in EXCLUDED)]
  assert not missing, f'{algorithm}: per-replica tensors neither in replica_state() nor excluded: {missing}'
  assert len(registered) == len(tr.replica_state())  # no buffer listed twice


def _state(tr):
  return [t.clone() for t in tr.replica_state() + _outputs(tr)]


SET_LOOPS = [('GAIL', ()), ('GAIL', GENERAL), ('SAC', ()), ('PWIL', ()), ('DRIL', PRE), ('RED', PRE)]


@pytest.mark.parametrize('algorithm,extra', SET_LOOPS, ids=['GAIL-fused', 'GAIL-general', 'SAC', 'PWIL', 'DRIL', 'RED'])
def test_set_hparams_before_first_step_equals_construction(algorithm, extra):
  """Eager: built with H1 and switched to H2 before the first step == built with H2, bit for bit, after 40 steps."""
  from il_b200.train import Trainer
  R, steps = 4, 40
  def run(tr):
    rs = np.random.RandomState(5)
    for step in range(1, steps + 1):
      _feed(tr, rs, step, np.arange(R))
      tr.train_step()
    torch.cuda.synchronize()
    return _state(tr)
  def make(shift):
    tr = Trainer(_cfg(algorithm, extra, R, steps, graphs=False), hparams=_hparams(algorithm, R, shift))
    tr.inject = True
    return tr
  switched = make(0)  # each trainer pre-trains right after its construction, so both draw the same host and device streams
  keep = dict(switched.hparams)
  switched.set_hparams(_hparams(algorithm, R, 2))
  assert all(switched.hparams[k] is v for k, v in keep.items())  # in place
  if algorithm in ('DRIL', 'RED'): switched.pretrain_discriminator()
  ref = make(2)
  if algorithm in ('DRIL', 'RED'): ref.pretrain_discriminator()
  for i, (a, b) in enumerate(zip(run(switched), run(ref))): assert torch.equal(a, b), f'{algorithm} {extra}: buffer {i}'


@pytest.mark.parametrize('algorithm,extra', SET_LOOPS[:4], ids=['GAIL-fused', 'GAIL-general', 'SAC', 'PWIL'])
def test_set_hparams_mid_run_under_graphs(algorithm, extra):
  """A graph-captured trainer switched to H2 at step 20 == an eager trainer given the same switch, bit for bit; nothing is re-captured."""
  R, steps = 4, 36
  outs = []
  for graphs in (True, False):
    tr = _trainer(algorithm, extra, R, steps, graphs=graphs)
    rs = np.random.RandomState(9)
    for step in range(1, steps + 1):
      if step == 20:
        g, l = dict(tr.graphs), dict(tr.graph_launches)
        tr.set_hparams(_hparams(algorithm, R, 3))
      _feed(tr, rs, step, np.arange(R))
      tr.train_step()
    torch.cuda.synchronize()
    if graphs: assert 'step+update' in g and tr.graphs == g and tr.graph_launches == l
    outs.append(_state(tr))
  for i, (a, b) in enumerate(zip(*outs)): assert torch.equal(a, b), f'{algorithm} {extra}: buffer {i}'


def test_set_hparams_rejections():
  from il_b200.train import Trainer
  tr = Trainer(_cfg('GAIL', (), 4, 20), hparams={'imitation.grad_penalty': torch.zeros(4, dtype=torch.float64)})
  with pytest.raises(ValueError, match='grad_penalty_any'):
    tr.set_hparams({'imitation.grad_penalty': [0.0, 1.0, 0.0, 0.0]})
  with pytest.raises(ValueError, match='not per-replica'):
    tr.set_hparams({'training.learning_rate': [1e-4] * 4})
  with pytest.raises(ValueError, match='>= 0'):
    tr.set_hparams({'imitation.grad_penalty': [-1.0, 0.0, 0.0, 0.0]})
  with pytest.raises(ValueError, match='overwritten'):
    tr.exploit([1, 2, 2, 3])


def test_cli_pbt(tmp_path):
  space = tmp_path / 'space.yaml'
  space.write_text('params:\n  training.learning_rate: {type: range, bounds: [1.0e-4, 1.0e-3], log_scale: true}\n'
                   '  reinforcement.discount: {type: range, bounds: [0.95, 0.99]}\n  imitation.grad_penalty: {type: choice, values: [0, 0.5, 1]}\n')
  out = tmp_path / 'out'
  cmd = [sys.executable, 'train.py', 'algorithm=GAIL', 'env=hopper', 'replicas=8', 'sweep.trials=4', f'sweep.space={space}', 'sweep.pbt.interval=1',
         'sweep.pbt.fraction=0.5', 'steps=80', 'training.start=10', 'evaluation.interval=20', 'evaluation.episodes=2', 'training.batch_size=32',
         'imitation.trajectories=2', 'reinforcement.actor.hidden_size=32', 'reinforcement.critic.hidden_size=32', 'memory.size=100', f'output_dir={out}']
  r = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=600)
  assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
  run_dir = next(p for p in out.rglob('sweep.pth')).parent
  res = torch.load(run_dir / 'sweep.pth', weights_only=False)
  assert set(res) == {'trials', 'seeds_per_trial', 'keys', 'values', 'scores', 'best', 'pbt'}
  recs = res['pbt']['records']
  assert [r['step'] for r in recs] == [20, 40, 60]  # evaluations at 20, 40, 60, 80; the last one only ranks
  for rec in recs:
    p = rec['parents']
    assert p.shape == (4, ) and (p[p] == p).all() and (p != np.arange(4)).sum() == 2
    lr, disc, gp = rec['values'].T
    assert ((lr >= 1e-4) & (lr <= 1e-3)).all() and ((disc >= 0.95) & (disc <= 0.99)).all() and set(gp) <= {0.0, 0.5, 1.0}
    assert rec['scores'].shape == (4, )
  assert np.array_equal(res['values'], recs[-1]['values']) and np.isfinite(res['scores']).all() and res['best'] == int(np.argmax(res['scores']))
  from il_b200 import sweep
  lin = sweep.lineage(res, res['best'])
  assert lin[0][0] == 0 and np.array_equal(lin[-1][1], res['values'][res['best']])
  from il_b200.config import CONF_DIR, load_config
  conf = tmp_path / 'conf'
  shutil.copytree(CONF_DIR, conf)
  shutil.copy(run_dir / 'sweep_best.yaml', conf / 'optimised_hyperparameters' / 'sweep_best.yaml')
  cfg = load_config(['algorithm=GAIL', 'optimised_hyperparameters=sweep_best'], conf_dir=str(conf))
  assert cfg.training.learning_rate == res['values'][res['best'], 0] and cfg.imitation.grad_penalty == res['values'][res['best'], 2]
