"""Pins oracle/loop.py — the restated step schedule of train.py:146-227 that the GPU loop tests and the CPU baseline are
built on — against the reference's REAL `train.train(cfg)`: the unmodified train.py / environments.py / memory.py /
models.py / training.py / evaluation.py run end to end (oracle/ref_train.py stubs only hydra, plotting and `gym.make`,
which returns the synthetic-environment twin) and the oracle loop, fed by the same global torch / numpy RNG streams,
must arrive at the same parameters after the same number of steps. What each reference run ends with is recorded in
tests/golden/loop_pinned.npz (`record`, written by `python -m oracle.make_golden loop_pinned`), so the comparison runs
without the reference tree."""
import functools
import json

import numpy as np
import pytest
import torch

from conftest import load_golden
from il_b200 import config
from oracle import loop

STEPS, MAX_EPISODE_STEPS, B, H, START = 60, 25, 16, 32, 8
ATOL = 2e-6  # fp32, same torch CPU ops on both sides; observed 3e-8 after 60 steps
FULL, SAMPLES = 128, 32 # recorded tensors above FULL entries keep a fixed sample of SAMPLES entries plus their sum and max |x| (fixture size)


def _cfg(algorithm, env, seed, extra=()):
  cfg = config.load_config([f'algorithm={algorithm}', f'env={env}', f'steps={STEPS}', f'training.start={START}', f'training.batch_size={B}', f'reinforcement.actor.hidden_size={H}',
                            f'reinforcement.critic.hidden_size={H}', 'imitation.trajectories=3', f'evaluation.interval={STEPS}', 'evaluation.episodes=2', 'logging.interval=10',
                            'memory.size=1000', f'seed={seed}', *extra])
  for k in ('replicas', 'device_rng', 'cuda_graphs', 'gemm_mode', 'output_dir'): cfg.pop(k, None)  # keys this build adds
  return cfg


def _sample_idx(size):
  return np.random.RandomState(size).choice(size, SAMPLES, replace=False)


class _Sampled:
  def __init__(self, shape, val, stat): self.shape, self.val, self.stat = tuple(int(d) for d in shape), val, stat


def record(run_id, ref, z):
  """Adds what `oracle.ref_train.run_reference_train` returned to the fixture dict `z`, keyed `<run_id>/<name>` in the
  order of the reference's state dicts (the order `_recorded` hands back)."""
  def put(name, v):
    v = np.asarray(v.detach().numpy() if torch.is_tensor(v) else v)
    if v.dtype.kind == 'f' and v.size > FULL:
      z[f'{run_id}/{name}@val'], z[f'{run_id}/{name}@shape'] = v.reshape(-1)[_sample_idx(v.size)], np.int64(v.shape)
      z[f'{run_id}/{name}@stat'] = np.float64([v.astype(np.float64).sum(), np.abs(v).max()])
    else:
      z[f'{run_id}/{name}'] = v
  for group in ('actor', 'critic'):
    for k, v in ref['agent'].get(group, {}).items(): put(f'{group}/{k}', v)
  if 'log_alpha' in ref['agent']: put('log_alpha', ref['agent']['log_alpha'])
  for k, v in ref.get('discriminator', {}).items(): put(f'discriminator/{k}', v)
  m = ref['metrics']
  put('train_returns', np.float64([r[0] for r in m['train_returns']]))
  put('update_steps', np.int64(m['update_steps']))
  for k in ('predicted_rewards', 'Q_values', 'entropies'):
    if m[k]: put(k, m[k][-1])
  if m['test_returns']: put('test_returns', np.float64(m['test_returns'][0]))
  put('score', np.float64(ref['score']))


def pack(z):
  """The fixture dict as one JSON index and one float64 vector (an npz entry per small array would cost more in headers
  than in data); float32 and small integers round-trip exactly."""
  index, chunks, offset = [], [], 0
  for k, v in z.items():
    index.append([k, v.dtype.str, list(v.shape), offset])
    chunks.append(v.astype(np.float64).reshape(-1))
    offset += v.size
  return dict(index=np.array(json.dumps(index)), values=np.concatenate(chunks))


@functools.lru_cache(maxsize=None)
def _fixture():
  g = load_golden('loop_pinned')
  values = g['values']
  return {k: values[off:off + int(np.prod(shape))].astype(dtype).reshape(shape) for k, dtype, shape, off in json.loads(str(g['index']))}


def _recorded(run_id):
  """The recorded run as {'actor': {name: array | _Sampled}, 'critic': {...}, 'discriminator': {...}, other name: array}."""
  z, out = _fixture(), {}
  for key in z:
    if not key.startswith(run_id + '/'): continue
    name = key[len(run_id) + 1:].split('@')[0]
    value = z[key] if '@' not in key else _Sampled(z[f'{run_id}/{name}@shape'], z[f'{run_id}/{name}@val'], z[f'{run_id}/{name}@stat'])
    group, _, k = name.partition('/')
    if k: out.setdefault(group, {}).setdefault(k, value)
    else: out.setdefault(group, value)
  assert out, f'{run_id}: not in tests/golden/loop_pinned.npz'
  return out


def _close(name, ref, mine, atol=ATOL):
  mine = torch.as_tensor(mine).detach().float()
  if isinstance(ref, _Sampled):
    assert ref.shape == tuple(mine.shape), (name, ref.shape, tuple(mine.shape))
    scale = max(1.0, float(ref.stat[1]))
    err = float((torch.as_tensor(ref.val) - mine.reshape(-1)[_sample_idx(mine.numel())]).abs().max())
    assert err <= atol * scale, f'{name}: max abs err {err:.3e} on the recorded entries'
    m64 = mine.double()
    assert abs(float(m64.sum()) - ref.stat[0]) <= atol * scale * mine.numel(), f'{name}: sum {float(m64.sum())} vs {ref.stat[0]}'
    assert abs(float(m64.abs().max()) - ref.stat[1]) <= atol * scale, f'{name}: max |x| {float(m64.abs().max())} vs {ref.stat[1]}'
    return
  ref = torch.as_tensor(ref).detach().float()
  assert ref.shape == mine.shape, (name, ref.shape, mine.shape)
  err = float((ref - mine).abs().max())
  assert err <= atol * max(1.0, float(ref.abs().max())), f'{name}: max abs err {err:.3e}'


CONFIGS = [
  # (algorithm, env, reference-side overrides, oracle-loop kwargs)
  ('GAIL', 'hopper', (), {}),
  ('GAIL', 'walker2d', ('imitation.mix_expert_data=mixed_batch', ), dict(mix_expert_data='mixed_batch')),
  ('GAIL', 'hopper', ('imitation.loss_function=Mixup', 'imitation.entropy_bonus=0.1', 'imitation.grad_penalty=0.5'), dict(imitation=dict(loss_function='Mixup', entropy_bonus=0.1, grad_penalty=0.5))),
  ('GAIL', 'hopper', ('imitation.loss_function=PUGAIL', 'imitation.nonnegative_margin=0.3', 'imitation.grad_penalty=0', 'imitation.spectral_norm=false',
                      'imitation.discriminator.reward_function=FAIRL'),
   dict(imitation=dict(loss_function='PUGAIL', nonnegative_margin=0.3, grad_penalty=0.0, spectral_norm=False, reward_function='FAIRL'))),
  ('GAIL', 'hopper', ('imitation.bc_aux_loss=true', ), dict(bc_aux_loss=True)),
  ('GAIL', 'hopper', ('imitation.discriminator.reward_shaping=true', 'imitation.discriminator.subtract_log_policy=true', 'imitation.discriminator.hidden_size=16'),
   dict(imitation=dict(reward_shaping=True, subtract_log_policy=True, hidden_size=16))),
  ('GAIL', 'halfcheetah', ('imitation.discriminator.depth=2', 'imitation.discriminator.activation=tanh', 'imitation.discriminator.hidden_size=16', 'imitation.discriminator.reward_function=GAIL'),
   dict(imitation=dict(depth=2, activation='tanh', hidden_size=16, reward_function='GAIL'))),
  ('GAIL', 'hopper', ('imitation.state_only=true', 'imitation.grad_penalty=0', 'imitation.discriminator.activation=sigmoid', 'imitation.discriminator.reward_shaping=true'),
   dict(imitation=dict(state_only=True, grad_penalty=0.0, activation='sigmoid', reward_shaping=True))),
  # AdRIL (balanced alternation, rounds of 20 steps so several round boundaries fall inside the run), unbalanced AdRIL, SQIL (update_freq 0)
  ('AdRIL', 'hopper', ('imitation.update_freq=20', ), dict(mix_expert_data='mixed_batch', imitation=dict(update_freq=20, balanced=True))),
  ('AdRIL', 'walker2d', ('imitation.update_freq=15', 'imitation.balanced=false'), dict(mix_expert_data='mixed_batch', imitation=dict(update_freq=15, balanced=False))),
  ('AdRIL', 'hopper', ('imitation.update_freq=0', ), dict(mix_expert_data='mixed_batch', imitation=dict(update_freq=0, balanced=True))),
  # DRIL (dropout policy ensemble, BC pretraining, quantile threshold, MC-dropout reward; bc_aux_loss from DRIL.yaml) and RED (predictor / target
  # embeddings, regression pretraining, median-heuristic bandwidth, with and without dropout / prefill)
  ('DRIL', 'hopper', ('imitation.pretraining.iterations=9', 'imitation.discriminator.hidden_size=16'),
   dict(bc_aux_loss=True, imitation=dict(hidden_size=16, activation='tanh', input_dropout=0.1, dropout=0.1, pretraining_iterations=9, learning_rate=3e-5, weight_decay=0.0))),
  ('DRIL', 'walker2d', ('imitation.pretraining.iterations=5', 'imitation.discriminator.hidden_size=16', 'imitation.discriminator.depth=2', 'imitation.discriminator.dropout=0.4',
                        'imitation.mix_expert_data=mixed_batch', 'imitation.quantile_cutoff=0.9', 'imitation.bc_aux_loss=false'),
   dict(mix_expert_data='mixed_batch', imitation=dict(hidden_size=16, depth=2, activation='tanh', input_dropout=0.1, dropout=0.4, pretraining_iterations=5, quantile_cutoff=0.9,
                                                      learning_rate=3e-5, weight_decay=0.0))),
  ('RED', 'hopper', ('imitation.pretraining.iterations=11', ), dict(imitation=dict(hidden_size=32, pretraining_iterations=11, learning_rate=3e-5, weight_decay=0.0))),
  ('RED', 'halfcheetah', ('imitation.pretraining.iterations=6', 'imitation.discriminator.input_dropout=0.2', 'imitation.discriminator.dropout=0.3', 'imitation.discriminator.depth=2',
                          'imitation.mix_expert_data=prefill_memory', 'imitation.weight_decay=0.5'),
   dict(mix_expert_data='prefill_memory', imitation=dict(hidden_size=32, depth=2, input_dropout=0.2, dropout=0.3, pretraining_iterations=6, learning_rate=3e-5, weight_decay=0.5))),
  ('SAC', 'hopper', (), {}),
  ('SAC', 'ant', ('training.weight_decay=0.01', ), dict(weight_decay=0.01)),
  ('GMMIL', 'halfcheetah', (), {}),
  ('GMMIL', 'hopper', ('imitation.mix_expert_data=mixed_batch', ), dict(mix_expert_data='mixed_batch')),
  ('GMMIL', 'hopper', ('imitation.mix_expert_data=prefill_memory', ), dict(mix_expert_data='prefill_memory')),
  ('PWIL', 'hopper', (), {}),
  ('PWIL', 'hopper', ('imitation.mix_expert_data=mixed_batch', ), dict(mix_expert_data='mixed_batch')),
  ('PWIL', 'walker2d', ('imitation.mix_expert_data=prefill_memory', ), dict(mix_expert_data='prefill_memory')),
]
LOOP_IDS = [f'{a}-{e}-{i}' for i, (a, e, _, _) in enumerate(CONFIGS)]
LOOP_SEED, BC_SEED, BC_ENV = 3, 5, 'hopper'
BC_RUNS = [('BC', 25), ('GAIL', 7)]


def _bc_cfg(algorithm, iterations):
  return _cfg(algorithm, BC_ENV, BC_SEED, [f'bc_pretraining.iterations={iterations}', 'bc_pretraining.learning_rate=0.001', 'bc_pretraining.weight_decay=0.01'])


def reference_runs():
  """(run id, config, raw expert dataset) of every reference `train.train` run the tests below compare with."""
  for run_id, (algorithm, env, extra, _) in zip(LOOP_IDS, CONFIGS):
    yield run_id, _cfg(algorithm, env, LOOP_SEED, extra), loop.synthesize_raw_dataset(env, True, 5, MAX_EPISODE_STEPS)
  for algorithm, iterations in BC_RUNS:
    yield f'bc-{algorithm}-{iterations}', _bc_cfg(algorithm, iterations), loop.synthesize_raw_dataset(BC_ENV, True, 5, MAX_EPISODE_STEPS)


@pytest.mark.parametrize('algorithm,env,extra,kwargs', CONFIGS, ids=LOOP_IDS)
def test_restated_loop_equals_the_reference_train_function(algorithm, env, extra, kwargs, request):
  seed = LOOP_SEED
  raw = loop.synthesize_raw_dataset(env, True, 5, MAX_EPISODE_STEPS)
  ref = _recorded(request.node.callspec.id)

  threads = torch.get_num_threads()
  torch.set_num_threads(1)
  try:
    ol = loop.OracleLoop(algorithm, env, seed=seed, batch_size=B, start=START, memory_size=STEPS, hidden_size=H, trajectories=3, max_episode_steps=MAX_EPISODE_STEPS,
                         expert_raw=raw, **kwargs)
    if algorithm in ('DRIL', 'RED'): ol.pretrain_discriminator()
    for _ in range(STEPS): ol.run_step()
  finally:
    torch.set_num_threads(threads)

  for i, (k, v) in enumerate(ref['actor'].items()): _close(f'actor.{k}', v, ol.agent.actor[i])
  critic = list(ref['critic'].items())
  assert len(critic) == 12
  for t in range(2):
    for i in range(6): _close(f'critic.{critic[6 * t + i][0]}', critic[6 * t + i][1], ol.agent.twin[t][i])
  _close('log_alpha', ref['log_alpha'], ol.agent.log_alpha)
  if algorithm == 'DRIL':  # discriminator.pth = the dropout policy's state dict (train.py:238)
    for i, (k, v) in enumerate(ref['discriminator'].items()): _close(f'dril.{k}', v, ol.disc[i])
  if algorithm == 'RED':
    sd = ref['discriminator']
    for i, (k, v) in enumerate((k, v) for k, v in sd.items() if k.startswith('predictor')): _close(f'red.{k}', v, ol.disc.predictor[i])
    for i, (k, v) in enumerate((k, v) for k, v in sd.items() if k.startswith('target')): _close(f'red.{k}', v, ol.disc.target[i])
  if algorithm == 'GAIL':
    sd, sn = ref['discriminator'], ol.disc.g_sn is not None
    for net, params, bufs in (('g', ol.disc.g, ol.disc.g_sn), ('h', ol.disc.h, ol.disc.h_sn)):
      if params is None: continue
      single = net == 'g' and ol.disc.h is not None  # with reward shaping g is one nn.Linear, not a Sequential (models.py:157)
      for l in range(len(params) // 2):
        pre = net if single else f'{net}.{[i for i in range(99) if f"{net}.{i}.bias" in sd][l]}'
        _close(f'{pre}.weight', sd[f'{pre}.parametrizations.weight.original' if sn else f'{pre}.weight'], params[2 * l])
        _close(f'{pre}.bias', sd[f'{pre}.bias'], params[2 * l + 1])
        if sn:
          # singular-vector estimates are ill-conditioned when the two largest singular values are close: 10x looser
          _close(f'{pre}.u', sd[f'{pre}.parametrizations.weight.0._u'], bufs[l][0], atol=10 * ATOL)
          _close(f'{pre}.v', sd[f'{pre}.parametrizations.weight.0._v'], bufs[l][1], atol=10 * ATOL)
    assert sum(k.endswith('bias') for k in sd) == (len(ol.disc.g) + len(ol.disc.h or [])) // 2
  # episode bookkeeping (train.py:161-168) and the logged tensors of the last logging step (train.py:205-210)
  got = ref['train_returns']
  assert len(got) == len(ol.episode_returns) and np.allclose(got, ol.episode_returns, rtol=1e-5, atol=1e-6)
  assert ref['update_steps'].tolist() == [s for s in range(10, STEPS + 1, 10) if s >= START]
  _close('predicted_rewards', ref['predicted_rewards'], ol.last['rewards'])
  _close('q_values', ref['Q_values'], ol.last['sac']['q_values'])
  _close('entropies', ref['entropies'], -ol.last['sac']['log_probs'])


@pytest.mark.parametrize('algorithm,iterations', BC_RUNS)
def test_bc_pretraining_equals_the_reference(algorithm, iterations):
  """train.py:95-115: BC on shuffled expert minibatches (the DataLoader's shuffling stream restated in OracleLoop.bc_pretrain);
  algorithm=BC returns after pretraining + evaluation, any other algorithm continues into the loop with the pretrained actor."""
  from oracle import port
  seed, env = BC_SEED, BC_ENV
  raw = loop.synthesize_raw_dataset(env, True, 5, MAX_EPISODE_STEPS)
  ref = _recorded(f'bc-{algorithm}-{iterations}')
  threads = torch.get_num_threads()
  torch.set_num_threads(1)
  try:
    ol = loop.OracleLoop('SAC' if algorithm == 'BC' else algorithm, env, seed=seed, batch_size=B, start=START, memory_size=STEPS, hidden_size=H, trajectories=3,
                         max_episode_steps=MAX_EPISODE_STEPS, expert_raw=raw, build_expert_memory=True)
    ol.bc_pretrain(iterations, 0.001, 0.01)
    if algorithm != 'BC':
      for _ in range(STEPS): ol.run_step()
  finally:
    torch.set_num_threads(threads)
  for i, (k, v) in enumerate(ref['actor'].items()): _close(f'actor.{k}', v, ol.agent.actor[i])
  if algorithm == 'BC':
    assert 'critic' not in ref and 'log_alpha' not in ref  # train.py:111 saves the actor only
    # the evaluation of train.py:104 on the evaluation env's own reset stream (second env made, oracle/ref_train.py)
    g = torch.Generator().manual_seed(seed + 10007)
    eval_env = port.SyntheticEnv(env, True, MAX_EPISODE_STEPS)
    noise = [torch.rand(eval_env.obs, generator=g) for _ in range(2)]
    mine = port.evaluate_agent(ol.agent.actor, eval_env, 2, noise)
    assert np.allclose(ref['test_returns'], mine, rtol=1e-5, atol=1e-6)
    assert abs(float(ref['score']) - np.mean(mine) / 1000.0) < 1e-7
  else:
    _close('log_alpha', ref['log_alpha'], ol.agent.log_alpha)
