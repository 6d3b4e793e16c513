"""Host logic of the replica-batched hyperparameter search (sweep.py): search-space parsing and validation, deterministic sampling,
replica -> trial mapping and sharding, per-trial scores (also reduced over two gloo ranks) and the best-trial overlay."""
import os
import shutil

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from il_b200 import distributed, sweep
from il_b200.config import CONF_DIR, load_config

SPACE = """params:
  training.learning_rate: {type: range, bounds: [1.0e-5, 1.0e-3], log_scale: true}
  reinforcement.discount: {type: range, bounds: [0.9, 0.999]}
  imitation.grad_penalty: {type: choice, values: [0, 0.5, 1, 5]}
"""


def _space(tmp_path, text=SPACE):
  p = tmp_path / 'space.yaml'
  p.write_text(text)
  return str(p)


def test_parse_range_log_choice(tmp_path):
  s = sweep.load_space(_space(tmp_path), 'GAIL')
  assert list(s) == ['training.learning_rate', 'reinforcement.discount', 'imitation.grad_penalty']
  assert s['training.learning_rate'] == dict(type='range', bounds=(1e-5, 1e-3), log_scale=True)
  assert s['reinforcement.discount'] == dict(type='range', bounds=(0.9, 0.999), log_scale=False)
  assert s['imitation.grad_penalty'] == dict(type='choice', values=[0.0, 0.5, 1.0, 5.0])


@pytest.mark.parametrize('text,match', [
  ('params:\n  training.learning_rate: {type: range, bounds: [0, 1], log_scale: true}\n', 'log_scale'),
  ('params:\n  training.learning_rate: {type: range, bounds: [2, 1]}\n', 'bad bounds'),
  ('params:\n  training.learning_rate: {type: choice, values: []}\n', 'without values'),
  ('params:\n  training.learning_rate: {type: fixed, value: 1}\n', 'range or choice'),
  ('params: {}\n', 'non-empty'),
])
def test_malformed_space_rejected(tmp_path, text, match):
  with pytest.raises(ValueError, match=match):
    sweep.load_space(_space(tmp_path, text))


@pytest.mark.parametrize('key', ['training.batch_size', 'reinforcement.actor.hidden_size', 'imitation.discriminator.depth', 'reinforcement.actor.activation',
                                 'training.start', 'imitation.loss_function', 'imitation.spectral_norm', 'imitation.pretraining.iterations',
                                 'imitation.discriminator.dropout'])
def test_non_batchable_keys_rejected(tmp_path, key):
  with pytest.raises(ValueError) as e:
    sweep.load_space(_space(tmp_path, SPACE + f'  {key}: {{type: choice, values: [1, 2]}}\n'))
  msg = str(e.value)
  assert key in msg and 'training.learning_rate' in msg and 'imitation.quantile_cutoff' in msg  # names the key, lists the batchable ones


def test_key_unused_by_algorithm_rejected(tmp_path):
  with pytest.raises(ValueError, match='imitation.grad_penalty'):
    sweep.load_space(_space(tmp_path), 'SAC')


def test_sampling_deterministic_and_in_bounds(tmp_path):
  s = sweep.load_space(_space(tmp_path))
  keys, v = sweep.sample(s, 500, seed=3)
  keys2, v2 = sweep.sample(s, 500, seed=3)
  assert keys == keys2 and v.dtype == np.float64 and v.shape == (500, 3)
  assert np.array_equal(v, v2)
  assert not np.array_equal(v, sweep.sample(s, 500, seed=4)[1])
  lr, disc, gp = v.T
  assert (lr >= 1e-5).all() and (lr <= 1e-3).all() and (disc >= 0.9).all() and (disc <= 0.999).all()
  assert set(gp) <= {0.0, 0.5, 1.0, 5.0} and len(set(gp)) == 4
  assert (np.log(lr) < np.log(1e-4)).mean() == pytest.approx(0.5, abs=0.1)  # log-uniform: half the draws below the geometric midpoint


def test_replicas_must_be_a_multiple_of_trials():
  with pytest.raises(ValueError, match='multiple'):
    sweep.trial_of(10, 4)
  cfg = load_config(['algorithm=GAIL', 'replicas=6', 'sweep.trials=4', 'sweep.space=unused.yaml'])
  with pytest.raises(ValueError, match='multiple'):
    sweep.setup(cfg)


def test_replica_to_trial_mapping_and_shards():
  assert sweep.trial_of(8, 4).tolist() == [0, 0, 1, 1, 2, 2, 3, 3]
  assert sweep.trial_of(6, 6).tolist() == list(range(6))
  values = np.array([[1.0, 10.0], [2.0, 20.0], [3.0, 30.0]])
  hp = sweep.replica_hparams(['a', 'b'], values, 6)
  assert hp['a'].dtype == torch.float64 and hp['a'].tolist() == [1, 1, 2, 2, 3, 3] and hp['b'].tolist() == [10, 10, 20, 20, 30, 30]
  parts = [sweep.shard(hp, *distributed.shard(6, r, 4)) for r in range(4)]
  assert torch.cat([p['b'] for p in parts]).tolist() == hp['b'].tolist()
  assert [p['a'].numel() for p in parts] == [2, 2, 1, 1]


def test_no_space_means_no_sweep():
  assert sweep.setup(load_config(['algorithm=GAIL'])) == ([], None)


def test_trial_scores():
  trials = sweep.trial_of(4, 2)
  e1 = np.array([[1.0, 3.0], [5.0, 7.0], [0.0, 0.0], [2.0, 2.0]])  # [replicas, episodes]
  e2 = e1 + 1
  sums = [sweep.trial_sums(e, trials, 2) for e in (e1, e2)]
  assert sums[0].tolist() == [[16.0, 4.0], [4.0, 4.0]]
  assert sweep.scores(sums, 2).tolist() == [4.5, 1.5]  # mean over evaluations of the per-trial mean over replicas x episodes


def _worker(rank, world, port, q):
  os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
  from il_b200 import distributed, sweep
  distributed.init('gloo')
  total, T = 6, 3
  lo, hi = distributed.shard(total, rank, world)
  normalized = np.arange(total * 2, dtype=np.float64).reshape(total, 2)[lo:hi]
  s = sweep.reduce_sums(sweep.trial_sums(normalized, sweep.trial_of(total, T)[lo:hi], T))
  distributed.barrier()
  q.put((rank, sweep.scores([s], T).tolist()))


@pytest.mark.timeout(120)
def test_trial_scores_two_ranks_gloo():
  ctx = mp.get_context('spawn')
  q = ctx.Queue()
  port = 29400 + (os.getpid() % 200)
  procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
  for p in procs: p.start()
  res = sorted(q.get(timeout=100) for _ in range(2))
  for p in procs: p.join(timeout=30)
  want = np.arange(12, dtype=np.float64).reshape(3, 4).mean(axis=1).tolist()  # trial t: replicas 2t, 2t+1 (the shard boundary splits trial 1)
  assert [r[1] for r in res] == [want, want]


def test_results_and_best_overlay_round_trip(tmp_path, capsys):
  conf = tmp_path / 'conf'
  shutil.copytree(CONF_DIR, conf)
  keys = ['training.learning_rate', 'reinforcement.discount', 'imitation.grad_penalty']
  values = np.array([[1e-4, 0.95, 0.0], [3.3e-4, 0.987654321, 0.5], [2e-5, 0.9, 5.0]])
  res = sweep.write_results(str(tmp_path) + os.sep, keys, values, 4, np.array([0.1, 0.7, np.nan]))
  assert res['best'] == 1 and 'top 3' in capsys.readouterr().out
  saved = torch.load(tmp_path / 'sweep.pth', weights_only=False)
  assert saved['trials'] == 3 and saved['seeds_per_trial'] == 4 and saved['keys'] == keys and saved['best'] == 1
  assert saved['values'].dtype == np.float64 and np.array_equal(saved['values'], values)
  text = (tmp_path / 'sweep_best.yaml').read_text()
  assert text.startswith('# @package _global_')
  shutil.copy(tmp_path / 'sweep_best.yaml', conf / 'optimised_hyperparameters' / 'sweep_best.yaml')
  cfg = load_config(['algorithm=GAIL', 'optimised_hyperparameters=sweep_best'], conf_dir=str(conf))
  assert cfg.training.learning_rate == 3.3e-4 and cfg.reinforcement.discount == 0.987654321 and cfg.imitation.grad_penalty == 0.5
  assert cfg.training.batch_size == 256 and cfg.imitation.loss_function == load_config(['algorithm=GAIL']).imitation.loss_function  # the rest stays


def test_results_without_evaluations(tmp_path):
  """check_time_usage=true or steps < evaluation.interval: no evaluation ran, every score is NaN and the results are still written."""
  values = np.array([[1e-4], [2e-4], [3e-4]])
  s = sweep.scores([], 3)
  assert s.shape == (3, ) and np.isnan(s).all()
  res = sweep.write_results(str(tmp_path) + os.sep, ['training.learning_rate'], values, 2, s)
  assert res['best'] == 0 and (tmp_path / 'sweep_best.yaml').exists()


def test_trainer_rejects_unsupported_per_replica_hyperparameters():
  from il_b200.train import MAX_SWEEP_REPLICAS, Trainer
  pwil = load_config(['algorithm=PWIL', 'imitation.mix_expert_data=mixed_batch'])
  with pytest.raises(ValueError, match='mix_expert_data'):
    Trainer._check_hparams({'imitation.reward_scale': [1.0, 2.0]}, pwil, 2, 'cpu')
  assert set(Trainer._check_hparams({'imitation.reward_scale': [1.0, 2.0]}, load_config(['algorithm=PWIL']), 2, 'cpu')) == {'imitation.reward_scale'}
  R = MAX_SWEEP_REPLICAS + 1
  with pytest.raises(ValueError, match=str(MAX_SWEEP_REPLICAS)):
    Trainer._check_hparams({'training.learning_rate': torch.full((R, ), 1e-4)}, load_config(['algorithm=SAC']), R, 'cpu')
  with pytest.raises(ValueError, match='hidden_size'):
    Trainer._check_hparams({'reinforcement.actor.hidden_size': [1.0, 2.0]}, load_config(['algorithm=SAC']), 2, 'cpu')
