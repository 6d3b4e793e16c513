"""Host logic of population-based training on the replica axis (sweep.py): selection, the replica map, exploration, lineage, the
rank-local populations over two gloo ranks, and the configurations it rejects."""
import os

import numpy as np
import pytest
import torch.multiprocessing as mp

from il_b200 import sweep
from il_b200.config import load_config

SPACE = """params:
  training.learning_rate: {type: range, bounds: [1.0e-5, 1.0e-3], log_scale: true}
  reinforcement.discount: {type: range, bounds: [0.9, 0.999]}
  imitation.grad_penalty: {type: choice, values: [0, 0.5, 1, 5]}
  bc_pretraining.learning_rate: {type: range, bounds: [1.0e-5, 1.0e-3]}
"""


def _space_file(tmp_path, text=SPACE):
  p = tmp_path / 'space.yaml'
  p.write_text(text)
  return str(p)


def _pbt(tmp_path, replicas=16, trials=8, world=1, extra=()):
  cfg = load_config(['algorithm=GAIL', f'replicas={replicas}', f'sweep.trials={trials}', f'sweep.space={_space_file(tmp_path)}', 'sweep.seed=11',
                     'sweep.pbt.interval=1', *extra])
  keys, values = sweep.setup(cfg)
  return sweep.pbt_config(cfg, world), keys, values


def test_defaults_and_off_by_default(tmp_path):
  assert sweep.pbt_config(load_config(['algorithm=GAIL', f'sweep.space={_space_file(tmp_path)}', 'replicas=4', 'sweep.trials=4'])) is None
  pbt, _, _ = _pbt(tmp_path)
  assert (pbt['interval'], pbt['fraction'], pbt['perturb'], pbt['resample'], pbt['seed']) == (1, 0.25, 0.2, 0.25, 11)
  assert pbt['grad_penalty_any'] is True and [p.tolist() for p in pbt['populations']] == [list(range(8))]


def test_selection_deterministic_disjoint_and_nan_last():
  rs = np.random.RandomState(0)
  pops = [np.arange(12)]
  for fraction in (0.1, 0.25, 0.5):
    scores = rs.standard_normal(12)
    scores[[3, 7]] = np.nan
    a = sweep.pbt_select(scores, pops, fraction, np.random.default_rng([5, 0]))
    b = sweep.pbt_select(scores, pops, fraction, np.random.default_rng([5, 0]))
    assert np.array_equal(a, b)
    k = int(np.floor(fraction * 12))
    exploited = np.flatnonzero(a != np.arange(12))
    assert len(exploited) == k
    order = sweep._ranking(scores)
    assert set(exploited) == set(order[12 - k:].tolist())  # the bottom k, NaN-scored trials first among them
    assert {3, 7} <= set(exploited) or k < 2
    assert set(a[exploited]) <= set(order[:k].tolist())  # parents come from the top k
    assert not set(a[exploited]) & set(exploited)  # bottom and top are disjoint
  many = {tuple(sweep.pbt_select(np.arange(12.0), pops, 0.25, np.random.default_rng([s, 0]))) for s in range(40)}
  assert len(many) > 1  # the parent is a random top trial


def test_replica_map_block_rule():
  parents = np.array([0, 1, 1, 0])
  m = sweep.replica_map(parents, 12)  # 3 seeds per trial
  assert m.tolist() == [0, 1, 2, 3, 4, 5, 3, 4, 5, 0, 1, 2]
  assert np.array_equal(m[m], m)


def test_explore_bounds_log_space_neighbours_and_frozen(tmp_path):
  pbt, keys, values = _pbt(tmp_path, extra=('sweep.pbt.resample=0', 'sweep.pbt.perturb=0.2'))
  space = pbt['space']
  T = len(values)
  parents = np.array([0, 1, 2, 3, 4, 5, 0, 1])
  rng = np.random.default_rng(1)
  for _ in range(50):
    new = sweep.pbt_explore(space, keys, values, parents, 0.2, 0.0, rng)
    assert np.array_equal(new[:6], values[:6])  # trials that were not exploited keep their values
    for t, p in ((6, 0), (7, 1)):
      lr, disc, gp, bc = new[t]
      assert 1e-5 <= lr <= 1e-3 and 0.9 <= disc <= 0.999
      step = abs(np.log(lr) - np.log(values[p, 0])) / (np.log(1e-3) - np.log(1e-5))  # a log-scale key moves by perturb in log space
      assert step == pytest.approx(0.2) or lr in (1e-5, 1e-3)
      assert abs(disc - values[p, 1]) == pytest.approx(0.2 * 0.099) or disc in (0.9, 0.999)
      vals = space['imitation.grad_penalty']['values']
      assert abs(vals.index(gp) - vals.index(values[p, 2])) == 1  # a choice moves to a neighbour
      assert bc == values[p, 3]  # bc_pretraining.* only acts before the loop: inherited, never perturbed
    values = new
  assert T == 8


def test_explore_resample_draws_in_bounds(tmp_path):
  pbt, keys, values = _pbt(tmp_path)
  parents = np.array([0, 1, 2, 3, 4, 5, 0, 1])
  new = sweep.pbt_explore(pbt['space'], keys, values, parents, 0.2, 1.0, np.random.default_rng(2))
  assert (new[6:, 0] >= 1e-5).all() and (new[6:, 0] <= 1e-3).all() and set(new[6:, 2]) <= {0.0, 0.5, 1.0, 5.0}
  assert np.array_equal(new[6:, 3], values[[0, 1], 3])


def test_pbt_step_deterministic_per_index(tmp_path):
  pbt, keys, values = _pbt(tmp_path)
  scores = np.linspace(0, 1, 8)
  a, b = sweep.pbt_step(pbt, keys, values, scores, 3), sweep.pbt_step(pbt, keys, values, scores, 3)
  assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
  assert set(np.flatnonzero(a[0] != np.arange(8))) == {0, 1}  # floor(0.25 x 8) lowest scores


def test_lineage_follows_parents():
  init = np.array([[1.0], [2.0], [3.0], [4.0]])
  r1 = dict(step=10, parents=np.array([0, 1, 1, 3]), values=np.array([[1.0], [2.0], [2.5], [4.0]]), scores=np.zeros(4))
  r2 = dict(step=20, parents=np.array([2, 1, 2, 3]), values=np.array([[2.7], [2.0], [2.5], [4.0]]), scores=np.zeros(4))
  res = dict(pbt=dict(initial=init, records=[r1, r2]))
  lin = sweep.lineage(res, 0)
  assert [(s, v.tolist()) for s, v in lin] == [(0, [2.0]), (10, [2.5]), (20, [2.7])]  # trial 0 <- trial 2 (at 20) <- trial 1 (at 10)
  assert [(s, v.tolist()) for s, v in sweep.lineage(res, 3)] == [(0, [4.0])]


def test_populations_reject_straddling_and_small_ranks():
  assert [p.tolist() for p in sweep.populations(16, 8, 2)] == [[0, 1, 2, 3], [4, 5, 6, 7]]
  with pytest.raises(ValueError, match='splits a trial'):
    sweep.populations(12, 6, 4)  # 3 replicas per rank, 2 seeds per trial
  with pytest.raises(ValueError, match='at least 2'):
    sweep.populations(8, 4, 4)  # one trial per rank


@pytest.mark.parametrize('extra,match', [
  (('algorithm=BC', ), 'BC'),
  (('check_time_usage=true', ), 'check_time_usage'),
  (('sweep.pbt.fraction=0.6', ), 'fraction'),
  (('sweep.pbt.fraction=0', ), 'fraction'),
  (('sweep.pbt.resample=1.5', ), 'resample'),
  (('sweep.pbt.perturb=-1', ), 'perturb'),
])
def test_rejections(tmp_path, extra, match):
  space = tmp_path / 'lr.yaml'
  space.write_text('params:\n  training.learning_rate: {type: range, bounds: [1.0e-5, 1.0e-3]}\n')
  cfg = load_config(['algorithm=GAIL', 'replicas=8', 'sweep.trials=4', f'sweep.space={space}', 'sweep.pbt.interval=2', *extra])
  with pytest.raises(ValueError, match=match):
    sweep.pbt_config(cfg, 1)


def test_rejects_pbt_without_space():
  with pytest.raises(ValueError, match='sweep.space'):
    sweep.pbt_config(load_config(['algorithm=GAIL', 'sweep.pbt.interval=1']), 1)


def _worker(rank, world, port, space, q):
  os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
  from il_b200 import distributed, sweep
  from il_b200.config import load_config
  distributed.init('gloo')
  total, T = 16, 8
  cfg = load_config(['algorithm=GAIL', f'replicas={total}', f'sweep.trials={T}', f'sweep.space={space}', 'sweep.pbt.interval=1', 'sweep.pbt.fraction=0.5'])
  keys, values = sweep.setup(cfg)
  pbt = sweep.pbt_config(cfg, world)
  lo, hi = distributed.shard(total, rank, world)
  normalized = np.random.RandomState(rank).standard_normal((hi - lo, 2))  # each rank's own returns; the reduced sums are global
  s = sweep.reduce_sums(sweep.trial_sums(normalized, sweep.trial_of(total, T)[lo:hi], T))
  parents, new = sweep.pbt_step(pbt, keys, values, sweep.latest_scores([s], T), 0)
  local = sweep.replica_map(parents, total)[lo:hi] - lo
  distributed.barrier()
  q.put((rank, parents.tolist(), new.tolist(), local.tolist()))


@pytest.mark.timeout(120)
def test_two_ranks_identical_decisions_rank_local(tmp_path):
  ctx = mp.get_context('spawn')
  q = ctx.Queue()
  port = 29600 + (os.getpid() % 200)
  procs = [ctx.Process(target=_worker, args=(r, 2, port, _space_file(tmp_path), q)) for r in range(2)]
  for p in procs: p.start()
  res = sorted(q.get(timeout=100) for _ in range(2))
  for p in procs: p.join(timeout=30)
  (_, p0, v0, l0), (_, p1, v1, l1) = res
  assert p0 == p1 and v0 == v1
  parents = np.array(p0)
  assert (parents != np.arange(8)).sum() == 4  # floor(0.5 x 4) per rank
  assert all((t < 4) == (parents[t] < 4) for t in range(8))  # no source crosses a rank
  assert min(l0 + l1) >= 0 and max(l0 + l1) < 8
