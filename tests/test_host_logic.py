"""CPU-only checks of the host-side logic of the drop-in: expert-data ingest (environments.py:63-125), the Hydra-free
configuration surface (train.py:21-23, conf/) and the replica sharding helpers. No CUDA call is made here."""
import json
import os

import numpy as np
import pytest
import torch
import yaml

from il_b200 import config, environments
from oracle import cases, port

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INGEST = [n for n, c in cases.CASES.items() if c['kind'] == 'ingest']


@pytest.mark.parametrize('name', INGEST)
def test_expert_ingest_equals_oracle_bit_for_bit(name):
  """il_b200.environments.build_expert_transitions (the product's get_dataset preprocessing, global numpy RNG for the
  subsampling offsets like environments.py:113) == the oracle port, which tests/golden pins against the reference."""
  c, inp = cases.CASES[name], cases.make_inputs(name)
  raw = {k: torch.from_numpy(inp[k].copy()) for k in ('observations', 'next_observations', 'actions', 'terminals', 'timeouts')}
  seed = int(inp['np_seed'][0])
  state = np.random.get_state()
  np.random.seed(seed)
  try:
    got = environments.build_expert_transitions(raw, c['trajectories'], c['subsample'], c['absorbing'])
  finally:
    np.random.set_state(state)
  want = port.build_expert_transitions(raw, c['trajectories'], c['subsample'], c['absorbing'], rng=np.random.RandomState(seed))
  assert got['num_trajectories'] == want['num_trajectories']
  for k in ('states', 'actions', 'next_states', 'terminals', 'timeouts', 'weights', 'rewards'):
    assert got[k].shape == want[k].shape, k
    assert torch.equal(got[k], want[k]), k
  assert inp['terminals'].tobytes() == raw['terminals'].numpy().tobytes(), 'the raw buffer must not be modified'


def test_expert_ingest_edge_cases():
  """Ragged input: a single one-step episode, an episode that ends by time limit (no absorbing row), subsample larger
  than an episode (the absorbing pair is always kept, environments.py:115)."""
  obs, A = 3, 2
  raw = dict(observations=torch.arange(18, dtype=torch.float32).view(6, obs), next_observations=torch.ones(6, obs), actions=torch.zeros(6, A),
             terminals=torch.tensor([1., 0, 0, 0, 0, 1]), timeouts=torch.tensor([0., 0, 0, 1, 0, 0]))
  tr = environments.build_expert_transitions(raw, 0, 1, True)
  assert tr['num_trajectories'] == 3
  # episode 0: 1 row + absorbing row; episode 1: 3 rows, timeout, no absorbing row; episode 2: 2 rows + absorbing row
  assert tr['states'].shape == (1 + 1 + 3 + 2 + 1, obs + 1)
  assert tr['states'][:, -1].tolist() == [0, 1, 0, 0, 0, 0, 0, 1]
  assert tr['terminals'].sum() == 0 and tr['timeouts'].tolist() == [0, 0, 0, 0, 1, 0, 0, 0]
  assert torch.all(tr['rewards'] == 0)
  state = np.random.get_state()
  np.random.seed(0)
  try:
    sub = environments.build_expert_transitions(raw, 1, 20, True)  # first episode only, subsample 20 > length
  finally:
    np.random.set_state(state)
  assert sub['states'].shape[0] == 2 and torch.equal(sub['weights'], torch.full((2,), 1 / 20))


def _flat(d, prefix=''):
  out = {}
  for k, v in d.items():
    if isinstance(v, dict): out.update(_flat(v, f'{prefix}{k}.'))
    else: out[prefix + k] = v
  return out


def test_config_defaults_and_overrides():
  cfg = config.load_config(['algorithm=GAIL', 'env=hopper', 'training.batch_size=512', 'imitation.discriminator.reward_function=FAIRL', 'replicas=8', 'cuda_graphs=false'])
  assert cfg.algorithm == 'GAIL' and cfg.env == 'hopper'
  assert cfg.training.batch_size == 512 and isinstance(cfg.training.batch_size, int)
  assert cfg.imitation.discriminator.reward_function == 'FAIRL'
  assert cfg.replicas == 8 and cfg.cuda_graphs is False
  # GAIL.yaml:5-7 overlays (discount / target temperature / polyak) on top of train_config.yaml:36-38
  assert cfg.reinforcement.discount == 0.97 and cfg.reinforcement.polyak_factor == 0.99 and cfg.reinforcement.target_temperature == -0.5
  assert cfg.imitation.weight_decay == 10 and cfg.imitation.learning_rate == 3e-5 and cfg.imitation.spectral_norm is True
  sac = config.load_config(['algorithm=SAC'])
  assert sac.reinforcement.discount == 0.99 and sac.reinforcement.polyak_factor == 0.995
  tuned = config.load_config(['algorithm=GAIL', 'optimised_hyperparameters=GAIL_5_trajectories'])
  assert tuned.training.batch_size == 1024 and tuned.imitation.loss_function == 'Mixup'
  with pytest.raises(FileNotFoundError): config.load_config(['algorithm=NOPE'])
  assert config.load_config(['algorithm=RED']).imitation.pretraining.iterations == 100000 and config.load_config(['algorithm=DRIL']).imitation.quantile_cutoff == 0.98
  assert config.load_config(['algorithm=AdRIL']).imitation.update_freq == 1250
  with pytest.raises(AttributeError): _ = cfg.training.no_such_key


CONF_FILES = (['train_config.yaml'] + [f'algorithm/{alg}.yaml' for alg in ('SAC', 'GAIL', 'GMMIL', 'PWIL', 'BC')]
              + [f'optimised_hyperparameters/{alg}_{n}_trajectories.yaml' for alg in ('BC', 'GAIL', 'GMMIL', 'PWIL') for n in (5, 10, 25)])
INIT_SEED, INIT_REPLICAS, INIT_DIMS = 7, 3, (12, 3, 256)  # S, A, H
INIT_SAMPLES, INIT_ATOL = 32, 1e-6  # orthogonal_ goes through a QR factorisation whose last bits follow the thread count and the CPU's LAPACK path


def _golden_json(name):
  with open(os.path.join(ROOT, 'tests', 'golden', name)) as f: return json.load(f)


def _init_idx(size):
  return np.random.RandomState(size).choice(size, min(size, INIT_SAMPLES), replace=False)


def _init_record(t):
  v = t.detach().double().reshape(-1)
  return dict(shape=list(t.shape), sample=v[_init_idx(v.numel())].tolist(), sum=float(v.sum()), absmax=float(v.abs().max()))


def record_reference_conf(conf_dir):
  """The values of the reference's conf/ files listed in CONF_FILES, flattened, without Hydra's own keys
  (tests/golden/reference_conf.json, written by `python -m oracle.make_golden reference_conf`)."""
  out = {}
  for name in CONF_FILES:
    with open(os.path.join(conf_dir, *name.split('/'))) as f: d = yaml.safe_load(f) or {}
    out[name] = _flat({k: v for k, v in d.items() if k not in ('defaults', 'hydra')})
  return out


def record_reference_init(ref):
  """Shape, a fixed sample of entries, sum and max |x| of every initial parameter of the reference's SoftActor and TwinCritic built after
  torch.manual_seed(INIT_SEED + r) (train.py:51-66), r < INIT_REPLICAS (tests/golden/reference_init.json, written by
  `python -m oracle.make_golden reference_init`)."""
  S, A, H = INIT_DIMS
  mc = ref.DictConfig(hidden_size=H, depth=2, activation='relu')
  out = {}
  for r in range(INIT_REPLICAS):
    torch.manual_seed(INIT_SEED + r)
    actor, critic = ref.models.SoftActor(S, A, mc), ref.models.TwinCritic(S, A, mc)
    for name, seq in (('actor', actor.actor), ('critic_1', critic.critic_1.critic), ('critic_2', critic.critic_2.critic)):
      out[f'{r}/{name}'] = [_init_record(t) for lin in seq if isinstance(lin, torch.nn.Linear) for t in (lin.weight, lin.bias)]
  return out


def test_conf_tree_carries_the_reference_values():
  """Every key of the reference's train_config.yaml / algorithm overlays / tuned overlays that this repo ships has
  the reference's value (this repo adds keys — replicas, device_rng, cuda_graphs, gemm_mode, output_dir — never changes one)."""
  ref = _golden_json('reference_conf.json')
  assert sorted(ref) == sorted(CONF_FILES)
  ours = _flat(config.load_config([]))
  for k, v in ref['train_config.yaml'].items():
    assert k in ours, f'train_config.yaml: {k} missing'
    assert ours[k] == v, (k, ours[k], v)
  for name in CONF_FILES[1:]:
    with open(os.path.join(ROOT, 'conf', *name.split('/'))) as f: mine = _flat(yaml.safe_load(f) or {})
    assert mine == ref[name], (name, mine, ref[name])


def test_parameter_initialisation_consumes_the_reference_rng_stream():
  """train.py:51-66 seeds torch once and builds actor, then the twin critic; replica r of this build must initialise
  like a reference run with seed + r (net.ReplicaRNG + net.init_fcnn_params, CPU side of ReplicaMLP)."""
  from il_b200 import net
  want = _golden_json('reference_init.json')
  S, A, H = INIT_DIMS
  rng = net.ReplicaRNG(seed=INIT_SEED, replicas=INIT_REPLICAS)
  for r in range(INIT_REPLICAS):
    with rng.replica(r):
      mine_actor = net.init_fcnn_params([S, H, H, 2 * A], 'relu')
      mine_c1, mine_c2 = net.init_fcnn_params([S + A, H, H, 1], 'relu'), net.init_fcnn_params([S + A, H, H, 1], 'relu')
    for name, mine in (('actor', mine_actor), ('critic_1', mine_c1), ('critic_2', mine_c2)):
      theirs = want[f'{r}/{name}']
      assert len(theirs) == len(mine) == 6, (r, name)
      for i, (t, ref) in enumerate(zip(mine, theirs)):
        got, where = _init_record(t), f'replica {r} {name} parameter {i}'
        assert got['shape'] == ref['shape'], where
        assert np.abs(np.subtract(got['sample'], ref['sample'])).max() <= INIT_ATOL, where
        assert abs(got['sum'] - ref['sum']) <= INIT_ATOL * t.numel() and abs(got['absmax'] - ref['absmax']) <= INIT_ATOL, where
  # the global stream is left untouched by the per-replica streams
  torch.manual_seed(123)
  a = torch.rand(3)
  torch.manual_seed(123)
  with rng.replica(0): net.init_fcnn_params([4, 4], 'relu')
  assert torch.equal(a, torch.rand(3))


def test_shard_and_statistics_helpers():
  from il_b200 import distributed
  for total, world in ((1024, 1), (1024, 8), (10, 4), (7, 8)):
    spans = [distributed.shard(total, rank, world) for rank in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == total
    assert all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:]))
    sizes = [hi - lo for lo, hi in spans]
    assert max(sizes) - min(sizes) <= 1


def test_cli_overrides_parse_like_hydra():
  """ADVICE r1: `training.learning_rate=3e-4` and `imitation.nonnegative_margin=inf` must arrive as floats (YAML 1.1 reads them as strings)."""
  from il_b200.config import load_config
  cfg = load_config(['algorithm=GAIL', 'env=hopper', 'training.learning_rate=3e-4', 'imitation.nonnegative_margin=inf', 'steps=1e5', 'training.batch_size=512',
                     'imitation.spectral_norm=false', 'imitation.loss_function=PUGAIL', 'imitation.discriminator.reward_function=FAIRL'])
  assert isinstance(cfg.training.learning_rate, float) and cfg.training.learning_rate == 3e-4
  assert cfg.imitation.nonnegative_margin == float('inf')
  assert cfg.steps == 1e5 and cfg.training.batch_size == 512 and isinstance(cfg.training.batch_size, int)
  assert cfg.imitation.spectral_norm is False and cfg.imitation.loss_function == 'PUGAIL' and cfg.imitation.discriminator.reward_function == 'FAIRL'
