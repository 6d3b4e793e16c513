"""Per-replica hyperparameters entry point by entry point (R = 4, small shapes and H = 256 / B = 256): arrays that all hold one value set
equal the scalar call on every output and state buffer, and with four different value sets replica k equals replica k of the scalar call
with set k — bit for bit. il_gail_update runs on both the register-tiled and the untiled kernel, with BCE, Mixup and PUGAIL and spectral
norm, and with a zero gradient penalty on one replica (the fused kernels choose the penalty pass per replica)."""

import pytest
import torch

pytestmark = pytest.mark.gpu
R = 4
LR = [3e-4, 1e-3, 5e-5, 2.5e-4]
WD = [0.0, 0.01, 8.5, 0.5]


class Cfg(dict):
  def __getattr__(self, k):
    v = self[k]
    return Cfg(v) if isinstance(v, dict) and not isinstance(v, Cfg) else v

  def get(self, k, d=None): return dict.get(self, k, d)


def _gen(seed): return torch.Generator().manual_seed(seed)


def _batch(S, A, B, seed, absorbing=True):
  import il_b200
  g = _gen(seed)
  u = lambda *s: torch.rand(*s, generator=g)
  d = dict(step=torch.arange(B, dtype=torch.float32).expand(R, B).clone(), states=torch.randn(R, B, S, generator=g), actions=u(R, B, A) * 1.8 - 0.9,
           rewards=torch.randn(R, B, generator=g), next_states=torch.randn(R, B, S, generator=g), terminals=(u(R, B) < 0.1).float(), timeouts=torch.zeros(R, B),
           weights=0.5 + u(R, B))
  return il_b200.TransitionBatch.from_dict({k: v.cuda() for k, v in d.items()}, absorbing=absorbing, device='cuda')


def _gemm(mode):
  from il_b200 import _lib
  _lib.check(_lib.lib().il_set_gemm_mode(_lib.handle(), _lib.GEMM_MODE[mode]))


@pytest.fixture(autouse=True)
def _restore_defaults():
  yield
  from il_b200 import _lib
  _gemm('fp32')
  _lib.set_option('gail_tiled', 1)


def _check(run, per, sets):
  """per: {name: [R] values}; sets[k]: the scalar values of replica k. Broadcast (set 1 everywhere) == scalar set 1; replica k == scalar set k."""
  out = run(per)
  bc = run({k: [v[1]] * R for k, v in per.items()})
  for k in range(R):
    ref = run(sets[k])
    assert set(ref) == set(out)
    for name, t in ref.items():
      assert torch.equal(out[name][k], t[k]), f'replica {k} differs from its scalar call in {name}'
      if k == 1: assert torch.equal(bc[name], t), f'broadcast arrays differ from the scalar call in {name}'


def _arrays(per, dtype=torch.float64):
  return {k: torch.tensor(v, dtype=dtype, device='cuda') if isinstance(v, list) else v for k, v in per.items()}


def _sets(per): return [{k: v[i] for k, v in per.items()} for i in range(R)]


def _state(**named):
  return {k: v.detach().clone().reshape(R, -1) for k, v in named.items()}


@pytest.mark.parametrize('tiled', [1, 0])
@pytest.mark.parametrize('loss', ['BCE', 'Mixup', 'PUGAIL'])
@pytest.mark.parametrize('H,B', [(64, 32), (256, 256)])
def test_gail_update(tiled, loss, H, B):
  import il_b200
  from il_b200 import _lib
  S, A = 11, 3
  per = dict(lr=LR, wd=WD, gp=[1.0, 0.28, 0.0, 5.0], eb=[0.0, 0.24, 1e-3, 0.5])
  pol, exp = [_batch(S, A, B, 10 + s) for s in range(2)], [_batch(S, A, B, 20 + s) for s in range(2)]
  g = _gen(3)
  eps_gp, eps_mix = [torch.rand(R, B, generator=g).cuda() for _ in range(2)], [torch.rand(R, B, generator=g).cuda() for _ in range(2)]
  icfg = Cfg(state_only=False, spectral_norm=True, loss_function=loss, grad_penalty=1.0, mixup_alpha=1, entropy_bonus=0.0, pos_class_prior=0.7, nonnegative_margin=0.1,
             discriminator=Cfg(hidden_size=H, depth=1, activation='relu', input_dropout=0.5, dropout=0.75, reward_shaping=False, subtract_log_policy=False, reward_function='AIRL'))
  def run(v):
    _lib.set_option('gail_tiled', tiled)
    torch.manual_seed(0)
    disc = il_b200.GAILDiscriminator(S, A, icfg, 0.97, replicas=R)
    assert not disc.general
    a = _arrays(v)
    opt = il_b200.AdamW(disc.parameters(), lr=a['lr'], weight_decay=a['wd'])
    losses = torch.zeros(R, 2, device='cuda')
    for s in range(2):
      disc.train()
      il_b200.adversarial_imitation_update(None, disc, pol[s], exp[s], opt, icfg, eps_gp=eps_gp[s], eps_mix=eps_mix[s], out_losses=losses, grad_penalty=a['gp'],
                                           entropy_bonus=a['eb'])
    torch.cuda.synchronize()
    return _state(params=disc.mlp.flat, m=opt.exp_avg, v=opt.exp_avg_sq, u=disc.u, sn_v=disc.v, losses=losses)
  _check(run, per, _sets(per))


@pytest.mark.parametrize('loss', ['BCE', 'Mixup'])
def test_gailx_update_shaping_log_policy(loss):
  import il_b200
  S, A, H, B = 11, 3, 32, 32
  per = dict(lr=LR, wd=WD, gp=[1.0, 0.28, 2.0, 5.0], eb=[0.0, 0.24, 1e-3, 0.5], discount=[0.97, 0.9, 0.999, 0.5])
  pol, exp = _batch(S, A, B, 10), _batch(S, A, B, 20)
  g = _gen(3)
  eps_gp, eps_mix = torch.rand(R, B, generator=g).cuda(), torch.rand(R, B, generator=g).cuda()
  icfg = Cfg(state_only=False, spectral_norm=True, loss_function=loss, grad_penalty=1.0, mixup_alpha=1, entropy_bonus=0.0, pos_class_prior=0.7, nonnegative_margin=float('inf'),
             discriminator=Cfg(hidden_size=H, depth=1, activation='relu', input_dropout=0.5, dropout=0.75, reward_shaping=True, subtract_log_policy=True, reward_function='AIRL'))
  torch.manual_seed(1)
  actor = il_b200.SoftActor(S, A, Cfg(hidden_size=32, depth=2, activation='relu'), replicas=R)
  def run(v):
    torch.manual_seed(0)
    a = _arrays(v)
    disc = il_b200.GAILDiscriminator(S, A, icfg, a['discount'], replicas=R)
    assert disc.general
    opt = il_b200.AdamW(disc.parameters(), lr=a['lr'], weight_decay=a['wd'])
    losses = torch.zeros(R, 2, device='cuda')
    for _ in range(2):
      disc.train()
      il_b200.adversarial_imitation_update(actor, disc, pol, exp, opt, icfg, eps_gp=eps_gp, eps_mix=eps_mix, out_losses=losses, grad_penalty=a['gp'], entropy_bonus=a['eb'],
                                           grad_penalty_any=True)
    disc.eval()
    lp = actor._run(pol.rows[..., :S], given=pol.rows[..., S:S + A], want=('log_prob', ))['log_prob']
    res = disc._run(pol, want_logits=True, log_policy=lp)
    torch.cuda.synchronize()
    return _state(params=disc.flat, m=opt.exp_avg, v=opt.exp_avg_sq, g_u=disc.g_u, g_v=disc.g_v, h_u=disc.h_u, h_v=disc.h_v, losses=losses, reward=res['reward'],
                  logits=res['logits'])
  _check(run, per, _sets(per))


@pytest.mark.parametrize('H,B,mode', [(64, 32, 'fp32'), (256, 256, 'tf32x3')])
def test_sac_update(H, B, mode):
  import il_b200
  S, A = 11, 3
  per = dict(lr=LR, wd=WD, discount=[0.99, 0.97, 0.9, 0.999], entropy_target=[-3.0, -1.5, -6.0, -2.43], polyak=[0.995, 0.98, 0.9, 0.971])
  batches = [_batch(S, A, B, 30 + s) for s in range(2)]
  g = _gen(4)
  eps = [(torch.randn(R, B, A, generator=g).cuda(), torch.randn(R, B, A, generator=g).cuda()) for _ in range(2)]
  mcfg = Cfg(hidden_size=H, depth=2, activation='relu')
  def run(v):
    _gemm(mode)
    torch.manual_seed(0)
    actor, critic = il_b200.SoftActor(S, A, mcfg, replicas=R), il_b200.TwinCritic(S, A, mcfg, replicas=R)
    target = il_b200.create_target_network(critic)
    log_alpha = torch.full((R, ), 0.1, device='cuda')
    a = _arrays(v)
    oa, oc = il_b200.AdamW(actor.parameters(), lr=a['lr'], weight_decay=a['wd']), il_b200.AdamW(critic.parameters(), lr=a['lr'], weight_decay=a['wd'])
    ot = il_b200.Adam([log_alpha], lr=a['lr'])
    f32 = lambda x: x.float() if torch.is_tensor(x) else x
    out = {}
    for s in range(2):
      il_b200.sac_update(actor, critic, log_alpha, target, batches[s], oa, oc, ot, f32(a['discount']), f32(a['entropy_target']), f32(a['polyak']), eps_next=eps[s][0],
                         eps_new=eps[s][1], out=out)
    torch.cuda.synchronize()
    return _state(actor=actor.mlp.flat, critic=critic.mlp.flat, target=target.mlp.flat, log_alpha=log_alpha, am=oa.exp_avg, av=oa.exp_avg_sq, cm=oc.exp_avg, cv=oc.exp_avg_sq,
                  tm=ot.exp_avg, tv=ot.exp_avg_sq, **{f'out_{k}': t for k, t in out.items()})
  _check(run, per, _sets(per))


@pytest.mark.parametrize('dropout', [False, True])
@pytest.mark.parametrize('H,B,mode', [(64, 32, 'fp32'), (256, 256, 'tf32x3')])
def test_bc_update(dropout, H, B, mode):
  import il_b200
  S, A = 11, 3
  per = dict(lr=LR, wd=WD)
  batches = [_batch(S, A, B, 40 + s, absorbing=False) for s in range(2)]
  g = _gen(5)
  mask = lambda w, p: ((torch.rand(R, B, w, generator=g) >= p).float() / (1 - p)).cuda()
  masks = [[mask(S, 0.2), mask(H, 0.3), mask(H, 0.3)] for _ in range(2)] if dropout else [None, None]
  mcfg = Cfg(hidden_size=H, depth=2, activation='relu', input_dropout=0.2 if dropout else 0, dropout=0.3 if dropout else 0)
  def run(v):
    _gemm(mode)
    torch.manual_seed(0)
    actor = il_b200.SoftActor(S, A, mcfg, replicas=R)
    a = _arrays(v)
    opt = il_b200.AdamW(actor.parameters(), lr=a['lr'], weight_decay=a['wd'])
    loss = torch.zeros(R, device='cuda')
    for s in range(2): il_b200.behavioural_cloning_update(actor, batches[s], opt, out_loss=loss, masks=masks[s])
    torch.cuda.synchronize()
    return _state(actor=actor.mlp.flat, m=opt.exp_avg, v=opt.exp_avg_sq, loss=loss)
  _check(run, per, _sets(per))


def test_red_update():
  import il_b200
  S, A, H, B = 11, 3, 64, 32
  per = dict(lr=LR, wd=WD)
  batches = [_batch(S, A, B, 50 + s, absorbing=False) for s in range(2)]
  g = _gen(6)
  mask = lambda w, p: ((torch.rand(R, B, w, generator=g) >= p).float() / (1 - p)).cuda()
  masks = [[mask(S + A, 0.2), mask(H, 0.3)] for _ in range(2)]
  icfg = Cfg(state_only=False, reward_bandwidth_scale=None, discriminator=Cfg(hidden_size=H, depth=1, activation='relu', input_dropout=0.2, dropout=0.3))
  def run(v):
    torch.manual_seed(0)
    disc = il_b200.REDDiscriminator(S, A, icfg, replicas=R)
    a = _arrays(v)
    opt = il_b200.AdamW(disc.parameters(), lr=a['lr'], weight_decay=a['wd'])
    loss = torch.zeros(R, device='cuda')
    for s in range(2): il_b200.target_estimation_update(disc, batches[s], opt, out_loss=loss, masks=masks[s])
    torch.cuda.synchronize()
    return _state(predictor=disc.predictor.flat, m=opt.exp_avg, v=opt.exp_avg_sq, loss=loss)
  _check(run, per, _sets(per))


def test_pwil_reward():
  import il_b200
  S, A, N, T = 11, 3, 40, 8
  per = dict(scale=[5.0, 1.0, 10.0, 0.5], bandwidth=[5.0, 2.0, 0.5, 9.0])
  g = _gen(7)
  z = torch.zeros
  mem = il_b200.ReplayMemory(N, S, A, True, transitions=dict(states=torch.randn(N, S, generator=g).cuda(), actions=torch.rand(N, A, generator=g).cuda() - 0.5, rewards=z(N),
                                                            next_states=z(N, S), terminals=z(N), timeouts=z(N), weights=torch.ones(N), num_trajectories=1), shared=True)
  states, actions = torch.randn(T + 3, R, S, generator=g).cuda(), (torch.rand(T + 3, R, A, generator=g) - 0.5).cuda()
  def run(v):
    a = _arrays(v)
    d = il_b200.PWILDiscriminator(S, A, Cfg(state_only=False, reward_scale=5, reward_bandwidth_scale=5), mem, T, replicas=R, reward_scale=a['scale'],
                                  reward_bandwidth_scale=a['bandwidth'])
    rewards = []
    for i in range(T + 3):
      rewards.append(d.compute_reward_batch(states[i], actions[i]).clone())
      if (i + 1) % T == 0: d.reset()
    torch.cuda.synchronize()
    return _state(rewards=torch.stack(rewards, dim=1), weights=d.expert_weights)
  _check(run, per, _sets(per))
