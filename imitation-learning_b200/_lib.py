"""ctypes binding of the C ABI in include/il_b200.h (the sm_100a shared library csrc/libil_b200.so).

PyTorch is used for device memory, streams and torch.distributed only; every hot-path computation goes through
the entry points bound here. There is no CPU fallback: creating a handle without a B200 raises.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
from typing import Dict, Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'csrc', 'libil_b200.so')
MAX_LAYERS = 6
ACT = {'relu': 0, 'tanh': 1, 'sigmoid': 2}
REWARD = {'AIRL': 0, 'GAIL': 1, 'FAIRL': 2}
LOSS = {'BCE': 0, 'Mixup': 1, 'PUGAIL': 2}
GEMM_MODE = {'fp32': 0, 'tf32x3': 1, 'tf32': 2}

c_f32p, c_i32p, c_i64p, c_u64p, vp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p  # raw device pointers


class Mlp(C.Structure):
  _fields_ = [('params', vp), ('stride', C.c_int64), ('n_layers', C.c_int32), ('activation', C.c_int32), ('dims', C.c_int32 * (MAX_LAYERS + 1)), ('_pad', C.c_int32)]


class Adam(C.Structure):
  _fields_ = [('m', vp), ('v', vp), ('step', vp), ('lr', C.c_double), ('beta1', C.c_double), ('beta2', C.c_double), ('eps', C.c_double), ('weight_decay', C.c_double), ('lr_r', vp),
              ('weight_decay_r', vp), ('replica_floats', C.c_int64)]


class Batch(C.Structure):
  _fields_ = [('rows', vp), ('replica_stride', C.c_int64), ('B', C.c_int32), ('S', C.c_int32), ('A', C.c_int32), ('row', C.c_int32)]


class Replay(C.Structure):
  _fields_ = [('rows', vp), ('replica_stride', C.c_int64), ('idx', vp), ('full', vp), ('num_trajectories', vp), ('size', C.c_int32), ('S', C.c_int32), ('A', C.c_int32),
              ('row', C.c_int32), ('absorbing', C.c_int32), ('shared', C.c_int32)]


class SacArgs(C.Structure):
  _fields_ = [('actor', Mlp), ('critic', Mlp), ('target', Mlp), ('actor_opt', Adam), ('critic_opt', Adam), ('alpha_opt', Adam), ('log_alpha', vp), ('batch', Batch),
              ('absorbing', vp), ('absorbing_from_state', C.c_int32), ('R', C.c_int32), ('eps_next', vp), ('eps_new', vp), ('discount', C.c_float),
              ('entropy_target', C.c_float), ('polyak_factor', C.c_float), ('_pad0', C.c_float), ('out_log_probs', vp), ('out_q_values', vp), ('out_losses', vp),
              ('workspace', vp), ('workspace_bytes', C.c_int64), ('discount_r', vp), ('entropy_target_r', vp), ('polyak_r', vp)]


class BcArgs(C.Structure):
  _fields_ = [('actor', Mlp), ('opt', Adam), ('batch', Batch), ('R', C.c_int32), ('_pad', C.c_int32), ('out_loss', vp), ('workspace', vp), ('workspace_bytes', C.c_int64)]


class Gail(C.Structure):
  _fields_ = [('g', Mlp), ('u', vp), ('v', vp), ('u_stride', C.c_int32), ('v_stride', C.c_int32), ('state_only', C.c_int32), ('reward_function', C.c_int32)]


class GailUpdateArgs(C.Structure):
  _fields_ = [('disc', Gail), ('opt', Adam), ('policy', Batch), ('expert', Batch), ('eps_gp', vp), ('eps_mix', vp), ('R', C.c_int32), ('loss_function', C.c_int32),
              ('training', C.c_int32), ('_pad', C.c_int32), ('grad_penalty', C.c_float), ('entropy_bonus', C.c_float), ('pos_class_prior', C.c_float),
              ('nonnegative_margin', C.c_float), ('out_losses', vp), ('workspace', vp), ('workspace_bytes', C.c_int64), ('grad_penalty_r', vp), ('entropy_bonus_r', vp)]


class Gailx(C.Structure):
  _fields_ = [('g', Mlp), ('h', Mlp), ('g_u', vp), ('g_v', vp), ('h_u', vp), ('h_v', vp), ('g_u_stride', C.c_int32), ('g_v_stride', C.c_int32), ('h_u_stride', C.c_int32),
              ('h_v_stride', C.c_int32), ('state_only', C.c_int32), ('reward_function', C.c_int32), ('subtract_log_policy', C.c_int32), ('discount', C.c_float),
              ('discount_r', vp)]


class GailxUpdateArgs(C.Structure):
  _fields_ = [('disc', Gailx), ('opt', Adam), ('params_floats', C.c_int64), ('policy', Batch), ('expert', Batch), ('eps_gp', vp), ('eps_mix', vp), ('logp_policy', vp),
              ('logp_expert', vp), ('logp_mix', vp), ('R', C.c_int32), ('loss_function', C.c_int32), ('training', C.c_int32), ('_pad', C.c_int32), ('grad_penalty', C.c_float),
              ('entropy_bonus', C.c_float), ('pos_class_prior', C.c_float), ('nonnegative_margin', C.c_float), ('out_losses', vp), ('workspace', vp), ('workspace_bytes', C.c_int64),
              ('grad_penalty_r', vp), ('entropy_bonus_r', vp)]


class Red(C.Structure):
  _fields_ = [('predictor', Mlp), ('target', Mlp), ('sigma', vp), ('state_only', C.c_int32), ('_pad', C.c_int32)]


class RedUpdateArgs(C.Structure):
  _fields_ = [('disc', Red), ('opt', Adam), ('batch', Batch), ('R', C.c_int32), ('_pad', C.c_int32), ('mask_in', vp), ('mask_hid', vp * MAX_LAYERS), ('out_loss', vp), ('workspace', vp),
              ('workspace_bytes', C.c_int64)]


class Pwil(C.Structure):
  _fields_ = [('atoms', vp), ('scale', vp), ('offset', vp), ('weights', vp), ('N', C.c_int32), ('d', C.c_int32), ('S', C.c_int32), ('A', C.c_int32), ('state_only', C.c_int32),
              ('time_horizon', C.c_int32), ('reward_scale', C.c_float), ('reward_bandwidth', C.c_float),
              ('reward_scale_r', vp), ('reward_bandwidth_r', vp)]


class Env(C.Structure):
  _fields_ = [('M', vp), ('N', vp), ('c', vp), ('w_r', vp), ('x', vp), ('t', vp), ('obs', C.c_int32), ('act', C.c_int32), ('absorbing', C.c_int32),
              ('max_episode_steps', C.c_int32), ('early_termination', C.c_int32), ('term_threshold', C.c_float)]


class EvalArgs(C.Structure):
  _fields_ = [('actor', Mlp), ('env', Env), ('R', C.c_int32), ('episodes', C.c_int32), ('max_steps', C.c_int32), ('traj_T', C.c_int32), ('state', vp), ('returns', vp),
              ('traj_states', vp), ('traj_actions', vp), ('traj_rewards', vp), ('traj_len', vp), ('out_counters', vp), ('workspace', vp), ('workspace_bytes', C.c_int64)]


i32, i64, u64, f32 = C.c_int32, C.c_int64, C.c_uint64, C.c_float
P = C.POINTER

# name -> (restype, argtypes); must list every symbol declared in include/il_b200.h (tests/test_abi.py checks)
SIGNATURES = {
  'il_create': (C.c_int, [C.c_int, P(vp)]),
  'il_destroy': (C.c_int, [vp]),
  'il_last_error': (C.c_char_p, []),
  'il_version': (C.c_int, []),
  'il_set_gemm_mode': (C.c_int, [vp, C.c_int]),
  'il_launch_count': (i64, [vp]),
  'il_set_option': (C.c_int, [vp, C.c_char_p, C.c_int]),
  'il_struct_sizes': (C.c_int, [P(i32)]),
  'il_mlp_param_offsets': (C.c_int, [P(i32), C.c_int, P(i64), P(i64), P(i64)]),
  'il_row_layout': (C.c_int, [C.c_int, C.c_int, P(i32), P(i32)]),
  'il_profile_begin': (C.c_int, [vp]),
  'il_profile_end': (C.c_int, [vp, P(C.c_double), P(C.c_double), P(i64)]),
  'il_profile_bytes': (C.c_int, [vp, P(C.c_double)]),
  'il_debug_gemm': (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, i64, C.c_int, C.c_int, vp, i64, C.c_int, C.c_int, vp, i64, C.c_int, vp, i64, C.c_int, vp, i64, C.c_int,
                              C.c_int, vp, i64, vp]),
  'il_fill_normal': (C.c_int, [vp, vp, i64, u64, u64, vp, vp]),
  'il_fill_uniform': (C.c_int, [vp, vp, i64, u64, u64, vp, vp]),
  'il_counter_add': (C.c_int, [vp, vp, u64, vp]),
  'il_replica_copy': (C.c_int, [vp, C.c_int, P(vp), P(i64), P(i64), C.c_int, vp, vp]),
  'il_actor_workspace_bytes': (i64, [P(Mlp), C.c_int, C.c_int]),
  'il_actor_forward': (C.c_int, [vp, P(Mlp), C.c_int, C.c_int, vp, i64, C.c_int, vp, vp, vp, vp, vp, vp, vp, i64, vp]),
  'il_critic_workspace_bytes': (i64, [P(Mlp), C.c_int, C.c_int]),
  'il_critic_forward': (C.c_int, [vp, P(Mlp), C.c_int, C.c_int, C.c_int, vp, i64, C.c_int, vp, i64, C.c_int, vp, vp, vp, i64, vp]),
  'il_polyak': (C.c_int, [vp, vp, vp, i64, f32, vp]),
  'il_sac_workspace_bytes': (i64, [P(SacArgs)]),
  'il_sac_update': (C.c_int, [vp, P(SacArgs), vp]),
  'il_bc_workspace_bytes': (i64, [P(BcArgs)]),
  'il_bc_update': (C.c_int, [vp, P(BcArgs), vp]),
  'il_adam_step': (C.c_int, [vp, vp, vp, P(Adam), i64, vp]),
  'il_adam_step_polyak': (C.c_int, [vp, vp, vp, P(Adam), i64, vp, C.c_float, vp]),
  'il_fill_dropout_mask': (C.c_int, [vp, vp, i64, f32, u64, u64, vp, vp]),
  'il_actor_dropout_workspace_bytes': (i64, [P(Mlp), C.c_int, C.c_int]),
  'il_actor_log_prob_dropout': (C.c_int, [vp, P(Mlp), C.c_int, C.c_int, C.c_int, vp, i64, C.c_int, vp, vp, P(vp), vp, vp, i64, vp]),
  'il_bc_update_dropout': (C.c_int, [vp, P(BcArgs), vp, P(vp), vp]),
  'il_dril_reward': (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, i64, C.c_int, vp, vp]),
  'il_red_workspace_bytes': (i64, [P(Red), C.c_int, C.c_int]),
  'il_red_update': (C.c_int, [vp, P(RedUpdateArgs), vp]),
  'il_red_sigma': (C.c_int, [vp, P(Red), C.c_int, P(Batch), vp, P(vp), vp, i64, vp]),
  'il_red_reward': (C.c_int, [vp, P(Red), C.c_int, P(Batch), vp, i64, C.c_int, vp, i64, vp]),
  'il_replay_append': (C.c_int, [vp, P(Replay), C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, C.c_int, vp]),
  'il_replay_wrap_absorbing': (C.c_int, [vp, P(Replay), C.c_int, vp, vp]),
  'il_replay_transfer': (C.c_int, [vp, P(Replay), C.c_int, P(Replay), vp]),
  'il_replay_sample_indices': (C.c_int, [vp, P(Replay), C.c_int, C.c_int, vp, vp, u64, u64, vp, vp]),
  'il_replay_gather': (C.c_int, [vp, P(Replay), C.c_int, vp, P(Batch), vp]),
  'il_mix_expert_rows': (C.c_int, [vp, P(Batch), P(Batch), C.c_int, vp]),
  'il_adril_relabel': (C.c_int, [vp, P(Batch), P(Batch), C.c_int, C.c_int, C.c_int, vp, vp, f32, vp, C.c_int, C.c_int, vp]),
  'il_gail_workspace_bytes': (i64, [P(GailUpdateArgs)]),
  'il_gail_update': (C.c_int, [vp, P(GailUpdateArgs), vp]),
  'il_gail_reward': (C.c_int, [vp, P(Gail), C.c_int, P(Batch), vp, i64, C.c_int, vp, vp]),
  'il_gailx_workspace_bytes': (i64, [P(GailxUpdateArgs)]),
  'il_gailx_update': (C.c_int, [vp, P(GailxUpdateArgs), vp]),
  'il_gailx_reward_workspace_bytes': (i64, [P(Gailx), C.c_int, C.c_int]),
  'il_gailx_reward': (C.c_int, [vp, P(Gailx), C.c_int, P(Batch), vp, vp, i64, C.c_int, vp, vp, i64, vp]),
  'il_gail_mix_batch': (C.c_int, [vp, P(Batch), P(Batch), vp, C.c_int, P(Batch), vp]),
  'il_gmmil_workspace_bytes': (i64, [C.c_int, C.c_int]),
  'il_gmmil_bandwidth': (C.c_int, [vp, C.c_int, P(Batch), P(Batch), C.c_int, vp, vp, i64, vp]),
  'il_gmmil_reward': (C.c_int, [vp, C.c_int, P(Batch), P(Batch), C.c_int, vp, vp, i64, C.c_int, vp]),
  'il_pwil_reset': (C.c_int, [vp, P(Pwil), C.c_int, vp, vp]),
  'il_pwil_reward': (C.c_int, [vp, P(Pwil), C.c_int, vp, vp, vp, vp, vp]),
  'il_env_reset': (C.c_int, [vp, P(Env), C.c_int, vp, vp, vp, vp, vp]),
  'il_env_step': (C.c_int, [vp, P(Env), C.c_int, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
  'il_rollout_bookkeep': (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, vp, vp, vp]),
  'il_eval_accumulate': (C.c_int, [vp, C.c_int, vp, vp, vp, vp, vp, vp]),
  'il_return_stats': (C.c_int, [vp, vp, i64, vp, vp]),
  'il_eval_workspace_bytes': (i64, [P(EvalArgs)]),
  'il_eval_rollout': (C.c_int, [vp, P(EvalArgs), vp]),
  'il_nccl_unique_id': (C.c_int, [vp]),
  'il_nccl_comm_create': (C.c_int, [vp, C.c_int, C.c_int, P(vp)]),
  'il_nccl_comm_destroy': (C.c_int, [vp]),
  'il_return_allreduce': (C.c_int, [vp, vp, vp, i64, vp, vp]),
}

_lock = threading.Lock()
_lib: Optional[C.CDLL] = None
_handles: Dict[int, int] = {}


def build(force: bool = False, verbose: bool = False) -> str:
  """Compiles csrc/*.cu for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
  import importlib.util
  spec = importlib.util.spec_from_file_location('il_b200_csrc_build', os.path.join(_HERE, 'csrc', 'build.py'))
  mod = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(mod)
  return mod.build(force=force, verbose=verbose)


def lib() -> C.CDLL:
  """Loads (building if needed) the shared library and binds every declared symbol."""
  global _lib
  with _lock:
    if _lib is None:
      if not os.path.exists(LIB_PATH): build()
      l = C.CDLL(LIB_PATH)
      for name, (res, args) in SIGNATURES.items():
        fn = getattr(l, name)  # AttributeError if the library does not export a declared symbol
        fn.restype, fn.argtypes = res, args
      _lib = l
  return _lib


def last_error() -> str:
  return lib().il_last_error().decode()


def check(rc: int):
  if rc != 0: raise RuntimeError(f'il_b200: {last_error()}')


def handle(device: Optional[int] = None) -> int:
  """One library handle per CUDA device; fails loudly when there is no B200 (no CPU fallback)."""
  if not torch.cuda.is_available():
    raise RuntimeError('il_b200: no CUDA device available; the hot path only exists as sm_100a kernels (no CPU fallback)')
  device = torch.cuda.current_device() if device is None else device
  with _lock:
    h = _handles.get(device)
  if h is None:
    out = vp()
    check(lib().il_create(device, C.byref(out)))
    h = out.value
    with _lock: _handles[device] = h
    mode = os.environ.get('IL_GEMM_MODE')
    if mode: check(lib().il_set_gemm_mode(h, GEMM_MODE[mode]))
  return h


def set_option(name: str, value: int):
  check(lib().il_set_option(handle(), name.encode(), int(value)))


def stream() -> int:
  return torch.cuda.current_stream().cuda_stream


def launch_count() -> int:
  return int(lib().il_launch_count(handle()))


def mask_array(masks):
  """ctypes array of MAX_LAYERS device pointers (NULL-padded) for the per-hidden-layer dropout masks."""
  arr = (vp * MAX_LAYERS)()
  for i, t in enumerate(masks or []): arr[i] = None if t is None else t.data_ptr()
  return arr


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
  if t is None: return None
  assert t.is_cuda, 'il_b200 expects CUDA tensors'
  return t.data_ptr()


def mlp_offsets(dims):
  n = len(dims) - 1
  d = (i32 * len(dims))(*dims)
  w, b, tot = (i64 * n)(), (i64 * n)(), i64()
  check(lib().il_mlp_param_offsets(d, n, w, b, C.byref(tot)))
  return list(w), list(b), tot.value


def row_layout(S: int, A: int):
  off, n = (i32 * 8)(), i32()
  check(lib().il_row_layout(S, A, off, C.byref(n)))
  names = ('states', 'actions', 'rewards', 'next_states', 'terminals', 'timeouts', 'weights', 'step')
  return dict(zip(names, list(off))), n.value


def py_mlp_offsets(dims):
  """Pure-Python mirror of il_mlp_param_offsets (usable without loading the library)."""
  al = lambda x, a: (x + a - 1) // a * a
  off, w, b = 0, [], []
  for l in range(len(dims) - 1):
    w.append(off)
    off = al(off + dims[l + 1] * dims[l], 4)
    b.append(off)
    off = al(off + dims[l + 1], 4)
  return w, b, al(off, 32)


def py_row_layout(S: int, A: int):
  off = dict(states=0, actions=S, rewards=S + A, next_states=S + A + 1, terminals=2 * S + A + 1, timeouts=2 * S + A + 2, weights=2 * S + A + 3, step=2 * S + A + 4)
  return off, (2 * S + A + 5 + 3) // 4 * 4
