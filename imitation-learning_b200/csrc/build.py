"""Builds libil_b200.so in-tree with nvcc for sm_100a only (no other arch, no fallback)."""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = ['api.cu', 'gemm.cu', 'tc_gemm.cu', 'mlp.cu', 'sac.cu', 'replay.cu', 'env.cu', 'eval.cu', 'gail.cu', 'gail_general.cu', 'dropout_nets.cu', 'gmmil_pwil.cu', 'replica.cu']
LIB = os.path.join(HERE, 'libil_b200.so')
NVCC = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17', '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _stale(target, deps):
  if not os.path.exists(target): return True
  t = os.path.getmtime(target)
  return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
  headers = [os.path.join(HERE, f) for f in os.listdir(HERE) if f.endswith(('.cuh', '.h'))] + [os.path.join(HERE, '..', '..', 'include', 'il_b200.h')]
  objs, procs = [], []
  for src in SOURCES:
    s, o = os.path.join(HERE, src), os.path.join(HERE, src.replace('.cu', '.o'))
    objs.append(o)
    if force or _stale(o, [s] + headers):
      cmd = [NVCC] + FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', s, '-o', o]
      procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
  failed = False
  for src, pr in procs:
    out, _ = pr.communicate()
    if pr.returncode != 0 or verbose: print(f'--- {src}\n{out}')
    failed |= pr.returncode != 0
  if failed: raise RuntimeError('nvcc failed')
  if force or procs or _stale(LIB, objs):
    subprocess.check_call([NVCC, '-shared', '-o', LIB] + objs + ['-lcudart', '-ldl'])
  return LIB


if __name__ == '__main__':
  print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
