"""Builds libbsuite_b200.so in-tree with nvcc for sm_100a.

    python -m bsuite_b200.build [--force]

The library is the only compiled artefact: CUDA kernels, the explicit host path
and the extern "C" surface of include/bsuite_b200.h.  It links cudart statically
and depends on nothing from torch.
"""

import os
import shutil
import subprocess
import sys
import time

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
FAMILIES = ('deep_sea', 'catch', 'cartpole', 'cartpole_swingup', 'mountain_car', 'memory_chain', 'bandit',
            'umbrella_chain', 'discounting_chain', 'mnist')
SOURCES = [os.path.join(CSRC, 'bsb_engine.cu'), os.path.join(CSRC, 'bsb_comm.cu'), os.path.join(CSRC, 'bsb_scoring.cu')] + [os.path.join(CSRC, f'fam_{name}.cu') for name in FAMILIES]
HEADERS = [os.path.join(CSRC, f) for f in ('bsb_rng.cuh', 'bsb_families.cuh', 'bsb_kernels.cuh', 'bsb_env.h',
                                           'bsb_dispatch.cuh', 'bsb_scoring.cuh')] + [
    os.path.join(os.path.dirname(HERE), 'include', 'bsuite_b200.h')]
OUTPUT = os.path.join(HERE, 'libbsuite_b200.so')
OBJ_DIR = os.path.join(HERE, 'build')

NVCC_FLAGS = [
    '-gencode', 'arch=compute_100a,code=sm_100a',
    '-O3', '-std=c++17', '-lineinfo',
    '--fmad=false',                       # CPython/numpy never fuse a*b+c (float-dynamics parity)
    '-Xcompiler', '-fPIC,-ffp-contract=off,-O2',
]


def find_nvcc() -> str:
  for candidate in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
    if candidate and os.path.exists(candidate):
      return candidate
  raise RuntimeError('nvcc not found: bsuite_b200 needs the CUDA toolkit to build (no CPU-only build exists)')


def _object_path(source: str) -> str:
  return os.path.join(OBJ_DIR, os.path.basename(source)[:-3] + '.o')


def _stale(target: str, deps) -> bool:
  if not os.path.exists(target):
    return True
  built = os.path.getmtime(target)
  return any(os.path.getmtime(p) > built for p in deps)


def is_stale() -> bool:
  return _stale(OUTPUT, SOURCES + HEADERS)


def _compile(nvcc: str, source: str, verbose: bool):
  cmd = [nvcc] + NVCC_FLAGS + ['-c', source, '-o', _object_path(source)]
  if os.environ.get('BSB_MIN_BLOCKS_PER_SM'):   # tuning experiment: cap registers via __launch_bounds__
    cmd.append('-DBSB_MIN_BLOCKS_PER_SM=' + os.environ['BSB_MIN_BLOCKS_PER_SM'])
  if verbose:
    cmd += ['-Xptxas', '-v']
  proc = subprocess.run(cmd, capture_output=True, text=True)
  if proc.returncode != 0:
    raise RuntimeError('nvcc failed:\n' + ' '.join(cmd) + '\n' + proc.stdout + proc.stderr)
  return proc.stderr


def build_library(force: bool = False, verbose: bool = False) -> str:
  """Compiles every translation unit for sm_100a (in parallel) and links libbsuite_b200.so in-tree."""
  import concurrent.futures
  if not force and not is_stale():
    return OUTPUT
  nvcc = find_nvcc()
  os.makedirs(OBJ_DIR, exist_ok=True)
  start = time.time()
  todo = [src for src in SOURCES if force or _stale(_object_path(src), [src] + HEADERS)]
  with concurrent.futures.ThreadPoolExecutor(max_workers=min(len(todo) or 1, os.cpu_count() or 1)) as pool:
    for log in pool.map(lambda src: _compile(nvcc, src, verbose), todo):
      if verbose:
        sys.stderr.write(log)
  cmd = [nvcc, '-shared', '-gencode', 'arch=compute_100a,code=sm_100a', '-o', OUTPUT] + [_object_path(s) for s in SOURCES] + ['-ldl']
  proc = subprocess.run(cmd, capture_output=True, text=True)
  if proc.returncode != 0:
    raise RuntimeError('link failed:\n' + ' '.join(cmd) + '\n' + proc.stdout + proc.stderr)
  sys.stderr.write(f'[bsuite_b200.build] built {OUTPUT} ({len(todo)} translation units) in {time.time() - start:.1f}s\n')
  return OUTPUT


if __name__ == '__main__':
  build_library(force='--force' in sys.argv, verbose='-v' in sys.argv)
