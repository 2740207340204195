"""Builds libdqnzoo_b200.so in-tree with nvcc for sm_100a (no GPU needed: cross-compile)."""

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, 'csrc')
LIB_DIR = os.path.join(HERE, 'lib')
LIB_PATH = os.path.join(LIB_DIR, 'libdqnzoo_b200.so')
SOURCES = ['dz_replay.cu', 'dz_frames.cu', 'dz_learner.cu', 'dz_tcp.cu', 'dz_umma.cu', 'dz_umma_net.cu', 'dz_preprocess.cu', 'dz_jaxprng.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC', '--expt-relaxed-constexpr']


def _nvcc():
  for cand in (os.environ.get('NVCC'), '/usr/local/cuda/bin/nvcc', 'nvcc'):
    if cand and (os.path.sep not in cand or os.path.exists(cand)):
      return cand
  raise RuntimeError('nvcc not found')


def needs_build():
  if not os.path.exists(LIB_PATH):
    return True
  t = os.path.getmtime(LIB_PATH)
  deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, '..', 'include', 'dqn_zoo_b200.h')]
  return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
  """Compiles every .cu under csrc/ and links the shared library.  Returns its path."""
  if not force and not needs_build():
    return LIB_PATH
  os.makedirs(LIB_DIR, exist_ok=True)
  objs = []
  procs = []
  for src in SOURCES:
    obj = os.path.join(LIB_DIR, src.replace('.cu', '.o'))
    cmd = [_nvcc()] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', os.path.join(CSRC, src), '-o', obj]
    procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs.append(obj)
  for src, p in procs:
    out, _ = p.communicate()
    if verbose or p.returncode:
      sys.stderr.write(out)
    if p.returncode:
      raise RuntimeError('nvcc failed on %s' % src)
  cmd = [_nvcc(), '-gencode', 'arch=compute_100a,code=sm_100a', '-shared', '-o', LIB_PATH] + objs
  subprocess.check_call(cmd)
  return LIB_PATH


if __name__ == '__main__':
  print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
