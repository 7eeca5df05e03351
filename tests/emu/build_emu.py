"""Build the CPU warp-emulator twin of the kernel library -- TEST INFRASTRUCTURE ONLY.

Compiles the product kernel sources (pymoc_b200/csrc/*.cu) with g++ and -DPMOC_EMU against
tests/emu/pmoc_emu.cpp into tests/emu/_pmoc_emu.so.  It exports the same C ABI with host
pointers standing in for device pointers, which lets `-m "not gpu"` tests exercise the
kernel logic on a GPU-less box.  The package never loads it.
"""
import concurrent.futures as cf
import hashlib
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
CSRC = os.path.join(ROOT, 'pymoc_b200', 'csrc')
OBJ = os.path.join(HERE, 'build')
LIB = os.path.join(HERE, '_pmoc_emu.so')
# blocks of two members in the host-buffer entry points: a test-sized ensemble already spans several blocks
# and all three streams
FLAGS = ['-O2', '-std=c++17', '-fPIC', '-ffp-contract=off', '-DPMOC_EMU', '-DPMOC_HOST_BLOCK_MEMBERS=2', '-I', HERE,
         '-Wno-unknown-pragmas']
LPLS = (2, 3, 4, 5, 6, 7, 8)


def _digest():
  h = hashlib.sha256()
  for d in (CSRC, HERE):
    for name in sorted(os.listdir(d)):
      if name.endswith(('.cu', '.cuh', '.cpp', '.h')):
        h.update(open(os.path.join(d, name), 'rb').read())
  h.update(open(os.path.join(ROOT, 'include', 'pymoc_b200.h'), 'rb').read())
  h.update(' '.join(FLAGS).encode())
  return h.hexdigest()


def _compile(src, obj, defs, lang):
  cmd = ['g++'] + FLAGS + defs + lang + ['-c', src, '-o', os.path.join(OBJ, obj)]
  r = subprocess.run(cmd, capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError('g++ failed for %s:\n%s' % (src, (r.stdout + r.stderr)[-6000:]))
  return os.path.join(OBJ, obj)


def build(force=False):
  os.makedirs(OBJ, exist_ok=True)
  stamp = os.path.join(OBJ, 'stamp')
  digest = _digest()
  if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == digest:
    return LIB
  cu = ['-x', 'c++']
  jobs = [(os.path.join(CSRC, 'pmoc_ops.cu'), 'ops.o', [], cu), (os.path.join(CSRC, 'pmoc_host.cu'), 'host.o', [], cu),
          (os.path.join(CSRC, 'pmoc_wide.cu'), 'wide.o', [], cu), (os.path.join(CSRC, 'pmoc_twcol.cu'), 'twcol.o', [], cu),
          (os.path.join(HERE, 'pmoc_emu.cpp'), 'emu.o', [], [])]
  jobs += [(os.path.join(CSRC, 'pmoc_model.cu'), 'model_%d.o' % n, ['-DPM_LPL=%d' % n], cu) for n in LPLS]
  with cf.ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:
    objs = list(ex.map(lambda j: _compile(*j), jobs))
  r = subprocess.run(['g++', '-shared', '-o', LIB] + objs + ['-lpthread'], capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError('link failed:\n' + r.stdout + r.stderr)
  open(stamp, 'w').write(digest)
  return LIB


if __name__ == '__main__':
  print(build(force=True))
