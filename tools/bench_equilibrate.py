"""Spin-up to equilibrium against fixed-length runs (Ensemble.run_to_equilibrium vs Ensemble.run), on cuda:0.

    python tools/bench_equilibrate.py [--workloads C4,C2] [--max-steps 36000] [--tols 1e-8,1e-6] [--out FILE]

Per workload (C4: the 32 768-member run_JansenNadeau_2018 lattice, K = 12, checked every 1200 iterations; C2: the
65 536-member column + Psi_SO lattice, K = 72, checked every 1152 = 16 K iterations, the multiple of K nearest to
1200), each on a freshly uploaded ensemble:
  * ``fixed``: one ``run(max_steps)``;
  * ``equilibrium``: ``run_to_equilibrium(max_steps, every, tol)`` for each tolerance: wall time, member-steps
    actually executed (the sum of every member's stop), fraction converged, members stopped as non-finite;
  * ``overhead``: ``tol = 0`` (no member converges, every chunk runs every member) against the fixed run: what the
    chunking, the checks and the per-check read-back of the counter cost.
Times are CUDA events around the call (the equilibrium call synchronises with the host after every check).  The card
name and its power limit are recorded with the numbers.  Prints one JSON object.

With ``--host`` (one tolerance, default 1e-4) each workload is instead run to equilibrium with its arrays in pinned
HOST memory, alternately, twice each:
  * ``host``: ``HostEnsemble.run_to_equilibrium`` (``pmoc_host_equilibrate``; state pushed, state, streamfunctions and
    diagnostics pulled): wall time of the synchronous call and the bytes it moved;
  * ``device_then_download``: ``Ensemble.run_to_equilibrium`` followed by a download of the same arrays into pinned
    buffers: wall time to the end of the download.
Both start from the same freshly built ensemble; the two results are compared bit for bit.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pymoc_b200 import _abi, configs  # noqa: E402
from pymoc_b200.ensemble import Ensemble, HostEnsemble  # noqa: E402

WORKLOADS = {  # name -> (builder, members, every)
    'C4': (lambda M: configs.c4_jansen_nadeau(M), 32768, 1200),
    'C2': (lambda M: configs.c2_column_so(M), 65536, 1152),
}


def card():
  import torch
  out = {'name': torch.cuda.get_device_name(0)}
  try:
    q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True, timeout=30)
    out['power_limit_and_max_sm_clock'] = q.stdout.strip()
  except (OSError, subprocess.SubprocessError) as e:
    out['power_limit_and_max_sm_clock'] = 'not available: %r' % (e,)
  return out


def timed(fn):
  import torch
  start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  torch.cuda.synchronize()
  start.record()
  res = fn()
  stop.record()
  torch.cuda.synchronize()
  return start.elapsed_time(stop), res


def fresh(spec):
  ens = Ensemble(spec)
  if spec.order == 'post':
    ens.diagnose()
  ens.be.sync()
  return ens


def bench(name, max_steps, tols):
  build, M, every = WORKLOADS[name]
  spec = build(M)
  assert every % spec.K == 0 and max_steps % spec.K == 0, (name, spec.K, every, max_steps)
  warm = fresh(spec)  # module load and first launches of both paths
  warm.run(spec.K)
  warm.run_to_equilibrium(2 * every, every, 0.0)
  del warm
  out = {'workload': spec.name, 'members': M, 'nz': spec.nz, 'K': spec.K, 'every': every, 'max_steps': max_steps}
  ens = fresh(spec)
  ms, _ = timed(lambda: ens.run(max_steps, sync=False))
  out['fixed'] = {'ms': ms, 'member_steps': M * max_steps}
  fixed_ms = ms
  out['equilibrium'] = []
  for tol in tols:
    ens = fresh(spec)
    ms, r = timed(lambda: ens.run_to_equilibrium(max_steps, every, tol))
    stopped, conv = r['stopped_at'], r['converged']
    executed = int(stopped.sum())
    out['equilibrium'].append({
        'tol': tol, 'ms': ms, 'member_steps': executed, 'member_steps_vs_fixed': executed / (M * max_steps),
        'time_vs_fixed': ms / fixed_ms, 'converged_fraction': float(conv.mean()),
        'nonfinite_stopped': int(((~conv) & (stopped < max_steps)).sum()),
        'stop_quantiles': [int(q) for q in np.quantile(stopped, [0.1, 0.5, 0.9])]})
  ens = fresh(spec)
  ms, r = timed(lambda: ens.run_to_equilibrium(max_steps, every, 0.0))
  out['overhead'] = {'tol0_ms': ms, 'fixed_ms': fixed_ms, 'ratio': ms / fixed_ms,
                     'checks': max_steps // every + (max_steps % every != 0),
                     'converged_at_tol0': int(r['converged'].sum())}
  return out


def bench_host(name, max_steps, tol, reps=2):
  """The host-buffer leg: HostEnsemble.run_to_equilibrium against the device call plus a download of the same
  arrays, alternated."""
  import torch
  build, M, every = WORKLOADS[name]
  spec = build(M)
  S, P, D = _abi.IO_STATE, _abi.IO_PSI, _abi.IO_DIAG
  warm = HostEnsemble(spec)
  warm.run_to_equilibrium(2 * every, every, 0.0)
  warm.close()
  out = {'workload': spec.name, 'members': M, 'nz': spec.nz, 'K': spec.K, 'every': every, 'max_steps': max_steps,
         'tol': tol, 'host': [], 'device_then_download': []}
  for _ in range(reps):
    host = HostEnsemble(spec)
    t0 = time.perf_counter()
    r_host = host.run_to_equilibrium(max_steps, every, tol, push=S, pull=S | P | D)
    ms = (time.perf_counter() - t0) * 1e3
    h2d, d2h = host.last_bytes()
    out['host'].append({'ms': ms, 'h2d_bytes': h2d, 'd2h_bytes': d2h})

    dev = fresh(spec)
    pinned = {k: torch.empty(tuple(b.shape), dtype=b.dtype, pin_memory=True) for k, b in dev._bufs.items()
              if k != 'scratch'}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r_dev = dev.run_to_equilibrium(max_steps, every, tol)
    for k, t in pinned.items():
      t.copy_(dev._bufs[k], non_blocking=True)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    out['device_then_download'].append({'ms': ms, 'd2h_bytes': sum(t.numel() * t.element_size() for t in pinned.values())})

    same = all(np.array_equal(r_host[k], r_dev[k]) for k in r_host)
    same = same and all(np.array_equal(host.be.download(host._bufs[k]), t.numpy(), equal_nan=True)
                        for k, t in pinned.items())
    out.setdefault('identical', True)
    out['identical'] = out['identical'] and bool(same)
    out['converged_fraction'] = float(r_dev['converged'].mean())
    host.close()
    del host, dev, pinned
  h, d = min(x['ms'] for x in out['host']), min(x['ms'] for x in out['device_then_download'])
  out['host_vs_device_then_download'] = h / d
  return out


def main():
  ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
  ap.add_argument('--workloads', default='C4,C2')
  ap.add_argument('--max-steps', type=int, default=36000)
  ap.add_argument('--tols', default=None,
                  help='comma list of tolerances (buoyancy, m s^-2, per check); default 1e-8,1e-6, with --host 1e-4')
  ap.add_argument('--host', action='store_true', help='the host-buffer leg (pinned arrays) instead')
  ap.add_argument('--out', default=None, help='also write the JSON object to this file')
  args = ap.parse_args()
  tols = [float(t) for t in (args.tols or ('1e-4' if args.host else '1e-8,1e-6')).split(',')]
  if args.host:
    results = [bench_host(w, args.max_steps, tols[0]) for w in args.workloads.split(',')]
  else:
    results = [bench(w, args.max_steps, tols) for w in args.workloads.split(',')]
  res = {'card': card(), 'results': results}
  line = json.dumps(res)
  print(line)
  if args.out:
    with open(args.out, 'w') as f:
      f.write(line + '\n')


if __name__ == '__main__':
  main()
