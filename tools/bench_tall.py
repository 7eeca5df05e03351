"""Throughput of the 'post'-order models above one warp's 256 levels (block-per-member kernels), on cuda:0.

    python tools/bench_tall.py [--out FILE.jsonl]

For each shape: C2 (column + Psi_SO) at nz = 256 (the warp kernel, for the cost of crossing the dispatch boundary),
257, 512, 1024, 2048 and 4096; explicit C3 (two columns + thermal wind + Psi_SO) at nz = 257 and 1024; C1 (column +
thermal wind, example_timestepping.py's K = 1) at nz = 257.  Profiles are those of the configs regridded to nz
uniform levels, dt scaled by (dz_new / dz_old)^2 and K = two model years of steps, as the scripts set it.  M is
the smallest power of two whose state (buoyancy of every column) is at least 256 MB, twice the 126 MB L2.

Each shape is warmed up (one diagnosis and a step window), then timed with CUDA events:
  * a window of steps that contains no diagnosis (it0 = 1): the step kernel alone;
  * pmoc_model_diagnose: one diagnosis of every member;
  * the rate over one whole K cycle, K step-times plus one diagnosis.  With K = 1 that cycle is timed directly.
It prints one JSON line per shape with member-steps/s, algorithmic FLOP/s (bench.algorithmic_flops) and their
fraction of the FP64 peak pmoc_fp64_peak measures, and a header line with the GPU's name, power limit and clock.
"""
import argparse
import ctypes
import dataclasses
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402
from pymoc_b200 import _lib, configs  # noqa: E402
from pymoc_b200.ensemble import Ensemble  # noqa: E402

STATE_BYTES = 256 << 20
DAY = 86400.


def regrid(spec, nz):
  """``spec`` on nz uniform levels: z-profiles interpolated, dt scaled by (dz_new / dz_old)^2 (never up), K = two
  model years of the new dt."""
  z0 = spec.z
  z = np.linspace(z0[0], z0[-1], nz)
  on_z = lambda a: np.ascontiguousarray(np.apply_along_axis(lambda r: np.interp(z, z0, r), -1, a))
  col = lambda c: None if c is None else dataclasses.replace(c, kappa=on_z(c.kappa), Area=on_z(c.Area), b0=on_z(c.b0))
  tw = spec.tw if spec.tw is None or spec.tw.b2 is None else dataclasses.replace(spec.tw, b2=on_z(spec.tw.b2))
  dt = spec.dt * min(1., ((z[1] - z[0]) / (z0[1] - z0[0]))**2)
  return dataclasses.replace(spec, z=z, dt=dt, K=max(1, int(np.floor(2. * 360 * DAY / dt))), basin=col(spec.basin),
                             north=col(spec.north), tw=tw)


def members(nz, ncol):
  return 1 << int(np.ceil(np.log2(STATE_BYTES / (8. * nz * ncol))))


def shapes():
  for nz in (256, 257, 512, 1024, 2048, 4096):
    yield 'C2', nz, lambda M, nz=nz: configs.c2_column_so(M, nz=nz, dt_days=10. * (199. / (nz - 1))**2)
  for nz in (257, 1024):
    yield 'C3', nz, lambda M, nz=nz: regrid(configs.c3_twocol_so(M), nz)
  yield 'C1', 257, lambda M: dataclasses.replace(regrid(configs.c1_timestepping(M), 257), K=1)  # the script's K


def card():
  q = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip()
  return {'gpu': torch.cuda.get_device_name(0), 'nvidia_smi': q}


def timed(fn, reps=3):
  """Best of ``reps`` CUDA-event timings of ``fn`` (seconds)."""
  best = float('inf')
  for _ in range(reps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    best = min(best, a.elapsed_time(b) * 1e-3)
  return best


def one(name, nz, make, peak):
  probe = make(2)
  ncol = 2 if probe.north is not None else 1
  M = members(nz, ncol)
  spec = make(M)
  K = spec.K
  ens = Ensemble(spec)
  ens.diagnose()
  flops = bench.algorithmic_flops(spec)
  out = dict(workload=name, nz=nz, M=M, K=K, dt_days=spec.dt / DAY, state_MB=M * nz * ncol * 8 / 2**20,
             flops_per_member_step=flops)
  if K == 1:
    ens.it = 1
    ens.run(4)  # warm-up
    n = max(4, int(2e9 / (M * nz)))
    t = timed(lambda: ens.run(n, sync=False))
    out.update(window_steps=n, window_s=t, cycle_s=t / n)
    rate = M * n / t
  else:
    n = max(2, min(K - 1, int(2e9 / (M * nz))))
    ens.it = 1
    ens.run(min(2, n), sync=True)  # warm-up of the step kernel

    def window():
      ens.it = 1  # [1, n] holds no iteration with it % K == 0
      ens.run(n, sync=False)

    t_step = timed(window) / n
    t_diag = timed(lambda: _diagnose(ens))
    out.update(window_steps=n, step_s=t_step, diagnose_s=t_diag, cycle_s=K * t_step + t_diag,
               step_only_member_steps_per_s=M / t_step)
    rate = M * K / (K * t_step + t_diag)
  out.update(member_steps_per_s=rate, flop_per_s=rate * flops, fraction_of_fp64_peak=rate * flops / peak)
  return out


def _diagnose(ens):
  from pymoc_b200 import _abi
  _abi.check(ens.lib, ens.lib.pmoc_model_diagnose(ctypes.byref(ens.model), ens.be.stream()))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--out', default=None, help='also append the JSON lines to this file')
  ap.add_argument('--only', default=None, help='comma list of workload:nz to run (default: all)')
  args = ap.parse_args()
  lib = _lib.lib()
  peak, mhz = ctypes.c_double(), ctypes.c_double()
  _lib.check(lib.pmoc_fp64_peak(ctypes.byref(peak), ctypes.byref(mhz), None))
  lines = [dict(card(), fp64_peak_flop_per_s=peak.value * 1e12, fp64_peak_clock_mhz=mhz.value)]
  print(json.dumps(lines[0]), flush=True)
  only = set(args.only.split(',')) if args.only else None
  for name, nz, make in shapes():
    if only and '%s:%d' % (name, nz) not in only:
      continue
    r = one(name, nz, make, peak.value * 1e12)  # pmoc_fp64_peak reports TFLOP/s
    lines.append(r)
    print(json.dumps(r), flush=True)
  if args.out:
    with open(args.out, 'a') as f:
      for r in lines:
        f.write(json.dumps(r) + '\n')


if __name__ == '__main__':
  main()
