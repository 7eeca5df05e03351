#!/usr/bin/env python
"""Benchmark of the PyMOC time-stepping hot path (BASELINE.json metric: member-timesteps/sec, fp64).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload C2] [--impl reference] [--dump-outputs DIR]

One bench "step" = one fused-kernel pass advancing every member of the ensemble by
``--nt`` model time steps (default: the workload's N from SURVEY.md section 8d).  Under
torchrun every rank holds ``--members`` members (weak scaling) and steps them with no
collective; a final NCCL all-gather of one diagnostic per member runs outside the timed
region.  Prints ONE JSON line (rank 0).

The headline workload is BASELINE.json ``configs[1]`` (C2: 65,536 members of column + Psi_SO, nz = 200).  The same
run also times the other BASELINE configurations -- C3 (``configs[2]``, explicit GM), C3_bvp (the literal
example_twocol_plusSO.py with its F2010 smoother: the north-star model), C4, C5 at nz = 4096 and C1 -- with CUDA
events and reports them under ``workloads`` (``--extras none`` skips them).

Keys beyond the base contract:
  roofline      FP64-pipe roofline of the fused kernel: algorithmic flops per member-step (SURVEY.md section 8d,
                restated in DESIGN.md) x member-steps/s, against the DFMA peak measured live by pmoc_fp64_peak on the
                same GPU (``peak_clock_mhz``: the SM clock that peak implies).  ``fp64_pipe_pct`` and
                ``executed_flops_per_member_step`` are what Nsight Compute measured for the same kernel (profiles/):
                the algorithmic count charges the reference's O(nb nz) remap and 11-flop stencil, the kernel executes
                an O(nb + nz) remap and a 5-flop stencil, so ``frac`` is an ALGORITHMIC fraction, not pipe utilisation.
  status_counts members per PMOC_ST_* status bit after the timed launches (include/pymoc_b200.h): how many members
                sit where the reference's own answer is decided by rounding noise (``parity_undefined``).
  cpu_baseline  the oracle's reference-faithful loop (NumPy/SciPy, oracle/pymoc_oracle.py) timed on the host cores
                of this box on a bounded sample of the same workload.
  e2e           the same metric through the host-buffer C-ABI handle (pmoc_host_open once; every step
                pmoc_host_step pushes the state from pinned HOST buffers, runs the fused kernel, pulls state +
                carried streamfunctions back).  ``stateless``: through pmoc_model_run_host, which also re-uploads
                every parameter array each call (round 1's e2e).  ``cadence120``: the handle called every 120 model
                steps, the diagnostic cadence of run_JansenNadeau_2018.py:218-226.

``--dump-outputs DIR`` writes what the headline workload's timed launches computed (see dump_outputs), so that two
builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pymoc_b200 import configs  # noqa: E402

WORKLOADS = {
    # name: (builder(M) -> spec, default members per GPU, default model steps per bench step)
    'C1': (lambda M: configs.c1_timestepping(M), 65536, 3000),
    'C2': (lambda M: configs.c2_column_so(M), 65536, 7200),
    'twocol': (lambda M: configs.twocol(M), 32768, 2400),
    'C3': (lambda M: configs.c3_twocol_so(M), 32768, 2400),
    # the literal script: F2010 smoother of Psi_GM (c = 0.1, bvp_with_Ek), parity at the stated 1e-5
    'C3_bvp': (lambda M: configs.c3_twocol_so(M, c=0.1), 32768, 2400),
    'twobasin': (lambda M: configs.twobasin(M), 32768, 2400),
    'C4': (lambda M: configs.c4_jansen_nadeau(M), 32768, 2400),
    'C5': (lambda M: configs.c5_single_global_basin(M), 32768, 2400),
    # BASELINE configs[4]: nz=4096 (block-per-member kernels), stable dt = 0.01 d, K = 72 000
    'C5_4096': (lambda M: configs.c5_single_global_basin(M, nz=4096, dt_days=0.01, kapfac_max=1.), 16384, 720),
}
# workloads timed next to the headline one (same process, CUDA events): name -> members per GPU in that role
EXTRAS = {'C3': 32768, 'C3_bvp': 32768, 'C4': 32768, 'C5_4096': 2048, 'C1': 65536}
E2E_EXTRAS = ('C3_bvp',)  # the north-star model also gets an end-to-end figure


def algorithmic_flops(spec):
  """FP64 flops per member-timestep, SURVEY.md section 8d (add/sub/mul/div/cmp = 1, FMA = 2)."""
  n, K, B = spec.nz, spec.K, spec.nb
  per_step = 11 * n + (2 * n if spec.basin.do_conv else 0)
  ncol = 1
  if spec.north is not None:
    per_step += 11 * n + (2 * n if spec.north.do_conv else 0)
    ncol = 2
  nclos = 1
  if getattr(spec, 'pac', None) is not None:  # third column, second thermal wind + remap, second Psi_SO
    per_step += 11 * n + (2 * n if spec.pac.do_conv else 0)
    ncol, nclos = 3, 2
  refresh = 3 * n * ncol
  if spec.tw is not None:
    refresh += nclos * 16 * n
    if spec.iso:
      refresh += nclos * (6 * B * (n - 1) + 8 * n + 2 * B + 2 * n * (math.ceil(math.log2(B)) + 5))
  if spec.so is not None:
    refresh += nclos * n * (math.ceil(math.log2(spec.so.y.size)) + 20)
    if spec.so.c is not None:
      refresh += 120 * n  # F2010 smoother (SURVEY.md section 8d: approximate)
  if spec.ml is not None:
    m = spec.ml.y.size
    per_step += m * (math.ceil(math.log2(n)) + 32) + n
  return per_step + refresh / K


# What Nsight Compute measured for each workload's fused kernel (`ncu --set full`, one launch; profiles/):
#   pipe: sm__pipe_fp64_cycles_active.avg.pct_of_peak_sustained_active
#   flops: executed FP64 flops per member-step = (dadd + dmul + 2 dfma thread instructions) / member-steps of the launch
#   dram: dram__bytes_read.sum + dram__bytes_write.sum per member of the launch (state and parameters are read once
#         and state + diagnostics written once per launch, whatever the number of steps)
NCU_FACTS = {  # round 2, profiles/r2_full_summary.txt (captures of the final kernels)
    'C1': dict(pipe=51.7, flops=2029., dram=(147.67e6 + 27.82e6) / 65536, source='profiles/r2_full_summary.txt'),
    'C2': dict(pipe=61.1, flops=1301., dram=(421.07e6 + 363.62e6) / 65536, source='profiles/r2_full_summary.txt'),
    'C3': dict(pipe=25.2, flops=2106., dram=(233.15e6 + 389.19e6) / 32768, source='profiles/r2_full_summary.txt'),
    'C3_bvp': dict(pipe=31.0, flops=4364., dram=(236.44e6 + 654.39e6) / 32768, source='profiles/r2_full_summary.txt'),
    'C4': dict(pipe=20.6, flops=10121., dram=(256.84e6 + 414.28e6) / 32768, source='profiles/r2_full_summary.txt'),
    # (block-per-member step kernel; its launches also read the per-member coefficient scratch)
    'C5_4096': dict(pipe=23.7, flops=187792., dram=(870.51e6 + 603.98e6) / 2048, source='profiles/r2_full_summary.txt'),
}


def dump_outputs(ens, out_dir, budget=60e6, seed=0):
  """Write the arrays a caller of the timed path receives after its last launch -- ``ens.state()`` and
  ``ens.diagnostics()`` -- as ``out_dir/<name>.npy`` in float64, for a fixed seeded sample of members sized so that
  all files together stay under 64 MB (``budget`` leaves room for the .npy headers); ``members.npy`` holds the
  sampled member indices."""
  outs = {**ens.state(), **ens.diagnostics()}
  per_member = 8 * (1 + sum(a.size // a.shape[0] for a in outs.values()))
  n = min(ens.M, int(budget // per_member))
  idx = np.sort(np.random.default_rng(seed).choice(ens.M, size=n, replace=False))
  os.makedirs(out_dir, exist_ok=True)
  np.save(os.path.join(out_dir, 'members.npy'), idx.astype(np.float64))
  for name, a in outs.items():
    np.save(os.path.join(out_dir, name + '.npy'), a[idx].astype(np.float64))


def config_of(workload, spec, m_local, world, nt):
  """The `config` object: a function of the command line and the workload definition only, so that the GPU arm
  and the reference arm print the same one."""
  M = m_local * world
  state_mb = m_local * spec.nz * 8 * 3 / 1e6
  return {'workload': '%s: %s' % (workload, spec.name), 'members_per_gpu': m_local, 'members': M,
          'nz': spec.nz, 'ny': spec.ny, 'K': spec.K, 'dt_days': spec.dt / 86400., 'model_steps_per_bench_step': nt,
          'l2': 'inputs (state + per-member parameters, %.0f MB per GPU) larger than the 126 MB L2' % state_mb,
          'parallelism': 'ensemble members sharded over %d GPU(s), no collective in the loop' % world}


# ---------------------------------------------------------------------------- CPU reference
def _cpu_task(args):
  workload, M, member, nsteps = args
  os.environ['OMP_NUM_THREADS'] = '1'
  import warnings
  warnings.filterwarnings('ignore')
  from oracle import pymoc_oracle as O
  with configs.members(member, member + 1):
    spec = WORKLOADS[workload][0](M)
  case = spec.member_case(0)
  t0 = time.perf_counter()
  O.run_coupled(case, nsteps, O.REFERENCE)
  return time.perf_counter() - t0


def cpu_reference(workload, M, nsteps=0, tasks_per_core=2, cores=None, target_s=15.0):
  """Reference-faithful CPU loop (the oracle in its default modes: solve_bvp, brentq, dense inv
  exactly where the reference calls them) on all host cores; returns member-steps/s.  With
  ``nsteps == 0`` the steps per task are sized from a short pilot so that the sample takes about
  ``target_s`` seconds of wall time (a bounded sample of the same workload)."""
  import multiprocessing as mp
  cores = cores or os.cpu_count() or 1
  ntask = cores * tasks_per_core
  members = [int(i * (M - 1) / max(ntask - 1, 1)) for i in range(ntask)]
  with configs.members(0, 1):
    K = WORKLOADS[workload][0](M).K
  ctx = mp.get_context('spawn')
  with ctx.Pool(cores) as pool:
    pilot_steps = 2 * K + 1
    t_pilot = max(pool.map(_cpu_task, [(workload, M, m, pilot_steps) for m in members[:cores]]))  # import + warm-up
    if nsteps <= 0:
      per_step = t_pilot / pilot_steps
      nsteps = int(max(pilot_steps, min(200000, target_s / (per_step * tasks_per_core))))
      nsteps = max(K, (nsteps // K) * K) + 1
    jobs = [(workload, M, m, nsteps) for m in members]
    t0 = time.perf_counter()
    pool.map(_cpu_task, jobs, chunksize=1)
    wall = time.perf_counter() - t0
  return ntask * nsteps / wall, cores, '%d members x %d steps of %s (members spread over the lattice)' % (
      ntask, nsteps, workload), wall


# ------------------------------------------------------------------------------ clocks
class ClockSampler(threading.Thread):
  Q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, index):
    super().__init__(daemon=True)
    self.index, self.rows, self.proc = index, [], None

  def run(self):
    try:
      self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                    '--format=csv,noheader,nounits', '-lms', '100'], stdout=subprocess.PIPE, text=True)
      for line in self.proc.stdout:
        self.rows.append([c.strip() for c in line.split(',')])
    except Exception:
      pass

  def stop(self):
    if self.proc is not None:
      self.proc.terminate()
    self.join(timeout=2)
    sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace('.', '').isdigit()]
    mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace('.', '').isdigit()]
    names = ('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap')
    reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower() == 'active'})
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': reasons, 'samples': len(sm)}


def bind_to_gpu_numa_node(local_rank):
  """Run this rank on the cores of its GPU's NUMA node, so that the pinned host buffers allocated afterwards are
  node-local (first touch).  Best effort: a box without the sysfs entries, or with one node, is left alone."""
  try:
    import torch
    p = torch.cuda.get_device_properties(local_rank)
    bus = '%04x:%02x:%02x.0' % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
  except Exception:
    bus = None
  try:
    if bus is None:
      bus = subprocess.run(['nvidia-smi', '-i', str(local_rank), '--query-gpu=pci.bus_id', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=10).stdout.strip().lower()
      if len(bus.split(':')[0]) == 8:
        bus = bus[4:]
    node = int(open('/sys/bus/pci/devices/%s/numa_node' % bus).read())
    if node < 0:
      return None
    cpus = set()
    for part in open('/sys/devices/system/node/node%d/cpulist' % node).read().strip().split(','):
      lo, _, hi = part.partition('-')
      cpus.update(range(int(lo), int(hi or lo) + 1))
    cpus &= os.sched_getaffinity(0)
    if cpus:
      os.sched_setaffinity(0, cpus)
      return node
  except Exception:
    pass
  return None


# ------------------------------------------------------------------------------ GPU arm
def gpu_arm(args):
  import torch
  import torch.distributed as dist
  from pymoc_b200 import _abi, _lib
  from pymoc_b200.ensemble import Ensemble, HostEnsemble
  from pymoc_b200.parallel import gather_members, shard_range

  rank = int(os.environ.get('RANK', 0))
  world = int(os.environ.get('WORLD_SIZE', 1))
  local = int(os.environ.get('LOCAL_RANK', 0))
  torch.cuda.set_device(local)
  numa_node = bind_to_gpu_numa_node(local)
  if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
    os.environ['NCCL_DEBUG'] = 'WARN'  # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
  if world > 1:
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
  lib = _lib.lib()

  peak = ctypes.c_double()
  mhz = ctypes.c_double()
  _lib.check(lib.pmoc_fp64_peak(ctypes.byref(peak), ctypes.byref(mhz), None))

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def allmax(x):
    t = torch.tensor([x], dtype=torch.float64, device='cuda')
    if world > 1:
      dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())

  def build_rank_spec(workload, m_local):
    M = m_local * world
    lo, hi = shard_range(M, rank, world)
    with configs.members(lo, hi):  # only this rank's block of the M-member lattice is ever built
      return WORKLOADS[workload][0](M), M

  def launches_per_run(spec, nt):
    if spec.nz <= 256:
      return 1
    nref = len([i for i in range(0, nt) if i % spec.K == 0])  # block-per-member kernels: geometry + diagnosis + step launches
    return 1 + nref + max(nref, 1)

  def time_workload(workload, m_local, nt, steps, warmup, sample_clocks=False):
    """`steps` timed launches of `nt` model steps each, CUDA events on the launching stream, max over ranks."""
    spec, M = build_rank_spec(workload, m_local)
    ens = Ensemble(spec)
    for _ in range(warmup):
      ens.run(nt, sync=False)
    barrier()
    sampler = None
    if sample_clocks:
      sampler = ClockSampler(local)
      sampler.start()
      time.sleep(0.3)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(steps):
      ens.run(nt, sync=False)
    e1.record()
    barrier()
    ms = allmax(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    ms_per_step = ms / steps
    value = M * nt / (ms_per_step * 1e-3)
    flops = algorithmic_flops(spec)
    achieved = value / world * flops / 1e12
    census = _abi.status_census(ens.diagnostics()['status'])
    facts = NCU_FACTS.get(workload, {})
    # bytes the launch has to move at least: parameters + state in, state + rewritten diagnostics out
    nbytes = lambda b: b.numel() * b.element_size()
    params = sum(nbytes(b) for b in ens._keep)
    state = sum(nbytes(ens._bufs[k]) for k in ('b_basin', 'b_north', 'b_pac', 'bs_ml') if k in ens._bufs)
    diags = sum(nbytes(b) for k, b in ens._bufs.items() if k.startswith(('Psi', 'psib', 'bgrid')))
    bound_bytes = params + 2 * state + diags
    traffic = facts['dram'] * m_local if facts.get('dram') else None
    out = {
        'value': value, 'unit': 'member-timesteps/s', 'ms_per_step': ms_per_step, 'steps': steps, 'warmup': warmup,
        'config': config_of(workload, spec, m_local, world, nt), 'gpu_launches': steps * launches_per_run(spec, nt),
        'status_counts': census,
        'roofline': {
            'bound': 'fp64',
            'bound_note': 'FP64 pipe (DFMA): the state stays on chip across the fused steps; BASELINE.json asks for '
                          '"% of FP64/HBM roofline", hbm_check shows the HBM side',
            'achieved': achieved, 'peak': peak.value, 'unit': 'TFLOP/s', 'frac': achieved / peak.value,
            'peak_source': 'pmoc_fp64_peak measured live (DFMA stream); MEASURED_PEAKS.json has no FP64 entry',
            'peak_clock_mhz': mhz.value, 'flops_per_member_step': flops,
            'fp64_pipe_pct': facts.get('pipe'), 'executed_flops_per_member_step': facts.get('flops'),
            'ncu_source': facts.get('source'),
            'traffic': traffic, 'traffic_source': 'ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, scaled by members',
            'traffic_bound_buffers': bound_bytes,
            'traffic_note': 'traffic_bound_buffers = parameters + 2 x state + diagnostics of the buffers bound to this launch',
            'hbm_check': {'achieved_GBs': (traffic or bound_bytes) / (ms_per_step * 1e-3) / 1e9, 'peak_GBs': 6540.5,
                          'note': 'MEASURED_PEAKS.json hbm_gbs; state stays on chip, HBM is idle'},
            'kernel_ms': ms_per_step},
    }
    if clocks:
      out['clocks'] = clocks
    return out, spec, ens

  def time_e2e(spec, nt, steps):
    """The same metric through the host-buffer handle: every step pushes the state from pinned host memory,
    runs the fused kernel and pulls state + carried streamfunctions back."""
    S, P = HostEnsemble.IO_STATE, HostEnsemble.IO_PSI
    hens = HostEnsemble(spec)
    hens.run(nt, push=S, pull=S | P)  # warm-up (memory pool, page faults)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
      hens.run(nt, push=S, pull=S | P)
    barrier()
    dt = allmax(time.perf_counter() - t0)
    h2d, d2h = hens.last_bytes()
    M = spec.M * world
    fin = hens.state()['b_basin']
    assert np.isfinite(fin).all(), 'non-finite members in the host-buffer run'
    hens.close()
    return {'value': M * nt * steps / dt, 'unit': 'member-timesteps/s', 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
            'steps': steps, 'model_steps_per_call': nt,
            'api': 'pmoc_host_open once; per step pmoc_host_step(push=STATE, pull=STATE|PSI), pinned host buffers'}

  build, m_default, nt_default = WORKLOADS[args.workload]
  m_local = args.members or m_default
  nt = args.nt or nt_default
  main, spec, ens = time_workload(args.workload, m_local, nt, args.steps, args.warmup, sample_clocks=True)
  M = m_local * world

  # final diagnostic gather (the only collective of the path), untimed
  diag_key = 'Psi_so' if spec.so is not None else 'Psi_tw'
  per_member = ens.buffer(diag_key).abs().amax(dim=1)
  gathered = gather_members(per_member, M)
  assert gathered.shape[0] == M
  # the lattices hold no member that the (explicit, CFL-limited) reference loses
  assert main['status_counts']['nan'] == 0, '%d of %d members non-finite' % (main['status_counts']['nan'], ens.M)
  if args.dump_outputs and rank == 0:  # (rank 0's members)
    dump_outputs(ens, args.dump_outputs)
  del ens

  e2e = None
  if args.e2e_steps > 0:
    e2e = time_e2e(spec, nt, args.e2e_steps)
    # the handle at the diagnostic cadence of the reference's scripts (120 model steps per call)
    if nt > 120:
      cad = time_e2e(spec, 120, max(args.e2e_steps, 5))
      e2e['cadence120'] = {k: cad[k] for k in ('value', 'h2d_bytes_per_step', 'd2h_bytes_per_step', 'steps', 'model_steps_per_call')}
    # round 1's stateless call: every parameter array re-uploaded, streams re-created, per call
    from pymoc_b200.backend import PinnedHostBackend
    sens = Ensemble(spec, backend=PinnedHostBackend())
    _lib.check(lib.pmoc_model_run_host(ctypes.byref(sens.model), 0, nt))
    barrier()
    t0 = time.perf_counter()
    it = nt
    for _ in range(args.e2e_steps):
      _lib.check(lib.pmoc_model_run_host(ctypes.byref(sens.model), it, nt))
      it += nt
    barrier()
    dt = allmax(time.perf_counter() - t0)
    h2d, d2h = ctypes.c_uint64(), ctypes.c_uint64()
    lib.pmoc_host_last_bytes(ctypes.byref(h2d), ctypes.byref(d2h))
    e2e['stateless'] = {'value': M * nt * args.e2e_steps / dt, 'h2d_bytes_per_step': int(h2d.value),
                        'd2h_bytes_per_step': int(d2h.value), 'api': 'pmoc_model_run_host'}
    e2e['numa_node'] = numa_node
    del sens

  workloads = {}
  if args.extras != 'none':
    names = [n for n in (EXTRAS if args.extras == 'all' else args.extras.split(',')) if n != args.workload]
    for name in names:
      w_nt = WORKLOADS[name][2]
      try:  # an extra workload must never cost the headline line
        res, w_spec, w_ens = time_workload(name, EXTRAS.get(name, WORKLOADS[name][1]), w_nt, max(2, min(args.steps, 3)), 1)
        del w_ens
        if name in E2E_EXTRAS and args.e2e_steps > 0:
          res['e2e'] = time_e2e(w_spec, w_nt, 2)
      except Exception as exc:  # noqa: BLE001 (reported in the line; every rank runs the same code)
        res = {'error': '%s: %s' % (type(exc).__name__, exc)}
      workloads[name] = res

  cpu = None
  if rank == 0 and world == 1 and not args.no_cpu:
    try:
      v, cores, sample, wall = cpu_reference(args.workload, min(M, 65536), args.cpu_steps)
      cpu = {'value': v, 'unit': 'member-timesteps/s', 'cores': cores, 'kind': 'port', 'sample': sample,
             'wall_s': round(wall, 2)}
    except Exception as exc:  # noqa: BLE001 (the GPU numbers above are still worth printing)
      cpu = {'value': None, 'unit': 'member-timesteps/s', 'cores': os.cpu_count(), 'kind': 'port',
             'sample': 'failed: %s: %s' % (type(exc).__name__, exc)}

  if rank == 0:
    line = {
        'metric': 'member-timesteps/sec, fp64', 'value': main['value'], 'unit': 'member-timesteps/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': main['ms_per_step'], 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': main['config'], 'roofline': main['roofline'], 'status_counts': main['status_counts'],
        'sweep_rank0': {k: [float(v.min()), float(v.max())] for k, v in spec.sweep.items()},
        'cpu_baseline': cpu, 'e2e': e2e, 'gpu_launches': main['gpu_launches'], 'clocks': main.get('clocks'),
        'workloads': workloads,
    }
    print(json.dumps(line))
  if world > 1:
    dist.destroy_process_group()


def reference_arm(args):
  rank = int(os.environ.get('RANK', 0))
  world = int(os.environ.get('WORLD_SIZE', 1))
  if rank != 0:
    return
  build, m_default, nt_default = WORKLOADS[args.workload]
  m_local = args.members or m_default
  M = m_local * world
  nt = args.nt or nt_default
  with configs.members(0, 1):
    spec = build(M)
  for _ in range(args.warmup):
    cpu_reference(args.workload, M, args.cpu_steps, tasks_per_core=1, target_s=4.0)
  vals = []
  t0 = time.perf_counter()
  for _ in range(args.steps):
    v, cores, sample, wall = cpu_reference(args.workload, M, args.cpu_steps, tasks_per_core=1, target_s=12.0)
    vals.append(v)
  total = time.perf_counter() - t0
  value = float(np.mean(vals))
  line = {
      'impl': 'reference', 'metric': 'member-timesteps/sec, fp64', 'value': value, 'unit': 'member-timesteps/s',
      'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total / args.steps * 1e3,
      'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
      'config': config_of(args.workload, spec, m_local, world, nt),
      'cpu_baseline': {'value': value, 'unit': 'member-timesteps/s', 'cores': cores, 'kind': 'port', 'sample': sample},
      'e2e': {'value': value, 'unit': 'member-timesteps/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
  }
  print(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=10)
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--workload', default='C2', choices=sorted(WORKLOADS))
  ap.add_argument('--members', type=int, default=0, help='members per GPU (default: workload size)')
  ap.add_argument('--nt', type=int, default=0, help='model time steps per bench step')
  ap.add_argument('--e2e-steps', type=int, default=3)
  ap.add_argument('--cpu-steps', type=int, default=0, help='model steps per CPU-baseline task (0: sized for ~15 s)')
  ap.add_argument('--no-cpu', action='store_true')
  ap.add_argument('--extras', default='all', help="'all', 'none' or a comma list: other workloads timed in the same run")
  ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                  help='write the outputs of the last timed launch of the headline workload as DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  args.warmup = max(args.warmup, 3) if args.impl == 'ours' else args.warmup
  if args.impl == 'reference':
    reference_arm(args)
  else:
    gpu_arm(args)


if __name__ == '__main__':
  main()
