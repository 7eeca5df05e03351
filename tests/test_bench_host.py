"""Host-side pieces of bench.py (no GPU): the algorithmic flop counts behind roofline.achieved, the CLI
contract of the reference arm."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_algorithmic_flops_match_survey_table():
  """SURVEY.md section 8d: C1 2 100, C2 2 280, C3 ~12 500 (with the BVP smoother's ~120n/K; the explicit twin
  is 12 100), C4 ~26 900 (of which 2 014 for the diagnostics-only Psib every Diag_iters, not counted here),
  C5 (nz = 4096) ~113 000 flops per member-step."""
  import bench
  from pymoc_b200 import configs
  want = {'C1': (configs.c1_timestepping(1), 2100), 'C2': (configs.c2_column_so(16, ntau=4), 2280),
          'C3': (configs.c3_twocol_so(1), 12100), 'C4': (configs.c4_jansen_nadeau(1), 26900 - 2014),
          'C5': (configs.c5_single_global_basin(1, nz=4096, dt_days=0.01), 113000)}
  for name, (spec, flops) in want.items():
    got = bench.algorithmic_flops(spec)
    assert abs(got - flops) / flops < 0.03, (name, got, flops)


def test_reference_arm_prints_one_json_line():
  """`bench.py --impl reference` (the oracle port on the host cores) needs no GPU: one JSON line with the keys
  the contract names."""
  env = dict(os.environ, PYTHONPATH=ROOT)
  out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0',
                        '--cpu-steps', '73', '--members', '64'], capture_output=True, text=True, env=env, timeout=600)
  assert out.returncode == 0, out.stderr[-2000:]
  lines = [l for l in out.stdout.splitlines() if l.strip()]
  assert len(lines) == 1
  d = json.loads(lines[0])
  assert d['impl'] == 'reference' and d['unit'] == 'member-timesteps/s' and d['value'] > 0
  assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
  assert d['e2e']['h2d_bytes_per_step'] == 0 and d['e2e']['d2h_bytes_per_step'] == 0


def test_dump_outputs_writes_a_fixed_sample_of_every_output(tmp_path):
  """--dump-outputs: every array of state() and diagnostics() as float64 .npy, for the same seeded member sample
  on every call, within the byte budget (the kernel sources run on the warp emulator)."""
  import numpy as np

  import bench
  from emu.emu_backend import EmuBackend
  from pymoc_b200 import configs
  from pymoc_b200.ensemble import Ensemble
  ens = Ensemble(configs.c3_twocol_so(64, axes=(4, 4, 2, 2)), backend=EmuBackend())
  ens.run(5)
  outs = {**ens.state(), **ens.diagnostics()}
  per_member = 8 * (1 + sum(a.size // a.shape[0] for a in outs.values()))
  for run in ('a', 'b'):
    bench.dump_outputs(ens, str(tmp_path / run), budget=20 * per_member)
  files = sorted(p.name for p in (tmp_path / 'a').iterdir())
  assert files == sorted(['members.npy'] + [k + '.npy' for k in outs])
  idx = np.load(tmp_path / 'a' / 'members.npy').astype(int)
  assert idx.size == 20 and len(set(idx)) == 20 and np.array_equal(idx, np.sort(idx))
  assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 20 * per_member + 128 * len(files)
  for name, a in outs.items():
    got = np.load(tmp_path / 'a' / (name + '.npy'))
    assert got.dtype == np.float64 and np.array_equal(got, a[idx].astype(np.float64)), name
    assert np.array_equal(got, np.load(tmp_path / 'b' / (name + '.npy'))), name
  bench.dump_outputs(ens, str(tmp_path / 'all'))  # a small ensemble fits the budget whole
  assert np.array_equal(np.load(tmp_path / 'all' / 'members.npy'), np.arange(64))


def test_both_arms_print_the_same_config_and_facts_are_consistent():
  """`config` is a function of the command line and the workload definition only (the driver compares the two arms'),
  and every ncu fact / extra workload names a workload that exists."""
  import bench
  from pymoc_b200 import configs
  with configs.members(0, 1):
    spec_a = bench.WORKLOADS['C3'][0](262144)
  with configs.members(1000, 1001):
    spec_b = bench.WORKLOADS['C3'][0](262144)
  assert bench.config_of('C3', spec_a, 32768, 8, 2400) == bench.config_of('C3', spec_b, 32768, 8, 2400)
  assert set(bench.NCU_FACTS) <= set(bench.WORKLOADS) and set(bench.EXTRAS) <= set(bench.WORKLOADS)
  assert set(bench.E2E_EXTRAS) <= set(bench.EXTRAS)
