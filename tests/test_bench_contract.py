"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '4', '--warmup', '3',
                          '--cpu-instances', '64'], capture_output=True, text=True, check=True, cwd=ROOT).stdout
    lines = [l for l in out.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'nmpc_solves_per_sec' and d['unit'] == 'solves/s'
    assert d['higher_is_better'] is True and d['n_gpus'] == 1 and d['steps'] == 4 and d['warmup'] == 3
    assert d['value'] > 0 and d['e2e']['value'] == d['value'] and d['e2e']['h2d_bytes_per_step'] == 0
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and 'sample' in cb
    assert d['config']['controller'] == 'force' and d['config']['horizon'] == 30 and d['vs_baseline'] is None
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_flop_and_byte_model_matches_design():
    sys.path.insert(0, ROOT)
    import bench
    # per IPM iteration (DESIGN.md 3.3): 13.6 kflop force, 27.4 kflop jerk (block-structured count)
    f_it_force = bench.flops_per_solve(2, 2, 1, 30, 4, 1.0, 0.0)
    f_it_jerk = bench.flops_per_solve(2, 3, 1, 30, 1, 1.0, 0.0)
    assert abs(f_it_force - 13620) < 1 and abs(f_it_jerk - 27440) < 1
    assert bench.bytes_per_solve(4, 2, 30) == 1616 and bench.bytes_per_solve(6, 2, 30) == 2128


import numpy as np
import pytest
import torch

DUMP_NAMES = {'drone', 'Xsim', 'U_ctrl', 'U_plant', 'a', 'status', 'qp_iter', 'cost', 'aed', 'failures'}


def test_dump_outputs_writes_the_last_step_and_samples_above_the_limit(tmp_path, monkeypatch):
    sys.path.insert(0, ROOT)
    import bench
    B, S = 10, 5
    g = torch.Generator().manual_seed(0)
    res = dict(Xsim=torch.rand(B, S + 1, 4, generator=g, dtype=torch.float64), U_ctrl=torch.rand(B, S, 2, generator=g, dtype=torch.float64),
               U_plant=torch.rand(B, S, 2, generator=g, dtype=torch.float64), a=torch.rand(B, S, 2, generator=g, dtype=torch.float64),
               status=torch.randint(0, 3, (B, S), generator=g, dtype=torch.int32), qp_iter=torch.randint(0, 20, (B, S), generator=g, dtype=torch.int32),
               cost=torch.rand(B, generator=g, dtype=torch.float64), aed=torch.rand(B, generator=g, dtype=torch.float64),
               failures=torch.randint(0, 3, (B,), generator=g, dtype=torch.int32))
    want = dict(Xsim=res['Xsim'][:, S], U_ctrl=res['U_ctrl'][:, S - 1], U_plant=res['U_plant'][:, S - 1], a=res['a'][:, S - 1],
                status=res['status'][:, S - 1], qp_iter=res['qp_iter'][:, S - 1], cost=res['cost'], aed=res['aed'], failures=res['failures'])

    def dump(name):
        bench.dump_outputs(str(tmp_path / name), res, S - 1, 0, 1)
        got = {f[:-4]: np.load(tmp_path / name / f) for f in os.listdir(tmp_path / name)}
        assert set(got) == DUMP_NAMES and all(v.dtype == np.float64 for v in got.values())
        rows = got['drone'].astype(int)
        for k, v in want.items():
            np.testing.assert_array_equal(got[k], v.double().numpy()[rows], err_msg=k)
        return rows

    assert dump('all').tolist() == list(range(B))
    limit = bench.DUMP_HEADER_BYTES * len(DUMP_NAMES) + 8 * 16 * 4 + 100      # 16 float64 per drone: room for 4 drones
    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', limit)
    rows = dump('sample')
    assert len(rows) == 4 and np.all(np.diff(rows) > 0) and np.array_equal(dump('again'), rows)
    assert sum(os.path.getsize(tmp_path / 'sample' / f) for f in os.listdir(tmp_path / 'sample')) <= limit


@pytest.mark.gpu
def test_both_arms_run_the_same_experiment(tmp_path):
    """`bench.py` and `bench.py --impl reference` draw the same instances (sharding.instance_inputs of the same global ids),
    print the same `config`, and do the same work per solve: the mean interior-point iteration count over the timed steps
    is identical, and the bench line carries every key the contract names.  --dump-outputs writes the last timed step."""
    common = ['--batch', '256', '--steps', '6', '--warmup', '3', '--cpu-instances', '256', '--cpu-steps', '6']
    run = lambda extra: json.loads([l for l in subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py')] + common + extra,
                                                              capture_output=True, text=True, check=True, cwd=ROOT).stdout.splitlines()
                                    if l.startswith('{')][-1])
    ours = run(['--skip-extra', '--e2e-steps', '4', '--dump-outputs', str(tmp_path)])
    ref = run(['--impl', 'reference'])
    dumped = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(dumped) == DUMP_NAMES and all(v.dtype == np.float64 and v.shape[0] == 256 for v in dumped.values())
    assert dumped['Xsim'].shape == (256, 4) and np.isfinite(dumped['Xsim']).all() and (dumped['status'] == 0).all()
    assert ours['config'] == ref['config'] and ours['metric'] == ref['metric'] and ours['unit'] == ref['unit']
    assert ours['qp_iter_mean'] == pytest.approx(ref['qp_iter_mean'], abs=1e-12)
    assert ours['cpu_baseline']['qp_iter_mean'] == pytest.approx(ours['qp_iter_mean'], abs=1e-12)
    assert ours['nonzero_status'] == ref['nonzero_status'] == 0
    for k in ('value', 'ms_per_step', 'n_gpus', 'steps', 'warmup', 'higher_is_better', 'scaling', 'dtype', 'data', 'clocks', 'e2e',
              'gpu_launches', 'roofline', 'cpu_baseline', 'per_step_launch', 'p50_step_latency_ms'):
        assert k in ours, k
    assert ours['gpu_launches'] >= 1 and ours['e2e']['h2d_bytes_per_step'] > 0 and ours['e2e']['value'] > 0
    assert ours['roofline']['frac'] > 0 and ours['cpu_baseline']['kind'] == 'port'
