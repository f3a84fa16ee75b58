"""The e2e control step of bench.py with the reference window uploaded every step against the reference table bound once and
the window selected by row (BatchedAcadosOcpSolver.set_ref_table + set_yref_row), in the same process, alternating.

  force / jerk: SolverFleet of 4 sub-fleets, pinned host buffers, the bench's seeded instances (bench.workload ->
                sharding.instance_inputs), `step` (set_yref_all of a pinned host window + step_into per sub-fleet) against
                `step_at` (set_yref_row + step_into).
  att:          one solver, device buffers, the step of attitude_model.follow_trajectory_batched: the window gathered on the
                device + set_yref_all + step_device, against set_yref_row + step_device.

Each leg: W warm-up steps, then K timed steps, host clock around work that ends in a synchronise; every leg starts from a
reset solver and the same states, so the final plant states of the two legs must be identical.  The GPU name and power limit
are read in the same run.
usage: python tools/e2e_ref_table.py --out RESULT.json [--warmup 10] [--steps 50] [--repeats 3] [--legs force,jerk,att]"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np
import torch

import bench
import drone_attitude_control_b200 as pkg


def device_record(index):
    rec = {'torch_name': torch.cuda.get_device_name(index)}
    try:
        q = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, pl, clk = [v.strip() for v in q.split(',')]
        rec.update(name=name, power_limit=pl, max_sm_clock=clk)
    except Exception as e:      # noqa: BLE001
        rec['nvidia_smi_error'] = repr(e)
    return rec


def fleet_leg(model, B, W, K, groups=4):
    N = 30
    inp = bench.workload(0, B, W + K, max(500 + N, W + K + N + 1), N)
    ref = inp['ref'].permute(2, 0, 1).contiguous()                      # [B, rows, 8] instance-major, as bench.py's e2e leg
    fleet = pkg.SolverFleet(model, batch=B, groups=groups, device=0)
    nx, nu, ny = fleet.nx, fleet.nu, fleet.ny
    per = N * ny + nx
    yh = [torch.cat([ref[:, i:i + N, :ny].reshape(B, N * ny), ref[:, i + N, :nx]], 1).contiguous().pin_memory() for i in range(W + K)]
    noise = inp['noise'][:W + K].contiguous().pin_memory()
    pin = lambda *sh, dt=torch.float64: torch.zeros(sh, dtype=dt).pin_memory()
    xb, u0, up, st = [pin(B, nx), pin(B, nx)], pin(B, nu), pin(B, 2), pin(B, dt=torch.int32)
    fleet.set_ref_table(ref)

    def run(table):
        fleet.reset()
        xb[0].zero_()
        xb[0][:, :4] = inp['x0'].t()
        if nx == 6:
            xb[0][:, 5] = 9.81
        bad = [0]

        def on_results(g, lo, hi):
            bad[0] += int((st[lo:hi] != 0).sum())

        def step(i, hook):
            if table:
                fleet.step_at(i, xb[i % 2], noise[i], u0, up, st, xb[(i + 1) % 2], on_results=hook)
            else:
                fleet.step(yh[i], xb[i % 2], noise[i], u0, up, st, xb[(i + 1) % 2], on_results=hook)
        for i in range(W):
            step(i, None)
        fleet.synchronize()
        t0 = time.perf_counter()
        for i in range(W, W + K):
            step(i, on_results)
        fleet.synchronize(on_results=on_results)
        dt = time.perf_counter() - t0
        return dt, xb[(W + K) % 2].clone(), bad[0]

    return run, {'model': model, 'drones': B, 'groups': groups, 'api': 'SolverFleet, pinned host buffers',
                 'h2d_bytes_per_step': {'upload': B * (per + nx + 1) * 8, 'table': B * (nx + 1) * 8},
                 'table_bytes_bound_once': int(ref.numel() * 8)}


def att_leg(B, W, K):
    from drone_attitude_control_b200.attitude_model import helix_table
    from drone_attitude_control_b200.sharding import instance_inputs
    dev = torch.device('cuda', 0)
    N, NX, NU = 30, 10, 4
    ny = NX + NU
    inp = instance_inputs(0, B, 0, seed=bench.SEED, mass_sigma=0.05, with_noise=False)
    c3 = torch.stack([inp['center'][:, 0], torch.zeros(B, dtype=torch.float64), inp['center'][:, 1]], 1)
    rows = W + K + N + 1
    ref = helix_table(inp['radius'] * 0.9, c3, inp['phase'], 0.2 * inp['radius'], rows, device=dev)      # as bench.py's att leg
    x0 = ref[:, 0, :NX].clone()
    x0[:, :4] += inp['dx0'].to(dev).T
    pp = torch.stack([0.03277 * inp['mass_scale'], torch.full((B,), 9.81, dtype=torch.float64)], 1).to(dev)
    s = pkg.BatchedAcadosOcpSolver('att', batch=B, device=0, numpy_io=False)
    s.set_ref_table(ref)
    xg = torch.zeros((B, NX), dtype=torch.float64, device=dev); xg[:, 6] = 1.0
    ug = torch.zeros((B, NU), dtype=torch.float64, device=dev); ug[:, 0] = 0.03277 * 9.81
    xs = [torch.empty_like(x0), torch.empty_like(x0)]
    u0 = torch.empty((B, NU), dtype=torch.float64, device=dev); up = torch.empty((B, 2), dtype=torch.float64, device=dev)
    st = torch.empty(B, dtype=torch.int32, device=dev)

    def run(table):
        s.reset()
        for k in range(N + 1):
            s.set(k, 'x', xg)
        for k in range(N):
            s.set(k, 'u', ug)
        xs[0].copy_(x0)

        def step(i):
            if table:
                s.set_yref_row(i)
            else:                                                       # follow_trajectory_batched's OCP.set_up_ocp
                s.set_yref_all(torch.cat((ref[:, i:i + N, :].reshape(B, N * ny), ref[:, i + N, :NX]), 1).contiguous())
            s.step_device(xs[i % 2], None, u0, up, st, xs[(i + 1) % 2], pp)
        for i in range(W):
            step(i)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for i in range(W, W + K):
            step(i)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dt, xs[(W + K) % 2].clone(), int((st != 0).sum())

    return run, {'model': 'att', 'drones': B, 'api': 'one solver, device buffers, step_device (bnmpc_step_for_x0)',
                 'h2d_bytes_per_step': {'upload': 0, 'table': 0},
                 'device_gather_bytes_per_step': {'upload': 2 * B * (N * ny + NX) * 8, 'table': 0},
                 'table_bytes_bound_once': int(ref.numel() * 8)}


def measure(name, run, meta, B, K, repeats):
    times = {'upload': [], 'table': []}
    x_ref, dx, bad = None, 0.0, {}
    for r in range(repeats):
        for leg in ('upload', 'table'):
            dt, x, nbad = run(leg == 'table')
            times[leg].append(dt)
            bad[leg] = nbad
            if x_ref is None:
                x_ref = x
            dx = max(dx, float((x - x_ref).abs().max()))
    out = dict(meta)
    for leg, ts in times.items():
        ms = [t / K * 1e3 for t in ts]
        out[leg] = {'ms_per_step': ms, 'ms_per_step_median': float(np.median(ms)),
                    'M_solves_per_s': [B * K / t * 1e-6 for t in ts],
                    'spread_pct': float((max(ms) - min(ms)) / np.median(ms) * 100),
                    'nonzero_status_last_step': bad[leg]}
    out['table_vs_upload_ms_per_step_pct'] = float((out['table']['ms_per_step_median'] / out['upload']['ms_per_step_median'] - 1) * 100)
    out['max_abs_state_difference'] = dx
    print(name, json.dumps({k: v for k, v in out.items() if k in ('upload', 'table', 'table_vs_upload_ms_per_step_pct', 'max_abs_state_difference')}), flush=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', required=True, help='where to write the JSON result')
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--repeats', type=int, default=3)
    ap.add_argument('--legs', default='force,jerk,att')
    a = ap.parse_args()
    assert torch.cuda.is_available(), 'this measurement needs the GPU'
    torch.cuda.set_device(0)
    res = {'device': device_record(0), 'warmup': a.warmup, 'steps': a.steps, 'repeats': a.repeats,
           'timing': 'host perf_counter around the K timed steps, ending in a synchronise; legs alternate upload / table in one process',
           'legs': {}}
    W, K, R = a.warmup, a.steps, a.repeats
    legs = a.legs.split(',')
    if 'force' in legs:
        run, meta = fleet_leg('force', 4096, W, K)
        res['legs']['force'] = measure('force', run, meta, 4096, K, R)
    if 'jerk' in legs:
        run, meta = fleet_leg('jerk', 16384, W, K)
        res['legs']['jerk'] = measure('jerk', run, meta, 16384, K, R)
    if 'att' in legs:
        run, meta = att_leg(4736, W, K)
        res['legs']['att'] = measure('att', run, meta, 4736, K, R)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, 'w') as f:
        json.dump(res, f, indent=1)
    print('wrote', a.out)


if __name__ == '__main__':
    main()
