"""Cost of the solution sensitivities against the solve, on the same instances (CUDA events).

For each case (force model with 4096 drones, jerk model with 16384 drones, FP64, reference horizon N = 30) it times, per
call: the solve (solve_for_x0_device), bnmpc_eval_sens_x0 with stages = 1 (the feedback gain of u0) and with stages = N + 1,
and the adjoint with a seed on u0 only.  Each timed solve starts from the solution of the previous one at another x0 (the
x0 sets alternate), so that it is a real re-solve, as in a closed loop; its mean QP iterations are recorded.  The
sensitivities are evaluated at the stored solution, which they leave as it is.  10 warm-up and 50 timed calls, three
repeats; the card's name and power limit are read in the same run.

    python tools/sens_bench.py [--out profiles/sens_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'tests'))

from common import random_solve_inputs  # noqa: E402
from drone_attitude_control_b200 import BatchedAcadosOcpSolver  # noqa: E402

WARMUP, TIMED, REPEATS = 10, 50, 3


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                       capture_output=True, text=True)
    name, power, clock = [v.strip() for v in q.stdout.strip().split(',')]
    return dict(name=name, power_limit=power, max_sm_clock=clock)


def timed(fn, stream):
    """mean ms per call of fn() over TIMED calls after WARMUP, REPEATS times"""
    out = []
    for _ in range(REPEATS):
        for _ in range(WARMUP):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(TIMED):
            fn()
        e1.record(stream)
        e1.synchronize()
        out.append(e0.elapsed_time(e1) / TIMED)
    return out


def case(model, B):
    sv = BatchedAcadosOcpSolver(model, batch=B, numpy_io=False)
    N, dev, st = sv.N, sv.device, sv._stream
    x0, yref = random_solve_inputs(model, B, seed=5)
    xa = torch.tensor(x0, device=dev)
    xb = xa + torch.tensor(np.random.default_rng(6).uniform(-0.02, 0.02, x0.shape), device=dev)
    sv.set_yref_all(torch.tensor(yref, device=dev))
    u0 = torch.empty((B, sv.nu), dtype=torch.float64, device=dev)
    status = torch.empty(B, dtype=torch.int32, device=dev)
    flip = [0]
    qp_iters = []

    def solve():
        flip[0] ^= 1
        sv.solve_for_x0_device(xa if flip[0] else xb, u0, status)

    res = dict(model=model, batch=B, horizon=N, precision='fp64', warmup=WARMUP, timed=TIMED, repeats=REPEATS)
    res['solve_ms'] = timed(solve, st)
    for _ in range(4):
        solve()
        qp_iters.append(float(sv.get_stats('qp_iter').double().mean()))
    res['solve_mean_qp_iter'] = float(np.mean(qp_iters))
    res['solve_status_nonzero'] = int((status != 0).sum())
    sx1, su1 = (torch.empty((B, 1, sv.nx, sv.nx), dtype=torch.float64, device=dev),
                torch.empty((B, 1, sv.nu, sv.nx), dtype=torch.float64, device=dev))
    sxN, suN = (torch.empty((B, N + 1, sv.nx, sv.nx), dtype=torch.float64, device=dev),
                torch.empty((B, N, sv.nu, sv.nx), dtype=torch.float64, device=dev))
    seed_u = torch.zeros((B, N, sv.nu), dtype=torch.float64, device=dev)
    seed_u[:, 0] = 1.0
    gx = torch.empty((B, sv.nx), dtype=torch.float64, device=dev)
    gy = torch.empty((B, N * sv.ny + sv.ny_e), dtype=torch.float64, device=dev)
    from drone_attitude_control_b200._lib import check, lib
    import ctypes as C
    p = lambda t: C.c_void_p(t.data_ptr())
    res['sens_x0_stages1_ms'] = timed(lambda: check(lib().bnmpc_eval_sens_x0(sv.handle, 1, p(sx1), p(su1), 1)), st)
    res['sens_x0_stagesN1_ms'] = timed(lambda: check(lib().bnmpc_eval_sens_x0(sv.handle, N + 1, p(sxN), p(suN), 1)), st)
    res['adjoint_seed_u0_ms'] = timed(lambda: check(lib().bnmpc_eval_adjoint_sens(sv.handle, None, p(seed_u), p(gx), p(gy), 1)), st)
    torch.cuda.synchronize()
    res['sens_nan_rows'] = int(torch.isnan(su1).any(-1).any(-1).any(-1).sum())
    for k in ('sens_x0_stages1_ms', 'sens_x0_stagesN1_ms', 'adjoint_seed_u0_ms'):
        res[k.replace('_ms', '_over_solve')] = float(np.median(res[k]) / np.median(res['solve_ms']))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    out = dict(card=card(), cases=[case('force', 4096), case('jerk', 16384)])
    txt = json.dumps(out, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(txt + '\n')


if __name__ == '__main__':
    main()
