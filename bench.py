#!/usr/bin/env python3
"""bench.py - NMPC solves/s of the fused closed-loop step (BASELINE.json metric) on N B200s, one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--model force|jerk] [--batch B]
                    [--dump-outputs DIR]

A "step" is one control step for the whole batch of drones: yref windowing + x0 embedding + SQP/HPIPM solve + converter
+ plant step + logs (bnmpc_closed_loop_run).  Workload of the headline at every N: BASELINE config 2, "force_model
batched closed-loop, 4096 drones with randomised x0 and trajectories, FP64" per GPU (weak scaling: each rank owns its
own 4096 instances, no data-path collective).

  value   K control steps of every drone in ONE launch (steps_per_launch = K: queue tickets of (drone, chunk of steps),
          the working set of a drone stays on chip inside a chunk - the Monte-Carlo throughput path), inputs resident in HBM
  per_step_launch   the same K steps as K launches (every launch ends with all drones at the same step - the latency
          path: p50 / p99 step latency), L2 flushed between launches
  e2e     the reference's own loop shape through the AcadosOcpSolver / AcadosSimSolver-style shim with pinned HOST
          buffers, every step: set_up_ocp (yref window), solve_for_x0 (x0 in, u0 + status out), Converter on the host,
          simulate_next_x (x, u, noise in, x_next out)
  extra   bounded runs of BASELINE configs 3 (jerk 16384, FP64 + FP32), 4 (262144 drones with plant-mass perturbation,
          SHARDED over the N ranks - strong scaling) and 5 (horizon 20 / 50 / 100 at 65536 drones)

--impl reference times the CPU restatement of the reference's path (oracle/nmpc_oracle.c, all host threads) - acados
itself is not installable here (DESIGN.md) - on the same instances (same generator, same global ids), a bounded sample.

--dump-outputs DIR writes what the timed closed loop returned for its last control step as DIR/<name>.npy (float64), so
that two builds can be compared output for output; the inputs are seeded and identical from run to run.

bench.py writes nothing into the source tree (which may be read-only): what it compiles at run time goes to a temporary
directory.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

sys.dont_write_bytecode = True          # no __pycache__ in the tree
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'nmpc_solves_per_sec'
UNIT = 'solves/s'
SEED = 2026
MODEL_DIMS = dict(force=(2, 2, 1, 4, 2, 4), jerk=(2, 3, 1, 6, 2, 1), force_dense=(1, 4, 2, 4, 2, 4), thrust=(1, 4, 2, 4, 2, 4))   # nblk n m nx nu erk


def flops_per_solve(nblk, n, m, N, erk_stages, qp_iters, linearisations=1.0):
    """Algorithmic flops (SURVEY 8d formulas, applied to the block structure the solver actually factorises):
    per stage factorisation s n^2 + s^2 n + s^3/3, one KKT solve 4n^2 + 4sn + 2s^2, residuals/barrier 2(2sn + s^2) + 10s;
    per IPM iteration N (F_f + 2 F_s + F_r); per linearisation N (S_rk 2 n^2 s + 2 s^2) - SQP to tolerance linearises once
    more than it solves QPs (the residual test that ends it), SQP_RTI exactly once."""
    s = n + m
    f_f = s * n * n + s * s * n + s ** 3 / 3.0
    f_s = 4 * n * n + 4 * s * n + 2 * s * s
    f_r = 2 * (2 * s * n + s * s) + 10 * s
    f_it = nblk * N * (f_f + 2 * f_s + f_r)
    f_lin = nblk * N * (erk_stages * 2 * n * n * s + 2 * s * s)
    return linearisations * f_lin + qp_iters * f_it


def bytes_per_solve(nx, nu, N):
    """Algorithmic HBM bytes of one closed-loop step (SURVEY 8d): x0 + yref window in, u0 + status/iters out, plus the
    rollout's state r/w, noise and p."""
    return nx * 8 + (N * (nx + nu) + nx) * 8 + nu * 8 + 8 + 64 + 8 + 16


def config_dict(args):
    """What both arms print as `config` (identical for --impl ours and --impl reference)."""
    return {'workload': f'{args.model}_model batched closed loop, {args.batch} drones per GPU with randomised x0 and circle trajectories '
                        f'(BASELINE config 2), N_horizon {args.horizon}, {"SQP_RTI" if args.rti else "SQP to tol 1e-6"} + HPIPM-style IPM, '
                        f'noise sigma 0.01',
            'batch_per_gpu': args.batch, 'horizon': args.horizon, 'controller': args.model, 'precision': args.precision,
            'plant_mass_sigma': args.mass_sigma,
            'instances': f'sharding.instance_inputs(seed {SEED}): Philox draws keyed by the global instance id, per-instance circle tables',
            'reference_table': 'per-instance table [B, rows, 8] in HBM' if args.ref == 'table' else 'generated in the kernel (CircleRef)',
            'l2': 'GPU arm - value: one launch over per-instance tables larger than L2 (157 MB), L2 flushed before it; per_step_launch: '
                  'flushed between launches (256 MiB write, untimed)',
            'timing': 'GPU arm: CUDA events on the launch stream, max over ranks; CPU arm: perf_counter around the timed steps'}


class ClockSampler:
    """SM clock + throttle reasons during the timed region (pynvml; falls back to nvidia-smi)."""

    def __init__(self, index):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thr = None

    def _run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {getattr(nv, k): k for k in dir(nv) if k.startswith('nvmlClocksEventReason') or k.startswith('nvmlClocksThrottleReason')}
            while not self._stop.is_set():
                self.samples.append(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for bit, name in names.items():
                    if isinstance(bit, int) and bit and (r & bit) == bit and bit & (bit - 1) == 0:
                        self.reasons.add(name.replace('nvmlClocksEventReason', '').replace('nvmlClocksThrottleReason', ''))
                time.sleep(0.02)
        except Exception as e:   # noqa: BLE001
            self.reasons.add(f'sampler_error:{type(e).__name__}')

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=2)

    def summary(self):
        med = float(np.median(self.samples)) if self.samples else None
        rs = sorted(r for r in self.reasons if r not in ('None', 'GpuIdle', 'ApplicationsClocksSetting'))
        return {'sm_mhz': med, 'sm_max_mhz': self.max_mhz, 'reasons': rs, 'samples': len(self.samples)}


def workload(lo, hi, n_steps, rows, N, mass_sigma=0.0, with_noise=True):
    """BASELINE config 2 / 4 / SURVEY 8d inputs of the global instances lo..hi-1 as CPU tensors: the circle parameters, the
    reference table ref [rows, 8, b], x0 [4, b], the noise [n_steps, b] and the plant mass scale - from the per-instance
    Philox draws of sharding.instance_inputs, so the numbers do not depend on how many ranks share the batch and BOTH arms
    of the bench (GPU and CPU reference) run exactly these instances."""
    from drone_attitude_control_b200.generate_trajectory import gen_circle_traj_batched
    from drone_attitude_control_b200.sharding import instance_inputs
    inp = instance_inputs(lo, hi, n_steps, seed=SEED, mass_sigma=mass_sigma, with_noise=with_noise)
    n_rev = max(500, rows - N)
    ref = gen_circle_traj_batched(n_rev, rows - n_rev, inp['radius'], inp['center'], inp['phase'])      # [rows, 8, b]
    inp['ref'] = ref
    inp['x0'] = ref[0, :4, :].clone() + inp['dx0']
    return inp


def native_oracle(model):
    """The C restatement rebuilt for THIS host (bench.py runs on the GPU box): -O3 -march=native with the model's dimensions
    as compile-time constants (ORC_FIXED_NX / NU), so the CPU baseline is the port at its best.  Timing only - the parity
    tests use the generic build.  Built in a temporary directory, removed once the library is loaded."""
    from oracle import c_oracle as co
    nx, nu = (6, 2) if model == 'jerk' else (4, 2)
    src = os.path.join(ROOT, 'oracle', 'nmpc_oracle.c')
    flags = ['-O3', '-march=native', f'-DORC_FIXED_NX={nx}', f'-DORC_FIXED_NU={nu}']
    try:
        with tempfile.TemporaryDirectory(prefix='bnmpc_oracle_') as tmp:
            out = os.path.join(tmp, f'libnmpc_oracle_native_{nx}_{nu}.so')
            subprocess.check_call(['gcc'] + flags + ['-pthread', '-fPIC', '-shared', '-o', out, src, '-lm'])
            return co.load_variant(out), ' '.join(flags)
    except Exception as e:   # noqa: BLE001
        return co.lib(), f'generic build -O3 -mavx2 -mfma (native rebuild failed: {type(e).__name__})'


def cpu_closed_loop(args, inp, n_inst, warm, steps):
    """The oracle on the first n_inst instances of `inp`: returns (seconds for `steps` steps after `warm` warm-up steps,
    qp_iter mean over the timed steps, nonzero statuses, cores, build flags)."""
    from oracle import c_oracle as co
    L, flags = native_oracle(args.model)
    model = co.MODEL_JERK if args.model.startswith('jerk') else co.MODEL_FORCE
    cores = co.lib().orc_num_cores()
    refs = inp['ref'][:, :, :n_inst].permute(2, 0, 1).contiguous().numpy()
    x0 = inp['x0'][:, :n_inst].numpy().T.copy()
    noise = inp['noise'][:, :n_inst].contiguous().numpy()
    pc = np.repeat(np.array([[0.03277, 9.81]]), n_inst, 0)
    pp = pc.copy(); pp[:, 0] *= inp['mass_scale'][:n_inst].numpy()
    opts = co.default_opts(model, N=args.horizon, rti=args.rti)
    nw = min(cores, n_inst)
    co.closed_loop(opts, refs[:nw], x0[:nw], np.ascontiguousarray(noise[:2, :nw]), pc[:nw], pp[:nw], 2, outputs=False, L=L)     # warm the threads
    # the oracle API runs whole loops: time the (warm + steps)-step run and the warm-step run and subtract
    t0 = time.perf_counter(); co.closed_loop(opts, refs, x0, noise, pc, pp, warm, nthreads=cores, outputs=False, L=L); tw = time.perf_counter() - t0
    t0 = time.perf_counter(); out = co.closed_loop(opts, refs, x0, noise, pc, pp, warm + steps, nthreads=cores, outputs=True, L=L); tk = time.perf_counter() - t0
    qp = out['qp_iter'][:, warm:warm + steps]
    return max(tk - tw, 1e-9), float(qp.mean()), int((out['status'][:, warm:warm + steps] != 0).sum()), cores, flags


def run_ours(args):
    import ctypes as C
    import torch
    import torch.distributed as dist
    import drone_attitude_control_b200 as pkg
    from drone_attitude_control_b200 import _lib
    from drone_attitude_control_b200.sharding import shard_range

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if args.gpus != world:
        raise SystemExit(f'bench.py --gpus {args.gpus} but WORLD_SIZE is {world}: launch N > 1 as python -m torch.distributed.run '
                         f'--nnodes=1 --nproc-per-node {args.gpus} --master-addr 127.0.0.1 bench.py --gpus {args.gpus} ...')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    B, K, W, N = args.batch, args.steps, args.warmup, args.horizon
    S = W + 2 * K                                   # warm-up, K steps in one launch, K steps as K launches
    rows = max(500 + N, S + N + 1)
    inp = workload(rank * B, (rank + 1) * B, S, rows, N, mass_sigma=args.mass_sigma)   # weak scaling: global ids rank*B ..
    ref_im = inp['ref'].permute(2, 0, 1).contiguous().to(dev)                           # [B, rows, 8] instance-major
    x0, noise = inp['x0'].to(dev), inp['noise'].to(dev)
    loop = pkg.BatchedClosedLoop(args.model, batch=B, device=local, precision=args.precision, N_horizon=N, rti=args.rti)
    p_plant = None
    if args.mass_sigma > 0:                                                             # BASELINE config 4: model mismatch
        p_plant = torch.stack([0.03277 * inp['mass_scale'], torch.full((B,), 9.81, dtype=torch.float64)])
    ref_arg = pkg.CircleRef(inp['radius'], inp['center'], inp['phase'], n=max(500, rows - N)) if args.ref == 'circle' else ref_im
    loop.init(x0, ref_arg, noise=noise, p_plant=p_plant, n_steps=S, log=True)
    stream = torch.cuda.current_stream()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])

    loop.run(W)                                   # warm-up steps (untimed, one launch each)
    flush.fill_(1)
    barrier()
    # ---- value: K control steps of every drone in one launch ---------------------------------------------------------
    l0 = loop.solver.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        t0 = time.perf_counter()
        e0.record(stream)
        loop.run(K, steps_per_launch=args.steps_per_launch or K)
        e1.record(stream)
        barrier()
        wall = time.perf_counter() - t0
        launches = loop.solver.launch_count() - l0
        ms_multi = e0.elapsed_time(e1)
        # ---- the same K steps as K launches (latency path), L2 flushed between launches ------------------------------
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        for i in range(K):
            flush.fill_(i & 0xff)
            evs[i][0].record(stream)
            loop.run(1)
            evs[i][1].record(stream)
        barrier()
    step_ms = np.array([a.elapsed_time(b) for a, b in evs])
    ms_multi_all, ms_step_all = allmax(ms_multi), allmax(float(step_ms.sum()))
    value = world * B * K / (ms_multi_all * 1e-3)
    res = loop.results()
    qp = res['qp_iter'][:, W:W + K].double()
    st = res['status'][:, W:W + K]
    sqp_mean = float(loop.solver.get_stats('sqp_iter').double().mean())
    stats = torch.tensor([float(qp.sum()), float((st != 0).sum()), float(res['cost'].sum()), float(res['aed'].sum()), float(B),
                          float(res['failures'].sum())], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(stats)                    # the only collective of the headline: final per-step metrics (< 1 KB)
    qp_local = float(qp.sum())
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res, S - 1, rank, world)
    del loop, res

    # ---- e2e: the reference's loop shape through the shim with pinned host buffers, every step ------------------------
    e2e = None
    if not args.skip_e2e:
        e2e = run_e2e(args, pkg, dev, local, inp, ref_im, world, barrier, allmax, min(K, args.e2e_steps))
    del ref_im
    torch.cuda.empty_cache()

    # ---- extra: BASELINE configs 3, 4, 5, bounded ---------------------------------------------------------------------
    extra = None
    if not args.skip_extra:
        extra = run_extra(args, pkg, dev, local, rank, world, barrier, allmax, shard_range)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    # ---- roofline of the dominant kernel (k_loop_step = the whole step) ----------------------------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    tf = C.c_double()
    _lib.check(_lib.lib().bnmpc_measure_fma_peak(local, _lib.FP32 if args.precision == 'fp32' else _lib.FP64, C.byref(tf)))
    nblk, n, m, nx, nu, erk = MODEL_DIMS[args.model]
    lin = 1.0 if args.rti else sqp_mean + 1.0
    fl = flops_per_solve(nblk, n, m, N, erk, qp_local / (B * K), lin) * B * K       # per launch (K steps), this rank
    by = bytes_per_solve(nx, nu, N) * B * K
    ach_tf = fl / (ms_multi * 1e-3) * 1e-12
    ach_gbs = by / (ms_multi * 1e-3) * 1e-9
    hbm_peak = peaks.get('hbm_gbs', 6650.0)
    traffic, ncu_view = None, None
    try:       # dram bytes per launch and pipe utilisation of the dominant kernel from the committed ncu capture of this config
        ncu_view = json.load(open(os.path.join(ROOT, 'profiles', 'traffic.json'))).get(f'{args.model}_{args.precision}_B{B}_multistep')
        # (the capture covers a launch of `steps_in_capture` control steps: scale to this launch's K steps)
        traffic = ncu_view['traffic_bytes'] / ncu_view.get('steps_in_capture', 1) * K if ncu_view else None
    except Exception:
        pass
    cfg = config_dict(args)
    line = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms_multi_all / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64' if args.precision == 'fp64' else 'f32', 'data': 'synthetic', 'config': cfg,
        'launch_mode': f'value = {K} control steps of every drone in {launches} launch(es) (steps_per_launch = {args.steps_per_launch or K})',
        'per_step_launch': {'value': world * B * K / (ms_step_all * 1e-3), 'unit': UNIT, 'ms_per_step': ms_step_all / K,
                            'p50_step_latency_ms': float(np.median(step_ms)), 'p99_step_latency_ms': float(np.percentile(step_ms, 99)),
                            'gpu_launches': K},
        'p50_step_latency_ms': float(np.median(step_ms)), 'p99_step_latency_ms': float(np.percentile(step_ms, 99)),
        'qp_iter_mean': float(stats[0]) / (world * B * K), 'sqp_iter_mean': sqp_mean, 'nonzero_status': int(stats[1]),
        'failed_steps_whole_run': int(stats[5]),
        'closed_loop_cost_mean': float(stats[2]) / float(stats[4]), 'aed_mean': float(stats[3]) / float(stats[4]),
        'gpu_launches': int(launches), 'wall_s_timed_region': wall,
        'clocks': clk.summary(),
        'e2e': e2e,
        'roofline': {'bound': 'fp64' if args.precision == 'fp64' else 'fp32', 'achieved': ach_tf, 'peak': tf.value, 'unit': 'TFLOP/s',
                     'frac': ach_tf / tf.value if tf.value else None, 'traffic': traffic,
                     'peak_source': 'measured live: bnmpc_measure_fma_peak (MEASURED_PEAKS.json has no vector-pipe figure); '
                                    'a recorded copy with its clock record is profiles/fma_peak.json',
                     'kernel': 'k_loop_step', 'flops_per_launch': fl, 'ms_per_launch': ms_multi,
                     'linearisations_per_solve': lin, 'ncu': ncu_view,
                     'hbm': {'bound': 'hbm', 'achieved': ach_gbs, 'peak': hbm_peak, 'unit': 'GB/s', 'frac': ach_gbs / hbm_peak,
                             'bytes_per_launch': by,
                             'peak_source': 'MEASURED_PEAKS.json hbm_gbs' if 'hbm_gbs' in peaks else 'fallback 6650'}},
        'extra': extra,
    }
    if not args.skip_cpu and world == 1:
        n_inst = min(args.cpu_instances, B)
        inp_cpu = workload(0, n_inst, W + args.cpu_steps, max(500 + N, W + args.cpu_steps + N + 1), N, mass_sigma=args.mass_sigma)   # same ids, more steps
        dt, qpm, bad, cores, flags = cpu_closed_loop(args, inp_cpu, n_inst, W, args.cpu_steps)
        dense_ratio = flops_per_solve(1, nx, nu, N, erk, 1, 0) / flops_per_solve(nblk, n, m, N, erk, 1, 0)
        line['cpu_baseline'] = {'value': n_inst * args.cpu_steps / dt, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                'qp_iter_mean': qpm, 'nonzero_status': bad,
                                'sample': f'the first {n_inst} of the workload\'s instances (same global ids, same inputs) x {args.cpu_steps} '
                                          f'closed-loop steps after {W} warm-up steps, oracle/nmpc_oracle.c built {flags}, {cores} pthreads, '
                                          f'{dt:.1f} s; the port factorises dense {nx}-state stages (no x/z block split: '
                                          f'{dense_ratio:.1f}x the flops per IPM iteration of the GPU path)'}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20
DUMP_HEADER_BYTES = 1024        # room kept for the header of each .npy file


def dump_outputs(out_dir, res, step, rank, world):
    """--dump-outputs: what BatchedClosedLoop.results() gives a caller for control step `step` (the last timed one) - the
    plant state after it, controller and plant inputs, carried acceleration, status and QP iterations - and the per-drone
    totals of the run (closed-loop cost, AED, failed steps), one row per drone in global instance order, as float64 .npy.
    Above DUMP_LIMIT_BYTES the rows are a fixed seeded sample of the drones; `drone.npy` holds the global ids of the rows."""
    import torch
    arrays = {'Xsim': res['Xsim'][:, step + 1], 'U_ctrl': res['U_ctrl'][:, step], 'U_plant': res['U_plant'][:, step],
              'a': res['a'][:, step], 'status': res['status'][:, step], 'qp_iter': res['qp_iter'][:, step],
              'cost': res['cost'], 'aed': res['aed'], 'failures': res['failures']}
    arrays = {k: v.double().contiguous() for k, v in arrays.items()}
    if world > 1:                                   # every rank owns the same number of drones (weak scaling), in rank order
        import torch.distributed as dist
        for k, v in arrays.items():
            parts = [torch.empty_like(v) for _ in range(world)]
            dist.all_gather(parts, v)
            arrays[k] = torch.cat(parts)
    if rank != 0:
        return
    total = arrays['cost'].shape[0]
    row_bytes = 8 * (1 + sum(v[0].numel() for v in arrays.values()))
    max_rows = (DUMP_LIMIT_BYTES - DUMP_HEADER_BYTES * (1 + len(arrays))) // row_bytes
    rows = np.arange(total)
    if total > max_rows:
        rows = np.sort(np.random.default_rng(SEED).choice(total, max_rows, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'drone.npy'), rows.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f'{k}.npy'), v.cpu().numpy()[rows])


def run_e2e(args, pkg, dev, local, inp, ref_im, world, barrier, allmax, Ke):
    """follow_trajectory of the reference (src/force_model/controller.py:25-54 / src/jerk_model/controller.py:26-56) for the
    whole batch through the AcadosOcpSolver-style shim, host buffers in and out every step:
        set_up_ocp (yref window H2D) -> set x0 (H2D) -> solve -> get u0, status (D2H) -> Converter on the host ->
        simulate_next_x (x, u, noise H2D; x_next D2H) -> next step's x0.
    The window of step i+1 is known in advance, so its upload is enqueued on a copy stream behind step i's x0 and overlaps
    the solve; everything that depends on the solution is serial, as in the reference."""
    import torch
    B, N, W = args.batch, args.horizon, args.warmup
    s = pkg.BatchedAcadosOcpSolver(args.model, batch=B, device=local, precision=args.precision, N_horizon=N, rti=args.rti, numpy_io=False)
    ny, nx, nu = s.ny, s.nx, s.nu
    jerk = nx == 6
    nsub = int(s.cfg.sim_substeps)
    hc = float(s.cfg.sim_dt)
    ref_h = ref_im.cpu()                                      # [B, rows, 8]
    ycols = list(range(nx)) + [nx + j for j in range(nu)] if jerk else [0, 1, 2, 3, 4, 5]
    yh = [torch.cat([ref_h[:, i:i + N, ycols].reshape(B, N * ny), ref_h[:, i + N, :nx]], 1).contiguous().pin_memory()
          for i in range(W + Ke)]
    noise_h = inp['noise'][:W + Ke].contiguous().pin_memory()      # [steps, B]
    pin = lambda *sh, dt=torch.float64: torch.empty(sh, dtype=dt).pin_memory()
    x0h, u_host, st_host = pin(B, nx), pin(B, nu), pin(B, dt=torch.int32)
    xs_h, up_h, xn_h = pin(B, 4), pin(B, nsub, 2), pin(B, 4)
    acc = torch.zeros(B, 2, dtype=torch.float64)
    per = N * ny + nx
    ydev = [torch.empty((B, per), dtype=torch.float64, device=dev) for _ in range(2)]
    yev = [torch.cuda.Event(), torch.cuda.Event()]
    copy_stream = torch.cuda.Stream(device=dev)
    mass = 0.03277

    def prefetch(i):      # upload the reference window of step i on the copy stream (overlaps the solve of step i-1)
        with torch.cuda.stream(copy_stream):
            ydev[i % 2].copy_(yh[i], non_blocking=True)
            yev[i % 2].record(copy_stream)

    x0b = [pin(B, nx), pin(B, nx)]

    def start():
        s.reset()
        xs_h.copy_(inp['x0'].t())
        acc[:, 0] = 0.0; acc[:, 1] = 9.81
        x0b[0][:, :4] = xs_h
        if jerk:
            x0b[0][:, 4:] = acc
        prefetch(0)

    def step_fused(i, last):
        """one C-ABI call per control step: x0 + noise in; solve, Converter, plant step on the device; u0, u_plant, status and
        the next x0 out"""
        torch.cuda.current_stream().wait_event(yev[i % 2])
        s.set_yref_all(ydev[i % 2])                                      # OCP.set_up_ocp
        s.step_into(x0b[i % 2], noise_h[i], u_host, up_h[:, 0], st_host, x0b[(i + 1) % 2], wait=False)
        if not last:
            prefetch(i + 1)
        s.synchronize()

    def step_calls(i, last):
        """the reference's call sequence: solve_for_x0, Converter on the host, simulate_next_x"""
        torch.cuda.current_stream().wait_event(yev[i % 2])
        s.set_yref_all(ydev[i % 2])
        x0h[:, :4] = xs_h
        if jerk:
            x0h[:, 4:] = acc
        s.solve_for_x0_into(x0h, u_host, st_host, wait=False)           # x0 in, solve, u0 + status out (pinned host)
        if not last:
            prefetch(i + 1)
        s.synchronize()
        if jerk:                                                         # Converter.convert, jerk dynamics.py:76-83
            for j in range(nsub):
                acc.add_(u_host, alpha=hc)
                f = mass * acc
                up_h[:, j, 0] = torch.atan2(f[:, 0], f[:, 1]); up_h[:, j, 1] = torch.sqrt(f[:, 0] ** 2 + f[:, 1] ** 2)
        else:                                                            # dynamics.py:66-70
            up_h[:, 0, 0] = torch.atan2(u_host[:, 0], u_host[:, 1]); up_h[:, 0, 1] = torch.sqrt(u_host[:, 0] ** 2 + u_host[:, 1] ** 2)
        s.simulate_next_x_into(xs_h, up_h, noise_h[i], xn_h, wait=True)  # OCP.simulate_next_x incl. the noise draw
        xs_h.copy_(xn_h)

    def run(step):
        start()
        for i in range(W):
            step(i, False)
        barrier()
        t0 = time.perf_counter()
        for i in range(W, W + Ke):
            step(i, i == W + Ke - 1)
        barrier()
        return allmax(time.perf_counter() - t0)

    dt_calls = run(step_calls)
    x_calls = xs_h.clone()
    dt_one = run(step_fused)
    x_one = x0b[(W + Ke) % 2].clone()
    same = float((x_one[:, :4] - x_calls).abs().max())                 # both paths walked the same closed loop
    s = None                                                            # (frees the single solver's workspace)
    upf = pin(B, 2)

    # ---- the same step for the fleet split into G solver objects on G streams (SolverFleet): a sub-fleet is synchronised
    #      only right before its own next step is enqueued, so the tail of one launch overlaps the next sub-fleet's launch
    G = max(1, min(args.e2e_groups, B))
    fleet = pkg.SolverFleet(args.model, batch=B, groups=G, device=local, precision=args.precision, N_horizon=N, rti=args.rti)
    bad_steps = [0]

    def on_results(g, lo, hi):                                          # the reference's status check, per sub-fleet
        bad_steps[0] += int((st_host[lo:hi] != 0).sum())

    def run_fleet():
        fleet.reset()
        x0b[0][:, :4] = inp['x0'].t()
        if jerk:
            x0b[0][:, 4] = 0.0; x0b[0][:, 5] = 9.81
        for i in range(W):
            fleet.step(yh[i], x0b[i % 2], noise_h[i], u_host, upf, st_host, x0b[(i + 1) % 2])
        fleet.synchronize()
        bad_steps[0] = 0
        barrier()
        t0 = time.perf_counter()
        for i in range(W, W + Ke):
            fleet.step(yh[i], x0b[i % 2], noise_h[i], u_host, upf, st_host, x0b[(i + 1) % 2], on_results=on_results)
        fleet.synchronize(on_results=on_results)
        barrier()
        return allmax(time.perf_counter() - t0)

    dt = run_fleet()
    same_fleet = float((x0b[(W + Ke) % 2] - x_one).abs().max())          # identical to the single solver object (bit for bit)
    bad = int((st_host != 0).sum())
    return {'value': world * B * Ke / dt, 'unit': UNIT, 'steps': Ke, 'ms_per_step': dt / Ke * 1e3,
            'h2d_bytes_per_step': int(B * (per + nx + 1) * 8), 'd2h_bytes_per_step': int(B * (nu * 8 + 2 * 8 + 4 + nx * 8)),
            'nonzero_status_last_step': bad, 'nonzero_status_steps_seen_by_host': bad_steps[0], 'groups': G,
            'api': f'per control step, pinned host buffers, SolverFleet of {G} solver objects on {G} streams (sub-fleets of {B // G} drones, '
                   'software-pipelined: a sub-fleet is synchronised - and its statuses checked on the host - right before its own next step '
                   'is enqueued); per sub-fleet BatchedAcadosOcpSolver.set_yref_all (OCP.set_up_ocp: the yref window, H2D) + step_into = '
                   'bnmpc_step_for_x0 (x0 and the noise draw in; x0 embedding, solve, get(0,u), Converter.convert and simulate_next_x on the '
                   'device; u0, u_plant, status and the next x0 out)',
            'max_abs_state_difference_to_single_solver': same_fleet,
            'single_solver': {'value': world * B * Ke / dt_one, 'unit': UNIT, 'ms_per_step': dt_one / Ke * 1e3,
                              'api': 'the same calls on ONE solver object for the whole batch, synchronised every step; the upload of the '
                                     'next step\'s window rides a copy stream behind this step\'s x0'},
            'reference_call_sequence': {'value': world * B * Ke / dt_calls, 'unit': UNIT, 'ms_per_step': dt_calls / Ke * 1e3,
                                        'h2d_bytes_per_step': int(B * (per + nx + 4 + 2 * nsub + 1) * 8),
                                        'd2h_bytes_per_step': int(B * (nu * 8 + 4 + 4 * 8)),
                                        'api': 'solve_for_x0 (x0 in, u0 + status out), Converter on the host, simulate_next_x (x, u, noise in, '
                                               'x_next out): two device round trips per step, as the reference\'s loop makes them',
                                        'max_abs_state_difference_to_fused_call': same}}


def run_extra(args, pkg, dev, local, rank, world, barrier, allmax, shard_range):
    """Bounded runs of BASELINE configs 3, 4, 5 with the multi-step launch path (inputs resident, circle reference generated in
    the kernel, noise drawn in the kernel by Philox): solves/s, statuses, algorithmic roofline fraction."""
    import ctypes as C
    import torch
    from drone_attitude_control_b200 import _lib
    from drone_attitude_control_b200.sharding import instance_inputs
    peak = {}

    def fma_peak(prec):
        if prec not in peak:
            tf = C.c_double()
            _lib.check(_lib.lib().bnmpc_measure_fma_peak(local, _lib.FP32 if prec == 'fp32' else _lib.FP64, C.byref(tf)))
            peak[prec] = tf.value
        return peak[prec]

    def one(model, total, N, prec, steps, warm, mass_sigma, sharded, table=False, rti=False):
        lo, hi = shard_range(total, rank, world) if sharded else (rank * total, (rank + 1) * total)
        b = hi - lo
        inp = instance_inputs(lo, hi, 0, seed=SEED, mass_sigma=mass_sigma, with_noise=False)
        om = 2 * np.pi / 10
        if table:      # per-instance reference tables in HBM, as in the headline configuration
            from drone_attitude_control_b200.generate_trajectory import gen_circle_traj_batched
            cref = gen_circle_traj_batched(500, N, inp['radius'], inp['center'], inp['phase'], device=dev).permute(2, 0, 1).contiguous()
        else:
            cref = pkg.CircleRef(inp['radius'], inp['center'], inp['phase'], n=500)
        r, ph, c = inp['radius'], inp['phase'], inp['center']
        x0 = torch.stack([c[:, 0] + r * torch.cos(ph), c[:, 1] + r * torch.sin(ph), -r * om * torch.sin(ph), r * om * torch.cos(ph)]) + inp['dx0']
        loop = pkg.BatchedClosedLoop(model, batch=b, device=local, precision=prec, N_horizon=N, rti=rti)
        pp = torch.stack([0.03277 * inp['mass_scale'], torch.full((b,), 9.81, dtype=torch.float64)]) if mass_sigma > 0 else None
        loop.init(x0, cref, noise=pkg.PhiloxNoise(seed=SEED, std=0.01, first_instance=lo), p_plant=pp, n_steps=warm + steps, log=False)
        loop.run(warm, steps_per_launch=warm)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); loop.run(steps, steps_per_launch=steps); e1.record()
        barrier()
        ms = allmax(e0.elapsed_time(e1))
        qp = loop.solver.get_stats('qp_iter').double()
        sq = loop.solver.get_stats('sqp_iter').double()
        st = torch.tensor([float(loop.failures().sum()), float(qp.sum()), float(sq.sum()), float(b)], dtype=torch.float64, device=dev)
        if world > 1:
            import torch.distributed as dist
            dist.all_reduce(st)
        tot = int(st[3])
        nblk, n, m, nx, nu, erk = MODEL_DIMS[model]
        fl = flops_per_solve(nblk, n, m, N, erk, float(st[1]) / tot, 1.0 if rti else float(st[2]) / tot + 1.0) * tot * steps
        ach = fl / (ms * 1e-3) * 1e-12
        del loop
        torch.cuda.empty_cache()
        return {'model': model, 'instances_total': tot, 'instances_this_rank': b, 'sharded_over_ranks': bool(sharded), 'horizon': N,
                'precision': prec, 'nlp_solver': 'SQP_RTI' if rti else 'SQP', 'steps': steps, 'warmup': warm, 'ms': ms, 'reference': 'tables in HBM' if table else 'generated in the kernel', 'value': tot * steps / (ms * 1e-3), 'unit': UNIT,
                'failed_steps': int(st[0]), 'qp_iter_mean_last_step': float(st[1]) / tot,
                'roofline_frac': ach / fma_peak(prec), 'achieved_tflops': ach}

    out = {'note': 'multi-step launches (steps_per_launch = steps), noise drawn in the kernel (PhiloxNoise), reference tables in HBM (config 3) '
                   'or generated in the kernel (configs 4, 5), CUDA events, max over ranks'}
    # the metric's name says SQP-RTI; the reference's OCP is configured nlp_solver_type = 'SQP' (src/force_model/ocp.py:83), which the
    # headline follows - this is config 2 with one QP per control step (acados SQP_RTI), 4096 drones per GPU, tables in HBM
    out['config2_force_4096_sqp_rti'] = one('force', 4096, 30, 'fp64', 100, 10, 0.0, False, table=True, rti=True)
    out['config3_jerk_16384_fp64'] = one('jerk', 16384, 30, 'fp64', 20, 5, 0.0, False, table=True)
    out['config3_jerk_16384_fp32'] = one('jerk', 16384, 30, 'fp32', 20, 5, 0.0, False, table=True)
    out['config4_force_262144_mass_perturbed_sharded'] = dict(one('force', 262144, 30, 'fp64', 10, 3, 0.05, True), scaling='strong')
    for N in (20, 50, 100):
        out[f'config5_force_65536_N{N}'] = one('force', 65536, N, 'fp64', 4 if N > 30 else 8, 2, 0.0, False)
    out['north_star_att_3d_nx10_nu4'] = att_extra(args, dev, local, rank, world, barrier, allmax)
    out['north_star_att_3d_nx10_nu4_sqp_rti'] = att_extra(args, dev, local, rank, world, barrier, allmax, steps=12, warm=8, rti=True)
    return out


def att_extra(args, dev, local, rank, world, barrier, allmax, per_rank=4736, steps=6, warm=4, rti=False):
    """The 3-D attitude-and-total-thrust OCP of the north-star (nx 10, nu 4; not in the reference): closed loop of `per_rank`
    drones per GPU on per-instance helix references with a 5 % plant-mass perturbation, device-resident, one
    bnmpc_step_for_x0 per control step (solve kernel + plant kernel); SQP to tolerance.  With --skip-cpu unset, rank 0 also
    times the C restatement (oracle/, kind "port") on a bounded sample of the same instances on all host cores."""
    import torch
    from drone_attitude_control_b200.attitude_model import follow_trajectory_batched, helix_table
    from drone_attitude_control_b200.sharding import instance_inputs
    lo, hi = rank * per_rank, (rank + 1) * per_rank
    inp = instance_inputs(lo, hi, 0, seed=SEED, mass_sigma=0.05, with_noise=False)
    b = hi - lo
    c3 = torch.stack([inp['center'][:, 0], torch.zeros(b, dtype=torch.float64), inp['center'][:, 1]], 1)
    rows = warm + steps + 30
    ref = helix_table(inp['radius'] * 0.9, c3, inp['phase'], 0.2 * inp['radius'], rows, device=dev)
    x0 = ref[:, 0, :10].clone()
    x0[:, :4] += inp['dx0'].to(dev).T
    pp = torch.stack([0.03277 * inp['mass_scale'], torch.full((b,), 9.81, dtype=torch.float64)], 1).to(dev)
    state = {}

    def run(first, n, x):
        kw = {} if 'solver' in state or not rti else {'rti': True}
        r = follow_trajectory_batched(ref[:, first:], x, n, p_plant=pp, device=local, log=True, solver=state.get('solver'), **kw)
        state['solver'] = r['solver']
        return r
    r0 = run(0, warm, x0)                                     # warm-up: the cold-start solves
    torch.cuda.synchronize(); barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); r1 = run(warm, steps, r0['Xsim'][:, -1].contiguous()); e1.record()
    barrier()
    ms = allmax(e0.elapsed_time(e1))
    st = torch.tensor([float((r1['status'] != 0).sum()), float(r1['qp_iter'].sum()), float(r1['sqp_iter'].sum()), float(b)], dtype=torch.float64, device=dev)
    if world > 1:
        import torch.distributed as dist
        dist.all_reduce(st)
    tot = int(st[3])
    perr = float((r1['Xsim'][:, 1:, :3] - ref[:, warm + 1:warm + steps + 1, :3]).norm(dim=2).mean())
    out = {'model': 'att', 'nlp_solver': 'SQP_RTI' if rti else 'SQP', 'mean_position_error_m': perr, 'instances_total': tot, 'horizon': 30, 'precision': 'fp64', 'steps': steps, 'warmup': warm, 'ms': ms,
           'value': tot * steps / (ms * 1e-3), 'unit': UNIT, 'failed_steps': int(st[0]), 'qp_iter_mean': float(st[1]) / (tot * steps),
           'sqp_iter_mean': float(st[2]) / (tot * steps), 'launches_per_step': 2,
           'path': 'bnmpc_set_yref_all + bnmpc_step_for_x0 per control step, device buffers'}
    fl = flops_per_solve(1, 10, 4, 30, 4, out['qp_iter_mean'], 1.0 if rti else out['sqp_iter_mean'] + 1.0) * tot * steps
    out['achieved_tflops'] = fl / (ms * 1e-3) * 1e-12
    tf = C_peak(local)
    out['roofline_frac'] = out['achieved_tflops'] / tf if tf else None
    if not args.skip_cpu and rank == 0 and not rti:
        import time
        from oracle import c_oracle as co
        ns = min(b, 8 * max(1, co.lib().orc_num_cores()))
        oc = co.default_opts(co.MODEL_ATT)
        xs = r0['Xsim'][:ns, -1].cpu().numpy()
        it = np.zeros((ns, 31, 10)); it[:, :, 6] = 1.0
        t0 = time.perf_counter()
        w = co.closed_loop_att(oc, ref[:ns, warm:].cpu().numpy(), xs, None, np.tile([0.03277, 9.81], (ns, 1)), pp[:ns].cpu().numpy(), steps)
        dt_ = time.perf_counter() - t0
        out['cpu_baseline'] = {'value': ns * steps / dt_, 'unit': UNIT, 'cores': int(co.lib().orc_num_cores()), 'kind': 'port',
                               'sample': f'{ns} of the same instances x {steps} steps from the same plant states (cold iterate), all host cores',
                               'qp_iter_mean': float(w['qp_iter'].mean())}
    return out


def C_peak(local):
    import ctypes as C
    from drone_attitude_control_b200 import _lib
    tf = C.c_double()
    _lib.check(_lib.lib().bnmpc_measure_fma_peak(local, _lib.FP64, C.byref(tf)))
    return tf.value


def run_reference(args):
    """--impl reference: the CPU restatement of the reference's path on the host cores, same metric, same config, same
    instances (sharding.instance_inputs of the same global ids), a bounded sample per step."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    K, W, N = args.steps, args.warmup, args.horizon
    Bs = min(args.cpu_instances, args.batch)
    rows = max(500 + N, W + K + N + 1)
    inp = workload(0, Bs, W + K, rows, N, mass_sigma=args.mass_sigma)
    dt, qpm, bad, cores, flags = cpu_closed_loop(args, inp, Bs, W, K)
    value = Bs * K / dt
    world = int(os.environ.get('WORLD_SIZE', '1'))
    sample = (f'the first {Bs} of the workload\'s {args.batch} instances per step (same global ids and inputs as the GPU arm), '
              f'oracle/nmpc_oracle.c built {flags}, {cores} pthreads')
    print(json.dumps({
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': dt / K * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f64' if args.precision == 'fp64' else 'f32', 'data': 'synthetic', 'config': config_dict(args),
        'qp_iter_mean': qpm, 'nonzero_status': bad,
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--model', default='force', choices=['force', 'jerk', 'force_dense', 'thrust'])
    ap.add_argument('--batch', type=int, default=4096, help='instances per GPU')
    ap.add_argument('--horizon', type=int, default=30)
    ap.add_argument('--precision', default='fp64', choices=['fp64', 'fp32'])
    ap.add_argument('--rti', action='store_true')
    ap.add_argument('--ref', default='table', choices=['table', 'circle'], help='trajectory table in HBM, or generated in the kernel')
    ap.add_argument('--mass-sigma', type=float, default=0.0, help='BASELINE config 4: plant mass = 0.03277 (1 + N(0, sigma)) clipped to +-15 %%')
    ap.add_argument('--steps-per-launch', type=int, default=0, help='control steps per launch of the `value` leg (default: all K in one launch)')
    ap.add_argument('--skip-e2e', action='store_true')
    ap.add_argument('--skip-cpu', action='store_true')
    ap.add_argument('--skip-extra', action='store_true')
    ap.add_argument('--e2e-steps', type=int, default=50)
    ap.add_argument('--e2e-groups', type=int, default=4, help='solver objects (streams) the e2e leg splits the batch into (SolverFleet)')
    ap.add_argument('--cpu-instances', type=int, default=4096)
    ap.add_argument('--cpu-steps', type=int, default=400, help='closed-loop steps of the cpu_baseline sample (~10-20 s of CPU work on 16 cores)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed control step as DIR/<name>.npy (float64)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs dumps the GPU path; the reference arm has no outputs to dump')
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
