"""AcadosOcpSolver / AcadosSimSolver-style surface over libbnmpc (batched, CUDA only).

The reference drives acados through `acados_template.AcadosOcpSolver` / `AcadosSimSolver`
(reference src/force_model/ocp.py:95-96,104; calls at src/force_model/controller.py:30-39, src/force_model/ocp.py:108-112,
120-122).  These classes keep the same method names and meaning for `batch` independent instances:

    set(stage, field, value)   get(stage, field)   solve() -> status   get_stats(name)   print_statistics()
    solve_for_x0(x0_bar)       get_cost()          reset()
    eval_solution_sensitivity()             eval_adjoint_solution_sensitivity(seed_x, seed_u)
    eval_param_sensitivity()                eval_adjoint_param_sensitivity(seed_x, seed_u)

`value` is a `[batch, dim]` tensor (CUDA or CPU) or numpy array; with batch == 1 a plain `(dim,)` numpy vector is
accepted and `get` returns one, so the reference's `follow_trajectory` runs against this class unchanged apart from the
constructor.  `solve()` returns the acados status int for batch == 1 and an int32 tensor `[batch]` otherwise.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib
from ._lib import FIELDS, STATS, BnmpcError, check, default_config, lib


def _require_cuda(device):
    if not torch.cuda.is_available():
        raise BnmpcError('no CUDA device: this solver runs on the GPU only (there is no CPU fallback)')
    return torch.device('cuda', device if isinstance(device, int) else torch.device(device).index or 0)


class BatchedAcadosOcpSolver:
    """`AcadosOcpSolver` of the reference's OCP (src/force_model/ocp.py:21-96 or src/jerk_model/ocp.py:20-95) for `batch` drones."""

    def __init__(self, model='force', batch=1, device=0, precision='fp64', N_horizon=None, rti=False, numpy_io=None, **overrides):
        self.device = _require_cuda(device)
        kw = dict(overrides)
        if N_horizon is not None:
            kw['horizon'] = int(N_horizon)
        kw['precision'] = _lib.FP32 if precision in ('fp32', 'float32', _lib.FP32) else _lib.FP64
        kw['rti'] = int(bool(rti))
        if kw['precision'] == _lib.FP32:
            # what single precision can certify: stationarity / equality / inequality residuals carry ~1e-5 of round-off,
            # the complementarity tolerance stays at acados' 1e-6 (the multipliers of this OCP are tiny, DESIGN.md 2)
            kw.setdefault('qp_tol', [1e-4, 1e-4, 1e-4, 1e-6])
            kw.setdefault('tol', [1e-3, 1e-3, 1e-3, 1e-5])
        self.cfg = default_config(model, **kw)
        self.model = model
        self.batch = int(batch)
        self.numpy_io = (self.batch == 1) if numpy_io is None else bool(numpy_io)
        self._h = C.c_void_p()
        check(lib().bnmpc_create(C.byref(self.cfg), self.batch, self.device.index, C.byref(self._h)))
        dims = (C.c_int32 * 7)()
        check(lib().bnmpc_dims(self._h, dims))
        self.nx, self.nu, self.ny, self.ny_e, self.N, self.np_, self.nblk = [int(v) for v in dims]
        self._bind_stream()
        self._time_tot = 0.0
        self.solve_count = 0        # solves (and resets) so far: a sensitivity belongs to the solution of one of them

    # -- plumbing ------------------------------------------------------------------------------------------------------
    def _bind_stream(self):
        with torch.cuda.device(self.device):
            self._stream = torch.cuda.current_stream()
        check(lib().bnmpc_set_stream(self._h, C.c_void_p(self._stream.cuda_stream)))

    def __del__(self):
        h, self._h = getattr(self, '_h', None), None
        if h:
            try:
                lib().bnmpc_destroy(h)
            except Exception:
                pass

    @property
    def handle(self):
        return self._h

    def _dim(self, stage, field):
        N = self.N
        return {'x': self.nx if 0 <= stage <= N else 0, 'u': self.nu if 0 <= stage < N else 0,
                'yref': (self.ny if 0 <= stage < N else (self.ny_e if stage == N else 0)),
                'lbx': self.nx if 0 <= stage < N else 0, 'ubx': self.nx if 0 <= stage < N else 0, 'p': self.np_,
                'lbu': self.nu if 0 <= stage < N else 0, 'ubu': self.nu if 0 <= stage < N else 0,
                'pi': self.nx if 0 <= stage < N else 0,
                'lam': 2 * self.nu if stage == 0 else (2 * (self.nu + self.nx) if 0 < stage < N else 0)}[field]

    def _as_arg(self, value, dim):
        """-> (keepalive, pointer, on_device) for a [batch, dim] float64 buffer"""
        if isinstance(value, torch.Tensor):
            t = value.detach().to(torch.float64)
            if t.dim() == 1 and self.batch == 1:
                t = t[None]
            if tuple(t.shape) != (self.batch, dim):
                raise ValueError(f'expected shape ({self.batch}, {dim}), got {tuple(value.shape)}')
            t = t.contiguous()
            if t.is_cuda and t.device != self.device:
                t = t.to(self.device)
            return t, C.c_void_p(t.data_ptr()), int(t.is_cuda)
        a = np.ascontiguousarray(value, dtype=np.float64)
        if a.ndim == 1 and self.batch == 1:
            a = a[None]
        if a.shape != (self.batch, dim):
            raise ValueError(f'expected shape ({self.batch}, {dim}), got {np.shape(value)}')
        return a, C.c_void_p(a.ctypes.data), 0

    # -- the acados surface ---------------------------------------------------------------------------------------------
    def set(self, stage, field, value):
        if field not in FIELDS:
            raise ValueError(f'unknown field {field!r}')
        dim = self._dim(int(stage), field)
        if dim == 0:
            raise ValueError(f'field {field!r} does not exist at stage {stage}')
        keep, ptr, on_dev = self._as_arg(value, dim)
        check(lib().bnmpc_set(self._h, int(stage), FIELDS[field], ptr, on_dev))
        if on_dev == 0:
            pass   # the library copied the host buffer before returning (pageable) or on its stream (pinned)
        self._keep = keep

    def get(self, stage, field):
        if field not in FIELDS:
            raise ValueError(f'unknown field {field!r}')
        dim = self._dim(int(stage), field)
        if dim == 0:
            raise ValueError(f'field {field!r} does not exist at stage {stage}')
        if self.numpy_io:
            out = np.empty((self.batch, dim))
            check(lib().bnmpc_get(self._h, int(stage), FIELDS[field], C.c_void_p(out.ctypes.data), 0))
            return out[0] if self.batch == 1 else out
        out = torch.empty((self.batch, dim), dtype=torch.float64, device=self.device)
        check(lib().bnmpc_get(self._h, int(stage), FIELDS[field], C.c_void_p(out.data_ptr()), 1))
        return out

    def set_yref_all(self, yref):
        """OCP.set_up_ocp in one call: [batch, N*ny + ny_e] = yref_0 .. yref_{N-1}, yref_N (src/force_model/ocp.py:117-122)."""
        keep, ptr, on_dev = self._as_arg(yref, self.N * self.ny + self.ny_e)
        check(lib().bnmpc_set_yref_all(self._h, ptr, on_dev))
        self._keep_y = keep

    def set_ref_table(self, table):
        """Bind the whole reference trajectory once (bnmpc_set_ref_table): [rows, cols] shared by all drones or [batch, rows,
        cols] one per drone, row r = [xref_r (nx) | uref_r (nu) | ignored] - the gen_circle_traj table (8 columns) of the
        force / jerk models, the [xref | uref] table (14 columns) of the 3-D model.  torch (CUDA or CPU) or numpy; the
        solver keeps its own copy.  None releases the binding.  Select a window with set_yref_row(i)."""
        if table is None:
            check(lib().bnmpc_set_ref_table(self._h, None, 0, 0, 0, 0))
            return
        if isinstance(table, torch.Tensor):
            t = table.detach().to(torch.float64)
        else:
            t = torch.from_numpy(np.asarray(table, dtype=np.float64))
        if t.dim() == 3 and t.shape[0] != self.batch:
            raise ValueError(f'per-drone table: expected {self.batch} tables, got {t.shape[0]}')
        if t.dim() not in (2, 3) or t.shape[-1] < self.nx + self.nu or t.shape[-2] < self.N + 1:
            raise ValueError(f'expected a table [rows >= {self.N + 1}, cols >= {self.nx + self.nu}] or [{self.batch}, rows, cols], '
                             f'got {tuple(t.shape)}')
        if t.is_cuda and t.device != self.device:
            t = t.to(self.device)
        t = t.contiguous()
        if t.is_cuda:
            torch.cuda.current_stream(t.device).synchronize()       # the copy runs on the solver's stream
        rows, cols = int(t.shape[-2]), int(t.shape[-1])
        check(lib().bnmpc_set_ref_table(self._h, C.c_void_p(t.data_ptr()), rows, cols, 1 if t.dim() == 2 else 2, int(t.is_cuda)))

    def set_yref_row(self, i):
        """OCP.set_up_ocp(i, xref, uref) (src/force_model/ocp.py:117-122) on the table of set_ref_table: the solves read
        yref_k = rows i + k of it, no upload.  set_yref_all() switches back to uploaded windows."""
        check(lib().bnmpc_set_yref_row(self._h, int(i)))

    def solve(self):
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record(self._stream)
        check(lib().bnmpc_solve(self._h))
        self.solve_count += 1
        ev1.record(self._stream)
        self._ev = (ev0, ev1)
        st = self.get_stats('status')
        if self.batch == 1:
            return int(st[0]) if not isinstance(st, int) else st
        return st

    def get_status(self):
        return self.get_stats('status')

    def get_stats(self, name):
        if name == 'time_tot':
            ev0, ev1 = self._ev
            ev1.synchronize()
            return ev0.elapsed_time(ev1) * 1e-3
        if name not in STATS:
            raise ValueError(f'unknown statistic {name!r}')
        if self.numpy_io:
            out = np.empty(self.batch, np.int32)
            check(lib().bnmpc_get_stats(self._h, STATS[name], C.c_void_p(out.ctypes.data), 0))
            return out
        out = torch.empty(self.batch, dtype=torch.int32, device=self.device)
        check(lib().bnmpc_get_stats(self._h, STATS[name], C.c_void_p(out.data_ptr()), 1))
        return out

    def print_statistics(self):
        st, si, qi = (np.asarray(torch.as_tensor(self.get_stats(k)).cpu()) for k in ('status', 'sqp_iter', 'qp_iter'))
        print('bnmpc statistics: instances %d | status histogram %s | sqp_iter max %d | qp_iter min/mean/max %d/%.1f/%d' % (
            self.batch, np.bincount(st, minlength=5).tolist(), si.max(), qi.min(), qi.mean(), qi.max()))

    def solve_for_x0(self, x0_bar, fail_on_nonzero_status=True):
        """acados' solve_for_x0 (used by the reference's dev scripts, src/force_model/ocp.py:162-164): embed x0, solve, return
        u0 - one library call (one kernel launch in FP64).  Raises on a non-zero status like acados does, unless
        fail_on_nonzero_status=False (then the statuses are available through get_stats('status'))."""
        keep, ptr, on_dev = self._as_arg(x0_bar, self.nx)
        if on_dev:
            u0 = torch.empty((self.batch, self.nu), dtype=torch.float64, device=self.device)
            st = torch.empty(self.batch, dtype=torch.int32, device=self.device)
            up, sp = C.c_void_p(u0.data_ptr()), C.c_void_p(st.data_ptr())
        else:
            u0 = np.empty((self.batch, self.nu)); st = np.empty(self.batch, np.int32)
            up, sp = C.c_void_p(u0.ctypes.data), C.c_void_p(st.ctypes.data)
        ev0 = torch.cuda.Event(enable_timing=True); ev1 = torch.cuda.Event(enable_timing=True)
        ev0.record(self._stream)
        check(lib().bnmpc_solve_for_x0(self._h, ptr, up, sp, on_dev))
        self.solve_count += 1
        ev1.record(self._stream)
        self._ev = (ev0, ev1)
        self._keep = keep
        if fail_on_nonzero_status:
            bad = bool((st != 0).any())
            if bad:
                raise BnmpcError(f'solver returned status {st}')
        if not on_dev and self.numpy_io:
            return u0[0] if self.batch == 1 else u0
        return u0 if on_dev else torch.from_numpy(u0).to(self.device)

    def solve_for_x0_into(self, x0_host, u0_host, status_host, wait=True):
        """Zero-allocation form for tight loops: pinned host tensors in and out (x0 [B, nx], u0 [B, nu] float64,
        status [B] int32); returns when the results are in host memory.  wait=False (BNMPC_HOST_ASYNC) only enqueues the
        copies and the solve; call synchronize() before reading the outputs - work enqueued in between (e.g. the upload
        of the next step's reference window on another stream) then runs behind this step's x0 upload, not in front."""
        check(lib().bnmpc_solve_for_x0(self._h, C.c_void_p(x0_host.data_ptr()), C.c_void_p(u0_host.data_ptr()),
                                       C.c_void_p(status_host.data_ptr()), 0 if wait else 2))
        self.solve_count += 1

    def solve_for_x0_device(self, x0_dev, u0_dev, status_dev):
        """Same with device tensors: everything stays on the solver's stream, nothing synchronises."""
        check(lib().bnmpc_solve_for_x0(self._h, C.c_void_p(x0_dev.data_ptr()), C.c_void_p(u0_dev.data_ptr()),
                                       C.c_void_p(status_dev.data_ptr()), 1))
        self.solve_count += 1

    def step_into(self, x0_host, eps_host, u0_host, up_host, status_host, xn_host, p_plant_host=None, wait=True):
        """One iteration of the reference's follow_trajectory for all drones in one call (bnmpc_step_for_x0): x0 embedding,
        solve, get(0,'u'), Converter.convert, simulate_next_x with the noise draw - pinned host tensors x0 [B, nx], eps [B]
        (or None) in; u0 [B, nu], u_plant [B, 2], status [B], x_next [B, nx] out (x_next is the next step's x0)."""
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(lib().bnmpc_step_for_x0(self._h, ptr(x0_host), ptr(eps_host), ptr(p_plant_host), ptr(u0_host), ptr(up_host),
                                      ptr(status_host), ptr(xn_host), 0 if wait else 2))
        self.solve_count += 1

    def step_device(self, x0_dev, eps_dev, u0_dev, up_dev, status_dev, xn_dev, p_plant_dev=None):
        """step_into with device tensors: everything is enqueued on the solver's stream, nothing synchronises."""
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(lib().bnmpc_step_for_x0(self._h, ptr(x0_dev), ptr(eps_dev), ptr(p_plant_dev), ptr(u0_dev), ptr(up_dev),
                                      ptr(status_dev), ptr(xn_dev), 1))
        self.solve_count += 1

    def simulate_next_x_into(self, x_host, u_host, eps_host, xn_host, p_plant_host=None, wait=True):
        """OCP.simulate_next_x (src/force_model/ocp.py:106-115, src/jerk_model/ocp.py:106-116) for all drones with the plant
        integrator this OCP was configured with (AcadosSim of create_simulator): pinned host tensors x [B, 4], u [B, substeps,
        2] = (theta, Fd) per sub-step, eps [B] (the noise draw, or None) in, x_next [B, 4] out.  wait=False only enqueues."""
        nsub = int(u_host.shape[1]) if u_host.dim() == 3 else 1
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        check(lib().bnmpc_sim_step(self._h, nsub, ptr(x_host), ptr(u_host), ptr(p_plant_host), ptr(eps_host), ptr(xn_host),
                                   0 if wait else 2))

    def get_cost(self):
        """acados get_cost(): the NLP objective at the current iterate (LINEAR_LS, stage cost scaled by dt)."""
        io, self.numpy_io = self.numpy_io, False
        try:
            W = torch.tensor(list(self.cfg.W)[:self.ny], dtype=torch.float64, device=self.device)
            We = torch.tensor(list(self.cfg.W_e)[:self.ny_e], dtype=torch.float64, device=self.device)
            tot = torch.zeros(self.batch, dtype=torch.float64, device=self.device)
            for k in range(self.N):
                r = torch.cat([self.get(k, 'x'), self.get(k, 'u')], 1) - self.get(k, 'yref')
                tot += 0.5 * self.cfg.dt * (r * r * W).sum(1)
            r = self.get(self.N, 'x') - self.get(self.N, 'yref')
            tot += 0.5 * (r * r * We).sum(1)
        finally:
            self.numpy_io = io
        return float(tot[0]) if self.batch == 1 else tot

    # -- solution sensitivities (acados' eval_solution_sensitivity; models force, jerk and force_dense) --------------------
    def eval_solution_sensitivity(self, stages=None, with_respect_to='initial_state'):
        """d x_k / d x0 and d u_k / d x0 at the solution of the last solve (bnmpc_eval_sens_x0), stages 0 .. stages-1
        (default N + 1): returns (sens_x [batch, stages, nx, nx], sens_u [batch, min(stages, N), nu, nx]) - torch tensors on
        the solver's device, or numpy without the batch dimension when batch == 1, as get() does.  sens_u[:, 0] is the
        feedback gain of u0.  Rows of an instance whose last solve did not succeed are NaN.  Only 'initial_state' is
        supported here; the sensitivities with respect to the stage-wise model parameters p = (mass, g) are
        eval_param_sensitivity (acados' 'p_global' is a different object)."""
        if with_respect_to != 'initial_state':
            raise ValueError(f"with_respect_to={with_respect_to!r}: only 'initial_state' is supported")
        stages = self.N + 1 if stages is None else int(stages)
        if not 1 <= stages <= self.N + 1:
            raise ValueError(f'stages must be within 1 .. {self.N + 1}, got {stages}')
        shapes = ((self.batch, stages, self.nx, self.nx), (self.batch, min(stages, self.N), self.nu, self.nx))
        if self.numpy_io:
            sx, su = np.empty(shapes[0]), np.empty(shapes[1])
            check(lib().bnmpc_eval_sens_x0(self._h, stages, C.c_void_p(sx.ctypes.data), C.c_void_p(su.ctypes.data), 0))
            return (sx[0], su[0]) if self.batch == 1 else (sx, su)
        sx, su = (torch.empty(sh, dtype=torch.float64, device=self.device) for sh in shapes)
        check(lib().bnmpc_eval_sens_x0(self._h, stages, C.c_void_p(sx.data_ptr()), C.c_void_p(su.data_ptr()), 1))
        return sx, su

    def _seed(self, v, shape):
        if v is None:
            return None
        t = v.detach().to(torch.float64) if isinstance(v, torch.Tensor) else torch.from_numpy(np.asarray(v, dtype=np.float64))
        if t.dim() == len(shape) - 1 and self.batch == 1:
            t = t[None]
        if tuple(t.shape) != shape:
            raise ValueError(f'expected seed shape {shape}, got {tuple(v.shape)}')
        return t.to(self.device).contiguous()

    def adjoint_device(self, seed_x=None, seed_u=None):
        """eval_adjoint_solution_sensitivity with device tensors in and out, asynchronous on the solver's stream."""
        return self._adjoint(seed_x, seed_u, False)

    def _adjoint_device_p(self, seed_x=None, seed_u=None):
        """(grad_x0, grad_yref, grad_p) as device tensors from one bnmpc_eval_adjoint_sens_p call, asynchronous on the
        solver's stream (autograd.solve_u0 with p)."""
        return self._adjoint(seed_x, seed_u, True)

    def _adjoint(self, seed_x, seed_u, with_p):
        sx = self._seed(seed_x, (self.batch, self.N + 1, self.nx))
        su = self._seed(seed_u, (self.batch, self.N, self.nu))
        if sx is None and su is None:
            raise ValueError('seed_x and seed_u are both None')
        gx = torch.empty((self.batch, self.nx), dtype=torch.float64, device=self.device)
        gy = torch.empty((self.batch, self.N * self.ny + self.ny_e), dtype=torch.float64, device=self.device)
        ptr = lambda t: C.c_void_p(t.data_ptr()) if t is not None else None
        self._keep = (sx, su)
        if not with_p:
            check(lib().bnmpc_eval_adjoint_sens(self._h, ptr(sx), ptr(su), ptr(gx), ptr(gy), 1))
            return gx, gy
        gp = torch.empty((self.batch, self.np_), dtype=torch.float64, device=self.device)
        check(lib().bnmpc_eval_adjoint_sens_p(self._h, ptr(sx), ptr(su), ptr(gx), ptr(gy), ptr(gp), 1))
        return gx, gy, gp

    def eval_adjoint_solution_sensitivity(self, seed_x=None, seed_u=None):
        """Adjoint of eval_solution_sensitivity (bnmpc_eval_adjoint_sens): seed_x [batch, N+1, nx], seed_u [batch, N, nu]
        (None = 0, not both) -> (grad_x0 [batch, nx], grad_yref [batch, N*ny + ny_e]) = sum over the stages of the
        sensitivities' transposes times the seeds, with respect to x0 and to the set_yref_all window.  One linear solve per
        drone whatever the seed.  Output types as for eval_solution_sensitivity."""
        gx, gy = self.adjoint_device(seed_x, seed_u)
        if self.numpy_io:
            gx, gy = gx.cpu().numpy(), gy.cpu().numpy()
            return (gx[0], gy[0]) if self.batch == 1 else (gx, gy)
        return gx, gy

    # -- sensitivities with respect to the model parameters p = (mass, g) (set(0, 'p', ..); models force, jerk, force_dense) --
    def eval_param_sensitivity(self, stages=None):
        """d x_k / d p and d u_k / d p at the solution of the last solve (bnmpc_eval_sens_p), p = (mass, g) of each drone's
        controller model, stages 0 .. stages-1 (default N + 1): returns (sens_x [batch, stages, nx, np],
        sens_u [batch, min(stages, N), nu, np]) with the conventions of eval_solution_sensitivity.  sens_x[:, 0] = 0 (x_0 is
        fixed by x0); sens_u[:, 0, :, 0] is how u0 changes per unit of mass estimate."""
        stages = self.N + 1 if stages is None else int(stages)
        if not 1 <= stages <= self.N + 1:
            raise ValueError(f'stages must be within 1 .. {self.N + 1}, got {stages}')
        shapes = ((self.batch, stages, self.nx, self.np_), (self.batch, min(stages, self.N), self.nu, self.np_))
        if self.numpy_io:
            sx, su = np.empty(shapes[0]), np.empty(shapes[1])
            check(lib().bnmpc_eval_sens_p(self._h, stages, C.c_void_p(sx.ctypes.data), C.c_void_p(su.ctypes.data), 0))
            return (sx[0], su[0]) if self.batch == 1 else (sx, su)
        sx, su = (torch.empty(sh, dtype=torch.float64, device=self.device) for sh in shapes)
        check(lib().bnmpc_eval_sens_p(self._h, stages, C.c_void_p(sx.data_ptr()), C.c_void_p(su.data_ptr()), 1))
        return sx, su

    def eval_adjoint_param_sensitivity(self, seed_x=None, seed_u=None):
        """Adjoint of eval_param_sensitivity (bnmpc_eval_adjoint_sens_p): seed_x [batch, N+1, nx], seed_u [batch, N, nu]
        (None = 0, not both) -> grad_p [batch, np] = sum over the stages of the sensitivities' transposes times the seeds.
        One linear solve per drone whatever the seed.  Output types as for eval_solution_sensitivity."""
        _, _, gp = self._adjoint(seed_x, seed_u, True)
        if self.numpy_io:
            gp = gp.cpu().numpy()
            return gp[0] if self.batch == 1 else gp
        return gp

    def reset(self):
        check(lib().bnmpc_reset(self._h))
        self.solve_count += 1

    def synchronize(self):
        check(lib().bnmpc_synchronize(self._h))

    def launch_count(self):
        return int(lib().bnmpc_launch_count(self._h))

    def workspace_bytes(self):
        return int(lib().bnmpc_workspace_bytes(self._h))


class BatchedAcadosSimSolver:
    """`AcadosSimSolver` of the plant model (reference src/plant.py, create_simulator src/force_model/ocp.py:98-104 /
    src/jerk_model/ocp.py:97-104): set('x'|'u'|'p', v), solve(), get('x'), simulate(x=, u=).  One solve() is one ERK step
    of length T with `num_stages` stages."""

    def __init__(self, T, num_stages=4, batch=1, device=0, numpy_io=None, model='plant'):
        """model 'plant': the planar plant of src/plant.py (x [4], u = (theta, Fd)); 'att': the 3-D attitude model as its own
        plant (x [10], u = (T, wx, wy, wz))."""
        self.device = _require_cuda(device)
        self.batch = int(batch)
        self.numpy_io = (self.batch == 1) if numpy_io is None else bool(numpy_io)
        self.nx, self.nu = (10, 4) if model == 'att' else (4, 2)
        cfg = default_config('att' if model == 'att' else 'force', horizon=1, sim_erk_stages=int(num_stages), sim_substeps=1, sim_dt=float(T))
        self._h = C.c_void_p()
        check(lib().bnmpc_create(C.byref(cfg), self.batch, self.device.index, C.byref(self._h)))
        with torch.cuda.device(self.device):
            self._stream = torch.cuda.current_stream()
        check(lib().bnmpc_set_stream(self._h, C.c_void_p(self._stream.cuda_stream)))
        self._x = torch.zeros((self.batch, self.nx), dtype=torch.float64, device=self.device)
        self._u = torch.zeros((self.batch, self.nu), dtype=torch.float64, device=self.device)
        self._p = None
        self._xn = torch.zeros((self.batch, self.nx), dtype=torch.float64, device=self.device)

    def __del__(self):
        h, self._h = getattr(self, '_h', None), None
        if h:
            try:
                lib().bnmpc_destroy(h)
            except Exception:
                pass

    def _t(self, v, dim):
        t = torch.as_tensor(np.asarray(v) if not isinstance(v, torch.Tensor) else v, dtype=torch.float64)
        if t.dim() == 1 and self.batch == 1:
            t = t[None]
        if tuple(t.shape) != (self.batch, dim):
            raise ValueError(f'expected shape ({self.batch}, {dim}), got {tuple(t.shape)}')
        return t.to(self.device).contiguous()

    def set(self, field, value):
        if field == 'x':
            self._x = self._t(value, self.nx)
        elif field == 'u':
            self._u = self._t(value, self.nu)
        elif field == 'p':
            self._p = self._t(value, 2)
        else:
            raise ValueError(f'unknown field {field!r}')

    def solve(self):
        pp = C.c_void_p(self._p.data_ptr()) if self._p is not None else None
        check(lib().bnmpc_sim_step(self._h, 1, C.c_void_p(self._x.data_ptr()), C.c_void_p(self._u.data_ptr()), pp, None,
                                   C.c_void_p(self._xn.data_ptr()), 1))
        return 0

    def get(self, field):
        if field != 'x':
            raise ValueError(f'unknown field {field!r}')
        if self.numpy_io:
            a = self._xn.cpu().numpy()
            return a[0].copy() if self.batch == 1 else a
        return self._xn.clone()

    def simulate(self, x=None, u=None, p=None):
        if x is not None:
            self.set('x', x)
        if u is not None:
            self.set('u', u)
        if p is not None:
            self.set('p', p)
        self.solve()
        return self.get('x')
