"""A fleet of drones stepped as a software pipeline of sub-fleets.

One control step of `BatchedAcadosOcpSolver` for B drones ends when its LONGEST solve ends: interior-point iteration counts
differ 4x between drones, so at 4096 drones a fifth of the warp time of a per-step launch is spent waiting for the last few
(DESIGN.md 5, "queue tail").  The drones are independent - each one's next step depends only on its own previous step, as in the
reference's follow_trajectory (src/force_model/controller.py:25-54, one drone per loop) - so nothing requires the whole fleet to
finish step i before any drone starts step i+1.  `SolverFleet` splits the batch into G solver objects, each on its own CUDA
stream, and steps them round-robin: sub-fleet g is synchronised (its results of step i are in host memory, the `on_results`
hook sees them) only right before ITS step i+1 is enqueued, while the kernels of the other sub-fleets keep the SMs busy.  The
tail of one sub-fleet's launch overlaps the bulk of the next one's, the uploads of one overlap the solves of another, and every
drone still sees exactly the reference's sequence  set_up_ocp -> x0 embedding -> solve -> get(0,'u') -> Converter ->
simulate_next_x  per step.  Results are identical to one solver object for the whole batch (instances are independent).
"""
import torch

from .acados_shim import BatchedAcadosOcpSolver


def group_bounds(batch, groups):
    """[lo_0, lo_1, ..., batch]: contiguous slices of near-equal size (the first batch % groups slices get one more)."""
    batch, groups = int(batch), int(groups)
    if batch < 1 or groups < 1:
        raise ValueError('batch and groups must be positive')
    groups = min(groups, batch)
    q, r = divmod(batch, groups)
    out = [0]
    for g in range(groups):
        out.append(out[-1] + q + (1 if g < r else 0))
    return out


class SolverFleet:
    """G `BatchedAcadosOcpSolver`s over contiguous slices of `batch` drones, each on its own stream (see the module docstring).

    All buffers handed to `step` are PINNED host tensors covering the whole batch; sub-fleet g reads and writes rows
    lo_g:hi_g of them.  `x_next` of one step is meant to be passed as `x0` of the next (double-buffer it): the copies of a
    sub-fleet are ordered on its stream, so its next step may be enqueued before the host has looked at anything."""

    def __init__(self, model='force', batch=1, groups=4, device=0, solver_factory=None, **solver_kw):
        """solver_factory(batch) -> solver object (default: a BatchedAcadosOcpSolver of `model` on a CUDA stream of its own);
        anything with set_yref_all / step_into / synchronize / reset works, plus set_ref_table / set_yref_row for step_at (the CPU
        tests drive the pipeline with a recorder)."""
        self.bounds = group_bounds(batch, groups)
        self.groups = len(self.bounds) - 1
        self.batch = int(batch)
        self.solvers, self.streams = [], []
        for g in range(self.groups):
            b = self.bounds[g + 1] - self.bounds[g]
            if solver_factory is not None:
                self.solvers.append(solver_factory(b))
                continue
            dev = torch.device('cuda', device) if not isinstance(device, torch.device) else device
            st = torch.cuda.Stream(device=dev)
            with torch.cuda.stream(st):                     # the solver binds the current stream when it is created
                s = BatchedAcadosOcpSolver(model, batch=b, device=device, numpy_io=False, **solver_kw)
            self.solvers.append(s)
            self.streams.append(st)
        s0 = self.solvers[0]
        self.nx, self.nu, self.ny, self.ny_e, self.N = s0.nx, s0.nu, s0.ny, s0.ny_e, s0.N
        self.cfg = getattr(s0, 'cfg', None)
        self._pending = [False] * self.groups

    def slices(self):
        return [(self.bounds[g], self.bounds[g + 1]) for g in range(self.groups)]

    def reset(self):
        self.synchronize()
        for s in self.solvers:
            s.reset()

    def step(self, yref, x0, eps, u0, u_plant, status, x_next, p_plant=None, on_results=None):
        """One control step of every drone (OCP.set_up_ocp + one iteration of follow_trajectory, bnmpc_set_yref_all +
        bnmpc_step_for_x0 per sub-fleet).  yref [B, N*ny + ny_e], x0 [B, nx], eps [B] or None, p_plant [B, 2] or None in;
        u0 [B, nu], u_plant [B, 2], status [B] int32, x_next [B, nx] out.  Returns with the step ENQUEUED: rows lo_g:hi_g of the
        outputs are valid after `wait(g)` / `synchronize()` - or inside `on_results(g, lo, hi)`, which the next call of `step`
        invokes for each sub-fleet once its previous step is back on the host and before its next one is enqueued (the place
        of the reference's status check and logging, src/force_model/controller.py:33-41)."""
        self._step(lambda s, lo, hi: s.set_yref_all(yref[lo:hi]), x0, eps, u0, u_plant, status, x_next, p_plant, on_results)

    def set_ref_table(self, table):
        """Bind the reference trajectory to every sub-fleet once (BatchedAcadosOcpSolver.set_ref_table): a shared table
        [rows, cols] goes to all of them, a per-drone table [B, rows, cols] gives sub-fleet g its rows lo_g:hi_g."""
        per_drone = table.ndim == 3
        if per_drone and table.shape[0] != self.batch:
            raise ValueError(f'per-drone table: expected {self.batch} tables, got {table.shape[0]}')
        for g, s in enumerate(self.solvers):
            lo, hi = self.bounds[g], self.bounds[g + 1]
            s.set_ref_table(table[lo:hi] if per_drone else table)

    def step_at(self, i, x0, eps, u0, u_plant, status, x_next, p_plant=None, on_results=None):
        """`step` with the reference window taken from the table of set_ref_table at row i (OCP.set_up_ocp(i, xref, uref),
        bnmpc_set_yref_row + bnmpc_step_for_x0 per sub-fleet): no reference upload.  Same buffers, pipeline and hook."""
        self._step(lambda s, lo, hi: s.set_yref_row(i), x0, eps, u0, u_plant, status, x_next, p_plant, on_results)

    def _step(self, set_ref, x0, eps, u0, u_plant, status, x_next, p_plant, on_results):
        for g, s in enumerate(self.solvers):
            lo, hi = self.bounds[g], self.bounds[g + 1]
            if self._pending[g]:
                s.synchronize()
                self._pending[g] = False
                if on_results is not None:
                    on_results(g, lo, hi)
            set_ref(s, lo, hi)
            s.step_into(x0[lo:hi], None if eps is None else eps[lo:hi], u0[lo:hi], u_plant[lo:hi], status[lo:hi], x_next[lo:hi],
                        p_plant_host=None if p_plant is None else p_plant[lo:hi], wait=False)
            self._pending[g] = True

    def wait(self, g):
        if self._pending[g]:
            self.solvers[g].synchronize()
            self._pending[g] = False

    def synchronize(self, on_results=None):
        for g in range(self.groups):
            was = self._pending[g]
            self.wait(g)
            if was and on_results is not None:
                on_results(g, self.bounds[g], self.bounds[g + 1])

    def launch_count(self):
        return sum(s.launch_count() for s in self.solvers)
