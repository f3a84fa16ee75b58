"""The reference trajectory bound to a solver once (bnmpc_set_ref_table) and the yref window selected by row
(bnmpc_set_yref_row) - OCP.set_up_ocp(iter, xref, uref) of the reference (src/force_model/ocp.py:117-122) without a window
upload per control step.  The solves read the window straight from the table; everything they compute must be bit for bit
what the same calls compute after bnmpc_set_yref_all of that window, in both precisions, for every model, for shared and
per-drone tables, and through every solve entry point."""
import ctypes as C

import numpy as np
import pytest
import torch

from common import random_loop_inputs, thrust_refs
from oracle import c_oracle as co

E_ARG = -1
MODEL_ID = {'force': 0, 'jerk': 1}


def _window(tab, i, N, nx, ny):
    """bnmpc_set_yref_all's [B, N*ny + nx] from per-drone tables [B, rows, cols]"""
    B = tab.shape[0]
    return np.ascontiguousarray(np.concatenate([tab[:, i:i + N, :ny].reshape(B, N * ny), tab[:, i + N, :nx]], 1))


def _inputs(model, B, S, seed):
    """per-drone tables [B, rows, cols], plant start states, noise [S, B], plant parameters [B, 2]"""
    if model == 'att':
        from test_att import att_inputs
        refs, x0, _, pp = att_inputs(B, seed, rows=S + 40)
        return refs, x0, np.random.default_rng(seed).normal(0, 0.002, (S, B)), pp
    refs, x0, noise, _, pp = random_loop_inputs(B, S, seed, mass_sigma=0.05)
    return (thrust_refs(refs) if model == 'thrust' else refs), x0, noise, pp


def _full(tab, B):
    return tab if tab.ndim == 3 else np.broadcast_to(tab, (B,) + tab.shape)


def _solver(model, B, precision='fp64'):
    import drone_attitude_control_b200 as pkg
    s = pkg.BatchedAcadosOcpSolver(model, batch=B, device=0, precision=precision, numpy_io=False)
    if model == 'att':             # start iterate of follow_trajectory_batched: level attitude, hover thrust
        xg = torch.zeros((B, 10), dtype=torch.float64, device='cuda'); xg[:, 6] = 1.0
        ug = torch.zeros((B, 4), dtype=torch.float64, device='cuda'); ug[:, 0] = 0.03277 * 9.81
        for k in range(s.N + 1):
            s.set(k, 'x', xg)
        for k in range(s.N):
            s.set(k, 'u', ug)
    return s


def _x0_full(x0, nx):
    if nx == 6:                    # jerk model: plant state + the carried acceleration a_i = (0, g)
        return np.hstack([x0, np.tile([0.0, 9.81], (x0.shape[0], 1))])
    return x0


def _closed_loop(model, tab, x0, noise, pp, S, precision, use_table):
    """S control steps of step_into with the window uploaded (set_yref_all) or selected in the bound table (set_yref_row)"""
    B = x0.shape[0]
    s = _solver(model, B, precision)
    nx, nu, N, ny = s.nx, s.nu, s.N, s.ny
    full = _full(tab, B)
    pin = lambda *sh, dt=torch.float64: torch.zeros(sh, dtype=dt).pin_memory()
    xa, xb, u0, up, st = pin(B, nx), pin(B, nx), pin(B, nu), pin(B, 2), pin(B, dt=torch.int32)
    xa.copy_(torch.tensor(_x0_full(x0, nx)))
    ppt = torch.tensor(pp).pin_memory()
    if use_table:
        s.set_ref_table(tab)
    out = []
    for i in range(S):
        if use_table:
            s.set_yref_row(i)
        else:
            s.set_yref_all(torch.tensor(_window(full, i, N, nx, ny)))
        s.step_into(xa, torch.tensor(noise[i]).pin_memory(), u0, up, st, xb, p_plant_host=ppt)
        out.append(dict(u0=u0.numpy().copy(), u_plant=up.numpy().copy(), status=st.numpy().copy(), x_next=xb.numpy().copy(),
                        sqp_iter=s.get_stats('sqp_iter').cpu().numpy(), qp_iter=s.get_stats('qp_iter').cpu().numpy()))
        xa, xb = xb, xa
    return out


def _assert_same_loop(a, b):
    for i, (ra, rb) in enumerate(zip(a, b)):
        for k in ra:
            assert np.array_equal(ra[k], rb[k]), (i, k)


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize('layout', ['shared', 'per_drone'])
@pytest.mark.parametrize('precision', ['fp64', 'fp32'])
@pytest.mark.parametrize('model', ['force', 'jerk', 'att'])
def test_closed_loop_on_the_table_is_bit_identical_to_uploaded_windows(model, precision, layout):
    B, S = 96, 10
    refs, x0, noise, pp = _inputs(model, B, S, seed=301 + len(model))
    tab = np.ascontiguousarray(refs[0] if layout == 'shared' else refs)
    if layout == 'shared':         # every drone starts at its offset from the start of the one shared trajectory
        nxp = x0.shape[1]
        x0 = refs[0, 0, :nxp] + (x0 - refs[:, 0, :nxp])
    up = _closed_loop(model, tab, x0, noise, pp, S, precision, use_table=False)
    tb = _closed_loop(model, tab, x0, noise, pp, S, precision, use_table=True)
    _assert_same_loop(up, tb)
    st = np.stack([r['status'] for r in up])
    assert (st == 0).mean() > 0.9 and np.stack([r['qp_iter'] for r in up]).max() > 0


@pytest.mark.gpu
def test_closed_loop_on_the_table_at_full_size():
    B, S = 4096, 20
    refs, x0, noise, pp = _inputs('force', B, S, seed=307)
    up = _closed_loop('force', refs, x0, noise, pp, S, 'fp64', use_table=False)
    tb = _closed_loop('force', torch.tensor(refs, device='cuda'), x0, noise, pp, S, 'fp64', use_table=True)
    _assert_same_loop(up, tb)
    assert (np.stack([r['status'] for r in up]) == 0).mean() > 0.99


def _collect(s):
    N = s.N
    return dict(status=s.get_stats('status').cpu().numpy(), sqp_iter=s.get_stats('sqp_iter').cpu().numpy(),
                qp_iter=s.get_stats('qp_iter').cpu().numpy(),
                x=np.stack([s.get(k, 'x').cpu().numpy() for k in range(N + 1)], 1),
                u=np.stack([s.get(k, 'u').cpu().numpy() for k in range(N)], 1),
                pi=np.stack([s.get(k, 'pi').cpu().numpy() for k in range(N)], 1))


def _assert_same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp64', 'fp32'])
@pytest.mark.parametrize('model', ['force', 'jerk', 'force_dense', 'thrust', 'att'])
def test_every_solve_entry_point_reads_the_window(model, precision):
    """bnmpc_solve and bnmpc_solve_for_x0 after set_yref_row equal the same calls after set_yref_all of the window - also on a
    handle with per-stage bounds (the second instantiation of the solve kernel)"""
    B, row = 64, 11
    refs, x0, _, _ = _inputs(model, B, 2, seed=311)

    def run(use_table, stage_bounds):
        s = _solver(model, B, precision)
        x0f = _x0_full(x0, s.nx)
        if stage_bounds:
            s.set(3, 'ubu', s.get(3, 'ubu') * 0.9)
        if use_table:
            s.set_ref_table(refs)
            s.set_yref_row(row)
        else:
            s.set_yref_all(_window(refs, row, s.N, s.nx, s.ny))
        s.set(0, 'lbx', x0f); s.set(0, 'ubx', x0f)
        s.solve()
        r = {'solve_' + k: v for k, v in _collect(s).items()}
        u0 = s.solve_for_x0(torch.tensor(x0f + 0.01, device='cuda'), fail_on_nonzero_status=False)
        r.update({'x0_' + k: v for k, v in _collect(s).items()})
        r['u0'] = u0.cpu().numpy()
        return r

    for sb in (False, True):
        a, b = run(False, sb), run(True, sb)
        _assert_same(a, b)
        assert a['solve_qp_iter'].max() > 0


@pytest.mark.gpu
@pytest.mark.parametrize('precision', ['fp64', 'fp32'])
def test_switching_the_yref_source(precision):
    B, row, N = 40, 17, 30
    refs, x0, _, _ = _inputs('force', B, 2, seed=321)
    other = refs[::-1].copy()
    cast = (lambda a: a) if precision == 'fp64' else (lambda a: a.astype(np.float32).astype(np.float64))

    def fresh():
        s = _solver('force', B, precision)
        s.set(0, 'lbx', x0); s.set(0, 'ubx', x0)
        return s

    def solve(s):
        s.solve()
        return _collect(s)

    # get(k, 'yref') reads the table's rows row + k (the x-part at k = N) and changes nothing
    s = fresh(); s.set_ref_table(refs); s.set_yref_row(row)
    for k in (0, 1, 13, N - 1):
        assert np.array_equal(s.get(k, 'yref').cpu().numpy(), cast(refs[:, row + k, :6]))
    assert np.array_equal(s.get(N, 'yref').cpu().numpy(), cast(refs[:, row + N, :4]))
    first = solve(s)
    launches = s.launch_count()
    s.get(5, 'yref'); s.get(N, 'yref')
    assert s.launch_count() == launches + 2                 # one read kernel per get, no gather into the stored yref
    second = solve(s)
    s2 = fresh(); s2.set_ref_table(refs); s2.set_yref_row(row)
    _assert_same(first, solve(s2)); _assert_same(second, solve(s2))
    # set(k, 'yref', v) on the selected table == set_yref_all(window) + set(k, 'yref', v)
    v = refs[:, 3, :6] + 0.05
    s = fresh(); s.set_ref_table(refs); s.set_yref_row(row); s.set(4, 'yref', v)
    s2 = fresh(); s2.set_yref_all(_window(refs, row, N, 4, 6)); s2.set(4, 'yref', v)
    for k in (0, 4, 5, N):
        assert np.array_equal(s.get(k, 'yref').cpu().numpy(), s2.get(k, 'yref').cpu().numpy())
    _assert_same(solve(s), solve(s2))
    # set_yref_all after set_yref_row: the uploaded window is the source again
    s = fresh(); s.set_ref_table(refs); s.set_yref_row(row); s.set_yref_all(_window(refs, row + 40, N, 4, 6))
    s2 = fresh(); s2.set_yref_all(_window(refs, row + 40, N, 4, 6))
    _assert_same(solve(s), solve(s2))
    # releasing or re-binding the selected table keeps the window of the next solve; a new row selects in the new table
    s2 = fresh(); s2.set_yref_all(_window(refs, row, N, 4, 6))
    want = solve(s2)
    s = fresh(); s.set_ref_table(refs); s.set_yref_row(row); s.set_ref_table(None)
    _assert_same(solve(s), want)
    s = fresh(); s.set_ref_table(refs); s.set_yref_row(row); s.set_ref_table(other)
    _assert_same(solve(s), want)
    s.reset(); s.set_yref_row(row)
    s2 = fresh(); s2.set_yref_all(_window(other, row, N, 4, 6))
    _assert_same(solve(s), solve(s2))


@pytest.mark.gpu
def test_errors_leave_the_handle_usable():
    import drone_attitude_control_b200 as pkg
    L = pkg.lib()
    B, N = 8, 30
    refs, x0, _, _ = _inputs('force', B, 2, seed=331)
    s = _solver('force', B)
    h = s.handle
    p = C.c_void_p(np.ascontiguousarray(refs).ctypes.data)
    rows = refs.shape[1]
    assert L.bnmpc_set_yref_row(h, 0) == E_ARG and b'no reference table' in L.bnmpc_last_error()
    assert L.bnmpc_set_ref_table(h, p, rows, 8, 3, 0) == E_ARG and b'layout' in L.bnmpc_last_error()
    assert L.bnmpc_set_ref_table(h, p, rows, 5, 2, 0) == E_ARG and b'cols' in L.bnmpc_last_error()
    assert L.bnmpc_set_ref_table(h, p, N, 8, 2, 0) == E_ARG and b'rows' in L.bnmpc_last_error()
    ws = s.workspace_bytes()
    tab = np.ascontiguousarray(refs[:, :N + 5])
    assert L.bnmpc_set_ref_table(h, C.c_void_p(tab.ctypes.data), N + 5, 8, 2, 0) == 0
    assert s.workspace_bytes() == ws + tab.nbytes
    assert L.bnmpc_set_yref_row(h, -1) == E_ARG and b'row out of range' in L.bnmpc_last_error()
    assert L.bnmpc_set_yref_row(h, 5) == E_ARG
    assert L.bnmpc_set_yref_row(h, 4) == 0
    with pytest.raises(ValueError):
        s.set_ref_table(refs[:B - 1])                       # one table per drone
    with pytest.raises(ValueError):
        s.set_ref_table(refs[0, :, :5])                     # cols < nx + nu
    with pytest.raises(ValueError):
        s.set_ref_table(refs[0, :N])                        # rows < N + 1
    with pytest.raises(ValueError):
        s.set_ref_table(refs[0, 0])
    s.set(0, 'lbx', x0); s.set(0, 'ubx', x0)
    s.solve()
    got = _collect(s)
    s2 = _solver('force', B)
    s2.set_yref_all(_window(tab, 4, N, 4, 6)); s2.set(0, 'lbx', x0); s2.set(0, 'ubx', x0)
    s2.solve()
    _assert_same(got, _collect(s2))
    assert (got['status'] == 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize('model,groups', [('force', 3), ('jerk', 4)])
def test_solver_fleet_step_at(model, groups):
    """SolverFleet.step_at: the same closed loop as the oracle and, bit for bit, as SolverFleet.step with uploaded windows;
    the hook sees every (sub-fleet, step) once"""
    import drone_attitude_control_b200 as pkg
    B, S = 50, 8
    om = MODEL_ID[model]
    refs, x0, noise, pc, pp = random_loop_inputs(B, S, seed=71 + om, mass_sigma=0.05)
    want = co.closed_loop(co.default_opts(om), refs, x0, noise, pc, pp, S)
    pin = lambda *sh, dt=torch.float64: torch.zeros(sh, dtype=dt).pin_memory()
    ppt = torch.tensor(pp).pin_memory()
    eps = torch.tensor(noise).pin_memory()

    def run(use_table):
        fleet = pkg.SolverFleet(model, batch=B, groups=groups, device=0)
        nx, nu, N, ny = fleet.nx, fleet.nu, fleet.N, fleet.ny
        xb, u0, up, st = [pin(B, nx), pin(B, nx)], pin(B, nu), pin(B, 2), pin(B, dt=torch.int32)
        xb[0].copy_(torch.tensor(_x0_full(x0, nx)))
        seen, step_of = [], [0] * groups

        def on_results(g, lo, hi):
            i = step_of[g]
            step_of[g] += 1
            seen.append((i, lo, hi, st[lo:hi].numpy().copy(), u0[lo:hi].numpy().copy(), up[lo:hi].numpy().copy(),
                         xb[(i + 1) % 2][lo:hi].numpy().copy()))

        if use_table:
            fleet.set_ref_table(refs)
        for i in range(S):
            if use_table:
                fleet.step_at(i, xb[i % 2], eps[i], u0, up, st, xb[(i + 1) % 2], p_plant=ppt, on_results=on_results)
            else:
                y = torch.tensor(_window(refs, i, N, nx, ny)).pin_memory()
                fleet.step(y, xb[i % 2], eps[i], u0, up, st, xb[(i + 1) % 2], p_plant=ppt, on_results=on_results)
        fleet.synchronize(on_results=on_results)
        assert step_of == [S] * groups
        assert sorted((i, lo) for i, lo, *_ in seen) == sorted((i, lo) for i in range(S) for lo, _ in fleet.slices())
        return sorted(seen, key=lambda e: (e[0], e[1]))

    got = run(True)
    for i, lo, hi, st, u, _, x in got:
        assert np.array_equal(st, want['status'][lo:hi, i])
        np.testing.assert_allclose(u, want['U_ctrl'][lo:hi, i], rtol=0, atol=1e-9)
        np.testing.assert_allclose(x[:, :4], want['Xsim'][lo:hi, i + 1], rtol=0, atol=1e-9)
    for a, b in zip(got, run(False)):
        assert a[:3] == b[:3]
        for va, vb in zip(a[3:], b[3:]):
            assert np.array_equal(va, vb)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
def test_fleet_step_at_order_on_cpu():
    """SolverFleet.step_at with recording stand-ins: the table reaches each sub-fleet once (its own rows of a per-drone table,
    the whole of a shared one), every step is set_yref_row(i) followed by the sub-fleet's step, and the synchronisation
    order is the one of SolverFleet.step"""
    from drone_attitude_control_b200.fleet import SolverFleet
    log = []

    class Rec:
        nx, nu, ny, ny_e, N = 4, 2, 6, 4, 30

        def __init__(self, b):
            self.b, self.id = b, len(made)
            made.append(self)

        def set_ref_table(self, t):
            log.append(('table', self.id, tuple(t.shape), float(t[0, 0, 0]) if t.ndim == 3 else None))

        def set_yref_row(self, i):
            log.append(('row', self.id, i))

        def step_into(self, x0, eps, u0, up, st, xn, p_plant_host=None, wait=True):
            assert not wait and x0.shape[0] == self.b and xn.shape[0] == self.b and (eps is None or eps.shape[0] == self.b)
            log.append(('step', self.id, float(x0[0, 0])))
            xn.copy_(x0 + 1.0)
            st.fill_(self.id)

        def synchronize(self):
            log.append(('sync', self.id))

        def reset(self):
            log.append(('reset', self.id))

    made = []
    B, G, S = 10, 3, 4
    fleet = SolverFleet(batch=B, groups=G, solver_factory=Rec)
    table = torch.arange(B, dtype=torch.float64)[:, None, None].expand(B, 40, 8).contiguous()
    fleet.set_ref_table(table)
    assert [e for e in log] == [('table', 0, (4, 40, 8), 0.0), ('table', 1, (3, 40, 8), 4.0), ('table', 2, (3, 40, 8), 7.0)]
    fleet.set_ref_table(table[0])
    assert [e[:3] for e in log[3:]] == [('table', g, (40, 8)) for g in range(G)]
    with pytest.raises(ValueError):
        fleet.set_ref_table(table[:B - 1])
    del log[:]
    xb = [torch.zeros(B, 4, dtype=torch.float64), torch.zeros(B, 4, dtype=torch.float64)]
    xb[0][:, 0] = torch.arange(B, dtype=torch.float64) * 100
    u0, up, st = torch.zeros(B, 2), torch.zeros(B, 2), torch.zeros(B, dtype=torch.int32)
    seen = []
    for i in range(S):
        fleet.step_at(i, xb[i % 2], None, u0, up, st, xb[(i + 1) % 2],
                      on_results=lambda g, lo, hi: seen.append((g, lo, hi, len([e for e in log if e[0] == 'step' and e[1] == g]))))
    fleet.synchronize(on_results=lambda g, lo, hi: seen.append((g, lo, hi, S)))
    for g in range(G):
        mine = [e for e in log if e[1] == g]
        assert [e[0] for e in mine] == ['row', 'step'] + ['sync', 'row', 'step'] * (S - 1) + ['sync']
        assert [e[2] for e in mine if e[0] == 'row'] == list(range(S))
    order = [(e[0], e[1]) for e in log if e[0] in ('sync', 'step')]
    assert order[:G] == [('step', 0), ('step', 1), ('step', 2)] and order[G:G + 4] == [('sync', 0), ('step', 0), ('sync', 1), ('step', 1)]
    assert sorted(seen) == sorted((g, lo, hi, k) for g, (lo, hi) in enumerate(fleet.slices()) for k in range(1, S + 1))
    assert torch.equal(xb[S % 2][:, 0], torch.arange(B, dtype=torch.float64) * 100 + S)
    assert st.tolist() == [0] * 4 + [1] * 3 + [2] * 3
