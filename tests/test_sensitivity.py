"""Solution sensitivities of the batched solve (bnmpc_eval_sens_x0 / bnmpc_eval_adjoint_sens, the shim's
eval_solution_sensitivity / eval_adjoint_solution_sensitivity, autograd.solve_u0).  There is no acados here, so parity
with acados' eval_solution_sensitivity is unpinned; the pins are central finite differences of solves and the dense-KKT
restatement of tests/sens_oracle.py at the stored solution of an oracle.nmpc_oracle.OracleOcpSolver, which the product
templates (host build: tests/hostsim_sens, and the device) must match at identical stored iterates."""
import ctypes as C

import numpy as np
import pytest
import torch

import hostsim as hs
import hostsim_sens as hss
import sens_oracle as so
from common import random_solve_inputs
from oracle import c_oracle as co
from oracle import nmpc_oracle as o

E_ARG, E_UNSUPPORTED = -1, -5
SPECS = {'force': o.force_ocp, 'jerk': o.jerk_ocp, 'force_dense': o.force_ocp}
HSS_MODEL = {'force': hss.MODEL_FORCE, 'jerk': hss.MODEL_JERK, 'force_dense': hss.MODEL_FORCE_DENSE}


def _rel(a, b):
    return float(np.abs(np.asarray(a) - np.asarray(b)).max() / max(np.abs(np.asarray(b)).max(), 1e-300))


def _oracle_solve(spec, x0, yref, bnd=None):
    s = o.OracleOcpSolver(spec)
    ny = spec.nx + spec.nu
    for k in range(spec.N):
        s.set(k, 'yref', yref[k * ny:(k + 1) * ny])
    s.set(spec.N, 'yref', yref[spec.N * ny:])
    s.set(0, 'lbx', x0)
    if bnd is not None:
        _set_oracle_bounds(s, bnd)
    s.solve()
    return s


def _set_oracle_bounds(s, bnd):
    """per-stage bounds [N, 2, nu + nx] (the solver's layout) -> the oracle's per-stage boxes"""
    nu = s.spec.nu
    s.lbu_k[:], s.ubu_k[:] = bnd[:, 0, :nu], bnd[:, 1, :nu]
    s.lbx_k[1:], s.ubx_k[1:] = bnd[1:, 0, nu:], bnd[1:, 1, nu:]


def _margin(s):
    """smallest distance of the solution to a bound"""
    N = s.spec.N
    return min((s.u - s.lbu_k).min(), (s.ubu_k - s.u).min(), (s.x[1:N] - s.lbx_k[1:]).min(), (s.ubx_k[1:] - s.x[1:N]).min())


def _interior(model, n, seed, B=16, margin=0.02):
    """instances whose solutions keep every bound inactive by more than `margin` (then the barrier terms lam / t of the KKT
    matrix are far below the cost Hessian and the sensitivity is the derivative of the QP solution)"""
    spec = SPECS[model](tol=1e-10)
    x0, yref = random_solve_inputs(model, B, seed, spread=0.01)
    out = []
    for i in range(B):
        s = _oracle_solve(spec, x0[i], yref[i])
        if s.status == 0 and _margin(s) > margin:
            out.append((x0[i], yref[i], s))
        if len(out) == n:
            break
    assert out
    return spec, out


def _lam_dev(s):
    """the oracle's multipliers (QP variable order) -> the solver's LAM layout [N, 2, nu + nx]"""
    sp = s.spec
    lam = np.zeros((sp.N, 2, sp.nu + sp.nx))
    for side, v in enumerate(s.lam):
        for k in range(sp.N):
            lam[k, side, :sp.nu] = v[s.off_u[k]:s.off_u[k] + sp.nu]
            if k >= 1:
                lam[k, side, sp.nu:] = v[s.off_x[k]:s.off_x[k] + sp.nx]
    return lam


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the oracle restatement against finite differences, and the product templates (host build) against the oracle
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_oracle_forward_matches_finite_differences(model):
    spec, cases = _interior(model, 2, seed=21)
    h = 1e-4
    for x0, yref, s in cases:
        sx, su = so.solution_sensitivity(s)
        fx, fu = np.zeros_like(sx), np.zeros_like(su)
        for j in range(spec.nx):
            e = np.zeros(spec.nx); e[j] = h
            a, b = _oracle_solve(spec, x0 + e, yref), _oracle_solve(spec, x0 - e, yref)
            assert a.status == b.status == 0
            fx[:, :, j] = (a.x - b.x) / (2 * h)
            fu[:, :, j] = (a.u - b.u) / (2 * h)
        assert _rel(sx, fx) <= 1e-6 and _rel(su, fu) <= 1e-6, (_rel(sx, fx), _rel(su, fu))
        np.testing.assert_array_equal(sx[0], np.eye(spec.nx))


@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_oracle_adjoint_matches_forward_and_finite_differences(model):
    _, cases = _interior(model, 1, seed=22)
    x0, yref, _ = cases[0]
    spec = SPECS[model](tol=1e-12)        # (the finite differences resolve 1e-6 only with the QP solved this tightly)
    s = _oracle_solve(spec, x0, yref)
    rng = np.random.default_rng(5)
    sdx, sdu = rng.normal(size=(spec.N + 1, spec.nx)), rng.normal(size=(spec.N, spec.nu))
    gx, gy = so.adjoint_solution_sensitivity(s, sdx, sdu)
    sx, su = so.solution_sensitivity(s)
    want = np.einsum('kij,ki->j', sx, sdx) + np.einsum('kij,ki->j', su, sdu)
    assert _rel(gx, want) <= 1e-12, _rel(gx, want)
    # grad_yref along random directions d: d/dh of sum(seed . solution)(yref + h d)
    h = 1e-3
    J = lambda t: float((t.x * sdx).sum() + (t.u * sdu).sum())
    for _ in range(3):
        d = rng.normal(size=yref.shape)
        fd = (J(_oracle_solve(spec, x0, yref + h * d)) - J(_oracle_solve(spec, x0, yref - h * d))) / (2 * h)
        assert abs(fd - gy @ d) <= 1e-6 * abs(fd), (fd, gy @ d)
    assert np.all(gy[:spec.nx] == 0)        # the x-part of stage 0: x_0 = x0 whatever the reference


def _active_cases(model, seed, B=3):
    """instances whose input bounds are driven active by a large x0 offset"""
    spec = SPECS[model]()
    x0, yref = random_solve_inputs(model, B, seed)
    x0 = x0.copy()
    x0[:, 2:4] += 0.2 if model == 'jerk' else 0.4
    return spec, x0, yref


def _stage_bounds(spec, B, seed):
    rng = np.random.default_rng(seed)
    bnd = np.zeros((B, spec.N, 2, spec.nu + spec.nx))
    bnd[:, :, 0] = np.concatenate([spec.lbu, spec.lbx])
    bnd[:, :, 1] = np.concatenate([spec.ubu, spec.ubx])
    bnd[:, 3:9, 1, :spec.nu] = spec.ubu * (0.7 + 0.05 * rng.random((B, 6, spec.nu)))
    j, lim = (4, 2.0) if spec.nx == 6 else (2, 0.2)      # jerk: a_x, force: v_x
    bnd[:, 5:12, 0, spec.nu + j] = -lim
    bnd[:, 5:12, 1, spec.nu + j] = lim
    return bnd


@pytest.mark.parametrize('model', ['force', 'jerk', 'force_dense'])
@pytest.mark.parametrize('case', ['interior', 'active', 'stage_bounds'])
def test_product_templates_match_oracle_restatement(model, case):
    """the device templates (host build) against the dense-KKT restatement at identical stored iterates"""
    B = 3
    if case == 'active':
        spec, x0, yref = _active_cases(model, seed=31, B=B)
    else:
        spec = SPECS[model]()
        x0, yref = random_solve_inputs(model, B, seed=32)
    bnd = _stage_bounds(spec, B, seed=33) if case == 'stage_bounds' else None
    sols = [_oracle_solve(spec, x0[i], yref[i], None if bnd is None else bnd[i]) for i in range(B)]
    assert all(s.status == 0 for s in sols)
    if case != 'interior':
        assert min(_margin(s) for s in sols) < 1e-6          # some bound is active
    x = np.stack([s.x for s in sols]); u = np.stack([s.u for s in sols]); lam = np.stack([_lam_dev(s) for s in sols])
    p = np.repeat(np.array([[o.MASS, o.GRAVITY_ACC]]), B, 0)
    oo = hs.opts_from_oracle(co.default_opts(co.MODEL_JERK if model == 'jerk' else co.MODEL_FORCE))
    sx, su = hss.sens(HSS_MODEL[model], hss.FP64, oo, p, x, u, lam, bnd=bnd)
    rng = np.random.default_rng(34)
    sdx, sdu = rng.normal(size=(B, spec.N + 1, spec.nx)), rng.normal(size=(B, spec.N, spec.nu))
    gx, gy = hss.sens(HSS_MODEL[model], hss.FP64, oo, p, x, u, lam, bnd=bnd, seed_x=sdx, seed_u=sdu)
    gx0, _ = hss.sens(HSS_MODEL[model], hss.FP64, oo, p, x, u, lam, bnd=bnd, seed_u=sdu)
    for i, s in enumerate(sols):
        wx, wu = so.solution_sensitivity(s)
        assert _rel(sx[i], wx) <= 1e-10 and _rel(su[i], wu) <= 1e-10, (i, _rel(sx[i], wx), _rel(su[i], wu))
        wgx, wgy = so.adjoint_solution_sensitivity(s, sdx[i], sdu[i])
        assert _rel(gx[i], wgx) <= 1e-10 and _rel(gy[i], wgy) <= 1e-10, (i, _rel(gx[i], wgx), _rel(gy[i], wgy))
        wgx0, _ = so.adjoint_solution_sensitivity(s, None, sdu[i])
        assert _rel(gx0[i], wgx0) <= 1e-10
    # fewer stages: the leading part of the full result
    sx2, su2 = hss.sens(HSS_MODEL[model], hss.FP64, oo, p, x, u, lam, bnd=bnd, stages=2)
    np.testing.assert_allclose(sx2, sx[:, :2], rtol=0, atol=1e-12 * np.abs(sx).max())
    np.testing.assert_allclose(su2, su[:, :2], rtol=0, atol=1e-12 * np.abs(su).max())


def test_product_templates_nan_without_a_solution():
    spec = o.force_ocp()
    x0, yref = random_solve_inputs('force', 3, seed=35)
    sols = [_oracle_solve(spec, x0[i], yref[i]) for i in range(3)]
    x = np.stack([s.x for s in sols]); u = np.stack([s.u for s in sols]); lam = np.stack([_lam_dev(s) for s in sols])
    p = np.repeat(np.array([[o.MASS, o.GRAVITY_ACC]]), 3, 0)
    oo = hs.opts_from_oracle(co.default_opts(co.MODEL_FORCE))
    sx, su = hss.sens(hss.MODEL_FORCE, hss.FP64, oo, p, x, u, lam, status=[0, 1, 0], have_mult=[1, 1, 0])
    assert np.all(np.isfinite(sx[0])) and np.all(np.isfinite(su[0]))
    assert np.all(np.isnan(sx[1:])) and np.all(np.isnan(su[1:]))
    gx, gy = hss.sens(hss.MODEL_FORCE, hss.FP64, oo, p, x, u, lam, status=[0, 1, 0], have_mult=[1, 1, 0],
                      seed_u=np.ones((3, spec.N, 2)))
    assert np.all(np.isfinite(gx[0])) and np.all(np.isnan(gx[1:])) and np.all(np.isnan(gy[1:]))


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
def _solver(model, B, N=30, precision='fp64', tight=True, tol=1e-10):
    from drone_attitude_control_b200 import BatchedAcadosOcpSolver
    kw = dict(tol=[tol] * 4, qp_tol=[tol] * 4) if tight and precision == 'fp64' else {}
    if tight and precision == 'fp32':
        # what single precision can certify, as the shim's defaults, but with the complementarity driven 1000 times lower:
        # the multipliers of inactive bounds enter the KKT matrix as lam / t
        kw = dict(qp_tol=[1e-4, 1e-4, 1e-4, 1e-9], tol=[1e-3, 1e-3, 1e-3, 1e-8])
    return BatchedAcadosOcpSolver(model, batch=B, N_horizon=N, precision=precision, numpy_io=False, **kw)


def _inputs(model, B, N, seed, active=0, spread=0.08):
    """x0 [B, nx], yref [B, N*ny + nx]; the first `active` instances get an x0 offset that drives input bounds active"""
    x0, yref = random_solve_inputs('jerk' if model == 'jerk' else 'force', B, seed, spread=spread, N=N)
    x0 = x0.copy()
    x0[:active, 2:4] += 0.4
    return x0, yref


def _solve(sv, x0, yref):
    sv.set_yref_all(torch.tensor(yref, device=sv.device))
    sv.solve_for_x0(torch.tensor(x0, device=sv.device), fail_on_nonzero_status=False)
    return sv.get_stats('status').cpu().numpy()


def _oracle_at_device(sv, model, idx):
    """OracleOcpSolvers holding the device's stored solution of instances idx (iterate, multipliers, status)"""
    N, nx, nu = sv.N, sv.nx, sv.nu
    xs = torch.stack([sv.get(k, 'x') for k in range(N + 1)], 1).cpu().numpy()
    us = torch.stack([sv.get(k, 'u') for k in range(N)], 1).cpu().numpy()
    lams = [sv.get(k, 'lam').cpu().numpy() for k in range(N)]
    st = sv.get_stats('status').cpu().numpy()
    out = []
    for i in idx:
        s = o.OracleOcpSolver(SPECS[model](N=N))
        s.x[:], s.u[:] = xs[i], us[i]
        ll, lu = np.zeros(s.nv), np.zeros(s.nv)
        for k in range(N):
            L = lams[k][i]
            ll[s.off_u[k]:s.off_u[k] + nu] = L[:nu]
            if k == 0:
                lu[s.off_u[k]:s.off_u[k] + nu] = L[nu:]
            else:
                ll[s.off_x[k]:s.off_x[k] + nx] = L[nu:nu + nx]
                lu[s.off_u[k]:s.off_u[k] + nu] = L[nu + nx:2 * nu + nx]
                lu[s.off_x[k]:s.off_x[k] + nx] = L[2 * nu + nx:]
        s.lam, s.status = (ll, lu), int(st[i])
        out.append(s)
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk', 'force_dense'])
@pytest.mark.parametrize('B,N', [(1, 30), (256, 30), (4096, 30), (256, 100)])
def test_device_matches_oracle_restatement(model, B, N):
    sv = _solver(model, B, N)
    x0, yref = _inputs(model, B, N, seed=41, active=max(1, B // 8))
    st = _solve(sv, x0, yref)
    sx, su = (t.cpu().numpy() for t in sv.eval_solution_sensitivity())
    rng = np.random.default_rng(42)
    sdx, sdu = rng.normal(size=(B, N + 1, sv.nx)), rng.normal(size=(B, N, sv.nu))
    gx, gy = (t.cpu().numpy() for t in sv.eval_adjoint_solution_sensitivity(sdx, sdu))
    idx = sorted(set([0, B - 1] + list(rng.choice(B, min(B, 6), replace=False))))
    for i, s in zip(idx, _oracle_at_device(sv, model, idx)):
        assert st[i] == 0
        wx, wu = so.solution_sensitivity(s)
        wgx, wgy = so.adjoint_solution_sensitivity(s, sdx[i], sdu[i])
        errs = (_rel(sx[i], wx), _rel(su[i], wu), _rel(gx[i], wgx), _rel(gy[i], wgy))
        assert max(errs) <= 1e-9, (i, errs)


def _margins(sv, model):
    """status and distance of the solution to the nearest bound of every instance of a solved device solver"""
    ora = _oracle_at_device(sv, model, range(sv.batch))
    return np.array([s.status for s in ora]), np.array([_margin(s) for s in ora])


def fp32_against_fp64(model, B=256, N=30):
    """worst relative deviation (to the largest entry) of the FP32 sensitivities, computed in FP32 at the FP32 solution,
    from FP64 over the instances whose FP64 solution keeps every bound inactive by more than 0.05"""
    x0, yref = _inputs(model, B, N, seed=43, spread=0.01)
    res = {}
    for prec in ('fp64', 'fp32'):
        sv = _solver(model, B, N, precision=prec)
        st = _solve(sv, x0, yref)
        sx, su = (t.cpu().numpy() for t in sv.eval_solution_sensitivity())
        gx, gy = (t.cpu().numpy() for t in sv.eval_adjoint_solution_sensitivity(seed_u=np.ones((B, N, sv.nu))))
        res[prec] = (st, sx, su, gx, gy)
        if prec == 'fp64':
            _, margin = _margins(sv, model)
    ok = (res['fp64'][0] == 0) & (res['fp32'][0] == 0) & (margin > 0.05)
    return int(ok.sum()), max(_rel(a[ok], b[ok]) for a, b in zip(res['fp32'][1:], res['fp64'][1:]))


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_device_fp32_against_fp64(model):
    n, err = fp32_against_fp64(model)
    assert n >= 16 and err <= 1e-4, (n, err)      # (measured on a B200: 2.3e-6 force, 1.7e-6 jerk)


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_device_matches_finite_differences(model):
    B, N, h = 64, 30, 1e-4
    x0, yref = _inputs(model, B, N, seed=44, spread=0.01)
    sv = _solver(model, B, N, tol=1e-12)        # (the finite differences resolve 1e-6 only with the QP solved this tightly)
    _solve(sv, x0, yref)
    st, margin = _margins(sv, model)
    interior = np.nonzero((st == 0) & (margin > 0.02))[0]
    assert len(interior) >= 4
    sx, su = (t.cpu().numpy() for t in sv.eval_solution_sensitivity())
    fx, fu = np.zeros_like(sx), np.zeros_like(su)
    for j in range(sv.nx):
        out = []
        for sg in (1, -1):
            xp = x0.copy(); xp[:, j] += sg * h
            _solve(sv, xp, yref)
            out.append((torch.stack([sv.get(k, 'x') for k in range(N + 1)], 1).cpu().numpy(),
                        torch.stack([sv.get(k, 'u') for k in range(N)], 1).cpu().numpy()))
        fx[..., j] = (out[0][0] - out[1][0]) / (2 * h)
        fu[..., j] = (out[0][1] - out[1][1]) / (2 * h)
    for i in interior:
        assert _rel(sx[i], fx[i]) <= 1e-6 and _rel(su[i], fu[i]) <= 1e-6, (i, _rel(sx[i], fx[i]), _rel(su[i], fu[i]))


def _state(sv):
    N = sv.N
    f = lambda fld, n: torch.stack([sv.get(k, fld) for k in range(n)], 1).cpu().numpy()
    return dict(x=f('x', N + 1), u=f('u', N), pi=f('pi', N), lam=[sv.get(k, 'lam').cpu().numpy() for k in range(N)],
                stats=[sv.get_stats(k).cpu().numpy() for k in ('status', 'sqp_iter', 'qp_iter')])


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_sensitivity_leaves_the_handle_unchanged(model):
    B, N = 512, 30
    x0, yref = _inputs(model, B, N, seed=45, active=32)
    x1 = x0 + 0.01
    runs = []
    for between in (False, True):
        sv = _solver(model, B, N, tight=False)
        _solve(sv, x0, yref)
        if between:
            for call in (lambda: sv.eval_solution_sensitivity(), lambda: sv.eval_solution_sensitivity(stages=1),
                         lambda: sv.eval_adjoint_solution_sensitivity(seed_u=torch.ones(B, N, sv.nu, dtype=torch.float64)),
                         lambda: sv.eval_adjoint_solution_sensitivity(seed_x=torch.ones(B, N + 1, sv.nx, dtype=torch.float64))):
                n0 = sv.launch_count()
                call()
                assert sv.launch_count() == n0 + 1
        sv.set_yref_all(torch.tensor(yref, device=sv.device))
        u0 = sv.solve_for_x0(torch.tensor(x1, device=sv.device), fail_on_nonzero_status=False).cpu().numpy()
        runs.append((u0, _state(sv)))
    (ua, sa), (ub, sb) = runs
    np.testing.assert_array_equal(ua, ub)
    for k in sa:
        for a, b in zip(sa[k], sb[k]) if isinstance(sa[k], list) else [(sa[k], sb[k])]:
            np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_nan_rows_and_errors():
    import drone_attitude_control_b200 as pkg
    from drone_attitude_control_b200 import BatchedAcadosOcpSolver
    L = pkg.lib()
    B, N = 64, 30
    x0, yref = _inputs('force', B, N, seed=46)
    fresh = _solver('force', B, N, tight=False)
    sx, su = fresh.eval_solution_sensitivity()
    assert torch.isnan(sx).all() and torch.isnan(su).all()
    gx, gy = fresh.eval_adjoint_solution_sensitivity(seed_u=torch.ones(B, N, 2, dtype=torch.float64))
    assert torch.isnan(gx).all() and torch.isnan(gy).all()
    res = []
    for bad in (False, True):
        sv = _solver('force', B, N, tight=False)
        xb = x0.copy()
        if bad:
            xb[5] = np.nan
        st = _solve(sv, xb, yref)
        assert (st[5] == 1) == bad
        res.append([t.cpu().numpy() for t in sv.eval_solution_sensitivity()] +
                   [t.cpu().numpy() for t in sv.eval_adjoint_solution_sensitivity(seed_u=np.ones((B, N, 2)))])
    keep = np.arange(B) != 5
    for a, b in zip(*res):
        assert np.all(np.isnan(b[5]))
        np.testing.assert_array_equal(a[keep], b[keep])
    sv = _solver('force', 4, N, tight=False)
    h = sv.handle
    buf = torch.empty(4 * (N + 2) * 16, dtype=torch.float64, device=sv.device)
    p = C.c_void_p(buf.data_ptr())
    assert L.bnmpc_eval_sens_x0(h, 0, p, None, 1) == E_ARG
    assert L.bnmpc_eval_sens_x0(h, N + 2, p, None, 1) == E_ARG
    assert L.bnmpc_eval_adjoint_sens(h, None, None, p, None, 1) == E_ARG
    with pytest.raises(ValueError):
        sv.eval_solution_sensitivity(with_respect_to='p_global')
    for model in ('thrust', 'att'):
        other = BatchedAcadosOcpSolver(model, batch=2, numpy_io=False)
        assert L.bnmpc_eval_sens_x0(other.handle, 1, p, None, 1) == E_UNSUPPORTED
        assert L.bnmpc_eval_adjoint_sens(other.handle, p, None, p, None, 1) == E_UNSUPPORTED


@pytest.mark.gpu
def test_numpy_io_single_drone():
    x0, yref = _inputs('force', 1, 30, seed=47)
    from drone_attitude_control_b200 import BatchedAcadosOcpSolver
    sv = BatchedAcadosOcpSolver('force', batch=1)
    sv.set_yref_all(yref[0])
    sv.solve_for_x0(x0[0])
    sx, su = sv.eval_solution_sensitivity(stages=1)
    assert isinstance(sx, np.ndarray) and sx.shape == (1, 4, 4) and su.shape == (1, 2, 4)
    gx, gy = sv.eval_adjoint_solution_sensitivity(seed_u=np.eye(1, 60).reshape(30, 2))
    assert isinstance(gx, np.ndarray) and gx.shape == (4,) and gy.shape == (184,)
    np.testing.assert_allclose(gx, su[0, 0], rtol=1e-12, atol=1e-14)        # seed on u0[0]: row 0 of the gain


@pytest.mark.gpu
def test_grad_yref_from_bound_table_is_bit_identical():
    from common import random_loop_inputs
    B, N, row = 128, 30, 17
    refs, x0, _, _, _ = random_loop_inputs(B, 1, seed=48)
    win = np.concatenate([refs[:, row:row + N, :6].reshape(B, -1), refs[:, row + N, :4]], 1)
    xs = refs[:, row, :4] + 0.02
    seed_u = torch.randn(B, N, 2, dtype=torch.float64, generator=torch.Generator().manual_seed(3))
    out = []
    for table in (False, True):
        sv = _solver('force', B, N, tight=False)
        if table:
            sv.set_ref_table(refs)
            sv.set_yref_row(row)
        else:
            sv.set_yref_all(torch.tensor(win, device=sv.device))
        sv.solve_for_x0(torch.tensor(xs, device=sv.device), fail_on_nonzero_status=False)
        out.append([t.cpu().numpy() for t in sv.eval_adjoint_solution_sensitivity(seed_u=seed_u)])
    for a, b in zip(*out):
        np.testing.assert_array_equal(a, b)


@pytest.mark.gpu
def test_autograd_gradcheck_and_stale_backward():
    from drone_attitude_control_b200.autograd import solve_u0
    B, N = 3, 30
    cases = _interior('force', B, seed=49)[1]
    assert len(cases) == B
    x0, yref = np.stack([c[0] for c in cases]), np.stack([c[1] for c in cases])
    main, fd = _solver('force', B, N, tol=1e-12), _solver('force', B, N, tol=1e-12)
    calls = []

    def f(x, y):
        # gradcheck differentiates the first evaluation and then perturbs the inputs: the perturbed solves run on a second
        # solver so that the first one still holds the solution its backward differentiates
        calls.append(1)
        return solve_u0(main if len(calls) == 1 else fd, x, y)

    xt = torch.tensor(x0, device=main.device, requires_grad=True)
    yt = torch.tensor(yref, device=main.device, requires_grad=True)
    assert torch.autograd.gradcheck(f, (xt, yt), eps=1e-4, atol=1e-6, rtol=1e-5)
    u0 = solve_u0(main, xt, yt)
    main.solve_for_x0(torch.tensor(x0, device=main.device))
    with pytest.raises(RuntimeError, match='solved again'):
        u0.sum().backward()
