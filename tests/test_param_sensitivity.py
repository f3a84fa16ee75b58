"""Sensitivities of the batched solve with respect to the model parameters p = (mass, g) (bnmpc_eval_sens_p /
bnmpc_eval_adjoint_sens_p, the shim's eval_param_sensitivity / eval_adjoint_param_sensitivity, autograd.solve_u0 with p).
The pins are central finite differences of solves in p and the dense-KKT restatement of tests/sens_oracle_p.py at the
stored solution of an oracle.nmpc_oracle.OracleOcpSolver, which the product templates (host build: tests/hostsim_sens_p,
and the device) must match at identical stored iterates."""
import ctypes as C
import dataclasses

import numpy as np
import pytest
import torch

import hostsim as hs
import hostsim_sens as hss
import hostsim_sens_p as hssp
import sens_oracle_p as sop
from common import random_solve_inputs
from oracle import c_oracle as co
from oracle import nmpc_oracle as o
from test_sensitivity import (HSS_MODEL, SPECS, _active_cases, _inputs, _lam_dev, _margin, _oracle_at_device, _rel,
                              _set_oracle_bounds, _solver, _stage_bounds, _state)

E_ARG, E_UNSUPPORTED = -1, -5
P_NOM = np.array([o.MASS, o.GRAVITY_ACC])
# central-difference steps relative to each parameter (mass 0.033, g 9.81).  With no bound active the solution is affine
# in g (g only shifts the drift of affine dynamics).  In the force model the input cancels a change of g almost entirely,
# so d x / d g is ~1e-4 of d u / d g and needs a longer step for the solver's tolerance not to drown it; in the jerk model
# a longer step moves the vertical acceleration onto its bound.  The solution is rational in the mass: 1e-3 keeps the
# truncation error below 1e-6 while the solver's tolerance (~1e-11 in the solution) divided by the step stays there too.
FD_STEP = {'force': (1e-3, 1e-2), 'jerk': (1e-3, 1e-4)}


def _p_of(B, seed):
    """per-drone controller parameters around the nominal ones (mass +-10 %, g +-2 %)"""
    rng = np.random.default_rng(seed)
    return P_NOM * (1 + np.stack([rng.uniform(-0.1, 0.1, B), rng.uniform(-0.02, 0.02, B)], 1))


def _solve(spec, x0, yref, p, bnd=None):
    s = o.OracleOcpSolver(spec, p=p)
    ny = spec.nx + spec.nu
    for k in range(spec.N):
        s.set(k, 'yref', yref[k * ny:(k + 1) * ny])
    s.set(spec.N, 'yref', yref[spec.N * ny:])
    s.set(0, 'lbx', x0)
    if bnd is not None:
        _set_oracle_bounds(s, bnd)
    s.solve()
    return s


def _rel_cols(a, b):
    """worst relative error over the parameter columns (last axis), each relative to its own largest entry"""
    return max(_rel(np.asarray(a)[..., j], np.asarray(b)[..., j]) for j in range(np.shape(b)[-1]))


# ------------------------------------------------------------------------------------------------------------------------
# CPU: the oracle restatement against finite differences, and the product templates (host build) against the oracle
# ------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_oracle_param_sensitivity_matches_finite_differences(model):
    spec = SPECS[model](tol=1e-12)        # (the finite differences resolve 1e-6 only with the QP solved this tightly)
    x0, yref = random_solve_inputs(model, 16, seed=61, spread=0.01)
    p = _p_of(16, seed=62)
    cases = []
    for i in range(16):
        s = _solve(spec, x0[i], yref[i], p[i])
        if s.status == 0 and _margin(s) > 0.02:
            cases.append((i, s))
    assert len(cases) >= 2
    rng = np.random.default_rng(63)
    for i, s in cases[:2]:
        sx, su = sop.param_sensitivity(s)
        fx, fu = np.zeros_like(sx), np.zeros_like(su)
        for j in range(2):
            h = FD_STEP[model][j] * p[i, j]
            e = np.zeros(2); e[j] = h
            a, b = _solve(spec, x0[i], yref[i], p[i] + e), _solve(spec, x0[i], yref[i], p[i] - e)
            assert a.status == b.status == 0
            fx[..., j] = (a.x - b.x) / (2 * h)
            fu[..., j] = (a.u - b.u) / (2 * h)
        assert _rel_cols(sx, fx) <= 1e-6 and _rel_cols(su, fu) <= 1e-6, (_rel_cols(sx, fx), _rel_cols(su, fu))
        assert np.all(sx[0] == 0)
        if model == 'jerk':
            assert np.all(fx[..., 0] == 0) and np.all(sx[..., 0] == 0) and np.all(su[..., 0] == 0)
        else:
            assert np.abs(su[..., 0]).max() > 1.0          # the force model's inputs scale with the mass
        sdx, sdu = rng.normal(size=(spec.N + 1, spec.nx)), rng.normal(size=(spec.N, spec.nu))
        gp = sop.adjoint_param_sensitivity(s, sdx, sdu)
        want = np.einsum('kij,ki->j', sx, sdx) + np.einsum('kij,ki->j', su, sdu)
        assert _rel(gp, want) <= 1e-12, _rel(gp, want)


def _templates_case(model, case, erk, B=3):
    if case == 'active':
        spec, x0, yref = _active_cases(model, seed=64, B=B)
    else:
        spec = SPECS[model]()
        x0, yref = random_solve_inputs(model, B, seed=32)
    spec = dataclasses.replace(spec, erk_stages=erk)
    bnd = _stage_bounds(spec, B, seed=66) if case == 'stage_bounds' else None
    p = _p_of(B, seed=67)
    sols = [_solve(spec, x0[i], yref[i], p[i], None if bnd is None else bnd[i]) for i in range(B)]
    assert all(s.status == 0 for s in sols)
    if case != 'interior':
        assert min(_margin(s) for s in sols) < 1e-6          # some bound is active
    oo = hs.opts_from_oracle(co.default_opts(co.MODEL_JERK if model == 'jerk' else co.MODEL_FORCE))
    oo.erk_stages = erk
    st = dict(x=np.stack([s.x for s in sols]), u=np.stack([s.u for s in sols]), lam=np.stack([_lam_dev(s) for s in sols]),
              pi=np.stack([s.pi for s in sols]), bnd=bnd)
    return spec, sols, oo, p, st


@pytest.mark.parametrize('erk', [4, 1, 0])
@pytest.mark.parametrize('model', ['force', 'jerk', 'force_dense'])
@pytest.mark.parametrize('case', ['interior', 'active', 'stage_bounds'])
def test_product_templates_match_oracle_restatement(model, case, erk):
    """forward and adjoint in p of the device templates (host build) against the dense-KKT restatement at identical stored
    iterates, for the explicit schemes with 4 and 1 stages and the implicit Gauss-Legendre scheme (erk_stages = 0)"""
    spec, sols, oo, p, st = _templates_case(model, case, erk)
    B, M = len(sols), HSS_MODEL[model]
    sx, su = hssp.sens_p(M, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], bnd=st['bnd'])
    rng = np.random.default_rng(68)
    sdx, sdu = rng.normal(size=(B, spec.N + 1, spec.nx)), rng.normal(size=(B, spec.N, spec.nu))
    gx, gy, gp = hssp.sens_p(M, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], bnd=st['bnd'], seed_x=sdx, seed_u=sdu)
    _, _, gpu = hssp.sens_p(M, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], bnd=st['bnd'], seed_u=sdu)
    for i, s in enumerate(sols):
        wx, wu = sop.param_sensitivity(s)
        assert _rel_cols(sx[i], wx) <= 1e-10 and _rel_cols(su[i], wu) <= 1e-10, (i, _rel_cols(sx[i], wx), _rel_cols(su[i], wu))
        wgp = sop.adjoint_param_sensitivity(s, sdx[i], sdu[i])
        assert _rel(gp[i], wgp) <= 1e-10, (i, gp[i], wgp)
        assert _rel(gpu[i], sop.adjoint_param_sensitivity(s, None, sdu[i])) <= 1e-10
    # the adjoint is the seed contracted with the forward result
    want = np.einsum('bkij,bki->bj', sx, sdx) + np.einsum('bkij,bki->bj', su, sdu)
    assert _rel(gp, want) <= 1e-10, _rel(gp, want)
    # grad_x0 / grad_yref of the same evaluation are those of the adjoint without grad_p, bit for bit
    gx0, gy0 = hss.sens(M, hss.FP64, oo, p, st['x'], st['u'], st['lam'], bnd=st['bnd'], seed_x=sdx, seed_u=sdu)
    np.testing.assert_array_equal(gx, gx0)
    np.testing.assert_array_equal(gy, gy0)
    gx1, gy1, none = hssp.sens_p(M, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], bnd=st['bnd'], seed_x=sdx,
                                 seed_u=sdu, with_grad_p=False)
    assert none is None
    np.testing.assert_array_equal(gx1, gx0)
    np.testing.assert_array_equal(gy1, gy0)
    # fewer stages: the leading part of the full result
    sx2, su2 = hssp.sens_p(M, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], bnd=st['bnd'], stages=2)
    np.testing.assert_allclose(sx2, sx[:, :2], rtol=0, atol=1e-12 * np.abs(sx).max())
    np.testing.assert_allclose(su2, su[:, :2], rtol=0, atol=1e-12 * np.abs(su).max())
    assert np.all(sx[:, 0] == 0)
    if model == 'jerk':          # the mass does not enter the jerk model
        assert np.all(sx[..., 0] == 0) and np.all(su[..., 0] == 0) and np.all(gp[:, 0] == 0)


def test_product_templates_fp32_and_nan_rows():
    spec, sols, oo, p, st = _templates_case('force', 'interior', 4)
    B = len(sols)
    sx64, su64 = hssp.sens_p(hssp.MODEL_FORCE, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'])
    sx32, su32 = hssp.sens_p(hssp.MODEL_FORCE, hssp.FP32, oo, p, st['x'], st['u'], st['lam'], st['pi'])
    assert _rel_cols(sx32, sx64) <= 1e-4 and _rel_cols(su32, su64) <= 1e-4
    status, have_mult = [0, 1, 0], [1, 1, 0]
    sx, su = hssp.sens_p(hssp.MODEL_FORCE, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], status=status,
                        have_mult=have_mult)
    assert np.all(np.isfinite(sx[0])) and np.all(np.isfinite(su[0]))
    assert np.all(np.isnan(sx[1:])) and np.all(np.isnan(su[1:]))
    gx, gy, gp = hssp.sens_p(hssp.MODEL_FORCE, hssp.FP64, oo, p, st['x'], st['u'], st['lam'], st['pi'], status=status,
                            have_mult=have_mult, seed_u=np.ones((B, spec.N, 2)))
    assert np.all(np.isfinite(gp[0])) and np.all(np.isnan(gp[1:])) and np.all(np.isnan(gx[1:])) and np.all(np.isnan(gy[1:]))


# ------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------
def _solve_dev(sv, x0, yref, p):
    sv.set(0, 'p', torch.tensor(p, device=sv.device))
    sv.set_yref_all(torch.tensor(yref, device=sv.device))
    sv.solve_for_x0(torch.tensor(x0, device=sv.device), fail_on_nonzero_status=False)
    return sv.get_stats('status').cpu().numpy()


def _oracle_at_device_p(sv, model, idx, p):
    """_oracle_at_device plus the multipliers of the dynamics and the parameters of each instance"""
    pis = torch.stack([sv.get(k, 'pi') for k in range(sv.N)], 1).cpu().numpy()
    out = _oracle_at_device(sv, model, idx)
    for i, s in zip(idx, out):
        s.pi[:] = pis[i]
        s.p[:] = p[i]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk', 'force_dense'])
@pytest.mark.parametrize('B,N', [(1, 30), (256, 30), (4096, 30), (256, 100)])
def test_device_matches_oracle_restatement(model, B, N):
    sv = _solver(model, B, N)
    x0, yref = _inputs(model, B, N, seed=71, active=max(1, B // 8))
    p = _p_of(B, seed=72)
    st = _solve_dev(sv, x0, yref, p)
    sx, su = (t.cpu().numpy() for t in sv.eval_param_sensitivity())
    rng = np.random.default_rng(73)
    sdx, sdu = rng.normal(size=(B, N + 1, sv.nx)), rng.normal(size=(B, N, sv.nu))
    gp = sv.eval_adjoint_param_sensitivity(sdx, sdu).cpu().numpy()
    idx = sorted(set([0, B - 1] + list(rng.choice(B, min(B, 6), replace=False))))
    for i, s in zip(idx, _oracle_at_device_p(sv, model, idx, p)):
        assert st[i] == 0
        wx, wu = sop.param_sensitivity(s)
        wgp = sop.adjoint_param_sensitivity(s, sdx[i], sdu[i])
        errs = (_rel_cols(sx[i], wx), _rel_cols(su[i], wu), _rel(gp[i], wgp))
        assert max(errs) <= 1e-9, (i, errs)
    ok = st == 0                 # (the other instances have NaN rows)
    if model == 'jerk':
        assert np.all(sx[ok, ..., 0] == 0) and np.all(su[ok, ..., 0] == 0) and np.all(gp[ok, 0] == 0)


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_device_matches_finite_differences(model):
    B, N = 64, 30
    x0, yref = _inputs(model, B, N, seed=74, spread=0.01)
    p = _p_of(B, seed=75)
    # Solved this tightly: at 1e-12 the interior point stops with multipliers of ~1e-11 on bounds 0.05 away, and the mass
    # derivative of the solution it returns differs from that of the exact solution by up to 2e-6 (the oracle agrees).
    tol = 1e-14
    sv = _solver(model, B, N, tol=tol)
    _solve_dev(sv, x0, yref, p)
    ora = _oracle_at_device(sv, model, range(B))
    st, margin = np.array([s.status for s in ora]), np.array([_margin(s) for s in ora])
    interior = np.nonzero((st == 0) & (margin > 0.02))[0]
    assert len(interior) >= 4
    sx, su = (t.cpu().numpy() for t in sv.eval_param_sensitivity())
    fx, fu = np.zeros_like(sx), np.zeros_like(su)
    for j in range(2):
        h = FD_STEP[model][j] * p[:, j]
        out = []
        for sg in (1, -1):
            # each perturbed solve starts cold, like the one differentiated: a re-solve warm-started from the previous
            # solution ends at a point that differs by a few 1e-6 in these difference quotients
            pp = p.copy(); pp[:, j] += sg * h
            sp = _solver(model, B, N, tol=tol)
            assert np.all(_solve_dev(sp, x0, yref, pp)[interior] == 0)
            out.append((torch.stack([sp.get(k, 'x') for k in range(N + 1)], 1).cpu().numpy(),
                        torch.stack([sp.get(k, 'u') for k in range(N)], 1).cpu().numpy()))
        fx[..., j] = (out[0][0] - out[1][0]) / (2 * h[:, None, None])
        fu[..., j] = (out[0][1] - out[1][1]) / (2 * h[:, None, None])
    # (d x / d g of the force model is ~1e-4 of d x / d mass and cancels almost entirely: finite differences of device
    # solves do not resolve it to 1e-6 of itself, so the states are compared relative to their largest entry, as for x0)
    for i in interior:
        assert _rel(sx[i], fx[i]) <= 1e-6 and _rel_cols(su[i], fu[i]) <= 1e-6, (i, _rel(sx[i], fx[i]), _rel_cols(su[i], fu[i]))


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_device_fp32_against_fp64(model):
    """the protocol of test_sensitivity.fp32_against_fp64: FP32 at the FP32 solution against FP64, on the instances whose
    FP64 solution keeps every bound inactive by more than 0.05"""
    B, N = 256, 30
    x0, yref = _inputs(model, B, N, seed=43, spread=0.01)
    p = _p_of(B, seed=76)
    seed_u = np.ones((B, N, 2))
    res = {}
    for prec in ('fp64', 'fp32'):
        sv = _solver(model, B, N, precision=prec)
        st = _solve_dev(sv, x0, yref, p)
        sx, su = (t.cpu().numpy() for t in sv.eval_param_sensitivity())
        res[prec] = (st, sx, su, sv.eval_adjoint_param_sensitivity(seed_u=seed_u).cpu().numpy())
        if prec == 'fp64':
            margin = np.array([_margin(s) for s in _oracle_at_device(sv, model, range(B))])
    ok = (res['fp64'][0] == 0) & (res['fp32'][0] == 0) & (margin > 0.05)
    assert ok.sum() >= 16
    err = max(_rel(a[ok], b[ok]) for a, b in zip(res['fp32'][1:], res['fp64'][1:]))
    assert err <= 1e-4, err


@pytest.mark.gpu
def test_nan_rows_and_errors():
    import drone_attitude_control_b200 as pkg
    from drone_attitude_control_b200 import BatchedAcadosOcpSolver
    L = pkg.lib()
    B, N = 64, 30
    x0, yref = _inputs('force', B, N, seed=77)
    p = _p_of(B, seed=78)
    fresh = _solver('force', B, N, tight=False)
    sx, su = fresh.eval_param_sensitivity()
    assert torch.isnan(sx).all() and torch.isnan(su).all()
    assert torch.isnan(fresh.eval_adjoint_param_sensitivity(seed_u=torch.ones(B, N, 2, dtype=torch.float64))).all()
    res = []
    for bad in (False, True):
        sv = _solver('force', B, N, tight=False)
        xb = x0.copy()
        if bad:
            xb[5] = np.nan
        st = _solve_dev(sv, xb, yref, p)
        assert (st[5] == 1) == bad
        res.append([t.cpu().numpy() for t in sv.eval_param_sensitivity()] +
                   [sv.eval_adjoint_param_sensitivity(seed_u=np.ones((B, N, 2))).cpu().numpy()])
    keep = np.arange(B) != 5
    for a, b in zip(*res):
        assert np.all(np.isnan(b[5]))
        np.testing.assert_array_equal(a[keep], b[keep])
    sv = _solver('force', 4, N, tight=False)
    h = sv.handle
    buf = torch.empty(4 * (N + 2) * 16, dtype=torch.float64, device=sv.device)
    q = C.c_void_p(buf.data_ptr())
    assert L.bnmpc_eval_sens_p(h, 0, q, None, 1) == E_ARG
    assert L.bnmpc_eval_sens_p(h, N + 2, q, None, 1) == E_ARG
    assert L.bnmpc_eval_sens_p(h, 1, q, None, 2) == E_ARG
    assert L.bnmpc_eval_adjoint_sens_p(h, None, None, q, None, q, 1) == E_ARG
    with pytest.raises(ValueError):
        sv.eval_param_sensitivity(stages=N + 2)
    for model in ('thrust', 'att'):
        other = BatchedAcadosOcpSolver(model, batch=2, numpy_io=False)
        assert L.bnmpc_eval_sens_p(other.handle, 1, q, None, 1) == E_UNSUPPORTED
        assert L.bnmpc_eval_adjoint_sens_p(other.handle, q, None, None, None, q, 1) == E_UNSUPPORTED


@pytest.mark.gpu
@pytest.mark.parametrize('model', ['force', 'jerk'])
def test_one_launch_and_the_handle_is_unchanged(model):
    B, N = 512, 30
    x0, yref = _inputs(model, B, N, seed=79, active=32)
    p = _p_of(B, seed=80)
    x1 = x0 + 0.01
    runs = []
    for between in (False, True):
        sv = _solver(model, B, N, tight=False)
        _solve_dev(sv, x0, yref, p)
        if between:
            ones = lambda *sh: torch.ones(*sh, dtype=torch.float64)
            for call in (lambda: sv.eval_param_sensitivity(), lambda: sv.eval_param_sensitivity(stages=1),
                         lambda: sv.eval_adjoint_param_sensitivity(seed_u=ones(B, N, sv.nu)),
                         lambda: sv.eval_adjoint_param_sensitivity(seed_x=ones(B, N + 1, sv.nx)),
                         lambda: sv._adjoint_device_p(seed_u=ones(B, N, sv.nu))):
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
@pytest.mark.parametrize('on_device', [0, 1])
def test_adjoint_without_grad_p_is_bit_identical(on_device):
    """bnmpc_eval_adjoint_sens_p(.., grad_p = NULL) and bnmpc_eval_adjoint_sens give the same grad_x0 / grad_yref bit for
    bit; with grad_p (a separate kernel instantiation) they agree to rounding; host and device buffers give the same bits"""
    import drone_attitude_control_b200 as pkg
    L = pkg.lib()
    B, N = 256, 30
    x0, yref = _inputs('force', B, N, seed=81, active=16)
    sv = _solver('force', B, N, tight=False)
    _solve_dev(sv, x0, yref, _p_of(B, seed=82))
    rng = np.random.default_rng(83)
    sdx, sdu = rng.normal(size=(B, N + 1, 4)), rng.normal(size=(B, N, 2))
    ny = N * 6 + 4

    def bufs():
        if on_device:
            t = [torch.tensor(sdx, device=sv.device), torch.tensor(sdu, device=sv.device)]
            t += [torch.full(sh, 7.0, dtype=torch.float64, device=sv.device) for sh in ((B, 4), (B, ny), (B, 2))]
            return t, [C.c_void_p(a.data_ptr()) for a in t], lambda a: a.cpu().numpy()
        t = [np.ascontiguousarray(sdx), np.ascontiguousarray(sdu)] + [np.full(sh, 7.0) for sh in ((B, 4), (B, ny), (B, 2))]
        return t, [C.c_void_p(a.ctypes.data) for a in t], lambda a: a.copy()

    out = []
    for variant in range(3):
        t, ptr, get = bufs()
        if variant == 0:
            rc = L.bnmpc_eval_adjoint_sens(sv.handle, ptr[0], ptr[1], ptr[2], ptr[3], on_device)
        else:
            rc = L.bnmpc_eval_adjoint_sens_p(sv.handle, ptr[0], ptr[1], ptr[2], ptr[3], ptr[4] if variant == 2 else None,
                                             on_device)
        assert rc == 0
        torch.cuda.synchronize()
        out.append([get(a) for a in t[2:]])
    np.testing.assert_array_equal(out[1][0], out[0][0])
    np.testing.assert_array_equal(out[1][1], out[0][1])
    for a, b in zip(out[2][:2], out[0][:2]):
        assert _rel(a, b) <= 1e-12, _rel(a, b)
    assert np.all(out[1][2] == 7.0)         # grad_p = NULL: nothing written there
    want = sv.eval_adjoint_param_sensitivity(sdx, sdu).cpu().numpy()
    np.testing.assert_array_equal(out[2][2], want)


@pytest.mark.gpu
def test_numpy_io_single_drone():
    from drone_attitude_control_b200 import BatchedAcadosOcpSolver
    x0, yref = _inputs('force', 1, 30, seed=84)
    sv = BatchedAcadosOcpSolver('force', batch=1)
    sv.set(0, 'p', P_NOM * [1.05, 1.0])
    sv.set_yref_all(yref[0])
    sv.solve_for_x0(x0[0])
    sx, su = sv.eval_param_sensitivity(stages=1)
    assert isinstance(sx, np.ndarray) and sx.shape == (1, 4, 2) and su.shape == (1, 2, 2)
    gp = sv.eval_adjoint_param_sensitivity(seed_u=np.eye(1, 60).reshape(30, 2))
    assert isinstance(gp, np.ndarray) and gp.shape == (2,)
    np.testing.assert_allclose(gp, su[0, 0], rtol=1e-12, atol=1e-14)        # seed on u0[0]: row 0 of d u0 / d p


@pytest.mark.gpu
def test_autograd_gradcheck_with_p():
    from drone_attitude_control_b200.autograd import solve_u0
    B, N = 3, 30
    spec = SPECS['force'](tol=1e-10)
    x0, yref = random_solve_inputs('force', 16, seed=85, spread=0.01)
    p0 = _p_of(16, seed=86)
    pick = [i for i in range(16) if (lambda s: s.status == 0 and _margin(s) > 0.02)(_solve(spec, x0[i], yref[i], p0[i]))]
    assert len(pick) >= B
    pick = pick[:B]
    x0, yref, p0 = x0[pick], yref[pick], p0[pick]
    main, fd = _solver('force', B, N, tol=1e-12), _solver('force', B, N, tol=1e-12)
    calls = []
    pt = torch.tensor(p0, device=main.device)

    def f(x, y, s):
        # p = p0 exp(s): one eps suits both parameters.  gradcheck differentiates the first evaluation and then perturbs
        # the inputs: the perturbed solves run on a second solver so that the first one still holds its solution
        calls.append(1)
        return solve_u0(main if len(calls) == 1 else fd, x, y, pt * torch.exp(s))

    xt = torch.tensor(x0, device=main.device, requires_grad=True)
    yt = torch.tensor(yref, device=main.device, requires_grad=True)
    st = torch.zeros((B, 2), dtype=torch.float64, device=main.device, requires_grad=True)
    assert torch.autograd.gradcheck(f, (xt, yt, st), eps=1e-4, atol=1e-6, rtol=1e-5)
    # p = None keeps the parameters the solver has: the same u0, and the gradients of the call with p for x0 and yref (to
    # rounding: with p the backward is the adjoint kernel that also evaluates grad_p)
    main.set(0, 'p', pt)
    u_a = solve_u0(main, xt, yt)
    ga = torch.autograd.grad(u_a.sum(), (xt, yt))
    u_b = solve_u0(main, xt, yt, pt.clone().requires_grad_(True))
    gb = torch.autograd.grad(u_b.sum(), (xt, yt))
    torch.testing.assert_close(u_a, u_b, rtol=0, atol=0)
    for a, b in zip(ga, gb):
        torch.testing.assert_close(a, b, rtol=1e-12, atol=1e-12 * float(b.abs().max()))
