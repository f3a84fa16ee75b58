"""Numpy restatement of the solution sensitivities with respect to the model parameters p = (mass, g)
(bnmpc_eval_sens_p / bnmpc_eval_adjoint_sens_p) at the stored solution of an oracle.nmpc_oracle.OracleOcpSolver: the
dense x0-eliminated KKT matrix of tests/sens_oracle.py (from the oracle's own linearisation and QP) with the derivative in p
of the KKT residual as right-hand side, assembled from the oracle's own integrator.  Test infrastructure only."""
import numpy as np

from oracle import nmpc_oracle as o
from sens_oracle import kkt


def _dynamics_dp(s, k):
    """d phi_k / d p [nx, 2], d A_k / d p [2, nx, nx], d B_k / d p [2, nx, nu] at the stored (x_k, u_k), from the oracle's own
    integrator (erk_step, the scheme of spec.erk_stages).  Closed forms: for the force and jerk models the parameters enter
    f only through q = 1 / mass (as q u) and g (as a constant drift), so every stage derivative of the explicit and implicit
    schemes - and hence phi, A and B - is affine in (q, g) for fixed (x, u).  A central difference in q or in g is then exact
    up to round-off for any step; the step is half the parameter, and the affinity is asserted through the second
    difference.  d / d mass = -q^2 d / d q."""
    sp = s.spec
    m, g = s.p
    q = 1.0 / m

    def ev(qq, gg):
        xn, S = o.erk_step(sp.f, sp.jac, s.x[k], s.u[k], np.array([1.0 / qq, gg]), sp.dt, sp.erk_stages)
        return np.concatenate([xn, S.ravel()])

    mid = ev(q, g)
    out = []
    for j, (hq, hg) in enumerate(((q / 2, 0.0), (0.0, max(abs(g), 1.0) / 2))):
        hi, lo = ev(q + hq, g + hg), ev(q - hq, g - hg)
        scale = max(np.abs(mid).max(), 1.0)
        assert np.abs(hi - 2 * mid + lo).max() <= 1e-12 * scale, 'phi is not affine in (1/mass, g)'
        d = (hi - lo) / (2 * (hq + hg))
        out.append(d * (-q * q) if j == 0 else d)
    nx, nu = sp.nx, sp.nu
    phi_p = np.stack([d[:nx] for d in out], 1)
    S_p = [d[nx:].reshape(nx, nx + nu) for d in out]
    return phi_p, np.stack([S[:, :nx] for S in S_p]), np.stack([S[:, nx:] for S in S_p])


def param_residual(s):
    """[dR; dc] [nv + ne, 2]: the derivative in p = (mass, g) of the KKT residual at the stored solution, with the oracle's
    conventions c_k = phi_k(x_k, u_k; p) - x_{k+1}, grad_u L = dt W (u - yref) + B_k' pi_k, grad_x L = ... + A_k' pi_k -
    pi_{k-1}: dc_k = d phi_k / d p, dR = (d B_k / d p)' pi_k (u-part, k < N), (d A_k / d p)' pi_k (x-part, 1 <= k < N)."""
    sp = s.spec
    D = np.zeros((s.nv + sp.N * sp.nx, 2))
    for k in range(sp.N):
        phi_p, A_p, B_p = _dynamics_dp(s, k)
        D[s.nv + k * sp.nx:s.nv + (k + 1) * sp.nx] = phi_p
        for j in range(2):
            D[s.off_u[k]:s.off_u[k] + sp.nu, j] = B_p[j].T @ s.pi[k]
            if k >= 1:
                D[s.off_x[k]:s.off_x[k] + sp.nx, j] = A_p[j].T @ s.pi[k]
    return D


def param_sensitivity(s, stages=None):
    """d x_k / d p [stages, nx, 2] and d u_k / d p [min(stages, N), nu, 2] = the z-part of -K^{-1} [dR; dc]; sens_x[0] = 0
    (x_0 is fixed by x0).  NaN without a successful solve."""
    sp = s.spec
    stages = sp.N + 1 if stages is None else int(stages)
    sx, su = np.full((stages, sp.nx, 2), np.nan), np.full((min(stages, sp.N), sp.nu, 2), np.nan)
    m = kkt(s)
    if m is None:
        return sx, su
    K, _ = m
    dz = -np.linalg.solve(K, param_residual(s))[:s.nv]
    for k in range(stages):
        sx[k] = 0.0 if k == 0 else dz[s.off_x[k]:s.off_x[k] + sp.nx]
    for k in range(min(stages, sp.N)):
        su[k] = dz[s.off_u[k]:s.off_u[k] + sp.nu]
    return sx, su


def adjoint_param_sensitivity(s, seed_x=None, seed_u=None):
    """grad_p [2] = sum over the stages of (d x_k / d p)' seed_x[k] + (d u_k / d p)' seed_u[k] = -[dR; dc]' K^{-1} [seed; 0]
    (K is symmetric); seed_x[0] does not enter (x_0 is fixed).  NaN without a successful solve."""
    sp = s.spec
    sdx = np.zeros((sp.N + 1, sp.nx)) if seed_x is None else np.asarray(seed_x, float)
    sdu = np.zeros((sp.N, sp.nu)) if seed_u is None else np.asarray(seed_u, float)
    m = kkt(s)
    if m is None:
        return np.full(2, np.nan)
    K, _ = m
    rhs = np.zeros(K.shape[0])
    for k in range(sp.N):
        rhs[s.off_u[k]:s.off_u[k] + sp.nu] = sdu[k]
    for k in range(1, sp.N + 1):
        rhs[s.off_x[k]:s.off_x[k] + sp.nx] = sdx[k]
    return -param_residual(s).T @ np.linalg.solve(K, rhs)
