"""Numpy restatement of the solution sensitivities (bnmpc_eval_sens_x0 / bnmpc_eval_adjoint_sens) at the stored solution
of an oracle.nmpc_oracle.OracleOcpSolver: the x0-eliminated KKT matrix assembled densely from the oracle's own QP
(OracleOcpSolver._linearise / _build_qp) and solved with a dense LU, so that agreement with the product's Riccati passes is
agreement between independent linear-algebra paths.  Test infrastructure only."""
import numpy as np

from oracle import nmpc_oracle as o


def kkt(s):
    """Dense x0-eliminated KKT matrix [[diag(H), G'], [G, 0]] at the stored iterate of `s`: H = dt W (W_e at stage N) +
    lam_lb / t_lb + lam_ub / t_ub with the multipliers of the last successful QP (s.lam) and the slacks recomputed from x / u,
    t_lb = max(v - lb, t_min), t_ub = max(ub - v, t_min); G the dynamics Jacobian of the stored iterate.  Returns (K, A) or
    None when the last solve did not succeed or there are no multipliers yet."""
    sp = s.spec
    if s.status != o.ACADOS_SUCCESS or s.lam is None:
        return None
    A, B, b = s._linearise()
    Hd, _, G, _, lb, ub, _ = s._build_qp(A, B, b)      # lb / ub: the boxes minus the iterate
    bounded = np.isfinite(lb)
    t_lb = np.maximum(np.where(bounded, -lb, 1.0), sp.t_min)
    t_ub = np.maximum(np.where(bounded, ub, 1.0), sp.t_min)
    lam_lb, lam_ub = s.lam
    H = Hd + np.where(bounded, lam_lb / t_lb + lam_ub / t_ub, 0.0)
    nv, ne = s.nv, G.shape[0]
    K = np.zeros((nv + ne, nv + ne))
    K[np.arange(nv), np.arange(nv)] = H
    K[:nv, nv:] = G.T
    K[nv:, :nv] = G
    return K, A


def solution_sensitivity(s, stages=None):
    """d x_k / d x0 [stages, nx, nx] and d u_k / d x0 [min(stages, N), nu, nx]: x0 enters only through the stage-0 dynamics
    offset b_0 = A_0 (x0 - x_0), so d(z, pi) / d x0 = -K^{-1} [0; A_0].  NaN without a successful solve."""
    sp = s.spec
    stages = sp.N + 1 if stages is None else int(stages)
    sx, su = np.full((stages, sp.nx, sp.nx), np.nan), np.full((min(stages, sp.N), sp.nu, sp.nx), np.nan)
    m = kkt(s)
    if m is None:
        return sx, su
    K, A = m
    rhs = np.zeros((K.shape[0], sp.nx))
    rhs[s.nv:s.nv + sp.nx] = -A[0]
    dz = np.linalg.solve(K, rhs)[:s.nv]
    for k in range(stages):
        sx[k] = np.eye(sp.nx) if k == 0 else dz[s.off_x[k]:s.off_x[k] + sp.nx]
    for k in range(min(stages, sp.N)):
        su[k] = dz[s.off_u[k]:s.off_u[k] + sp.nu]
    return sx, su


def adjoint_solution_sensitivity(s, seed_x=None, seed_u=None):
    """Vector-Jacobian products of the same derivative: seed_x [N+1, nx], seed_u [N, nu] (None = 0) -> grad_x0 [nx],
    grad_yref [N*(nx+nu) + nx] (set_yref_all layout).  With w = K^{-1} [seed; 0] (K is symmetric): grad_x0 = seed_x[0] -
    A_0' w_pi0 and, the cost gradient depending on yref through -dt W / -W_e, grad_yref = dt W w / W_e w (0 for the x-part of
    stage 0)."""
    sp = s.spec
    ny = sp.nx + sp.nu
    sdx = np.zeros((sp.N + 1, sp.nx)) if seed_x is None else np.asarray(seed_x, float)
    sdu = np.zeros((sp.N, sp.nu)) if seed_u is None else np.asarray(seed_u, float)
    m = kkt(s)
    if m is None:
        return np.full(sp.nx, np.nan), np.full(sp.N * ny + sp.nx, np.nan)
    K, A = m
    rhs = np.zeros(K.shape[0])
    for k in range(sp.N):
        rhs[s.off_u[k]:s.off_u[k] + sp.nu] = sdu[k]
    for k in range(1, sp.N + 1):
        rhs[s.off_x[k]:s.off_x[k] + sp.nx] = sdx[k]
    w = np.linalg.solve(K, rhs)
    gx = sdx[0] - A[0].T @ w[s.nv:s.nv + sp.nx]
    gy = np.zeros(sp.N * ny + sp.nx)
    for k in range(sp.N):
        gy[k * ny + sp.nx:(k + 1) * ny] = sp.dt * sp.w[sp.nx:] * w[s.off_u[k]:s.off_u[k] + sp.nu]
        if k >= 1:
            gy[k * ny:k * ny + sp.nx] = sp.dt * sp.w[:sp.nx] * w[s.off_x[k]:s.off_x[k] + sp.nx]
    gy[sp.N * ny:] = sp.w_e * w[s.off_x[sp.N]:s.off_x[sp.N] + sp.nx]
    return gx, gy
