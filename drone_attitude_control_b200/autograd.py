"""The batched MPC as a differentiable layer: u0 = solve_u0(solver, x0, yref) with gradients for x0 and yref.

Backward is one adjoint sensitivity evaluation (bnmpc_eval_adjoint_sens) at the solution the forward solve left in the
solver, so the solver must not solve again between forward and backward; that is checked.  Models force, jerk and
force_dense (the ones whose solution sensitivities the library evaluates)."""
import torch


class _SolveU0(torch.autograd.Function):
    @staticmethod
    def forward(ctx, solver, x0, yref):
        solver.set_yref_all(yref.detach().to(solver.device, torch.float64).contiguous())
        x = x0.detach().to(solver.device, torch.float64).contiguous()
        u0 = torch.empty((solver.batch, solver.nu), dtype=torch.float64, device=solver.device)
        status = torch.empty(solver.batch, dtype=torch.int32, device=solver.device)
        solver.solve_for_x0_device(x, u0, status)
        ctx.solver, ctx.solve_count = solver, solver.solve_count
        ctx.x0_dtype, ctx.yref_dtype = x0.dtype, yref.dtype
        return u0

    @staticmethod
    def backward(ctx, grad_u0):
        solver = ctx.solver
        if solver.solve_count != ctx.solve_count:
            raise RuntimeError('solve_u0: the solver has solved again since this forward pass; its solution is gone, '
                               'so gradients of this u0 cannot be evaluated (use one solver per graph)')
        seed_u = torch.zeros((solver.batch, solver.N, solver.nu), dtype=torch.float64, device=solver.device)
        seed_u[:, 0] = grad_u0.to(torch.float64)
        grad_x0, grad_yref = solver.adjoint_device(seed_u=seed_u)
        return None, grad_x0.to(ctx.x0_dtype), grad_yref.to(ctx.yref_dtype)


def solve_u0(solver, x0, yref):
    """u0 [batch, nu] of `solver` (a BatchedAcadosOcpSolver) for x0 [batch, nx] and the reference window yref
    [batch, N*ny + ny_e] (set_yref_all layout): set_yref_all + solve_for_x0_device forward, the adjoint sensitivity with
    seed_u[0] = grad_u0 backward.  Gradients of a drone whose solve did not succeed are NaN."""
    return _SolveU0.apply(solver, x0, yref)
