// bnmpc_loop.cuh - the glue either side of solve(): acados-style field access (set/get), yref windowing, converters,
// plant step, logged quantities.  Reference (BroilerCompiler/drone-attitude-control):
//   OCP.set_up_ocp        src/force_model/ocp.py:117-122, src/jerk_model/ocp.py:118-123
//   follow_trajectory     src/force_model/controller.py:18-56, src/jerk_model/controller.py:18-58
//   Converter.convert     src/force_model/dynamics.py:66-70, src/jerk_model/dynamics.py:76-83
//   OCP.simulate_next_x   src/force_model/ocp.py:106-115, src/jerk_model/ocp.py:106-116
#pragma once
#include "bnmpc_core.cuh"

namespace bnmpc {

// field ids of the C-ABI (include/bnmpc.h)
enum { F_X = 0, F_U = 1, F_YREF = 2, F_LBX = 3, F_UBX = 4, F_P = 5, F_PI = 6, F_LAM = 7, F_LBU = 8, F_UBU = 9 };
enum { KIND_FORCE = 0, KIND_JERK = 1, KIND_THRUST = 2, KIND_ATT = 3 };
enum { REF_BATCH_MINOR = 0, REF_SHARED = 1, REF_INSTANCE_MAJOR = 2, REF_CIRCLE = 3 };   // bnmpc_closed_loop_args.ref_shared

// which block / local index holds global input g, state g
template <class M> BN_HD constexpr int ublk(int g) { for (int b = 0; b < M::NBLK; b++) for (int j = 0; j < M::NUB; j++) if (M::ug(b, j) == g) return b; return 0; }
template <class M> BN_HD constexpr int uloc(int g) { for (int b = 0; b < M::NBLK; b++) for (int j = 0; j < M::NUB; j++) if (M::ug(b, j) == g) return j; return 0; }
template <class M> BN_HD constexpr int xblk(int g) { for (int b = 0; b < M::NBLK; b++) for (int j = 0; j < M::NXB; j++) if (M::xg(b, j) == g) return b; return 0; }
template <class M> BN_HD constexpr int xloc(int g) { for (int b = 0; b < M::NBLK; b++) for (int j = 0; j < M::NXB; j++) if (M::xg(b, j) == g) return j; return 0; }

// AoS dimension of a field at a stage (0 = not valid there)
BN_HD int field_dim(int NX, int NU, int NP, int field, int stage, int N) {
    switch (field) {
    case F_X: return (stage >= 0 && stage <= N) ? NX : 0;
    case F_U: return (stage >= 0 && stage < N) ? NU : 0;
    case F_YREF: return (stage >= 0 && stage < N) ? NX + NU : (stage == N ? NX : 0);
    case F_LBX: case F_UBX: return (stage >= 0 && stage < N) ? NX : 0;      // stage 0: the x0 embedding; 1..N-1: state box
    case F_LBU: case F_UBU: return (stage >= 0 && stage < N) ? NU : 0;
    case F_P: return NP;
    case F_PI: return (stage >= 0 && stage < N) ? NX : 0;
    case F_LAM: return (stage == 0) ? 2 * NU : ((stage > 0 && stage < N) ? 2 * (NU + NX) : 0);
    }
    return 0;
}

// element j of the AoS vector of (field, stage) <-> its place in the persistent state of instance `inst`
template <class T>
BN_HD T* field_ptr(const Gs<T>& gs, int NX, int NU, int NP, int inst, int field, int k, int j) {
    const int N = gs.N, SG = NU + NX;
    switch (field) {
    case F_X: return gs.V + (size_t)inst * (N + 1) * SG + k * SG + NU + j;
    case F_U: return gs.V + (size_t)inst * (N + 1) * SG + k * SG + j;
    case F_YREF:   // acados order [x-part; u-part] (Vx = [I; 0], Vu = [0; I]), stored as is
        return gs.YREF + (size_t)inst * (N * SG + NX) + k * SG + j;
    case F_LBX: case F_UBX: return gs.X0 + (size_t)inst * NX + j;
    case F_P: return gs.PAR + (size_t)inst * NP + j;
    case F_PI: return gs.PI + (size_t)inst * N * NX + k * NX + j;
    case F_LAM: {  // acados order [lbu, lbx, ubu, ubx]; stage 0 has no x bounds
        const int half = (k == 0) ? NU : SG;
        const int side = j >= half, v = j - side * half;
        return gs.LAM + (size_t)inst * N * 2 * SG + k * 2 * SG + side * SG + v;
    }
    }
    return nullptr;
}

// ---------------------------------------------------------------------------------------------------------------------
// fused closed loop
// ---------------------------------------------------------------------------------------------------------------------
struct LoopArgs {
    int step;            // absolute index of the first control step of this launch (row of ref / noise / logs)
    int n_steps;         // control steps of every instance in this launch (1: one launch per control step)
    int chunk;           // consecutive steps of one instance a warp runs before it hands the instance back to the queue
    int kind;            // KIND_FORCE | KIND_JERK | KIND_THRUST (converter + logged quantities)
    int ref_layout, log_stride, batch, ref_rows;   // ref_layout: REF_BATCH_MINOR | REF_SHARED | REF_INSTANCE_MAJOR | REF_CIRCLE
    size_t Bp;           // stride of the handle-owned state arrays
    const double* ref; const double* noise;
    // noise generated on the device instead of read from `noise`: eps = noise_std * N(0,1) drawn from Philox4x32-10 with
    // key = seed and counter = (global instance id, control step) - see philox_normal()
    unsigned long long noise_seed; double noise_std; long long inst0; int noise_philox;
    double *Xsim, *U_plant, *U_ctrl, *a_log; int32_t *status, *qp_iter;
    // handle-owned loop state
    double *xs, *acc, *cost, *abs_err; const double *p_plant;
    int32_t* fail_count; // [batch] control steps whose solve ended with a non-zero status (sticky until closed_loop_init)
    int* next_step;      // [batch] first control step of the instance that has not been run yet (multi-step launches)
    int ls_generation;   // lockstep kernel: instances of a CTA start their QPs together (see ls_pslot)
    long long* prof;     // debug: CTA 0 records (clock64, masks) at every barrier of the lockstep schedule, prof[0] = count
    int prof_cap;
};

// Philox4x32-10 (Salmon et al., SC'11): counter (c0..c3), key (k0, k1) -> four 32-bit words.  Used for the plant noise
// of reference src/force_model/ocp.py:114-115 (np.random.normal(0, noise)) when the caller does not supply the draws:
// counter = (instance lo, instance hi, step, 0), key = seed, so a draw depends only on (seed, global instance, step) and
// not on the batch size, the sharding or the launch shape.
BN_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    for (int r = 0; r < 10; r++) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// standard normal by Box-Muller from two 53-bit uniforms of one Philox block: u1 in (0, 1], u2 in [0, 1)
BN_HD double philox_normal(unsigned long long seed, long long inst, int step) {
    uint32_t r[4];
    philox4x32_10((uint32_t)inst, (uint32_t)((unsigned long long)inst >> 32), (uint32_t)step, 0u, (uint32_t)seed, (uint32_t)(seed >> 32), r);
    const double two53 = 1.0 / 9007199254740992.0;
    const double u1 = (double)((((uint64_t)r[0] << 32 | r[1]) >> 11) + 1) * two53;
    const double u2 = (double)(((uint64_t)r[2] << 32 | r[3]) >> 11) * two53;
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586476925 * u2);
}

// where the cost reference of instance `inst` at control step `step` comes from
BN_HD YrefSrc loop_yref(int inst, int step, int N, const LoopArgs& a) {
    const size_t Bt = (size_t)a.batch;
    YrefSrc ys;
    ys.yref = nullptr; ys.ref = a.ref; ys.row0 = step; ys.circle_n = 0;
    if (a.ref_layout == REF_CIRCLE) { ys.ref_rs = 0; ys.ref_cs = 0; ys.ref_off = (size_t)inst * 4; ys.circle_n = a.ref_rows - N; }
    else if (a.ref_layout == REF_SHARED) { ys.ref_rs = 8; ys.ref_cs = 1; ys.ref_off = 0; }
    else if (a.ref_layout == REF_INSTANCE_MAJOR) { ys.ref_rs = 8; ys.ref_cs = 1; ys.ref_off = (size_t)inst * a.ref_rows * 8; }
    else { ys.ref_rs = 8 * Bt; ys.ref_cs = Bt; ys.ref_off = (size_t)inst; }
    return ys;
}

// start of a control step of instance `inst`: controller parameters and x0_bar = Xsim[i] (+ a_i for the jerk model),
// controller.py:29-31 / jerk controller.py:30-32.  The caller synchronises the group afterwards.
template <class M, class T, class G, class PS>
BN_HD void loop_begin(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs, const LoopArgs& a) {
    constexpr int NX = M::NX, NP = M::NP;
    T p[NP];
#pragma unroll
    for (int j = 0; j < NP; j++) p[j] = gs.PAR[(size_t)inst * NP + j];
    sv.set_par(p);
    for (int gi = sv.g.lane; gi < NX; gi += G::L)
        sv.X0S(gi) = T(gi < 4 ? ld_cg(a.xs + (size_t)gi * a.Bp + inst) : ld_cg(a.acc + (size_t)(gi - 4) * a.Bp + inst));
}

// end of a control step, on the leader lane of the instance: logged cost, converter, plant step, noise, logs
// (controller.py:37-54 / jerk controller.py:38-56).  With keep_x0 the new plant state also becomes the x0_bar of the next
// step in place (the instance stays on this group for its next control step).
template <class M, class T, class G, class PS>
BN_HD void loop_finish(Solver<M, T, G, PS>& sv, int inst, int step, int status, int qp_it, const YrefSrc& ys, const LoopArgs& a,
                       bool keep_x0) {
    using SL = typename Solver<M, T, G, PS>::SL;
    constexpr int m = M::NUB, NX = M::NX, NU = M::NU, NBLK = M::NBLK;
    const size_t Bp = a.Bp, Bt = (size_t)a.batch;
    if (sv.g.lane == 0) {
        auto refv = [&](int row, int col) -> double {
            if (ys.circle_n > 0) return circle_ref(a.ref + ys.ref_off, row, col, ys.circle_n);
            return a.ref[(size_t)row * ys.ref_rs + (size_t)col * ys.ref_cs + ys.ref_off];
        };
        const int cost_stage = (a.kind == KIND_JERK) ? 1 : 0;   // controller.py:39 get(0,'x') / jerk controller.py:39 get(1,'x')
        double u0[NU], xo[4];
#pragma unroll
        for (int gi = 0; gi < NU; gi++) u0[gi] = double(sv.S(SL::VAL + uloc<M>(gi), ublk<M>(gi)));
#pragma unroll
        for (int gi = 0; gi < 4; gi++) xo[gi] = double(sv.S(SL::VAL + m + xloc<M>(gi), cost_stage * NBLK + xblk<M>(gi)));
        const double pc_mass = double(sv.par[0]);
        double xs[4], pp[2];
#pragma unroll
        for (int j = 0; j < 4; j++) xs[j] = ld_cg(a.xs + (size_t)j * Bp + inst);
        pp[0] = a.p_plant[inst]; pp[1] = a.p_plant[Bp + inst];
        const double wc[4] = {1e2, 1e2, 1.0, 1.0};            // controller.py:40
        double c = 0.0;
#pragma unroll
        for (int j = 0; j < 4; j++) { const double d = xo[j] - refv(step, j); c += wc[j] * d * d; }
        a.cost[inst] = ld_cg(a.cost + inst) + c;
        a.abs_err[inst] = ld_cg(a.abs_err + inst) + (fabs(refv(step, 0) - xs[0]) + fabs(refv(step, 1) - xs[1]));   // store_results.py:233-236
        // a non-zero solver status does not stop the loop (the reference raises, controller.py:33-36): the plant is driven
        // with the u0 of the iterate the solver returned, the step is logged, and the instance's failure count goes up
        if (status != ST_SUCCESS && a.fail_count) a.fail_count[inst] = ld_cg(a.fail_count + inst) + 1;
        double up[2], alog[2];
        if (a.kind == KIND_JERK) {
            double ai[2] = {ld_cg(a.acc + inst), ld_cg(a.acc + Bp + inst)};
            const double hc = sv.o.sim_dt;
            for (int j = 0; j < sv.o.sim_substeps; j++) {     // jerk dynamics.py:76-83 + jerk ocp.py:106-113
                ai[0] += u0[0] * hc; ai[1] += u0[1] * hc;
                const double fx = pc_mass * ai[0], fz = pc_mass * ai[1];
                up[0] = atan2(fx, fz); up[1] = sqrt(fx * fx + fz * fz);
                plant_step<double>(sv.o.sim_erk_stages, pp, hc, up, xs);
            }
            a.acc[inst] = ai[0]; a.acc[Bp + inst] = ai[1];
            alog[0] = ai[0]; alog[1] = ai[1];
            if constexpr (NX >= 6) { if (keep_x0) { sv.X0S(4) = T(ai[0]); sv.X0S(5) = T(ai[1]); } }
        } else if (a.kind == KIND_THRUST) {               // the OCP input already is the plant input (theta, Fd)
            up[0] = u0[0]; up[1] = u0[1];
            for (int j = 0; j < sv.o.sim_substeps; j++) plant_step<double>(sv.o.sim_erk_stages, pp, sv.o.sim_dt, up, xs);
            // logged with the nominal mass drone.MASS like the force path (params.py:42), whatever p_ctrl holds
            alog[0] = u0[1] * sin(u0[0]) / 0.03277; alog[1] = u0[1] * cos(u0[0]) / 0.03277;
        } else {
            up[0] = atan2(u0[0], u0[1]); up[1] = sqrt(u0[0] * u0[0] + u0[1] * u0[1]);     // dynamics.py:66-70
            for (int j = 0; j < sv.o.sim_substeps; j++) plant_step<double>(sv.o.sim_erk_stages, pp, sv.o.sim_dt, up, xs);
            // controller.py:38 divides by the constant drone.MASS (params.py:42) - the nominal mass, whatever p_ctrl holds
            alog[0] = u0[0] / 0.03277; alog[1] = u0[1] / 0.03277;
        }
        double eps = 0.0;                                                                  // ocp.py:114-115
        if (a.noise_philox) eps = a.noise_std * philox_normal(a.noise_seed, a.inst0 + inst, step);
        else if (a.noise) eps = a.noise[(size_t)step * Bt + inst];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            xs[j] += eps; a.xs[(size_t)j * Bp + inst] = xs[j];
            if (keep_x0) sv.X0S(j) = T(xs[j]);
        }
        const size_t l2 = (size_t)step * 2 * Bt + inst;
        if (a.U_ctrl) { a.U_ctrl[l2] = u0[0]; a.U_ctrl[l2 + Bt] = u0[1]; }
        if (a.U_plant) { a.U_plant[l2] = up[0]; a.U_plant[l2 + Bt] = up[1]; }
        if (a.a_log) { a.a_log[l2] = alog[0]; a.a_log[l2 + Bt] = alog[1]; }
        if (a.Xsim) {
#pragma unroll
            for (int j = 0; j < 4; j++) a.Xsim[((size_t)(step + 1) * 4 + j) * Bt + inst] = xs[j];
        }
        if (a.status) a.status[(size_t)step * Bt + inst] = status;
        if (a.qp_iter) a.qp_iter[(size_t)step * Bt + inst] = qp_it;
    }
}

// one instance, one control step, executed by the lanes of the solver's group
template <class M, class T, class G, class PS>
BN_HD void closed_loop_step(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs, const LoopArgs& a) {
    const YrefSrc ys = loop_yref(inst, a.step, sv.N, a);
    loop_begin<M, T>(sv, inst, gs, a);
    sv.g.sync();
    sv.template sqp_solve<T>(inst, gs, ys);
    loop_finish<M, T>(sv, inst, a.step, gs.status[inst], gs.qp_iter[inst], ys, a, false);
    sv.g.sync();
}

// Queue ticket `ticket` of a multi-step launch = (instance, chunk of LoopArgs::chunk consecutive control steps): the
// instance's working set stays on chip for the whole chunk (only the first step loads the persistent state from HBM;
// every step still stores it, which is write-only traffic and keeps the state of the last good solve available to the
// failure path).  `wq` orders the chunks of an instance (ready / publish, see bnmpc_lockstep.cuh).
template <class M, class T, class G, class PS, class WQ>
BN_HD void closed_loop_chunk(Solver<M, T, G, PS>& sv, int ticket, const Gs<T>& gs, const LoopArgs& a, WQ& wq) {
    const int B = gs.B;
    const int c = ticket / B, pos = ticket - c * B;
    const int inst = sv.o.order ? sv.o.order[pos] : pos;
    const int s0 = a.step + c * a.chunk;
    const int s1 = s0 + a.chunk < a.step + a.n_steps ? s0 + a.chunk : a.step + a.n_steps;
    if (c > 0) wq.wait(inst, s0);
    loop_begin<M, T>(sv, inst, gs, a);
    bool have_mult = ld_cg(gs.have_mult + inst) != 0;
    sv.load_state(gs, inst, have_mult);
    sv.g.sync();
    for (int step = s0; step < s1; step++) {
        const YrefSrc ys = loop_yref(inst, step, sv.N, a);
        int sqp_it = 0, qp_it = 0;
        const int status = sv.template sqp_core<T>(ys, have_mult, sqp_it, qp_it);
        sv.store_result(gs, inst, status, sqp_it, qp_it, have_mult);
        const bool more = step + 1 < s1;
        loop_finish<M, T>(sv, inst, step, status, qp_it, ys, a, more);
        sv.g.sync();
        // a failed QP leaves its own multipliers on chip; the next solve starts from those of the last good solve
        if (more && status == ST_QP_FAILURE) { sv.load_state(gs, inst, have_mult); sv.g.sync(); }
    }
    if (s1 < a.step + a.n_steps) wq.publish(inst, s1);
}

// The reference table bound to a handle for the solve() path (bnmpc_set_ref_table + bnmpc_set_yref_row): OCP.set_up_ocp(row,
// xref, uref) with yref_k = table row `row + k`, columns [xref (NX) | uref (NU) | ignored].  ref == nullptr: the yref
// stored in Gs::YREF.  The table is FP64 in both precisions; Solver::yref_at converts what it reads.
struct ApiRef {
    const double* ref;   // [rows][cols] shared by all instances, or [B][rows][cols] (instance-major)
    int rows, cols;
    int shared;          // 1 = one table for all instances, 0 = one table per instance
    int row;             // first row of the window
};

// row `row + k` of instance inst's table
BN_HD const double* api_ref_row(const ApiRef& t, int inst, int k) {
    return t.ref + (t.shared ? (size_t)0 : (size_t)inst * t.rows * t.cols) + (size_t)(t.row + k) * t.cols;
}

// one instance, one ocp_solver.solve() with the x0 / yref / p stored through the API (yref from `tab` when it has a table)
template <class M, class T, class G, class PS>
BN_HD void api_solve(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs, const ApiRef& tab = ApiRef{nullptr, 0, 0, 0, 0}) {
    constexpr int NX = M::NX, NU = M::NU, NP = M::NP;
    YrefSrc ys;
    ys.ref = nullptr; ys.ref_rs = 0; ys.ref_cs = 0; ys.ref_off = 0; ys.row0 = 0; ys.circle_n = 0;
    if (tab.ref) {
        ys.yref = nullptr; ys.ref = tab.ref; ys.ref_rs = (size_t)tab.cols; ys.ref_cs = 1; ys.row0 = tab.row;
        ys.ref_off = tab.shared ? (size_t)0 : (size_t)inst * tab.rows * tab.cols;
    } else {
        ys.yref = gs.YREF + (size_t)inst * (gs.N * (NU + NX) + NX);
    }
    {
        T p[NP];
#pragma unroll
        for (int j = 0; j < NP; j++) p[j] = gs.PAR[(size_t)inst * NP + j];
        sv.set_par(p);
        for (int gi = sv.g.lane; gi < NX; gi += G::L) sv.X0S(gi) = gs.X0[(size_t)inst * NX + gi];
        sv.bnd = gs.BND ? gs.BND + (size_t)inst * gs.N * 2 * (NU + NX) : nullptr;
    }
    sv.g.sync();
    sv.template sqp_solve<T>(inst, gs, ys);
    if (sv.g.lane == 0) {      // ocp_solver.get(0, 'u') for free: the solution is still in shared memory
        using SL = typename Solver<M, T, G, PS>::SL;
#pragma unroll
        for (int gi = 0; gi < NU; gi++) gs.U0[(size_t)inst * NU + gi] = double(sv.S(SL::VAL + uloc<M>(gi), ublk<M>(gi)));
    }
    sv.g.sync();
}

// ---------------------------------------------------------------------------------------------------------------------
// solution sensitivities at the stored solutions (bnmpc_eval_sens_x0 / bnmpc_eval_adjoint_sens), FP64 in and out
// ---------------------------------------------------------------------------------------------------------------------
struct SensArgs {
    int stages;                     // forward: stages 0 .. stages-1 of sens_x, 0 .. min(stages, N)-1 of sens_u
    double *sens_x, *sens_u;        // [B][stages][NX][NX] = d x_k / d x0, [B][min(stages, N)][NU][NX] = d u_k / d x0, or NULL
    const double *seed_x, *seed_u;  // adjoint: [B][N+1][NX], [B][N][NU], NULL = 0
    double *grad_x0, *grad_yref;    // [B][NX], [B][N*(NX+NU) + NX] (the bnmpc_set_yref_all layout), or NULL
};

// Binds the instance and factorises its KKT matrix (Solver::sens_factor).  false: the last solve did not succeed or left no
// multipliers - there is no solution to differentiate and the caller writes NaN rows.
template <class M, class T, class G, class PS>
BN_HD bool sens_begin(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs) {
    constexpr int NX = M::NX, NU = M::NU, NP = M::NP;
    if (gs.status[inst] != ST_SUCCESS || gs.have_mult[inst] == 0) return false;
    T p[NP];
#pragma unroll
    for (int j = 0; j < NP; j++) p[j] = gs.PAR[(size_t)inst * NP + j];
    sv.set_par(p);
    sv.bnd = gs.BND ? gs.BND + (size_t)inst * gs.N * 2 * (NU + NX) : nullptr;
    sv.sens_factor(gs, inst);
    return true;
}

template <class G>
BN_HD void nan_fill(const G& g, double* p, size_t count) {
    if (!p) return;
    for (size_t e = (size_t)g.lane; e < count; e += G::L) p[e] = (double)NAN;
}

// Forward: x0 enters the QP only through b_0 = A_0 (x0 - x_0) (Solver::build_qp), so direction e_j is one Newton solve with
// RB = A_0 e_j at stage 0 and a zero gradient; its step is column j of d(x_k, u_k) / d x0.  sens_x[0] = I.
template <class M, class T, class G, class PS>
BN_HD void api_sens_x0(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs, const SensArgs& a) {
    using SL = typename Solver<M, T, G, PS>::SL;
    constexpr int n = M::NXB, m = M::NUB, s = n + m, NBLK = M::NBLK, NX = M::NX, NU = M::NU;
    const int N = sv.N, ns = a.stages, nsu = a.stages < N ? a.stages : N;
    double* sx = a.sens_x ? a.sens_x + (size_t)inst * ns * NX * NX : nullptr;
    double* su = a.sens_u ? a.sens_u + (size_t)inst * nsu * NU * NX : nullptr;
    if (!sens_begin(sv, inst, gs)) {
        nan_fill(sv.g, sx, (size_t)ns * NX * NX);
        nan_fill(sv.g, su, (size_t)nsu * NU * NX);
        sv.g.sync();
        return;
    }
    for (int j = 0; j < NX; j++) {
        const int bj = xblk<M>(j), lj = xloc<M>(j);
        for (int sb = sv.g.lane; sb < sv.NSB; sb += G::L) {
            const int k = sb / NBLK, b = sb % NBLK;
            sv.use_block(b);
#pragma unroll
            for (int v = 0; v < s; v++) sv.S(SL::GV + v, sb) = T(0);
            if (k < N) {
#pragma unroll
                for (int r = 0; r < n; r++) {
                    T e = T(0);      // A_0[r][lj], selected with constant indices so that A stays in registers
#pragma unroll
                    for (int c = 0; c < n; c++) if (k == 0 && b == bj && c == lj) e = sv.maA(T(0), T(1), r, c);
                    sv.S(SL::RB + r, sb) = e;
                }
            }
        }
        sv.g.sync();
        sv.sens_solve(ns > 2);
        for (int sb = sv.g.lane; sb < sv.NSB; sb += G::L) {
            const int k = sb / NBLK, b = sb % NBLK;
            if (sx && k < ns) {
#pragma unroll
                for (int r = 0; r < n; r++)
                    sx[((size_t)k * NX + M::xg(b, r)) * NX + j] = k == 0 ? (M::xg(b, r) == j ? 1.0 : 0.0) : double(sv.S(SL::DZA + m + r, sb));
            }
            if (su && k < nsu) {
#pragma unroll
                for (int c = 0; c < m; c++) su[((size_t)k * NU + M::ug(b, c)) * NX + j] = double(sv.S(SL::DZA + c, sb));
            }
        }
        sv.g.sync();
    }
}

// Adjoint: the KKT matrix is symmetric, so the Newton solve with the seed as gradient (RB = 0) gives the vector-Jacobian
// products.  With that step (dz, dpi): grad_x0 = seed_x[0] + A_0' dpi_0, and since the cost gradient depends on yref through
// -dt W (stages < N) / -W_e (stage N), grad_yref = -dt W dz / -W_e dz (0 for the x-part of stage 0: x_0 is not a variable).
template <class M, class T, class G, class PS>
BN_HD void api_sens_adj(Solver<M, T, G, PS>& sv, int inst, const Gs<T>& gs, const SensArgs& a) {
    using SL = typename Solver<M, T, G, PS>::SL;
    constexpr int n = M::NXB, m = M::NUB, s = n + m, NBLK = M::NBLK, NX = M::NX, NU = M::NU, ny = NX + NU;
    const int N = sv.N;
    const double* sdx = a.seed_x ? a.seed_x + (size_t)inst * (N + 1) * NX : nullptr;
    const double* sdu = a.seed_u ? a.seed_u + (size_t)inst * N * NU : nullptr;
    double* gx = a.grad_x0 ? a.grad_x0 + (size_t)inst * NX : nullptr;
    double* gy = a.grad_yref ? a.grad_yref + (size_t)inst * (N * ny + NX) : nullptr;
    if (!sens_begin(sv, inst, gs)) {
        nan_fill(sv.g, gx, NX);
        nan_fill(sv.g, gy, (size_t)N * ny + NX);
        sv.g.sync();
        return;
    }
    for (int sb = sv.g.lane; sb < sv.NSB; sb += G::L) {
        const int k = sb / NBLK, b = sb % NBLK;
#pragma unroll
        for (int v = 0; v < s; v++) {
            T sd = T(0);
            if (sv.has(k, v)) {
                if (v < m) { if (sdu) sd = T(sdu[(size_t)k * NU + M::ug(b, v)]); }
                else if (sdx) sd = T(sdx[(size_t)k * NX + M::xg(b, v - m)]);
            }
            sv.S(SL::GV + v, sb) = sd;
        }
        if (k < N) {
#pragma unroll
            for (int r = 0; r < n; r++) sv.S(SL::RB + r, sb) = T(0);
        }
    }
    sv.g.sync();
    sv.sens_solve(gy != nullptr);
    if (gx) {
        for (int b = sv.g.lane; b < NBLK; b += G::L) {
            sv.use_block(b);
            const int sb1 = NBLK + b;
            T dpi[n];       // dpi_0 = p_1 + P_1 dx_1 (the multiplier step of Solver::qp_update)
#pragma unroll
            for (int r = 0; r < n; r++) {
                T d = sv.S(SL::GV + m + r, sb1);
#pragma unroll
                for (int l = 0; l < n; l++) d += sv.S(SL::P + sv.pidx(r, l), sb1) * sv.S(SL::DZA + m + l, sb1);
                dpi[r] = d;
            }
#pragma unroll
            for (int c = 0; c < n; c++) {
                T acc = sdx ? T(sdx[M::xg(b, c)]) : T(0);
#pragma unroll
                for (int r = 0; r < n; r++) acc = sv.maA(acc, dpi[r], r, c);
                gx[M::xg(b, c)] = double(acc);
            }
        }
    }
    if (gy) {
        for (int sb = sv.g.lane; sb < sv.NSB; sb += G::L) {
            const int k = sb / NBLK, b = sb % NBLK;
            sv.use_block(b);
#pragma unroll
            for (int v = 0; v < s; v++) {
                if (v < m && k == N) continue;
                const size_t e = (size_t)k * ny + (v < m ? NX + M::ug(b, v) : M::xg(b, v - m));
                const T h = k < N ? sv.Hd[v] : sv.He[v - m];
                gy[e] = sv.has(k, v) ? double(-h * sv.S(SL::DZA + v, sb)) : 0.0;
            }
        }
    }
    sv.g.sync();
}

}  // namespace bnmpc
