// hostsim_sens - TEST HARNESS ONLY.  The solution-sensitivity path of the product (api_sens_x0 / api_sens_adj of
// csrc/bnmpc_loop.cuh with Solver::sens_factor / sens_solve of csrc/bnmpc_core.cuh, the templates k_sens instantiates) compiled
// for the host CPU, one emulated lane per instance, so that the CPU-only test run can check it against the numpy
// restatement (tests/sens_oracle.py).  Not part of libbnmpc.so.
#define __host__
#define __device__
#define __forceinline__ inline __attribute__((always_inline))
#define __noinline__ __attribute__((noinline))
#include <string.h>
#include <vector>

#include "../../drone_attitude_control_b200/csrc/bnmpc_loop.cuh"

using namespace bnmpc;

namespace {
struct HostGroup {
    static constexpr int L = 1;
    static constexpr bool PAR_SCAN = false;
    int lane = 0;
    template <class T> T max(T v) const { return v; }
    template <class T> T sum(T v) const { return v; }
    bool any(bool p) const { return p; }
    bool all(bool p) const { return p; }
    void sync() const {}
};

// The stored solution given by the caller: x [B][N+1][NX], u [B][N][NU], lam [B][N][2][NU+NX] (the layout of Gs::LAM),
// status / have_mult [B], parameters p [B][2], per-stage bounds [B][N][2][NU+NX] or NULL.
template <class M, class T>
int sens_t(const Opts* o, int mode, int B, const double* p, const double* x, const double* u, const double* lam, const int* status,
           const int* have_mult, const double* bnd, int stages, double* sens_x, double* sens_u, const double* seed_x,
           const double* seed_u, double* grad_x0, double* grad_yref) {
    constexpr int NX = M::NX, NU = M::NU, NP = M::NP, SG = NX + NU;
    const int N = o->N;
    std::vector<T> V((size_t)B * (N + 1) * SG, T(0)), LAM((size_t)B * N * 2 * SG), PAR((size_t)B * NP);
    std::vector<int32_t> st(status, status + B), hm(have_mult, have_mult + B);
    for (int i = 0; i < B; i++) {
        for (int k = 0; k <= N; k++) {
            for (int j = 0; j < NX; j++) V[((size_t)i * (N + 1) + k) * SG + NU + j] = T(x[((size_t)i * (N + 1) + k) * NX + j]);
            if (k < N) for (int j = 0; j < NU; j++) V[((size_t)i * (N + 1) + k) * SG + j] = T(u[((size_t)i * N + k) * NU + j]);
        }
        for (int j = 0; j < NP; j++) PAR[(size_t)i * NP + j] = T(p[(size_t)i * 2 + j]);
    }
    for (size_t e = 0; e < LAM.size(); e++) LAM[e] = T(lam[e]);
    Gs<T> gs;
    memset(&gs, 0, sizeof(gs));
    gs.V = V.data(); gs.LAM = LAM.data(); gs.PAR = PAR.data(); gs.status = st.data(); gs.have_mult = hm.data();
    gs.BND = const_cast<double*>(bnd); gs.B = B; gs.N = N;
    const SensArgs a{stages, sens_x, sens_u, seed_x, seed_u, grad_x0, grad_yref};
    std::vector<T> sm(SmLayout<M, true>::elems(N), T(0));
    HostGroup g;
    const SmemPriv<M, T> ps;
    for (int i = 0; i < B; i++) {
        Solver<M, T, HostGroup, SmemPriv<M, T>> sv(sm.data(), 0, *o, g, ps);
        if (mode == 0) api_sens_x0<M, T>(sv, i, gs, a);
        else api_sens_adj<M, T>(sv, i, gs, a);
    }
    return 0;
}
}  // namespace

extern "C" {
int hss_sizeof_opts(void) { return (int)sizeof(Opts); }
// mode 0: d(x_k, u_k) / d x0 (bnmpc_eval_sens_x0), 1: adjoint (bnmpc_eval_adjoint_sens); model 0 force, 1 jerk, 2 force_dense
int hss_sens(int model, int prec, const Opts* o, int mode, int B, const double* p, const double* x, const double* u, const double* lam,
             const int* status, const int* have_mult, const double* bnd, int stages, double* sens_x, double* sens_u,
             const double* seed_x, const double* seed_u, double* grad_x0, double* grad_yref) {
#define HSS(MODEL, TYPE) return sens_t<MODEL, TYPE>(o, mode, B, p, x, u, lam, status, have_mult, bnd, stages, sens_x, sens_u, seed_x, seed_u, grad_x0, grad_yref)
    switch (model * 2 + prec) {
    case 0: HSS(Model_force, double);
    case 1: HSS(Model_force, float);
    case 2: HSS(Model_jerk, double);
    case 3: HSS(Model_jerk, float);
    case 4: HSS(Model_force_dense, double);
    case 5: HSS(Model_force_dense, float);
    }
#undef HSS
    return -2;
}
}
