// bnmpc_api.cu - the C-ABI of include/bnmpc.h: handle, workspace, staging, kernel launches.  No solver arithmetic here.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/bnmpc.h"
#include "bnmpc_kernels.cuh"

using namespace bnmpc;

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }

#define CK(call)                                                                                                   \
    do {                                                                                                           \
        cudaError_t e_ = (call);                                                                                   \
        if (e_ != cudaSuccess) return fail(BNMPC_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));      \
    } while (0)

struct Handle {
    bnmpc_config cfg;
    Opts opts;
    const ModelOps* ops;
    int batch, device, ctas, warps;    // persistent CTAs per launch (one per SM) and instances per CTA (in flight per SM)
    int wpg;                       // warps per instance of the closed-loop kernel (1 at the reference horizon, 2 / 4 for long horizons)
    int *queue, qi;                // work-queue counters (one per launch, recycled), next counter to use
    int* order;                    // queue position -> instance, refreshed before every launch (longest expected solve first)
    cudaStream_t stream;
    bool own_stream;
    GsAny gs;                      // persistent per-instance state in HBM
    char* gs_base;
    size_t gs_bytes, nV, nPI, nLAM, nYREF;   // elements per instance
    int32_t* ints;                 // status | sqp_iter | qp_iter | have_mult
    double* stage[4];              // device staging buffers for host<->device AoS copies
    size_t stage_cap[4];
    // closed-loop state, stride Bp
    size_t Bp;
    double *xs, *acc, *cost, *abs_err, *p_plant;
    int32_t* fail_count;           // [batch] closed-loop steps with a non-zero solver status since closed_loop_init
    int* next_step;                // [batch] next control step of every instance (orders the step chunks of a multi-step launch)
    int loop_kernel;               // 0: one warp per instance with a work queue (k_loop_step), 1: slotted lockstep (k_loop_ls)
    int chunk_override;            // BNMPC_CHUNK: steps per queue ticket of a multi-step launch (0 = automatic)
    int ls_generation;             // BNMPC_LS_GENERATION: see LoopArgs::ls_generation
    long long* prof; int prof_cap; // bnmpc_debug_profile
    int64_t launches;
    // reference table bound by bnmpc_set_ref_table ([rows][cols], or [batch][rows][cols] when not shared), FP64
    double* tab; size_t tab_cap;   // device copy, its capacity in doubles
    int tab_rows, tab_cols, tab_shared;
    bool tab_sel; int tab_row;     // the table (window at tab_row) is the yref source of the solves, not Gs::YREF
    double* sens_stage; size_t sens_cap;   // device staging of the sensitivity evaluations with host buffers, its capacity in doubles
};

const ModelOps* pick_ops(int model, int precision) {
    switch (model) {
    case BNMPC_MODEL_FORCE: return ops_force(precision);
    case BNMPC_MODEL_JERK: return ops_jerk(precision);
    case BNMPC_MODEL_FORCE_DENSE: return ops_force_dense(precision);
    case BNMPC_MODEL_THRUST: return ops_thrust(precision);
    case BNMPC_MODEL_ATT: return ops_att(precision);
    }
    return nullptr;
}

Opts make_opts(const bnmpc_config& c) {
    Opts o;
    memset(&o, 0, sizeof(o));
    o.N = c.horizon; o.erk_stages = c.erk_stages; o.sqp_max_iter = c.sqp_max_iter; o.qp_max_iter = c.qp_max_iter; o.rti = c.rti;
    o.sim_erk_stages = c.sim_erk_stages; o.sim_substeps = c.sim_substeps; o.dt = c.dt; o.sim_dt = c.sim_dt;
    memcpy(o.W, c.W, sizeof(o.W)); memcpy(o.W_e, c.W_e, sizeof(o.W_e));
    memcpy(o.lbx, c.lbx, sizeof(o.lbx)); memcpy(o.ubx, c.ubx, sizeof(o.ubx));
    memcpy(o.lbu, c.lbu, sizeof(o.lbu)); memcpy(o.ubu, c.ubu, sizeof(o.ubu));
    memcpy(o.tol, c.tol, sizeof(o.tol)); memcpy(o.qp_tol, c.qp_tol, sizeof(o.qp_tol));
    o.mu0 = c.mu0; o.thr0 = c.thr0; o.alpha_min = c.alpha_min; o.lam_min = c.lam_min; o.t_min = c.t_min;
    return o;
}

int use_device(Handle* h) {
    CK(cudaSetDevice(h->device));
    return 0;
}

// device view of a caller buffer of `count` doubles: the pointer itself, or a staged copy of host memory
int stage_in(Handle* h, int slot, const double* p, size_t count, int on_device, const double** out) {
    if (on_device) { *out = p; return 0; }
    if (h->stage_cap[slot] < count) {
        if (h->stage[slot]) CK(cudaFree(h->stage[slot]));
        h->stage[slot] = nullptr; h->stage_cap[slot] = 0;
        CK(cudaMalloc(&h->stage[slot], count * sizeof(double)));
        h->stage_cap[slot] = count;
    }
    CK(cudaMemcpyAsync(h->stage[slot], p, count * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    *out = h->stage[slot];
    return 0;
}

int stage_out_begin(Handle* h, int slot, double* p, size_t count, int on_device, double** dev) {
    if (on_device) { *dev = p; return 0; }
    if (h->stage_cap[slot] < count) {
        if (h->stage[slot]) CK(cudaFree(h->stage[slot]));
        h->stage[slot] = nullptr; h->stage_cap[slot] = 0;
        CK(cudaMalloc(&h->stage[slot], count * sizeof(double)));
        h->stage_cap[slot] = count;
    }
    *dev = h->stage[slot];
    return 0;
}

int stage_out_end(Handle* h, int slot, double* p, size_t count, int on_device) {
    if (on_device) return 0;
    CK(cudaMemcpyAsync(p, h->stage[slot], count * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

// ocp_solver.set / get for all instances: AoS [B][dim] (FP64) <-> persistent state
template <class T, bool TO_STATE>
__global__ void k_field(const __grid_constant__ Gs<T> gs, int NX, int NU, int NP, int field, int stage, double* aos, int dim, int aos_stride) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = (int)(idx / dim), j = (int)(idx % dim);
    if (inst >= gs.B) return;
    T* p = field_ptr(gs, NX, NU, NP, inst, field, stage, j);
    if (TO_STATE) *p = T(aos[(size_t)inst * aos_stride + j]); else aos[(size_t)inst * aos_stride + j] = double(*p);
}

// per-stage bounds [B][N][2][NU+NX]: fill with the configuration's boxes / copy one (stage, side, u|x) slice to or from AoS
__global__ void k_bnd_init(int B, int N, int NX, int NU, const __grid_constant__ Opts o, double* bnd) {
    const int SG = NU + NX;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)B * N * 2 * SG) return;
    const int j = (int)(idx % SG), side = (int)((idx / SG) % 2);
    bnd[idx] = j < NU ? (side ? o.ubu[j] : o.lbu[j]) : (side ? o.ubx[j - NU] : o.lbx[j - NU]);
}
template <bool TO_STATE>
__global__ void k_bnd_field(int B, int N, int NX, int NU, int stage, int side, int is_x, double* bnd, double* aos) {
    const int SG = NU + NX, dim = is_x ? NX : NU;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)B * dim) return;
    const int inst = (int)(idx / dim), j = (int)(idx % dim);
    double* p = bnd + (((size_t)inst * N + stage) * 2 + side) * SG + (is_x ? NU : 0) + j;
    if (TO_STATE) *p = aos[idx]; else aos[idx] = *p;
}

// OCP.set_up_ocp in one call: [B][N*ny + ny_e]
template <class T>
__global__ void k_yref_all(const __grid_constant__ Gs<T> gs, int NX, int NU, int NP, const double* aos) {
    const int ny = NX + NU, per = gs.N * ny + NX;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = (int)(idx / per), e = (int)(idx % per);
    if (inst >= gs.B) return;
    const int k = e < gs.N * ny ? e / ny : gs.N, j = e - k * ny;
    *field_ptr(gs, NX, NU, NP, inst, F_YREF, k, j) = T(aos[idx]);
}

// the window of the bound table -> Gs::YREF, all stages (what bnmpc_set_yref_all of that window stores)
template <class T>
__global__ void k_yref_from_table(const __grid_constant__ Gs<T> gs, int NX, int NU, int NP, const __grid_constant__ ApiRef t) {
    const int ny = NX + NU, per = gs.N * ny + NX;
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = (int)(idx / per), e = (int)(idx % per);
    if (inst >= gs.B) return;
    const int k = e < gs.N * ny ? e / ny : gs.N, j = e - k * ny;
    *field_ptr(gs, NX, NU, NP, inst, F_YREF, k, j) = T(api_ref_row(t, inst, k)[j]);
}
// get(k, 'yref') from the bound table: the values the solve reads (rounded to T), AoS [B][dim]
template <class T>
__global__ void k_yref_table_get(int B, const __grid_constant__ ApiRef t, int k, int dim, double* aos) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int inst = (int)(idx / dim), j = (int)(idx % dim);
    if (inst >= B) return;
    aos[idx] = double(T(api_ref_row(t, inst, k)[j]));
}

// p_ctrl [NP][B] batch-minor -> parameters
template <class T>
__global__ void k_par_from_bm(const __grid_constant__ Gs<T> gs, int NP, const double* p_ctrl) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= gs.B) return;
    for (int j = 0; j < NP; j++) gs.PAR[(size_t)i * NP + j] = T(p_ctrl[(size_t)j * gs.B + i]);
}

template <class T>
cudaError_t launch_field(Handle* h, int field, int stage, double* aos, int dim, int stride, int to_state) {
    const size_t tot = (size_t)h->batch * dim;
    const int grid = (int)((tot + 127) / 128);
    const Gs<T> g = gs_cast<T>(h->gs);
    if (to_state) k_field<T, true><<<grid, 128, 0, h->stream>>>(g, h->ops->nx, h->ops->nu, h->ops->np, field, stage, aos, dim, stride);
    else k_field<T, false><<<grid, 128, 0, h->stream>>>(g, h->ops->nx, h->ops->nu, h->ops->np, field, stage, aos, dim, stride);
    h->launches++;
    return cudaGetLastError();
}
cudaError_t field_xfer(Handle* h, int field, int stage, double* aos, int dim, int stride, int to_state) {
    return h->ops->elem_size == 8 ? launch_field<double>(h, field, stage, aos, dim, stride, to_state)
                                  : launch_field<float>(h, field, stage, aos, dim, stride, to_state);
}

__global__ void k_sim_step(int B, int ns, int nsub, double hstep, const double* x, const double* u, const double* p_plant,
                           const double* eps, double* xn) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    double xs[4], pp[2] = {0.03277, 9.81};
#pragma unroll
    for (int j = 0; j < 4; j++) xs[j] = x[(size_t)i * 4 + j];
    if (p_plant) { pp[0] = p_plant[(size_t)i * 2]; pp[1] = p_plant[(size_t)i * 2 + 1]; }
    for (int j = 0; j < nsub; j++) {
        const double up[2] = {u[((size_t)i * nsub + j) * 2], u[((size_t)i * nsub + j) * 2 + 1]};
        plant_step<double>(ns, pp, hstep, up, xs);
    }
    const double e = eps ? eps[i] : 0.0;
#pragma unroll
    for (int j = 0; j < 4; j++) xn[(size_t)i * 4 + j] = xs[j] + e;
}

// the same for the 3-D attitude model (its plant IS the controller model): x [B][10], u [B][nsub][4]; the noise draw is
// added to position and velocity (the quaternion is left on the unit sphere's neighbourhood the integrator keeps it in)
__global__ void k_sim_step_att(int B, int ns, int nsub, double hstep, const double* x, const double* u, int u_inst, int u_sub, const double* p_plant,
                               const double* eps, double* xn) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    constexpr int NX = Model_att::NX, NU = Model_att::NU;
    double xs[NX], pp[2] = {0.03277, 9.81};
#pragma unroll
    for (int j = 0; j < NX; j++) xs[j] = x[(size_t)i * NX + j];
    if (p_plant) { pp[0] = p_plant[(size_t)i * 2]; pp[1] = p_plant[(size_t)i * 2 + 1]; }
    const FullFn<Model_att, double> fn{pp};
    for (int j = 0; j < nsub; j++) {
        double up[NU], x2[NX], dA[1], dB[1];
#pragma unroll
        for (int c = 0; c < NU; c++) up[c] = u[(size_t)i * u_inst + (size_t)j * u_sub + c];
        erk_dispatch<NX, NU, false>(ns, fn, xs, up, hstep, x2, dA, dB);
#pragma unroll
        for (int c = 0; c < NX; c++) xs[c] = x2[c];
    }
    const double e = eps ? eps[i] : 0.0;
#pragma unroll
    for (int j = 0; j < NX; j++) xn[(size_t)i * NX + j] = xs[j] + (j < 6 ? e : 0.0);
}

// Converter.convert + OCP.simulate_next_x for every instance from the u0 the solve kernel left in gs.U0 (bnmpc_step_for_x0):
// force dynamics.py:66-70 / jerk dynamics.py:76-83, then `nsub` plant sub-steps and the noise draw (ocp.py:106-115).
// x0 [B][nx] = plant state (+ carried acceleration a_i for the jerk model); out_x [B][nx] the same after the step.
__global__ void k_convert_sim(int B, int kind, int nx, int ns, int nsub, double hstep, const double* x0, const double* u0, const double* par_mass,
                              int par_stride, int par_is_float, const double* p_plant, const double* eps, double* out_x, double* out_up) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    double xs[4], pp[2] = {0.03277, 9.81}, up[2] = {0.0, 0.0};
#pragma unroll
    for (int j = 0; j < 4; j++) xs[j] = x0[(size_t)i * nx + j];
    if (p_plant) { pp[0] = p_plant[(size_t)i * 2]; pp[1] = p_plant[(size_t)i * 2 + 1]; }
    const double u[2] = {u0[(size_t)i * 2], u0[(size_t)i * 2 + 1]};
    if (kind == KIND_JERK) {
        const double mass = par_is_float ? (double)((const float*)par_mass)[(size_t)i * par_stride] : par_mass[(size_t)i * par_stride];
        double ai[2] = {x0[(size_t)i * nx + 4], x0[(size_t)i * nx + 5]};
        for (int j = 0; j < nsub; j++) {
            ai[0] += u[0] * hstep; ai[1] += u[1] * hstep;
            const double fx = mass * ai[0], fz = mass * ai[1];
            up[0] = atan2(fx, fz); up[1] = sqrt(fx * fx + fz * fz);
            plant_step<double>(ns, pp, hstep, up, xs);
        }
        out_x[(size_t)i * nx + 4] = ai[0]; out_x[(size_t)i * nx + 5] = ai[1];
    } else {
        if (kind == KIND_THRUST) { up[0] = u[0]; up[1] = u[1]; }
        else { up[0] = atan2(u[0], u[1]); up[1] = sqrt(u[0] * u[0] + u[1] * u[1]); }
        for (int j = 0; j < nsub; j++) plant_step<double>(ns, pp, hstep, up, xs);
    }
    const double e = eps ? eps[i] : 0.0;
#pragma unroll
    for (int j = 0; j < 4; j++) out_x[(size_t)i * nx + j] = xs[j] + e;
    out_up[(size_t)i * 2] = up[0]; out_up[(size_t)i * 2 + 1] = up[1];
}

// gen_circle_traj for every instance, written instance-major [B][rows][8] with the arithmetic the solver uses on the fly
__global__ void k_circle_table(int B, int rows, int n, const double* prm, double* out) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)B * rows * 8) return;
    const int col = (int)(idx % 8), row = (int)((idx / 8) % rows), inst = (int)(idx / ((size_t)rows * 8));
    out[idx] = circle_ref(prm + (size_t)inst * 4, row, col, n);
}

__global__ void k_philox_noise(int B, int n_steps, int first_step, unsigned long long seed, double std_, long long inst0, double* out) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)B * n_steps) return;
    const int i = (int)(idx % B), s = (int)(idx / B);
    out[idx] = std_ * philox_normal(seed, inst0 + i, first_step + s);
}

__global__ void k_fill_int(int n, int v, int* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = v;
}

__global__ void k_loop_init(int B, size_t Bp, const double* x0, const double* p_ctrl, const double* p_plant, double* xs, double* acc,
                            double* cost, double* abs_err, double* pp, int32_t* fail_count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    fail_count[i] = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) xs[(size_t)j * Bp + i] = x0[(size_t)j * B + i];
    acc[i] = 0.0;                                             // jerk controller.py:23  a_i = [0, g]
    acc[Bp + i] = p_ctrl ? p_ctrl[(size_t)B + i] : 9.81;
    cost[i] = 0.0; abs_err[i] = 0.0;
    pp[i] = p_plant ? p_plant[i] : 0.03277;
    pp[Bp + i] = p_plant ? p_plant[(size_t)B + i] : 9.81;
}

__global__ void k_loop_state(int B, size_t Bp, const double* xs, const double* acc, const double* cost, const double* abs_err,
                             double* o_cost, double* o_err, double* o_x, double* o_acc) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    if (o_cost) o_cost[i] = cost[i];
    if (o_err) o_err[i] = abs_err[i];
    if (o_x) for (int j = 0; j < 4; j++) o_x[(size_t)j * B + i] = xs[(size_t)j * Bp + i];
    if (o_acc) for (int j = 0; j < 2; j++) o_acc[(size_t)j * B + i] = acc[(size_t)j * Bp + i];
}

template <class T>
__global__ void k_fma_peak(T* out, int iters) {
    T a[8];
#pragma unroll
    for (int i = 0; i < 8; i++) a[i] = T(threadIdx.x + i) * T(1e-3);
    const T b = T(1.0000001), c = T(1e-7);
    for (int it = 0; it < iters; it++) {
#pragma unroll
        for (int r = 0; r < 8; r++)
#pragma unroll
            for (int i = 0; i < 8; i++) a[i] = a[i] * b + c;
    }
    T s = T(0);
#pragma unroll
    for (int i = 0; i < 8; i++) s += a[i];
    if (s == T(-1)) out[0] = s;   // never true; keeps the chains alive
}

template <class T>
int fma_peak(double* tflops) {
    T* d = nullptr;
    CK(cudaMalloc(&d, sizeof(T)));
    cudaDeviceProp pr;
    int dev = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaGetDeviceProperties(&pr, dev));
    const int blocks = pr.multiProcessorCount * 8, tpb = 256, iters = 4096;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 6; rep++) {
        CK(cudaEventRecord(e0));
        k_fma_peak<T><<<blocks, tpb>>>(d, iters);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        const double fl = 2.0 * 64.0 * iters * (double)blocks * tpb;
        if (rep > 0 && fl / (ms * 1e-3) * 1e-12 > best) best = fl / (ms * 1e-3) * 1e-12;
    }
    CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1)); CK(cudaFree(d));
    *tflops = best;
    return 0;
}

// rcp_vec against the plain division, bit for bit (bnmpc_selftest_rcp)
__device__ __forceinline__ uint64_t mix64(uint64_t x) {
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}
__global__ void k_rcp_check(long long per_thread, int solver_range, unsigned long long* bad) {
    uint64_t sd = mix64((uint64_t)blockIdx.x * blockDim.x + threadIdx.x + 0x1234567ULL * (solver_range + 1));
    unsigned long long nbad = 0;
    for (long long it = 0; it < per_thread; it++) {
        double t[6], r[6];
#pragma unroll
        for (int i = 0; i < 6; i++) {
            sd = mix64(sd + 0x9e3779b97f4a7c15ULL);
            uint64_t bits = sd;
            if (solver_range) bits = (sd & 0x000fffffffffffffULL) | ((uint64_t)(1023 - 47 + (int)((sd >> 52) % 68)) << 52);
            t[i] = __longlong_as_double((long long)bits);
        }
        rcp_vec<double, 6>(t, r);
#pragma unroll
        for (int i = 0; i < 6; i++) {
            const double ref = 1.0 / t[i];
            if (__double_as_longlong(r[i]) != __double_as_longlong(ref) && !(r[i] != r[i] && ref != ref)) nbad++;
        }
    }
    if (nbad) atomicAdd(bad, nbad);
}

constexpr int QUEUE_LEN = 1024;

// counter of the work queue for the next launch; the ring is re-zeroed (stream-ordered) when it wraps
int next_queue(Handle* h, int** q) {
    if (h->qi == QUEUE_LEN) {
        CK(cudaMemsetAsync(h->queue, 0, sizeof(int) * QUEUE_LEN, h->stream));
        h->qi = 0;
    }
    *q = h->queue + h->qi++;
    return 0;
}

// Longest-expected-first order of the work queue: counting sort of the instances by the interior-point iterations (plus
// the SQP iterations, which carry the linearisation) of their previous solve, descending.  One CTA; the order among equal
// keys is arbitrary, which is fine - the order only moves work in time.
__global__ void k_order(const int32_t* __restrict__ qp_iter, const int32_t* __restrict__ sqp_iter, int B, int* __restrict__ order) {
    __shared__ int hist[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        int k = qp_iter[i] + 2 * sqp_iter[i];
        atomicAdd(&hist[k > 255 ? 255 : (k < 0 ? 0 : k)], 1);
    }
    __syncthreads();
    if (threadIdx.x == 0) {            // start of bucket k = number of instances with a larger key
        int run = 0;
        for (int k = 255; k >= 0; k--) { const int c = hist[k]; hist[k] = run; run += c; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        int k = qp_iter[i] + 2 * sqp_iter[i];
        order[atomicAdd(&hist[k > 255 ? 255 : (k < 0 ? 0 : k)], 1)] = i;
    }
}

// refresh the queue order before a launch (only when there are more instances than warps in flight)
int refresh_order(Handle* h) {
    if (!h->opts.order) return 0;
    k_order<<<1, 1024, 0, h->stream>>>(h->gs.qp_iter, h->gs.sqp_iter, h->batch, h->order);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}

// 'lbu' / 'ubu' at any stage and 'lbx' / 'ubx' at stages >= 1 live in per-instance storage that exists only once such a
// field has been set (until then every stage uses the boxes of the configuration and the solve kernels carry no lookup)
bool is_stage_bound(int field, int stage) {
    return field == F_LBU || field == F_UBU || ((field == F_LBX || field == F_UBX) && stage >= 1);
}
int ensure_bounds(Handle* h) {
    if (h->gs.BND) return 0;
    const size_t tot = (size_t)h->batch * h->cfg.horizon * 2 * (h->ops->nu + h->ops->nx);
    CK(cudaMalloc(&h->gs.BND, tot * sizeof(double)));
    k_bnd_init<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->batch, h->cfg.horizon, h->ops->nx, h->ops->nu, h->opts, h->gs.BND);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}
int bound_xfer(Handle* h, int field, int stage, double* aos, int to_state) {
    const int is_x = (field == F_LBX || field == F_UBX), side = (field == F_UBX || field == F_UBU);
    const size_t tot = (size_t)h->batch * (is_x ? h->ops->nx : h->ops->nu);
    const unsigned grid = (unsigned)((tot + 127) / 128);
    if (to_state) k_bnd_field<true><<<grid, 128, 0, h->stream>>>(h->batch, h->cfg.horizon, h->ops->nx, h->ops->nu, stage, side, is_x, h->gs.BND, aos);
    else k_bnd_field<false><<<grid, 128, 0, h->stream>>>(h->batch, h->cfg.horizon, h->ops->nx, h->ops->nu, stage, side, is_x, h->gs.BND, aos);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}

// the yref source of the next solve: the bound table's window, or Gs::YREF
ApiRef api_ref(const Handle* h) {
    if (!h->tab_sel) return ApiRef{nullptr, 0, 0, 0, 0};
    return ApiRef{h->tab, h->tab_rows, h->tab_cols, h->tab_shared, h->tab_row};
}

// selected table -> Gs::YREF (one gather kernel, converting to T), which is the yref source from then on
int materialise_window(Handle* h) {
    if (!h->tab_sel) return 0;
    const ApiRef t = api_ref(h);
    const size_t tot = ((size_t)h->cfg.horizon * (h->ops->nx + h->ops->nu) + h->ops->nx) * h->batch;
    const unsigned grid = (unsigned)((tot + 127) / 128);
    if (h->ops->elem_size == 8) k_yref_from_table<double><<<grid, 128, 0, h->stream>>>(gs_cast<double>(h->gs), h->ops->nx, h->ops->nu, h->ops->np, t);
    else k_yref_from_table<float><<<grid, 128, 0, h->stream>>>(gs_cast<float>(h->gs), h->ops->nx, h->ops->nu, h->ops->np, t);
    CK(cudaGetLastError()); h->launches++;
    h->tab_sel = false;
    return 0;
}

// staging area of a sensitivity evaluation with host buffers: `count` doubles, handle-owned, grown on demand
int sens_staging(Handle* h, size_t count, double** out) {
    if (h->sens_cap < count) {
        CK(cudaStreamSynchronize(h->stream));
        if (h->sens_stage) CK(cudaFree(h->sens_stage));
        h->sens_stage = nullptr; h->sens_cap = 0;
        CK(cudaMalloc(&h->sens_stage, count * sizeof(double)));
        h->sens_cap = count;
    }
    *out = h->sens_stage;
    return 0;
}

int launch_sens(Handle* h, const SensArgs& a, int mode) {
    int* q;
    if (int rc = next_queue(h, &q)) return rc;
    CK(h->ops->sens(h->gs, h->opts, a, mode, h->ctas, h->warps, q, h->stream)); h->launches++;
    return 0;
}

int reset_iterate(Handle* h) {
    const size_t es = h->ops->elem_size, B = h->batch;
    CK(cudaMemsetAsync(h->gs.V, 0, B * h->nV * es, h->stream));
    CK(cudaMemsetAsync(h->gs.PI, 0, B * h->nPI * es, h->stream));
    CK(cudaMemsetAsync(h->gs.LAM, 0, B * h->nLAM * es, h->stream));
    CK(cudaMemsetAsync(h->ints, 0, sizeof(int32_t) * 4 * h->batch, h->stream));
    return 0;
}

}  // namespace

extern "C" {

int bnmpc_version(void) { return BNMPC_VERSION; }
const char* bnmpc_last_error(void) { return g_err.c_str(); }

int bnmpc_config_default(int model, bnmpc_config* c) {
    if (!c) return fail(BNMPC_E_ARG, "cfg is NULL");
    if (model < 0 || model > BNMPC_MODEL_ATT) return fail(BNMPC_E_ARG, "unknown model");
    memset(c, 0, sizeof(*c));
    const bool jerk = (model == BNMPC_MODEL_JERK);
    // reference src/params.py:37-61,113-122
    const double MASS = 0.03277, G = 9.81, GR = G * MASS;
    c->model = model; c->horizon = 30; c->precision = BNMPC_FP64; c->sqp_max_iter = 100; c->qp_max_iter = 50; c->rti = 0;
    c->dt = 1.0 / 50;
    for (int i = 0; i < 4; i++) { c->tol[i] = 1e-6; c->qp_tol[i] = 1e-6; }
    c->mu0 = 1.0; c->thr0 = 0.1; c->alpha_min = 1e-8; c->lam_min = 1e-16; c->t_min = 1e-16;
    const double wx[4] = {1e2, 1e2, 1.0, 1.0};
    if (model == BNMPC_MODEL_ATT) {
        // our 3-D extension, numbers in the spirit of src/force_model/ocp.py:38-78 and src/params.py:45-61: position weight 100,
        // velocity 1, attitude 10 on the vector part of the quaternion (0 on its scalar part), thrust and body rates 0.1;
        // |p| <= 1.2, |v| <= 1, quaternion components within [-1.5, 1.5] (never active), thrust in [0.1, 2] x m g,
        // body rates within +-6 rad/s; ERK4 for the OCP and for the plant
        c->erk_stages = 4;
        const double w[14] = {1e2, 1e2, 1e2, 1.0, 1.0, 1.0, 0.0, 10.0, 10.0, 10.0, 1e-1, 1e-1, 1e-1, 1e-1};
        for (int i = 0; i < 14; i++) c->W[i] = w[i];
        for (int i = 0; i < 10; i++) c->W_e[i] = w[i];
        const double lb[10] = {-1.2, -1.2, -1.2, -1, -1, -1, -1.5, -1.5, -1.5, -1.5};
        for (int i = 0; i < 10; i++) { c->lbx[i] = lb[i]; c->ubx[i] = -lb[i]; }
        c->lbu[0] = 0.1 * GR; c->ubu[0] = 2.0 * GR;
        for (int i = 1; i < 4; i++) { c->lbu[i] = -6.0; c->ubu[i] = 6.0; }
        c->sim_erk_stages = 4; c->sim_substeps = 1; c->sim_dt = c->dt;
        return 0;
    }
    for (int i = 0; i < 4; i++) { c->W[i] = wx[i]; c->W_e[i] = wx[i]; }
    if (jerk) {
        // src/jerk_model/ocp.py:27-79, 84-92, 97-104
        c->erk_stages = 1;
        c->W[4] = c->W[5] = 0.0; c->W[6] = c->W[7] = 1e-1;
        const double lb[6] = {-1.2, -1.2, -1, -1, -5, -5 + G}, ub[6] = {1.2, 1.2, 1, 1, 5, 5 + G};
        memcpy(c->lbx, lb, sizeof(lb)); memcpy(c->ubx, ub, sizeof(ub));
        c->lbu[0] = c->lbu[1] = -5; c->ubu[0] = c->ubu[1] = 5;
        c->sim_erk_stages = 1; c->sim_substeps = 10; c->sim_dt = 1.0 / 500;
    } else {
        // src/force_model/ocp.py:28-78, 83-93, 98-104
        c->erk_stages = 4;
        c->W[4] = c->W[5] = 1e-1;
        const double lb[4] = {-1.2, -1.2, -1, -1}, ub[4] = {1.2, 1.2, 1, 1};
        memcpy(c->lbx, lb, sizeof(lb)); memcpy(c->ubx, ub, sizeof(ub));
        c->lbu[0] = c->lbu[1] = -0.2 * GR; c->ubu[0] = c->ubu[1] = 1.3 * GR;
        c->sim_erk_stages = 4; c->sim_substeps = 1; c->sim_dt = c->dt;
        if (model == BNMPC_MODEL_THRUST) {   // our nonlinear extension: u = (theta, Fd)
            c->lbu[0] = -1.0; c->ubu[0] = 1.0; c->lbu[1] = 0.05; c->ubu[1] = 0.6;
        }
    }
    return 0;
}


int bnmpc_create(const bnmpc_config* cfg, int batch, int device, void** handle) {
    if (!cfg || !handle) return fail(BNMPC_E_ARG, "NULL argument");
    if (batch < 1) return fail(BNMPC_E_ARG, "batch must be >= 1");
    if (cfg->horizon < 1 || cfg->horizon > 1024) return fail(BNMPC_E_ARG, "horizon out of range");
    if (cfg->erk_stages < 0 || cfg->erk_stages > 4 || cfg->sim_erk_stages < 1 || cfg->sim_erk_stages > 4)
        return fail(BNMPC_E_ARG, "erk_stages must be 0 (implicit Gauss-Legendre) or 1..4, sim_erk_stages 1..4");
    if (cfg->precision != BNMPC_FP64 && cfg->precision != BNMPC_FP32) return fail(BNMPC_E_ARG, "unknown precision");
    const ModelOps* ops = pick_ops(cfg->model, cfg->precision);
    if (!ops) return fail(BNMPC_E_ARG, "unknown model");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1)
        return fail(BNMPC_E_CUDA, "no CUDA device: libbnmpc has no CPU path");
    if (device < 0 || device >= ndev) return fail(BNMPC_E_ARG, "device index out of range");
    if (ops->smem_bytes(cfg->horizon) > 226 * 1024 || ops->tmem_cols(cfg->horizon, 1, 1) == 0)
        return fail(BNMPC_E_UNSUPPORTED, "horizon too long: the working set of one instance exceeds 227 KB of shared memory or 512 tensor-memory columns");
    CK(cudaSetDevice(device));
    Handle* h = new Handle();
    memset(h, 0, sizeof(*h));
    h->cfg = *cfg; h->opts = make_opts(*cfg); h->ops = ops; h->batch = batch; h->device = device;
    // from here on every failure path releases the handle
#define CKH(call)                                                                                                    \
    do {                                                                                                             \
        cudaError_t e_ = (call);                                                                                     \
        if (e_ != cudaSuccess) {                                                                                     \
            const std::string m_ = std::string(#call) + ": " + cudaGetErrorString(e_);                               \
            bnmpc_destroy(h);                                                                                        \
            return fail(BNMPC_E_CUDA, m_);                                                                           \
        }                                                                                                            \
    } while (0)
    CKH(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->own_stream = true;
    const size_t SGd = ops->nu + ops->nx, Nn = cfg->horizon, es = ops->elem_size;
    h->nV = (Nn + 1) * SGd; h->nPI = Nn * ops->nx; h->nLAM = Nn * 2 * SGd;
    h->nYREF = Nn * SGd + ops->nx;
    const size_t per = h->nV + h->nYREF + h->nPI + h->nLAM + ops->nx + ops->np;
    h->gs_bytes = per * batch * es;
    h->Bp = ((size_t)batch + 31) / 32 * 32;
    bool ok = cudaMalloc(&h->gs_base, h->gs_bytes) == cudaSuccess;
    ok = ok && cudaMalloc(&h->ints, sizeof(int32_t) * 4 * batch) == cudaSuccess;
    ok = ok && cudaMalloc(&h->queue, sizeof(int) * QUEUE_LEN) == cudaSuccess;
    ok = ok && cudaMalloc(&h->xs, sizeof(double) * 11 * h->Bp) == cudaSuccess;
    ok = ok && cudaMalloc(&h->gs.U0, sizeof(double) * (size_t)batch * ops->nu) == cudaSuccess;
    ok = ok && cudaMalloc(&h->order, sizeof(int) * (size_t)batch) == cudaSuccess;
    ok = ok && cudaMalloc(&h->fail_count, sizeof(int32_t) * (size_t)batch) == cudaSuccess;
    ok = ok && cudaMalloc(&h->next_step, sizeof(int) * (size_t)batch) == cudaSuccess;
    if (!ok) {
        const std::string msg = std::string("cudaMalloc failed: ") + cudaGetErrorString(cudaGetLastError());
        bnmpc_destroy(h);
        return fail(BNMPC_E_CUDA, msg);
    }
    h->acc = h->xs + 4 * h->Bp; h->cost = h->acc + 2 * h->Bp; h->abs_err = h->cost + h->Bp; h->p_plant = h->abs_err + h->Bp;
    {
        char* p = h->gs_base;
        h->gs.V = p; p += h->nV * batch * es; h->gs.PI = p; p += h->nPI * batch * es; h->gs.LAM = p; p += h->nLAM * batch * es;
        h->gs.YREF = p; p += h->nYREF * batch * es; h->gs.X0 = p; p += (size_t)ops->nx * batch * es; h->gs.PAR = p;
    }
    h->gs.status = h->ints; h->gs.sqp_iter = h->ints + batch; h->gs.qp_iter = h->ints + 2 * batch; h->gs.have_mult = h->ints + 3 * batch;
    h->gs.B = batch; h->gs.N = cfg->horizon;
    {
        int warps = 0;
        cudaDeviceProp pr;
        CKH(cudaGetDeviceProperties(&pr, device));
        int wpg = 1;
        CKH(ops->cta_shape(cfg->horizon, &warps, &wpg));
        if (warps < 1) { bnmpc_destroy(h); return fail(BNMPC_E_UNSUPPORTED, "kernel does not fit on an SM for this horizon"); }
        if (const char* e = getenv("BNMPC_WARPS_PER_SM")) {     // tuning knob: fewer instances in flight per SM than would fit
            const int v = atoi(e);
            if (v >= 1 && v < warps) warps = v;
        }
        if (batch < warps * pr.multiProcessorCount)             // small batches spread over the SMs instead of filling a few
            warps = (batch + pr.multiProcessorCount - 1) / pr.multiProcessorCount;
        h->warps = warps;
        // warps per instance of the closed-loop kernel: with few instances per SM (long horizon, or a small batch spread over
        // the SMs) each one gets a group of 2 or 4 warps for its 32-lane passes, up to the launch bound and the tensor memory
        wpg = 1;
        int optin = 0;
        CKH(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
        for (int g = ops->max_wpg; g >= 2; g /= 2) {
            const long stat = ops->loop_static_bytes(g);           // (the group kernels carry the scans' exchange area)
            if (warps * g <= ops->max_warps && ops->tmem_cols(cfg->horizon, warps * g, g) != 0 && stat >= 0 &&
                (size_t)warps * ops->smem_bytes(cfg->horizon) + (size_t)stat <= (size_t)optin) { wpg = g; break; }
        }
        if (const char* e = getenv("BNMPC_WARPS_PER_INSTANCE")) {   // tuning knob: 1 switches the warp groups off
            const int v = atoi(e);
            if (v >= 1 && v < wpg) wpg = (v >= 2) ? 2 : 1;
        }
        h->wpg = wpg;
        const int want = (batch + warps - 1) / warps;
        h->ctas = want < pr.multiProcessorCount ? want : pr.multiProcessorCount;
        // longest-first order: pays from about two instances per warp on (measured: +3 % at 3.5 per warp, +5 % for the jerk
        // model at 2.3, -2 % at 1.7 where the extra launch costs more than the shorter tail saves)
        h->opts.order = (batch > 2 * h->ctas * warps && !getenv("BNMPC_NO_ORDER")) ? h->order : nullptr;
    }
    CKH(cudaMemsetAsync(h->queue, 0, sizeof(int) * QUEUE_LEN, h->stream));
    h->qi = 0;
    CKH(cudaMemsetAsync(h->gs_base, 0, h->gs_bytes, h->stream));
    CKH(cudaMemsetAsync(h->ints, 0, sizeof(int32_t) * 4 * batch, h->stream));
    CKH(cudaMemsetAsync(h->xs, 0, sizeof(double) * 11 * h->Bp, h->stream));
    CKH(cudaMemsetAsync(h->fail_count, 0, sizeof(int32_t) * batch, h->stream));
    CKH(cudaMemsetAsync(h->next_step, 0, sizeof(int) * batch, h->stream));
    h->loop_kernel = 0;
    if (const char* e = getenv("BNMPC_LOOP_KERNEL")) h->loop_kernel = (strcmp(e, "ls") == 0) ? 1 : 0;
    if (const char* e = getenv("BNMPC_CHUNK")) h->chunk_override = atoi(e);
    if (const char* e = getenv("BNMPC_LS_GENERATION")) h->ls_generation = atoi(e);
    // nominal parameters p = (mass, g) for every instance (reference src/params.py:37,42)
    double* pnom = nullptr;
    const double pn[2] = {0.03277, 9.81};
    { const double* d; int rc = stage_in(h, 0, pn, 2, 0, &d); if (rc) { bnmpc_destroy(h); return rc; } pnom = const_cast<double*>(d); }
    CKH(field_xfer(h, F_P, 0, pnom, ops->np, 0, 1));
    CKH(cudaStreamSynchronize(h->stream));
#undef CKH
    *handle = h;
    return 0;
}

int bnmpc_destroy(void* handle) {
    Handle* h = (Handle*)handle;
    if (!h) return 0;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->gs_base) cudaFree(h->gs_base);
    if (h->ints) cudaFree(h->ints);
    if (h->queue) cudaFree(h->queue);
    if (h->order) cudaFree(h->order);
    if (h->fail_count) cudaFree(h->fail_count);
    if (h->next_step) cudaFree(h->next_step);
    if (h->xs) cudaFree(h->xs);
    if (h->gs.U0) cudaFree(h->gs.U0);
    if (h->gs.BND) cudaFree(h->gs.BND);
    if (h->tab) cudaFree(h->tab);
    if (h->sens_stage) cudaFree(h->sens_stage);
    for (int i = 0; i < 4; i++) if (h->stage[i]) cudaFree(h->stage[i]);
    if (h->own_stream && h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return 0;
}

int bnmpc_set_stream(void* handle, void* cuda_stream) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (use_device(h)) return BNMPC_E_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    if (h->own_stream) { CK(cudaStreamDestroy(h->stream)); h->own_stream = false; }
    h->stream = (cudaStream_t)cuda_stream;
    return 0;
}

int bnmpc_synchronize(void* handle) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (use_device(h)) return BNMPC_E_CUDA;
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_dims(void* handle, int32_t dims[7]) {
    Handle* h = (Handle*)handle;
    if (!h || !dims) return fail(BNMPC_E_ARG, "NULL argument");
    dims[0] = h->ops->nx; dims[1] = h->ops->nu; dims[2] = h->ops->nx + h->ops->nu; dims[3] = h->ops->nx;
    dims[4] = h->cfg.horizon; dims[5] = h->ops->np; dims[6] = h->ops->nblk;
    return 0;
}

int64_t bnmpc_workspace_bytes(void* handle) {
    Handle* h = (Handle*)handle;
    return h ? (int64_t)(h->gs_bytes + sizeof(int32_t) * 4 * h->batch + sizeof(double) * 11 * h->Bp + sizeof(double) * h->tab_cap +
                         sizeof(double) * h->sens_cap) : 0;
}

int bnmpc_set(void* handle, int stage, int field, const double* value, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !value) return fail(BNMPC_E_ARG, "NULL argument");
    if (field < BNMPC_F_X || field > BNMPC_F_UBU) return fail(BNMPC_E_FIELD, "unknown field");
    if (field == BNMPC_F_PI || field == BNMPC_F_LAM) return fail(BNMPC_E_FIELD, "field is read-only");
    const int dim = field_dim(h->ops->nx, h->ops->nu, h->ops->np, field, stage, h->cfg.horizon);
    if (dim <= 0) return fail(BNMPC_E_STAGE, "field does not exist at this stage");
    if (use_device(h)) return BNMPC_E_CUDA;
    const double* d;
    if (int rc = stage_in(h, 0, value, (size_t)h->batch * dim, on_device, &d)) return rc;
    if (is_stage_bound(field, stage)) {
        if (int rc = ensure_bounds(h)) return rc;
        return bound_xfer(h, field, stage, const_cast<double*>(d), 1);
    }
    if (field == F_YREF)           // one stage of the table's window: the whole window becomes the stored yref first
        if (int rc = materialise_window(h)) return rc;
    CK(field_xfer(h, field, stage, const_cast<double*>(d), dim, dim, 1));
    return 0;
}

int bnmpc_get(void* handle, int stage, int field, double* out, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !out) return fail(BNMPC_E_ARG, "NULL argument");
    if (field < BNMPC_F_X || field > BNMPC_F_UBU) return fail(BNMPC_E_FIELD, "unknown field");
    const int dim = field_dim(h->ops->nx, h->ops->nu, h->ops->np, field, stage, h->cfg.horizon);
    if (dim <= 0) return fail(BNMPC_E_STAGE, "field does not exist at this stage");
    if (use_device(h)) return BNMPC_E_CUDA;
    double* d;
    if (int rc = stage_out_begin(h, 1, out, (size_t)h->batch * dim, on_device, &d)) return rc;
    if (is_stage_bound(field, stage)) {          // (reading a bound materialises the storage: it then holds the configuration's boxes)
        if (int rc = ensure_bounds(h)) return rc;
        if (int rc = bound_xfer(h, field, stage, d, 0)) return rc;
        return stage_out_end(h, 1, out, (size_t)h->batch * dim, on_device);
    }
    if (field == F_YREF && h->tab_sel) {           // read straight from the table: no handle state changes
        const size_t tot = (size_t)h->batch * dim;
        const unsigned grid = (unsigned)((tot + 127) / 128);
        if (h->ops->elem_size == 8) k_yref_table_get<double><<<grid, 128, 0, h->stream>>>(h->batch, api_ref(h), stage, dim, d);
        else k_yref_table_get<float><<<grid, 128, 0, h->stream>>>(h->batch, api_ref(h), stage, dim, d);
        CK(cudaGetLastError()); h->launches++;
        return stage_out_end(h, 1, out, (size_t)h->batch * dim, on_device);
    }
    CK(field_xfer(h, field, stage, d, dim, dim, 0));
    return stage_out_end(h, 1, out, (size_t)h->batch * dim, on_device);
}

int bnmpc_set_yref_all(void* handle, const double* value, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !value) return fail(BNMPC_E_ARG, "NULL argument");
    if (use_device(h)) return BNMPC_E_CUDA;
    h->tab_sel = false;            // the uploaded window is the yref source again
    const int N = h->cfg.horizon;
    const size_t per = (size_t)N * (h->ops->nx + h->ops->nu) + h->ops->nx;
    if (h->ops->elem_size == 8) {   // the state keeps yref in exactly this layout: a plain copy, no kernel
        CK(cudaMemcpyAsync(h->gs.YREF, value, per * h->batch * sizeof(double), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
        return 0;
    }
    const double* d;
    if (int rc = stage_in(h, 2, value, per * h->batch, on_device, &d)) return rc;
    {
        const size_t tot = per * h->batch;
        const int grid = (int)((tot + 127) / 128);
        k_yref_all<float><<<grid, 128, 0, h->stream>>>(gs_cast<float>(h->gs), h->ops->nx, h->ops->nu, h->ops->np, d);   // (FP64 returned above)
        CK(cudaGetLastError()); h->launches++;
    }
    return 0;
}

int bnmpc_set_ref_table(void* handle, const double* table, int rows, int cols, int layout, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (table) {
        if (layout != 1 && layout != 2) return fail(BNMPC_E_ARG, "layout must be 1 (one [rows][cols] table shared by all instances) or 2 ([batch][rows][cols], instance-major)");
        if (cols < h->ops->nx + h->ops->nu) return fail(BNMPC_E_ARG, "cols must be >= nx + nu: a row is [xref | uref | ignored]");
        if (rows < h->cfg.horizon + 1) return fail(BNMPC_E_ARG, "rows must be >= N + 1: a window is N + 1 rows");
    }
    if (use_device(h)) return BNMPC_E_CUDA;
    // the window the next solve would read stays what it is: if the old table is selected it becomes the stored yref
    if (int rc = materialise_window(h)) return rc;
    if (!table) {
        if (h->tab) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(h->tab)); }
        h->tab = nullptr; h->tab_cap = 0; h->tab_rows = h->tab_cols = 0;
        return 0;
    }
    const size_t count = (size_t)(layout == 1 ? 1 : h->batch) * rows * cols;
    if (h->tab_cap < count) {
        CK(cudaStreamSynchronize(h->stream));         // (kernels already enqueued may still read the old table)
        if (h->tab) CK(cudaFree(h->tab));
        h->tab = nullptr; h->tab_cap = 0;
        CK(cudaMalloc(&h->tab, count * sizeof(double)));
        h->tab_cap = count;
    }
    h->tab_rows = rows; h->tab_cols = cols; h->tab_shared = layout == 1;
    CK(cudaMemcpyAsync(h->tab, table, count * sizeof(double), on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));             // the caller's buffer is free when this returns
    return 0;
}

int bnmpc_set_yref_row(void* handle, int row) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (!h->tab) return fail(BNMPC_E_ARG, "no reference table bound (bnmpc_set_ref_table)");
    if (row < 0 || row + h->cfg.horizon >= h->tab_rows) return fail(BNMPC_E_ARG, "row out of range: needs 0 <= row and row + N < rows");
    h->tab_sel = true; h->tab_row = row;
    return 0;
}

int bnmpc_reset(void* handle) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (use_device(h)) return BNMPC_E_CUDA;
    return reset_iterate(h);
}

int bnmpc_solve(void* handle) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (use_device(h)) return BNMPC_E_CUDA;
    if (int rc = refresh_order(h)) return rc;
    int* q;
    if (int rc = next_queue(h, &q)) return rc;
    CK((h->gs.BND ? h->ops->solve_sb : h->ops->solve)(h->gs, h->opts, api_ref(h), h->ctas, h->warps, q, h->stream)); h->launches++;
    return 0;
}

int bnmpc_solve_for_x0(void* handle, const double* x0, double* u0, int32_t* status, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !x0) return fail(BNMPC_E_ARG, "NULL argument");
    if (use_device(h)) return BNMPC_E_CUDA;
    const int B = h->batch, nx = h->ops->nx, nu = h->ops->nu;
    if (on_device < 0 || on_device > BNMPC_HOST_ASYNC) return fail(BNMPC_E_ARG, "on_device must be 0, 1 or BNMPC_HOST_ASYNC");
    const cudaMemcpyKind in = on_device == 1 ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    const cudaMemcpyKind out = on_device == 1 ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    if (h->ops->elem_size == 8) {
        CK(cudaMemcpyAsync(h->gs.X0, x0, sizeof(double) * B * nx, in, h->stream));            // lbx_0 = ubx_0 = x0_bar
    } else {
        const double* d;
        if (int rc = stage_in(h, 0, x0, (size_t)B * nx, on_device == 1, &d)) return rc;
        CK(field_xfer(h, F_LBX, 0, const_cast<double*>(d), nx, nx, 1));
    }
    if (int rc = refresh_order(h)) return rc;
    int* q;
    if (int rc = next_queue(h, &q)) return rc;
    CK((h->gs.BND ? h->ops->solve_sb : h->ops->solve)(h->gs, h->opts, api_ref(h), h->ctas, h->warps, q, h->stream)); h->launches++;
    if (u0) CK(cudaMemcpyAsync(u0, h->gs.U0, sizeof(double) * B * nu, out, h->stream));   // gathered by the solve kernel
    if (status) CK(cudaMemcpyAsync(status, h->gs.status, sizeof(int32_t) * B, out, h->stream));
    if (!on_device) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_eval_sens_x0(void* handle, int stages, double* sens_x, double* sens_u, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (!h->ops->sens) return fail(BNMPC_E_UNSUPPORTED, "solution sensitivities need the exact Hessian of the Lagrangian: models FORCE, JERK and FORCE_DENSE only");
    const int N = h->cfg.horizon;
    if (stages < 1 || stages > N + 1) return fail(BNMPC_E_ARG, "stages must be within 1 .. N+1");
    if (on_device != 0 && on_device != 1) return fail(BNMPC_E_ARG, "on_device must be 0 or 1");
    if (use_device(h)) return BNMPC_E_CUDA;
    const size_t B = h->batch, nx = h->ops->nx, nu = h->ops->nu;
    const size_t nsx = sens_x ? B * stages * nx * nx : 0, nsu = sens_u ? B * (stages < N ? stages : N) * nu * nx : 0;
    SensArgs a{stages, sens_x, sens_u, nullptr, nullptr, nullptr, nullptr};
    double* d = nullptr;
    if (!on_device) {
        if (int rc = sens_staging(h, nsx + nsu, &d)) return rc;
        a.sens_x = sens_x ? d : nullptr; a.sens_u = sens_u ? d + nsx : nullptr;
    }
    if (int rc = launch_sens(h, a, 0)) return rc;
    if (on_device) return 0;
    if (sens_x) CK(cudaMemcpyAsync(sens_x, d, nsx * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sens_u) CK(cudaMemcpyAsync(sens_u, d + nsx, nsu * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_eval_sens_p(void* handle, int stages, double* sens_x, double* sens_u, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (!h->ops->sens) return fail(BNMPC_E_UNSUPPORTED, "solution sensitivities need the exact Hessian of the Lagrangian: models FORCE, JERK and FORCE_DENSE only");
    const int N = h->cfg.horizon;
    if (stages < 1 || stages > N + 1) return fail(BNMPC_E_ARG, "stages must be within 1 .. N+1");
    if (on_device != 0 && on_device != 1) return fail(BNMPC_E_ARG, "on_device must be 0 or 1");
    if (use_device(h)) return BNMPC_E_CUDA;
    const size_t B = h->batch, nx = h->ops->nx, nu = h->ops->nu, np = h->ops->np;
    const size_t nsx = sens_x ? B * stages * nx * np : 0, nsu = sens_u ? B * (stages < N ? stages : N) * nu * np : 0;
    SensArgs a{stages, sens_x, sens_u, nullptr, nullptr, nullptr, nullptr, nullptr};
    double* d = nullptr;
    if (!on_device) {
        if (int rc = sens_staging(h, nsx + nsu, &d)) return rc;
        a.sens_x = sens_x ? d : nullptr; a.sens_u = sens_u ? d + nsx : nullptr;
    }
    if (int rc = launch_sens(h, a, 2)) return rc;
    if (on_device) return 0;
    if (sens_x) CK(cudaMemcpyAsync(sens_x, d, nsx * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (sens_u) CK(cudaMemcpyAsync(sens_u, d + nsx, nsu * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_eval_adjoint_sens_p(void* handle, const double* seed_x, const double* seed_u, double* grad_x0, double* grad_yref,
                              double* grad_p, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (!h->ops->sens) return fail(BNMPC_E_UNSUPPORTED, "solution sensitivities need the exact Hessian of the Lagrangian: models FORCE, JERK and FORCE_DENSE only");
    if (!seed_x && !seed_u) return fail(BNMPC_E_ARG, "seed_x and seed_u are both NULL");
    if (on_device != 0 && on_device != 1) return fail(BNMPC_E_ARG, "on_device must be 0 or 1");
    if (use_device(h)) return BNMPC_E_CUDA;
    const size_t B = h->batch, nx = h->ops->nx, nu = h->ops->nu, N = h->cfg.horizon, np = h->ops->np;
    const size_t nsx = seed_x ? B * (N + 1) * nx : 0, nsu = seed_u ? B * N * nu : 0;
    const size_t ngx = grad_x0 ? B * nx : 0, ngy = grad_yref ? B * (N * (nx + nu) + nx) : 0, ngp = grad_p ? B * np : 0;
    SensArgs a{0, nullptr, nullptr, seed_x, seed_u, grad_x0, grad_yref, grad_p};
    double* d = nullptr;
    if (!on_device) {       // one staging area: seed_x | seed_u | grad_x0 | grad_yref | grad_p
        if (int rc = sens_staging(h, nsx + nsu + ngx + ngy + ngp, &d)) return rc;
        if (seed_x) CK(cudaMemcpyAsync(d, seed_x, nsx * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        if (seed_u) CK(cudaMemcpyAsync(d + nsx, seed_u, nsu * sizeof(double), cudaMemcpyHostToDevice, h->stream));
        a.seed_x = seed_x ? d : nullptr; a.seed_u = seed_u ? d + nsx : nullptr;
        a.grad_x0 = grad_x0 ? d + nsx + nsu : nullptr; a.grad_yref = grad_yref ? d + nsx + nsu + ngx : nullptr;
        a.grad_p = grad_p ? d + nsx + nsu + ngx + ngy : nullptr;
    }
    if (int rc = launch_sens(h, a, grad_p ? 3 : 1)) return rc;
    if (on_device) return 0;
    if (grad_x0) CK(cudaMemcpyAsync(grad_x0, a.grad_x0, ngx * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (grad_yref) CK(cudaMemcpyAsync(grad_yref, a.grad_yref, ngy * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    if (grad_p) CK(cudaMemcpyAsync(grad_p, a.grad_p, ngp * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_eval_adjoint_sens(void* handle, const double* seed_x, const double* seed_u, double* grad_x0, double* grad_yref, int on_device) {
    return bnmpc_eval_adjoint_sens_p(handle, seed_x, seed_u, grad_x0, grad_yref, nullptr, on_device);
}

int bnmpc_step_for_x0(void* handle, const double* x0, const double* eps, const double* p_plant, double* u0, double* u_plant,
                      int32_t* status, double* x_next, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !x0 || !x_next) return fail(BNMPC_E_ARG, "NULL argument");
    if (on_device < 0 || on_device > BNMPC_HOST_ASYNC) return fail(BNMPC_E_ARG, "on_device must be 0, 1 or BNMPC_HOST_ASYNC");
    if (use_device(h)) return BNMPC_E_CUDA;
    const int B = h->batch, nx = h->ops->nx, nu = h->ops->nu;
    const bool dev = on_device == 1;
    const cudaMemcpyKind out = dev ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    // inputs: x0 | p_plant | eps in one staging buffer (host modes)
    const size_t n0 = (size_t)B * nx, n1 = p_plant ? (size_t)B * 2 : 0, n2 = eps ? (size_t)B : 0;
    const double *dx = x0, *dp = p_plant, *de = eps;
    if (!dev) {
        if (h->stage_cap[3] < n0 + n1 + n2) {
            if (h->stage[3]) CK(cudaFree(h->stage[3]));
            h->stage[3] = nullptr; h->stage_cap[3] = 0;
            CK(cudaMalloc(&h->stage[3], (n0 + n1 + n2) * sizeof(double)));
            h->stage_cap[3] = n0 + n1 + n2;
        }
        double* d = h->stage[3];
        CK(cudaMemcpyAsync(d, x0, n0 * 8, cudaMemcpyHostToDevice, h->stream));
        if (p_plant) CK(cudaMemcpyAsync(d + n0, p_plant, n1 * 8, cudaMemcpyHostToDevice, h->stream));
        if (eps) CK(cudaMemcpyAsync(d + n0 + n1, eps, n2 * 8, cudaMemcpyHostToDevice, h->stream));
        dx = d; dp = p_plant ? d + n0 : nullptr; de = eps ? d + n0 + n1 : nullptr;
    }
    // lbx_0 = ubx_0 = x0_bar
    if (h->ops->elem_size == 8) CK(cudaMemcpyAsync(h->gs.X0, dx, n0 * 8, cudaMemcpyDeviceToDevice, h->stream));
    else CK(field_xfer(h, F_LBX, 0, const_cast<double*>(dx), nx, nx, 1));
    if (int rc = refresh_order(h)) return rc;
    int* q;
    if (int rc = next_queue(h, &q)) return rc;
    CK((h->gs.BND ? h->ops->solve_sb : h->ops->solve)(h->gs, h->opts, api_ref(h), h->ctas, h->warps, q, h->stream)); h->launches++;
    // Converter + plant step + noise on the device, results staged as x_next | u_plant
    double* dout;
    if (int rc = stage_out_begin(h, 1, nullptr, n0 + (size_t)B * 2, 0, &dout)) return rc;
    double* dxn = dev ? x_next : dout;
    double* dup = (dev && u_plant) ? u_plant : dout + n0;
    if (h->ops->kind == KIND_ATT) {     // no converter: the OCP input is the plant input, held for the sub-steps; u_plant = (T, wx)
        k_sim_step_att<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->cfg.sim_erk_stages, h->cfg.sim_substeps, h->cfg.sim_dt, dx, h->gs.U0, 4, 0, dp, de, dxn);
        CK(cudaGetLastError()); h->launches++;
        CK(cudaMemcpy2DAsync(dup, 2 * sizeof(double), h->gs.U0, nu * sizeof(double), 2 * sizeof(double), B, cudaMemcpyDeviceToDevice, h->stream));
    } else {
    k_convert_sim<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->ops->kind, nx, h->cfg.sim_erk_stages, h->cfg.sim_substeps, h->cfg.sim_dt, dx, h->gs.U0,
                                                           (const double*)h->gs.PAR, h->ops->np, h->ops->elem_size == 4, dp, de, dxn, dup);
    CK(cudaGetLastError()); h->launches++;
    }
    if (!dev) {
        CK(cudaMemcpyAsync(x_next, dout, n0 * 8, out, h->stream));
        if (u_plant) CK(cudaMemcpyAsync(u_plant, dout + n0, (size_t)B * 2 * 8, out, h->stream));
    }
    if (u0) CK(cudaMemcpyAsync(u0, h->gs.U0, sizeof(double) * B * nu, out, h->stream));
    if (status) CK(cudaMemcpyAsync(status, h->gs.status, sizeof(int32_t) * B, out, h->stream));
    if (on_device == 0) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_get_stats(void* handle, int which, int32_t* out, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !out) return fail(BNMPC_E_ARG, "NULL argument");
    if (which < BNMPC_STAT_STATUS || which > BNMPC_STAT_QP_ITER) return fail(BNMPC_E_FIELD, "unknown statistic");
    if (use_device(h)) return BNMPC_E_CUDA;
    const int32_t* src = h->ints + (size_t)which * h->batch;
    CK(cudaMemcpyAsync(out, src, sizeof(int32_t) * h->batch, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    if (!on_device) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_sim_step(void* handle, int substeps, const double* x, const double* u, const double* p_plant, const double* eps,
                   double* x_next, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !x || !u || !x_next) return fail(BNMPC_E_ARG, "NULL argument");
    if (substeps < 1) return fail(BNMPC_E_ARG, "substeps must be >= 1");
    if (use_device(h)) return BNMPC_E_CUDA;
    const int B = h->batch, nsub = substeps;
    // one staging buffer: x | u | p | eps, and a second one for the result
    const bool att = h->ops->kind == KIND_ATT;      // 3-D model: x [B][10], u [B][substeps][4]
    const size_t nx_ = (size_t)B * (att ? 10 : 4), nu_ = (size_t)B * nsub * (att ? 4 : 2), np_ = p_plant ? (size_t)B * 2 : 0, ne_ = eps ? (size_t)B : 0;
    const double *dx = x, *du = u, *dp = p_plant, *de = eps;
    if (on_device < 0 || on_device > BNMPC_HOST_ASYNC) return fail(BNMPC_E_ARG, "on_device must be 0, 1 or BNMPC_HOST_ASYNC");
    if (on_device != 1) {
        // one staging buffer on the device: x | u | p | eps
        const size_t tot = nx_ + nu_ + np_ + ne_;
        if (h->stage_cap[3] < tot) {
            if (h->stage[3]) CK(cudaFree(h->stage[3]));
            h->stage[3] = nullptr; h->stage_cap[3] = 0;
            CK(cudaMalloc(&h->stage[3], tot * sizeof(double)));
            h->stage_cap[3] = tot;
        }
        double* d = h->stage[3];
        CK(cudaMemcpyAsync(d, x, nx_ * 8, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(d + nx_, u, nu_ * 8, cudaMemcpyHostToDevice, h->stream));
        if (p_plant) CK(cudaMemcpyAsync(d + nx_ + nu_, p_plant, np_ * 8, cudaMemcpyHostToDevice, h->stream));
        if (eps) CK(cudaMemcpyAsync(d + nx_ + nu_ + np_, eps, ne_ * 8, cudaMemcpyHostToDevice, h->stream));
        dx = d; du = d + nx_; dp = p_plant ? d + nx_ + nu_ : nullptr; de = eps ? d + nx_ + nu_ + np_ : nullptr;
    }
    double* dout;
    if (int rc = stage_out_begin(h, 1, x_next, nx_, on_device == 1, &dout)) return rc;
    if (att) k_sim_step_att<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->cfg.sim_erk_stages, nsub, h->cfg.sim_dt, dx, du, nsub * 4, 4, dp, de, dout);
    else k_sim_step<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->cfg.sim_erk_stages, nsub, h->cfg.sim_dt, dx, du, dp, de, dout);
    CK(cudaGetLastError()); h->launches++;
    if (on_device == 1) return 0;
    CK(cudaMemcpyAsync(x_next, dout, nx_ * 8, cudaMemcpyDeviceToHost, h->stream));
    if (on_device == 0) CK(cudaStreamSynchronize(h->stream));      // BNMPC_HOST_ASYNC: the caller synchronises
    return 0;
}

int bnmpc_closed_loop_init(void* handle, const double* x0, const double* p_ctrl, const double* p_plant) {
    Handle* h = (Handle*)handle;
    if (!h || !x0) return fail(BNMPC_E_ARG, "NULL argument");
    if (use_device(h)) return BNMPC_E_CUDA;
    if (int rc = reset_iterate(h)) return rc;
    const int B = h->batch;
    k_loop_init<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->Bp, x0, p_ctrl, p_plant, h->xs, h->acc, h->cost, h->abs_err, h->p_plant, h->fail_count);
    CK(cudaGetLastError()); h->launches++;
    if (p_ctrl) {
        if (h->ops->elem_size == 8) k_par_from_bm<double><<<(B + 127) / 128, 128, 0, h->stream>>>(gs_cast<double>(h->gs), h->ops->np, p_ctrl);
        else k_par_from_bm<float><<<(B + 127) / 128, 128, 0, h->stream>>>(gs_cast<float>(h->gs), h->ops->np, p_ctrl);
        CK(cudaGetLastError()); h->launches++;
    } else {
        const double pn[2] = {0.03277, 9.81};
        const double* d;
        if (int rc = stage_in(h, 0, pn, 2, 0, &d)) return rc;
        CK(field_xfer(h, F_P, 0, const_cast<double*>(d), h->ops->np, 0, 1));
    }
    return 0;
}

int bnmpc_closed_loop_run(void* handle, const bnmpc_closed_loop_args* a) {
    Handle* h = (Handle*)handle;
    if (!h || !a || !a->ref) return fail(BNMPC_E_ARG, "NULL argument");
    if (a->n_steps < 0 || a->first_step < 0) return fail(BNMPC_E_ARG, "negative step count");
    if (a->first_step + a->n_steps + h->cfg.horizon > a->ref_rows) return fail(BNMPC_E_ARG, "ref has too few rows for first_step + n_steps + N");
    if (a->noise_philox && a->noise) return fail(BNMPC_E_ARG, "noise array and noise_philox are exclusive");
    if (h->ops->kind == KIND_ATT) return fail(BNMPC_E_UNSUPPORTED, "the 3-D attitude model has no fused closed loop: step it with bnmpc_step_for_x0");
    if (h->gs.BND) return fail(BNMPC_E_UNSUPPORTED, "per-stage bounds ('lbu'/'ubu', 'lbx'/'ubx' at stages >= 1) belong to the solve() path; the fused closed loop uses the boxes of the configuration, like the reference's follow_trajectory");
    const bool logs = a->noise || a->Xsim || a->U_plant || a->U_ctrl || a->a_log || a->status || a->qp_iter;
    if (logs && a->log_stride < a->first_step + a->n_steps) return fail(BNMPC_E_ARG, "log_stride too small");
    if (use_device(h)) return BNMPC_E_CUDA;
    LoopArgs la;
    memset(&la, 0, sizeof(la));
    if (a->ref_shared < 0 || a->ref_shared > 3) return fail(BNMPC_E_ARG, "ref_shared must be 0 (batch-minor), 1 (shared), 2 (instance-major) or 3 (circle parameters)");
    if (a->ref_shared == 3 && a->ref_rows - h->cfg.horizon < 2) return fail(BNMPC_E_ARG, "circle reference needs ref_rows >= horizon + 2");
    la.kind = h->ops->kind; la.ref_layout = a->ref_shared; la.ref_rows = a->ref_rows; la.log_stride = a->log_stride; la.batch = h->batch; la.Bp = h->Bp;
    la.ref = a->ref; la.noise = a->noise; la.Xsim = a->Xsim; la.U_plant = a->U_plant; la.U_ctrl = a->U_ctrl; la.a_log = a->a_log;
    la.status = a->status; la.qp_iter = a->qp_iter;
    la.noise_philox = a->noise_philox; la.noise_seed = a->noise_seed; la.noise_std = a->noise_std; la.inst0 = a->first_instance;
    la.xs = h->xs; la.acc = h->acc; la.cost = h->cost; la.abs_err = h->abs_err; la.p_plant = h->p_plant;
    la.fail_count = h->fail_count; la.next_step = h->next_step;
    la.ls_generation = h->ls_generation; la.prof = h->prof; la.prof_cap = h->prof_cap;
    const int spl = a->steps_per_launch > 1 ? a->steps_per_launch : 1;
    const int slots = h->ctas * h->warps;
    for (int s = 0; s < a->n_steps;) {
        const int ns = (a->n_steps - s) < spl ? (a->n_steps - s) : spl;
        la.step = a->first_step + s; la.n_steps = ns;
        if (int rc = refresh_order(h)) return rc;
        int* q;
        if (int rc = next_queue(h, &q)) return rc;
        if (ns == 1) {
            la.chunk = 1;
            if (h->loop_kernel == 1) CK(h->ops->loop_ls(h->gs, h->opts, la, h->ctas, h->warps, q, h->stream));
            else CK(h->ops->loop_step(h->gs, h->opts, la, h->ctas, h->warps, h->wpg, q, h->stream));
            h->launches++;
        } else {
            const bool ls = h->loop_kernel == 1;
            // steps of an instance per queue ticket: long enough to amortise the load of the persistent state, short enough
            // for ~12 tickets per resident warp so that the launch ends without a tail (measured, 4096 drones x 60 steps: chunks
            // of 3 / 10 / 60 steps 9.31 / 9.52 / 8.45 M solves/s); one ticket per instance when every
            // instance has a warp of its own anyway
            long long chunk = h->batch <= slots ? ns : ((long long)h->batch * ns) / (12LL * slots);
            if (h->chunk_override > 0) chunk = h->chunk_override;
            if (chunk < 1) chunk = 1;
            if (chunk > ns) chunk = ns;
            la.chunk = (int)chunk;
            if (chunk < ns) {
                k_fill_int<<<(h->batch + 255) / 256, 256, 0, h->stream>>>(h->batch, la.step, h->next_step);
                CK(cudaGetLastError()); h->launches++;
            }
            if (ls) CK(h->ops->loop_ls(h->gs, h->opts, la, h->ctas, h->warps, q, h->stream));
            else CK(h->ops->loop_step(h->gs, h->opts, la, h->ctas, h->warps, h->wpg, q, h->stream));
            h->launches++;
        }
        s += ns;
    }
    return 0;
}

int bnmpc_philox_noise(void* handle, uint64_t seed, double noise_std, int64_t first_instance, int first_step, int n_steps, double* out) {
    Handle* h = (Handle*)handle;
    if (!h || !out) return fail(BNMPC_E_ARG, "NULL argument");
    if (n_steps < 0 || first_step < 0) return fail(BNMPC_E_ARG, "negative step count");
    if (use_device(h)) return BNMPC_E_CUDA;
    const size_t tot = (size_t)h->batch * n_steps;
    if (tot == 0) return 0;
    k_philox_noise<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->batch, n_steps, first_step, seed, noise_std, first_instance, out);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}

int bnmpc_debug_profile(void* handle, long long* buf, int cap) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    h->prof = buf; h->prof_cap = buf ? cap : 0;
    return 0;
}

int bnmpc_closed_loop_failures(void* handle, int32_t* out, int on_device) {
    Handle* h = (Handle*)handle;
    if (!h || !out) return fail(BNMPC_E_ARG, "NULL argument");
    if (use_device(h)) return BNMPC_E_CUDA;
    CK(cudaMemcpyAsync(out, h->fail_count, sizeof(int32_t) * h->batch, on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, h->stream));
    if (!on_device) CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int bnmpc_gen_circle_table(void* handle, const double* params, int rows, double* table) {
    Handle* h = (Handle*)handle;
    if (!h || !params || !table) return fail(BNMPC_E_ARG, "NULL argument");
    if (rows - h->cfg.horizon < 2) return fail(BNMPC_E_ARG, "rows must be >= horizon + 2");
    if (use_device(h)) return BNMPC_E_CUDA;
    const size_t tot = (size_t)h->batch * rows * 8;
    k_circle_table<<<(unsigned)((tot + 255) / 256), 256, 0, h->stream>>>(h->batch, rows, rows - h->cfg.horizon, params, table);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}

int bnmpc_closed_loop_state(void* handle, double* cost, double* abs_err, double* x, double* acc) {
    Handle* h = (Handle*)handle;
    if (!h) return fail(BNMPC_E_ARG, "NULL handle");
    if (use_device(h)) return BNMPC_E_CUDA;
    const int B = h->batch;
    k_loop_state<<<(B + 127) / 128, 128, 0, h->stream>>>(B, h->Bp, h->xs, h->acc, h->cost, h->abs_err, cost, abs_err, x, acc);
    CK(cudaGetLastError()); h->launches++;
    return 0;
}

int bnmpc_measure_fma_peak(int device, int precision, double* tflops) {
    if (!tflops) return fail(BNMPC_E_ARG, "NULL argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail(BNMPC_E_CUDA, "no CUDA device: libbnmpc has no CPU path");
    if (device < 0 || device >= ndev) return fail(BNMPC_E_ARG, "device index out of range");
    CK(cudaSetDevice(device));
    return precision == BNMPC_FP32 ? fma_peak<float>(tflops) : fma_peak<double>(tflops);
}

int bnmpc_selftest_rcp(int device, int64_t count, int solver_range, int64_t* mismatches) {
    if (!mismatches || count < 1) return fail(BNMPC_E_ARG, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return fail(BNMPC_E_CUDA, "no CUDA device: libbnmpc has no CPU path");
    if (device < 0 || device >= ndev) return fail(BNMPC_E_ARG, "device index out of range");
    CK(cudaSetDevice(device));
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, sizeof(*d)));
    CK(cudaMemset(d, 0, sizeof(*d)));
    const int blocks = 592, tpb = 256;
    const long long per_thread = (count + (long long)blocks * tpb - 1) / ((long long)blocks * tpb);
    k_rcp_check<<<blocks, tpb>>>(per_thread, solver_range, d);
    CK(cudaGetLastError());
    unsigned long long hbad = 0;
    CK(cudaMemcpy(&hbad, d, sizeof(hbad), cudaMemcpyDeviceToHost));
    CK(cudaFree(d));
    *mismatches = (int64_t)hbad;
    return 0;
}

int64_t bnmpc_launch_count(void* handle) {
    Handle* h = (Handle*)handle;
    return h ? h->launches : 0;
}

}  // extern "C"
