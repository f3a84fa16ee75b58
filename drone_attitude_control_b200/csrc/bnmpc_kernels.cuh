// bnmpc_kernels.cuh - __global__ wrappers around the solver templates and the per-model launch table.
// Each model_*.cu instantiates BNMPC_DEFINE_MODEL_OPS for one generated model (both precisions); bnmpc_api.cu only
// sees the ModelOps table, so the heavy templates compile in parallel translation units.
//
// Launch shape: ONE PERSISTENT CTA per SM with as many warps as the on-chip memories hold instances (16 for the force
// model, 12 for the jerk model at N = 30); every warp pulls OCP instances from an atomic work queue and solves them one
// at a time (instance solve lengths differ by 4x, so the queue balances itself).  Warps of a CTA never synchronise
// during the solves; the CTA exists because of tensor memory:
//
//   * shared memory holds the part of an instance's working set that the Riccati sweeps and neighbouring stages touch
//     (SmLayout: 29 doubles per (stage, block) item for the force model, 14.4 KB per instance);
//   * TENSOR MEMORY holds the lane-private part (gradient q, multipliers lam, slacks t and their reciprocals, plus the
//     dynamics offset b_k where the record has room: 23 doubles per item for the force model).  A warp owns the 32 TMEM lanes of its quarter (warp id mod 4) in
//     the column group of its warp quad (warp id / 4); lane l keeps the records of its items in consecutive columns and
//     moves a whole record with one tcgen05.ld / tcgen05.st (.32x32b.x32).  TMEM is used purely as a software-managed,
//     lane-private scratchpad - no tcgen05.mma is involved: these are 3x3 / 4x4 FP64 problems.
//
// Measured (force model, 65536 instances, M solves/s): three CTAs of 4 warps at 168 registers 6.20; ONE CTA of 12 warps
// at 168 registers 7.20; one CTA at 128 registers with 8 / 10 / 11 / 12 / 13 / 14 warps 5.03 / 5.08 / 5.58 / 6.57 / 5.87 /
// 6.04 - only whole multiples of the four SM sub-partitions pay.  With the block constants bound per lane the force kernel
// needs 124-128 registers, and with Phi_k formed in the scans 16 instances fit shared memory: 16 warps 8.54 vs 12 warps
// 7.63.  The launch bound is per model (LaunchShape): the largest multiple of four warps (at most BNMPC_MAX_WARPS = 16)
// whose instances fit shared memory at the reference horizon N = 30 - 16 for the force model (128 registers), 12 for the
// jerk model (168 registers), 8 for the dense 4-state models (255 registers).  The warps actually launched per CTA
// follow from the horizon of the handle and the tensor-memory columns (cta_shape below).
#pragma once
#include <cuda_runtime.h>
#include <string.h>

#include "bnmpc_lockstep.cuh"

#ifndef BNMPC_MAX_WARPS
#define BNMPC_MAX_WARPS 16       // warps of the one resident CTA per SM the register allocator leaves room for (launch bound)
#endif

namespace bnmpc {

// type-erased Gs<T> (identical layout for every T)
struct GsAny {
    void *V, *PI, *LAM, *YREF, *X0, *PAR;
    int32_t *status, *sqp_iter, *qp_iter, *have_mult;
    double* U0;
    double* BND;
    int B, N;
};
template <class T> inline Gs<T> gs_cast(const GsAny& a) {
    static_assert(sizeof(Gs<T>) == sizeof(GsAny), "layout");
    Gs<T> g; memcpy(&g, &a, sizeof(g)); return g;
}

struct ModelOps {
    const char* name;
    int nx, nu, np, nblk, nxb, nub, kind, jac_const, elem_size, sm_rows;
    int max_wpg, max_warps;                                         // largest warp group per instance the closed-loop kernel was built for; launch bound
    size_t (*smem_bytes)(int N);                                    // dynamic shared memory of one instance (one warp)
    int (*tmem_cols)(int N, int warps, int wpg);                    // tensor-memory columns a CTA of `warps` allocates (0 = too many)
    // `tab`: the handle's bound reference table and window row when it is the yref source (ApiRef::ref == nullptr: Gs::YREF)
    cudaError_t (*solve)(const GsAny&, const Opts&, const ApiRef& tab, int ctas, int warps, int* queue, cudaStream_t);
    // the same for handles whose instances carry per-stage bounds (GsAny::BND): a second instantiation of the solve kernel, so
    // that the lookup costs the common case nothing
    cudaError_t (*solve_sb)(const GsAny&, const Opts&, const ApiRef& tab, int ctas, int warps, int* queue, cudaStream_t);
    cudaError_t (*loop_step)(const GsAny&, const Opts&, const LoopArgs&, int ctas, int warps, int wpg, int* queue, cudaStream_t);
    // slotted lockstep schedule (bnmpc_lockstep.cuh): LoopArgs::n_steps control steps per launch, tickets of LoopArgs::chunk steps
    cudaError_t (*loop_ls)(const GsAny&, const Opts&, const LoopArgs&, int ctas, int warps, int* queue, cudaStream_t);
    // warps per CTA and warps per instance (wpg; instances in flight per SM = warps / wpg), warps = 0: does not fit
    cudaError_t (*cta_shape)(int N, int* warps, int* wpg);
    long (*loop_static_bytes)(int wpg);                             // static shared memory of the closed-loop kernel (-1: none)
    // solution sensitivities at the stored solutions, mode 0: d(x_k, u_k) / d x0, 1: adjoint, 2: d(x_k, u_k) / d p,
    // 3: adjoint with grad_p (bnmpc_eval_sens_x0 / bnmpc_eval_adjoint_sens_p / bnmpc_eval_sens_p); nullptr for the models
    // whose Gauss-Newton Hessian is not the Lagrangian's (THRUST, ATT)
    cudaError_t (*sens)(const GsAny&, const Opts&, const SensArgs&, int mode, int ctas, int warps, int* queue, cudaStream_t);
};

// ---------------------------------------------------------------------------------------------------------------------
// tensor memory as lane-private storage
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* w) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]), "=r"(w[4]), "=r"(w[5]), "=r"(w[6]), "=r"(w[7]),
          "=r"(w[8]), "=r"(w[9]), "=r"(w[10]), "=r"(w[11]), "=r"(w[12]), "=r"(w[13]), "=r"(w[14]), "=r"(w[15]),
          "=r"(w[16]), "=r"(w[17]), "=r"(w[18]), "=r"(w[19]), "=r"(w[20]), "=r"(w[21]), "=r"(w[22]), "=r"(w[23]),
          "=r"(w[24]), "=r"(w[25]), "=r"(w[26]), "=r"(w[27]), "=r"(w[28]), "=r"(w[29]), "=r"(w[30]), "=r"(w[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t* w) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};\n"
        :: "r"(taddr),
           "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]), "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7]),
           "r"(w[8]), "r"(w[9]), "r"(w[10]), "r"(w[11]), "r"(w[12]), "r"(w[13]), "r"(w[14]), "r"(w[15]),
           "r"(w[16]), "r"(w[17]), "r"(w[18]), "r"(w[19]), "r"(w[20]), "r"(w[21]), "r"(w[22]), "r"(w[23]),
           "r"(w[24]), "r"(w[25]), "r"(w[26]), "r"(w[27]), "r"(w[28]), "r"(w[29]), "r"(w[30]), "r"(w[31])
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory"); }

__device__ __forceinline__ double words_to(uint32_t lo, uint32_t hi, double) { return __hiloint2double((int)hi, (int)lo); }
__device__ __forceinline__ float words_to(uint32_t lo, uint32_t, float) { return __uint_as_float(lo); }

template <class M, class T, bool SB = false>
struct TmemPriv {
    static constexpr bool IN_SMEM = false;
    static constexpr bool STAGE_BOUNDS = SB;                        // per-stage bounds looked up per item (API solve kernel only)
    static constexpr int s = M::NXB + M::NUB, n = M::NXB;
    static constexpr int WPE = (int)sizeof(T) / 4;                 // 32-bit words per element
    static constexpr bool TI_PRIV = true;                          // the reciprocals 1/t travel with the record (7 s elements)
    static constexpr int CH = (7 * s * WPE + 31) / 32;             // .x32 chunks per record (q, lam, t, 1/t)
    static constexpr bool QB_PRIV = (7 * s + n) * WPE <= CH * 32;  // room for the dynamics offset b_k in the same chunks
    static constexpr int NQ = QB_PRIV ? n : 0;
    // what else the chunks have room for: the bound residuals rd and the stationarity residual rg of the predictor pass
    static constexpr bool RD_PRIV = (7 * s + NQ + 2 * s) * WPE <= CH * 32;
    static constexpr int NRD = RD_PRIV ? 2 * s : 0;
    static constexpr bool RG_PRIV = RD_PRIV && (7 * s + NQ + NRD + s) * WPE <= CH * 32;
    static constexpr int NRG = RG_PRIV ? s : 0;
    static constexpr int NE = 7 * s + NQ + NRD + NRG;              // elements of a record: q, lam, t [, b], 1/t [, rd] [, rg]
    static constexpr int CPR = CH * 32;                            // columns per round of items
    uint32_t base;                                                 // lane quarter of this warp | first column

    // columns the four warps of a quad share (one lane quarter each); L = lanes of the group that owns an instance
    static __host__ __device__ int cols_per_quad(int N, int L = 32) {
        return ((N + 1) * M::NBLK + L - 1) / L * CPR;
    }
    static __host__ __device__ int cols_needed(int N, int warps, int L = 32) { // allocation of a CTA: power of two >= 32, 0 if it does not fit
        const int need = (warps + 3) / 4 * cols_per_quad(N, L);
        int c = 32;
        while (c < need) c <<= 1;
        return c <= 512 ? c : 0;
    }
    // TMEM address of this warp's records: lane quarter = warp id mod 4 (the hardware's access rule), column group = warp id / 4
    static __device__ __forceinline__ uint32_t warp_base(uint32_t tbase, int N, int L = 32) {
        const uint32_t w = threadIdx.x >> 5;
        return tbase + (((w & 3u) * 32u) << 16) + (w >> 2) * (uint32_t)cols_per_quad(N, L);
    }
    __device__ __forceinline__ void load(T*, int rd, int, bool, PrivRec<T, s, n>& r) const {
        __syncwarp();                                              // tcgen05.ld/st are warp-collective (.aligned)
        uint32_t w[CH * 32];
#pragma unroll
        for (int c = 0; c < CH; c++) tmem_ld32(base + rd * CPR + c * 32, w + c * 32);
        tmem_wait_ld();
        T e[NE];
#pragma unroll
        for (int i = 0; i < NE; i++) e[i] = words_to(w[i * WPE], w[i * WPE + WPE - 1], T());
#pragma unroll
        for (int v = 0; v < s; v++) r.q[v] = e[v];
#pragma unroll
        for (int v = 0; v < 2 * s; v++) { r.lam[v] = e[s + v]; r.tt[v] = e[3 * s + v]; }
        if constexpr (QB_PRIV) {
#pragma unroll
            for (int v = 0; v < n; v++) r.qb[v] = e[5 * s + v];
        }
#pragma unroll
        for (int v = 0; v < 2 * s; v++) r.ti[v] = e[5 * s + NQ + v];
        if constexpr (RD_PRIV) {
#pragma unroll
            for (int v = 0; v < 2 * s; v++) r.rd[v] = e[7 * s + NQ + v];
        }
        if constexpr (RG_PRIV) {
#pragma unroll
            for (int v = 0; v < s; v++) r.rg[v] = e[7 * s + NQ + NRD + v];
        }
    }
    __device__ __forceinline__ void store(T*, int rd, int, bool, const PrivRec<T, s, n>& r) const {
        T e[NE];
#pragma unroll
        for (int v = 0; v < s; v++) e[v] = r.q[v];
#pragma unroll
        for (int v = 0; v < 2 * s; v++) { e[s + v] = r.lam[v]; e[3 * s + v] = r.tt[v]; }
        if constexpr (QB_PRIV) {
#pragma unroll
            for (int v = 0; v < n; v++) e[5 * s + v] = r.qb[v];
        }
#pragma unroll
        for (int v = 0; v < 2 * s; v++) e[5 * s + NQ + v] = r.ti[v];
        if constexpr (RD_PRIV) {
#pragma unroll
            for (int v = 0; v < 2 * s; v++) e[7 * s + NQ + v] = r.rd[v];
        }
        if constexpr (RG_PRIV) {
#pragma unroll
            for (int v = 0; v < s; v++) e[7 * s + NQ + NRD + v] = r.rg[v];
        }
        uint32_t w[CH * 32];
        __syncwarp();
#pragma unroll
        for (int i = 0; i < CH * 32; i++) w[i] = 0u;
#pragma unroll
        for (int i = 0; i < NE; i++) {
            if constexpr (WPE == 2) { w[2 * i] = (uint32_t)__double2loint((double)e[i]); w[2 * i + 1] = (uint32_t)__double2hiint((double)e[i]); }
            else w[i] = __float_as_uint((float)e[i]);
        }
#pragma unroll
        for (int c = 0; c < CH; c++) tmem_st32(base + rd * CPR + c * 32, w + c * 32);
        tmem_wait_st();
    }
};

// per-CTA tensor memory allocation (warp 0 allocates and frees; the address travels through shared memory)
__device__ __forceinline__ uint32_t tmem_alloc_cta(uint32_t cols) {
    __shared__ uint32_t tmem_base_s;
    if ((threadIdx.x >> 5) == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n"
                     :: "r"((uint32_t)__cvta_generic_to_shared(&tmem_base_s)), "r"(cols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    return tmem_base_s;
}
__device__ __forceinline__ void tmem_free_cta(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if ((threadIdx.x >> 5) == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" :: "r"(base), "r"(cols) : "memory");
}

// Element offset of this warp's working set inside the CTA's dynamic shared memory.  The value goes through an opaque
// `mov` so that it lives in ONE register: left to itself the compiler re-derived it from threadIdx and the horizon at
// every group of shared-memory accesses (16 % of all executed instructions in the ncu profile of that version).
__device__ __forceinline__ int warp_smem_off(int stride_elems, int group_lanes = 32) {
    int off = stride_elems * (int)(threadIdx.x / group_lanes);
    asm volatile("mov.b32 %0, %0;" : "+r"(off));
    return off;
}

// launch bound of a model: instances that fit shared memory at the reference horizon, whole warp quads, <= BNMPC_MAX_WARPS
template <class M, class T>
struct LaunchShape {
    static constexpr size_t REF_BYTES = SmLayout<M, false, TmemPriv<M, T>::QB_PRIV>::elems(30) * sizeof(T);
    static constexpr int FIT = (int)((227 * 1024 - 1024) / REF_BYTES);
    static constexpr int MAX_WARPS = FIT >= BNMPC_MAX_WARPS ? BNMPC_MAX_WARPS : (FIT >= 4 ? FIT / 4 * 4 : (FIT >= 1 ? FIT : 1));
};

// next instance of the work queue (one atomic per warp).  `order` maps the queue position to an instance: the host side
// sorts the instances by the iterations of their previous solve, longest first, so that the tail of a launch is made of
// short solves (instances are independent: the order changes the timing, never a result).
__device__ __forceinline__ int next_instance(int* queue, const int* order, int B) {
    int i = 0;
    if ((threadIdx.x & 31) == 0) {
        i = atomicAdd(queue, 1);
        if (order != nullptr && i < B) i = order[i];
    }
    return __shfl_sync(0xffffffffu, i, 0);
}

template <class G>
struct DevTickets {
    int* queue; int* next_step; const G& g;
    // value of the group's first lane -> all lanes of the group
    __device__ __forceinline__ int bcast(int v) const {
        if constexpr (G::L == 32) return __shfl_sync(0xffffffffu, v, 0);
        else {
            __shared__ int word[16];
            if (g.lane == 0) word[g.gid()] = v;
            g.sync();
            v = word[g.gid()];
            g.sync();
            return v;
        }
    }
    __device__ __forceinline__ int take() const {
        int i = 0;
        if (g.lane == 0) i = atomicAdd(queue, 1);
        return bcast(i);
    }
    __device__ __forceinline__ bool ready(int inst, int step) const {
        int v = 0;
        if (g.lane == 0) v = *(volatile int*)(next_step + inst);
        v = bcast(v);
        if (v != step) return false;
        __threadfence();
        return true;
    }
    __device__ __forceinline__ void wait(int inst, int step) const {      // free-running groups only (never inside a CTA-wide schedule)
        while (!ready(inst, step)) __nanosleep(200);
    }
    __device__ __forceinline__ void publish(int inst, int next) const {
        __threadfence();
        g.sync();
        if (g.lane == 0) *(volatile int*)(next_step + inst) = next;
    }
};

template <class M, class T, bool SB>
__global__ void __launch_bounds__(32 * LaunchShape<M, T>::MAX_WARPS, 1)
k_solve(const __grid_constant__ Gs<T> gs, const __grid_constant__ Opts o, const __grid_constant__ ApiRef tab, int* queue, int tmem_cols) {
    const uint32_t tbase = tmem_alloc_cta(tmem_cols);
    const WarpGroup<32> g;
    const TmemPriv<M, T, SB> ps{TmemPriv<M, T, SB>::warp_base(tbase, o.N)};
    Solver<M, T, WarpGroup<32>, TmemPriv<M, T, SB>> sv(nullptr, warp_smem_off(o.smem_stride), o, g, ps);
    for (int inst = next_instance(queue, o.order, gs.B); inst < gs.B; inst = next_instance(queue, o.order, gs.B)) api_solve<M, T>(sv, inst, gs, tab);
    tmem_free_cta(tbase, tmem_cols);
}

// Solution sensitivities at the stored solutions, MODE 0: forward in x0 (api_sens_x0), 1: adjoint (api_sens_adj), 2: forward
// in p (api_sens_p), 3: adjoint with the gradient in p as well.  The
// launch shape, work queue and shared-memory layout of k_solve, with the per-stage-bound lookup compiled in.  The passes
// involved (factorisation, Newton solve) keep nothing in the lane-private record, so the kernel allocates no tensor memory.
template <class M, class T, int MODE>
__global__ void __launch_bounds__(32 * LaunchShape<M, T>::MAX_WARPS, 1)
k_sens(const __grid_constant__ Gs<T> gs, const __grid_constant__ Opts o, const __grid_constant__ SensArgs a, int* queue) {
    const WarpGroup<32> g;
    const TmemPriv<M, T, true> ps{0u};
    Solver<M, T, WarpGroup<32>, TmemPriv<M, T, true>> sv(nullptr, warp_smem_off(o.smem_stride), o, g, ps);
    for (int inst = next_instance(queue, nullptr, gs.B); inst < gs.B; inst = next_instance(queue, nullptr, gs.B)) {
        if constexpr (MODE == 0) api_sens_x0<M, T>(sv, inst, gs, a);
        else if constexpr (MODE == 1) api_sens_adj<M, T>(sv, inst, gs, a);
        else if constexpr (MODE == 2) api_sens_p<M, T>(sv, inst, gs, a);
        else api_sens_adj<M, T, true>(sv, inst, gs, a);
    }
}

// WPG warps per instance (see WarpGroup): 1 at the reference horizon, 2 / 4 where the horizon leaves room for only 8 / 4
// instances per SM
template <class M, class T, int WPG>
__global__ void __launch_bounds__(32 * LaunchShape<M, T>::MAX_WARPS, 1)
k_loop_step(const __grid_constant__ Gs<T> gs, const __grid_constant__ Opts o, const __grid_constant__ LoopArgs a, int* queue, int tmem_cols) {
    const uint32_t tbase = tmem_alloc_cta(tmem_cols);
    using G = WarpGroup<32 * WPG>;
    const G g;
    const TmemPriv<M, T> ps{TmemPriv<M, T>::warp_base(tbase, o.N, G::L)};
    Solver<M, T, G, TmemPriv<M, T>> sv(nullptr, warp_smem_off(o.smem_stride, G::L), o, g, ps);
    // queue tickets = (instance, chunk of control steps), issued instance-round-robin; with one control step per launch a
    // ticket is simply an instance (one copy of the solver code for both cases: the kernel's hot loop is instruction-fetch
    // sensitive, see profiles/README.md)
    DevTickets<G> wq{queue, a.next_step, g};
    const int total = gs.B * ((a.n_steps + a.chunk - 1) / a.chunk);
    for (int t = wq.take(); t < total; t = wq.take()) closed_loop_chunk<M, T>(sv, t, gs, a, wq);
    tmem_free_cta(tbase, tmem_cols);
}

// ---------------------------------------------------------------------------------------------------------------------
// slotted lockstep kernel (bnmpc_lockstep.cuh)
// ---------------------------------------------------------------------------------------------------------------------
// one lane of the sweep warp: it serves block `b` of the instance of warp slot `slot`
struct SweepLane {
    static constexpr int L = 1;
    static constexpr bool PAR_SCAN = false;
    int lane;
    __device__ __forceinline__ SweepLane() : lane(0) {}
    template <class T> __device__ __forceinline__ T max(T v) const { return v; }
    template <class T> __device__ __forceinline__ T sum(T v) const { return v; }
    __device__ __forceinline__ bool any(bool p) const { return p; }
    __device__ __forceinline__ bool all(bool p) const { return p; }
    __device__ __forceinline__ void sync() const {}
};

struct LsShared {
    int wstate[BNMPC_MAX_WARPS];          // LsWarp::published() of every warp, refreshed before the first barrier of a half-round
    double par[BNMPC_MAX_WARPS][2];       // model parameters of every warp's instance, for the lanes of the sweep warp
};

// KIND 0: factorisation, 1: backward scan, 2: forward scan - for all instances of `mask` (bit = warp slot) at once, NBLK
// lanes per instance, executed by one warp.  The lane's view of "its" instance is a Solver bound to that warp's working set.
template <class M, class T, int KIND>
__device__ __forceinline__ void ls_sweep(const Opts& o, const LsShared& sh, unsigned mask, int ws_of_slot) {
    constexpr int NBLK = M::NBLK;
    const int lane = (int)(threadIdx.x & 31), slot = lane / NBLK, b = lane % NBLK;
    if (!((mask >> slot) & 1u) || slot >= BNMPC_MAX_WARPS) return;
    const SweepLane gl;
    const TmemPriv<M, T> ps{0u};
    Solver<M, T, SweepLane, TmemPriv<M, T>> svs(nullptr, o.smem_stride * slot, o, gl, ps);
    T p[M::NP];
#pragma unroll
    for (int j = 0; j < M::NP; j++) p[j] = T(sh.par[slot][j]);
    svs.set_par(p);
    svs.bind_block(b);
    if (KIND == 0) svs.kkt_factor_blk(b);
    else if (KIND == 1) svs.back_scan_blk(b);
    else svs.fwd_scan_blk(b, (ws_of_slot & 7) - 1);
}

template <class M, class T>
__global__ void __launch_bounds__(32 * LaunchShape<M, T>::MAX_WARPS, 1)
k_loop_ls(const __grid_constant__ Gs<T> gs, const __grid_constant__ Opts o, const __grid_constant__ LoopArgs a, int* queue, int tmem_cols) {
    __shared__ LsShared sh;
    const uint32_t tbase = tmem_alloc_cta(tmem_cols);
    const WarpGroup<32> g;
    const TmemPriv<M, T> ps{TmemPriv<M, T>::warp_base(tbase, o.N)};
    using SV = Solver<M, T, WarpGroup<32>, TmemPriv<M, T>>;
    SV sv(nullptr, warp_smem_off(o.smem_stride), o, g, ps);
    LsWarp<M, T, WarpGroup<32>, TmemPriv<M, T>> w;
    w.reset();
    DevTickets<WarpGroup<32>> wq{queue, a.next_step, g};
    const int W = (int)(blockDim.x >> 5), warp = (int)(threadIdx.x >> 5), lane = (int)(threadIdx.x & 31);
    static_assert(LaunchShape<M, T>::MAX_WARPS * M::NBLK <= 32, "the sweeps of a CTA must fit one warp");
    const bool prof = a.prof != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
    int nprof = 1;
    auto mark = [&](int tag, unsigned m0, unsigned m1) {
        if (prof && nprof + 2 <= a.prof_cap) { a.prof[nprof++] = clock64(); a.prof[nprof++] = ((long long)tag << 56) | ((long long)m0 << 24) | (long long)(m1 & 0xffffffu); }
    };
    unsigned ipm_prev = 0;
    for (;;) {
        const int inst_before = w.inst;
        mark(0, 0, 0);
        ls_pslot<M, T>(1, w, sv, gs, a, wq, (ipm_prev & ~(1u << warp)) != 0);
        if (w.inst != inst_before && w.inst >= 0 && lane < M::NP) sh.par[warp][lane] = double(sv.par[lane]);
        if (lane == 0) sh.wstate[warp] = w.published();
        mark(1, 0, 0);
        __syncthreads();
        const int ws = lane < W ? sh.wstate[lane] : 0;
        const unsigned alive_m = __ballot_sync(0xffffffffu, (ws & LS_ALIVE) != 0);
        const unsigned fac_m = __ballot_sync(0xffffffffu, (ws & 7) == 1), ipm_m = __ballot_sync(0xffffffffu, (ws & 7) != 0);
        if (!alive_m) break;
        ipm_prev = ipm_m;
        const bool others = (ipm_m & ~(1u << warp)) != 0;
        const int ws_slot = __shfl_sync(0xffffffffu, ws, lane / M::NBLK);       // state of the warp slot this lane would sweep for
        mark(2, fac_m, ipm_m);
        if (fac_m) { if (warp == 0) ls_sweep<M, T, 0>(o, sh, fac_m, ws_slot); mark(3, 0, 0); __syncthreads(); }
        mark(4, 0, 0);
        ls_pslot<M, T>(2, w, sv, gs, a, wq, others);
        mark(5, 0, 0);
        __syncthreads();
        mark(6, 0, 0);
        if (ipm_m) { if (warp == 0) ls_sweep<M, T, 1>(o, sh, ipm_m, ws_slot); mark(7, 0, 0); __syncthreads(); }
        mark(8, 0, 0);
        ls_pslot<M, T>(3, w, sv, gs, a, wq, others);
        mark(9, 0, 0);
        __syncthreads();
        mark(10, 0, 0);
        if (ipm_m) { if (warp == 0) ls_sweep<M, T, 2>(o, sh, ipm_m, ws_slot); mark(11, 0, 0); __syncthreads(); }
        mark(12, 0, 0);
        ls_pslot<M, T>(4, w, sv, gs, a, wq, others);
    }
    if (prof) a.prof[0] = nprof;
    tmem_free_cta(tbase, tmem_cols);
}

// GROUPS: also instantiate the closed-loop kernel with 2 and 4 warps per instance (long horizons)
// LOOP: the model has a fused closed loop (k_loop_step / k_loop_ls); false = the acados-style solve() surface only (the 3-D
// attitude model: its closed loop runs through bnmpc_step_for_x0, one call per control step)
template <class M, class T, bool GROUPS = false, bool LOOP = true>
struct OpsImpl {
    static size_t smem_bytes(int N) { return (SmLayout<M, false, TmemPriv<M, T>::QB_PRIV>::elems(N) * sizeof(T) + 15) / 16 * 16; }
    static int tmem_cols(int N, int warps, int wpg) { return TmemPriv<M, T>::cols_needed(N, warps, 32 * wpg); }
    // dynamic shared memory is opted in once per kernel up to the device limit (handles with different horizons share
    // the kernel, so the attribute must not follow the last handle created)
    template <class K>
    static cudaError_t prep(K kern, size_t) {
        int dev = 0, optin = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return e;
        cudaFuncAttributes fa;
        e = cudaFuncGetAttributes(&fa, kern);
        if (e != cudaSuccess) return e;
        const int stat = fa.sharedSizeBytes > 1024 ? (int)fa.sharedSizeBytes : 1024;                  // the static part (the 2- / 4-warp
        e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin - stat);   // kernels carry the scans' exchange area)
        if (e != cudaSuccess) return e;
        return cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    }
    // Warps of the one CTA per SM = instances in flight per SM: bounded by registers (the launch bound), by shared memory
    // (the opt-in maximum of a block minus the static part) and by tensor memory (512 columns, one column group per warp quad).
    static cudaError_t cta_shape(int N, int* warps, int* wpg) {
        cudaError_t e = cudaSuccess;
        if constexpr (LOOP) {
            e = prep(k_loop_step<M, T, 1>, 0);
            if (e != cudaSuccess) return e;
            if constexpr (GROUPS) {
                e = prep(k_loop_step<M, T, 2>, 0);
                if (e != cudaSuccess) return e;
                e = prep(k_loop_step<M, T, 4>, 0);
                if (e != cudaSuccess) return e;
            }
            e = prep(k_loop_ls<M, T>, 0);
            if (e != cudaSuccess) return e;
        }
        e = prep(k_solve<M, T, false>, 0);
        if (e != cudaSuccess) return e;
        e = prep(k_solve<M, T, true>, 0);
        if (e != cudaSuccess) return e;
        if constexpr (M::JAC_CONST) {
            e = prep(k_sens<M, T, 0>, 0);
            if (e != cudaSuccess) return e;
            e = prep(k_sens<M, T, 1>, 0);
            if (e != cudaSuccess) return e;
            e = prep(k_sens<M, T, 2>, 0);
            if (e != cudaSuccess) return e;
            e = prep(k_sens<M, T, 3>, 0);
            if (e != cudaSuccess) return e;
        }
        int dev = 0, optin = 0;
        e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return e;
        e = cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
        if (e != cudaSuccess) return e;
        int w = (int)((size_t)(optin - 1024) / smem_bytes(N));
        if (w > LaunchShape<M, T>::MAX_WARPS) w = LaunchShape<M, T>::MAX_WARPS;
        while (w > 0 && tmem_cols(N, w, 1) == 0) w--;
        if (w > 4) w = w / 4 * 4;                                // whole warp quads: one warp more on one sub-partition costs more than it adds
        *warps = w;
        int g = 1;
        *wpg = g;
        return cudaSuccess;
    }
    // static shared memory of the closed-loop kernel with wpg warps per instance (-1: no such kernel)
    static long loop_static_bytes(int wpg) {
        if constexpr (!LOOP) return -1;
        else {
            cudaFuncAttributes fa;
            cudaError_t e = cudaErrorInvalidValue;
            if (wpg == 1) e = cudaFuncGetAttributes(&fa, k_loop_step<M, T, 1>);
            else if constexpr (GROUPS) {
                if (wpg == 2) e = cudaFuncGetAttributes(&fa, k_loop_step<M, T, 2>);
                else if (wpg == 4) e = cudaFuncGetAttributes(&fa, k_loop_step<M, T, 4>);
            }
            return e == cudaSuccess ? (long)fa.sharedSizeBytes : -1;
        }
    }
    static cudaError_t solve(const GsAny& a, const Opts& o_, const ApiRef& tab, int ctas, int warps, int* queue, cudaStream_t st) {
        Opts o = o_;
        o.smem_stride = (int)(smem_bytes(o.N) / sizeof(T));
        k_solve<M, T, false><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, tab, queue, tmem_cols(o.N, warps, 1));
        return cudaGetLastError();
    }
    static cudaError_t solve_sb(const GsAny& a, const Opts& o_, const ApiRef& tab, int ctas, int warps, int* queue, cudaStream_t st) {
        Opts o = o_;
        o.smem_stride = (int)(smem_bytes(o.N) / sizeof(T));
        k_solve<M, T, true><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, tab, queue, tmem_cols(o.N, warps, 1));
        return cudaGetLastError();
    }
    // `warps` = instances per CTA, each run by a group of wpg warps
    static cudaError_t loop_step(const GsAny& a, const Opts& o_, const LoopArgs& la, int ctas, int warps, int wpg, int* queue, cudaStream_t st) {
        if constexpr (!LOOP) return cudaErrorNotSupported;
        else {
        Opts o = o_;
        o.smem_stride = (int)(smem_bytes(o.N) / sizeof(T));
        const int cols = tmem_cols(o.N, warps * wpg, wpg);
        const size_t sm = smem_bytes(o.N) * warps;
        if (wpg == 1) k_loop_step<M, T, 1><<<ctas, 32 * warps, sm, st>>>(gs_cast<T>(a), o, la, queue, cols);
        else if constexpr (GROUPS) {
            if (wpg == 2) k_loop_step<M, T, 2><<<ctas, 64 * warps, sm, st>>>(gs_cast<T>(a), o, la, queue, cols);
            else k_loop_step<M, T, 4><<<ctas, 128 * warps, sm, st>>>(gs_cast<T>(a), o, la, queue, cols);
        } else return cudaErrorInvalidValue;
        return cudaGetLastError();
        }
    }
    static cudaError_t loop_ls(const GsAny& a, const Opts& o_, const LoopArgs& la, int ctas, int warps, int* queue, cudaStream_t st) {
        if constexpr (!LOOP) return cudaErrorNotSupported;
        else {
        Opts o = o_;
        o.smem_stride = (int)(smem_bytes(o.N) / sizeof(T));
        k_loop_ls<M, T><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, la, queue, tmem_cols(o.N, warps, 1));
        return cudaGetLastError();
        }
    }
    static cudaError_t sens(const GsAny& a, const Opts& o_, const SensArgs& sa, int mode, int ctas, int warps, int* queue, cudaStream_t st) {
        if constexpr (!M::JAC_CONST) return cudaErrorNotSupported;
        else {
        Opts o = o_;
        o.smem_stride = (int)(smem_bytes(o.N) / sizeof(T));
        if (mode == 0) k_sens<M, T, 0><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, sa, queue);
        else if (mode == 1) k_sens<M, T, 1><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, sa, queue);
        else if (mode == 2) k_sens<M, T, 2><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, sa, queue);
        else k_sens<M, T, 3><<<ctas, 32 * warps, smem_bytes(o.N) * warps, st>>>(gs_cast<T>(a), o, sa, queue);
        return cudaGetLastError();
        }
    }
    static ModelOps make(int kind) {
        return ModelOps{M::name(), M::NX, M::NU, M::NP, M::NBLK, M::NXB, M::NUB, kind, M::JAC_CONST ? 1 : 0, (int)sizeof(T),
                        SmLayout<M, false, TmemPriv<M, T>::QB_PRIV>::ROWS, GROUPS ? 4 : 1, LaunchShape<M, T>::MAX_WARPS, &smem_bytes, &tmem_cols, &solve, &solve_sb, &loop_step, &loop_ls, &cta_shape, &loop_static_bytes,
                        M::JAC_CONST ? &sens : nullptr};
    }
};

#define BNMPC_DEFINE_MODEL_OPS(MODEL, KIND, FN, GROUPS) BNMPC_DEFINE_MODEL_OPS_(MODEL, KIND, FN, GROUPS, true)
#define BNMPC_DEFINE_MODEL_OPS_(MODEL, KIND, FN, GROUPS, LOOP)                                \
    namespace bnmpc {                                                                         \
    const ModelOps* FN(int precision) {                                                       \
        static const ModelOps d = OpsImpl<MODEL, double, GROUPS, LOOP>::make(KIND);            \
        static const ModelOps f = OpsImpl<MODEL, float, GROUPS, LOOP>::make(KIND);             \
        return precision == 0 ? &d : &f;                                                      \
    }                                                                                         \
    }

const ModelOps* ops_force(int precision);
const ModelOps* ops_jerk(int precision);
const ModelOps* ops_force_dense(int precision);
const ModelOps* ops_thrust(int precision);
const ModelOps* ops_att(int precision);

}  // namespace bnmpc
