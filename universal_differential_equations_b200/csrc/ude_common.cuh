// ude_common.cuh -- shared pieces of the sm_100a kernels of the UDE hot path (+ the forward kernel).
//
//   ude_forward_kernel : whole fixed-step Tsit5 solve of an ensemble in ONE launch.  One thread
//                        integrates T trajectories: state and stage derivatives live in registers,
//                        the embedded chain's weights are read as constant-bank FFMA operands (or
//                        from a TMA-staged shared-memory copy), every stage's UDE right-hand side =
//                        known physics + chain forward is fused into the Runge-Kutta stage loop.
//                        Writes the saved states, the per-step states and the dense output (k_1..k_7).
//   ude_adjoint_kernel : the InterpolatingAdjoint backward solve in ONE launch: reverse-time Tsit5 on
//                        lambda, u(t) from the stored dense output, chain VJP, loss jumps at the save
//                        points (optionally forming the L2 cotangent in-kernel) and the running
//                        parameter-gradient quadrature.  mu' = -lambda^T df/dtheta never feeds back,
//                        so sum_n mu_n is accumulated directly: the H x H layer's contribution is a
//                        per-warp outer-product GEMM over the warp's 32 trajectories (staged through
//                        shared memory, accumulators resident in registers across all steps).
//   ude_reduce_kernel  : deterministic fixed-order sum of the per-CTA partial gradients / losses.
//
// Reference semantics being replaced (file:line relative to the reference repo):
//   RHS closures          LotkaVolterra/scenario_1.jl:69-76, scenario_2.jl:90-98, hudson_bay.jl:85-91
//   Tsit5 perform_step!   [OrdinaryDiffEq]  call sites Fisher-KPP-CNN.jl:136, seir_exposure.jl:66,132
//   InterpolatingAdjoint  [DiffEqSensitivity] call sites seir_exposure.jl:71,140, Fisher-KPP-CNN.jl:136
//   L2 loss               scenario_1.jl:91-94
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "params.h"
#include "tsit5.cuh"

namespace b200ude {

constexpr int MODEL_LV = 0, MODEL_SEIR = 1, MODEL_FKPP = 2, MODEL_NODE = 3, MODEL_SEIR_NODE = 4;
constexpr int ACT_IDENTITY = 0, ACT_TANH = 1, ACT_RBF = 2, ACT_RUNTIME = -1;
constexpr int GRAD_LANE = 0;   // every lane keeps all P partial sums in registers (small chains)
constexpr int GRAD_WARPGEMM = 1;  // H x H layer via per-warp smem-staged outer-product GEMM

constexpr int MAX_THETA = 12288;  // floats; 48 KB of the 64 KB constant bank (the script's 7-64-64-64-7 neural ODE has 9287)
static __constant__ __align__(16) float c_theta[MAX_THETA];
static __constant__ float c_consts[16];
static __constant__ float c_lossw[16];
static __constant__ int c_acts[8];

// weight sources ---------------------------------------------------------------------------------
struct WConst {  // constant bank: sm_100a reads it through LDCU.128 into uniform registers (4 weights per load)
    __device__ __forceinline__ float operator()(int i) const { return c_theta[i]; }
};
struct WSmem {  // shared-memory copy (bulk-copied once per CTA); compile-time offsets -> LDS[.128]
    const float *p;
    __device__ __forceinline__ float operator()(int i) const { return p[i]; }
};
template <int STRIDE>
struct WLane {  // one theta per lane in dynamic shared memory laid out [P][STRIDE]: lane l reads column l, so the warp's 32
                // different weights at one index sit in 32 different banks (LDS with a compile-time offset i * STRIDE)
    int lane;
    __device__ __forceinline__ float operator()(int i) const
    {
        extern __shared__ __align__(16) float s_lane[];
        return s_lane[i * STRIDE + lane];
    }
};

// compile-time description of one UDE -----------------------------------------------------------
template <int MODEL_, int D_, int DIN_, int H_, int NHID_, int DOUT_, int ACT_, int NPREFIX_, int GRAD_>
struct Cfg {
    static constexpr int MODEL = MODEL_, D = D_, DIN = DIN_, H = H_, NHID = NHID_, DOUT = DOUT_;
    static constexpr int ACT = ACT_, NPREFIX = NPREFIX_, GRAD = GRAD_;
    static constexpr int OFF_W0 = NPREFIX;
    static constexpr int OFF_B0 = OFF_W0 + DIN * H;
    __host__ __device__ static constexpr int off_w(int l) { return OFF_B0 + H + (l - 1) * (H * H + H); }
    __host__ __device__ static constexpr int off_b(int l) { return off_w(l) + H * H; }
    static constexpr int OFF_WOUT = OFF_B0 + H + (NHID - 1) * (H * H + H);
    static constexpr int OFF_BOUT = OFF_WOUT + H * DOUT;
    static constexpr int P = OFF_BOUT + DOUT;  // (+ suffix for FKPP, none for LV/SEIR)
    static constexpr int JB = (H % 4 == 0) ? 4 : (H % 5 == 0 ? 5 : 1);  // output block of the H x H sweep
};

// the reference-shaped LV UDE: 2 -> 5 -> 5 -> 5 -> 2 chain, per-layer activations, NP trainable linear rates in front of the chain
// (LotkaVolterra/scenario_1.jl:62-73, scenario_2.jl:79-98, hudson_bay.jl:77-91, loop_recoveries.jl:7-12)
template <int NP>
using CfgLV5 = Cfg<MODEL_LV, 2, 2, 5, 3, 2, ACT_RUNTIME, NP, GRAD_LANE>;

// activations -------------------------------------------------------------------------------------
// TM = 0: tanh(x) = 1 - 2/(2^(2 log2(e) x) + 1): MUFU.EX2 + MUFU.RCP, abs. error ~1e-7
// TM = 1: tanh.approx.f32 (one MUFU, rel. error 2^-11) -- opt-in
template <int TM>
__device__ __forceinline__ float tanh_dev(float x)
{
    if constexpr (TM == 1) {
        float y;
        asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
        return y;
    } else {
        float e, r;
        asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * 2.885390081777927f));
        asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(e + 1.0f));
        return fmaf(-2.0f, r, 1.0f);
    }
}
__device__ __forceinline__ float rbf_dev(float x)
{
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * x * -1.4426950408889634f));
    return e;
}
template <int ACT, int TM>
__device__ __forceinline__ float act_dev(float a, int layer)
{
    if constexpr (ACT == ACT_TANH) return tanh_dev<TM>(a);
    else if constexpr (ACT == ACT_RBF) return rbf_dev(a);
    else if constexpr (ACT == ACT_IDENTITY) return a;
    else {
        const int k = c_acts[layer];
        return k == ACT_TANH ? tanh_dev<TM>(a) : (k == ACT_RBF ? rbf_dev(a) : a);
    }
}
// derivative of the activation from pre-activation a and output h
template <int ACT>
__device__ __forceinline__ float actder_dev(float a, float h, int layer)
{
    if constexpr (ACT == ACT_TANH) return fmaf(-h, h, 1.0f);
    else if constexpr (ACT == ACT_RBF) return -2.0f * a * h;
    else if constexpr (ACT == ACT_IDENTITY) return 1.0f;
    else {
        const int k = c_acts[layer];
        return k == ACT_TANH ? fmaf(-h, h, 1.0f) : (k == ACT_RBF ? -2.0f * a * h : 1.0f);
    }
}

// chain forward (T trajectories per thread) -------------------------------------------------------
template <class C, int T, int TM, class W>
__device__ __forceinline__ void chain_forward(const W &w, const float (&x)[C::DIN][T], float (&y)[C::DOUT][T])
{
    constexpr int H = C::H, JB = C::JB;
    float h[H][T];
#pragma unroll
    for (int j = 0; j < H; ++j) {
#pragma unroll
        for (int t = 0; t < T; ++t) {
            float a = w(C::OFF_B0 + j);
#pragma unroll
            for (int m = 0; m < C::DIN; ++m) a = fmaf(w(C::OFF_W0 + m * H + j), x[m][t], a);
            h[j][t] = act_dev<C::ACT, TM>(a, 0);
        }
    }
#pragma unroll
    for (int m = 0; m < C::DOUT; ++m)
#pragma unroll
        for (int t = 0; t < T; ++t) y[m][t] = w(C::OFF_BOUT + m);
#pragma unroll
    for (int l = 1; l < C::NHID; ++l) {
        float hn[H][T];
#pragma unroll
        for (int jb = 0; jb < H / JB; ++jb) {
            float acc[JB][T];
#pragma unroll
            for (int jj = 0; jj < JB; ++jj)
#pragma unroll
                for (int t = 0; t < T; ++t) acc[jj][t] = w(C::off_b(l) + jb * JB + jj);
#pragma unroll
            for (int i = 0; i < H; ++i)
#pragma unroll
                for (int jj = 0; jj < JB; ++jj)
#pragma unroll
                    for (int t = 0; t < T; ++t)
                        acc[jj][t] = fmaf(w(C::off_w(l) + i * H + jb * JB + jj), h[i][t], acc[jj][t]);
#pragma unroll
            for (int jj = 0; jj < JB; ++jj)
#pragma unroll
                for (int t = 0; t < T; ++t) {
                    const float v = act_dev<C::ACT, TM>(acc[jj][t], l);
                    if (l == C::NHID - 1) {  // last hidden layer: feed the output layer directly
#pragma unroll
                        for (int m = 0; m < C::DOUT; ++m)
                            y[m][t] = fmaf(w(C::OFF_WOUT + (jb * JB + jj) * C::DOUT + m), v, y[m][t]);
                    } else {
                        hn[jb * JB + jj][t] = v;
                    }
                }
        }
        if (l < C::NHID - 1) {
#pragma unroll
            for (int j = 0; j < H; ++j)
#pragma unroll
                for (int t = 0; t < T; ++t) h[j][t] = hn[j][t];
        }
    }
    if constexpr (C::NHID == 1) {
#pragma unroll
        for (int j = 0; j < H; ++j)
#pragma unroll
            for (int m = 0; m < C::DOUT; ++m)
#pragma unroll
                for (int t = 0; t < T; ++t) y[m][t] = fmaf(w(C::OFF_WOUT + j * C::DOUT + m), h[j][t], y[m][t]);
    }
}

// UDE right-hand side: known physics fused with the chain ------------------------------------------
template <class C, class W>
__device__ __forceinline__ void phys_rates(const W &w, float &a1, float &a2)
{
    a1 = c_consts[0];
    a2 = c_consts[1];
    if constexpr (C::NPREFIX == 1) a2 = w(0);
    if constexpr (C::NPREFIX == 2) { a1 = w(0); a2 = w(1); }
}

template <class C, int T, int TM, class W>
__device__ __forceinline__ void ude_rhs(const W &w, const float (&u)[C::D][T], float (&du)[C::D][T])
{
    static_assert(C::MODEL == MODEL_LV, "only the LV family has a kernel in this build");
    float y[C::DOUT][T];
    chain_forward<C, T, TM>(w, u, y);
    float a1, a2;
    phys_rates<C>(w, a1, a2);
#pragma unroll
    for (int t = 0; t < T; ++t) {
        du[0][t] = fmaf(a1, u[0][t], y[0][t]);    // du1 =  p1*u1 + NN1(u)   scenario_1.jl:71
        du[1][t] = fmaf(-a2, u[1][t], y[1][t]);   // du2 = -p4*u2 + NN2(u)   scenario_1.jl:72
    }
}

// The right-hand side is deliberately NOT inlined into the Runge-Kutta loops: with the body inlined
// 6x inside the time-step loop ptxas hoists the ~1.2k loop-invariant weight loads out of the loop and
// spills them to local memory (5 KB stack frame, 6k LDL per step measured in SASS).  As a real
// function the loads stay next to their FFMAs, the code is 6x smaller and the call costs ~20
// instructions per ~1500.
template <int D, int T>
struct StateT {
    float v[D][T];
};
template <class C, int T, int TM, class W>
__device__ __noinline__ StateT<C::D, T> ude_rhs_call(W w, StateT<C::D, T> u)
{
    StateT<C::D, T> du;
    ude_rhs<C, T, TM>(w, u.v, du.v);
    return du;
}

// forward kernel -----------------------------------------------------------------------------------

template <class W>
struct WeightStage;
template <>
struct WeightStage<WConst> {
    static constexpr bool kSmem = false;
    __device__ static WConst load(const float *, int) { return WConst{}; }
};
template <>
struct WeightStage<WSmem> {
    static constexpr bool kSmem = true;
    // One elected thread bulk-copies theta into shared memory with the TMA (1-D cp.async.bulk +
    // mbarrier transaction count); everybody waits on the barrier's phase 0.
    __device__ static WSmem load(const float *theta, int P)
    {
        extern __shared__ __align__(16) float s_dyn[];
        __shared__ __align__(8) uint64_t bar;
        const uint32_t bar_a = (uint32_t)__cvta_generic_to_shared(&bar);
        const uint32_t dst_a = (uint32_t)__cvta_generic_to_shared(s_dyn);
        const uint32_t bytes = (uint32_t)(((P + 3) / 4) * 16);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar_a));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar_a), "r"(bytes) : "memory");
            asm volatile(
                "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_a),
                "l"(theta), "r"(bytes), "r"(bar_a)
                : "memory");
        }
        uint32_t done = 0;
        while (!done) {
            asm volatile(
                "{\n\t.reg .pred p;\n\t"
                "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\t"
                "selp.u32 %0, 1, 0, p;\n\t}"
                : "=r"(done)
                : "r"(bar_a)
                : "memory");
        }
        return WSmem{s_dyn};
    }
};

// Whole fixed-step Tsit5 solve of trajectories n[0..T) from p.u0: writes the saved states, the per-step states and the dense
// output (stores masked by live[]) and leaves the final state in us.
template <class C, int T, int TM, class W>
__device__ __forceinline__ void tsit5_record(const W &w, const FwdParams &p, const int (&n)[T], const bool (&live)[T], StateT<C::D, T> &us)
{
    constexpr int D = C::D;
    const size_t N = (size_t)p.N;
    float (&u)[D][T] = us.v;
    float k[7][D][T];
#pragma unroll
    for (int t = 0; t < T; ++t)
#pragma unroll
        for (int c = 0; c < D; ++c) u[c][t] = __ldg(p.u0 + (size_t)c * N + n[t]);
    const float dt = p.dt;
    auto store_state = [&](float *base, int row) {
#pragma unroll
        for (int t = 0; t < T; ++t)
            if (live[t]) {
#pragma unroll
                for (int c = 0; c < D; ++c) base[((size_t)row * D + c) * N + n[t]] = u[c][t];
            }
    };
    auto store_k = [&](int row, const float (&kk)[D][T]) {
#pragma unroll
        for (int t = 0; t < T; ++t)
            if (live[t]) {
#pragma unroll
                for (int c = 0; c < D; ++c) p.dense[((size_t)row * D + c) * N + n[t]] = kk[c][t];
            }
    };
    store_state(p.out, 0);
    store_state(p.ustep, 0);
    {
        const StateT<D, T> r = ude_rhs_call<C, T, TM>(w, us);
#pragma unroll
        for (int c = 0; c < D; ++c)
#pragma unroll
            for (int t = 0; t < T; ++t) k[0][c][t] = r.v[c][t];
    }
    store_k(0, k[0]);
    int isave = 1;
#pragma unroll 1
    for (int s = 0; s < p.n_steps; ++s) {
#pragma unroll
        for (int i = 1; i < 7; ++i) {
            StateT<D, T> gs;
            float (&g)[D][T] = gs.v;
#pragma unroll
            for (int c = 0; c < D; ++c)
#pragma unroll
                for (int t = 0; t < T; ++t) {
                    float acc = 0.0f;
#pragma unroll
                    for (int j = 0; j < i; ++j)
                        if (Tsit5::a(i, j) != 0.0) acc = fmaf((float)Tsit5::a(i, j), k[j][c][t], acc);
                    g[c][t] = fmaf(dt, acc, u[c][t]);
                }
            if (i == 6) {  // stage 7's argument is u_{n+1} (row 7 = b, FSAL)
#pragma unroll
                for (int c = 0; c < D; ++c)
#pragma unroll
                    for (int t = 0; t < T; ++t) u[c][t] = g[c][t];
            }
            {
                const StateT<D, T> r = ude_rhs_call<C, T, TM>(w, gs);
#pragma unroll
                for (int c = 0; c < D; ++c)
#pragma unroll
                    for (int t = 0; t < T; ++t) k[i][c][t] = r.v[c][t];
            }
            if (i < 6) store_k(s * 6 + i, k[i]);
        }
        store_k((s + 1) * 6, k[6]);
        store_state(p.ustep, s + 1);
        if ((s + 1) % p.save_every == 0) {
            store_state(p.out, isave);
            ++isave;
        }
#pragma unroll
        for (int c = 0; c < D; ++c)
#pragma unroll
            for (int t = 0; t < T; ++t) k[0][c][t] = k[6][c][t];
    }
}

template <class C, int T, int TM, class W, int BLOCK, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB) ude_forward_kernel(FwdParams p)
{
    constexpr int D = C::D;
    const W w = WeightStage<W>::load(p.theta, p.P);
    const int NT = gridDim.x * BLOCK;
    const int tid = blockIdx.x * BLOCK + threadIdx.x;
    int n[T];
    bool live[T];
#pragma unroll
    for (int t = 0; t < T; ++t) {
        n[t] = tid + t * NT;
        live[t] = n[t] < p.N;
        if (!live[t]) n[t] = p.N - 1;  // duplicate work of the last trajectory; stores are masked
    }
    StateT<D, T> us;
    tsit5_record<C, T, TM>(w, p, n, live, us);
    float (&u)[D][T] = us.v;
    if (p.status) {
#pragma unroll
        for (int t = 0; t < T; ++t)
            if (live[t]) {
                bool ok = true;
#pragma unroll
                for (int c = 0; c < D; ++c) ok = ok && (fabsf(u[c][t]) <= 3.0e38f);  // false for NaN/Inf
                p.status[n[t]] = ok ? 0 : 1;
            }
    }
}



// push the per-handle tables into THIS translation unit's constant bank (stream-ordered)
static inline cudaError_t upload_tables(const ConstTables &t, cudaStream_t st)
{
    // theta changes every optimiser step: always re-sent (device-to-device, stream-ordered, ~5 KB).
    cudaError_t e = cudaMemcpyToSymbolAsync(c_theta, t.d_theta, sizeof(float) * t.P, 0, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return e;
    static SerialCache cache;
    if (cache.hit(t.serial)) return cudaSuccess;
    e = cudaMemcpyToSymbolAsync(c_consts, t.consts, sizeof(t.consts), 0, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbolAsync(c_lossw, t.lossw, sizeof(t.lossw), 0, cudaMemcpyHostToDevice, st);
    if (e != cudaSuccess) return e;
    e = cudaMemcpyToSymbolAsync(c_acts, t.acts, sizeof(t.acts), 0, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) cache.set(t.serial);
    return e;
}

template <class C, int T, int TM, class W, int MINB>
static inline cudaError_t launch_forward(const FwdParams &p, cudaStream_t st)
{
    auto kern = ude_forward_kernel<C, T, TM, W, FWD_BLOCK, MINB>;
    const int per_block = FWD_BLOCK * T;
    const int grid = (p.N + per_block - 1) / per_block;
    const size_t smem = WeightStage<W>::kSmem ? sizeof(float) * ((C::P + 3) / 4) * 4 : 0;
    kern<<<grid, FWD_BLOCK, smem, st>>>(p);
    return cudaGetLastError();
}

}  // namespace b200ude
