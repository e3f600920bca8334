// ude_adjoint.cuh -- InterpolatingAdjoint backward solve as one fused sm_100a kernel per launch.
//
// Replaces, for the whole ensemble at once, what DiffEqSensitivity does for
//   concrete_solve(...; sensealg = InterpolatingAdjoint(autojacvec = ReverseDiffVJP()))
//   (SEIR_exposure/seir_exposure.jl:71,140; FisherKPP/Fisher-KPP-CNN.jl:136):
// reverse-time Tsit5 on lambda with u(t) from the forward dense output, the chain VJP (what the
// ReverseDiff tape computes), the loss jumps at the save points (discrete callback; optionally the
// L2 cotangent 2 w (u - data) of scenario_1.jl:91-94 is formed in-kernel) and the quadrature of
// mu' = -lambda^T df/dtheta.  mu never feeds back into lambda, so sum_n mu_n is accumulated directly:
//   * ude_adjoint_lane_kernel  (small chains, P <~ 100): every lane keeps all P partial sums in registers;
//   * lv32::adjoint_kernel (lv32_packed.cuh, 2 -> 32 -> 32 -> 2): the 32 x 32 layer's gradient is a
//     per-warp outer-product GEMM over the warp's trajectories, operands staged through shared memory.
// Both end with a fixed-order CTA reduction into partial[blockIdx][P+1]; ude_reduce_kernel sums the
// CTAs in a fixed order, so gradients are bitwise reproducible run to run.
#pragma once
#include "ude_common.cuh"

namespace b200ude {

// ---- pieces shared by both adjoint kernels -------------------------------------------------------
// NC = true: the forward record and the data are read through the non-coherent read-only path (they are written by an earlier
// launch).  A kernel that writes its own record in the same launch (the batched trainer, k_batch.cu) reads it with NC = false.
template <bool NC>
__device__ __forceinline__ float ld_rec(const float *a)
{
    if constexpr (NC) return __ldg(a);
    else return *a;
}

// u(t_{s+1} - c_i dt) from the stored dense output of forward step s (Tsit5 free interpolant).
// The k's are re-read per stage (L1-resident after the first touch) instead of being held in
// registers across the stage evaluations.
template <int D, int I, bool NC = true>
__device__ __forceinline__ void interp_state(const AdjParams &p, int s, size_t n, size_t N, float dt, float (&x)[D])
{
#pragma unroll
    for (int c = 0; c < D; ++c) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < 7; ++j)
            if (Tsit5::bw(I, j) != 0.0)
                acc = fmaf((float)Tsit5::bw(I, j), ld_rec<NC>(p.dense + ((size_t)(s * 6 + j) * D + c) * N + n), acc);
        x[c] = fmaf(dt, acc, ld_rec<NC>(p.ustep + ((size_t)s * D + c) * N + n));
    }
}

template <int D, int I>
__device__ __forceinline__ void stage_arg(const float (&lam)[D], const float (&kl)[6][D], float dt, float (&g)[D])
{
#pragma unroll
    for (int c = 0; c < D; ++c) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < I; ++j)
            if (Tsit5::a(I, j) != 0.0) acc = fmaf((float)Tsit5::a(I, j), kl[j][c], acc);
        g[c] = fmaf(dt, acc, lam[c]);
    }
}

// ---- discrete adjoint (exact gradient of the fixed-step Tsit5 scheme; what ForwardDiffSensitivity computes,
// scenario_1.jl:86): stage argument g_i = u_n + dt sum_{j<i} a_ij k_j from the stored step start and stage derivatives ...
template <int D, int I, bool NC = true>
__device__ __forceinline__ void fwd_stage_state(const AdjParams &p, int s, size_t n, size_t N, float dt, float (&x)[D])
{
#pragma unroll
    for (int c = 0; c < D; ++c) {
        float acc = 0.0f;
#pragma unroll
        for (int j = 0; j < I; ++j)
            if (Tsit5::a(I, j) != 0.0)
                acc = fmaf((float)Tsit5::a(I, j), ld_rec<NC>(p.dense + ((size_t)(s * 6 + j) * D + c) * N + n), acc);
        x[c] = fmaf(dt, acc, ld_rec<NC>(p.ustep + ((size_t)s * D + c) * N + n));
    }
}
// ... and the cotangent of k_i: kbar_i = dt (b_i ubar_{n+1} + sum_{j>i} a_ji gbar_j), gbar_j = J_u(g_j)^T kbar_j of the later stages
template <int D, int I>
__device__ __forceinline__ void disc_stage_cot(const float (&lam)[D], const float (&gb)[6][D], float dt, float (&kb)[D])
{
#pragma unroll
    for (int c = 0; c < D; ++c) {
        float acc = (float)Tsit5::b(I) * lam[c];
#pragma unroll
        for (int j = I + 1; j < 6; ++j)
            if (Tsit5::a(j, I) != 0.0) acc = fmaf((float)Tsit5::a(j, I), gb[j][c], acc);
        kb[c] = dt * acc;
    }
}

// lambda += dL/du(t_isave); with fused_l2 also accumulates the loss
template <int D, bool NC = true>
__device__ __forceinline__ void loss_jump(const AdjParams &p, int isave, size_t n, size_t N, float (&lam)[D], float &loss)
{
#pragma unroll
    for (int c = 0; c < D; ++c) {
        const size_t idx = ((size_t)isave * D + c) * N + n;
        if (p.fused_l2) {
            // saved state i is the state at step i*save_every (the handle's own per-step store)
            const size_t idu = ((size_t)(isave * p.save_every) * D + c) * N + n;
            const float r = ld_rec<NC>(p.ustep + idu) - ld_rec<NC>(p.cot + idx);
            const float wgt = c_lossw[c];
            loss = fmaf(wgt * r, r, loss);
            lam[c] = fmaf(2.0f * wgt, r, lam[c]);
        } else {
            lam[c] += ld_rec<NC>(p.cot + idx);
        }
    }
}

// =====================================================================================================
// small chains: per-lane register accumulators
// =====================================================================================================
// Backward sweep of trajectory n: gacc[P] = its parameter gradient, lam = dL/du0, loss = its fused-L2 loss (fused_l2 only).
// DISC selects the discrete adjoint (reverse accumulation through the stages) over the interpolating one.
template <class C, int TM, class W, bool DISC, bool NC = true>
__device__ __forceinline__ void lane_adjoint(const W &w, const AdjParams &p, size_t n, float (&gacc)[C::P], float (&lam)[C::D], float &loss)
{
    static_assert(C::MODEL == MODEL_LV, "only the LV family has a kernel in this build");
    constexpr int D = C::D, H = C::H, NHID = C::NHID, DIN = C::DIN, DOUT = C::DOUT, P = C::P;
    constexpr bool NEED_PRE = (C::ACT != ACT_TANH && C::ACT != ACT_IDENTITY);
    const size_t N = (size_t)p.N;
    const float dt = p.dt;
#pragma unroll
    for (int q = 0; q < P; ++q) gacc[q] = 0.0f;

    float a1, a2;
    phys_rates<C>(w, a1, a2);

    loss = 0.0f;
    const int n_save = p.n_steps / p.save_every + 1;
#pragma unroll
    for (int c = 0; c < D; ++c) lam[c] = 0.0f;
    loss_jump<D, NC>(p, n_save - 1, n, N, lam, loss);

    auto stage_eval = [&](const float sc, const float (&x)[DIN], const float (&g)[D], float (&klI)[D]) {
        const float isc = 1.0f / sc;  // sc = dt*b_i: quadrature weight of this stage
        float hs[NHID][H];
        float pre[NHID][H];  // only written/read when the activation's derivative needs it
#pragma unroll
        for (int j = 0; j < H; ++j) {
            float a = w(C::OFF_B0 + j);
#pragma unroll
            for (int m = 0; m < DIN; ++m) a = fmaf(w(C::OFF_W0 + m * H + j), x[m], a);
            if constexpr (NEED_PRE) pre[0][j] = a;
            hs[0][j] = act_dev<C::ACT, TM>(a, 0);
        }
#pragma unroll
        for (int l = 1; l < NHID; ++l) {
#pragma unroll
            for (int j = 0; j < H; ++j) {
                float a = w(C::off_b(l) + j);
#pragma unroll
                for (int i2 = 0; i2 < H; ++i2) a = fmaf(w(C::off_w(l) + i2 * H + j), hs[l - 1][i2], a);
                if constexpr (NEED_PRE) pre[l][j] = a;
                hs[l][j] = act_dev<C::ACT, TM>(a, l);
            }
        }
        // reverse sweep; every cotangent carries the quadrature weight sc
        float sg[DOUT];
#pragma unroll
        for (int m = 0; m < DOUT; ++m) sg[m] = sc * g[m];  // LV: d(du)/d(NN) = I
        float q[NHID][H];
#pragma unroll
        for (int j = 0; j < H; ++j) {
            float a = 0.0f;
#pragma unroll
            for (int m = 0; m < DOUT; ++m) a = fmaf(w(C::OFF_WOUT + j * DOUT + m), sg[m], a);
            q[NHID - 1][j] = a * actder_dev<C::ACT>(NEED_PRE ? pre[NHID - 1][j] : 0.f, hs[NHID - 1][j], NHID - 1);
        }
#pragma unroll
        for (int l = NHID - 1; l >= 1; --l) {
#pragma unroll
            for (int i2 = 0; i2 < H; ++i2) {
                float a = 0.0f;
#pragma unroll
                for (int j = 0; j < H; ++j) a = fmaf(w(C::off_w(l) + i2 * H + j), q[l][j], a);
                q[l - 1][i2] = a * actder_dev<C::ACT>(NEED_PRE ? pre[l - 1][i2] : 0.f, hs[l - 1][i2], l - 1);
            }
        }
        float dx[DIN];
#pragma unroll
        for (int m = 0; m < DIN; ++m) {
            float a = 0.0f;
#pragma unroll
            for (int j = 0; j < H; ++j) a = fmaf(w(C::OFF_W0 + m * H + j), q[0][j], a);
            dx[m] = a * isc;
        }
        klI[0] = fmaf(a1, g[0], dx[0]);   // (df/du)^T g, LV physics: diag(a1, -a2)
        klI[1] = fmaf(-a2, g[1], dx[1]);
        if constexpr (C::NPREFIX == 1) gacc[0] = fmaf(-x[1], sg[1], gacc[0]);
        if constexpr (C::NPREFIX == 2) {
            gacc[0] = fmaf(x[0], sg[0], gacc[0]);
            gacc[1] = fmaf(-x[1], sg[1], gacc[1]);
        }
#pragma unroll
        for (int j = 0; j < H; ++j) {
#pragma unroll
            for (int m = 0; m < DIN; ++m) gacc[C::OFF_W0 + m * H + j] = fmaf(q[0][j], x[m], gacc[C::OFF_W0 + m * H + j]);
            gacc[C::OFF_B0 + j] += q[0][j];
        }
#pragma unroll
        for (int l = 1; l < NHID; ++l)
#pragma unroll
            for (int j = 0; j < H; ++j) {
#pragma unroll
                for (int i2 = 0; i2 < H; ++i2)
                    gacc[C::off_w(l) + i2 * H + j] = fmaf(q[l][j], hs[l - 1][i2], gacc[C::off_w(l) + i2 * H + j]);
                gacc[C::off_b(l) + j] += q[l][j];
            }
#pragma unroll
        for (int j = 0; j < H; ++j)
#pragma unroll
            for (int m = 0; m < DOUT; ++m)
                gacc[C::OFF_WOUT + j * DOUT + m] = fmaf(sg[m], hs[NHID - 1][j], gacc[C::OFF_WOUT + j * DOUT + m]);
#pragma unroll
        for (int m = 0; m < DOUT; ++m) gacc[C::OFF_BOUT + m] += sg[m];
    };

#pragma unroll 1
    for (int s = p.n_steps - 1; s >= 0; --s) {
        float kl[6][D];
#define B200UDE_LANE_STAGE(I)                                   \
    {                                                           \
        float x[DIN], g[D];                                     \
        interp_state<D, I, NC>(p, s, n, N, dt, x);              \
        stage_arg<D, I>(lam, kl, dt, g);                        \
        stage_eval(dt * (float)Tsit5::b(I), x, g, kl[I]);       \
    }
#define B200UDE_LANE_DSTAGE(I)                                  \
    {                                                           \
        float x[DIN], kb[D];                                    \
        fwd_stage_state<D, I, NC>(p, s, n, N, dt, x);           \
        disc_stage_cot<D, I>(lam, kl, dt, kb);                  \
        stage_eval(1.0f, x, kb, kl[I]);                         \
    }
        if constexpr (DISC) {
            // reverse accumulation through the forward stages 6..1 of step s; kl[i] holds gbar_i = J_u(g_i)^T kbar_i
            B200UDE_LANE_DSTAGE(5)
            B200UDE_LANE_DSTAGE(4)
            B200UDE_LANE_DSTAGE(3)
            B200UDE_LANE_DSTAGE(2)
            B200UDE_LANE_DSTAGE(1)
            B200UDE_LANE_DSTAGE(0)
#pragma unroll
            for (int c = 0; c < D; ++c) {
                float acc = lam[c];
#pragma unroll
                for (int j = 0; j < 6; ++j) acc += kl[j][c];
                lam[c] = acc;
            }
        } else {
        // k_7 of the backward step only feeds FSAL / error estimation: not needed
        B200UDE_LANE_STAGE(0)
        B200UDE_LANE_STAGE(1)
        B200UDE_LANE_STAGE(2)
        B200UDE_LANE_STAGE(3)
        B200UDE_LANE_STAGE(4)
        B200UDE_LANE_STAGE(5)
#pragma unroll
        for (int c = 0; c < D; ++c) {
            float acc = 0.0f;
#pragma unroll
            for (int j = 0; j < 6; ++j) acc = fmaf((float)Tsit5::b(j), kl[j][c], acc);
            lam[c] = fmaf(dt, acc, lam[c]);
        }
        }
#undef B200UDE_LANE_STAGE
#undef B200UDE_LANE_DSTAGE
        if (s % p.save_every == 0) loss_jump<D, NC>(p, s / p.save_every, n, N, lam, loss);
    }
}

template <class C, int TM, class W, int BLOCK, int MINB, bool DISC = false>
__global__ void __launch_bounds__(BLOCK, MINB) ude_adjoint_lane_kernel(AdjParams p)
{
    constexpr int D = C::D, P = C::P;
    constexpr int NWARP = BLOCK / 32;
    const W w = WeightStage<W>::load(p.theta, p.P);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t N = (size_t)p.N;
    const int gid = blockIdx.x * BLOCK + threadIdx.x;
    const bool live = gid < p.N;
    const size_t n = live ? (size_t)gid : (size_t)(p.N - 1);

    extern __shared__ __align__(16) unsigned char s_raw[];
    constexpr int THETA_SMEM_FLOATS = WeightStage<W>::kSmem ? ((P + 3) / 4) * 4 : 0;

    float gacc[P], lam[D], loss;
    lane_adjoint<C, TM, W, DISC>(w, p, n, gacc, lam, loss);
    if (p.grad_u0 && live) {
#pragma unroll
        for (int c = 0; c < D; ++c) p.grad_u0[(size_t)c * N + n] = lam[c];
    }

    // CTA reduction, fixed order
    __syncthreads();
    float *red = reinterpret_cast<float *>(s_raw + sizeof(float) * THETA_SMEM_FLOATS);  // [P+1]
    for (int q2 = threadIdx.x; q2 < P + 1; q2 += BLOCK) red[q2] = 0.0f;
    __syncthreads();
    const float lv = live ? 1.0f : 0.0f;  // padding lanes duplicated trajectory N-1: contribute zero
    loss *= lv;
#pragma unroll
    for (int q2 = 0; q2 < P; ++q2) {
        float v = gacc[q2] * lv;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        gacc[q2] = v;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) loss += __shfl_xor_sync(0xffffffffu, loss, o);
    for (int wv = 0; wv < NWARP; ++wv) {
        if (warp == wv && lane == 0) {
#pragma unroll
            for (int q2 = 0; q2 < P; ++q2) red[q2] += gacc[q2];
            red[P] += loss;
        }
        __syncthreads();
    }
    float *dst = p.partial + (size_t)blockIdx.x * (P + 1);
    for (int q2 = threadIdx.x; q2 < P + 1; q2 += BLOCK) dst[q2] = red[q2];
}

// fixed-order reduction of the per-CTA partials: out[q] = sum_b partial[b][q]; q == P1-1 is the loss.
// One warp per output entry (8 entries per 256-thread CTA): lane l sums partials l, l+32, ... in order,
// then a fixed butterfly combines the lanes -> deterministic, and ~1000 partials cost a few microseconds.
static __global__ void ude_reduce_kernel(const float *__restrict__ partial, int nblocks, int P1, float *__restrict__ grad,
                                         float *__restrict__ loss)
{
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (q >= P1) return;
    float acc = 0.f;
    for (int b = lane; b < nblocks; b += 32) acc += partial[(size_t)b * P1 + q];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) {
        if (q == P1 - 1) {
            if (loss) *loss = acc;
        } else {
            grad[q] = acc;
        }
    }
}

// ---- the same reduction fused with the cross-GPU sum over NVLink peer memory (one launch, no NCCL) ----------------------
// Every rank owns an exchange buffer (cudaMalloc'ed, mapped into every peer process with CUDA IPC):
//   uint32 flags[16]   flags[src] = number of CTAs of rank `src` whose pushes have landed here (monotonic)
//   uint32 ticket      local CTA counter (monotonic)
//   uint32 epoch       number of completed calls (device-resident so that launch arguments never change: the call can sit
//                      in a replayed CUDA graph, b200ude_train_adam); read by every CTA at its start, bumped by the last CTA
//   float  slots[2][16][P1pad]   [epoch parity][source rank][entry]
// Phase 1 (all CTAs, one warp per entry): local fixed-order sum over the partial rows, PUSHED with plain stores into
// slots[parity][rank][q] of every rank (remote stores over NVLink are fire-and-forget), system-scope fence, then one
// release increment of flags[rank] on every rank per CTA.  Phase 2 (the last CTA of this rank to finish phase 1): acquire-
// spin until every source's flag reached epoch * gridDim.x, then sum the `world` slots of every entry in rank order ->
// all ranks obtain bitwise identical sums.  Parity double-buffering makes the next call's pushes safe: a rank can push for
// epoch e+2 only after it finished epoch e+1, which needed every peer's e+1 push, which a peer issues only after it finished
// reading epoch e.  A bounded spin (about 2 s) turns a lost peer into NaN results instead of a hang.
struct PeerCtx {
    float *slots[16];        // every rank's slot array (this process's mappings), [2][16][P1pad]
    unsigned *flags[16];     // every rank's flags
    unsigned *ticket;        // this rank's CTA counter
    int rank, world, P1pad;
};

static __global__ void ude_reduce_exchange_kernel(const float *__restrict__ partial, int nblocks, int P1, PeerCtx ctx,
                                                  float *__restrict__ grad, float *__restrict__ loss)
{
    __shared__ int s_last;
    // no CTA of this launch can have bumped it yet: the bump happens after ALL CTAs took their ticket, which follows this read
    const unsigned epoch = *reinterpret_cast<volatile unsigned *>(ctx.ticket + 1) + 1u;
    const int lane = threadIdx.x & 31;
    const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int par = (int)(epoch & 1u);
    if (q < P1) {
        float acc = 0.f;
        for (int b = lane; b < nblocks; b += 32) acc += partial[(size_t)b * P1 + q];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane < ctx.world) {
            float *dst = ctx.slots[lane] + ((size_t)par * 16 + ctx.rank) * ctx.P1pad + q;
            *reinterpret_cast<volatile float *>(dst) = acc;
            __threadfence_system();
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence_system();
        for (int r = 0; r < ctx.world; ++r) atomicAdd_system(ctx.flags[r] + ctx.rank, 1u);
        const unsigned t = atomicAdd(ctx.ticket, 1u);
        s_last = ((t + 1u) % gridDim.x) == 0u;
    }
    __syncthreads();
    if (!s_last) return;
    __shared__ int s_ok;
    if (threadIdx.x == 0) s_ok = 1;
    __syncthreads();
    if (threadIdx.x < ctx.world) {
        const unsigned target = epoch * gridDim.x;
        volatile unsigned *f = ctx.flags[ctx.rank] + threadIdx.x;
        const long long t0 = clock64();
        while ((int)(*f - target) < 0) {
            if (clock64() - t0 > 4000000000ll) { s_ok = 0; break; }   // ~2 s at 1.9 GHz
            __nanosleep(100);
        }
        __threadfence_system();
    }
    __syncthreads();
    const float *mine = ctx.slots[ctx.rank] + (size_t)par * 16 * ctx.P1pad;
    for (int e = threadIdx.x; e < P1; e += blockDim.x) {
        float tot = 0.f;
        for (int r = 0; r < ctx.world; ++r) tot += __ldcg(mine + (size_t)r * ctx.P1pad + e);
        if (!s_ok) tot = __int_as_float(0x7fc00000);
        if (e == P1 - 1) {
            if (loss) *loss = tot;
        } else {
            grad[e] = tot;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) *reinterpret_cast<volatile unsigned *>(ctx.ticket + 1) = epoch;
}

}  // namespace b200ude
