// ude_batch.cuh -- batched independent trainings of the LV 2 -> 5 -> 5 -> 5 -> 2 UDE: M members, each with its own theta, data,
// u0, gradient and ADAM moments, one member per thread and no coupling between members anywhere (no ensemble sum, no shared
// optimiser state).  The device counterpart of LotkaVolterra/run_loops.jl:55-62, which calls recover_dynamics
// (loop_recoveries.jl) once per noisy data set, one run after another.
//
// One thread runs a member's whole iteration in registers: the fixed-step Tsit5 forward solve (tsit5_record), the fused-L2
// backward sweep (lane_adjoint, interpolating or discrete), the member's loss and the Flux.ADAM update -- the arithmetic of
// adam_kernel (b200ude.cu), applied to one member.  All `iters` iterations run inside one launch: members never exchange data,
// so no iteration needs a grid-wide synchronisation.
//
// Layouts: theta of the CTA's members in shared memory as [P][BLOCK] (WLane: lane l reads column l, conflict-free); the ADAM
// moments in global memory as [P][ldm] and the forward record as [..][D][M] (member-fastest: the warp's accesses coalesce).
// The record is written and read back by the same thread in the same launch, so it is read with ordinary loads (NC = false).
//
// Every member keeps its own ADAM step count (advanced only by its own updates) and, like sciml_train, the best pre-update theta
// seen so far with its loss (strictly lower loss replaces it; non-finite losses never do).
// A member whose final state, loss or gradient is non-finite stops: status B200UDE_TRAJ_NONFINITE, theta, moments and step count
// keep their last values, the loss slots of its remaining iterations are NaN.  The other members compute exactly what they would
// without it: a member's results depend on its own inputs only (not on M or its position), bit for bit.
#pragma once
#include "ude_adjoint.cuh"

namespace b200ude {

template <class C, bool DISC, int BLOCK>
__device__ __forceinline__ void batch_member(const WLane<BLOCK> &w, const BatchParams &p, size_t n)
{
    constexpr int D = C::D, P = C::P;
    const size_t M = (size_t)p.M;
    FwdParams fp;
    fp.u0 = p.u0; fp.out = p.out; fp.ustep = p.ustep; fp.dense = p.dense; fp.status = nullptr; fp.theta = nullptr;
    fp.N = p.M; fp.n_steps = p.n_steps; fp.save_every = p.save_every; fp.P = P; fp.dt = p.dt;
    AdjParams ap;
    ap.ustep = p.ustep; ap.dense = p.dense; ap.cot = p.data; ap.grad_u0 = nullptr; ap.partial = nullptr; ap.theta = nullptr;
    ap.N = p.M; ap.n_steps = p.n_steps; ap.save_every = p.save_every; ap.P = P; ap.fused_l2 = 1; ap.dt = p.dt;
    const int nn[1] = {(int)n};
    const bool live[1] = {true};
    const int iters = p.mode == BATCH_TRAIN ? p.iters : 1;
    int32_t status = 0;
    int it = 0;
#pragma unroll 1
    for (; it < iters; ++it) {
        StateT<D, 1> us;
        tsit5_record<C, 1, 0>(w, fp, nn, live, us);
        bool ok = true;
#pragma unroll
        for (int c = 0; c < D; ++c) ok = ok && (fabsf(us.v[c][0]) <= 3.0e38f);   // false for NaN / Inf
        if (p.mode == BATCH_FORWARD) {
            status = ok ? 0 : 1;
            break;
        }
        float gacc[P], lam[D], loss;
        lane_adjoint<C, 0, WLane<BLOCK>, DISC, false>(w, ap, n, gacc, lam, loss);
        ok = ok && (fabsf(loss) <= 3.0e38f);
#pragma unroll
        for (int q = 0; q < P; ++q) ok = ok && (fabsf(gacc[q]) <= 3.0e38f);
        if (p.mode == BATCH_LOSS_GRAD) {
            p.loss[n] = loss;
#pragma unroll
            for (int q = 0; q < P; ++q) p.grad[n * P + q] = gacc[q];
            status = ok ? 0 : 1;
            break;
        }
        // ADAM (adam_kernel's arithmetic): L = loss_scale * L_data + l2_reg * sum theta[NPREFIX:]^2 is recorded at the pre-update
        // theta; g = loss_scale * grad + 2 l2_reg theta (the L2 term skips the trainable physics rates)
        float sq = 0.0f;
        if (p.l2_reg != 0.0f) {
#pragma unroll
            for (int q = C::NPREFIX; q < P; ++q) sq = fmaf(w(q), w(q), sq);
        }
        const float total = fmaf(p.loss_scale, loss, p.l2_reg * sq);
        if (p.loss_history) p.loss_history[(size_t)it * M + n] = total;
        if (total < p.best_loss[n]) {   // step count and best loss stay in global memory: no registers held across the loop
            p.best_loss[n] = total;
#pragma unroll 1
            for (int q = 0; q < P; ++q) p.best[n * P + q] = w(q);
        }
        if (!ok) {
            status = 1;
            ++it;
            break;
        }
        const int t = p.t[n] + 1;
        p.t[n] = t;
        const float c1 = (float)(1.0 / (1.0 - pow((double)p.beta1, (double)t)));
        const float c2 = (float)(1.0 / (1.0 - pow((double)p.beta2, (double)t)));
        extern __shared__ __align__(16) float s_lane[];
#pragma unroll
        for (int q = 0; q < P; ++q) {
            float &th = s_lane[q * BLOCK + w.lane];
            const size_t iq = (size_t)q * p.ldm + n;
            const float g = fmaf(p.loss_scale, gacc[q], q >= C::NPREFIX ? 2.0f * p.l2_reg * th : 0.0f);
            const float m = fmaf(p.beta1, p.m[iq], (1.0f - p.beta1) * g);
            const float v = fmaf(p.beta2, p.v[iq], (1.0f - p.beta2) * g * g);
            p.m[iq] = m;
            p.v[iq] = v;
            th = th - p.eta * (m * c1) / (sqrtf(v * c2) + p.eps);
        }
    }
    if (p.loss_history)
        for (; it < iters; ++it) p.loss_history[(size_t)it * M + n] = __int_as_float(0x7fc00000);
    if (p.status) p.status[n] = status;
}

template <class C, bool DISC, int BLOCK>
__global__ void __launch_bounds__(BLOCK) ude_batch_kernel(BatchParams p)
{
    constexpr int P = C::P;
    extern __shared__ __align__(16) float s_lane[];   // [P][BLOCK]
    const size_t first = (size_t)blockIdx.x * BLOCK;
    const int rows = (int)min((size_t)BLOCK, (size_t)p.M - first);
    // the CTA's rows of theta [M][P] are contiguous in global memory: coalesced reads, transposed into the lanes' columns
    for (int i = threadIdx.x; i < rows * P; i += BLOCK) s_lane[(i % P) * BLOCK + i / P] = p.theta[first * P + i];
    __syncthreads();
    if ((int)threadIdx.x < rows) batch_member<C, DISC, BLOCK>(WLane<BLOCK>{(int)threadIdx.x}, p, first + threadIdx.x);
    if (p.mode == BATCH_TRAIN) {
        __syncthreads();
        for (int i = threadIdx.x; i < rows * P; i += BLOCK) p.theta[first * P + i] = s_lane[(i % P) * BLOCK + i / P];
    }
}

}  // namespace b200ude
