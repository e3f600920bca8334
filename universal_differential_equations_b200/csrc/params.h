// params.h -- plain structs shared by the C-ABI layer and the kernel translation units.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

namespace b200ude {

struct FwdParams {
    const float *u0;    // [D][N]
    float *out;         // [n_save][D][N]
    float *ustep;       // [n_steps+1][D][N]  state at every step start (adjoint's interpolation base)
    float *dense;       // [n_steps*6+1][D][N] stage derivatives: row n*6+i = k_{i+1} of step n; k_7(n) = k_1(n+1)
    int32_t *status;    // [N] or nullptr
    const float *theta; // device copy of theta (shared-memory weight variant only)
    int N, n_steps, save_every, P;
    float dt;
};

struct AdjParams {
    const float *ustep;   // [n_steps+1][D][N]
    const float *dense;   // [n_steps*6+1][D][N]
    const float *cot;     // fused_l2 ? data [n_save][D][N] : dL/dout [n_save][D][N]
    float *grad_u0;       // [D][N] or nullptr
    float *partial;       // [gridDim.x][P+1]  per-CTA partial gradient, last entry = partial loss
    const float *theta;   // device theta (shared-memory weight variant only)
    int N, n_steps, save_every, P;
    int fused_l2;         // 1: cot is the data, form 2 w (u - data) and the loss in-kernel
    float dt;
    // sub-range launches (warp-collective LV kernels only): trajectories [n0, n0 + n_cnt) of the N, partial rows from row0
    // (n_cnt = 0: all N).  Lets the host-buffer path start the adjoint of the first half while the second half's data still uploads.
    int n0 = 0, n_cnt = 0, row0 = 0;
};

// per-handle tables every launch pushes into the launching translation unit's constant bank
struct ConstTables {
    uint64_t serial;  // unique per handle: the small tables are re-sent only when it changes
    const float *d_theta;
    int P;
    float consts[16];
    float lossw[16];
    int acts[8];
};

struct Variant {
    int fwd_smem = 0;    // 0: constant-bank weights, 1: shared-memory (TMA-staged) weights
    int fwd_T = 1;       // trajectories per thread in the forward kernel
    int adj_smem = 0;
    int approx_tanh = 0;
    int fwd_tc = 0;      // 1: tcgen05 (3xTF32) forward kernel
    int adj_tc = 0;      // 1: tcgen05 (3xTF32) adjoint kernel, FFMA2 gradient GEMM; 2: mma.sync gradient GEMM
    int discrete = 0;    // 1: discrete adjoint (exact gradient of the fixed-step scheme) instead of the interpolating adjoint
    int fwd_wm = 0;      // 1: warp-collective mma.sync forward kernel (lv32_wm.cuh)
    int adj_wm = 0;      // 1: warp-collective mma.sync adjoint kernel
    int wm_groups = 1;   // groups per warp in the warp-collective forward kernel (1 or 2)
    int wm_rows = 0;     // trajectories per group / 8: 1, 2, or 0 = by ensemble size (<= wm_r1_max -> 1)
    int wm_r1_max = 4736;   // 8 trajectories per warp while that still leaves one warp per scheduler (148 x 4 x 8)
};

// function attributes (dynamic shared-memory size) are per device: one-time flags are kept per device ordinal
struct PerDeviceOnce {
    bool done[64] = {};
    bool &flag()
    {
        int dev = 0;
        cudaGetDevice(&dev);
        return done[dev & 63];
    }
};

// "which handle's small tables are in this device's constant bank": the bank is per device, so the cache is too
// (one host thread per GPU may create and drive handles concurrently)
struct SerialCache {
    std::atomic<uint64_t> last[64] = {};
    static int dev()
    {
        int d = 0;
        cudaGetDevice(&d);
        return d & 63;
    }
    bool hit(uint64_t serial) const { return last[dev()].load(std::memory_order_acquire) == serial; }
    void set(uint64_t serial) { last[dev()].store(serial, std::memory_order_release); }
};

constexpr int FWD_BLOCK = 128;      // small-chain forward kernels
constexpr int FWD_BLOCK_LV32 = 32;  // packed LV32 forward: one warp (64 trajectories) per CTA -> even spread over the SMs
constexpr int ADJ_BLOCK_GEMM = 32;   // H=32 adjoint: one warp (64 trajectories) per CTA
constexpr int ADJ_BLOCK_LANE = 128;  // small-chain adjoint

// batched independent trainings (k_batch.cu, ude_batch.cuh): M members of the LV 2-5-5-5-2 UDE, one theta / gradient / ADAM state
// per member, one member per thread.  Member-fastest layouts except theta.
constexpr int BATCH_FORWARD = 0, BATCH_LOSS_GRAD = 1, BATCH_TRAIN = 2;
constexpr int BATCH_BLOCK = 32;   // members per CTA: theta of the CTA in shared memory as [P][32] (11 KB at P = 89)
struct BatchParams {
    const float *u0;        // [D][M]
    const float *data;      // [n_save][D][M]  (loss / gradient / train)
    float *out;             // [n_save][D][M]  forward: the result; otherwise scratch
    int32_t *status;        // [M]
    float *theta;           // [M][P]: every member's theta contiguous (train writes the updated thetas back)
    float *m, *v;           // [P][ldm] ADAM moments (train)
    float *ustep, *dense;   // forward record [n_steps+1][D][M], [n_steps*6+1][D][M]
    float *loss;            // [M]     (loss / gradient)
    float *grad;            // [M][P]  (loss / gradient)
    float *loss_history;    // [iters][M] or nullptr (train)
    int32_t *t;             // [M] ADAM steps each member has taken (train; advanced only by the member's own updates)
    float *best;            // [M][P] the member's best pre-update theta so far (train)
    float *best_loss;       // [M] its loss (+inf: none yet)
    int M, ldm, n_steps, save_every, mode, iters;
    float dt, eta, beta1, beta2, eps, loss_scale, l2_reg;
};

// runtime shape of a UDE handled by the generic kernels (k_generic.cu)
struct GenericShape {
    uint64_t serial;
    int model, D, din, dout, n_layers, n_prefix, P;
    int widths[8];
    int acts[8];
};

// adaptive stepping: save grid + tolerances + the per-trajectory record of accepted steps
struct AdaptiveGrid {
    float t0, save_dt, abstol, reltol;
    int n_save, max_steps;
    float *tgrid;   // [max_steps+1][N]
    int *nacc;      // [N]
};
constexpr int L2_BLOCKS = 296;

// launchers (one translation unit per kernel family; each owns its constant-bank symbols)
cudaError_t launch_fwd_lv32(const Variant &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_lv32(const Variant &, const ConstTables &, const AdjParams &, cudaStream_t, int *grid_out);
cudaError_t launch_fwd_lv5(int n_prefix, const Variant &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_lv5(int n_prefix, const Variant &, const ConstTables &, const AdjParams &, cudaStream_t, int *grid_out);
int adj_grid_lv32(int N);
cudaError_t launch_fwd_lv32_wm(const Variant &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_lv32_wm(const Variant &, const ConstTables &, const AdjParams &, cudaStream_t, int *rows_out);
int adj_rows_lv32_wm(int N);
cudaError_t launch_tanh_selftest(const float *x, float *y, size_t n, cudaStream_t);
cudaError_t launch_fwd_lv32_adaptive(const Variant &, const ConstTables &, const FwdParams &, const AdaptiveGrid &, cudaStream_t);
cudaError_t launch_adj_lv32_adaptive(const Variant &, const ConstTables &, const AdjParams &, const AdaptiveGrid &, cudaStream_t, int *rows_out);
int adj_grid_lv5(int N);
cudaError_t launch_batch(int n_prefix, bool discrete, const ConstTables &, const BatchParams &, cudaStream_t);
cudaError_t launch_fwd_generic(const GenericShape &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_generic(const GenericShape &, const ConstTables &, const AdjParams &, cudaStream_t, int *rows_out);
int adj_rows_generic(int N);
cudaError_t launch_fwd_vern7(const GenericShape &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_fwd_vern7_adaptive(const GenericShape &, const ConstTables &, const FwdParams &, const AdaptiveGrid &, cudaStream_t);
cudaError_t launch_fwd_adaptive(const GenericShape &, const ConstTables &, const FwdParams &, const AdaptiveGrid &, cudaStream_t);
cudaError_t launch_adj_adaptive(const GenericShape &, const ConstTables &, const AdjParams &, const AdaptiveGrid &, cudaStream_t, int *rows_out);
cudaError_t launch_l2_cot(const ConstTables &, const float *out, const float *data, float *cot, float *block_loss, int D, size_t N, int n_save, cudaStream_t);
cudaError_t launch_l2_finish(const float *block_loss, float *loss, cudaStream_t);
cudaError_t launch_fwd_fkpp(const GenericShape &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_fkpp(const GenericShape &, const ConstTables &, const AdjParams &, cudaStream_t, int *rows_out);
int adj_rows_fkpp(int N, int Nx);
cudaError_t launch_fwd_seir(const Variant &, const ConstTables &, const FwdParams &, cudaStream_t);
cudaError_t launch_adj_seir(const Variant &, const ConstTables &, const AdjParams &, cudaStream_t, int *rows_out);
cudaError_t launch_fwd_seir_vern7(const Variant &, const ConstTables &, const FwdParams &, cudaStream_t);
int adj_rows_seir(int N);
cudaError_t launch_fwd_seir_adaptive(const Variant &, const ConstTables &, const FwdParams &, const AdaptiveGrid &, cudaStream_t);
cudaError_t launch_adj_seir_adaptive(const Variant &, const ConstTables &, const AdjParams &, const AdaptiveGrid &, cudaStream_t, int *rows_out);
// RKC2 recurrence tables of a handle (computed on the host, b200ude.cu)
struct RkcHost {
    int s = 0;
    float mt1 = 0;
    float mu[65] = {}, nu[65] = {}, mt[65] = {}, ga[65] = {}, c[65] = {}, w[65] = {};
};
cudaError_t launch_fwd_fkpp16_rkc(const Variant &, const ConstTables &, const RkcHost &, const FwdParams &, int Nx, cudaStream_t);
cudaError_t launch_adj_fkpp16_rkc(const Variant &, const ConstTables &, const RkcHost &, const AdjParams &, int Nx, cudaStream_t, int *rows_out);
cudaError_t launch_fwd_fkpp16(const Variant &, const ConstTables &, const FwdParams &, int Nx, cudaStream_t);
cudaError_t launch_adj_fkpp16(const Variant &, const ConstTables &, const AdjParams &, int Nx, cudaStream_t, int *rows_out);
int adj_rows_fkpp16(int N, int Nx);
// exchange buffers of the fused reduce + all-reduce (ude_adjoint.cuh): every rank's buffer as mapped in this process
constexpr int PEER_HEADER_BYTES = 256;   // flags[16], ticket, padding
struct PeerLinks {
    void *base[16];
    int rank = 0, world = 0, P1pad = 0;
};
cudaError_t launch_reduce_exchange(const float *partial, int nblocks, int P1, const PeerLinks &, float *grad, float *loss, cudaStream_t);
cudaError_t launch_reduce(const float *partial, int nblocks, int P1, float *grad, float *loss, cudaStream_t);

// ---- double-precision path (dtype = B200UDE_F64; k_f64.cu / ude_f64.cuh) ----
struct Shape64Host {
    uint64_t serial;
    int model, D, din, dout, n_layers, n_prefix, P;
    int widths[8], acts[8];
    const double *theta;
    double consts[16], lossw[16];
};
struct Fwd64Host {
    const double *u0;
    double *out, *ustep, *dense;
    int32_t *status;
    int N, n_steps, save_every;
    double dt;
};
struct Adj64Host {
    const double *ustep, *dense, *cot;
    double *grad_u0, *partial;
    int N, n_steps, save_every, fused_l2;
    double dt;
};
struct Adapt64Host {
    double t0, save_dt, abstol, reltol;
    int n_save, max_steps;
    double *tgrid;
    int *nacc;
};
int adj_rows_f64(int N);
cudaError_t launch_fwd_f64(const Shape64Host &, const Fwd64Host &, int solver, const Adapt64Host *adaptive_or_null, cudaStream_t);
cudaError_t launch_adj_f64(const Shape64Host &, const Adj64Host &, const Adapt64Host *adaptive_or_null, cudaStream_t, int *rows_out);
cudaError_t launch_reduce_f64(const double *partial, int nrows, int P1, double *grad, double *loss, cudaStream_t);
cudaError_t launch_l2_cot_f64(const Shape64Host &, const double *out, const double *data, double *cot, double *loss, size_t N, int n_save, cudaStream_t);

}  // namespace b200ude
