// b200ude.cu -- C-ABI entry points (include/b200ude.h) over the sm_100a kernels.
//
// No torch types, no exceptions across the boundary, no CPU fallback: if there is no usable
// CUDA device, or the requested configuration has no kernel, the call fails with a code and a
// message.  Nothing here includes or links the CPU oracle.
#include "../../include/b200ude.h"

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <new>
#include <algorithm>
#include <atomic>
#include <string>

#include "params.h"

using namespace b200ude;

namespace {

thread_local std::string g_create_error;

// kernel families compiled into this build (one translation unit each, see k_*.cu)
//   K_LV32   LV 2 -> 32 -> 32 -> 2 tanh                      BASELINE config 2
//   K_LV5Px  LV 2 -> 5 -> 5 -> 5 -> 2, per-layer activations, x trainable linear rates
//            scenario_1.jl:62-73 (x=0), scenario_2.jl:79-98 (x=1), hudson_bay.jl:77-91 (x=2)
//   K_GENERIC  any LV / SEIR / SEIR_NODE / NODE form with chain widths <= 64 and <= 5 layers (k_generic.cu): functional
//            coverage (seir_exposure.jl:52-64,114-130 shapes), not tuned; also Vern7 and the adaptive path of untuned chains
//   K_FKPP     Fisher-KPP UPDE: pointwise chain 1 -> ... -> 1 + 3-tap periodic stencil (Fisher-KPP-CNN.jl:111-126)
//   K_SEIR64   SEIR exposure UDE 3 -> 64 -> 64 -> 1 tanh, tensor-core kernels (k_seir.cu)      BASELINE config 3
//   K_FKPP16   Fisher-KPP UPDE with the 1 -> 16 -> 16 -> 1 tanh reaction chain (k_fkpp.cu)                BASELINE config 4
enum KernelId { K_NONE = 0, K_LV32, K_LV5P0, K_LV5P1, K_LV5P2, K_GENERIC, K_FKPP, K_SEIR64, K_FKPP16, K_F64 };

int kernel_num_params(KernelId k)
{
    switch (k) {
    case K_LV32: return 2 * 32 + 32 + 32 * 32 + 32 + 32 * 2 + 2;
    case K_SEIR64: return 3 * 64 + 64 + 64 * 64 + 64 + 64 + 1;
    case K_FKPP16: return 16 + 16 + 256 + 16 + 16 + 1 + 5;
    case K_LV5P0: return 87;
    case K_LV5P1: return 88;
    case K_LV5P2: return 89;
    default: return 0;
    }
}

std::atomic<uint64_t> g_serial{0};   // handles may be created from several host threads (one per GPU)

}  // namespace

struct b200ude_handle {
    b200ude_desc desc;
    KernelId kid = K_NONE;
    Variant var;
    ConstTables tab;
    GenericShape gen;
    int P = 0, n_save = 0, D = 0;
    size_t cap = 0;  // max trajectories
    size_t N = 0;    // trajectories of the last forward
    bool have_forward = false;
    bool have_theta = false;
    int sm_count = 0;
    size_t wm_fwd_max = 0, wm_adj_max = 0;   // largest ensembles the warp-collective LV kernels are chosen for (auto mode)
    // device buffers
    float *d_theta = nullptr;
    float *d_ustep = nullptr;
    float *d_dense = nullptr;
    float *d_partial = nullptr;
    size_t partial_blocks = 0;
    // adaptive stepping
    bool adaptive = false;
    float *d_tgrid = nullptr, *d_cot = nullptr, *d_block_loss = nullptr;
    int *d_nacc = nullptr;
    const float *last_out = nullptr;
    AdaptiveGrid ag{};
    // host-buffer path
    float *d_u0 = nullptr, *d_out = nullptr, *d_data = nullptr, *d_gu0 = nullptr, *d_grad = nullptr, *d_loss = nullptr;
    int32_t *d_status = nullptr;
    float *h_loss = nullptr;  // pinned
    cudaStream_t own_stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // host-buffer path: the data upload overlaps the forward kernel
    cudaEvent_t data_ready = nullptr, data_ready2 = nullptr;
    RkcHost rkc;                    // solver = B200UDE_RKC2: recurrence tables for desc.n_stages
    // fused reduce + all-reduce over NVLink peer memory (b200ude_peer_*)
    void *d_peer_buf = nullptr;     // this rank's exchange buffer (cudaMalloc, exported with CUDA IPC)
    PeerLinks peer;                 // every rank's buffer as mapped here
    bool peer_attached = false;
    // on-device optimiser (b200ude_adam_*, b200ude_train_adam)
    float *d_u0_keep = nullptr, *d_aux_out = nullptr;   // Vern7: u0 of the last forward, saved states of the Tsit5 re-solve
    bool vern7_pending = false;
    float *d_adam_m = nullptr, *d_adam_v = nullptr, *d_train_out = nullptr;
    int *d_adam_t = nullptr;
    int adam_t = 0;   // host mirror of the step counter
    // double-precision path (dtype = B200UDE_F64, kid = K_F64): every device array of the handle and of the callers is double
    Shape64Host sh64{};
    double *q_theta = nullptr, *q_ustep = nullptr, *q_dense = nullptr, *q_partial = nullptr, *q_tgrid = nullptr, *q_cot = nullptr;
    double *q_u0_keep = nullptr, *q_aux_out = nullptr;
    const double *q_last_out = nullptr;
    size_t dev_bytes = 0;
    std::string err;
};

// ---- batched independent trainings (b200ude_batch_*, k_batch.cu) ---------------------------------------------------------------
struct b200ude_batch_handle {
    b200ude_desc desc;
    int P = 0, n_save = 0;
    size_t cap = 0;        // member capacity
    size_t members = 0;    // members whose theta set_params has stored
    ConstTables tab;
    float *d_theta = nullptr;             // [cap][P]
    float *d_m = nullptr, *d_v = nullptr; // [P][cap]
    float *d_ustep = nullptr, *d_dense = nullptr, *d_out = nullptr;   // forward record [..][D][M], saved-state scratch
    int32_t *d_t = nullptr;               // [cap] ADAM steps each member has taken since set_params
    float *d_best = nullptr;              // [cap][P] each member's best pre-update theta since set_params
    float *d_best_loss = nullptr;         // [cap] its loss (+inf: no finite loss yet)
    std::string err;
};

namespace {

// where a failure's message goes: the handle's own string, or the calling thread's last create() error
std::string &err_of(b200ude_handle *h) { return h ? h->err : g_create_error; }
std::string &err_of(b200ude_batch_handle *h) { return h ? h->err : g_create_error; }
std::string &err_of(std::nullptr_t) { return g_create_error; }

template <class H>
int32_t fail(H h, int32_t code, const char *fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    err_of(h) = buf;
    return code;
}

#define CUDA_TRY(h, expr)                                                                                \
    do {                                                                                                 \
        cudaError_t e_ = (expr);                                                                         \
        if (e_ != cudaSuccess) {                                                                         \
            return fail((h), (int32_t)e_, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
        }                                                                                                \
    } while (0)

template <class T>
cudaError_t dalloc(b200ude_handle *h, T **p, size_t count)
{
    cudaError_t e = cudaMalloc((void **)p, count * sizeof(T));
    if (e == cudaSuccess) h->dev_bytes += count * sizeof(T);
    return e;
}

// RKC2 (Sommeijer, Shampine, Verwer 1998) recurrence coefficients, stage abscissae and the quadrature weights of the stage
// integrands (from running the recurrence on unit impulses)
void rkc2_tables(int s, RkcHost *out)
{
    const double eps = 2.0 / 13.0, w0 = 1.0 + eps / ((double)s * s);
    double T[65], dT[65], d2T[65], b[65] = {0}, mu[65] = {0}, nu[65] = {0}, mt[65] = {0}, ga[65] = {0}, c[65] = {0};
    double W[65][65];   // 33 KB of stack, host side only
    T[0] = 1; T[1] = w0; dT[0] = 0; dT[1] = 1; d2T[0] = 0; d2T[1] = 0;
    for (int j = 2; j <= s; ++j) {
        T[j] = 2 * w0 * T[j - 1] - T[j - 2];
        dT[j] = 2 * T[j - 1] + 2 * w0 * dT[j - 1] - dT[j - 2];
        d2T[j] = 4 * dT[j - 1] + 2 * w0 * d2T[j - 1] - d2T[j - 2];
    }
    const double w1 = dT[s] / d2T[s];
    for (int j = 2; j <= s; ++j) b[j] = d2T[j] / (dT[j] * dT[j]);
    b[0] = b[1] = b[2];
    const double mt1 = b[1] * w1;
    for (int j = 2; j <= s; ++j) {
        mu[j] = 2 * b[j] * w0 / b[j - 1];
        nu[j] = -b[j] / b[j - 2];
        mt[j] = 2 * b[j] * w1 / b[j - 1];
        ga[j] = -(1.0 - b[j - 1] * T[j - 1]) * mt[j];
    }
    memset(W, 0, sizeof W);
    c[0] = 0; c[1] = mt1; W[1][0] = mt1;
    for (int j = 2; j <= s; ++j) {
        c[j] = mu[j] * c[j - 1] + nu[j] * c[j - 2] + mt[j] + ga[j];
        for (int k = 0; k < j; ++k) W[j][k] = mu[j] * W[j - 1][k] + nu[j] * W[j - 2][k];
        W[j][j - 1] += mt[j];
        W[j][0] += ga[j];
    }
    *out = RkcHost();
    out->s = s; out->mt1 = (float)mt1;
    for (int j = 0; j <= s; ++j) {
        out->mu[j] = (float)mu[j]; out->nu[j] = (float)nu[j]; out->mt[j] = (float)mt[j]; out->ga[j] = (float)ga[j]; out->c[j] = (float)c[j];
        out->w[j] = j < s ? (float)W[s][j] : 0.0f;
    }
}

int env_int(const char *name, int dflt)
{
    const char *s = getenv(name);
    return s && *s ? atoi(s) : dflt;
}

bool generic_ok(const b200ude_desc &d)
{
    if (d.n_layers < 1 || d.n_layers > 5) return false;
    for (int l = 0; l <= d.n_layers; ++l)
        if (d.widths[l] < 1 || d.widths[l] > 64) return false;
    for (int l = 0; l < d.n_layers; ++l)
        if (d.acts[l] < 0 || d.acts[l] > 2) return false;
    const int din = d.widths[0], dout = d.widths[d.n_layers];
    if (d.model == B200UDE_MODEL_LV) return d.state_dim == 2 && din == 2 && dout == 2 && d.n_prefix >= 0 && d.n_prefix <= 2 && d.n_consts >= 2;
    if (d.model == B200UDE_MODEL_SEIR) return d.state_dim == 7 && din == 3 && dout == 1 && d.n_prefix == 0 && d.n_consts >= 9;
    if (d.model == B200UDE_MODEL_FKPP) return d.state_dim >= 3 && d.state_dim <= 256 && din == 1 && dout == 1 && d.n_prefix == 0 && d.n_suffix == 5 && d.n_loss_weights == 0;
    if (d.model == B200UDE_MODEL_SEIR_NODE) return d.state_dim == 7 && din == 7 && dout == 7 && d.n_prefix == 0 && d.n_consts >= 9;
    if (d.model == B200UDE_MODEL_NODE) return d.state_dim >= 1 && d.state_dim <= 8 && din == d.state_dim && dout == d.state_dim && d.n_prefix == 0;
    return false;
}

// kernel family of the LV 2-32-32-2 chain for an ensemble of N: mode 1 = always warp-collective, 0 = never, -1 = by size
bool use_wm(int mode, size_t N, size_t n_max) { return mode > 0 || (mode < 0 && N <= n_max); }

KernelId pick_kernel(const b200ude_desc &d)
{
    if (d.model == B200UDE_MODEL_LV && d.state_dim == 2 && d.acts[d.n_layers - 1] == B200UDE_ACT_IDENTITY) {
        if (d.n_layers == 3 && d.widths[0] == 2 && d.widths[1] == 32 && d.widths[2] == 32 && d.widths[3] == 2 &&
            d.acts[0] == B200UDE_ACT_TANH && d.acts[1] == B200UDE_ACT_TANH && d.n_prefix == 0)
            return K_LV32;
        if (d.n_layers == 4 && d.widths[0] == 2 && d.widths[1] == 5 && d.widths[2] == 5 && d.widths[3] == 5 && d.widths[4] == 2) {
            if (d.n_prefix == 0) return K_LV5P0;
            if (d.n_prefix == 1) return K_LV5P1;
            if (d.n_prefix == 2) return K_LV5P2;
        }
    }
    if (!generic_ok(d)) return K_NONE;
    if (d.model == B200UDE_MODEL_SEIR && d.n_layers == 3 && d.widths[1] == 64 && d.widths[2] == 64 && d.acts[0] == B200UDE_ACT_TANH &&
        d.acts[1] == B200UDE_ACT_TANH && d.acts[2] == B200UDE_ACT_IDENTITY && d.n_suffix == 0 && env_int("B200UDE_SEIR_TC", 1))
        return K_SEIR64;
    if (d.model == B200UDE_MODEL_FKPP && d.n_layers == 3 && d.widths[1] == 16 && d.widths[2] == 16 && d.acts[0] == B200UDE_ACT_TANH &&
        d.acts[1] == B200UDE_ACT_TANH && d.acts[2] == B200UDE_ACT_IDENTITY && env_int("B200UDE_FKPP_TUNED", 1))
        return K_FKPP16;
    return d.model == B200UDE_MODEL_FKPP ? K_FKPP : K_GENERIC;
}


// Tsit5 forward solve with the dense record (stage derivatives) the interpolating adjoint reads
int32_t tsit5_forward(b200ude_handle *h, const float *u0, size_t N, float *out, int32_t *status, cudaStream_t st)
{
    FwdParams p;
    p.u0 = u0; p.out = out; p.ustep = h->d_ustep; p.dense = h->d_dense; p.status = status; p.theta = h->d_theta;
    p.N = (int)N; p.n_steps = h->desc.n_steps; p.save_every = h->desc.save_every; p.P = h->P; p.dt = (float)h->desc.dt;
    cudaError_t e = cudaSuccess;
    if (h->adaptive) {
        e = h->kid == K_LV32 ? launch_fwd_lv32_adaptive(h->var, h->tab, p, h->ag, st)
            : h->kid == K_SEIR64 ? launch_fwd_seir_adaptive(h->var, h->tab, p, h->ag, st) : launch_fwd_adaptive(h->gen, h->tab, p, h->ag, st);
        CUDA_TRY(h, e);
        h->last_out = out;
        return B200UDE_OK;
    }
    if (h->desc.solver == B200UDE_RKC2) {
        CUDA_TRY(h, launch_fwd_fkpp16_rkc(h->var, h->tab, h->rkc, p, h->D, st));
        return B200UDE_OK;
    }
    switch (h->kid) {
    case K_LV32:
        // small / medium ensembles: the warp-collective family (latency per stage ~4x lower); large ones: tcgen05
        e = use_wm(h->var.fwd_wm, N, h->wm_fwd_max) ? launch_fwd_lv32_wm(h->var, h->tab, p, st) : launch_fwd_lv32(h->var, h->tab, p, st);
        break;
    case K_LV5P0: e = launch_fwd_lv5(0, h->var, h->tab, p, st); break;
    case K_LV5P1: e = launch_fwd_lv5(1, h->var, h->tab, p, st); break;
    case K_LV5P2: e = launch_fwd_lv5(2, h->var, h->tab, p, st); break;
    case K_GENERIC: e = launch_fwd_generic(h->gen, h->tab, p, st); break;
    case K_FKPP: e = launch_fwd_fkpp(h->gen, h->tab, p, st); break;
    case K_SEIR64: e = launch_fwd_seir(h->var, h->tab, p, st); break;
    case K_FKPP16: e = launch_fwd_fkpp16(h->var, h->tab, p, h->D, st); break;
    default: return fail(h, B200UDE_EUNSUPPORTED, "forward: no kernel");
    }
    CUDA_TRY(h, e);
    return B200UDE_OK;
}

int32_t do_forward(b200ude_handle *h, const float *u0, size_t N, float *out, int32_t *status, cudaStream_t st)
{
    CUDA_TRY(h, cudaSetDevice(h->desc.device));   // launches, symbol copies and function attributes go to the handle's device
    if (!h->have_theta) return fail(h, B200UDE_ESTATE, "forward: set_params has not been called");
    if (N == 0 || N > h->cap) return fail(h, B200UDE_EINVAL, "forward: N=%zu outside (0, max_trajectories=%zu]", N, h->cap);
    if (!u0 || !out) return fail(h, B200UDE_EINVAL, "forward: null pointer");
    if (h->desc.solver == B200UDE_VERN7) {
        // Vern7 writes the saved states only.  Its lazy dense output is not available (SURVEY.md App. A.3), so the
        // interpolating adjoint of a Vern7 solve runs over a Tsit5 re-solve from the same u0 with the same step /
        // tolerances, launched by the first adjoint call (do_adjoint); u0 is kept for that.
        FwdParams p;
        p.u0 = u0; p.out = out; p.ustep = nullptr; p.dense = nullptr; p.status = status; p.theta = h->d_theta;
        p.N = (int)N; p.n_steps = h->desc.n_steps; p.save_every = h->desc.save_every; p.P = h->P; p.dt = (float)h->desc.dt;
        if (h->adaptive) CUDA_TRY(h, launch_fwd_vern7_adaptive(h->gen, h->tab, p, h->ag, st));
        else if (h->kid == K_SEIR64) CUDA_TRY(h, launch_fwd_seir_vern7(h->var, h->tab, p, st));   // tensor-core kernels (seir_tc.cuh)
        else CUDA_TRY(h, launch_fwd_vern7(h->gen, h->tab, p, st));
        if (!h->d_u0_keep && dalloc(h, &h->d_u0_keep, (size_t)h->D * h->cap) != cudaSuccess)
            return fail(h, B200UDE_ENOMEM, "forward: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        CUDA_TRY(h, cudaMemcpyAsync(h->d_u0_keep, u0, sizeof(float) * (size_t)h->D * N, cudaMemcpyDeviceToDevice, st));
        h->N = N;
        h->have_forward = false;
        h->vern7_pending = true;
        return B200UDE_OK;
    }
    int32_t rc = tsit5_forward(h, u0, N, out, status, st);
    if (rc) return rc;
    h->N = N;
    h->have_forward = true;
    return B200UDE_OK;
}

// split: two events (data of the first / second half of the trajectories resident) for the host-buffer path: the warp-collective LV
// adjoint then runs as two sub-range launches, the first one under the second half's upload
int32_t do_adjoint(b200ude_handle *h, bool l2, const float *cot, float *loss, float *grad_theta,
                   float *grad_u0, cudaStream_t st, bool peer = false, const cudaEvent_t *split = nullptr, size_t split_at = 0)
{
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    if (peer && !h->peer_attached) return fail(h, B200UDE_ESTATE, "adjoint_l2_allreduce: b200ude_peer_attach has not been called");
    if (peer && h->adaptive) return fail(h, B200UDE_EUNSUPPORTED, "adjoint_l2_allreduce: not available with adaptive stepping (all-reduce the result of b200ude_adjoint_l2 instead)");
    if (h->desc.solver == B200UDE_VERN7 && h->vern7_pending) {
        if (!h->d_aux_out && dalloc(h, &h->d_aux_out, (size_t)h->n_save * (size_t)h->D * h->cap) != cudaSuccess)
            return fail(h, B200UDE_ENOMEM, "adjoint: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        int32_t rc = tsit5_forward(h, h->d_u0_keep, h->N, h->d_aux_out, nullptr, st);
        if (rc) return rc;
        h->vern7_pending = false;
        h->have_forward = true;
    }
    if (!h->have_forward) return fail(h, B200UDE_ESTATE, "adjoint: no stored forward solution (call b200ude_forward first)");
    if (!cot || !grad_theta) return fail(h, B200UDE_EINVAL, "adjoint: null pointer");
    const bool split_ok = split && h->kid == K_LV32 && !h->adaptive && h->desc.solver != B200UDE_RKC2 && !h->var.discrete &&
                          use_wm(h->var.adj_wm, h->N, h->wm_adj_max) && split_at > 0 && split_at < h->N;
    if (split && !split_ok) {   // every other kernel family reads the whole data array
        CUDA_TRY(h, cudaStreamWaitEvent(st, split[0], 0));
        CUDA_TRY(h, cudaStreamWaitEvent(st, split[1], 0));
    }
    AdjParams p;
    p.ustep = h->d_ustep; p.dense = h->d_dense; p.cot = cot; p.grad_u0 = grad_u0; p.partial = h->d_partial;
    p.theta = h->d_theta; p.N = (int)h->N; p.n_steps = h->desc.n_steps; p.save_every = h->desc.save_every; p.P = h->P;
    p.fused_l2 = l2 ? 1 : 0;
    p.dt = (float)h->desc.dt;
    cudaError_t e = cudaSuccess;
    int grid = 0;
    if (h->adaptive) {
        if (l2) {   // form the cotangent 2 w (out - data) from the interpolated saved states of the last forward
            CUDA_TRY(h, launch_l2_cot(h->tab, h->last_out, cot, h->d_cot, h->d_block_loss, h->D, h->N, h->n_save, st));
            p.cot = h->d_cot;
            p.fused_l2 = 0;
        }
        if (h->kid == K_LV32) CUDA_TRY(h, launch_adj_lv32_adaptive(h->var, h->tab, p, h->ag, st, &grid));
        else if (h->kid == K_SEIR64) CUDA_TRY(h, launch_adj_seir_adaptive(h->var, h->tab, p, h->ag, st, &grid));
        else CUDA_TRY(h, launch_adj_adaptive(h->gen, h->tab, p, h->ag, st, &grid));
        CUDA_TRY(h, launch_reduce(h->d_partial, grid, h->P + 1, grad_theta, loss, st));
        if (l2 && loss) CUDA_TRY(h, launch_l2_finish(h->d_block_loss, loss, st));
        return B200UDE_OK;
    }
    if (h->desc.solver == B200UDE_RKC2) {
        CUDA_TRY(h, launch_adj_fkpp16_rkc(h->var, h->tab, h->rkc, p, h->D, st, &grid));
        if (peer) CUDA_TRY(h, launch_reduce_exchange(h->d_partial, grid, h->P + 1, h->peer, grad_theta, loss, st));
        else CUDA_TRY(h, launch_reduce(h->d_partial, grid, h->P + 1, grad_theta, loss, st));
        return B200UDE_OK;
    }
    switch (h->kid) {
    case K_LV32:
        if (split_ok) {
            int g0 = 0, g1 = 0;
            AdjParams q = p;
            q.n0 = 0; q.n_cnt = (int)split_at; q.row0 = 0;
            CUDA_TRY(h, cudaStreamWaitEvent(st, split[0], 0));
            e = launch_adj_lv32_wm(h->var, h->tab, q, st, &g0);
            if (e == cudaSuccess) {
                q.n0 = (int)split_at; q.n_cnt = (int)(h->N - split_at); q.row0 = g0;
                CUDA_TRY(h, cudaStreamWaitEvent(st, split[1], 0));
                e = launch_adj_lv32_wm(h->var, h->tab, q, st, &g1);
            }
            grid = g0 + g1;
        } else {
            e = (!h->var.discrete && use_wm(h->var.adj_wm, h->N, h->wm_adj_max)) ? launch_adj_lv32_wm(h->var, h->tab, p, st, &grid)
                                                                                  : launch_adj_lv32(h->var, h->tab, p, st, &grid);
        }
        break;
    case K_LV5P0: e = launch_adj_lv5(0, h->var, h->tab, p, st, &grid); break;
    case K_LV5P1: e = launch_adj_lv5(1, h->var, h->tab, p, st, &grid); break;
    case K_LV5P2: e = launch_adj_lv5(2, h->var, h->tab, p, st, &grid); break;
    case K_GENERIC: e = launch_adj_generic(h->gen, h->tab, p, st, &grid); break;
    case K_FKPP: e = launch_adj_fkpp(h->gen, h->tab, p, st, &grid); break;
    case K_SEIR64: e = launch_adj_seir(h->var, h->tab, p, st, &grid); break;
    case K_FKPP16: e = launch_adj_fkpp16(h->var, h->tab, p, h->D, st, &grid); break;
    default: return fail(h, B200UDE_EUNSUPPORTED, "adjoint: no kernel");
    }
    CUDA_TRY(h, e);
    if (peer) {
        CUDA_TRY(h, launch_reduce_exchange(h->d_partial, grid, h->P + 1, h->peer, grad_theta, loss, st));
    } else {
        CUDA_TRY(h, launch_reduce(h->d_partial, grid, h->P + 1, grad_theta, loss, st));
    }
    return B200UDE_OK;
}


// ---- ADAM on the device (Flux.ADAM(eta, (beta1, beta2)), eps = 1e-8: scenario_1.jl:114, seir_exposure.jl:160) ----
// One CTA: L = loss_scale * L_data + l2_reg * sum theta^2, g = loss_scale * grad + 2 l2_reg theta, then the
// bias-corrected update of theta in place.  The step counter lives in device memory so that the launch arguments
// do not change from iteration to iteration (the training loop is replayed as a CUDA graph).
struct AdamArgs {
    float *theta, *m, *v;
    const float *grad, *loss;   // loss may be null
    float *loss_history;        // [..] or null; slot (t - 1 - t_base) receives the pre-update loss
    int *t;
    int P, t_base, reg_from;   // the L2 term covers theta[reg_from:] (scenario_2.jl:113: sum(abs2, theta[2:end]) skips the trainable physics rate)
    float eta, beta1, beta2, eps, loss_scale, l2_reg;
};

__global__ void __launch_bounds__(1024, 1) adam_kernel(AdamArgs a)
{
    __shared__ float red[32];
    __shared__ int s_t;
    if (threadIdx.x == 0) s_t = *a.t + 1;
    float sq = 0.0f;
    if (a.l2_reg != 0.0f)
        for (int i = a.reg_from + threadIdx.x; i < a.P; i += blockDim.x) sq = fmaf(a.theta[i], a.theta[i], sq);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sq;
    __syncthreads();
    const int t = s_t;
    if (threadIdx.x == 0) {
        float tot = 0.0f;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) tot += red[w];   // fixed order
        if (a.loss_history && a.loss) a.loss_history[t - 1 - a.t_base] = fmaf(a.loss_scale, *a.loss, a.l2_reg * tot);
        *a.t = t;
    }
    const float c1 = (float)(1.0 / (1.0 - pow((double)a.beta1, (double)t)));
    const float c2 = (float)(1.0 / (1.0 - pow((double)a.beta2, (double)t)));
    for (int i = threadIdx.x; i < a.P; i += blockDim.x) {
        const float th = a.theta[i];
        const float g = fmaf(a.loss_scale, a.grad[i], i >= a.reg_from ? 2.0f * a.l2_reg * th : 0.0f);
        const float m = fmaf(a.beta1, a.m[i], (1.0f - a.beta1) * g);
        const float v = fmaf(a.beta2, a.v[i], (1.0f - a.beta2) * g * g);
        a.m[i] = m;
        a.v[i] = v;
        a.theta[i] = th - a.eta * (m * c1) / (sqrtf(v * c2) + a.eps);
    }
}

int32_t ensure_adam(b200ude_handle *h)
{
    if (h->kid == K_F64) return fail(h, B200UDE_EUNSUPPORTED, "adam: not available for B200UDE_F64 handles (update theta on the host side)");
    if (h->d_adam_m) return B200UDE_OK;
    bool ok = dalloc(h, &h->d_adam_m, (size_t)h->P) == cudaSuccess && dalloc(h, &h->d_adam_v, (size_t)h->P) == cudaSuccess &&
              dalloc(h, &h->d_adam_t, 1) == cudaSuccess;
    if (!ok) return fail(h, B200UDE_ENOMEM, "adam: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    // synchronous with respect to the host and to every stream that is used afterwards
    cudaMemset(h->d_adam_m, 0, sizeof(float) * h->P);
    cudaMemset(h->d_adam_v, 0, sizeof(float) * h->P);
    cudaMemset(h->d_adam_t, 0, sizeof(int));
    cudaDeviceSynchronize();
    h->adam_t = 0;
    return B200UDE_OK;
}

int32_t check_adam(b200ude_handle *h, const b200ude_adam *o)
{
    if (!o || o->struct_size != sizeof(b200ude_adam)) return fail(h, B200UDE_EINVAL, "adam: bad options struct");
    if (!(o->eta > 0) || !(o->beta1 >= 0 && o->beta1 < 1) || !(o->beta2 >= 0 && o->beta2 < 1) || !(o->eps > 0))
        return fail(h, B200UDE_EINVAL, "adam: need eta > 0, 0 <= beta < 1, eps > 0");
    if (!h->have_theta) return fail(h, B200UDE_ESTATE, "adam: no parameters set (call b200ude_set_params first)");
    return ensure_adam(h);
}

cudaError_t launch_adam(b200ude_handle *h, const b200ude_adam *o, const float *grad, const float *loss, float *hist, int t_base, cudaStream_t st)
{
    AdamArgs a;
    a.theta = h->d_theta; a.m = h->d_adam_m; a.v = h->d_adam_v; a.grad = grad; a.loss = loss; a.loss_history = hist;
    a.t = h->d_adam_t; a.P = h->P; a.t_base = t_base; a.reg_from = h->desc.n_prefix > 0 ? h->desc.n_prefix : 0;
    a.eta = (float)o->eta; a.beta1 = (float)o->beta1; a.beta2 = (float)o->beta2; a.eps = (float)o->eps;
    a.loss_scale = (float)(o->loss_scale == 0.0 ? 1.0 : o->loss_scale); a.l2_reg = (float)o->l2_reg;
    adam_kernel<<<1, 1024, 0, st>>>(a);
    return cudaGetLastError();
}

// ---- double-precision path (kid = K_F64) ----------------------------------------------------------------------------------
Adapt64Host adapt64(const b200ude_handle *h)
{
    return Adapt64Host{h->desc.t0, h->desc.dt * h->desc.save_every, h->desc.abstol, h->desc.reltol, h->n_save, h->desc.max_steps, h->q_tgrid, h->d_nacc};
}

int32_t tsit5_forward64(b200ude_handle *h, const double *u0, size_t N, double *out, int32_t *status, cudaStream_t st)
{
    Fwd64Host p{u0, out, h->q_ustep, h->q_dense, status, (int)N, h->desc.n_steps, h->desc.save_every, h->desc.dt};
    const Adapt64Host a = adapt64(h);
    CUDA_TRY(h, launch_fwd_f64(h->sh64, p, 0, h->adaptive ? &a : nullptr, st));
    h->q_last_out = out;
    return B200UDE_OK;
}

int32_t do_forward64(b200ude_handle *h, const double *u0, size_t N, double *out, int32_t *status, cudaStream_t st)
{
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    if (!h->have_theta) return fail(h, B200UDE_ESTATE, "forward: set_params has not been called");
    if (N == 0 || N > h->cap) return fail(h, B200UDE_EINVAL, "forward: N=%zu outside (0, max_trajectories=%zu]", N, h->cap);
    if (!u0 || !out) return fail(h, B200UDE_EINVAL, "forward: null pointer");
    if (h->desc.solver == B200UDE_VERN7) {
        // saved states only; the interpolating adjoint runs over a Tsit5 re-solve with the same step / tolerances (as in fp32)
        Fwd64Host p{u0, out, nullptr, nullptr, status, (int)N, h->desc.n_steps, h->desc.save_every, h->desc.dt};
        const Adapt64Host a = adapt64(h);
        CUDA_TRY(h, launch_fwd_f64(h->sh64, p, 1, h->adaptive ? &a : nullptr, st));
        if (!h->q_u0_keep && dalloc(h, &h->q_u0_keep, (size_t)h->D * h->cap) != cudaSuccess)
            return fail(h, B200UDE_ENOMEM, "forward: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        CUDA_TRY(h, cudaMemcpyAsync(h->q_u0_keep, u0, sizeof(double) * (size_t)h->D * N, cudaMemcpyDeviceToDevice, st));
        h->N = N;
        h->have_forward = false;
        h->vern7_pending = true;
        return B200UDE_OK;
    }
    int32_t rc = tsit5_forward64(h, u0, N, out, status, st);
    if (rc) return rc;
    h->N = N;
    h->have_forward = true;
    return B200UDE_OK;
}

int32_t do_adjoint64(b200ude_handle *h, bool l2, const double *cot, double *loss, double *grad_theta, double *grad_u0, cudaStream_t st)
{
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    if (h->desc.solver == B200UDE_VERN7 && h->vern7_pending) {
        if (!h->q_aux_out && dalloc(h, &h->q_aux_out, (size_t)h->n_save * (size_t)h->D * h->cap) != cudaSuccess)
            return fail(h, B200UDE_ENOMEM, "adjoint: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
        int32_t rc = tsit5_forward64(h, h->q_u0_keep, h->N, h->q_aux_out, nullptr, st);
        if (rc) return rc;
        h->vern7_pending = false;
        h->have_forward = true;
    }
    if (!h->have_forward) return fail(h, B200UDE_ESTATE, "adjoint: no stored forward solution (call b200ude_forward first)");
    if (!cot || !grad_theta) return fail(h, B200UDE_EINVAL, "adjoint: null pointer");
    Adj64Host p{h->q_ustep, h->q_dense, cot, grad_u0, h->q_partial, (int)h->N, h->desc.n_steps, h->desc.save_every, l2 ? 1 : 0, h->desc.dt};
    int rows = 0;
    if (h->adaptive) {
        const Adapt64Host a = adapt64(h);
        double *loss_l2 = nullptr;
        if (l2) {   // cotangent 2 w (out - data) from the interpolated saved states of the last Tsit5 forward; the loss goes straight to `loss`
            CUDA_TRY(h, launch_l2_cot_f64(h->sh64, h->q_last_out, cot, h->q_cot, loss, h->N, h->n_save, st));
            p.cot = h->q_cot;
            p.fused_l2 = 0;
            loss_l2 = loss;
        }
        CUDA_TRY(h, launch_adj_f64(h->sh64, p, &a, st, &rows));
        CUDA_TRY(h, launch_reduce_f64(h->q_partial, rows, h->P + 1, grad_theta, loss_l2 ? nullptr : loss, st));
        return B200UDE_OK;
    }
    CUDA_TRY(h, launch_adj_f64(h->sh64, p, nullptr, st, &rows));
    CUDA_TRY(h, launch_reduce_f64(h->q_partial, rows, h->P + 1, grad_theta, loss, st));
    return B200UDE_OK;
}

int32_t f64_unsupported(b200ude_handle *h, const char *what)
{
    return fail(h, B200UDE_EUNSUPPORTED, "%s: not available for B200UDE_F64 handles (device-pointer forward / adjoint entry points only)", what);
}

}  // namespace

namespace {

// the checks every batch call shares; fills the fields of p that do not depend on the call
int32_t batch_prepare(b200ude_batch_handle *h, size_t M, const void *u0, int mode, BatchParams &p)
{
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    if (h->members == 0) return fail(h, B200UDE_ESTATE, "batch: b200ude_batch_set_params has not been called");
    if (M == 0 || M > h->members) return fail(h, B200UDE_EINVAL, "batch: M=%zu outside (0, members set=%zu]", M, h->members);
    if (!u0) return fail(h, B200UDE_EINVAL, "batch: null u0");
    p = BatchParams{};
    p.u0 = (const float *)u0; p.out = h->d_out; p.theta = h->d_theta; p.m = h->d_m; p.v = h->d_v;
    p.ustep = h->d_ustep; p.dense = h->d_dense;
    p.t = h->d_t; p.best = h->d_best; p.best_loss = h->d_best_loss;
    p.M = (int)M; p.ldm = (int)h->cap; p.n_steps = h->desc.n_steps; p.save_every = h->desc.save_every; p.mode = mode; p.iters = 1;
    p.dt = (float)h->desc.dt;
    return B200UDE_OK;
}

__global__ void fill_kernel(float *a, float v, size_t n)
{
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) a[i] = v;
}

int32_t batch_launch(b200ude_batch_handle *h, const BatchParams &p, cudaStream_t st)
{
    CUDA_TRY(h, launch_batch(h->desc.n_prefix, h->desc.sensealg == B200UDE_DISCRETE_ADJOINT, h->tab, p, st));
    return B200UDE_OK;
}

}  // namespace

// ---- exported entry points ------------------------------------------------------------------------
extern "C" {

int32_t b200ude_version(void) { return B200UDE_ABI_VERSION; }

const char *b200ude_last_error(const b200ude_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int32_t b200ude_create(const b200ude_desc *d, b200ude_handle **out)
{
    if (!d || !out) return fail(nullptr, B200UDE_EINVAL, "create: null argument");
    *out = nullptr;
    if (d->struct_size != sizeof(b200ude_desc))
        return fail(nullptr, B200UDE_EINVAL, "create: struct_size %u != %zu (ABI mismatch)", d->struct_size, sizeof(b200ude_desc));
    if (d->dtype != B200UDE_F32 && d->dtype != B200UDE_F64) return fail(nullptr, B200UDE_EINVAL, "create: unknown dtype %d", d->dtype);
    if (d->n_layers < 1 || d->n_layers > B200UDE_MAX_LAYERS) return fail(nullptr, B200UDE_EINVAL, "create: n_layers=%d out of range", d->n_layers);
    if (d->solver != B200UDE_TSIT5 && d->solver != B200UDE_VERN7 && d->solver != B200UDE_RKC2)
        return fail(nullptr, B200UDE_EINVAL, "create: unknown solver %d", d->solver);
    if (d->sensealg != B200UDE_INTERPOLATING_ADJOINT && d->sensealg != B200UDE_DISCRETE_ADJOINT)
        return fail(nullptr, B200UDE_EUNSUPPORTED, "create: unknown sensealg %d", d->sensealg);
    if (!(d->dt > 0) || d->n_steps < 1 || d->save_every < 1 || d->n_steps % d->save_every != 0)
        return fail(nullptr, B200UDE_EINVAL, "create: need dt>0, n_steps>=1, save_every>=1 dividing n_steps");
    if (d->max_trajectories == 0 || d->max_trajectories > (1ull << 26)) return fail(nullptr, B200UDE_EINVAL, "create: max_trajectories out of range");
    if (d->n_loss_weights != 0 && d->n_loss_weights != d->state_dim) return fail(nullptr, B200UDE_EINVAL, "create: n_loss_weights must be 0 or state_dim");
    KernelId kid = pick_kernel(*d);
    const bool want64 = d->dtype == B200UDE_F64;
    if (want64) {
        // fp64: the runtime-shape one-trajectory-per-thread kernels (ude_f64.cuh): LV / SEIR / NODE forms, Tsit5 and Vern7,
        // fixed step and adaptive, interpolating adjoint
        if (!generic_ok(*d) || d->model == B200UDE_MODEL_FKPP || d->solver == B200UDE_RKC2 || d->sensealg != B200UDE_INTERPOLATING_ADJOINT)
            return fail(nullptr, B200UDE_EUNSUPPORTED,
                        "create: B200UDE_F64 kernels exist for the LV / SEIR / NODE forms (chain widths <= 64), Tsit5 / Vern7, interpolating adjoint");
        if (d->adaptive && (!(d->abstol > 0) || !(d->reltol > 0) || d->max_steps < 1))
            return fail(nullptr, B200UDE_EINVAL, "create: adaptive stepping needs abstol > 0, reltol > 0, max_steps >= 1");
        kid = K_F64;
    }
    if (!want64 && d->solver == B200UDE_VERN7) {
        if (!generic_ok(*d) || d->model == B200UDE_MODEL_FKPP)
            return fail(nullptr, B200UDE_EUNSUPPORTED, "create: Vern7 kernels exist for the LV / SEIR / NODE forms only");
        // fixed-step Vern7 of the SEIR 3-64-64-1 chain runs on the tensor-core kernels (and so does the Tsit5 re-solve its
        // adjoint uses); every other Vern7 configuration on the runtime-shape kernels
        if (!(kid == K_SEIR64 && !d->adaptive && env_int("B200UDE_SEIR_VERN7_TC", 1))) kid = K_GENERIC;
    }
    if (!want64 && d->adaptive) {
        if (!(d->abstol > 0) || !(d->reltol > 0) || d->max_steps < 1)
            return fail(nullptr, B200UDE_EINVAL, "create: adaptive stepping needs abstol > 0, reltol > 0, max_steps >= 1");
        if (!generic_ok(*d) || d->model == B200UDE_MODEL_FKPP)
            return fail(nullptr, B200UDE_EUNSUPPORTED, "create: adaptive stepping is implemented for the LV / SEIR / NODE forms (chain widths <= 64)");
        // adaptive solves run on the runtime-shape kernels, except the headline chain (tensor-core kernels with CTA-uniform attempt loops)
        if (!((kid == K_LV32 || kid == K_SEIR64) && d->solver == B200UDE_TSIT5 && env_int("B200UDE_ADAPTIVE_TC", 1))) kid = K_GENERIC;
    }
    if (d->solver == B200UDE_RKC2) {
        if (d->n_stages < 2 || d->n_stages > 64) return fail(nullptr, B200UDE_EINVAL, "create: RKC2 needs 2 <= n_stages <= 64 (stability interval ~ 0.65 n_stages^2 >= dt * spectral radius)");
        if (kid != K_FKPP16 || d->state_dim % 2 != 0 || d->adaptive || d->sensealg != B200UDE_INTERPOLATING_ADJOINT || !env_int("B200UDE_FKPP_PACKED", 1))
            return fail(nullptr, B200UDE_EUNSUPPORTED,
                        "create: RKC2 has kernels for the Fisher-KPP UPDE with the 1-16-16-1 chain on even grids (fixed step, interpolating adjoint)");
    }
    if (d->sensealg == B200UDE_DISCRETE_ADJOINT &&
        (d->adaptive || d->solver != B200UDE_TSIT5 || !(kid == K_LV32 || kid == K_LV5P0 || kid == K_LV5P1 || kid == K_LV5P2)))
        return fail(nullptr, B200UDE_EUNSUPPORTED,
                    "create: the discrete adjoint has kernels for fixed-step Tsit5 on the LV chains 2-32-32-2 and 2-5-5-5-2 (the scripts that use ForwardDiffSensitivity)");
    if (kid == K_NONE)
        return fail(nullptr, B200UDE_EUNSUPPORTED,
                    "create: no sm_100a kernel for this model/chain (built: LV 2-32-32-2 tanh; LV 2-5-5-5-2; generic LV/SEIR/NODE chains with widths <= 64, <= 5 layers)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(nullptr, B200UDE_ENODEVICE, "create: no CUDA device (%s)", cudaGetErrorString(e));
    if (d->device < 0 || d->device >= ndev) return fail(nullptr, B200UDE_EINVAL, "create: device %d of %d", d->device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, d->device);
    if (e != cudaSuccess) return fail(nullptr, (int32_t)e, "create: cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, B200UDE_ENODEVICE, "create: device %d is sm_%d%d; this library carries sm_100a code only", d->device, prop.major, prop.minor);
    e = cudaSetDevice(d->device);
    if (e != cudaSuccess) return fail(nullptr, (int32_t)e, "create: cudaSetDevice: %s", cudaGetErrorString(e));

    b200ude_handle *h = new (std::nothrow) b200ude_handle();
    if (!h) return fail(nullptr, B200UDE_ENOMEM, "create: out of host memory");
    const uint64_t serial = ++g_serial;   // taken once: gen.serial and tab.serial must agree
    h->desc = *d;
    h->kid = kid;
    h->D = d->state_dim;
    h->n_save = d->n_steps / d->save_every + 1;
    h->cap = (size_t)d->max_trajectories;
    h->sm_count = prop.multiProcessorCount;
    h->adaptive = d->adaptive != 0;
    h->P = kernel_num_params(kid);
    if (kid == K_GENERIC || kid == K_FKPP || kid == K_F64) {
        int P = d->n_prefix + d->n_suffix;
        for (int l = 0; l < d->n_layers; ++l) P += d->widths[l] * d->widths[l + 1] + d->widths[l + 1];
        h->P = P;
        h->gen.serial = serial;   // same serial as the tables set below
        h->gen.model = d->model; h->gen.D = d->state_dim; h->gen.din = d->widths[0]; h->gen.dout = d->widths[d->n_layers];
        h->gen.n_layers = d->n_layers; h->gen.n_prefix = d->n_prefix; h->gen.P = P;
        for (int l = 0; l < 8; ++l) { h->gen.widths[l] = l <= d->n_layers ? d->widths[l] : 0; h->gen.acts[l] = l < d->n_layers ? d->acts[l] : 0; }
        if (kid != K_F64 && P > 12288) { delete h; return fail(nullptr, B200UDE_EUNSUPPORTED, "create: %d parameters exceed the constant-bank budget", P); }
    }
    h->var.approx_tanh = (d->flags & B200UDE_FLAG_APPROX_TANH) ? 1 : 0;
    h->var.discrete = d->sensealg == B200UDE_DISCRETE_ADJOINT ? 1 : 0;
    if (d->solver == B200UDE_RKC2) rkc2_tables(d->n_stages, &h->rkc);
    // tuning knobs for experiments (defaults are the measured-best variant, see DESIGN.md)
    h->var.fwd_smem = env_int("B200UDE_FWD_SMEM", 0);
    h->var.fwd_T = env_int("B200UDE_FWD_T", 1) == 2 ? 2 : 1;
    h->var.adj_smem = env_int("B200UDE_ADJ_SMEM", 0);
    // default: tcgen05 (3xTF32) kernels; B200UDE_FWD_TC=0 / B200UDE_ADJ_TC=0 select the FFMA2-packed CUDA-core kernels
    h->var.fwd_tc = env_int("B200UDE_FWD_TC", 1);
    h->var.adj_tc = env_int("B200UDE_ADJ_TC", 2);   // 2: gradient GEMM on mma.sync (3xTF32), 1: on the FMA pipe (FFMA2)
    // warp-collective mma.sync family (lv32_wm.cuh): -1 = chosen per call from the ensemble size, 0 = off, 1 = always
    h->var.fwd_wm = env_int("B200UDE_FWD_WM", -1);
    h->var.adj_wm = env_int("B200UDE_ADJ_WM", -1);
    h->var.wm_groups = env_int("B200UDE_WM_G", 1);
    h->var.wm_rows = env_int("B200UDE_WM_R", 0);
    h->var.wm_r1_max = env_int("B200UDE_WM_R1_MAX", 4736);
    h->wm_fwd_max = (size_t)env_int("B200UDE_WM_FWD_MAX", 1 << 26);
    h->wm_adj_max = (size_t)env_int("B200UDE_WM_ADJ_MAX", 1 << 26);

    if (kid == K_F64) {
        const size_t N64 = h->cap, D64 = (size_t)h->D;
        const size_t rec = h->adaptive ? (size_t)d->max_steps : (size_t)d->n_steps;
        h->partial_blocks = (size_t)adj_rows_f64((int)N64);
        bool ok64 = dalloc(h, &h->q_theta, (size_t)h->P + 1) == cudaSuccess && dalloc(h, &h->q_ustep, (rec + 1) * D64 * N64) == cudaSuccess &&
                    dalloc(h, &h->q_dense, (rec * 6 + 1) * D64 * N64) == cudaSuccess &&
                    dalloc(h, &h->q_partial, h->partial_blocks * (size_t)(h->P + 1)) == cudaSuccess;
        if (h->adaptive)
            ok64 = ok64 && dalloc(h, &h->q_tgrid, (rec + 1) * N64) == cudaSuccess && dalloc(h, &h->d_nacc, N64) == cudaSuccess &&
                   dalloc(h, &h->q_cot, (size_t)h->n_save * D64 * N64) == cudaSuccess;
        if (!ok64) {
            g_create_error = std::string("create: device allocation failed: ") + cudaGetErrorString(cudaGetLastError());
            b200ude_destroy(h);
            return B200UDE_ENOMEM;
        }
        cudaMemset(h->q_theta, 0, sizeof(double) * ((size_t)h->P + 1));
        Shape64Host &sh = h->sh64;
        sh.serial = serial; sh.model = d->model; sh.D = d->state_dim; sh.din = d->widths[0]; sh.dout = d->widths[d->n_layers];
        sh.n_layers = d->n_layers; sh.n_prefix = d->n_prefix; sh.P = h->P; sh.theta = h->q_theta;
        for (int l = 0; l < 8; ++l) { sh.widths[l] = l <= d->n_layers ? d->widths[l] : 0; sh.acts[l] = l < d->n_layers ? d->acts[l] : 0; }
        for (int i = 0; i < 16; ++i) {
            sh.consts[i] = i < d->n_consts ? d->consts[i] : 0.0;
            sh.lossw[i] = d->n_loss_weights > 0 ? (i < d->n_loss_weights ? d->loss_weights[i] : 0.0) : 1.0;
        }
        if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
            g_create_error = "create: stream allocation failed";
            b200ude_destroy(h);
            return B200UDE_ENOMEM;
        }
        *out = h;
        return B200UDE_OK;
    }
    const size_t N = h->cap, D = (size_t)h->D;
    h->partial_blocks = (size_t)(kid == K_LV32 ? std::max(adj_grid_lv32((int)N), adj_rows_lv32_wm((int)N)) : kid == K_GENERIC ? adj_rows_generic((int)N) : kid == K_FKPP ? adj_rows_fkpp((int)N, d->state_dim) : kid == K_SEIR64 ? adj_rows_seir((int)N) : kid == K_FKPP16 ? adj_rows_fkpp16((int)N, d->state_dim) : adj_grid_lv5((int)N));
    bool ok = true;
    ok = ok && dalloc(h, &h->d_theta, (size_t)((h->P + 3) / 4) * 4) == cudaSuccess;
    const size_t rec_steps = h->adaptive ? (size_t)d->max_steps : (size_t)d->n_steps;   // capacity of the step record
    ok = ok && dalloc(h, &h->d_ustep, (rec_steps + 1) * D * N) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_dense, (rec_steps * 6 + 1) * D * N) == cudaSuccess;
    if (h->adaptive) {
        ok = ok && dalloc(h, &h->d_tgrid, (rec_steps + 1) * N) == cudaSuccess;
        ok = ok && dalloc(h, &h->d_nacc, N) == cudaSuccess;
        ok = ok && dalloc(h, &h->d_cot, (size_t)h->n_save * D * N) == cudaSuccess;
        ok = ok && dalloc(h, &h->d_block_loss, (size_t)L2_BLOCKS) == cudaSuccess;
    }
    ok = ok && dalloc(h, &h->d_partial, h->partial_blocks * (size_t)(h->P + 1)) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_grad, (size_t)h->P) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_loss, 1) == cudaSuccess;
    if (!ok) {
        cudaError_t le = cudaGetLastError();
        g_create_error = std::string("create: device allocation failed: ") + cudaGetErrorString(le);
        b200ude_destroy(h);
        return B200UDE_ENOMEM;
    }
    cudaMemset(h->d_theta, 0, sizeof(float) * ((h->P + 3) / 4) * 4);
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->data_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&h->data_ready2, cudaEventDisableTiming) != cudaSuccess ||
        cudaMallocHost((void **)&h->h_loss, sizeof(float)) != cudaSuccess) {
        g_create_error = "create: stream / pinned allocation failed";
        b200ude_destroy(h);
        return B200UDE_ENOMEM;
    }
    h->tab.serial = serial;
    h->ag.t0 = (float)d->t0; h->ag.save_dt = (float)(d->dt * d->save_every); h->ag.abstol = (float)d->abstol; h->ag.reltol = (float)d->reltol;
    h->ag.n_save = h->n_save; h->ag.max_steps = d->max_steps; h->ag.tgrid = h->d_tgrid; h->ag.nacc = h->d_nacc;
    h->tab.d_theta = h->d_theta;
    h->tab.P = h->P;
    for (int i = 0; i < 16; ++i) {
        h->tab.consts[i] = i < d->n_consts ? (float)d->consts[i] : 0.0f;
        h->tab.lossw[i] = d->n_loss_weights > 0 ? (i < d->n_loss_weights ? (float)d->loss_weights[i] : 0.0f) : 1.0f;
    }
    for (int i = 0; i < 8; ++i) h->tab.acts[i] = i < d->n_layers ? d->acts[i] : 0;
    *out = h;
    return B200UDE_OK;
}

void b200ude_destroy(b200ude_handle *h)
{
    if (!h) return;
    cudaFree(h->d_theta); cudaFree(h->d_ustep); cudaFree(h->d_dense); cudaFree(h->d_partial);
    cudaFree(h->d_u0); cudaFree(h->d_out); cudaFree(h->d_data); cudaFree(h->d_gu0); cudaFree(h->d_grad);
    cudaFree(h->d_loss); cudaFree(h->d_status);
    b200ude_peer_detach(h);
    cudaFree(h->d_peer_buf);
    cudaFree(h->d_u0_keep); cudaFree(h->d_aux_out);
    cudaFree(h->d_adam_m); cudaFree(h->d_adam_v); cudaFree(h->d_adam_t); cudaFree(h->d_train_out);
    cudaFree(h->d_tgrid); cudaFree(h->d_nacc); cudaFree(h->d_cot); cudaFree(h->d_block_loss);
    cudaFree(h->q_theta); cudaFree(h->q_ustep); cudaFree(h->q_dense); cudaFree(h->q_partial); cudaFree(h->q_tgrid); cudaFree(h->q_cot);
    cudaFree(h->q_u0_keep); cudaFree(h->q_aux_out);
    if (h->h_loss) cudaFreeHost(h->h_loss);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->data_ready) cudaEventDestroy(h->data_ready);
    if (h->data_ready2) cudaEventDestroy(h->data_ready2);
    delete h;
}

size_t b200ude_num_params(const b200ude_handle *h) { return h ? (size_t)h->P : 0; }
size_t b200ude_num_save(const b200ude_handle *h) { return h ? (size_t)h->n_save : 0; }
size_t b200ude_device_bytes(const b200ude_handle *h) { return h ? h->dev_bytes : 0; }

int32_t b200ude_set_params(b200ude_handle *h, const void *theta, size_t P, int32_t mem, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!theta || P != (size_t)h->P) return fail(h, B200UDE_EINVAL, "set_params: P=%zu, expected %d", P, h->P);
    cudaStream_t st = (cudaStream_t)stream;
    if (h->kid == K_F64)
        CUDA_TRY(h, cudaMemcpyAsync(h->q_theta, theta, sizeof(double) * P, mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    else
    CUDA_TRY(h, cudaMemcpyAsync(h->d_theta, theta, sizeof(float) * P,
                                mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    h->have_theta = true;
    return B200UDE_OK;
}

int32_t b200ude_forward(b200ude_handle *h, const void *u0, size_t N, void *out, int32_t *status, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return do_forward64(h, (const double *)u0, N, (double *)out, status, (cudaStream_t)stream);
    return do_forward(h, (const float *)u0, N, (float *)out, status, (cudaStream_t)stream);
}

int32_t b200ude_adjoint(b200ude_handle *h, const void *dL_dout, void *grad_theta, void *grad_u0, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return do_adjoint64(h, false, (const double *)dL_dout, nullptr, (double *)grad_theta, (double *)grad_u0, (cudaStream_t)stream);
    return do_adjoint(h, false, (const float *)dL_dout, nullptr, (float *)grad_theta, (float *)grad_u0,
                      (cudaStream_t)stream);
}

int32_t b200ude_adjoint_l2(b200ude_handle *h, const void *data, void *loss, void *grad_theta, void *grad_u0, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return do_adjoint64(h, true, (const double *)data, (double *)loss, (double *)grad_theta, (double *)grad_u0, (cudaStream_t)stream);
    return do_adjoint(h, true, (const float *)data, (float *)loss, (float *)grad_theta, (float *)grad_u0,
                      (cudaStream_t)stream);
}

// ---- host-buffer entry points -------------------------------------------------------------------
static int32_t ensure_host_path(b200ude_handle *h)
{
    if (h->d_u0) return B200UDE_OK;
    const size_t N = h->cap, D = (size_t)h->D;
    bool ok = true;
    ok = ok && dalloc(h, &h->d_u0, D * N) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_out, (size_t)h->n_save * D * N) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_data, (size_t)h->n_save * D * N) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_gu0, D * N) == cudaSuccess;
    ok = ok && dalloc(h, &h->d_status, N) == cudaSuccess;
    if (!ok) return fail(h, B200UDE_ENOMEM, "host path: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    return B200UDE_OK;
}

int32_t b200ude_solve_host(b200ude_handle *h, const void *theta, const void *u0, size_t N, void *out, int32_t *status)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return f64_unsupported(h, "solve_host");
    if (!theta || !u0 || !out) return fail(h, B200UDE_EINVAL, "solve_host: null pointer");
    if (N == 0 || N > h->cap) return fail(h, B200UDE_EINVAL, "solve_host: N=%zu outside (0, %zu]", N, h->cap);
    int32_t rc = ensure_host_path(h);
    if (rc) return rc;
    cudaStream_t st = h->own_stream;
    const size_t D = (size_t)h->D;
    rc = b200ude_set_params(h, theta, (size_t)h->P, B200UDE_HOST, st);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h->d_u0, u0, sizeof(float) * D * N, cudaMemcpyHostToDevice, st));
    rc = do_forward(h, h->d_u0, N, h->d_out, status ? h->d_status : nullptr, st);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(out, h->d_out, sizeof(float) * (size_t)h->n_save * D * N, cudaMemcpyDeviceToHost, st));
    if (status) CUDA_TRY(h, cudaMemcpyAsync(status, h->d_status, sizeof(int32_t) * N, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    return B200UDE_OK;
}

int32_t b200ude_loss_gradient_host(b200ude_handle *h, const void *theta, const void *u0, const void *data, size_t N,
                                   double *loss, void *grad_theta, void *grad_u0)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return f64_unsupported(h, "loss_gradient_host");
    if (!theta || !u0 || !data || !grad_theta) return fail(h, B200UDE_EINVAL, "loss_gradient_host: null pointer");
    if (N == 0 || N > h->cap) return fail(h, B200UDE_EINVAL, "loss_gradient_host: N=%zu outside (0, %zu]", N, h->cap);
    int32_t rc = ensure_host_path(h);
    if (rc) return rc;
    cudaStream_t st = h->own_stream;
    const size_t D = (size_t)h->D;
    rc = b200ude_set_params(h, theta, (size_t)h->P, B200UDE_HOST, st);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(h->d_u0, u0, sizeof(float) * D * N, cudaMemcpyHostToDevice, st));
    // the data (n_save x larger than u0) is only needed by the adjoint: upload it on a second stream while
    // the forward kernel runs (pinned host memory makes the two overlap)
    // ... in two halves of the trajectories (strided copies: the layout is trajectory-fastest), so that the adjoint of the first half
    // can start under the second half's upload when the link is slower than the forward kernel
    const size_t half = N >= 8192 ? ((N / 2 + 15) / 16) * 16 : N;
    const size_t rows = (size_t)h->n_save * D;
    CUDA_TRY(h, cudaMemcpy2DAsync(h->d_data, sizeof(float) * N, data, sizeof(float) * N, sizeof(float) * half, rows, cudaMemcpyHostToDevice, h->copy_stream));
    CUDA_TRY(h, cudaEventRecord(h->data_ready, h->copy_stream));
    if (half < N)
        CUDA_TRY(h, cudaMemcpy2DAsync(h->d_data + half, sizeof(float) * N, (const float *)data + half, sizeof(float) * N, sizeof(float) * (N - half), rows,
                                      cudaMemcpyHostToDevice, h->copy_stream));
    CUDA_TRY(h, cudaEventRecord(h->data_ready2, h->copy_stream));
    rc = do_forward(h, h->d_u0, N, h->d_out, nullptr, st);
    if (rc) return rc;
    const cudaEvent_t ev[2] = {h->data_ready, h->data_ready2};
    rc = do_adjoint(h, true, h->d_data, h->d_loss, h->d_grad, grad_u0 ? h->d_gu0 : nullptr, st, false, ev, half);
    if (rc) return rc;
    CUDA_TRY(h, cudaMemcpyAsync(grad_theta, h->d_grad, sizeof(float) * (size_t)h->P, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaMemcpyAsync(h->h_loss, h->d_loss, sizeof(float), cudaMemcpyDeviceToHost, st));
    if (grad_u0) CUDA_TRY(h, cudaMemcpyAsync(grad_u0, h->d_gu0, sizeof(float) * D * N, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(h, cudaStreamSynchronize(st));
    if (loss) *loss = (double)*h->h_loss;
    return B200UDE_OK;
}

// ---- on-device optimiser ---------------------------------------------------------------------------
int32_t b200ude_get_params(b200ude_handle *h, void *theta, size_t P, int32_t mem, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!theta || P != (size_t)h->P) return fail(h, B200UDE_EINVAL, "get_params: P=%zu, expected %d", P, h->P);
    if (h->kid == K_F64)
        CUDA_TRY(h, cudaMemcpyAsync(theta, h->q_theta, sizeof(double) * P, mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost,
                                    (cudaStream_t)stream));
    else
    CUDA_TRY(h, cudaMemcpyAsync(theta, h->d_theta, sizeof(float) * P,
                                mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    if (mem != B200UDE_DEVICE) CUDA_TRY(h, cudaStreamSynchronize((cudaStream_t)stream));
    return B200UDE_OK;
}

int32_t b200ude_adam_reset(b200ude_handle *h, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    int32_t rc = ensure_adam(h);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaMemsetAsync(h->d_adam_m, 0, sizeof(float) * h->P, st));
    CUDA_TRY(h, cudaMemsetAsync(h->d_adam_v, 0, sizeof(float) * h->P, st));
    CUDA_TRY(h, cudaMemsetAsync(h->d_adam_t, 0, sizeof(int), st));
    h->adam_t = 0;
    return B200UDE_OK;
}

int32_t b200ude_adam_step(b200ude_handle *h, const b200ude_adam *opt, const void *grad_theta, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!grad_theta) return fail(h, B200UDE_EINVAL, "adam_step: null gradient");
    int32_t rc = check_adam(h, opt);
    if (rc) return rc;
    CUDA_TRY(h, launch_adam(h, opt, (const float *)grad_theta, nullptr, nullptr, h->adam_t, (cudaStream_t)stream));
    h->adam_t += 1;
    return B200UDE_OK;
}

int32_t b200ude_train_adam(b200ude_handle *h, const b200ude_adam *opt, const void *u0, const void *data, size_t N,
                           int32_t iters, void *loss_history, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!u0 || !data || iters < 1) return fail(h, B200UDE_EINVAL, "train_adam: null pointer or iters < 1");
    if (N == 0 || N > h->cap) return fail(h, B200UDE_EINVAL, "train_adam: N=%zu outside (0, %zu]", N, h->cap);
    int32_t rc = check_adam(h, opt);
    if (rc) return rc;
    if (!h->d_train_out && dalloc(h, &h->d_train_out, (size_t)h->n_save * (size_t)h->D * h->cap) != cudaSuccess)
        return fail(h, B200UDE_ENOMEM, "train_adam: device allocation failed: %s", cudaGetErrorString(cudaGetLastError()));
    cudaStream_t st = stream ? (cudaStream_t)stream : h->own_stream;   // the legacy default stream cannot be captured
    if (!stream) {
        // own_stream is non-blocking: order it after everything the caller enqueued on the legacy default stream (set_params,
        // adam_reset, the producers of u0 / data); the call synchronises own_stream before it returns
        CUDA_TRY(h, cudaEventRecord(h->data_ready, (cudaStream_t)0));
        CUDA_TRY(h, cudaStreamWaitEvent(h->own_stream, h->data_ready, 0));
    }
    const int t_base = h->adam_t;
    auto one_iteration = [&]() -> int32_t {
        int32_t r = do_forward(h, (const float *)u0, N, h->d_train_out, nullptr, st);
        if (r) return r;
        // with peers attached (b200ude_peer_attach) the gradient and the loss are the sums over all ranks: every rank runs the
        // same iterations in lock step and applies the identical update to its replica of theta
        r = do_adjoint(h, true, (const float *)data, h->d_loss, h->d_grad, nullptr, st, h->peer_attached);
        if (r) return r;
        CUDA_TRY(h, launch_adam(h, opt, h->d_grad, h->d_loss, (float *)loss_history, t_base, st));
        return B200UDE_OK;
    };
    // iteration 1 eagerly (one-time function attributes, constant tables), the rest as replays of one captured graph
    rc = one_iteration();
    if (rc) return rc;
    if (iters > 1) {
        cudaGraph_t graph = nullptr;
        cudaGraphExec_t exec = nullptr;
        bool graphed = false;
        if (env_int("B200UDE_TRAIN_GRAPH", 1) && cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal) == cudaSuccess) {
            const int32_t r = one_iteration();
            const cudaError_t ce = cudaStreamEndCapture(st, &graph);
            if (r == B200UDE_OK && ce == cudaSuccess && graph && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) graphed = true;
            else cudaGetLastError();
        }
        for (int it = 1; it < iters; ++it) {
            if (graphed) CUDA_TRY(h, cudaGraphLaunch(exec, st));
            else if ((rc = one_iteration()) != 0) break;   // same kernels, launched one by one
        }
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        if (rc) return rc;
    }
    h->adam_t = t_base + iters;
    if (!stream) CUDA_TRY(h, cudaStreamSynchronize(st));
    return B200UDE_OK;
}

// ---- multi-GPU: fused final reduction + all-reduce over NVLink peer memory ------------------------------------
static size_t peer_buf_bytes(const b200ude_handle *h)
{
    const size_t P1pad = (size_t)((h->P + 1 + 31) / 32) * 32;
    return (size_t)PEER_HEADER_BYTES + sizeof(float) * 2 * 16 * P1pad;
}

int32_t b200ude_peer_export(b200ude_handle *h, void *handle_out)
{
    if (!h) return B200UDE_EINVAL;
    if (h->kid == K_F64) return fail(h, B200UDE_EUNSUPPORTED, "peer_export: not available for B200UDE_F64 handles (all-reduce the result of b200ude_adjoint_l2)");
    if (!handle_out) return fail(h, B200UDE_EINVAL, "peer_export: null pointer");
    static_assert(sizeof(cudaIpcMemHandle_t) == B200UDE_PEER_HANDLE_BYTES, "CUDA IPC handle size");
    if (!h->d_peer_buf) {
        CUDA_TRY(h, cudaMalloc(&h->d_peer_buf, peer_buf_bytes(h)));
        h->dev_bytes += peer_buf_bytes(h);
        CUDA_TRY(h, cudaMemset(h->d_peer_buf, 0, peer_buf_bytes(h)));
        CUDA_TRY(h, cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t ipc;
    CUDA_TRY(h, cudaIpcGetMemHandle(&ipc, h->d_peer_buf));
    memcpy(handle_out, &ipc, sizeof(ipc));
    return B200UDE_OK;
}

int32_t b200ude_peer_attach(b200ude_handle *h, int32_t rank, int32_t world, const void *handles)
{
    if (!h) return B200UDE_EINVAL;
    if (!handles || world < 1 || world > 16 || rank < 0 || rank >= world) return fail(h, B200UDE_EINVAL, "peer_attach: need 1 <= world <= 16, 0 <= rank < world");
    if (!h->d_peer_buf) return fail(h, B200UDE_ESTATE, "peer_attach: call b200ude_peer_export first");
    if (h->peer_attached) return fail(h, B200UDE_ESTATE, "peer_attach: already attached");
    for (int r = 0; r < 16; ++r) h->peer.base[r] = nullptr;
    for (int r = 0; r < world; ++r) {
        if (r == rank) { h->peer.base[r] = h->d_peer_buf; continue; }
        cudaIpcMemHandle_t ipc;
        memcpy(&ipc, (const char *)handles + (size_t)r * sizeof(ipc), sizeof(ipc));
        cudaError_t e = cudaIpcOpenMemHandle(&h->peer.base[r], ipc, cudaIpcMemLazyEnablePeerAccess);
        if (e != cudaSuccess) {
            for (int q = 0; q < r; ++q) if (q != rank && h->peer.base[q]) cudaIpcCloseMemHandle(h->peer.base[q]);
            return fail(h, (int32_t)e, "peer_attach: cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
        }
    }
    h->peer.rank = rank; h->peer.world = world; h->peer.P1pad = ((h->P + 1 + 31) / 32) * 32;
    h->peer_attached = true;
    return B200UDE_OK;
}

int32_t b200ude_peer_detach(b200ude_handle *h)
{
    if (!h) return B200UDE_EINVAL;
    if (h->peer_attached)
        for (int r = 0; r < h->peer.world; ++r)
            if (r != h->peer.rank && h->peer.base[r]) cudaIpcCloseMemHandle(h->peer.base[r]);
    h->peer_attached = false;
    return B200UDE_OK;
}

int32_t b200ude_adjoint_l2_allreduce(b200ude_handle *h, const void *data, void *loss, void *grad_theta, void *grad_u0, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    return do_adjoint(h, true, (const float *)data, (float *)loss, (float *)grad_theta, (float *)grad_u0, (cudaStream_t)stream, true);
}

int32_t b200ude_selftest_tanh(int32_t device, const void *x, void *y, size_t n, void *stream)
{
    if (!x || !y || n == 0) return fail(nullptr, B200UDE_EINVAL, "selftest_tanh: null pointer or n == 0");
    CUDA_TRY(nullptr, cudaSetDevice(device));
    CUDA_TRY(nullptr, launch_tanh_selftest((const float *)x, (float *)y, n, (cudaStream_t)stream));
    return B200UDE_OK;
}

// ---- batched independent trainings -------------------------------------------------------------------------------------------
int32_t b200ude_batch_create(const b200ude_desc *d, b200ude_batch_handle **out)
{
    if (!d || !out) return fail(nullptr, B200UDE_EINVAL, "batch_create: null argument");
    *out = nullptr;
    if (d->struct_size != sizeof(b200ude_desc))
        return fail(nullptr, B200UDE_EINVAL, "batch_create: struct_size %u != %zu (ABI mismatch)", d->struct_size, sizeof(b200ude_desc));
    if (d->dtype != B200UDE_F32 && d->dtype != B200UDE_F64) return fail(nullptr, B200UDE_EINVAL, "batch_create: unknown dtype %d", d->dtype);
    if (d->n_layers < 1 || d->n_layers > B200UDE_MAX_LAYERS) return fail(nullptr, B200UDE_EINVAL, "batch_create: n_layers=%d out of range", d->n_layers);
    if (d->solver != B200UDE_TSIT5 && d->solver != B200UDE_VERN7 && d->solver != B200UDE_RKC2)
        return fail(nullptr, B200UDE_EINVAL, "batch_create: unknown solver %d", d->solver);
    if (d->sensealg != B200UDE_INTERPOLATING_ADJOINT && d->sensealg != B200UDE_DISCRETE_ADJOINT)
        return fail(nullptr, B200UDE_EUNSUPPORTED, "batch_create: unknown sensealg %d", d->sensealg);
    if (!(d->dt > 0) || d->n_steps < 1 || d->save_every < 1 || d->n_steps % d->save_every != 0)
        return fail(nullptr, B200UDE_EINVAL, "batch_create: need dt>0, n_steps>=1, save_every>=1 dividing n_steps");
    if (d->max_trajectories == 0 || d->max_trajectories > (1ull << 26))
        return fail(nullptr, B200UDE_EINVAL, "batch_create: max_trajectories (the member capacity) out of range");
    if (d->n_loss_weights != 0 && d->n_loss_weights != d->state_dim)
        return fail(nullptr, B200UDE_EINVAL, "batch_create: n_loss_weights must be 0 or state_dim");
    bool acts_ok = true;
    for (int l = 0; l < d->n_layers; ++l) acts_ok = acts_ok && d->acts[l] >= 0 && d->acts[l] <= 2;
    if (!acts_ok) return fail(nullptr, B200UDE_EINVAL, "batch_create: unknown activation");
    const bool lv5 = d->model == B200UDE_MODEL_LV && d->state_dim == 2 && d->n_layers == 4 && d->widths[0] == 2 && d->widths[1] == 5 &&
                     d->widths[2] == 5 && d->widths[3] == 5 && d->widths[4] == 2 && d->acts[3] == B200UDE_ACT_IDENTITY &&
                     d->n_prefix >= 0 && d->n_prefix <= 2 && d->n_suffix == 0;
    if (!lv5 || d->dtype != B200UDE_F32 || d->solver != B200UDE_TSIT5 || d->adaptive)
        return fail(nullptr, B200UDE_EUNSUPPORTED,
                          "batch_create: batched trainings have kernels for the LV 2-5-5-5-2 chain (identity output layer, 0..2 trainable "
                          "rates), fp32, fixed-step Tsit5");
    if (d->n_consts < 2) return fail(nullptr, B200UDE_EINVAL, "batch_create: the LV model needs n_consts >= 2");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail(nullptr, B200UDE_ENODEVICE, "batch_create: no CUDA device (%s)", cudaGetErrorString(e));
    if (d->device < 0 || d->device >= ndev) return fail(nullptr, B200UDE_EINVAL, "batch_create: device %d of %d", d->device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, d->device);
    if (e != cudaSuccess) return fail(nullptr, (int32_t)e, "batch_create: cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return fail(nullptr, B200UDE_ENODEVICE, "batch_create: device %d is sm_%d%d; this library carries sm_100a code only", d->device, prop.major, prop.minor);
    e = cudaSetDevice(d->device);
    if (e != cudaSuccess) return fail(nullptr, (int32_t)e, "batch_create: cudaSetDevice: %s", cudaGetErrorString(e));

    b200ude_batch_handle *h = new (std::nothrow) b200ude_batch_handle();
    if (!h) return fail(nullptr, B200UDE_ENOMEM, "batch_create: out of host memory");
    h->desc = *d;
    h->P = 87 + d->n_prefix;
    h->n_save = d->n_steps / d->save_every + 1;
    h->cap = (size_t)d->max_trajectories;
    const size_t M = h->cap, P = (size_t)h->P, D = 2;
    bool ok = cudaMalloc((void **)&h->d_theta, sizeof(float) * M * P) == cudaSuccess &&
              cudaMalloc((void **)&h->d_m, sizeof(float) * M * P) == cudaSuccess &&
              cudaMalloc((void **)&h->d_v, sizeof(float) * M * P) == cudaSuccess &&
              cudaMalloc((void **)&h->d_ustep, sizeof(float) * ((size_t)d->n_steps + 1) * D * M) == cudaSuccess &&
              cudaMalloc((void **)&h->d_dense, sizeof(float) * ((size_t)d->n_steps * 6 + 1) * D * M) == cudaSuccess &&
              cudaMalloc((void **)&h->d_out, sizeof(float) * (size_t)h->n_save * D * M) == cudaSuccess &&
              cudaMalloc((void **)&h->d_t, sizeof(int32_t) * M) == cudaSuccess &&
              cudaMalloc((void **)&h->d_best, sizeof(float) * M * P) == cudaSuccess &&
              cudaMalloc((void **)&h->d_best_loss, sizeof(float) * M) == cudaSuccess;
    if (!ok) {
        g_create_error = std::string("batch_create: device allocation failed: ") + cudaGetErrorString(cudaGetLastError());
        b200ude_batch_destroy(h);
        return B200UDE_ENOMEM;
    }
    h->tab.serial = ++g_serial;
    h->tab.d_theta = nullptr;
    h->tab.P = h->P;
    for (int i = 0; i < 16; ++i) {
        h->tab.consts[i] = i < d->n_consts ? (float)d->consts[i] : 0.0f;
        h->tab.lossw[i] = d->n_loss_weights > 0 ? (i < d->n_loss_weights ? (float)d->loss_weights[i] : 0.0f) : 1.0f;
    }
    for (int i = 0; i < 8; ++i) h->tab.acts[i] = i < d->n_layers ? d->acts[i] : 0;
    *out = h;
    return B200UDE_OK;
}

void b200ude_batch_destroy(b200ude_batch_handle *h)
{
    if (!h) return;
    cudaFree(h->d_theta); cudaFree(h->d_m); cudaFree(h->d_v);
    cudaFree(h->d_ustep); cudaFree(h->d_dense); cudaFree(h->d_out);
    cudaFree(h->d_t); cudaFree(h->d_best); cudaFree(h->d_best_loss);
    delete h;
}

const char *b200ude_batch_last_error(const b200ude_batch_handle *h) { return h ? h->err.c_str() : g_create_error.c_str(); }

size_t b200ude_batch_num_params(const b200ude_batch_handle *h) { return h ? (size_t)h->P : 0; }

int32_t b200ude_batch_set_params(b200ude_batch_handle *h, const void *theta, size_t M, int32_t mem, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!theta || M == 0 || M > h->cap) return fail(h, B200UDE_EINVAL, "batch_set_params: null theta or M=%zu outside (0, %zu]", M, h->cap);
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = sizeof(float) * M * (size_t)h->P;
    CUDA_TRY(h, cudaMemcpyAsync(h->d_theta, theta, bytes, mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
    CUDA_TRY(h, cudaMemsetAsync(h->d_m, 0, sizeof(float) * h->cap * (size_t)h->P, st));
    CUDA_TRY(h, cudaMemsetAsync(h->d_v, 0, sizeof(float) * h->cap * (size_t)h->P, st));
    CUDA_TRY(h, cudaMemsetAsync(h->d_t, 0, sizeof(int32_t) * h->cap, st));
    CUDA_TRY(h, cudaMemcpyAsync(h->d_best, h->d_theta, bytes, cudaMemcpyDeviceToDevice, st));
    fill_kernel<<<(unsigned)std::min<size_t>((h->cap + 255) / 256, 1024), 256, 0, st>>>(h->d_best_loss, std::numeric_limits<float>::infinity(), h->cap);
    CUDA_TRY(h, cudaGetLastError());
    h->members = M;
    return B200UDE_OK;
}

int32_t b200ude_batch_get_params(b200ude_batch_handle *h, void *theta, size_t M, int32_t mem, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!theta || M == 0 || M > h->members) return fail(h, B200UDE_EINVAL, "batch_get_params: null theta or M=%zu outside (0, %zu]", M, h->members);
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(h, cudaMemcpyAsync(theta, h->d_theta, sizeof(float) * M * (size_t)h->P,
                                 mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
    if (mem != B200UDE_DEVICE) CUDA_TRY(h, cudaStreamSynchronize(st));
    return B200UDE_OK;
}

int32_t b200ude_batch_forward(b200ude_batch_handle *h, const void *u0, size_t M, void *out, int32_t *status, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    BatchParams p;
    int32_t rc = batch_prepare(h, M, u0, BATCH_FORWARD, p);
    if (rc) return rc;
    if (!out) return fail(h, B200UDE_EINVAL, "batch_forward: null out");
    p.out = (float *)out;
    p.status = status;
    return batch_launch(h, p, (cudaStream_t)stream);
}

int32_t b200ude_batch_loss_gradient(b200ude_batch_handle *h, const void *u0, const void *data, size_t M, void *loss, void *grad,
                                    int32_t *status, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    BatchParams p;
    int32_t rc = batch_prepare(h, M, u0, BATCH_LOSS_GRAD, p);
    if (rc) return rc;
    if (!data || !loss || !grad) return fail(h, B200UDE_EINVAL, "batch_loss_gradient: null pointer");
    p.data = (const float *)data;
    p.loss = (float *)loss;
    p.grad = (float *)grad;
    p.status = status;
    return batch_launch(h, p, (cudaStream_t)stream);
}

int32_t b200ude_batch_train_adam(b200ude_batch_handle *h, const b200ude_adam *o, const void *u0, const void *data, size_t M, int32_t iters,
                                 void *loss_history, int32_t *status, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!o || o->struct_size != sizeof(b200ude_adam)) return fail(h, B200UDE_EINVAL, "batch_train_adam: bad options struct");
    if (!(o->eta > 0) || !(o->beta1 >= 0 && o->beta1 < 1) || !(o->beta2 >= 0 && o->beta2 < 1) || !(o->eps > 0))
        return fail(h, B200UDE_EINVAL, "batch_train_adam: need eta > 0, 0 <= beta < 1, eps > 0");
    if (!data || iters < 1) return fail(h, B200UDE_EINVAL, "batch_train_adam: null data or iters < 1");
    BatchParams p;
    int32_t rc = batch_prepare(h, M, u0, BATCH_TRAIN, p);
    if (rc) return rc;
    p.data = (const float *)data;
    p.loss_history = (float *)loss_history;
    p.status = status;
    p.iters = iters;
    p.eta = (float)o->eta; p.beta1 = (float)o->beta1; p.beta2 = (float)o->beta2; p.eps = (float)o->eps;
    p.loss_scale = (float)(o->loss_scale == 0.0 ? 1.0 : o->loss_scale); p.l2_reg = (float)o->l2_reg;
    return batch_launch(h, p, (cudaStream_t)stream);
}

int32_t b200ude_batch_get_best(b200ude_batch_handle *h, void *theta, void *loss, size_t M, int32_t mem, void *stream)
{
    if (!h) return B200UDE_EINVAL;
    if (!theta || !loss || M == 0 || M > h->members)
        return fail(h, B200UDE_EINVAL, "batch_get_best: null pointer or M=%zu outside (0, %zu]", M, h->members);
    CUDA_TRY(h, cudaSetDevice(h->desc.device));
    cudaStream_t st = (cudaStream_t)stream;
    const cudaMemcpyKind kind = mem == B200UDE_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
    CUDA_TRY(h, cudaMemcpyAsync(theta, h->d_best, sizeof(float) * M * (size_t)h->P, kind, st));
    CUDA_TRY(h, cudaMemcpyAsync(loss, h->d_best_loss, sizeof(float) * M, kind, st));
    if (mem != B200UDE_DEVICE) CUDA_TRY(h, cudaStreamSynchronize(st));
    return B200UDE_OK;
}

}  // extern "C"
