/*
 * b200ude.h -- C ABI of the B200-native UDE training path.
 *
 * This is the drop-in boundary for ONE hot path of
 * ChrisRackauckas/universal_differential_equations: the forward solve of a
 * universal differential equation (known physics + embedded dense chain) for an
 * ensemble of trajectories and its interpolating-adjoint gradient.  The
 * reference has no FFI of its own: the seam is Julia dispatch on
 *     concrete_solve(prob::ODEProblem, Tsit5()/Vern7(), u0, p; saveat, abstol,
 *                    reltol, sensealg = InterpolatingAdjoint(autojacvec = ReverseDiffVJP()))
 *         SEIR_exposure/seir_exposure.jl:137-141, FisherKPP/Fisher-KPP-CNN.jl:136,
 *         LotkaVolterra/scenario_1.jl:82-88
 * and its reverse rule (DiffEqSensitivity._concrete_solve_adjoint), driven by
 *     DiffEqFlux.sciml_train(loss, theta, opt; cb, maxiters)
 *         seir_exposure.jl:160-161, Fisher-KPP-CNN.jl:236-238.
 * A Julia shim (INTEGRATION.md) defines those methods on top of the entry
 * points below with `ccall`; the Python mirror in
 * universal_differential_equations_b200/sciml.py binds the same symbols with
 * ctypes and is what the tests and bench.py exercise.
 *
 * Conventions
 *  - every function returns int32_t: 0 = OK, <0 usage error, >0 CUDA runtime error
 *    (message via b200ude_last_error); nothing throws or longjmps across the ABI.
 *  - all arrays are plain pointers + sizes; the caller owns every array it passes;
 *    the handle owns theta's device copy, the stored forward solution and scratch.
 *  - ensemble layouts are trajectory-fastest (structure of arrays):
 *        u0 [d][N]      out / data / dL_dout [n_save][d][N]      grad_u0 [d][N]
 *    i.e. a Julia Array of size (N, d) / (N, d, n_save).
 *  - theta is the reference's own flat layout: [n_prefix trainable physics scalars |
 *    per dense layer: vec(W) column-major (W is out x in), then b | n_suffix scalars]
 *    (Lux ComponentVector scenario_1.jl:113, DiffEqFlux initial_params
 *    seir_exposure.jl:115, Flux.destructure Fisher-KPP-CNN.jl:106).
 *  - `stream` is a cudaStream_t passed as void* (NULL = default stream); calls taking a
 *    stream are asynchronous with respect to the host unless stated otherwise.
 *  - a handle is not thread-safe; use one handle per host thread and device.  The default kernels of the LV 2-32-32-2 chain
 *    (warp-collective family) and the fp64 kernels read theta from the handle's own device copy: any number of such handles
 *    can be in flight on a device.  The other kernel families read the active handle's theta and tables from the constant
 *    bank, so work of DIFFERENT handles of those kinds on one device must be stream-ordered (not concurrent).
 *  - the interpolating adjoint of a Vern7 handle runs over a Tsit5 re-solve from the same u0 with the same step / tolerances
 *    (Vern7's lazy dense output is not available): with the fused L2 entry point the reported loss is that of the re-solve.
 */
#ifndef B200UDE_H
#define B200UDE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200UDE_ABI_VERSION 1

/* dtype */
#define B200UDE_F32 0
#define B200UDE_F64 1 /* double precision: EVERY device array of the calls (theta, u0, out, data, dL_dout, grad_theta, grad_u0, loss) is
                        * double.  Runtime-shape kernels for the LV / SEIR / NODE forms, Tsit5 and Vern7, fixed step and adaptive,
                        * interpolating adjoint -- the precision the reference's scenario 1 / 2 and SEIR scripts run in (Float64,
                        * abstol = reltol = 1e-6).  Entry points: create / set_params / get_params / forward / adjoint / adjoint_l2;
                        * the host-buffer, ADAM and peer entry points return B200UDE_EUNSUPPORTED for such handles. */

/* model kinds: the UDE right-hand sides of the reference */
#define B200UDE_MODEL_LV 0   /* du1 = a1*u1 + NN1(u), du2 = -a2*u2 + NN2(u)   scenario_1.jl:69-73,
                                a2 trainable (n_prefix=1) scenario_2.jl:90-95, a1,a2 trainable (n_prefix=2)
                                hudson_bay.jl:85-91; consts = {p_[1], p_[4]} */
#define B200UDE_MODEL_SEIR 1 /* 7-state exposure UDE, NN([S/N, I, D/N])      seir_exposure.jl:117-130;
                                consts = F,beta0,alpha,kappa,mu,sigma,gamma,d,lambda (:33) */
#define B200UDE_MODEL_FKPP 2 /* pointwise reaction net + D0 * 3-tap periodic stencil, n_suffix = 5
                                Fisher-KPP-CNN.jl:111-126, scenario_3.jl:103-114 */
#define B200UDE_MODEL_NODE 3 /* du = NN(u) */
#define B200UDE_MODEL_SEIR_NODE 4 /* the SEIR script's black-box baseline dudt_node: dS,dE,dI,dR,dD = first five outputs of
                                     NN([S/N,E,I,R,N,D/N,C]), dN = -mu N, dC = sigma E   seir_exposure.jl:52-64; consts as MODEL_SEIR */

/* activations of the dense chain */
#define B200UDE_ACT_IDENTITY 0
#define B200UDE_ACT_TANH 1
#define B200UDE_ACT_RBF 2 /* exp(-x^2), scenario_1.jl:59 */

/* solver (OrdinaryDiffEq algorithm the reference passes to solve/concrete_solve) */
#define B200UDE_TSIT5 0
#define B200UDE_VERN7 1
#define B200UDE_RKC2 2 /* second-order Runge-Kutta-Chebyshev with desc.n_stages stages per step: the closed-form stabilised explicit
                          method of the class of ROCK2 (Climate/NeuralPDE/npde.jl:61,82; ROCK2's own coefficient tables are not in the
                          reference); real stability interval ~ 0.65 n_stages^2; dense output = cubic Hermite; the interpolating
                          adjoint steps lambda backwards with RKC2 itself.  Fisher-KPP UPDE (1-16-16-1 chain, even grids), fixed step */

/* sensealg */
#define B200UDE_INTERPOLATING_ADJOINT 0 /* InterpolatingAdjoint(autojacvec = ReverseDiffVJP())  seir_exposure.jl:71,140 */
#define B200UDE_DISCRETE_ADJOINT 1      /* exact gradient of the discrete fixed-step scheme by reverse accumulation through the
                                           stages: the quantity ForwardDiffSensitivity() computes in forward mode
                                           (scenario_1.jl:86, scenario_2.jl:108, hudson_bay.jl:102); LV chains, Tsit5 fixed step */

/* memory space of a pointer argument */
#define B200UDE_HOST 0
#define B200UDE_DEVICE 1

/* flags */
#define B200UDE_FLAG_APPROX_TANH 1u /* tanh.approx.f32 (2^-11 rel. error) instead of the ex2/rcp form */

/* per-trajectory status words written by b200ude_forward */
#define B200UDE_TRAJ_OK 0
#define B200UDE_TRAJ_NONFINITE 1
#define B200UDE_TRAJ_MAXSTEPS 2 /* adaptive: more than max_steps accepted steps needed */

/* error codes */
#define B200UDE_OK 0
#define B200UDE_EINVAL (-1)       /* bad descriptor / argument */
#define B200UDE_EUNSUPPORTED (-2) /* configuration has no sm_100a kernel in this build */
#define B200UDE_ESTATE (-3)       /* call order violated (e.g. adjoint before forward) */
#define B200UDE_ENOMEM (-4)
#define B200UDE_ENODEVICE (-5)    /* no CUDA device / not an sm_100 part */

#define B200UDE_MAX_LAYERS 6

typedef struct b200ude_handle b200ude_handle;

typedef struct b200ude_desc {
    uint32_t struct_size; /* = sizeof(b200ude_desc); checked */
    int32_t device;       /* CUDA device ordinal */
    int32_t dtype;        /* B200UDE_F32 | B200UDE_F64 */
    int32_t model;        /* B200UDE_MODEL_* */
    int32_t state_dim;    /* d */
    int32_t n_layers;     /* dense layers of the embedded chain */
    int32_t widths[B200UDE_MAX_LAYERS + 1]; /* widths[0] = chain input, widths[n_layers] = chain output */
    int32_t acts[B200UDE_MAX_LAYERS];
    int32_t n_prefix;     /* trainable physics scalars before the chain in theta */
    int32_t n_suffix;     /* trainable scalars after the chain in theta */
    int32_t n_consts;
    double consts[16];    /* fixed physics constants */
    int32_t solver;       /* B200UDE_TSIT5 | B200UDE_VERN7 | B200UDE_RKC2 */
    int32_t sensealg;     /* B200UDE_INTERPOLATING_ADJOINT | B200UDE_DISCRETE_ADJOINT */
    double t0;            /* tspan[1] */
    double dt;            /* fixed step (adaptive = false); saveat = t0 + i*save_every*dt */
    int32_t n_steps;      /* number of steps; tspan[2] = t0 + n_steps*dt */
    int32_t save_every;   /* save the state every this many steps (and at t0) */
    double abstol, reltol; /* adaptive stepping tolerances (used when adaptive = 1) */
    int32_t n_loss_weights; /* 0 => all ones; else = state_dim */
    double loss_weights[16]; /* per-component weight of the fused L2 loss (seir_exposure.jl:146 uses rows 2:4) */
    uint64_t max_trajectories; /* capacity: scratch is sized for this many trajectories */
    uint32_t flags;
    int32_t adaptive;   /* 0: fixed step dt (adaptive = false). 1: Tsit5 with OrdinaryDiffEq's PI controller, abstol / reltol;
                           saveat = t0 + i*save_every*dt, i = 0..n_steps/save_every (dt only defines the save grid) */
    int32_t max_steps;  /* adaptive: capacity of ACCEPTED steps per trajectory (status 2 when exceeded) */
    int32_t n_stages;   /* B200UDE_RKC2: stages per step (2..64); choose dt * spectral_radius <= 0.65 n_stages^2.  0 otherwise */
} b200ude_desc;

int32_t b200ude_version(void);

/* Message of the last error on this handle (h may be NULL: last create() error of the calling thread). */
const char *b200ude_last_error(const b200ude_handle *h);

int32_t b200ude_create(const b200ude_desc *desc, b200ude_handle **out);
void b200ude_destroy(b200ude_handle *h);

/* length P of theta, number of saved time points, bytes of device memory held by the handle */
size_t b200ude_num_params(const b200ude_handle *h);
size_t b200ude_num_save(const b200ude_handle *h);
size_t b200ude_device_bytes(const b200ude_handle *h);

/* theta[P] (float) from host or device memory -> the handle's device copy. */
int32_t b200ude_set_params(b200ude_handle *h, const void *theta, size_t P, int32_t mem, void *stream);

/* FORWARD  (replaces: the UDE RHS closure + OrdinaryDiffEq perform_step! loop behind
 * concrete_solve(prob, Tsit5(), u0, p; saveat, ...), one trajectory per ensemble member).
 * u0 [d][N], out [n_save][d][N], status [N] (may be NULL): DEVICE pointers.
 * Also stores the dense output (stage derivatives) the adjoint interpolates.  With adaptive = 1 `out` must stay valid
 * until the matching adjoint call (the fused L2 adjoint reads the interpolated saved states from it). */
int32_t b200ude_forward(b200ude_handle *h, const void *u0, size_t N, void *out, int32_t *status,
                        void *stream);

/* ADJOINT  (replaces: DiffEqSensitivity InterpolatingAdjoint backward solve + ReverseDiffVJP).
 * Uses the forward solution stored by the last b200ude_forward on this handle.
 * dL_dout [n_save][d][N]: cotangent of the saved states (the Zygote pullback's Delta).
 * grad_theta [P]: SUM over the N trajectories (overwritten). grad_u0 [d][N] or NULL. DEVICE pointers. */
int32_t b200ude_adjoint(b200ude_handle *h, const void *dL_dout, void *grad_theta, void *grad_u0,
                        void *stream);

/* ADJOINT with the L2 trajectory-matching loss fused (scenario_1.jl:91-94, seir_exposure.jl:144-147):
 * L = sum_n sum_i sum_k w_k (out - data)^2, Delta = 2 w (out - data) formed in-kernel.
 * data [n_save][d][N]; loss: float[1] (sum over the ensemble, overwritten). DEVICE pointers. */
int32_t b200ude_adjoint_l2(b200ude_handle *h, const void *data, void *loss, void *grad_theta,
                           void *grad_u0, void *stream);

/* HOST-BUFFER entry points (what a host-language binding calls with ordinary arrays): copy
 * inputs host->device, run the kernels, copy results back, synchronise.  Pinned host memory makes
 * the copies asynchronous; pageable memory works but is slower. */
int32_t b200ude_solve_host(b200ude_handle *h, const void *theta, const void *u0, size_t N, void *out,
                           int32_t *status);
int32_t b200ude_loss_gradient_host(b200ude_handle *h, const void *theta, const void *u0,
                                   const void *data, size_t N, double *loss, void *grad_theta,
                                   void *grad_u0 /* may be NULL */);

/* ON-DEVICE OPTIMISER  (replaces the ADAM phase of DiffEqFlux.sciml_train(loss, theta, ADAM(eta); cb, maxiters)
 * seir_exposure.jl:160, Fisher-KPP-CNN.jl:236, Optimization.solve(optprob, ADAM(0.1); maxiters) scenario_1.jl:114,
 * for the trajectory-matching loss  L = loss_scale * sum w (u - data)^2 + l2_reg * sum theta[n_prefix:]^2
 * (the L2 term skips the n_prefix trainable physics rates, as scenario_2.jl:113 does with theta[2:end])
 * (scenario_1.jl:91-94; scenario_2.jl:113-116 divides by the number of points and adds the L2 term).
 * The update is Flux.ADAM: m = b1 m + (1-b1) g, v = b2 v + (1-b2) g^2,
 * theta -= eta * (m / (1 - b1^t)) / (sqrt(v / (1 - b2^t)) + eps); the moments and t live in the handle. */
typedef struct b200ude_adam {
    uint32_t struct_size; /* = sizeof(b200ude_adam) */
    uint32_t reserved;
    double eta, beta1, beta2, eps; /* Flux defaults: 0.001, 0.9, 0.999, 1e-8 */
    double loss_scale;             /* 0 is read as 1 */
    double l2_reg;
} b200ude_adam;

/* the handle's current theta -> theta[P] (host: synchronises the stream; device: asynchronous) */
int32_t b200ude_get_params(b200ude_handle *h, void *theta, size_t P, int32_t mem, void *stream);
/* zero the ADAM moments and the step counter */
int32_t b200ude_adam_reset(b200ude_handle *h, void *stream);
/* one ADAM update of the handle's theta with a caller-supplied DEVICE gradient [P] (e.g. after an all-reduce over GPUs);
 * loss_scale / l2_reg are applied to it as above */
int32_t b200ude_adam_step(b200ude_handle *h, const b200ude_adam *opt, const void *grad_theta, void *stream);
/* `iters` full iterations without a host round trip: forward, fused-L2 adjoint, fixed-order reduce, ADAM update -- the first
 * launched directly, the rest as replays of one captured CUDA graph.  u0 [d][N], data [n_save][d][N]: DEVICE pointers.
 * loss_history: DEVICE float[iters] or NULL; slot i = loss at the pre-update theta of iteration i (what the reference's
 * callback records).  stream NULL = the handle's own stream, synchronised before returning.  With peers attached
 * (b200ude_peer_attach, below) every iteration uses the loss and gradient summed over ALL ranks: the call is then a collective,
 * every rank runs the same iterations in lock step and applies the identical update to its replica of theta. */
int32_t b200ude_train_adam(b200ude_handle *h, const b200ude_adam *opt, const void *u0, const void *data, size_t N,
                           int32_t iters, void *loss_history, void *stream);

/* MULTI-GPU (one process per GPU; the ensemble shards, theta is replicated -- SURVEY.md section 8e).  The only exchange of
 * the path, the sum over ranks of [grad_theta (P); loss], can run inside the final reduction kernel over NVLink peer memory:
 * every rank exports an exchange buffer (CUDA IPC), the host program gathers the `world` handles in rank order by whatever
 * means it has (MPI, torch.distributed, a file), attaches, and synchronises all ranks once (a host barrier) before the first
 * call.  b200ude_adjoint_l2_allreduce is then b200ude_adjoint_l2 whose loss and grad_theta are the sums over ALL ranks
 * (bitwise identical on every rank); it is a collective: every rank must call it the same number of times.  grad_u0 stays
 * local.  Fixed-step handles only.  A peer that never arrives turns the results into NaN after ~2 s instead of hanging. */
#define B200UDE_PEER_HANDLE_BYTES 64
int32_t b200ude_peer_export(b200ude_handle *h, void *handle_out /* B200UDE_PEER_HANDLE_BYTES */);
int32_t b200ude_peer_attach(b200ude_handle *h, int32_t rank, int32_t world, const void *handles /* world x 64 bytes, rank order */);
int32_t b200ude_peer_detach(b200ude_handle *h);
int32_t b200ude_adjoint_l2_allreduce(b200ude_handle *h, const void *data, void *loss, void *grad_theta, void *grad_u0,
                                     void *stream);

/* BATCHED INDEPENDENT TRAININGS  (replaces the loop of LotkaVolterra/run_loops.jl:55-62, which calls recover_dynamics
 * (loop_recoveries.jl) once per noisy data set, one run after another: each run trains its own theta with ADAM(0.1) on its own
 * data and u0).  A batch handle holds M "members", each with its own theta, gradient and ADAM moments, one trajectory per member;
 * nothing is shared between members (no ensemble sum, no shared optimiser state).  A member's results are bitwise independent of M,
 * of its position in the batch and of the other members, and repeated calls are bitwise identical.
 * Descriptor: b200ude_desc as for b200ude_create, restricted to the LV model with the 2-5-5-5-2 chain (identity output layer, per-layer
 * activations, n_prefix 0..2 trainable rates: scenario 1 / the loop, scenario 2, Hudson Bay), fp32, fixed-step Tsit5, either sensealg;
 * max_trajectories is the member capacity.  Anything else is B200UDE_EUNSUPPORTED; the descriptor is validated before the device is
 * probed.  There is no CPU fallback.
 * Layouts: u0 [d][M], data / out [n_save][d][M], status / loss [M], loss_history [iters][M] (member-fastest);
 * theta / grad [M][P]: each member's flat theta is contiguous in the reference's own order (a Julia P x M matrix, one column per run).
 * All arrays except a HOST theta are DEVICE pointers.  The physics constants, loss weights and activations of a batch handle sit in the
 * constant bank of the batch kernels (not shared with the other families): work of two batch handles with different descriptors on one
 * device must be stream-ordered; a batch handle may run concurrently with any non-batch handle. */
typedef struct b200ude_batch_handle b200ude_batch_handle;
int32_t b200ude_batch_create(const b200ude_desc *desc, b200ude_batch_handle **out);
void b200ude_batch_destroy(b200ude_batch_handle *h);
/* message of the last error on this handle (h may be NULL: last b200ude_batch_create error of the calling thread) */
const char *b200ude_batch_last_error(const b200ude_batch_handle *h);
/* P, the length of one member's theta (87 + n_prefix) */
size_t b200ude_batch_num_params(const b200ude_batch_handle *h);
/* theta [M][P] from host or device memory -> the handle's thetas of members 0..M-1; zeroes every member's ADAM moments and step
 * count and makes theta its best theta so far (with loss +inf).  Later calls may use any M' <= M of these members: each member
 * keeps its own step count, so a member trained by fewer calls than another continues from its own state. */
int32_t b200ude_batch_set_params(b200ude_batch_handle *h, const void *theta, size_t M, int32_t mem, void *stream);
/* the current thetas of members 0..M-1 -> theta [M][P] (host: synchronises the stream; device: asynchronous) */
int32_t b200ude_batch_get_params(b200ude_batch_handle *h, void *theta, size_t M, int32_t mem, void *stream);
/* FORWARD of every member at its own theta from its own u0: out [n_save][d][M], status [M] (may be NULL; B200UDE_TRAJ_NONFINITE when
 * the final state is not finite). */
int32_t b200ude_batch_forward(b200ude_batch_handle *h, const void *u0, size_t M, void *out, int32_t *status, void *stream);
/* per-member fused L2 loss  loss[n] = sum_i sum_k w_k (u_n - data_n)^2  and its gradient grad [M][P] with respect to the member's own
 * theta (the desc's sensealg), status [M] or NULL (non-finite state, loss or gradient).  What a host-side batched optimiser calls. */
int32_t b200ude_batch_loss_gradient(b200ude_batch_handle *h, const void *u0, const void *data, size_t M, void *loss, void *grad,
                                    int32_t *status, void *stream);
/* `iters` ADAM iterations of every member in ONE launch (forward, fused-L2 adjoint, the member's loss, Flux.ADAM with its own moments;
 * options and loss as b200ude_train_adam: L = loss_scale * L_data + l2_reg * sum theta[n_prefix:]^2).  loss_history [iters][M] or
 * NULL: slot (i, n) = member n's loss at its pre-update theta of iteration i.  A member whose state, loss or gradient turns non-finite
 * stops there: status[n] = B200UDE_TRAJ_NONFINITE, its theta and moments keep their last finite values, its remaining loss slots are
 * NaN, and every other member is unaffected.  status [M] may be NULL.  Successive calls continue every member's moments and its own
 * step count (advanced only by the member's own updates: a stopped member's stays where it stopped).  Each member also keeps the
 * best pre-update theta since set_params and its loss, as sciml_train does (b200ude_batch_get_best). */
int32_t b200ude_batch_train_adam(b200ude_batch_handle *h, const b200ude_adam *opt, const void *u0, const void *data, size_t M,
                                 int32_t iters, void *loss_history, int32_t *status, void *stream);
/* every member's best theta since set_params -> theta [M][P] and its loss -> loss [M] (the lowest recorded pre-update loss of
 * b200ude_batch_train_adam; +inf and the set_params theta when there was no finite one) -- what sciml_train returns as its minimizer.
 * Host: synchronises the stream; device: asynchronous. */
int32_t b200ude_batch_get_best(b200ude_batch_handle *h, void *theta, void *loss, size_t M, int32_t mem, void *stream);

/* SELF-TEST of a device building block (no reference counterpart): y[i] = the kernels' tanh (1 - 2 / (1 + 2^(2 log2(e) x)) with one
 * reciprocal per four values, the variant the warp-collective LV kernels use) for n device floats; the parity tests compare it
 * with tanh in fp64.  device = CUDA ordinal. */
int32_t b200ude_selftest_tanh(int32_t device, const void *x, void *y, size_t n, void *stream);

/* TERMINAL-PDE / SDE PATH (SURVEY.md section 8 f4, BASELINE config 5) -- replaces, for highdim_pde/lambaem.jl:18-34,
 *     solve(TerminalPDEProblem(g, f, mu, sigma, x0, tspan), NNPDENS(u0, sigmaT_grad_u, opt = ADAM(eta));
 *           maxiters, trajectories = m, alg = LambaEM(), ...)                                   [EXT NeuralNetDiffEq 1.1.0]
 * i.e. the deep-BSDE method: dX = mu dt + sigma dW, du = -f dt + z . dW with z = sigmaT_grad_u([X; t]) and u(0) = u0(x0), all
 * `trajectories` paths advanced together, loss = mean (g(X_T) - u_T)^2, reverse-mode gradient through the discretised solve,
 * Flux.ADAM on both networks; the solution is u0(x0).  Problem family of the script (Hamilton-Jacobi-Bellman):
 *     mu = 0, sigma = sigma I, f(X, u, z, p, t) = -lambda |z|^2, g(X) = log(g_a + g_b |X|^2)
 * Networks as in the script: u0 = Dense(d, hidden, relu), Dense(hidden, hidden, relu), Dense(hidden, 1);
 * sigmaT_grad_u = Dense(d + 1, hidden, relu) x3 -> Dense(hidden, d); theta = [u0 net; sigmaT_grad_u net], each layer vec(W)
 * (out x in, column-major) then b -- Flux.params order.  relu'(0) = 1 (Flux 0.9 / Tracker differentiating max(zero(x), x)).
 * Time stepping: Euler-Maruyama with the fixed step T / n_steps (LambaEM is EM with step-size control).  Brownian increments:
 * sqrt(dt) * Box-Muller(Philox4x32-10) with counter (path, component / 4, step, 0) and key = seed; iteration i of
 * b200ude_bsde_train_adam uses seed0 + i.  dtype selects float or double for every buffer of the calls.
 * Streams: these calls take no stream; they run on the handle's own stream and return when the work is complete.  Device arrays
 * handed in (theta, a gradient for b200ude_bsde_adam_step) must be ready -- finish or synchronise the producing stream first. */
typedef struct b200ude_bsde_handle b200ude_bsde_handle;
typedef struct b200ude_bsde_desc {
    uint32_t struct_size; /* = sizeof(b200ude_bsde_desc) */
    int32_t device;
    int32_t dtype;        /* B200UDE_F32 | B200UDE_F64 */
    int32_t dim;          /* d */
    int32_t hidden;       /* hls (the script: 10 + d) */
    int32_t n_steps;
    double T;             /* tspan = (0, T) */
    double lambda, sigma; /* f = -lambda |z|^2; sigma = sqrt(2) in the script */
    double g_a, g_b;      /* g(X) = log(g_a + g_b |X|^2); 0.5, 0.5 in the script */
    const double *x0;     /* HOST double[dim]; copied by create */
    uint64_t max_paths;   /* capacity (trajectories) */
} b200ude_bsde_desc;
int32_t b200ude_bsde_create(const b200ude_bsde_desc *desc, b200ude_bsde_handle **out);
void b200ude_bsde_destroy(b200ude_bsde_handle *h);
const char *b200ude_bsde_last_error(const b200ude_bsde_handle *h);
size_t b200ude_bsde_num_params(const b200ude_bsde_handle *h);
/* mem = B200UDE_HOST | B200UDE_DEVICE; set_params also zeroes the ADAM state */
int32_t b200ude_bsde_set_params(b200ude_bsde_handle *h, const void *theta, size_t P, int32_t mem);
int32_t b200ude_bsde_get_params(b200ude_bsde_handle *h, void *theta, size_t P, int32_t mem);
/* one evaluation at the handle's theta: loss[1], grad[P], u0[1] = u0(x0) (host or device pointers of the handle's dtype; NULL =
 * not wanted).  path_offset shifts the Philox path counter and total_paths (0 = n_paths) is the denominator of the mean, so
 * that ranks of a multi-GPU job evaluate disjoint paths and their losses / gradients simply add. */
int32_t b200ude_bsde_loss_gradient(b200ude_bsde_handle *h, size_t n_paths, uint64_t seed, uint64_t path_offset, size_t total_paths,
                                   void *loss, void *grad, void *u0);
/* `iters` NNPDENS iterations on the device (forward paths, loss, backward sweep, ADAM), the first launched directly, the rest
 * as replays of one CUDA graph.  loss_history / u0_history: DEVICE arrays [iters] of the handle's dtype or NULL; slot i = the
 * loss / u0(x0) at the pre-update theta of iteration i (what the script's `verbose` callback prints). */
int32_t b200ude_bsde_train_adam(b200ude_bsde_handle *h, const b200ude_adam *opt, size_t n_paths, int32_t iters, uint64_t seed0,
                                void *loss_history, void *u0_history);
/* device time of the last b200ude_bsde_train_adam call in ms (CUDA events on the handle's stream around all its iterations) */
double b200ude_bsde_last_train_ms(const b200ude_bsde_handle *h);
/* fp64 handles with widths <= 112 run fused sweeps (csrc/bsde.cu): ms[0..2] = device time of the forward sweep, the cotangent sweep
 * and the batched weight-gradient GEMMs of the last b200ude_bsde_loss_gradient call (CUDA events on the handle's stream) */
int32_t b200ude_bsde_last_sweep_ms(b200ude_bsde_handle *h, double *ms);
/* one ADAM update with a caller-supplied DEVICE gradient [P] of the handle's dtype (multi-GPU: b200ude_bsde_loss_gradient on
 * every rank's path shard, all-reduce of the gradient, then this call on every rank) */
int32_t b200ude_bsde_adam_step(b200ude_bsde_handle *h, const b200ude_adam *opt, const void *grad);

#ifdef __cplusplus
}
#endif
#endif /* B200UDE_H */
