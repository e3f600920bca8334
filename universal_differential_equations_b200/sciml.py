"""Host-side mirror of the reference's call surface for the UDE training path.

The reference scripts are Julia; their seam for this path is multiple dispatch on

    concrete_solve(prob, Tsit5(), u0, p; saveat, sensealg=InterpolatingAdjoint(autojacvec=ReverseDiffVJP()))
        SEIR_exposure/seir_exposure.jl:137-141, FisherKPP/Fisher-KPP-CNN.jl:136
    solve(remake(prob_nn; u0, tspan, p), Vern7(); saveat, abstol, reltol, sensealg)
        LotkaVolterra/scenario_1.jl:82-88
    DiffEqFlux.sciml_train(loss, p, ADAM(0.01); cb, maxiters)   seir_exposure.jl:160-161
    FastChain(FastDense(3, 64, tanh), ...), initial_params(ann)  seir_exposure.jl:114-115
    Lux.Chain(Lux.Dense(2, 5, rbf), ...)                         scenario_1.jl:62-64

Julia is not available in the build/test environment, so this module restates that
surface in Python with the same names, argument meaning and error behaviour, on top
of the C-ABI library (the Julia `ccall` shim a maintainer would add is in
INTEGRATION.md).  torch is used only for device memory, streams and autograd
plumbing (the pullback of `concrete_solve` calls the adjoint kernel, the way Zygote
calls DiffEqSensitivity's rule); every number is produced by the sm_100a kernels.

Arbitrary closures cannot cross a C ABI: the right-hand side must be one of the UDE
forms the library recognises (`LotkaVolterraUDE` ...), built from a dense chain.
"""
from __future__ import annotations

import ctypes as C
import math
import warnings
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence

import numpy as np
import torch

from . import _lib

# --------------------------------------------------------------------------- activations
tanh = "tanh"
identity = "identity"
rbf = "rbf"  # rbf(x) = exp.(-(x.^2)), scenario_1.jl:59
_ACT_CODE = {"identity": _lib.ACT_IDENTITY, "tanh": _lib.ACT_TANH, "rbf": _lib.ACT_RBF}


# --------------------------------------------------------------------------- dense chains
@dataclass(frozen=True)
class FastDense:
    """DiffEqFlux.FastDense(in, out, activation) / Lux.Dense / Flux.Dense."""
    n_in: int
    n_out: int
    act: str = identity


Dense = FastDense


@dataclass(frozen=True)
class FastChain:
    """DiffEqFlux.FastChain / Lux.Chain / Flux.Chain of dense layers.

    Flat parameter layout (identical to `initial_params`, Lux ComponentVector and
    Flux.destructure): per layer vec(W) column-major with W of shape out x in, then b.
    """
    layers: tuple

    def __init__(self, *layers):
        object.__setattr__(self, "layers", tuple(layers))
        for a, b in zip(self.layers[:-1], self.layers[1:]):
            if a.n_out != b.n_in:
                raise ValueError(f"DimensionMismatch: layer output {a.n_out} feeds layer input {b.n_in}")

    @property
    def widths(self):
        return (self.layers[0].n_in,) + tuple(l.n_out for l in self.layers)

    @property
    def acts(self):
        return tuple(l.act for l in self.layers)

    def num_params(self):
        return sum(l.n_in * l.n_out + l.n_out for l in self.layers)


Chain = FastChain


def initial_params(chain: FastChain, rng: Optional[np.random.Generator] = None) -> np.ndarray:
    """Glorot-uniform Float32 weights, zero biases (DiffEqFlux.initial_params / Lux.setup)."""
    rng = rng or np.random.default_rng()
    parts = []
    for l in chain.layers:
        lim = math.sqrt(6.0 / (l.n_in + l.n_out))
        W = rng.uniform(-lim, lim, size=(l.n_out, l.n_in)).astype(np.float32)
        parts += [W.ravel(order="F"), np.zeros(l.n_out, np.float32)]
    return np.concatenate(parts)


# --------------------------------------------------------------------------- UDE right-hand sides
@dataclass(frozen=True)
class LotkaVolterraUDE:
    """du1 = p1*u1 + U(u)[1];  du2 = -p4*u2 + U(u)[2]        (scenario_1.jl:69-73)

    trainable_rates = 0: p1, p4 known (p_true[1], p_true[4]);
    trainable_rates = 1: theta = [delta; U], du2 = -delta*u2 + ...  (scenario_2.jl:90-95);
    trainable_rates = 2: theta = [p1, p2; U]                         (hudson_bay.jl:85-91).
    """
    chain: FastChain
    p_true: Sequence[float] = (1.3, 0.9, 0.8, 1.8)  # scenario_1.jl:39
    trainable_rates: int = 0

    model = _lib.MODEL_LV
    state_dim = 2

    def consts(self):
        return (float(self.p_true[0]), float(self.p_true[3]))

    def num_params(self):
        return self.trainable_rates + self.chain.num_params()


SEIR_P = (10.0, 0.5944, 0.4239, 1117.3, 0.02, 1 / 3, 1 / 5, 0.2, 1 / 11.2)  # F, beta0, alpha, kappa, mu, sigma, gamma, d, lambda (seir_exposure.jl:33)


@dataclass(frozen=True)
class SEIRExposureUDE:
    """7-state SEIR-type model whose exposure term is the chain: z = ann([S/N, I, D/N], p)  (seir_exposure.jl:117-130).

    dS = -b0*S*F/N - z - mu*S;  dE = b0*S*F/N + z - (sigma+mu)*E;  dI, dR, dN, dD, dC as in `corona!` (:16-29).
    """
    chain: FastChain
    p_true: Sequence[float] = SEIR_P

    model = _lib.MODEL_SEIR
    state_dim = 7

    def consts(self):
        return tuple(float(x) for x in self.p_true)

    def num_params(self):
        return self.chain.num_params()


@dataclass(frozen=True)
class FisherKPPUDE:
    """Fisher-KPP universal PDE on a periodic grid of `nx` points (FisherKPP/Fisher-KPP-CNN.jl:111-126,
    LotkaVolterra/scenario_3.jl:103-114):  du_i = rx_nn(u_i) + D0 * (w1 u_{i-1} + w2 u_i + w3 u_{i+1}).

    theta = [chain(1 -> ... -> 1); w1, w2, w3, conv-bias (unused); D0]  (Fisher-KPP-CNN.jl:106-109).
    """
    chain: FastChain
    nx: int

    model = _lib.MODEL_FKPP
    n_suffix = 5

    @property
    def state_dim(self):
        return self.nx

    def consts(self):
        return ()

    def num_params(self):
        return self.chain.num_params() + 5


@dataclass(frozen=True)
class NeuralODE:
    """du = ann(u, p): the black-box form (seir_exposure.jl:52-64 without its input scaling)."""
    chain: FastChain

    model = _lib.MODEL_NODE

    @property
    def state_dim(self):
        return self.chain.widths[0]

    def consts(self):
        return ()

    def num_params(self):
        return self.chain.num_params()


@dataclass
class SEIRNeuralODE:
    """dudt_node of the SEIR script (seir_exposure.jl:52-64): dS,dE,dI,dR,dD = first five outputs of
    ann_node([S/N,E,I,R,N,D/N,C]), dN = -mu N, dC = sigma E; chain 7 -> ... -> 7 (the script: 7-64-64-64-7 tanh)."""
    chain: FastChain
    p_: Sequence[float] = SEIR_P   # seir_exposure.jl:33

    model = _lib.MODEL_SEIR_NODE
    state_dim = 7

    def consts(self):
        return tuple(float(x) for x in self.p_)

    def num_params(self):
        return self.chain.num_params()


# --------------------------------------------------------------------------- problem / algorithm types
@dataclass
class ODEProblem:
    """ODEProblem(f, u0, tspan, p) -- f must be a recognised UDE form."""
    f: object
    u0: object
    tspan: tuple
    p: object = None


def remake(prob: ODEProblem, **kw) -> ODEProblem:
    return ODEProblem(kw.get("f", prob.f), kw.get("u0", prob.u0), kw.get("tspan", prob.tspan), kw.get("p", prob.p))


@dataclass
class EnsembleProblem:
    """EnsembleProblem(prob; u0s): the same problem for N initial conditions u0s[d, N] sharing theta."""
    prob: ODEProblem
    u0s: object


class Tsit5:
    code = _lib.TSIT5


class Vern7:
    code = _lib.VERN7


def _rkc2_beta(s):
    """Length of the real stability interval of s-stage RKC2 (damping 2/13): (w0 + 1) T''_s(w0) / T'_s(w0) ~ 0.65 s^2."""
    w0 = 1.0 + (2.0 / 13.0) / (s * s)
    T0, T1, d0, d1, e0, e1 = 1.0, w0, 0.0, 1.0, 0.0, 0.0
    for _ in range(2, s + 1):
        T0, T1, d0, d1, e0, e1 = T1, 2 * w0 * T1 - T0, d1, 2 * T1 + 2 * w0 * d1 - d0, e1, 4 * d1 + 2 * w0 * e1 - e0
    return (w0 + 1.0) * e1 / d1


class RKC2:
    """Stabilised explicit second-order Runge-Kutta-Chebyshev solver -- what this path offers where the reference calls
    `ROCK2(eigen_est = ...)` (Climate/NeuralPDE/npde.jl:61,82; named by the north star for the stiff Fisher-KPP grid):
    same class of method (explicit, stability interval growing with the square of the stage count), closed-form
    coefficients (ROCK2's tables are not in the reference).  Give `stages`, or `eigen_est` (an upper bound of the spectral
    radius of the RHS Jacobian, as the reference's ROCK2 call does) from which the stage count is chosen for the step."""
    code = _lib.RKC2

    def __init__(self, stages=None, eigen_est=None):
        self.stages, self.eigen_est = stages, eigen_est

    def n_stages(self, dt):
        if self.stages is not None:
            return int(self.stages)
        if self.eigen_est is None:
            raise ValueError("RKC2 needs stages= or eigen_est=")
        s = 2
        while _rkc2_beta(s) < 1.05 * dt * float(self.eigen_est):
            s += 1
            if s > 64:
                raise ValueError("dt * eigen_est needs more than 64 stages: reduce dt")
        return s


class ROCK2(RKC2):
    """The name the reference's scripts use (npde.jl:61,82,122).  NOT the ROCK2 algorithm: ROCK2's orthogonal-polynomial
    recurrence tables are not in the reference, so this selects RKC2 -- a different second-order stabilised explicit
    method of the same class -- and says so once per process."""
    _warned = False

    def __init__(self, stages=None, eigen_est=None):
        if not ROCK2._warned:
            warnings.warn("ROCK2(...) selects RKC2 (second-order Runge-Kutta-Chebyshev), not OrdinaryDiffEq's ROCK2: same "
                          "order and stability class, different stage recurrence; results agree to the solver tolerance, not bitwise",
                          RuntimeWarning, stacklevel=2)
            ROCK2._warned = True
        super().__init__(stages, eigen_est)


class ReverseDiffVJP:
    pass


class ZygoteVJP:
    pass


@dataclass
class InterpolatingAdjoint:
    autojacvec: object = field(default_factory=ReverseDiffVJP)
    code = _lib.INTERPOLATING_ADJOINT


class ForwardDiffSensitivity:
    """ForwardDiffSensitivity() of the LV scripts (scenario_1.jl:86, scenario_2.jl:108, hudson_bay.jl:102): the exact
    derivative of the discrete solver scheme.  The reference pushes dual numbers through the solver (cost O(P) forward
    solves); here the same quantity comes from reverse accumulation through the Tsit5 stages (one backward sweep,
    B200UDE_DISCRETE_ADJOINT).  Fixed-step Tsit5 on the LV chains."""
    code = _lib.DISCRETE_ADJOINT


# --------------------------------------------------------------------------- engine
def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _desc(f, device_index, dtype, alg, sensealg, t0, dt, n_steps, save_every, loss_weights, max_trajectories):
    """struct b200ude_desc of a UDE form on a fixed grid."""
    d = _lib.Desc()
    d.struct_size = C.sizeof(_lib.Desc)
    d.device = device_index
    d.dtype = _lib.F64 if dtype == torch.float64 else _lib.F32
    d.model = f.model
    d.state_dim = f.state_dim
    chain = f.chain
    d.n_layers = len(chain.layers)
    for i, w in enumerate(chain.widths):
        d.widths[i] = w
    for i, a in enumerate(chain.acts):
        d.acts[i] = _ACT_CODE[a]
    d.n_prefix = getattr(f, "trainable_rates", 0)
    d.n_suffix = getattr(f, "n_suffix", 0)
    cs = f.consts()
    d.n_consts = len(cs)
    for i, c in enumerate(cs):
        d.consts[i] = c
    d.solver = alg.code
    d.n_stages = alg.n_stages(float(dt)) if isinstance(alg, RKC2) else 0
    d.sensealg = sensealg.code
    d.t0, d.dt, d.n_steps, d.save_every = t0, dt, n_steps, save_every
    if loss_weights is not None:
        d.n_loss_weights = len(loss_weights)
        for i, w in enumerate(loss_weights):
            d.loss_weights[i] = float(w)
    d.max_trajectories = int(max_trajectories)
    return d


class UDESolver:
    """One C-ABI handle: a UDE form, a fixed Tsit5 grid and a capacity of trajectories."""

    def __init__(self, f, t0, dt, n_steps, save_every=1, max_trajectories=1, device=None,
                 loss_weights=None, alg=None, sensealg=None, approx_tanh=False, adaptive=False, abstol=1e-6, reltol=1e-3,
                 max_steps=512, dtype=torch.float32):
        alg = alg or Tsit5()
        sensealg = sensealg or InterpolatingAdjoint()
        if not isinstance(sensealg, (InterpolatingAdjoint, ForwardDiffSensitivity)):
            raise TypeError(f"unsupported sensealg {sensealg!r}")
        if not torch.cuda.is_available():
            raise RuntimeError("b200ude needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else torch.device(device).index or 0)
        self.f = f
        self.n_steps, self.save_every, self.dt, self.t0 = int(n_steps), int(save_every), float(dt), float(t0)
        if dtype not in (torch.float32, torch.float64):
            raise TypeError("dtype must be torch.float32 or torch.float64")
        self.dtype = dtype
        d = _desc(f, self.device.index, dtype, alg, sensealg, self.t0, self.dt, self.n_steps, self.save_every, loss_weights, max_trajectories)
        d.flags = _lib.FLAG_APPROX_TANH if approx_tanh else 0
        # adaptive = true: OrdinaryDiffEq's defaults abstol = 1e-6, reltol = 1e-3 when the kwargs are omitted (Fisher-KPP-CNN.jl:136)
        d.adaptive = 1 if adaptive else 0
        d.abstol, d.reltol, d.max_steps = float(abstol), float(reltol), int(max_steps)
        self._L = _lib.lib()
        h = C.c_void_p()
        rc = self._L.b200ude_create(C.byref(d), C.byref(h))
        if rc != 0:
            raise _lib.B200UDEError(rc, (self._L.b200ude_last_error(None) or b"").decode())
        self._h = h
        self.P = int(self._L.b200ude_num_params(h))
        self.n_save = int(self._L.b200ude_num_save(h))
        self.d = f.state_dim
        self.capacity = int(max_trajectories)
        self.adaptive, self.max_steps = bool(adaptive), int(max_steps)
        self.generation = 0   # bumped by every set_params / forward: identifies the forward record the handle holds

    def close(self):
        if getattr(self, "_h", None):
            self._L.b200ude_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- device-pointer API (inputs already resident in HBM) -------------------------------
    def set_params(self, theta: torch.Tensor):
        theta = theta.detach()
        if theta.dtype != self.dtype or theta.numel() != self.P:
            raise ValueError(f"theta must be {self.dtype}[{self.P}]")
        if theta.is_cuda:
            theta = theta.contiguous()
            _lib.check(self._h, self._L.b200ude_set_params(self._h, theta.data_ptr(), self.P, _lib.DEVICE, _stream_ptr(self.device)))
        else:
            arr = theta.contiguous()
            _lib.check(self._h, self._L.b200ude_set_params(self._h, arr.data_ptr(), self.P, _lib.HOST, _stream_ptr(self.device)))
        self._theta_keepalive = theta
        self.generation += 1

    def forward(self, u0: torch.Tensor, out: Optional[torch.Tensor] = None, status: Optional[torch.Tensor] = None):
        """u0[d, N] (cuda, the solver's dtype) -> out[n_save, d, N]."""
        assert u0.is_cuda and u0.dtype == self.dtype and u0.dim() == 2 and u0.shape[0] == self.d
        u0 = u0.contiguous()
        N = u0.shape[1]
        if out is None:
            out = torch.empty((self.n_save, self.d, N), device=u0.device, dtype=self.dtype)
        sp = status.data_ptr() if status is not None else None
        _lib.check(self._h, self._L.b200ude_forward(self._h, u0.data_ptr(), N, out.data_ptr(), sp, _stream_ptr(self.device)))
        self.generation += 1
        return out

    def adjoint(self, dL_dout: torch.Tensor, want_grad_u0=True):
        """dL_dout[n_save, d, N] -> (grad_theta[P] summed over the ensemble, grad_u0[d, N])."""
        dL_dout = dL_dout.contiguous()
        N = dL_dout.shape[2]
        assert dL_dout.dtype == self.dtype
        gth = torch.empty(self.P, device=dL_dout.device, dtype=self.dtype)
        gu0 = torch.empty((self.d, N), device=dL_dout.device, dtype=self.dtype) if want_grad_u0 else None
        _lib.check(self._h, self._L.b200ude_adjoint(self._h, dL_dout.data_ptr(), gth.data_ptr(),
                                                  gu0.data_ptr() if gu0 is not None else None, _stream_ptr(self.device)))
        return gth, gu0

    def adjoint_l2(self, data: torch.Tensor, want_grad_u0=False, grad_theta=None, loss=None):
        """Fused L2 loss + adjoint: data[n_save, d, N] -> (loss[1], grad_theta[P], grad_u0)."""
        data = data.contiguous()
        N = data.shape[2]
        assert data.dtype == self.dtype
        if grad_theta is None:
            grad_theta = torch.empty(self.P, device=data.device, dtype=self.dtype)
        if loss is None:
            loss = torch.empty(1, device=data.device, dtype=self.dtype)
        gu0 = torch.empty((self.d, N), device=data.device, dtype=self.dtype) if want_grad_u0 else None
        _lib.check(self._h, self._L.b200ude_adjoint_l2(self._h, data.data_ptr(), loss.data_ptr(), grad_theta.data_ptr(),
                                                     gu0.data_ptr() if gu0 is not None else None, _stream_ptr(self.device)))
        return loss, grad_theta, gu0

    # -- host-buffer API (what a host-language binding calls) ---------------------------------
    def solve_host(self, theta: np.ndarray, u0: np.ndarray):
        theta = np.ascontiguousarray(theta, np.float32)
        u0 = np.ascontiguousarray(u0, np.float32)
        N = u0.shape[1]
        out = np.empty((self.n_save, self.d, N), np.float32)
        status = np.empty(N, np.int32)
        self.generation += 1
        _lib.check(self._h, self._L.b200ude_solve_host(self._h, theta.ctypes.data, u0.ctypes.data, N, out.ctypes.data, status.ctypes.data))
        return out, status

    def loss_gradient_host(self, theta, u0, data, grad_theta=None, grad_u0=None):
        """Pinned torch CPU tensors or numpy arrays in, (loss, grad_theta[, grad_u0]) out; synchronous."""
        def ptr(a):
            return a.data_ptr() if isinstance(a, torch.Tensor) else a.ctypes.data
        N = u0.shape[1]
        if grad_theta is None:
            grad_theta = np.empty(self.P, np.float32)
        loss = C.c_double(0.0)
        self.generation += 1
        _lib.check(self._h, self._L.b200ude_loss_gradient_host(self._h, ptr(theta), ptr(u0), ptr(data), N, C.byref(loss), ptr(grad_theta),
                                                             ptr(grad_u0) if grad_u0 is not None else None))
        return loss.value, grad_theta, grad_u0


    # -- multi-GPU: fused reduce + all-reduce over NVLink peer memory (dist.PeerAllReduce drives these) ----
    def peer_export(self) -> bytes:
        buf = C.create_string_buffer(_lib.PEER_HANDLE_BYTES)
        _lib.check(self._h, self._L.b200ude_peer_export(self._h, buf))
        return buf.raw

    def peer_attach(self, rank: int, world: int, handles: bytes):
        assert len(handles) == world * _lib.PEER_HANDLE_BYTES
        _lib.check(self._h, self._L.b200ude_peer_attach(self._h, rank, world, handles))

    def peer_detach(self):
        _lib.check(self._h, self._L.b200ude_peer_detach(self._h))

    def adjoint_l2_allreduce(self, data: torch.Tensor, want_grad_u0=False, grad_theta=None, loss=None):
        """adjoint_l2 whose loss and grad_theta are summed over all attached ranks inside the reduction kernel."""
        data = data.contiguous()
        N = data.shape[2]
        if grad_theta is None:
            grad_theta = torch.empty(self.P, device=data.device, dtype=torch.float32)
        if loss is None:
            loss = torch.empty(1, device=data.device, dtype=torch.float32)
        gu0 = torch.empty((self.d, N), device=data.device, dtype=torch.float32) if want_grad_u0 else None
        _lib.check(self._h, self._L.b200ude_adjoint_l2_allreduce(self._h, data.data_ptr(), loss.data_ptr(), grad_theta.data_ptr(),
                                                               gu0.data_ptr() if gu0 is not None else None, _stream_ptr(self.device)))
        return loss, grad_theta, gu0

    # -- on-device optimiser ----------------------------------------------------------------
    @staticmethod
    def _adam_struct(opt, loss_scale=1.0, l2_reg=0.0):
        a = _lib.Adam()
        a.struct_size = C.sizeof(_lib.Adam)
        a.eta, (a.beta1, a.beta2), a.eps = opt.eta, opt.beta, opt.eps
        a.loss_scale, a.l2_reg = loss_scale, l2_reg
        return a

    def get_params(self) -> torch.Tensor:
        th = torch.empty(self.P, device=self.device, dtype=self.dtype)
        _lib.check(self._h, self._L.b200ude_get_params(self._h, th.data_ptr(), self.P, _lib.DEVICE, _stream_ptr(self.device)))
        return th

    def adam_reset(self):
        _lib.check(self._h, self._L.b200ude_adam_reset(self._h, _stream_ptr(self.device)))

    def adam_step(self, opt, grad_theta: torch.Tensor, loss_scale=1.0, l2_reg=0.0):
        """One ADAM update of the handle's theta with a device gradient (e.g. all-reduced over ranks)."""
        a = self._adam_struct(opt, loss_scale, l2_reg)
        grad_theta = grad_theta.contiguous()
        _lib.check(self._h, self._L.b200ude_adam_step(self._h, C.byref(a), grad_theta.data_ptr(), _stream_ptr(self.device)))

    def train_adam(self, opt, u0: torch.Tensor, data: torch.Tensor, iters: int, loss_scale=1.0, l2_reg=0.0,
                   loss_history: Optional[torch.Tensor] = None) -> torch.Tensor:
        """`iters` iterations of forward + fused-L2 adjoint + ADAM on the device (one CUDA graph replayed); returns the
        per-iteration pre-update losses (device float32[iters])."""
        a = self._adam_struct(opt, loss_scale, l2_reg)
        u0, data = u0.contiguous(), data.contiguous()
        if loss_history is None:
            loss_history = torch.empty(iters, device=self.device, dtype=torch.float32)
        self.generation += 1
        _lib.check(self._h, self._L.b200ude_train_adam(self._h, C.byref(a), u0.data_ptr(), data.data_ptr(), u0.shape[1], iters,
                                                     loss_history.data_ptr(), _stream_ptr(self.device)))
        return loss_history


class UDEBatchSolver:
    """M independent trainings at once (b200ude_batch_*): the batch counterpart of UDESolver for the reference's LV UDE with the
    2-5-5-5-2 chain, fixed-step Tsit5, fp32.  Every member has its own theta, u0, data, gradient and ADAM moments; one trajectory per
    member.  The device counterpart of run_loops.jl:55-62's loop over recover_dynamics.  Arrays: theta / grad [M, P] (row n = member
    n's flat theta in the reference's order), u0 [d, M], data / out [n_save, d, M], loss / status [M], loss history [iters, M]."""

    def __init__(self, f, t0, dt, n_steps, save_every=1, max_members=1, device=None, loss_weights=None, sensealg=None):
        sensealg = sensealg or InterpolatingAdjoint()
        if not isinstance(sensealg, (InterpolatingAdjoint, ForwardDiffSensitivity)):
            raise TypeError(f"unsupported sensealg {sensealg!r}")
        if not torch.cuda.is_available():
            raise RuntimeError("b200ude needs a CUDA device (sm_100a); there is no CPU fallback")
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else torch.device(device).index or 0)
        self.f = f
        self.n_steps, self.save_every, self.dt, self.t0 = int(n_steps), int(save_every), float(dt), float(t0)
        d = _desc(f, self.device.index, torch.float32, Tsit5(), sensealg, self.t0, self.dt, self.n_steps, self.save_every, loss_weights,
                  max_members)
        self._L = _lib.lib()
        h = C.c_void_p()
        rc = self._L.b200ude_batch_create(C.byref(d), C.byref(h))
        if rc != 0:
            raise _lib.B200UDEError(rc, (self._L.b200ude_batch_last_error(None) or b"").decode())
        self._h = h
        self.P = int(self._L.b200ude_batch_num_params(h))
        self.n_save = self.n_steps // self.save_every + 1
        self.d = f.state_dim
        self.capacity = int(max_members)
        self.members = 0

    def close(self):
        if getattr(self, "_h", None):
            self._L.b200ude_batch_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        _lib.check_batch(self._h, rc)

    def _inputs(self, u0, data=None):
        """Checks u0 [d, M] (and data [n_save, d, M]): CUDA float32 on the solver's device, M within the members set; returns them
        contiguous with M."""
        for name, a in (("u0", u0), ("data", data)):
            if a is None:
                continue
            if not isinstance(a, torch.Tensor) or not a.is_cuda or a.dtype != torch.float32 or a.device != self.device:
                raise TypeError(f"{name} must be a float32 CUDA tensor on {self.device}")
        if u0.dim() != 2 or u0.shape[0] != self.d:
            raise ValueError(f"u0 must be [{self.d}, M], got {tuple(u0.shape)}")
        M = u0.shape[1]
        if not 0 < M <= self.members:
            raise ValueError(f"M = {M} members, but set_params stored {self.members}")
        if data is not None and tuple(data.shape) != (self.n_save, self.d, M):
            raise ValueError(f"data must be [{self.n_save}, {self.d}, {M}], got {tuple(data.shape)}")
        return u0.contiguous(), (data.contiguous() if data is not None else None), M

    def set_params(self, theta):
        """theta [M, P] (host or device, float32) -> members 0..M-1; zeroes their ADAM state."""
        theta = torch.as_tensor(theta).detach().to(torch.float32).contiguous()
        if theta.dim() != 2 or theta.shape[1] != self.P or not 0 < theta.shape[0] <= self.capacity:
            raise ValueError(f"theta must be [M, {self.P}] with 0 < M <= {self.capacity}")
        if theta.is_cuda and theta.device != self.device:
            raise ValueError(f"theta is on {theta.device}, the solver on {self.device}")
        mem = _lib.DEVICE if theta.is_cuda else _lib.HOST
        self._check(self._L.b200ude_batch_set_params(self._h, theta.data_ptr(), theta.shape[0], mem, _stream_ptr(self.device)))
        self._theta_keepalive = theta
        self.members = theta.shape[0]

    def get_params(self, M=None) -> torch.Tensor:
        """The current thetas of members 0..M-1 [M, P]."""
        M = self.members if M is None else M
        th = torch.empty((M, self.P), device=self.device, dtype=torch.float32)
        self._check(self._L.b200ude_batch_get_params(self._h, th.data_ptr(), M, _lib.DEVICE, _stream_ptr(self.device)))
        return th

    def get_best(self, M=None):
        """Every member's best pre-update theta since set_params [M, P] and its loss [M] (+inf when it recorded no finite loss)."""
        M = self.members if M is None else M
        th = torch.empty((M, self.P), device=self.device, dtype=torch.float32)
        loss = torch.empty(M, device=self.device, dtype=torch.float32)
        self._check(self._L.b200ude_batch_get_best(self._h, th.data_ptr(), loss.data_ptr(), M, _lib.DEVICE, _stream_ptr(self.device)))
        return th, loss

    def forward(self, u0: torch.Tensor):
        """u0 [d, M] -> (out [n_save, d, M], status [M])."""
        u0, _, M = self._inputs(u0)
        out = torch.empty((self.n_save, self.d, M), device=self.device, dtype=torch.float32)
        status = torch.empty(M, device=self.device, dtype=torch.int32)
        self._check(self._L.b200ude_batch_forward(self._h, u0.data_ptr(), M, out.data_ptr(), status.data_ptr(), _stream_ptr(self.device)))
        return out, status

    def loss_gradient(self, u0: torch.Tensor, data: torch.Tensor):
        """Per-member fused L2 loss and gradient: (loss [M], grad [M, P], status [M])."""
        u0, data, M = self._inputs(u0, data)
        loss = torch.empty(M, device=self.device, dtype=torch.float32)
        grad = torch.empty((M, self.P), device=self.device, dtype=torch.float32)
        status = torch.empty(M, device=self.device, dtype=torch.int32)
        self._check(self._L.b200ude_batch_loss_gradient(self._h, u0.data_ptr(), data.data_ptr(), M, loss.data_ptr(), grad.data_ptr(),
                                                        status.data_ptr(), _stream_ptr(self.device)))
        return loss, grad, status

    def train_adam(self, opt, u0: torch.Tensor, data: torch.Tensor, iters: int, loss_scale=1.0, l2_reg=0.0):
        """`iters` ADAM iterations of every member in one launch: (loss history [iters, M] at the pre-update thetas, status [M])."""
        u0, data, M = self._inputs(u0, data)
        a = UDESolver._adam_struct(opt, loss_scale, l2_reg)
        hist = torch.empty((iters, M), device=self.device, dtype=torch.float32)
        status = torch.empty(M, device=self.device, dtype=torch.int32)
        self._check(self._L.b200ude_batch_train_adam(self._h, C.byref(a), u0.data_ptr(), data.data_ptr(), M, iters, hist.data_ptr(),
                                                     status.data_ptr(), _stream_ptr(self.device)))
        return hist, status


class _SolveFn(torch.autograd.Function):
    """concrete_solve with its reverse rule: backward = InterpolatingAdjoint on the stored forward."""

    @staticmethod
    def forward(ctx, theta, u0, solver):
        solver.set_params(theta)
        status = torch.zeros(u0.shape[1], dtype=torch.int32, device=u0.device) if solver.adaptive else None
        out = solver.forward(u0, status=status)
        if status is not None:
            # OrdinaryDiffEq reports retcode != Success (MaxIters / Unstable / DtLessThanMin) with a warning; the kernels
            # fill the unreached save points of a failed trajectory with NaN so that the failure reaches the loss
            nbad = int((status != 0).sum())
            if nbad:
                warnings.warn(f"concrete_solve: {nbad} of {u0.shape[1]} trajectories failed "
                              f"(status 1 = non-finite, 2 = max_steps={solver.max_steps} reached); their unreached save points are NaN",
                              RuntimeWarning, stacklevel=3)
        # the forward record (step states, stage derivatives, theta) lives in the handle, which later calls with the same
        # key reuse: remember which forward it holds and what produced it, so that backward can restore it
        ctx.solver = solver
        ctx.gen = solver.generation
        ctx.theta, ctx.u0 = theta.detach(), u0.detach()
        ctx.need_u0 = u0.requires_grad
        return out

    @staticmethod
    def backward(ctx, gout):
        solver = ctx.solver
        if solver.generation != ctx.gen:
            # another forward / set_params used the handle since (two predictions in one loss, multiple shooting,
            # mini-batches): re-run this call's forward so that the adjoint reads its own record and theta
            solver.set_params(ctx.theta)
            solver.forward(ctx.u0)
        gth, gu0 = solver.adjoint(gout, want_grad_u0=True)
        return gth, (gu0 if ctx.need_u0 else None), None


_SOLVERS = {}


def _grid_from(tspan, saveat, dt):
    t0, t1 = float(tspan[0]), float(tspan[1])
    if np.ndim(saveat) > 0:
        sv = np.asarray(saveat, dtype=np.float64)
        if len(sv) < 2 or abs(sv[0] - t0) > 1e-12 * max(1.0, abs(t0)):
            raise ValueError("saveat must start at tspan[1] and contain at least two points")
        step = np.diff(sv)
        if np.max(np.abs(step - step[0])) > 1e-9 * abs(step[0]):
            raise ValueError("only uniformly spaced saveat is supported by the fixed-step path")
        save_dt = float(step[0])
    elif saveat is None:
        save_dt = t1 - t0
    else:
        save_dt = float(saveat)
    if dt is None:
        dt = save_dt
    save_every = int(round(save_dt / dt))
    n_steps = int(round((t1 - t0) / dt))
    if save_every < 1 or abs(save_every * dt - save_dt) > 1e-9 * save_dt or abs(n_steps * dt - (t1 - t0)) > 1e-9 * (t1 - t0):
        raise ValueError("dt must divide the saveat spacing and the time span")
    return t0, float(dt), n_steps, save_every


def concrete_solve(prob, alg, u0=None, p=None, *, saveat=None, dt=None, adaptive=None, abstol=None, reltol=None,
                   sensealg=None, loss_weights=None, max_steps=512, dtype=torch.float32):
    """Array(concrete_solve(prob, Tsit5(), u0, p; saveat, sensealg=InterpolatingAdjoint(...))).

    `prob` may be an ODEProblem (u0[d] -> d x n_save, like Julia's Array(sol)) or an
    EnsembleProblem (u0s[d, N] -> n_save x d x N).  Differentiable w.r.t. p and u0.
    adaptive defaults to true when no dt is given (as in OrdinaryDiffEq): Tsit5 with the PI controller and
    abstol / reltol (defaults 1e-6 / 1e-3); pass dt= for adaptive=false.
    """
    ens = isinstance(prob, EnsembleProblem)
    base = prob.prob if ens else prob
    u0 = (prob.u0s if ens else base.u0) if u0 is None else u0
    p = base.p if p is None else p
    dev = torch.device("cuda", torch.cuda.current_device())
    u0t = torch.as_tensor(u0, dtype=dtype, device=dev) if not isinstance(u0, torch.Tensor) else u0.to(dev, dtype)
    if u0t.dim() == 1:
        u0t = u0t[:, None]
    pt = torch.as_tensor(p, dtype=dtype, device=dev) if not isinstance(p, torch.Tensor) else p
    if pt.dtype != dtype or not pt.is_cuda:
        pt = pt.to(dev, dtype)
    t0, dtv, n_steps, save_every = _grid_from(base.tspan, saveat, dt)
    N = u0t.shape[1]
    if adaptive is None:
        adaptive = dt is None
    abstol = 1e-6 if abstol is None else abstol
    reltol = 1e-3 if reltol is None else reltol
    key = (id(base.f), t0, dtv, n_steps, save_every, type(alg).__name__, getattr(alg, "stages", None), getattr(alg, "eigen_est", None),
           type(sensealg).__name__ if sensealg is not None else None, dev.index, tuple(loss_weights) if loss_weights else None,
           bool(adaptive), abstol, reltol, max_steps, str(dtype))
    solver = _SOLVERS.get(key)
    if solver is None or solver.capacity < N:
        # a smaller cached solver is only dropped from the cache (not closed): autograd graphs that are still alive
        # may hold it for their backward pass; its handle is destroyed when the last reference goes
        solver = UDESolver(base.f, t0, dtv, n_steps, save_every, max_trajectories=max(N, 1), device=dev, alg=alg,
                           sensealg=sensealg, loss_weights=loss_weights, adaptive=adaptive, abstol=abstol, reltol=reltol, max_steps=max_steps, dtype=dtype)
        _SOLVERS[key] = solver
    out = _SolveFn.apply(pt, u0t, solver)
    return out if ens else out[:, :, 0].transpose(0, 1)


solve = concrete_solve


# --------------------------------------------------------------------------- optimisers / sciml_train
@dataclass
class ADAM:
    """Flux.ADAM(eta, (beta1, beta2)); eps = 1e-8 (verified against the reference's stored loss history)."""
    eta: float = 0.001
    beta: tuple = (0.9, 0.999)
    eps: float = 1e-8


@dataclass
class BFGS:
    """Optim.BFGS(initial_stepnorm = ...): dense inverse-Hessian BFGS with backtracking line search."""
    initial_stepnorm: float = 0.01


@dataclass
class TrainResult:
    minimizer: torch.Tensor
    minimum: float
    iterations: int
    final: Optional[torch.Tensor] = None   # theta after the last update (sciml_train_l2)


def _loss_and_grad(loss: Callable, theta: torch.Tensor):
    th = theta.detach().clone().requires_grad_(True)
    res = loss(th)
    extra = ()
    if isinstance(res, tuple):
        res, extra = res[0], tuple(res[1:])
    g, = torch.autograd.grad(res, th)
    return float(res.detach()), g.detach(), extra


def sciml_train(loss: Callable, theta0, opt, cb: Optional[Callable] = None, maxiters: int = 100) -> TrainResult:
    """DiffEqFlux.sciml_train(loss, theta, opt; cb, maxiters).

    loss(theta) returns the scalar loss or a tuple whose first entry is the loss (the rest is
    forwarded to cb, seir_exposure.jl:144-158).  cb(theta, l, extras...) returning True halts
    (Fisher-KPP-CNN-Small.jl:230).  The callback sees the loss at the pre-update theta of the iteration.
    """
    if isinstance(theta0, torch.Tensor):   # keep the caller's dtype and device (e.g. a float64 host replay)
        th = theta0.detach().clone()
        dev = th.device
    else:
        dev = torch.device("cuda", torch.cuda.current_device()) if torch.cuda.is_available() else torch.device("cpu")
        th = torch.as_tensor(theta0, dtype=torch.float32).to(dev).clone()
    best, best_th, it = float("inf"), th.clone(), 0
    if isinstance(opt, ADAM):
        m = torch.zeros_like(th)
        v = torch.zeros_like(th)
        b1, b2 = opt.beta
        for it in range(1, maxiters + 1):
            l, g, extra = _loss_and_grad(loss, th)
            if l < best:
                best, best_th = l, th.clone()
            if cb is not None and cb(th, l, *extra):
                break
            m = b1 * m + (1 - b1) * g
            v = b2 * v + (1 - b2) * g * g
            th = th - opt.eta * (m / (1 - b1 ** it)) / (torch.sqrt(v / (1 - b2 ** it)) + opt.eps)
        return TrainResult(best_th, best, it)
    if isinstance(opt, BFGS):
        n = th.numel()
        l, g, extra = _loss_and_grad(loss, th)
        Hinv = torch.eye(n, device=dev, dtype=torch.float64) * (opt.initial_stepnorm / max(float(g.abs().max()), 1e-30))
        for it in range(1, maxiters + 1):
            if l < best:
                best, best_th = l, th.clone()
            if cb is not None and cb(th, l, *extra):
                break
            d = -(Hinv @ g.double())
            gd = float(g.double() @ d)
            if not gd < 0:  # reset a non-descent direction
                Hinv = torch.eye(n, device=dev, dtype=torch.float64) * (opt.initial_stepnorm / max(float(g.abs().max()), 1e-30))
                d = -(Hinv @ g.double())
                gd = float(g.double() @ d)
            a, ok = 1.0, False
            for _ in range(30):
                th_new = (th.double() + a * d).to(th.dtype)
                l_new, g_new, extra_new = _loss_and_grad(loss, th_new)
                if math.isfinite(l_new) and l_new <= l + 1e-4 * a * gd:
                    ok = True
                    break
                a *= 0.5
            if not ok:
                break
            s = (th_new - th).double()
            y = (g_new - g).double()
            sy = float(s @ y)
            if sy > 1e-12:
                rho = 1.0 / sy
                Hy = Hinv @ y
                Hinv = Hinv - rho * (torch.outer(s, Hy) + torch.outer(Hy, s)) + (rho * rho * float(y @ Hy) + rho) * torch.outer(s, s)
            th, l, g, extra = th_new, l_new, g_new, extra_new
            if float(g.abs().max()) < 1e-8:
                break
        if l < best:
            best, best_th = l, th.clone()
        return TrainResult(best_th, best, it)
    raise TypeError(f"unknown optimiser {opt!r}")


def sciml_train_l2(solver: "UDESolver", theta0, u0: torch.Tensor, data: torch.Tensor, opt: "ADAM", cb: Optional[Callable] = None,
                   maxiters: int = 100, chunk: int = 50, loss_scale: float = 1.0, l2_reg: float = 0.0) -> TrainResult:
    """sciml_train(loss, theta, ADAM(eta); cb, maxiters) for the trajectory-matching loss
    loss_scale * sum w (u - data)^2 + l2_reg * sum theta^2 (scenario_1.jl:91-94,111-114; scenario_2.jl:113-116) with the whole
    iteration -- forward, adjoint, reduce, ADAM -- on the device (b200ude_train_adam).  The host looks in every `chunk`
    iterations: cb(theta_at_chunk_start, l) is called for each recorded loss of the chunk and can halt the run at that
    boundary; the returned minimizer is the best (theta, loss) pair seen at a chunk start.  chunk = 1 reproduces the
    reference's per-iteration callback and best-so-far bookkeeping exactly.  `.final` holds the last theta."""
    th = torch.as_tensor(theta0, dtype=torch.float32).to(solver.device)
    solver.set_params(th)
    solver.adam_reset()
    best, best_th, it, halted = float("inf"), th.clone(), 0, False
    while it < maxiters and not halted:
        k = min(chunk, maxiters - it)
        start = solver.get_params()
        losses = solver.train_adam(opt, u0, data, k, loss_scale, l2_reg).cpu().numpy()
        it += k
        if float(losses[0]) < best:
            best, best_th = float(losses[0]), start
        if cb is not None:
            for l in losses:
                if cb(start, float(l)):
                    halted = True
                    break
    res = TrainResult(best_th, best, it)
    res.final = solver.get_params()
    return res


@dataclass
class BatchTrainResult:
    minimizers: torch.Tensor   # [M, P]: every member's best pre-update theta (sciml_train's minimizer; theta0 if no finite loss)
    minimum: torch.Tensor      # [M]: its loss (+inf: no finite loss)
    losses: torch.Tensor       # [maxiters, M]: loss at the pre-update theta of each iteration (NaN after a member stopped)
    status: torch.Tensor       # [M]: 0, or B200UDE_TRAJ_NONFINITE for a member whose state, loss or gradient turned non-finite
    final: torch.Tensor        # [M, P]: every member's theta after its last update (a stopped member: its last finite theta)


def sciml_train_batch(solver: "UDEBatchSolver", theta0, u0: torch.Tensor, data: torch.Tensor, opt: "ADAM", maxiters: int = 100,
                      loss_scale: float = 1.0, l2_reg: float = 0.0) -> BatchTrainResult:
    """sciml_train(loss, theta, ADAM(eta); maxiters) for M independent problems at once -- the ADAM phase of every run of
    run_loops.jl:55-62 (loop_recoveries.jl:71-77) in one device call.  theta0 [M, P], u0 [d, M], data [n_save, d, M]; the loss is
    loss_scale * sum w (u - data)^2 + l2_reg * sum theta[n_prefix:]^2 per member (the loop: l2_reg = 1e-4 / P).  As sciml_train, every
    member's minimizer is the theta of its lowest recorded loss -- what loop_recoveries.jl:78-84 hands to BFGS; `.final` is the last
    iterate."""
    solver.set_params(theta0)
    losses, status = solver.train_adam(opt, u0, data, maxiters, loss_scale, l2_reg)
    best, minimum = solver.get_best()
    return BatchTrainResult(best, minimum, losses, status, solver.get_params())
