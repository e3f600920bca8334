"""B200-native drop-in for the UDE training path of ChrisRackauckas/universal_differential_equations.

Only the hot path is here: ensemble forward solve of a universal differential equation
(known physics + embedded dense chain, Tsit5) and its interpolating-adjoint gradient,
as hand-written sm_100a kernels behind a C ABI (include/b200ude.h), plus a host-side
mirror of the reference's call surface (sciml.py).  See DESIGN.md.
"""
from . import _lib  # noqa: F401
from .sciml import (  # noqa: F401
    ADAM, BFGS, BatchTrainResult, Chain, Dense, EnsembleProblem, FastChain, FastDense, FisherKPPUDE, ForwardDiffSensitivity,
    InterpolatingAdjoint, LotkaVolterraUDE, NeuralODE, ODEProblem, SEIRExposureUDE, SEIRNeuralODE, ReverseDiffVJP, RKC2, ROCK2, Tsit5, UDEBatchSolver, UDESolver,
    Vern7, concrete_solve, identity, initial_params, rbf, remake, sciml_train, sciml_train_batch, sciml_train_l2, solve, tanh,
)
from . import pde  # noqa: F401
from . import jld2  # noqa: F401
from .pde import (  # noqa: F401
    BSDESolver, ConstantDiffusion, HJBNonlinearity, HJBTerminal, LambaEM, NNPDENS, TerminalPDEProblem, ZeroDrift, initial_params_pde, relu,
)
from .dist import PeerAllReduce, shard_range, allreduce_loss_grad  # noqa: F401


_ode_solve = solve


def solve(prob, algorithm, *args, **kw):  # noqa: F811
    """`solve(prob, alg; ...)`: ODE problems go to concrete_solve, TerminalPDEProblem + NNPDENS (with `alg = LambaEM()` as a
    keyword, lambaem.jl:33-34) to the deep-BSDE path."""
    if isinstance(prob, TerminalPDEProblem):
        return pde.solve(prob, algorithm, *args, **kw)
    return _ode_solve(prob, algorithm, *args, **kw)
