"""Host-side mirror of the reference call surface (no GPU needed): parameter layout, grid logic,
optimiser semantics, error behaviour."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

import universal_differential_equations_b200 as ude
from universal_differential_equations_b200 import sciml
from helpers import theta_scenario1_init


def test_chain_layout_matches_reference_flattening(O, golden):
    """initial_params / Lux ComponentVector order: per layer vec(W) column-major then b (KAT-1 layout)."""
    chain = ude.FastChain(ude.FastDense(2, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 2))
    assert chain.num_params() == 87 and chain.widths == (2, 5, 5, 5, 2)
    th = ude.initial_params(chain, np.random.default_rng(0))
    assert th.dtype == np.float32 and th.shape == (87,)
    assert np.all(th[10:15] == 0) and np.all(th[85:87] == 0)          # zero biases
    lim = np.sqrt(6.0 / 7)
    assert np.abs(th[:10]).max() <= lim                                 # Glorot-uniform bound of layer 1
    with pytest.raises(ValueError):
        ude.FastChain(ude.FastDense(2, 5), ude.FastDense(4, 2))
    f = ude.LotkaVolterraUDE(chain, trainable_rates=2)
    assert f.num_params() == 89 and f.consts() == (1.3, 1.8)


def test_grid_from_saveat():
    assert sciml._grid_from((0.0, 3.0), 0.1, None) == (0.0, 0.1, 30, 1)
    assert sciml._grid_from((0.0, 3.0), np.arange(0, 3.05, 0.1), 0.05) == (0.0, 0.05, 60, 2)
    with pytest.raises(ValueError):
        sciml._grid_from((0.0, 3.0), 0.1, 0.07)
    with pytest.raises(ValueError):
        sciml._grid_from((0.0, 3.0), np.array([0.0, 0.1, 0.3]), None)


def test_unsupported_requests_fail_loudly():
    chain = ude.FastChain(ude.FastDense(2, 32, ude.tanh), ude.FastDense(32, 32, ude.tanh), ude.FastDense(32, 2))
    prob = ude.ODEProblem(ude.LotkaVolterraUDE(chain), np.zeros(2), (0.0, 3.0), np.zeros(1218, np.float32))
    if not torch.cuda.is_available():
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            ude.UDESolver(prob.f, 0.0, 0.1, 30)
    with pytest.raises(TypeError):
        ude.UDESolver(prob.f, 0.0, 0.1, 30, sensealg=object())   # anything but InterpolatingAdjoint / ForwardDiffSensitivity


def test_sciml_train_adam_reproduces_reference_loss_history(O, golden):
    """sciml_train(loss, theta, ADAM(0.1)) driven by the oracle's loss/gradient replays the reference's
    stored losses[0..5] (scenario_1.jl:114): pins ADAM's betas, bias correction, eps scale and the
    callback convention (loss at the pre-update theta)."""
    g = golden["scenario_1"]
    m = O.lv_model((2, 5, 5, 5, 2), ("rbf", "rbf", "rbf", "identity"))
    X = g["X"]

    class OracleLoss(torch.autograd.Function):
        @staticmethod
        def forward(ctx, th):
            t64 = th.detach().cpu().numpy().astype(np.float64)
            out, dense = O.solve_fixed(m, t64, X[:, 0], 0.1 / 16, 480, save_every=16, want_dense=True)
            r = out - X.T
            gth, _ = O.adjoint_fixed(m, t64, out, dense, 0.1 / 16, 480, 2 * r, save_every=16)
            ctx.g = torch.from_numpy(gth)
            return torch.tensor((r**2).sum(), dtype=torch.float64)

        @staticmethod
        def backward(ctx, go):
            return (go * ctx.g).to(torch.float64)
    seen = []
    th0 = torch.from_numpy(theta_scenario1_init(g))
    def loss(th):
        return OracleLoss.apply(th.double())

    def cb(th, l):
        seen.append(l)
        return len(seen) >= 6
    res = ude.sciml_train(loss, th0, ude.ADAM(0.1), cb=cb, maxiters=10)   # float64 host tensor in -> float64 replay
    ref = g["losses"][:6]
    assert len(seen) == 6 and res.iterations == 6
    assert np.all(np.abs(np.array(seen) - ref) <= 2e-6 * ref), (seen, ref)


def test_sciml_train_bfgs_and_callback_halt():
    A = torch.tensor([[3.0, 0.5], [0.5, 1.0]])
    b = torch.tensor([1.0, -2.0])

    def loss(th):   # sciml_train puts a numpy theta on the current CUDA device when there is one
        return 0.5 * th @ (A.to(th.device) @ th) - b.to(th.device) @ th
    res = ude.sciml_train(loss, np.zeros(2, np.float32), ude.BFGS(initial_stepnorm=0.01), maxiters=200)
    sol = torch.linalg.solve(A, b)
    assert torch.allclose(res.minimizer.cpu(), sol, atol=1e-4)
    calls = []
    res = ude.sciml_train(loss, np.zeros(2, np.float32), ude.ADAM(0.05), cb=lambda th, l: calls.append(l) or len(calls) >= 3, maxiters=50)
    assert res.iterations == 3 and len(calls) == 3
    # loss returning (loss, extras...) forwards the extras to the callback (seir_exposure.jl:144-158)
    got = []
    ude.sciml_train(lambda th: (loss(th), "pred"), np.zeros(2, np.float32), ude.ADAM(0.05), cb=lambda th, l, pred: got.append(pred) or True, maxiters=5)
    assert got == ["pred"]


def test_rock2_stage_selection_from_eigen_est():
    """ROCK2(eigen_est = rho) picks the smallest RKC2 stage count whose real stability interval covers 1.05 dt rho."""
    from universal_differential_equations_b200.sciml import _rkc2_beta
    assert abs(_rkc2_beta(2) - 1.9629629629629626) < 1e-12 and 0.64 * 64 * 64 < _rkc2_beta(64) < 0.66 * 64 * 64
    for dt, rho in ((0.0125, 2603.0), (0.05, 160.8), (0.1, 2603.0)):
        s = ude.ROCK2(eigen_est=rho).n_stages(dt)
        assert _rkc2_beta(s) >= 1.05 * dt * rho and (s == 2 or _rkc2_beta(s - 1) < 1.05 * dt * rho)
    assert ude.ROCK2(stages=7).n_stages(0.3) == 7
    with pytest.raises(ValueError):
        ude.ROCK2().n_stages(0.1)
    with pytest.raises(ValueError):
        ude.ROCK2(eigen_est=1e9).n_stages(1.0)
