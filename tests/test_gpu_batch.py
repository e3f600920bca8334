"""Batched independent trainings on the B200 (b200ude_batch_*, UDEBatchSolver, sciml_train_batch) against the reference's 498 runs of
LotkaVolterra/run_loops.jl (tests/golden/scenario_1_loop.npz), the fp64 oracle, and the shared-theta path at N = 1."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RBF3 = ("rbf", "rbf", "rbf", "identity")
SUB, NS = 8, 240
DT = 0.1 / SUB
L2_REG = 1e-4 / 87


@pytest.fixture(scope="module")
def loop():
    return np.load(os.path.join(ROOT, "tests", "golden", "scenario_1_loop.npz"))


@pytest.fixture(scope="module")
def ude():
    import universal_differential_equations_b200 as ude
    return ude


def _model(ude):
    chain = ude.FastChain(ude.FastDense(2, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 2))
    return ude.LotkaVolterraUDE(chain)


def _loop_arrays(loop):
    import torch
    X = loop["X"]                                                  # [R, 2, 31]
    u0 = torch.from_numpy(np.ascontiguousarray(X[:, :, 0].T)).cuda()          # [2, R]
    data = torch.from_numpy(np.ascontiguousarray(X.transpose(2, 1, 0))).cuda()  # [31, 2, R]
    return u0, data


def _batch(ude, M, sensealg=None):
    return ude.UDEBatchSolver(_model(ude), 0.0, DT, NS, SUB, max_members=M, sensealg=sensealg)


@pytest.mark.parametrize("discrete", [False, True])
def test_kat12_all_runs_in_one_call(ude, loop, discrete):
    """train_adam with ADAM(0.1), l2 = 1e-4/87 over all 498 runs at once reproduces every run's stored losses[0:6] (the bounds of the
    single-run GPU KAT-4: 2e-4 relative on the first three, 5e-3 on all six)."""
    import torch
    u0, data = _loop_arrays(loop)
    s = _batch(ude, 498, ude.ForwardDiffSensitivity() if discrete else None)
    s.set_params(torch.from_numpy(loop["theta_init"]))
    hist, status = s.train_adam(ude.ADAM(0.1), u0, data, 6, l2_reg=L2_REG)
    torch.cuda.synchronize()
    h = hist.cpu().numpy().T                                       # [R, 6]
    assert (status.cpu().numpy() == 0).all()
    rel = np.abs(h / loop["losses_head"][:, :6] - 1)
    print(f"KAT-12 GPU (discrete={discrete}): max rel first three {rel[:, :3].max():.3e}, all six {rel.max():.3e}")
    assert rel[:, :3].max() < 2e-4 and rel.max() < 5e-3


def test_kat12_forward_at_trained_parameters(O, ude, loop):
    """forward at every run's trained_parameters: the loss matches losses[end] within 2e-6 + 2e-3 losses[end] (the CPU KAT's bound plus
    1e-6 for the fp32 solve) and the fp64 oracle's loss within 1e-5 + 1e-4 L (the trained losses are 2e-4 ... 7e-2, small enough for
    the fp32 rounding of the 62 residuals to need an absolute term), trajectories match the oracle within 3e-4 (1 + |u|); the four
    runs whose stored parameters are NaN come back with status NONFINITE."""
    import torch
    u0, data = _loop_arrays(loop)
    s = _batch(ude, 498)
    th = loop["theta_trained"]
    s.set_params(torch.from_numpy(th))
    out, status = s.forward(u0)
    torch.cuda.synchronize()
    out, status = out.cpu().numpy().astype(np.float64), status.cpu().numpy()
    finite = np.isfinite(th).all(1)
    assert (status[finite] == 0).all() and (status[~finite] == 1).all()
    m = O.lv_model((2, 5, 5, 5, 2), RBF3)
    worst_ref, worst_orc, worst_u = 0.0, 0.0, 0.0
    for i in np.where(finite)[0]:
        th64 = th[i].astype(np.float64)
        ref = O.solve_fixed(m, th64, loop["X"][i][:, 0].astype(np.float64), DT, NS, save_every=SUB)
        worst_u = max(worst_u, float((np.abs(out[:, :, i] - ref) / (1 + np.abs(ref))).max()))
        reg = L2_REG * (th64 ** 2).sum()
        l_gpu = ((out[:, :, i] - loop["X"][i].T) ** 2).sum() + reg
        l_orc = ((ref - loop["X"][i].T) ** 2).sum() + reg
        last = float(loop["losses_last"][i])
        worst_ref = max(worst_ref, abs(l_gpu - last) - 2e-3 * last)
        worst_orc = max(worst_orc, abs(l_gpu - l_orc) - 1e-4 * l_orc)
    print(f"forward at trained: max(|L-last| - 2e-3 last) {worst_ref:.3e}, max(|L-oracle| - 1e-4 L) {worst_orc:.3e}, max traj err {worst_u:.3e}")
    assert worst_ref <= 2e-6 and worst_orc <= 1e-5 and worst_u <= 3e-4


def _random_members(M, seed=0):
    from helpers import synthetic_ensemble
    rng = np.random.default_rng(seed)
    th = np.empty((M, 87), np.float32)
    off = 0
    for nin, nout in ((2, 5), (5, 5), (5, 5), (5, 2)):
        lim = np.sqrt(6.0 / (nin + nout))
        th[:, off:off + nin * nout] = rng.uniform(-lim, lim, (M, nin * nout))
        th[:, off + nin * nout:off + nin * nout + nout] = rng.uniform(-0.1, 0.1, (M, nout))
        off += nin * nout + nout
    u0, y = synthetic_ensemble(M, n_steps=30, dt=0.1, seed=seed)
    return th, u0, y


@pytest.mark.parametrize("discrete", [False, True])
@pytest.mark.parametrize("M", [498, 65536])
def test_loss_gradient_per_member_vs_oracle(O, ude, loop, M, discrete):
    """Per-member loss (1e-4) and gradient (norm-relative 2e-3) against the fp64 oracle at N = 1, for the 498 runs at their
    initial parameters and for 65 536 random members (a sample of 64 checked)."""
    import torch
    if M == 498:
        th, X = loop["theta_init"], loop["X"]
        u0, y = np.ascontiguousarray(X[:, :, 0].T), np.ascontiguousarray(X.transpose(2, 1, 0))
        check = np.arange(M)
    else:
        th, u0, y = _random_members(M)
        check = np.random.default_rng(1).choice(M, 64, replace=False)
    s = _batch(ude, M, ude.ForwardDiffSensitivity() if discrete else None)
    s.set_params(torch.from_numpy(th))
    loss, grad, status = s.loss_gradient(torch.from_numpy(u0).cuda(), torch.from_numpy(y).cuda())
    torch.cuda.synchronize()
    loss, grad = loss.cpu().numpy(), grad.cpu().numpy()
    assert (status.cpu().numpy() == 0).all()
    m = O.lv_model((2, 5, 5, 5, 2), RBF3)
    fn = O.ensemble_loss_grad_discrete if discrete else O.ensemble_loss_grad
    el, eg = 0.0, 0.0
    for k in check:
        res = fn(m, th[k].astype(np.float64), u0[:, [k]].astype(np.float64), y[:, :, [k]].astype(np.float64), np.ones(2), DT, NS, save_every=SUB)
        l_ref, g_ref = res[0], res[1]
        el = max(el, abs(loss[k] - l_ref) / abs(l_ref))
        eg = max(eg, np.linalg.norm(grad[k] - g_ref) / np.linalg.norm(g_ref))
    print(f"loss_gradient M={M} discrete={discrete}: max rel loss {el:.3e}, max rel grad {eg:.3e}")
    assert el < 1e-4 and eg < 2e-3


@pytest.mark.parametrize("discrete", [False, True])
def test_batch_agrees_with_the_shared_theta_path(ude, loop, discrete):
    """Members of a 498-run batch trained for 20 iterations agree (1e-5 relative) with b200ude_train_adam on an N = 1 handle with the same
    theta0, data and options, and sciml_train_batch agrees with looping sciml_train_l2 with a per-iteration callback (chunk = 1, the
    reference's bookkeeping): loss history, minimizer (best pre-update theta), minimum and final theta."""
    import torch
    u0, data = _loop_arrays(loop)
    sens = ude.ForwardDiffSensitivity() if discrete else None
    opt = ude.ADAM(0.1)
    th0 = torch.from_numpy(loop["theta_init"])
    res = ude.sciml_train_batch(_batch(ude, 498, sens), th0, u0, data, opt, 20, l2_reg=L2_REG)
    assert (res.status.cpu().numpy() == 0).all()
    hist_b, th_b = res.losses.cpu().numpy(), res.final.cpu().numpy()
    best_b, min_b = res.minimizers.cpu().numpy(), res.minimum.cpu().numpy()
    np.testing.assert_array_equal(min_b, np.nanmin(hist_b, axis=0))   # the best is the lowest recorded loss ...
    assert (np.argmin(hist_b, axis=0) > 0).any()                        # ... which is not always theta0
    one = ude.UDESolver(_model(ude), 0.0, DT, NS, SUB, max_trajectories=1, sensealg=sens)
    worst_l, worst_t = 0.0, 0.0
    for k in (0, 1, 137, 250, 497):
        one.set_params(th0[k].cuda())
        one.adam_reset()
        h1 = one.train_adam(opt, u0[:, k:k + 1], data[:, :, k:k + 1], 20, l2_reg=L2_REG).cpu().numpy()
        t1 = one.get_params().cpu().numpy()
        worst_l = max(worst_l, float(np.abs(h1 / hist_b[:, k] - 1).max()))
        worst_t = max(worst_t, float((np.abs(t1 - th_b[k]) / (1 + np.abs(t1))).max()))
        seen = []
        r2 = ude.sciml_train_l2(one, th0[k], u0[:, k:k + 1], data[:, :, k:k + 1], opt, cb=lambda th, l: seen.append(l) and False,
                                maxiters=20, chunk=1, l2_reg=L2_REG)
        worst_l = max(worst_l, float(np.abs(np.array(seen) / hist_b[:, k] - 1).max()), abs(r2.minimum / min_b[k] - 1))
        worst_t = max(worst_t, float((np.abs(r2.final.cpu().numpy() - th_b[k]) / (1 + np.abs(th_b[k]))).max()),
                      float((np.abs(r2.minimizer.cpu().numpy() - best_b[k]) / (1 + np.abs(best_b[k]))).max()))
    print(f"batch vs N=1 train_adam / sciml_train_l2 (discrete={discrete}): max rel loss {worst_l:.3e}, max rel theta {worst_t:.3e}")
    assert worst_l < 1e-5 and worst_t < 1e-5


def test_members_are_independent_and_calls_repeat_bitwise(ude, loop):
    """A member's loss history and final theta are bitwise the same alone, in the batch of 498 and in a permuted batch; two identical
    calls are bitwise identical."""
    import torch
    u0, data = _loop_arrays(loop)
    th0 = torch.from_numpy(loop["theta_init"])
    s = _batch(ude, 498)

    def run(idx):
        idx = torch.as_tensor(idx)
        s.set_params(th0[idx])
        h, st = s.train_adam(ude.ADAM(0.1), u0[:, idx.cuda()].contiguous(), data[:, :, idx.cuda()].contiguous(), 12, l2_reg=L2_REG)
        return h.cpu().numpy(), s.get_params().cpu().numpy(), st.cpu().numpy()

    h_all, t_all, st_all = run(np.arange(498))
    h_again, t_again, _ = run(np.arange(498))
    assert (st_all == 0).all()
    assert np.array_equal(h_all, h_again) and np.array_equal(t_all, t_again)
    perm = np.random.default_rng(3).permutation(498)
    h_p, t_p, _ = run(perm)
    assert np.array_equal(h_p[:, np.argsort(perm)], h_all) and np.array_equal(t_p[np.argsort(perm)], t_all)
    for k in (0, 31, 32, 250, 497):
        h1, t1, _ = run([k])
        assert np.array_equal(h1[:, 0], h_all[:, k]) and np.array_equal(t1[0], t_all[k]), k


def test_a_diverging_member_stops_alone(ude, loop):
    """A member whose trajectory overflows ends with status NONFINITE, its theta finite and unchanged (frozen at its last finite value),
    NaN loss slots after the failure, and every other member bitwise identical to the batch without it."""
    import torch
    u0, data = _loop_arrays(loop)
    th0 = loop["theta_init"].copy()
    s = _batch(ude, 498)
    opt = ude.ADAM(0.1)
    s.set_params(torch.from_numpy(th0))
    h_ref, st_ref = s.train_adam(opt, u0, data, 8, l2_reg=L2_REG)
    t_ref = s.get_params().cpu().numpy()
    bad = 137
    th_bad = th0.copy()
    th_bad[bad, 85:87] = 3e38          # output-layer biases: the Runge-Kutta stage sums overflow in the first step
    s.set_params(torch.from_numpy(th_bad))
    h, st = s.train_adam(opt, u0, data, 8, l2_reg=L2_REG)
    t = s.get_params().cpu().numpy()
    h, st, h_ref = h.cpu().numpy(), st.cpu().numpy(), h_ref.cpu().numpy()
    assert st[bad] == 1 and (np.delete(st, bad) == 0).all() and (st_ref.cpu().numpy() == 0).all()
    assert np.isfinite(t[bad]).all() and np.array_equal(t[bad], th_bad[bad])
    assert not np.isfinite(h[0, bad]) and np.isnan(h[1:, bad]).all()
    others = np.arange(498) != bad
    assert np.array_equal(h[:, others], h_ref[:, others]) and np.array_equal(t[others], t_ref[others])


def test_members_keep_their_own_step_count_across_calls(ude, loop):
    """Calls may use fewer members than set_params stored: after 10 iterations of members 0..99 and then 6 of all 498, members >= 100 are
    bitwise a fresh 6-iteration run (their bias correction starts at step 1) and members < 100 bitwise a 16-iteration run."""
    import torch
    u0, data = _loop_arrays(loop)
    th0 = torch.from_numpy(loop["theta_init"])
    s = _batch(ude, 498)
    opt = ude.ADAM(0.1)

    def fresh(iters):
        s.set_params(th0)
        h, st = s.train_adam(opt, u0, data, iters, l2_reg=L2_REG)
        return h.cpu().numpy(), s.get_params().cpu().numpy()

    h6, t6 = fresh(6)
    h16, t16 = fresh(16)
    s.set_params(th0)
    s.train_adam(opt, u0[:, :100].contiguous(), data[:, :, :100].contiguous(), 10, l2_reg=L2_REG)
    h, st = s.train_adam(opt, u0, data, 6, l2_reg=L2_REG)
    h, t = h.cpu().numpy(), s.get_params().cpu().numpy()
    assert (st.cpu().numpy() == 0).all()
    assert np.array_equal(h[:, 100:], h6[:, 100:]) and np.array_equal(t[100:], t6[100:])
    assert np.array_equal(h[:, :100], h16[10:, :100]) and np.array_equal(t[:100], t16[:100])


def test_a_member_failing_after_updates_keeps_its_last_state(ude, loop):
    """Member j trains 5 iterations, then a call whose data make its loss non-finite: it stops in that call's first iteration with its
    theta bitwise the 5-iteration theta and NaN in the call's later slots.  A third call with its good data then continues it bitwise like
    a run that never failed -- its moments and step count were frozen, not advanced -- and every other member is untouched throughout."""
    import torch
    u0, data = _loop_arrays(loop)
    th0 = torch.from_numpy(loop["theta_init"])
    s = _batch(ude, 498)
    opt = ude.ADAM(0.1)
    j = 211
    bad = data.clone()
    bad[20:, :, j] = 3e38                       # residuals whose squares overflow: the member's loss is +inf

    def run(second):
        s.set_params(th0)
        s.train_adam(opt, u0, data, 5, l2_reg=L2_REG)
        h2, st2 = s.train_adam(opt, u0, second, 4, l2_reg=L2_REG)
        t2 = s.get_params().cpu().numpy()
        h3, st3 = s.train_adam(opt, u0, data, 3, l2_reg=L2_REG)
        return h2.cpu().numpy(), st2.cpu().numpy(), t2, h3.cpu().numpy(), st3.cpu().numpy(), s.get_params().cpu().numpy()

    s.set_params(th0)
    s.train_adam(opt, u0, data, 5, l2_reg=L2_REG)
    t5 = s.get_params().cpu().numpy()
    h2, st2, t2, h3, st3, t3 = run(bad)
    g2, gst2, gt2, g3, gst3, gt3 = run(data)    # the same calls without the failure
    assert st2[j] == 1 and (np.delete(st2, j) == 0).all() and (gst2 == 0).all()
    assert np.array_equal(t2[j], t5[j]) and np.isfinite(t2[j]).all()
    assert not np.isfinite(h2[0, j]) and np.isnan(h2[1:, j]).all()
    others = np.arange(498) != j
    assert np.array_equal(h2[:, others], g2[:, others]) and np.array_equal(t2[others], gt2[others])
    # continued with its good data, j is bitwise a run whose second call was its first 3 iterations after the 5
    s.set_params(th0)
    s.train_adam(opt, u0, data, 5, l2_reg=L2_REG)
    c3, cst3 = s.train_adam(opt, u0, data, 3, l2_reg=L2_REG)
    assert st3[j] == 0 and np.array_equal(h3[:, j], c3.cpu().numpy()[:, j]) and np.array_equal(t3[j], s.get_params().cpu().numpy()[j])
    assert np.array_equal(h3[:, others], g3[:, others]) and np.array_equal(t3[others], gt3[others])


def test_zero_l2_reg_ignores_the_l2_sum_and_inputs_are_checked(ude, loop):
    """With l2_reg = 0 the recorded loss does not contain l2_reg * sum theta^2 (a theta whose squares overflow still gives finite losses,
    as adam_kernel does); malformed arrays raise before anything reaches the kernels."""
    import torch
    u0, data = _loop_arrays(loop)
    th = loop["theta_init"][:4].copy()
    th[1, 0] = 1e20                             # a first-layer weight: rbf saturates to 0, the trajectory stays finite, theta^2 overflows
    s = _batch(ude, 4)
    s.set_params(torch.from_numpy(th))
    h, st = s.train_adam(ude.ADAM(0.1), u0[:, :4].contiguous(), data[:, :, :4].contiguous(), 3)
    assert (st.cpu().numpy() == 0).all() and np.isfinite(h.cpu().numpy()).all()
    with pytest.raises(ValueError):
        s.forward(u0[:1, :4].contiguous())                      # [1, M]: wrong state dimension
    with pytest.raises(ValueError):
        s.loss_gradient(u0[:, :4].contiguous(), data[:, :, :3].contiguous())
    with pytest.raises(ValueError):
        s.forward(u0[:, :5].contiguous())                       # more members than set_params stored
    with pytest.raises(TypeError):
        s.forward(u0[:, :4].double())
