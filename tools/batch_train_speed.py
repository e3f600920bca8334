"""Speed of the batched independent trainings (b200ude_batch_train_adam) on the loop's workload: M members of the LV 2-5-5-5-2 rbf UDE,
200 ADAM iterations, Tsit5 dt = 0.1/8 over t = 0..3 (31 saved points), the loop's loss (L2 data term + 1e-4/87 sum theta^2).
Prints one JSON line per M with the device name and power limit, device ms per ADAM iteration (CUDA events after a warm-up call),
member-iterations/s, the same iterations as one launch per iteration (the alternative launch structure), the serial baseline (the
existing b200ude_train_adam on N = 1 handles, measured over a few members and extrapolated to M), the single-thread CPU oracle's rate,
and FLOPs per member-iteration counted from the shapes.
    python tools/batch_train_speed.py [--members 1,498,8192,65536] [--iters 200]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import universal_differential_equations_b200 as ude  # noqa: E402
from helpers import synthetic_ensemble  # noqa: E402

SUB, NS = 8, 240
DT = 0.1 / SUB
L2_REG = 1e-4 / 87
P = 87


def flops_per_member_iteration(n_steps=NS, p=P):
    """Floating-point operations of one member-iteration counted from the shapes (an FMA = 2; MUFU ex2 / rcp not counted)."""
    chain = 2 * (2 * 5 + 5 * 5 + 5 * 5 + 5 * 2) + 2 * 15      # dense FMAs + the rbf arguments -x^2 log2(e)
    rhs = chain + 2 * 2                                          # + the known physics
    fwd = n_steps * (6 * rhs + 2 * 2 * 21)                       # 6 new stages per step (FSAL), 21 tableau FMAs per component
    vjp = 2 * (2 * 5 + 5 * 5 + 5 * 5 + 5 * 2) + 3 * 15          # reverse sweep + activation derivatives
    stage = chain + vjp + 2 * p + 2 * 2 * 7 + 2 * 2 * 6          # recompute, VJP, gradient accumulation, state, cotangent algebra
    adjoint = n_steps * 6 * stage
    adam = 12 * p
    return fwd + adjoint + adam


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "unknown"
    return name, q


def model():
    chain = ude.FastChain(ude.FastDense(2, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 5, ude.rbf), ude.FastDense(5, 2))
    return ude.LotkaVolterraUDE(chain)


def members(M, seed=0):
    rng = np.random.default_rng(seed)
    th = np.stack([ude.initial_params(model().chain, rng) for _ in range(min(M, 1024))])
    th = np.resize(th, (M, P)).astype(np.float32)
    u0, y = synthetic_ensemble(M, n_steps=30, dt=0.1, seed=seed)
    return torch.from_numpy(th), torch.from_numpy(u0).cuda(), torch.from_numpy(y).cuda()


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", default="1,498,8192,65536")
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--serial-members", type=int, default=4)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device: speeds are measured on the GPU only")
    name, power = device_info()
    opt, iters = ude.ADAM(0.1), a.iters

    # serial baseline: the existing single-training path, one N = 1 handle trained after another
    th, u0, y = members(a.serial_members, seed=1)
    one = ude.UDESolver(model(), 0.0, DT, NS, SUB, max_trajectories=1, sensealg=ude.ForwardDiffSensitivity())
    one.set_params(th[0].cuda())
    one.train_adam(opt, u0[:, :1], y[:, :, :1], 5, l2_reg=L2_REG)                      # warm-up
    ms = 0.0
    for k in range(a.serial_members):
        one.set_params(th[k].cuda())
        one.adam_reset()
        ms += timed(lambda: one.train_adam(opt, u0[:, k:k + 1].contiguous(), y[:, :, k:k + 1].contiguous(), iters, l2_reg=L2_REG))
    serial_ms_per_iter = ms / (a.serial_members * iters)

    # CPU oracle (fp64, one thread): loss + gradient of one member
    from oracle import oracle as O
    m = O.lv_model((2, 5, 5, 5, 2), ("rbf", "rbf", "rbf", "identity"))
    th64, u064, y64 = th[0].numpy().astype(np.float64), u0[:, :1].cpu().numpy().astype(np.float64), y[:, :, :1].cpu().numpy().astype(np.float64)
    t0, n_cpu = time.perf_counter(), 20
    for _ in range(n_cpu):
        O.ensemble_loss_grad_discrete(m, th64, u064, y64, np.ones(2), DT, NS, save_every=SUB)
    cpu_rate = n_cpu / (time.perf_counter() - t0)

    fl = flops_per_member_iteration()
    for M in [int(x) for x in a.members.split(",")]:
        th, u0, y = members(M)
        s = ude.UDEBatchSolver(model(), 0.0, DT, NS, SUB, max_members=M, sensealg=ude.ForwardDiffSensitivity())
        s.set_params(th)
        s.train_adam(opt, u0, y, 2, l2_reg=L2_REG)                                      # warm-up
        torch.cuda.synchronize()
        s.set_params(th)
        one_launch = timed(lambda: s.train_adam(opt, u0, y, iters, l2_reg=L2_REG))
        s.set_params(th)
        n_sep = min(iters, 50)
        per_launch = timed(lambda: [s.train_adam(opt, u0, y, 1, l2_reg=L2_REG) for _ in range(n_sep)]) / n_sep
        ms_it = one_launch / iters
        rate = M / (ms_it * 1e-3)
        print(json.dumps({
            "device": name, "power_limit_and_max_sm_clock": power, "members": M, "adam_iters": iters,
            "ms_per_adam_iteration": round(ms_it, 4), "member_iterations_per_s": round(rate, 1),
            "ms_per_iteration_one_launch_per_iteration": round(per_launch, 4),
            "adam_phase_s": round(one_launch * 1e-3, 4),
            "serial_baseline": {"what": f"b200ude_train_adam on N=1 handles, measured over {a.serial_members} members, extrapolated to M",
                                "ms_per_iteration": round(serial_ms_per_iter, 4),
                                "adam_phase_s_extrapolated": round(serial_ms_per_iter * 1e-3 * iters * M, 3)},
            "cpu_oracle_member_iterations_per_s_one_thread": round(cpu_rate, 1),
            "flops_per_member_iteration": fl, "achieved_gflops": round(fl * rate * 1e-9, 1),
        }), flush=True)
        del s


if __name__ == "__main__":
    main()
