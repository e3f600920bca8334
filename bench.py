#!/usr/bin/env python3
"""bench.py -- ensemble trajectories/s, forward + interpolating adjoint (BASELINE.json's metric).

One "step" = one pass of the hot path over one batch of synthetic input: forward Tsit5 solve of every trajectory +
InterpolatingAdjoint gradient of the L2 trajectory-matching loss, summed over the ensemble (+ the sum over ranks of
[grad_theta; loss] when N_gpus > 1, fused into the final reduction kernel over NVLink peer memory).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--config lv|seir|fkpp|hjb] [--dump-outputs DIR]

--config lv (default, BASELINE config 2): 2->32->32->2 tanh chain, Glorot theta (seed 1), u0 ~ U(0.2,1) x U(2,5), 30 fixed
  Tsit5 steps of 0.1, states saved at every step, fp32.  The headline `value` is WEAK scaling (65 536 trajectories per GPU);
  the `strong` object of the same line is the metric's literal batch: 65 536 trajectories IN TOTAL over the N GPUs.
--config seir (config 3): 7-state SEIR exposure UDE, 3->64->64->1 chain, 84 steps of 0.25, saved daily, loss on E, I, R.
--config fkpp (config 4): Fisher-KPP UPDE on a 256-point grid, 1->16->16->1 reaction chain + 3-tap stencil, 200 steps.
--config hjb (config 5): highdim_pde/lambaem.jl's NNPDENS solve (d = 100, hls = 110, 20 Euler-Maruyama steps), 10 000 paths per GPU
  and iteration, fp64; a step = one iteration (forward paths + reverse sweep + ADAM); metric = paths/s.
Under torchrun one rank per GPU.  Rank 0 prints ONE JSON line.
--dump-outputs DIR: rank 0 writes what the last timed step returned as DIR/<name>.npy (lv / seir / fkpp: out[n_save, d, N] of its
  shard, grad_theta, loss; hjb: theta after the update, loss, u0 on 1 GPU or grad_theta, loss on several), so that two builds can be
  compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# the CPU legs run the OpenMP oracle: bind its threads before any OpenMP runtime is loaded -- but never in a multi-rank GPU run,
# where "close" binding would pin the main threads of ALL ranks to the same first core (measured: 8 ranks at 4.05 ms/step
# instead of 1.8)
if int(os.environ.get("WORLD_SIZE", "1")) == 1 or "reference" in sys.argv:
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")

import numpy as np  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_PER_GPU = 65536
UNIT = "trajectories/s"
FP32_PEAK_TFLOPS = 72.5     # measured FFMA/FFMA2 issue peak on this pool's B200 (profiles/r01_pipes_microbench.txt)
MUFU_PER_CLK_SM = 16.0      # measured (profiles/r01_pipes_microbench.txt): 0.499 warp instructions / clk / SM
HMMA_PER_CLK_SM = 0.468     # measured mma.sync m16n8k8.tf32 / m16n8k16.f16 warp instructions / clk / SM (profiles/r01_mma_sync_microbench.txt)


def host_cores():
    """Usable host cores: the affinity mask capped by the cgroup CPU quota (a 16-CPU quota on a 128-thread host
    is what made round 1's CPU arm swing 5x between boxes: 128 threads were time-sliced onto 16 CPUs)."""
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    cores = aff if quota is None else max(1, min(aff, int(quota)))
    return cores, aff, quota


# ----------------------------------------------------------------------------------------------- workloads
class LV:
    """BASELINE config 2."""
    name = "lv"
    metric = "ensemble trajectories/sec fwd+adjoint, LV UDE batch 65k"
    workload = "LV UDE ensemble, 2->32->32->2 tanh, Tsit5 dt=0.1 x30 saveat 0.1, fwd + InterpolatingAdjoint + L2 loss"
    n_steps, dt, every, D = 30, 0.1, 1, 2
    widths = (2, 32, 32, 2)
    P = 1218
    n_default = 65536
    fma_rhs = 2 * 32 + 32 * 32 + 32 * 2                                    # 1152 FMA per chain evaluation
    flop_fwd = 2.0 * fma_rhs * (1 + 6 * n_steps)                            # 181 RHS evaluations
    flop_adj = 2.0 * 3 * fma_rhs * (6 * n_steps)                            # 180 backward stages x (fwd + J_u^T + J_theta^T)
    bytes_fwd = 4.0 * (2 + 2 * (n_steps + 1) * 2 + (6 * n_steps + 1) * 2)   # u0 + out + per-step store + dense output
    bytes_adj = 4.0 * ((n_steps + 1) * 2 * 2 + (6 * n_steps + 1) * 2 + 2)   # per-step store + data + dense output + grad_u0
    loss_weights = None

    @staticmethod
    def synthetic(n, seed=0):
        from helpers import glorot_theta, synthetic_ensemble
        theta = glorot_theta(LV.widths, seed=1)
        u0, y = synthetic_ensemble(n, n_steps=LV.n_steps, dt=LV.dt, seed=seed)
        return theta, u0, y

    @staticmethod
    def make_solver(ude, n, dev):
        chain = ude.FastChain(ude.FastDense(2, 32, ude.tanh), ude.FastDense(32, 32, ude.tanh), ude.FastDense(32, 2))
        return ude.UDESolver(ude.LotkaVolterraUDE(chain), 0.0, LV.dt, LV.n_steps, LV.every, max_trajectories=n, device=dev)

    @staticmethod
    def oracle_model(O):
        return O.lv_model(), np.ones(2, np.float32)


class SEIR:
    """BASELINE config 3 in the reference's own shape (seir_exposure.jl:114-130): 7 states, chain 3->64->64->1 on [S/N, I, D/N]."""
    name = "seir"
    metric = "ensemble trajectories/sec fwd+adjoint, SEIR exposure UDE batch 65k"
    workload = "SEIR exposure UDE 7-state 3->64->64->1 tanh, Tsit5 dt=0.25 x84 over (0,21) saved daily, loss on E,I,R, fwd + InterpolatingAdjoint"
    n_steps, dt, every, D = 84, 0.25, 4, 7
    widths = (3, 64, 64, 1)
    P = 3 * 64 + 64 + 64 * 64 + 64 + 64 + 1
    n_default = 65536
    fma_rhs = 3 * 64 + 64 * 64 + 64
    flop_fwd = 2.0 * fma_rhs * (1 + 6 * n_steps)
    flop_adj = 2.0 * 3 * fma_rhs * (6 * n_steps)
    bytes_fwd = 4.0 * (7 + 7 * (n_steps // every + 1) + 7 * (n_steps + 1) + (6 * n_steps + 1) * 7)
    bytes_adj = 4.0 * (7 * (n_steps + 1) + 7 * (n_steps // every + 1) + (6 * n_steps + 1) * 7 + 7)
    loss_weights = [0, 1, 1, 1, 0, 0, 0]

    @staticmethod
    def synthetic(n, seed=0):
        from helpers import glorot_theta
        rng = np.random.default_rng(seed)
        theta = glorot_theta(SEIR.widths, seed=2)
        S0 = 14e6
        u0 = np.zeros((7, n), np.float32)
        u0[0] = 0.9 * S0 * rng.uniform(0.9, 1.0, n)
        u0[1:4] = rng.uniform(0, 50, (3, n))
        u0[4] = S0
        y = rng.uniform(0, 100, (SEIR.n_steps // SEIR.every + 1, 7, n)).astype(np.float32)
        return theta, u0, y

    @staticmethod
    def make_solver(ude, n, dev):
        chain = ude.FastChain(ude.FastDense(3, 64, ude.tanh), ude.FastDense(64, 64, ude.tanh), ude.FastDense(64, 1))
        return ude.UDESolver(ude.SEIRExposureUDE(chain), 0.0, SEIR.dt, SEIR.n_steps, SEIR.every, max_trajectories=n, device=dev,
                             loss_weights=SEIR.loss_weights)

    @staticmethod
    def oracle_model(O):
        return O.seir_model(), np.asarray(SEIR.loss_weights, np.float32)


class FKPP:
    """BASELINE config 4's shape (256-point grid, 1->16->16->1 reaction chain + 3-tap periodic stencil), Tsit5."""
    name = "fkpp"
    metric = "ensemble trajectories/sec fwd+adjoint, Fisher-KPP UPDE 256-point grid"
    workload = "Fisher-KPP UPDE 256-point grid, 1->16->16->1 tanh + 3-tap stencil, Tsit5 dt=1e-3 x200, fwd + InterpolatingAdjoint"
    Nx = 256
    n_steps, dt, every, D = 200, 1.0e-3, 20, 256
    widths = (1, 16, 16, 1)
    P = 16 + 16 + 256 + 16 + 16 + 1 + 5
    n_default = 8192
    fma_rhs = Nx * (16 + 256 + 16 + 4)
    flop_fwd = 2.0 * fma_rhs * (1 + 6 * n_steps)
    flop_adj = 2.0 * 3 * fma_rhs * (6 * n_steps)
    bytes_fwd = 4.0 * Nx * (1 + (n_steps // every + 1) + (n_steps + 1) + (6 * n_steps + 1))
    bytes_adj = 4.0 * Nx * ((n_steps + 1) + (n_steps // every + 1) + (6 * n_steps + 1) + 1)
    loss_weights = None

    @staticmethod
    def synthetic(n, seed=0):
        from helpers import glorot_theta
        rng = np.random.default_rng(seed)
        Nx = FKPP.Nx
        D0 = 0.01 * (Nx - 1) ** 2                       # D / dx^2 with the reference's D = 0.01 (Fisher-KPP-CNN.jl:16-25)
        theta = np.concatenate([glorot_theta(FKPP.widths, seed=3), [1.0, -2.0, 1.0, 0.0, D0]]).astype(np.float32)
        x = np.linspace(0, 1, Nx)
        d = rng.uniform(0.15, 0.5, n)[None, :]
        u0 = (0.5 * (np.tanh((x[:, None] - (0.5 - d / 2)) / (d / 10)) - np.tanh((x[:, None] - (0.5 + d / 2)) / (d / 10)))).astype(np.float32)
        y = np.repeat(u0[None], FKPP.n_steps // FKPP.every + 1, axis=0)
        return theta, u0, y

    @staticmethod
    def make_solver(ude, n, dev):
        layers = [ude.FastDense(1, 16, ude.tanh), ude.FastDense(16, 16, ude.tanh), ude.FastDense(16, 1)]
        return ude.UDESolver(ude.FisherKPPUDE(ude.FastChain(*layers), FKPP.Nx), 0.0, FKPP.dt, FKPP.n_steps, FKPP.every, max_trajectories=n, device=dev)

    @staticmethod
    def oracle_model(O):
        return O.fkpp_model(FKPP.Nx, FKPP.widths, ("tanh", "tanh", "identity")), np.ones(FKPP.Nx, np.float32)


CONFIGS = {"lv": LV, "seir": SEIR, "fkpp": FKPP}
HOST = None
DUMP_BYTES = 60_000_000     # data written by --dump-outputs: keeps the files, headers included, under 64 MB


def write_outputs(dirname, **arrays):
    """--dump-outputs: the host arrays as dirname/<name>.npy.  `out` (trajectories on the last axis) is cut to a fixed, seeded sample of
    trajectories when the files would pass DUMP_BYTES in all."""
    os.makedirs(dirname, exist_ok=True)
    out = arrays.get("out")
    room = DUMP_BYTES - sum(v.nbytes for k, v in arrays.items() if k != "out")
    if out is not None and out.nbytes > room:
        n = out.shape[-1]
        keep = np.sort(np.random.default_rng(0).choice(n, room // (out.nbytes // n), replace=False))
        arrays["out"] = np.ascontiguousarray(out[..., keep])
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), v)
    print(f"[bench] wrote {', '.join(f'{k}{list(v.shape)}' for k, v in arrays.items())} to {dirname}", file=sys.stderr)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        self.rows, self.stop = [], threading.Event()
        self.cmd = ["nvidia-smi", f"--id={index}",
                    "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                    "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                    "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits"]
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                o = subprocess.run(self.cmd, capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self.stop.wait(0.1)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_pass(cfg, theta, u0, y, threads):
    """One pass of the oracle port (C99/OpenMP, fp32, same algorithm) over the given trajectories; returns seconds."""
    from oracle import oracle as O
    m, w = cfg.oracle_model(O)
    t0 = time.perf_counter()
    O.ensemble_loss_grad(m, theta.astype(np.float32), u0, y, w, cfg.dt, cfg.n_steps, save_every=cfg.every, n_threads=threads, want_gu0=False)   # as the GPU arm's timed step: loss + grad_theta
    return time.perf_counter() - t0


def reference_arm(a, cfg):
    """The reference's own path (OrdinaryDiffEq.jl + SciMLSensitivity.jl) needs Julia, which this image does not have
    (BASELINE.md section 2): the CPU arm is the oracle port on the usable host cores."""
    cores, aff, quota = HOST
    n = a.n_per_gpu or cfg.n_default          # the SAME batch as the GPU arm's per-step workload (one GPU's share)
    if cfg is not LV and not a.n_per_gpu:
        n = min(n, 4096 if cfg is SEIR else 256)   # secondary configs: bounded sample (SEIR ~30x, FKPP ~1000x the LV cost per trajectory)
    theta, u0, y = cfg.synthetic(n)
    for _ in range(max(1, min(a.warmup, 2))):
        k = min(n, 1024)
        cpu_pass(cfg, theta, np.ascontiguousarray(u0[:, :k]), np.ascontiguousarray(y[:, :, :k]), cores)
    times = [cpu_pass(cfg, theta, u0, y, cores) for _ in range(a.steps)]
    med = float(np.median(times))
    value = n / med
    same = (cfg is LV and n == N_PER_GPU)
    print(json.dumps({
        "impl": "reference", "metric": cfg.metric, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": len(times),
        "warmup": a.warmup, "ms_per_step": 1e3 * med, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg.workload, "trajectories_per_step": n, "same_batch_as_gpu_arm": same,
                   "statistic": "median over the timed passes"},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} trajectories per step x {len(times)} steps (median), oracle C99/OpenMP fp32, {cores} threads "
                                   f"(affinity {aff}, cgroup quota {quota}), OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}",
                         "pass_seconds": [round(t, 4) for t in times]},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def kernel_names(run_step, torch):
    """Names of the kernels one step launches, observed with CUPTI (torch.profiler) on an untimed step."""
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            run_step()
            torch.cuda.synchronize()
        names = []
        for e in prof.events():
            if str(getattr(e, "device_type", "")).endswith("CUDA") and not e.name.startswith(("Memcpy", "Memset")):
                names.append(e.name)
        return names, "torch.profiler (CUPTI) on one untimed step"
    except Exception as ex:  # noqa: BLE001
        return None, f"profiler unavailable: {ex}"


def hjb_flops(d, hls, n_steps):
    """GEMM flops per path and iteration: forward (bias column included), data gradients (layers 2..4), weight + bias gradients (4 layers)."""
    mac_f = (d + 2) * hls + 2 * (hls + 1) * hls + (hls + 1) * d
    mac_d = 2 * hls * hls + hls * d
    return 2.0 * n_steps * (mac_f + mac_d + mac_f)


def main_hjb(a):
    """--config hjb (BASELINE config 5): highdim_pde/lambaem.jl's NNPDENS solve -- d = 100, hls = 110, 20 Euler-Maruyama steps, 10 000
    paths per GPU and iteration, fp64.  A step = one NNPDENS iteration (forward paths, loss, backward sweep, ADAM); metric = paths / s."""
    import math
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    d, hls, n_steps = 100, 110, 20
    m = a.n_per_gpu or 10000
    unit, metric = "paths/s", "NNPDENS paths per second (forward SDE + reverse sweep + ADAM), HJB d=100"
    workload = f"highdim_pde/lambaem.jl HJB d={d}, hls={hls}, {n_steps} EM steps, {m} paths per GPU and iteration, fp64"
    sys.path.insert(0, ROOT)
    if a.impl == "reference":
        if rank != 0:
            return
        from oracle import bsde_oracle as bo
        theta = bo.init_params(d, hls, 0)
        ms = min(m, 2000)
        bo.loss_and_grad(theta, d, hls, np.zeros(d), 1.0, n_steps, 200, 1)
        times = []
        for i in range(a.steps):
            t0 = time.perf_counter(); bo.loss_and_grad(theta, d, hls, np.zeros(d), 1.0, n_steps, ms, 1 + i); times.append(time.perf_counter() - t0)
        v = ms / float(np.median(times))
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": a.gpus, "steps": len(times), "warmup": 1,
                          "ms_per_step": 1e3 * float(np.median(times)), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
                          "data": "synthetic", "config": {"workload": workload, "paths_per_step": ms},
                          "cpu_baseline": {"value": v, "unit": unit, "cores": HOST[0], "kind": "port",
                                           "sample": f"{ms} paths per iteration (no ADAM update), oracle/bsde_oracle.py numpy fp64 (BLAS threads as the box gives)"},
                          "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    import torch
    import torch.distributed as dist
    import universal_differential_equations_b200 as ude
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    prob = ude.TerminalPDEProblem(ude.HJBTerminal(0.5, 0.5), ude.HJBNonlinearity(1.0), ude.ZeroDrift(), ude.ConstantDiffusion(math.sqrt(2.0)), np.zeros(d), (0.0, 1.0))
    u0 = ude.Chain(ude.Dense(d, hls, ude.relu), ude.Dense(hls, hls, ude.relu), ude.Dense(hls, 1))
    sg = ude.Chain(ude.Dense(d + 1, hls, ude.relu), ude.Dense(hls, hls, ude.relu), ude.Dense(hls, hls, ude.relu), ude.Dense(hls, d))
    alg = ude.NNPDENS(u0, sg, opt=ude.ADAM(0.03))
    s = ude.BSDESolver(prob, alg, n_steps, m, device=local, dtype=torch.float64)
    theta = ude.initial_params_pde(alg)
    s.set_params(theta)
    opt = ude.ADAM(0.03)
    clk = ClockSampler(local); clk.__enter__()
    g_all = torch.empty(s.P + 1, device=dev, dtype=torch.float64)

    def dist_step(i):
        # path shards: disjoint Philox path counters, mean over ALL paths; one all-reduce of [grad; loss]; identical ADAM update everywhere
        out = torch.empty(2, device=dev, dtype=torch.float64)
        torch.cuda.current_stream().synchronize()      # the handle works on its own stream: torch's queued work on g_all / out first
        ude._lib.check_bsde(s._h, s._L.b200ude_bsde_loss_gradient(s._h, m, 1 + i, rank * m, world * m, out.data_ptr(), g_all.data_ptr(), None))
        g_all[s.P] = out[0]
        dist.all_reduce(g_all)
        s.adam_step(opt, g_all[:s.P])

    if world == 1:
        s.train_adam(opt, m, max(a.warmup, 3), seed0=1)
        torch.cuda.synchronize()
        hist = s.train_adam(opt, m, a.steps, seed0=100)
        total_ms = s.last_train_ms()
        timing = "CUDA events on the handle's stream around the K iterations (1 direct launch + K-1 replays of one CUDA graph)"
    else:
        for i in range(max(a.warmup, 3)):
            dist_step(i)
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        for i in range(a.steps):
            dist_step(100 + i)
        torch.cuda.synchronize(); dist.barrier()
        t = torch.tensor([1e3 * (time.perf_counter() - t0)], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t)
        timing = "host clock around K synchronous iterations (each ends in a stream synchronize), max over ranks"
    value = world * m * a.steps / (total_ms * 1e-3)
    if a.dump_outputs and rank == 0:
        last = {"loss": hist[0][-1:], "u0": hist[1][-1:]} if world == 1 else {"grad_theta": g_all[:s.P], "loss": g_all[s.P:]}
        write_outputs(a.dump_outputs, theta=s.get_params(), **{k: v.cpu().numpy() for k, v in last.items()})

    # end to end through the host-buffer call a script makes per optimiser iteration: theta in from host, loss + gradient back to host
    th_h = np.ascontiguousarray(s.get_params())
    g_h, l_h, u_h = np.empty(s.P), np.empty(1), np.empty(1)
    e2e_steps = max(5, a.steps)
    for _ in range(2):
        s.set_params(th_h)
        ude._lib.check_bsde(s._h, s._L.b200ude_bsde_loss_gradient(s._h, m, 7, rank * m, world * m, l_h.ctypes.data, g_h.ctypes.data, u_h.ctypes.data))
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for i in range(e2e_steps):
        s.set_params(th_h)
        ude._lib.check_bsde(s._h, s._L.b200ude_bsde_loss_gradient(s._h, m, 7 + i, rank * m, world * m, l_h.ctypes.data, g_h.ctypes.data, u_h.ctypes.data))
        if world > 1:
            g_all[:s.P].copy_(torch.from_numpy(g_h)); dist.all_reduce(g_all); torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64); dist.all_reduce(t, op=dist.ReduceOp.MAX); e2e_s = float(t)
    names, names_src = (None, None)
    if rank == 0:
        names, names_src = kernel_names(lambda: s.loss_gradient(m, 3), torch)
    # roofline denominator: the library's own fp64 GEMM rate on this GPU, measured now (MEASURED_PEAKS.json has no fp64 entry)
    peak = None
    if rank == 0:
        A = torch.randn(4096, 4096, device=dev, dtype=torch.float64); B = torch.randn(4096, 4096, device=dev, dtype=torch.float64)
        for _ in range(2):
            A @ B
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); A @ B; e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        peak = 2 * 4096 ** 3 / (best * 1e-3) / 1e12
    t_probe = time.perf_counter()
    while rank == 0 and len(clk.rows) < 6 and time.perf_counter() - t_probe < 4.0:
        s.loss_gradient(m, 5)
    if world > 1:
        dist.barrier()
    clk.__exit__()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    fl = hjb_flops(d, hls, n_steps) * m
    ms_iter = total_ms / a.steps
    # dominant kernel: the fused forward sweep (csrc/bsde.cu::k_fused_forward2); its time from CUDA events on the handle's stream,
    # averaged over eager (non-graph) iterations of the same workload
    sweeps = []
    for i in range(5):
        s.loss_gradient(m, 50 + i)
        sweeps.append(s.last_sweep_ms())
    fwd_ms, bwd_ms, wg_ms = (float(np.mean([x[k] for x in sweeps])) for k in range(3))
    mac_f = (d + 2) * hls + 2 * (hls + 1) * hls + (hls + 1) * d          # [W | b] times the ones-augmented activations
    fwd_flops = 2.0 * n_steps * mac_f * m
    ach = fwd_flops / (fwd_ms * 1e-3) / 1e12
    dmma_peak = 36.5   # TFLOP/s, mma.sync.m8n8k4.f64 issue-rate microbenchmark on this GPU model (profiles/r02_dmma_microbench.txt)
    cpu = None
    if world == 1 and not a.no_cpu_baseline:
        from oracle import bsde_oracle as bo
        ms_ = min(m, a.cpu_sample or 1000)
        bo.loss_and_grad(theta, d, hls, np.zeros(d), 1.0, n_steps, 100, 1)
        tt = []
        for i in range(3):
            t0 = time.perf_counter(); bo.loss_and_grad(theta, d, hls, np.zeros(d), 1.0, n_steps, ms_, 1 + i); tt.append(time.perf_counter() - t0)
        cpu = {"value": ms_ / float(np.median(tt)), "unit": unit, "cores": HOST[0], "kind": "port",
               "sample": f"{ms_} of the {m} paths, median of 3 iterations, oracle/bsde_oracle.py (numpy fp64, BLAS threads)", "pass_seconds": [round(x, 4) for x in tt]}
    print(json.dumps({
        "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": ms_iter,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic (Brownian paths generated on the device, Philox4x32-10)",
        "config": {"workload": workload, "paths_per_gpu": m, "global_paths": world * m, "parallelism": f"path-sharded x{world}", "timing": timing,
                   "l2": "per-iteration working set (activations 2 x 3 x 110 x paths x 8 B + paths) exceeds L2 only above ~20 000 paths; no flush (state-carrying loop)",
                   "allreduce": "none (1 GPU)" if world == 1 else "NCCL all-reduce of [grad; loss] per iteration"},
        "e2e": {"value": world * m * e2e_steps / e2e_s, "unit": unit, "h2d_bytes_per_step": 8 * s.P, "d2h_bytes_per_step": 8 * (s.P + 2), "steps": e2e_steps,
                "note": "b200ude_bsde_set_params(host theta) + b200ude_bsde_loss_gradient(host loss / grad / u0), wall clock"},
        "gpu_launches": (sum(1 for k in names if "::k_" in k) if names else 0) * a.steps,
        "library_launches": (sum(1 for k in names if "::k_" not in k) if names else 0) * a.steps,
        "kernels_per_step": sorted(set(names)) if names else None, "kernels_source": names_src,
        "clocks": clk.summary(),
        "roofline": {"kernel": "k_fused_forward2 (fused DMMA forward sweep: 4 layers x 20 steps + Euler-Maruyama, two warps per 8-path tile, csrc/bsde.cu)", "bound": "tensor",
                     "achieved": ach, "peak": dmma_peak, "unit": "TFLOP/s", "frac": ach / dmma_peak, "traffic": None,
                     "peak_source": "fp64 tensor pipe: DMMA.8x8x4 issue-rate microbenchmark (tools/microbench/dmma.cu, profiles/r02_dmma_microbench.txt); "
                                    f"torch.matmul fp64 4096^3 in this run: {peak:.1f} TFLOP/s",
                     "algorithmic_flop_per_path_step": 2.0 * mac_f, "kernel_ms": fwd_ms,
                     "note": "share of the iteration: forward sweep / cotangent sweep / fused weight-gradient products in kernel_ms"},
        "kernel_ms": {"forward_sweep": fwd_ms, "cotangent_sweep": bwd_ms, "weight_gradient_products": wg_ms, "iteration": ms_iter},
        "iteration_gemm_tflops": fl / (ms_iter * 1e-3) / 1e12,
        "cpu_baseline": cpu,
    }))
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="lv", choices=sorted(CONFIGS) + ["hjb"])
    ap.add_argument("--n-per-gpu", type=int, default=0)
    ap.add_argument("--cpu-sample", type=int, default=0, help="trajectories in the in-line CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned to DIR/<name>.npy (GPU arm)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the GPU arm's results; the reference arm keeps none")
    global HOST
    if a.config == "hjb":
        HOST = host_cores()
        return main_hjb(a)
    cfg = CONFIGS[a.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))

    HOST = host_cores()   # before NCCL / CUDA initialisation can narrow the calling thread's affinity
    if a.impl == "reference":
        if rank == 0:
            reference_arm(a, cfg)
        return

    import torch
    import torch.distributed as dist
    import universal_differential_equations_b200 as ude

    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = a.n_per_gpu or cfg.n_default
    P, D = cfg.P, cfg.D
    n_save = cfg.n_steps // cfg.every + 1
    solver = cfg.make_solver(ude, n, dev)
    assert solver.P == P, (solver.P, P)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    # multi-GPU: the sum over ranks of [grad_theta; loss] runs inside the final reduction kernel over NVLink peer memory
    # (b200ude_adjoint_l2_allreduce); NCCL all-reduce only if the peer mapping cannot be set up on every rank
    peer = None
    if world > 1 and os.environ.get("B200UDE_PEER_ALLREDUCE", "1") != "0":
        ok = torch.ones(1, device=dev)
        try:
            peer = ude.PeerAllReduce(solver)
        except Exception as e:   # noqa: BLE001
            print(f"[bench] rank {rank}: peer-memory all-reduce unavailable ({e}); using NCCL", file=sys.stderr)
            ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok) == 0.0:
            if peer is not None:
                solver.peer_detach()
            peer = None

    class Shard:
        """One rank's share of an ensemble, resident in HBM."""

        def __init__(self, n_local, seed):
            self.n = n_local
            self.theta, self.u0, self.y = cfg.synthetic(n_local, seed=seed)
            self.th_d = torch.from_numpy(self.theta).to(dev)
            self.u0_d = torch.from_numpy(self.u0).to(dev)
            self.y_d = torch.from_numpy(self.y).to(dev)
            self.out_d = torch.empty((n_save, D, n_local), device=dev)
            self.buf = torch.zeros(P + 1, device=dev)          # [grad_theta ; loss] -- the one all-reduced message

    def step(sh, ev=None, collective=True):
        solver.set_params(sh.th_d)
        if ev:
            ev[0].record()
        solver.forward(sh.u0_d, out=sh.out_d)
        if ev:
            ev[1].record()
        if peer is not None and collective:
            solver.adjoint_l2_allreduce(sh.y_d, want_grad_u0=False, grad_theta=sh.buf[:P], loss=sh.buf[P:])
            if ev:
                ev[2].record()
        else:
            solver.adjoint_l2(sh.y_d, want_grad_u0=False, grad_theta=sh.buf[:P], loss=sh.buf[P:])
            if ev:
                ev[2].record()
            if collective:
                ude.allreduce_loss_grad(sh.buf)
        if ev:
            ev[3].record()

    def timed(sh):
        """W warm-up steps, then K steps timed with CUDA events on the launch stream; L2 flushed between iterations;
        barrier + synchronize on both sides; max over ranks."""
        for _ in range(a.warmup):
            step(sh)
        torch.cuda.synchronize()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(a.steps)]
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for i in range(a.steps):
            flush.zero_()                          # evict L2 between timed iterations (untimed)
            step(sh, evs[i])
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t_step = [e[0].elapsed_time(e[3]) for e in evs]
        total_ms = float(sum(t_step))
        if world > 1:
            t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            total_ms = float(t)
        return {"total_ms": total_ms, "fwd_ms": float(np.mean([e[0].elapsed_time(e[1]) for e in evs])),
                "adj_ms": float(np.mean([e[1].elapsed_time(e[2]) for e in evs])), "step_ms": float(np.mean(t_step))}

    clk = ClockSampler(local)
    clk.__enter__()                                  # samples run from the warm-up through the timed regions
    weak = Shard(n, seed=rank)                       # every rank owns a different shard of the (world * n) ensemble
    tw = timed(weak)
    value = world * n * a.steps / (tw["total_ms"] * 1e-3)
    if a.dump_outputs and rank == 0:                 # before the phases below reuse the shard's buffers
        write_outputs(a.dump_outputs, out=weak.out_d.cpu().numpy(), grad_theta=weak.buf[:P].cpu().numpy(), loss=weak.buf[P:].cpu().numpy())

    # ---- the metric's literal batch: 65 536 trajectories in total, sharded over the ranks (strong scaling) ----
    strong = None
    if cfg is LV and not a.no_strong:
        total = N_PER_GPU
        lo, hi = ude.shard_range(total, rank, world)
        if world == 1 and n == total:
            ts, ns = tw, n
        else:
            sh = Shard(hi - lo, seed=1000 + rank)
            ts, ns = timed(sh), hi - lo
            del sh
        strong = {"global_trajectories": total, "trajectories_per_gpu": ns, "value": total * a.steps / (ts["total_ms"] * 1e-3),
                  "unit": UNIT, "ms_per_step": ts["total_ms"] / a.steps, "scaling": "strong",
                  "kernel_ms": {"forward": ts["fwd_ms"], "adjoint_plus_reduce": ts["adj_ms"]},
                  "note": "BASELINE.json's literal batch: the 65 536 trajectories are sharded over the GPUs; same timing protocol as the headline value"}

    # ---- one-shot untimed check of the fused all-reduce against NCCL (the sums every rank must hold) ----
    allreduce_check = None
    if world > 1 and peer is not None:
        ref = torch.zeros(P + 1, device=dev)
        solver.set_params(weak.th_d)
        solver.forward(weak.u0_d, out=weak.out_d)
        solver.adjoint_l2(weak.y_d, want_grad_u0=False, grad_theta=ref[:P], loss=ref[P:])
        dist.all_reduce(ref, op=dist.ReduceOp.SUM)
        solver.adjoint_l2_allreduce(weak.y_d, want_grad_u0=False, grad_theta=weak.buf[:P], loss=weak.buf[P:])
        torch.cuda.synchronize()
        err = ((weak.buf - ref).abs().max() / ref.abs().max()).reshape(1)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        same = weak.buf.clone()
        dist.broadcast(same, src=0)
        ident = torch.tensor([1.0 if torch.equal(same, weak.buf) else 0.0], device=dev)
        dist.all_reduce(ident, op=dist.ReduceOp.MIN)
        allreduce_check = {"max_abs_diff_vs_nccl_rel": float(err), "bitwise_identical_on_all_ranks": bool(float(ident) == 1.0),
                           "entries": P + 1}

    # the timed region of the default run is shorter than nvidia-smi's sampling period: keep the same step running
    # (untimed) until the sampler has seen the GPU under this load a few times
    t_probe = time.perf_counter()
    while rank == 0 and len(clk.rows) < 6 and time.perf_counter() - t_probe < 4.0:
        step(weak, collective=False)           # rank-local: no collective outside the lock-stepped region
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clk.__exit__()
    clocks = clk.summary() if rank == 0 else None
    if clocks:
        clocks["window"] = "warm-up + timed steps + post-run probe of the same step (untimed)"

    # kernels of one step, observed (rank 0, untimed, no collective)
    names, names_src = (None, None)
    if rank == 0:
        names, names_src = kernel_names(lambda: step(weak, collective=False), torch)

    # ---- end-to-end through the host-buffer C-ABI call: pinned host inputs, H2D + kernels + D2H every step ----
    th_h = torch.from_numpy(weak.theta).pin_memory()
    u0_h = torch.from_numpy(weak.u0).pin_memory()
    y_h = torch.from_numpy(weak.y).pin_memory()
    g_h = torch.empty(P).pin_memory()
    for _ in range(4):
        solver.loss_gradient_host(th_h, u0_h, y_h, grad_theta=g_h)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_steps = max(5, a.steps)
    for _ in range(e2e_steps):
        l_h, _, _ = solver.loss_gradient_host(th_h, u0_h, y_h, grad_theta=g_h)
        if world > 1:
            weak.buf[:P].copy_(g_h, non_blocking=True)
            weak.buf[P] = l_h
            ude.allreduce_loss_grad(weak.buf)
            torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t)
    e2e_value = world * n * e2e_steps / e2e_s
    h2d = 4 * (P + weak.u0.size + weak.y.size)
    d2h = 4 * (P + 1)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    adj_ms, fwd_ms = tw["adj_ms"], tw["fwd_ms"]
    adj_name = next((k for k in (names or []) if "adjoint" in k), "adjoint kernel")
    fwd_name = next((k for k in (names or []) if "forward" in k), "forward kernel")
    traffic, traffic_src = None, "no ncu capture of this kernel committed for this round"
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from this round's ncu --set full capture
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")))
        ent = tj.get(cfg.name, {})
        if ent and ent.get("trajectories"):
            traffic = float(ent["dram_bytes"]) * (n / float(ent["trajectories"]))
            traffic_src = ent.get("source", "profiles/r02_ncu_traffic.json")
    except Exception:
        pass
    roofline = {
        "kernel": f"{adj_name} (+ the ~5 us fixed-order reduce; events bracket both)",
        "bound": "hbm", "achieved": n * cfg.bytes_adj / (adj_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
        "frac": n * cfg.bytes_adj / (adj_ms * 1e-3) / 1e9 / hbm_peak,
        "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6.65 TB/s (B200_PROFILING.md)",
        "algorithmic_bytes_per_trajectory": cfg.bytes_adj, "traffic": traffic, "traffic_source": traffic_src,
        "note": "the path is compute-bound by construction (SURVEY.md 8d, ~430 FLOP/B for config 2): roofline_pipes grades the kernels against the pipes they actually use",
    }
    sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
    line_extra = {}
    if cfg is LV:
        wm = any("wm::" in k for k in (names or []))
        # per-trajectory pipe work of the kernels that ran (DESIGN.md section 4.6): MUFU lane-ops, legacy tensor-pipe (HMMA) warp
        # instructions, FMA-pipe cycles and issue slots (static SASS counts of the stage loop bodies, cuobjdump), HBM bytes
        ev_f, ev_a = 1 + 6 * cfg.n_steps, 6 * cfg.n_steps
        mufu = 80.0 if wm else 128.0                       # per chain evaluation: 64 tanh x 1.25 (batched inversion) / x 2
        fam = {   # per trajectory and stage evaluation: (forward, adjoint)
            "hmma": (24.0 / 16.0, 96.0 / 16.0) if wm else (0.0, 96.0 / 32.0),          # warp-level mma.sync instructions
            "fma_cyc": (279.0 / 16.0, 500.0 / 16.0) if wm else (600.0 / 32.0, 1700.0 / 32.0),   # FMA-pipe cycles (FFMA2 = 2), per scheduler
            "issue": (500.0 / 16.0, 950.0 / 16.0) if wm else (887.0 / 32.0, 2268.0 / 32.0),     # warp instructions issued
        }
        clk_hz = sm_clock * 1e6

        def pipes(ms, evals, which, nbytes):
            t = ms * 1e-3
            b = {"mufu": n * evals * mufu / (148 * MUFU_PER_CLK_SM * clk_hz),
                 "tensor_mma_sync": n * evals * fam["hmma"][which] / (148 * HMMA_PER_CLK_SM * clk_hz),
                 "fma_pipe": n * evals * fam["fma_cyc"][which] / (148 * 4 * clk_hz),
                 "issue_slots": n * evals * fam["issue"][which] / (148 * 4 * clk_hz),
                 "hbm": n * nbytes / (hbm_peak * 1e9)}
            tmin = max(b.values())
            return {"ms": ms, "t_min_ms": 1e3 * tmin, "binding_pipe": max(b, key=b.get), "frac": tmin / t,
                    "pipe_ms": {k: 1e3 * v for k, v in b.items()}}
        line_extra["roofline_pipes"] = {
            "forward": pipes(fwd_ms, ev_f, 0, cfg.bytes_fwd), "adjoint": pipes(adj_ms, ev_a, 1, cfg.bytes_adj),
            "kernel_family": "warp-collective mma.sync (lv32_wm.cuh)" if wm else "tcgen05 (lv32_tc.cuh)",
            "peaks": {"mufu_lanes_per_clk_sm": MUFU_PER_CLK_SM, "mma_sync_warp_instr_per_clk_sm": HMMA_PER_CLK_SM, "issue_slots_per_clk_sm": 4, "fma_pipe_cycles_per_clk_sm": 4,
                      "hbm_gbs": hbm_peak, "sm_mhz": sm_clock},
            "peak_source": "tools/microbench (profiles/r01_pipes_microbench.txt, r01_mma_sync_microbench.txt), MEASURED_PEAKS.json",
            "note": "t_min = max over pipes of (work / measured pipe peak); frac = t_min / measured time; the tcgen05 pipe of the tensor-core family is far from binding and not listed",
        }
    line_extra["roofline_fp32"] = {
        "step_achieved_tflops": n * (cfg.flop_fwd + cfg.flop_adj) / (tw["step_ms"] * 1e-3) / 1e12, "peak": FP32_PEAK_TFLOPS,
        "note": "algorithmic FLOP rate for context only: most of these FLOPs run on tensor cores, so this is not a roofline fraction",
        "flop_per_trajectory": cfg.flop_fwd + cfg.flop_adj,
    }
    cpu = None
    if not a.no_cpu_baseline and world == 1:   # the in-line CPU leg is an N = 1 item (rank 0 of a multi-rank run has been re-pinned by NCCL)
        cores, aff, quota = HOST
        sample = min(a.cpu_sample or (8192 if cfg is LV else 512 if cfg is SEIR else 32), n)
        u0s, ys = np.ascontiguousarray(weak.u0[:, :sample]), np.ascontiguousarray(weak.y[:, :, :sample])
        k = min(sample, 256)
        cpu_pass(cfg, weak.theta, np.ascontiguousarray(u0s[:, :k]), np.ascontiguousarray(ys[:, :, :k]), cores)   # warm
        times = [cpu_pass(cfg, weak.theta, u0s, ys, cores) for _ in range(3)]
        med = float(np.median(times))
        cpu = {"value": sample / med, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{sample} of the {n} trajectories, median of 3 passes, oracle C99/OpenMP fp32 with {cores} threads "
                         f"(affinity {aff}, cgroup quota {quota})", "pass_seconds": [round(t, 4) for t in times]}
    line = {
        "metric": cfg.metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": tw["total_ms"] / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": cfg.workload, "trajectories_per_gpu": n, "global_trajectories": world * n, "parallelism": f"ensemble-sharded x{world}",
                   "l2": "flushed between timed iterations (256 MiB memset, untimed)",
                   "timing": "CUDA events per step on the launch stream, summed over steps, max over ranks",
                   "allreduce": ("none (1 GPU)" if world == 1 else
                                 "fused into the final reduction kernel over NVLink peer memory (CUDA IPC, b200ude_adjoint_l2_allreduce)" if peer is not None
                                 else "NCCL all-reduce of [grad_theta; loss]")},
        "strong": strong,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "note": "b200ude_loss_gradient_host: pinned host theta/u0/data -> H2D -> kernels -> D2H grad+loss, wall clock"},
        "gpu_launches": (len(names) if names else 3) * a.steps,
        "kernels_per_step": names, "kernels_source": names_src,
        "allreduce_check": allreduce_check,
        "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
        "kernel_ms": {"forward": fwd_ms, "adjoint_plus_reduce": adj_ms, "step": tw["step_ms"]},
    }
    line.update(line_extra)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
