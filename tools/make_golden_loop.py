"""Writes the fixtures of the batched-training known-answer tests (KAT-12) from the reference's
LotkaVolterra/results/Scenario_1_recovery_loop.jld2: one JLD2 group per run of run_loops.jl:55-62 ("1" ... "500"; runs the script's
try/catch skipped are absent), each holding X, t, initial_parameters, trained_parameters and losses (loop_recoveries.jl:145-152).

  tests/golden/scenario_1_loop.npz       run ids, X [R,2,31], t [31], theta_init / theta_trained [R,87], losses_head [R,16],
                                          losses_last [R], n_losses [R]  (float32, as the file stores them)
  tests/golden/scenario_1_loop_jld2.npz  `blob`: the file itself at full length with only the bytes the group walker visits for the root and a
                                          few groups kept (the rest zeroed, compressed), in the manner of tools/make_golden_jld2.py

The source file is guarded by its SHA-256.
    python tools/make_golden_loop.py --ref <checkout of the reference>"""
import argparse
import hashlib
import os
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
from universal_differential_equations_b200 import jld2  # noqa: E402
from make_golden_jld2 import header_ranges, object_ranges  # noqa: E402

REL = "LotkaVolterra/results/Scenario_1_recovery_loop.jld2"
SHA256 = "b0e287118aeefd850bf81c3fcf1cb87f00e631c95a076f3263dee8e9409cf285"
KEEP_GROUPS = ("1", "2", "17", "250", "500")     # groups the trimmed copy keeps readable
DATASETS = ("X", "t", "losses", "initial_parameters", "trained_parameters")
N_HEAD = 16


def extract(f):
    runs = sorted((k for k in f.keys() if k.isdigit()), key=int)
    X, th0, th1, head, last, n = [], [], [], [], [], []
    t = f.read(f"{runs[0]}/t")
    for r in runs:
        X.append(f.read(f"{r}/X"))
        (a,) = f.read_tree(f"{r}/initial_parameters")
        (b,) = f.read_tree(f"{r}/trained_parameters")
        th0.append(a)
        th1.append(b)
        losses = f.read(f"{r}/losses")
        head.append(losses[:N_HEAD])
        last.append(losses[-1])
        n.append(len(losses))
        assert np.array_equal(f.read(f"{r}/t"), t), r
    return dict(runs=np.array([int(r) for r in runs], np.int32), X=np.stack(X), t=t, theta_init=np.stack(th0),
                theta_trained=np.stack(th1), losses_head=np.stack(head), losses_last=np.array(last, np.float32),
                n_losses=np.array(n, np.int32))


def shrink(f, groups):
    sb = f.blob.find(jld2._SIG)
    keep = [(0, sb + 48)] + header_ranges(f, struct.unpack_from("<Q", f.blob, sb + 36)[0])
    for g in groups:
        keep += header_ranges(f, f._addr(g))
        for k in DATASETS:
            keep += object_ranges(f, f._addr(f"{g}/{k}"), k.endswith("_parameters"))
    out = bytearray(len(f.blob))
    for lo, hi in keep:
        out[lo:hi] = f.blob[lo:hi]
    return bytes(out)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref", required=True, help="checkout of ChrisRackauckas/universal_differential_equations")
    ap.add_argument("--out", default=os.path.join(ROOT, "tests", "golden"))
    a = ap.parse_args()
    path = os.path.join(a.ref, REL)
    blob = open(path, "rb").read()
    sha = hashlib.sha256(blob).hexdigest()
    if sha != SHA256:
        raise SystemExit(f"{REL}: sha256 {sha} != expected {SHA256}")
    f = jld2.JLD2File(path)
    arrays = extract(f)
    source = np.array(f"{REL} sha256={sha}")
    np.savez_compressed(os.path.join(a.out, "scenario_1_loop.npz"), _source=source, **arrays)
    small = shrink(f, KEEP_GROUPS)
    np.savez_compressed(os.path.join(a.out, "scenario_1_loop_jld2.npz"), blob=np.frombuffer(small, np.uint8), groups=np.array(KEEP_GROUPS),
                        _source=source)
    print(f"{len(arrays['runs'])} runs; losses per run {arrays['n_losses'].min()} .. {arrays['n_losses'].max()}")
    for fn in ("scenario_1_loop.npz", "scenario_1_loop_jld2.npz"):
        print("wrote", fn, os.path.getsize(os.path.join(a.out, fn)), "bytes")
