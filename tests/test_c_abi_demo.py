"""The boundary used from plain C99 (examples/c_abi_demo.c): the header compiles as strict C, the library links from C
with nothing but libcudart behind it, fails loudly without a device, and on a GPU reproduces the oracle."""
import os
import struct
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "universal_differential_equations_b200", "csrc")
NO_DEVICE = dict(os.environ, CUDA_VISIBLE_DEVICES="")     # the demo sees no device, on a GPU machine too


def _build(tmp_path):
    from universal_differential_equations_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    obj, exe = str(tmp_path / "demo.o"), str(tmp_path / "demo")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           "-c", os.path.join(ROOT, "examples", "c_abi_demo.c"), "-o", obj])
    subprocess.check_call(["gcc", "-o", exe, obj, "-L", CSRC, "-lb200ude", f"-Wl,-rpath,{CSRC}"])
    return exe


def _build_bsde(tmp_path):
    from universal_differential_equations_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    obj, exe = str(tmp_path / "bsde_demo.o"), str(tmp_path / "bsde_demo")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-I", os.path.join(ROOT, "include"),
                           "-c", os.path.join(ROOT, "examples", "c_abi_bsde_demo.c"), "-o", obj])
    subprocess.check_call(["gcc", "-o", exe, obj, "-L", CSRC, "-lb200ude", f"-Wl,-rpath,{CSRC}"])
    return exe


def _write_bsde_inputs(path):
    g = np.load(os.path.join(ROOT, "tests", "golden", "hjb_small.npz"))
    with open(path, "wb") as f:
        f.write(struct.pack("iiiiQ", int(g["d"]), int(g["hls"]), int(g["N"]), int(g["M"]), int(g["seed"])))
        f.write(np.asarray(g["x0"], np.float64).tobytes()); f.write(np.asarray(g["theta"], np.float64).tobytes())
    return g


def test_c_bsde_demo_compiles_links_and_fails_loudly_without_a_device(tmp_path):
    exe = _build_bsde(tmp_path)
    _write_bsde_inputs(str(tmp_path / "in.bin"))
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, env=NO_DEVICE)
    assert r.returncode == 1 and "b200ude_bsde_create failed (-5)" in r.stderr and not os.path.exists(tmp_path / "out.bin")


@pytest.mark.gpu
def test_c_bsde_demo_matches_the_frozen_vectors_on_the_gpu(tmp_path):
    """C99 -> libb200ude.so -> GPU against tests/golden/hjb_small.npz (no Python, torch or oracle in the loop)."""
    exe = _build_bsde(tmp_path)
    g = _write_bsde_inputs(str(tmp_path / "in.bin"))
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = np.frombuffer(open(tmp_path / "out.bin", "rb").read(), np.float64)
    P = g["theta"].size
    loss, u0, grad, after = raw[0], raw[1], raw[2:2 + P], raw[2 + P:]
    assert abs(loss - float(g["loss"])) <= 1e-10 * abs(loss) and abs(u0 - float(g["u0"])) <= 1e-10
    assert np.linalg.norm(grad - g["grad"]) <= 1e-9 * np.linalg.norm(g["grad"])
    assert np.isfinite(after).all() and after[0] != loss and len(set(after)) == 3     # three ADAM iterations moved the parameters


def _write_inputs(path, N, n_steps=30, dt=0.1):
    from helpers import glorot_theta, synthetic_ensemble
    theta = glorot_theta((2, 32, 32, 2), seed=1)
    u0, y = synthetic_ensemble(N, n_steps=n_steps, dt=dt)
    with open(path, "wb") as f:
        f.write(struct.pack("iif", N, n_steps, dt))
        f.write(theta.tobytes()); f.write(u0.tobytes()); f.write(y.tobytes())
    return theta, u0, y


def test_c_demo_compiles_links_and_fails_loudly_without_a_device(tmp_path):
    exe = _build(tmp_path)
    _write_inputs(str(tmp_path / "in.bin"), 4)
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True, env=NO_DEVICE)
    assert r.returncode == 1 and "b200ude_create failed (-5)" in r.stderr and not os.path.exists(tmp_path / "out.bin")


@pytest.mark.gpu
def test_c_demo_matches_oracle_on_the_gpu(tmp_path, O):
    N = 333
    exe = _build(tmp_path)
    theta, u0, y = _write_inputs(str(tmp_path / "in.bin"), N)
    r = subprocess.run([exe, str(tmp_path / "in.bin"), str(tmp_path / "out.bin")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    raw = open(tmp_path / "out.bin", "rb").read()
    loss = struct.unpack_from("d", raw, 0)[0]
    off = 8
    g = np.frombuffer(raw, np.float32, 1218, off); off += 4 * 1218
    gu = np.frombuffer(raw, np.float32, 2 * N, off).reshape(2, N); off += 8 * N
    out = np.frombuffer(raw, np.float32, 31 * 2 * N, off).reshape(31, 2, N); off += 4 * 31 * 2 * N
    status = np.frombuffer(raw, np.int32, N, off); off += 4 * N
    same = struct.unpack_from("i", raw, off)[0]
    m = O.lv_model()
    l64, g64, gu64, out64 = O.ensemble_loss_grad(m, theta.astype(np.float64), u0, y, np.ones(2), 0.1, 30, want_out=True)
    assert same == 1 and (status == 0).all()
    assert np.all(np.abs(out - out64) <= 3e-4 * (1 + np.abs(out64)))
    assert abs(loss - l64) <= 1e-4 * abs(l64)
    assert np.linalg.norm(g - g64) <= 2e-3 * np.linalg.norm(g64)
    assert np.abs(gu - gu64).max() <= 2e-3 * np.abs(gu64).max()
