"""universal_differential_equations_b200/jld2.py (reader + writer of plain numeric JLD2 datasets) against the reference's own result files (LotkaVolterra/results/*.jld2, written by
scenario_1.jl:210-213 ... hudson_bay.jl:231-235): the arrays it decodes by walking the HDF5 structure equal the committed golden vectors
(which tools/make_golden.py cut out at fixed byte offsets).  The result files come from tests/golden/jld2_results.npz (tools/make_golden_jld2.py):
each at its full length with every byte the reader visits as the reference wrote it and the bytes it never visits zeroed."""
import os

import numpy as np
import pytest

FILES = {"hudson_bay": "Hudson_Bay_recovery.jld2", "scenario_1": "Scenario_1_recovery_0.005.jld2",
         "scenario_2": "Scenario_2_recovery_0.005.jld2", "scenario_3": "Scenario_3_recovery_0.005.jld2"}


@pytest.fixture(scope="module")
def results_dir(tmp_path_factory):
    """A directory holding the reference's result files, written out from the committed fixture."""
    d = tmp_path_factory.mktemp("results")
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "jld2_results.npz"))
    for key, fn in FILES.items():
        (d / fn).write_bytes(z[key].tobytes())
    return str(d)


def test_save_load_round_trip(tmp_path):
    """Writer -> reader on arrays of both float types, both layouts (compact below 8 KiB, contiguous above), with valid checksums."""
    from universal_differential_equations_b200 import jld2
    rng = np.random.default_rng(0)
    arrays = {"X": rng.standard_normal((2, 31)), "t": np.linspace(0, 3, 31, dtype=np.float32), "losses": rng.random(3000),
              "big32": rng.standard_normal((7, 500)).astype(np.float32), "scalar_like": np.array([1.5])}
    path = str(tmp_path / "out.jld2")
    jld2.save(path, **arrays)
    f = jld2.JLD2File(path)
    assert f.superblock_ok and f.keys() == list(arrays)
    for k, a in arrays.items():
        assert f.header_bytes(k)[1], k
        got = f.read(k)
        assert got.dtype == a.dtype and got.shape == a.shape
        np.testing.assert_array_equal(got, a)
    assert jld2.load(path, "t")["t"].dtype == np.float32
    with pytest.raises(TypeError):
        jld2.save(path, n=np.arange(3))
    assert jld2.lookup3(b"") == 0xDEADBEEF and jld2.lookup3(b"Four score and seven years ago") == 0x17770551   # lookup3.c's own self-test values


def test_writer_reproduces_the_reference_files_own_bytes(tmp_path, results_dir):
    """The dataset object headers `save` emits for the reference's X / t arrays are byte-for-byte those JLD2 itself wrote
    (Hudson_Bay_recovery.jld2: compact layout), at the same addresses; for a contiguous dataset (scenario 1's loss history) everything but
    the data address agrees and the data follows the header as it does there.  The reference files' own checksums validate."""
    from universal_differential_equations_b200 import jld2
    ref = jld2.JLD2File(os.path.join(results_dir, "Hudson_Bay_recovery.jld2"))
    assert ref.superblock_ok and all(ref.header_bytes(k)[1] for k in ref.keys())
    path = str(tmp_path / "hb.jld2")
    jld2.save(path, julia_version="1.6.1", X=ref.read("X"), t=ref.read("t"))
    mine = jld2.JLD2File(path)
    for k in ("X", "t"):
        assert mine.links[k] == ref.links[k] and mine.header_bytes(k)[0] == ref.header_bytes(k)[0], k
    assert open(path, "rb").read()[:512] == ref.blob[:512]                       # the text header
    s1 = jld2.JLD2File(os.path.join(results_dir, "Scenario_1_recovery_0.005.jld2"))
    jld2.save(path, losses=s1.read("losses"))
    mine = jld2.JLD2File(path)
    a, b = mine.header_bytes("losses")[0], s1.header_bytes("losses")[0]
    assert len(a) == len(b) and a[:-20] == b[:-20] and a[-12:-4] == b[-12:-4]      # all but the 8-byte data address and the checksum
    np.testing.assert_array_equal(mine.read("losses"), s1.read("losses"))


def test_reader_reproduces_the_golden_vectors(golden, results_dir):
    from universal_differential_equations_b200 import jld2
    cases = {
        "scenario_1": ("Scenario_1_recovery_0.005.jld2", {"X": "X", "losses": "losses"}),
        "scenario_2": ("Scenario_2_recovery_0.005.jld2", {"X": "X", "t": "t", "losses": "losses"}),
        "scenario_3": ("Scenario_3_recovery_0.005.jld2", {"X": "X", "losses": "losses"}),
        "hudson_bay": ("Hudson_Bay_recovery.jld2", {"X": "X", "t": "t", "losses": "losses", "theta_init": "initial_parameters",
                                                    "theta_trained": "trained_parameters"}),
    }
    for name, (fn, keys) in cases.items():
        got = jld2.load(os.path.join(results_dir, fn), *keys.values())
        for gk, fk in keys.items():
            want = golden[name][gk]
            assert got[fk].dtype == want.dtype and got[fk].shape == want.shape, (name, gk, got[fk].shape, want.shape)
            np.testing.assert_array_equal(got[fk], want, err_msg=f"{name}:{gk}")


def test_reader_lists_structs_without_decoding_them(results_dir):
    from universal_differential_equations_b200 import jld2
    f = jld2.JLD2File(os.path.join(results_dir, "Scenario_1_recovery_0.005.jld2"))
    assert {"solution", "X", "t", "losses", "trained_parameters", "long_estimate"} <= set(f.keys())
    assert f.is_numeric("losses") and not f.is_numeric("solution")
    with pytest.raises(TypeError):
        f.read("solution")
    with pytest.raises(KeyError):
        f.read("nope")
    assert set(jld2.load(os.path.join(results_dir, "Hudson_Bay_recovery.jld2"))) >= {"X", "t", "losses", "model_parameter"}


def test_parameter_containers_are_followed_to_their_arrays(golden, results_dir):
    """`trained_parameters` (a ComponentVector) and `initial_parameters` (Lux's NamedTuple of layers) are Julia structs whose array fields
    are references to other objects of the file: read_tree follows them and returns the very arrays the golden vectors hold."""
    from universal_differential_equations_b200 import jld2
    f = jld2.JLD2File(os.path.join(results_dir, "Scenario_1_recovery_0.005.jld2"))
    (theta,) = f.read_tree("trained_parameters")
    np.testing.assert_array_equal(theta, golden["scenario_1"]["theta_trained"])
    layers = f.read_tree("initial_parameters")
    assert [a.shape for a in layers] == [(5, 2), (5, 1), (5, 5), (5, 1), (5, 5), (5, 1), (2, 5), (2, 1)]
    for k, w in zip(("W1_init", "W2_init", "W3_init", "W4_init"), layers[0::2]):
        np.testing.assert_array_equal(w, golden["scenario_1"][k])
    assert all(not b.any() for b in layers[1::2])                                  # Lux's zero biases
    f2 = jld2.JLD2File(os.path.join(results_dir, "Scenario_2_recovery_0.005.jld2"))
    np.testing.assert_array_equal(f2.read_tree("trained_parameters")[0], golden["scenario_2"]["theta_trained"])
    np.testing.assert_array_equal(f2.read_tree("initial_parameters")[0], golden["scenario_2"]["theta_init"])
    f3 = jld2.JLD2File(os.path.join(results_dir, "Scenario_3_recovery_0.005.jld2"))
    np.testing.assert_array_equal(f3.read_tree("trained_parameters")[0], golden["scenario_3"]["theta_trained"])
