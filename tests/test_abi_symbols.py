"""The C-ABI library loads here (no GPU) and exports exactly what include/b200ude.h declares;
create() fails loudly -- never silently falls back -- when no sm_100 device is present."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def libpath():
    from universal_differential_equations_b200 import _lib
    if not os.path.exists(_lib.SO_PATH):
        _lib.build()
    return _lib.SO_PATH


def _declared_functions():
    hdr = open(os.path.join(ROOT, "include", "b200ude.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    return sorted(set(re.findall(r"\b(b200ude_[a-z0-9_]+)\s*\(", hdr)))


def test_header_declares_expected_entry_points():
    from universal_differential_equations_b200 import _lib
    assert _declared_functions() == sorted(_lib.EXPORTS)


def test_library_exports_every_declared_symbol(libpath):
    L = C.CDLL(libpath)
    for name in _declared_functions():
        assert hasattr(L, name), name
    L.b200ude_version.restype = C.c_int32
    assert L.b200ude_version() == 1


def test_desc_struct_layout_matches_header(libpath):
    """struct_size is checked by create(): a wrong ctypes mirror is rejected with EINVAL, not UB."""
    from universal_differential_equations_b200 import _lib
    L = _lib.lib()
    d = _lib.Desc()
    d.struct_size = C.sizeof(_lib.Desc) + 8
    h = C.c_void_p()
    assert L.b200ude_create(C.byref(d), C.byref(h)) == _lib.EINVAL
    assert b"struct_size" in L.b200ude_last_error(None)


_CREATE_VALID_DESC = """
import ctypes as C
from universal_differential_equations_b200 import _lib
L = _lib.lib()
d = _lib.Desc()
d.struct_size = C.sizeof(_lib.Desc)
d.dtype, d.model, d.state_dim, d.n_layers = _lib.F32, _lib.MODEL_LV, 2, 3
for i, w in enumerate((2, 32, 32, 2)):
    d.widths[i] = w
d.acts[0] = d.acts[1] = _lib.ACT_TANH
d.n_consts = 2
d.consts[0], d.consts[1] = 1.3, 1.8
d.dt, d.n_steps, d.save_every, d.max_trajectories = 0.1, 30, 1, 16
h = C.c_void_p()
rc = L.b200ude_create(C.byref(d), C.byref(h))
print(rc, bool(h.value))
d.widths[1] = 65   # wider than any kernel family supports
print(L.b200ude_create(C.byref(d), C.byref(h)))
d.widths[1] = 32
d.dt = 0.0
print(L.b200ude_create(C.byref(d), C.byref(h)))
"""


def test_no_silent_cpu_fallback(libpath):
    """Without a CUDA device create() must fail with ENODEVICE (after validating the descriptor).  The call runs in a process
    that sees no device, so this holds on a GPU machine too (the GPU tests cover the success path)."""
    import subprocess
    import sys
    from universal_differential_equations_b200 import _lib
    r = subprocess.run([sys.executable, "-c", _CREATE_VALID_DESC], cwd=ROOT, capture_output=True, text=True,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert r.returncode == 0, r.stderr[-2000:]
    rc, handle, rc_wide, rc_dt = r.stdout.split()
    assert int(rc) == _lib.ENODEVICE and handle == "False"
    assert int(rc_wide) == _lib.EUNSUPPORTED     # an unsupported chain shape is reported as such even before the device is probed
    assert int(rc_dt) == _lib.EINVAL             # usage errors


def test_product_package_never_touches_the_oracle():
    pkg = os.path.join(ROOT, "universal_differential_equations_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", "Makefile")):
                txt = open(os.path.join(dirpath, f), errors="ignore").read()
                assert "ude_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f


def test_ctypes_mirrors_have_the_sizes_the_c_compiler_gives_the_header(tmp_path):
    """sizeof / offsetof of b200ude_desc and b200ude_adam as gcc lays them out == the ctypes mirrors in _lib.py
    (a drifted mirror would otherwise only show up as EINVAL from create() on a GPU box)."""
    import subprocess
    from universal_differential_equations_b200 import _lib
    src = tmp_path / "sz.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "b200ude.h"\n'
        'int main(void) { printf("%zu %zu %zu %zu %zu %zu %zu\\n", sizeof(b200ude_desc), offsetof(b200ude_desc, consts), '
        'offsetof(b200ude_desc, loss_weights), offsetof(b200ude_desc, max_trajectories), offsetof(b200ude_desc, max_steps), '
        'sizeof(b200ude_adam), offsetof(b200ude_adam, l2_reg)); return 0; }\n')
    exe = tmp_path / "sz"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    D, A = _lib.Desc, _lib.Adam
    want = [C.sizeof(D), D.consts.offset, D.loss_weights.offset, D.max_trajectories.offset, D.max_steps.offset, C.sizeof(A), A.l2_reg.offset]
    assert got == want, (got, want)


def test_bsde_desc_layout_and_no_cpu_fallback(libpath):
    """Terminal-PDE path: a wrong ctypes mirror of b200ude_bsde_desc is rejected (EINVAL), bad arguments are usage errors, and without a
    CUDA device create fails with ENODEVICE after validating the descriptor -- there is no CPU path behind b200ude_bsde_*."""
    import torch
    from universal_differential_equations_b200 import _lib
    L = _lib.lib()
    x0 = (C.c_double * 4)(0.0, 0.0, 0.0, 0.0)
    d = _lib.BsdeDesc(struct_size=C.sizeof(_lib.BsdeDesc) + 8, device=0, dtype=_lib.F64, dim=4, hidden=8, n_steps=5, T=1.0, lam=1.0, sigma=1.4,
                      g_a=0.5, g_b=0.5, x0=x0, max_paths=16)
    h = C.c_void_p()
    assert L.b200ude_bsde_create(C.byref(d), C.byref(h)) == _lib.EINVAL and b"struct_size" in L.b200ude_bsde_last_error(None)
    d.struct_size = C.sizeof(_lib.BsdeDesc)
    d.n_steps = 0
    assert L.b200ude_bsde_create(C.byref(d), C.byref(h)) == _lib.EINVAL
    d.n_steps = 5
    if not torch.cuda.is_available():
        assert L.b200ude_bsde_create(C.byref(d), C.byref(h)) == _lib.ENODEVICE and not h.value
    assert L.b200ude_bsde_num_params(None) == 0
    assert L.b200ude_bsde_set_params(None, None, 0, _lib.HOST) == _lib.EINVAL
