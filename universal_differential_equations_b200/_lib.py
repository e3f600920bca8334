"""ctypes binding of the C-ABI library (include/b200ude.h -> csrc/libb200ude.so).

This is the only place Python touches the product's native code.  There is no
CPU fallback: if the shared library is missing, or there is no sm_100 device,
the calls raise.  Nothing here imports the CPU oracle.
"""
import ctypes as C
import os
import shutil
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(CSRC, "libb200ude.so")

# ---- constants mirrored from include/b200ude.h -------------------------------
ABI_VERSION = 1
F32, F64 = 0, 1
MODEL_LV, MODEL_SEIR, MODEL_FKPP, MODEL_NODE, MODEL_SEIR_NODE = 0, 1, 2, 3, 4
ACT_IDENTITY, ACT_TANH, ACT_RBF = 0, 1, 2
TSIT5, VERN7, RKC2 = 0, 1, 2
INTERPOLATING_ADJOINT, DISCRETE_ADJOINT = 0, 1
HOST, DEVICE = 0, 1
FLAG_APPROX_TANH = 1
OK, EINVAL, EUNSUPPORTED, ESTATE, ENOMEM, ENODEVICE = 0, -1, -2, -3, -4, -5
MAX_LAYERS = 6

EXPORTS = [
    "b200ude_version", "b200ude_last_error", "b200ude_create", "b200ude_destroy",
    "b200ude_num_params", "b200ude_num_save", "b200ude_device_bytes", "b200ude_set_params",
    "b200ude_forward", "b200ude_adjoint", "b200ude_adjoint_l2", "b200ude_solve_host",
    "b200ude_loss_gradient_host", "b200ude_get_params", "b200ude_adam_reset", "b200ude_adam_step", "b200ude_train_adam",
    "b200ude_peer_export", "b200ude_peer_attach", "b200ude_peer_detach", "b200ude_adjoint_l2_allreduce", "b200ude_selftest_tanh",
    "b200ude_bsde_create", "b200ude_bsde_destroy", "b200ude_bsde_last_error", "b200ude_bsde_num_params", "b200ude_bsde_set_params",
    "b200ude_bsde_get_params", "b200ude_bsde_loss_gradient", "b200ude_bsde_train_adam", "b200ude_bsde_adam_step", "b200ude_bsde_last_train_ms", "b200ude_bsde_last_sweep_ms",
]
PEER_HANDLE_BYTES = 64


class Desc(C.Structure):
    """struct b200ude_desc"""
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("dtype", C.c_int32), ("model", C.c_int32),
        ("state_dim", C.c_int32), ("n_layers", C.c_int32),
        ("widths", C.c_int32 * (MAX_LAYERS + 1)), ("acts", C.c_int32 * MAX_LAYERS),
        ("n_prefix", C.c_int32), ("n_suffix", C.c_int32), ("n_consts", C.c_int32),
        ("consts", C.c_double * 16),
        ("solver", C.c_int32), ("sensealg", C.c_int32),
        ("t0", C.c_double), ("dt", C.c_double), ("n_steps", C.c_int32), ("save_every", C.c_int32),
        ("abstol", C.c_double), ("reltol", C.c_double),
        ("n_loss_weights", C.c_int32), ("loss_weights", C.c_double * 16),
        ("max_trajectories", C.c_uint64), ("flags", C.c_uint32), ("adaptive", C.c_int32), ("max_steps", C.c_int32),
        ("n_stages", C.c_int32),
    ]


class Adam(C.Structure):
    """struct b200ude_adam"""
    _fields_ = [
        ("struct_size", C.c_uint32), ("reserved", C.c_uint32),
        ("eta", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
        ("loss_scale", C.c_double), ("l2_reg", C.c_double),
    ]


class BsdeDesc(C.Structure):
    """struct b200ude_bsde_desc"""
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32), ("dtype", C.c_int32), ("dim", C.c_int32), ("hidden", C.c_int32),
        ("n_steps", C.c_int32), ("T", C.c_double), ("lam", C.c_double), ("sigma", C.c_double), ("g_a", C.c_double), ("g_b", C.c_double),
        ("x0", C.POINTER(C.c_double)), ("max_paths", C.c_uint64),
    ]


class B200UDEError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"b200ude error {code}: {msg}")
        self.code = code


def _nvcc():
    """$NVCC, else nvcc on PATH, else the toolkit's under $CUDA_HOME or the default install location (a user's PATH may lack it)."""
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    return os.environ.get("NVCC") or shutil.which("nvcc") or os.path.join(home, "bin", "nvcc")


def build(verbose=False):
    """Compile csrc/ for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    jobs = str(min(8, os.cpu_count() or 1))
    subprocess.check_call(["make", "-C", CSRC, "-j", jobs, f"NVCC={_nvcc()}"] + ([] if verbose else ["-s"]))
    return SO_PATH


_lib = None


def lib():
    """Load libb200ude.so; raises (never falls back) when it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise FileNotFoundError(
            f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C universal_differential_equations_b200/csrc`). There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    vp, sz, i32 = C.c_void_p, C.c_size_t, C.c_int32
    L.b200ude_version.restype = i32
    L.b200ude_last_error.restype = C.c_char_p
    L.b200ude_last_error.argtypes = [vp]
    L.b200ude_create.restype = i32
    L.b200ude_create.argtypes = [C.POINTER(Desc), C.POINTER(vp)]
    L.b200ude_destroy.restype = None
    L.b200ude_destroy.argtypes = [vp]
    for f in ("b200ude_num_params", "b200ude_num_save", "b200ude_device_bytes"):
        getattr(L, f).restype = sz
        getattr(L, f).argtypes = [vp]
    L.b200ude_set_params.restype = i32
    L.b200ude_set_params.argtypes = [vp, vp, sz, i32, vp]
    L.b200ude_forward.restype = i32
    L.b200ude_forward.argtypes = [vp, vp, sz, vp, vp, vp]
    L.b200ude_adjoint.restype = i32
    L.b200ude_adjoint.argtypes = [vp, vp, vp, vp, vp]
    L.b200ude_adjoint_l2.restype = i32
    L.b200ude_adjoint_l2.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b200ude_solve_host.restype = i32
    L.b200ude_solve_host.argtypes = [vp, vp, vp, sz, vp, vp]
    L.b200ude_loss_gradient_host.restype = i32
    L.b200ude_loss_gradient_host.argtypes = [vp, vp, vp, vp, sz, C.POINTER(C.c_double), vp, vp]
    L.b200ude_get_params.restype = i32
    L.b200ude_get_params.argtypes = [vp, vp, sz, i32, vp]
    L.b200ude_adam_reset.restype = i32
    L.b200ude_adam_reset.argtypes = [vp, vp]
    L.b200ude_adam_step.restype = i32
    L.b200ude_adam_step.argtypes = [vp, C.POINTER(Adam), vp, vp]
    L.b200ude_train_adam.restype = i32
    L.b200ude_train_adam.argtypes = [vp, C.POINTER(Adam), vp, vp, sz, i32, vp, vp]
    L.b200ude_peer_export.restype = i32
    L.b200ude_peer_export.argtypes = [vp, vp]
    L.b200ude_peer_attach.restype = i32
    L.b200ude_peer_attach.argtypes = [vp, i32, i32, vp]
    L.b200ude_peer_detach.restype = i32
    L.b200ude_peer_detach.argtypes = [vp]
    L.b200ude_adjoint_l2_allreduce.restype = i32
    L.b200ude_adjoint_l2_allreduce.argtypes = [vp, vp, vp, vp, vp, vp]
    L.b200ude_selftest_tanh.restype = i32
    L.b200ude_selftest_tanh.argtypes = [i32, vp, vp, sz, vp]
    u64 = C.c_uint64
    L.b200ude_bsde_create.restype = i32
    L.b200ude_bsde_create.argtypes = [C.POINTER(BsdeDesc), C.POINTER(vp)]
    L.b200ude_bsde_destroy.restype = None
    L.b200ude_bsde_destroy.argtypes = [vp]
    L.b200ude_bsde_last_error.restype = C.c_char_p
    L.b200ude_bsde_last_error.argtypes = [vp]
    L.b200ude_bsde_num_params.restype = sz
    L.b200ude_bsde_num_params.argtypes = [vp]
    L.b200ude_bsde_set_params.restype = i32
    L.b200ude_bsde_set_params.argtypes = [vp, vp, sz, i32]
    L.b200ude_bsde_get_params.restype = i32
    L.b200ude_bsde_get_params.argtypes = [vp, vp, sz, i32]
    L.b200ude_bsde_loss_gradient.restype = i32
    L.b200ude_bsde_loss_gradient.argtypes = [vp, sz, u64, u64, sz, vp, vp, vp]
    L.b200ude_bsde_train_adam.restype = i32
    L.b200ude_bsde_train_adam.argtypes = [vp, C.POINTER(Adam), sz, i32, u64, vp, vp]
    L.b200ude_bsde_last_train_ms.restype = C.c_double
    L.b200ude_bsde_last_train_ms.argtypes = [vp]
    L.b200ude_bsde_last_sweep_ms.restype = i32
    L.b200ude_bsde_last_sweep_ms.argtypes = [vp, C.POINTER(C.c_double)]
    L.b200ude_bsde_adam_step.restype = i32
    L.b200ude_bsde_adam_step.argtypes = [vp, C.POINTER(Adam), vp]
    if L.b200ude_version() != ABI_VERSION:
        raise RuntimeError("libb200ude.so ABI version mismatch")
    _lib = L
    return L


def check_bsde(handle, rc):
    if rc != 0:
        msg = lib().b200ude_bsde_last_error(handle)
        raise B200UDEError(rc, msg.decode() if msg else "")


def check(handle, rc):
    if rc != 0:
        msg = lib().b200ude_last_error(handle)
        raise B200UDEError(rc, msg.decode() if msg else "")
