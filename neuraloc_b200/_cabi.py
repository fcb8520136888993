"""ctypes binding of libnoc_b200.so — the C ABI declared in include/noc_b200.h.

This is the stub a maintainer of the reference would add (INTEGRATION.md): plain pointers and sizes,
no torch types.  The library is built in-tree (neuraloc_b200/libnoc_b200.so) by `make -C
neuraloc_b200/csrc` or `__graft_entry__.build()`; if it is missing every call raises — there is no
fallback path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NOC_LIB") or os.path.join(_HERE, "libnoc_b200.so")   # NOC_LIB: alternative build (tests)

F32, F64 = 0, 1
PROB_KINDS = {"Cross2D": 0, "SwarmTraj": 1, "Quadcopter": 2}
OBSTACLES = {None: 0, "softcorridor": 1, "hardcorridor": 2, "blocks": 3}
STEPPERS = {"rk1": 1, "rk4": 4}        # any other string: integrates nothing (OCflow.py:46-49)
MODE_MEAN, MODE_NOMEAN, MODE_INTERMEDIATES = 0, 1, 2

# every symbol include/noc_b200.h declares (tests check the library exports exactly these)
SYMBOLS = ["noc_version", "noc_last_error", "noc_device_info", "noc_ctrl_dim", "noc_stage_times", "noc_ocflow",
           "noc_ocflow_host", "noc_phi_eval", "noc_prob_eval", "noc_measure_fma_peak", "noc_tc_probe", "noc_launch_count",
           "noc_last_path", "noc_sample_rho0", "noc_philox_raw", "noc_ocflow_grad", "noc_baseline_loss", "noc_phi_vjp"]


class PhiT(C.Structure):
    _fields_ = [("d", C.c_int32), ("m", C.c_int32), ("nTh", C.c_int32), ("r", C.c_int32), ("h", C.c_double),
                ("A", C.c_void_p), ("c_w", C.c_void_p), ("c_b", C.c_void_p), ("w", C.c_void_p),
                ("K", C.POINTER(C.c_void_p)), ("b", C.POINTER(C.c_void_p))]


class ProbT(C.Structure):
    _fields_ = [("kind", C.c_int32), ("obstacle", C.c_int32), ("training", C.c_int32), ("nAgents", C.c_int32),
                ("agentDim", C.c_int32), ("alph_Q", C.c_double), ("alph_W", C.c_double), ("r", C.c_double),
                ("mass", C.c_double), ("grav", C.c_double), ("xtarget", C.c_void_p)]


_lib = None


class NocError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raise if the CUDA library has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NocError("libnoc_b200.so is not built (%s): run `make -C neuraloc_b200/csrc -j8` or "
                       "`python -c 'import __graft_entry__ as g; g.build()'`. There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i32, i64, dbl = C.c_void_p, C.c_int32, C.c_int64, C.c_double
    L.noc_version.restype = C.c_int
    L.noc_last_error.restype = C.c_char_p
    L.noc_launch_count.restype = i64
    L.noc_device_info.argtypes = [C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i64)]
    L.noc_ctrl_dim.argtypes = [C.POINTER(ProbT), i32]
    L.noc_stage_times.argtypes = [dbl, dbl, i32, C.POINTER(dbl)]
    common = [C.POINTER(PhiT), C.POINTER(ProbT), vp, i64, C.POINTER(dbl), dbl, dbl, i32, i32, C.POINTER(dbl), i32, i32,
              vp, vp, vp, vp]
    L.noc_ocflow.argtypes = common
    L.noc_ocflow_host.argtypes = common
    L.noc_ocflow_grad.argtypes = [C.POINTER(PhiT), C.POINTER(ProbT), vp, i64, C.POINTER(dbl), dbl, dbl, i32, C.POINTER(dbl), i32,
                                  vp, vp, vp, vp]
    L.noc_baseline_loss.argtypes = [C.POINTER(ProbT), vp, vp, i64, i32, i32, dbl, i32, vp, vp, vp]
    L.noc_phi_eval.argtypes = [C.POINTER(PhiT), vp, i64, i32, vp, vp, vp]
    L.noc_phi_vjp.argtypes = [C.POINTER(PhiT), vp, i64, vp, vp, i32, vp, vp, vp]
    L.noc_prob_eval.argtypes = [C.POINTER(ProbT), vp, vp, i64, i32, i32, vp, vp, vp, vp]
    L.noc_measure_fma_peak.argtypes = [i32, C.POINTER(dbl)]
    L.noc_tc_probe.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    L.noc_sample_rho0.argtypes = [vp, i32, i32, dbl, C.c_uint64, i64, i64, i32, vp, vp]
    L.noc_philox_raw.argtypes = [C.c_uint64, i64, i64, vp, vp]
    for name in SYMBOLS:
        if name not in ("noc_last_error", "noc_launch_count"):
            getattr(L, name).restype = C.c_int
    if L.noc_version() != 1:
        raise NocError("libnoc_b200.so ABI version %d, binding expects 1" % L.noc_version())
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NocError("noc error %d: %s" % (rc, lib().noc_last_error().decode("utf-8", "replace")))


PATH_NAMES = {-1: "none", 0: "tile", 1: "sample", 2: "tensor"}


def last_path():
    """Kernel family of this thread's last rollout: 'tile' (FMA), 'sample' (small batch) or 'tensor' (tcgen05)."""
    return PATH_NAMES[int(lib().noc_last_path())]


def launch_count():
    return int(lib().noc_launch_count())
