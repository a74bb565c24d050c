"""ctypes binding of libtvf.so (include/tvf.h).

There is no CPU fallback: if the library is missing, or no CUDA device is
usable, loading / handle creation raises.
"""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# TVF_LIBPATH: development switch (benchmarking compile-time variants of the library); never a CPU fallback
LIB_PATH = os.environ.get("TVF_LIBPATH") or os.path.join(_HERE, "libtvf.so")

c_double_p = C.POINTER(C.c_double)
c_int32_p = C.POINTER(C.c_int32)

TVF_OK = 0
TVF_ERR_ARG = -1
TVF_ERR_CUDA = -2
TVF_ERR_TOO_FEW_POINTS = -3
TVF_ERR_NOMEM = -4

ST_EIG_NOCONV = 1
ST_EPIPOLE_ZERO = 2
ST_NO_POSE_2 = 4
ST_NO_POSE_3 = 8
ST_NONFINITE = 16
ST_BA_NOCONV = 32
ST_COV_SINGULAR = 64
ST_RANSAC_FAILED = 128

LINEARF_ERRMSG = ("At least 8 correspondences are necessary to compute the "
                  "fundamental matrix linearly\\n")

class PoseOut(C.Structure):
    """tvf_pose_out of include/tvf.h: every optional output of a pose call (host or device pointers)."""
    _fields_ = [(k, C.c_void_p) for k in ("Rt2", "Rt3", "reconst", "T", "repr_err", "F21", "F31", "iter", "votes", "status")]


class SweepLevel(C.Structure):
    """tvf_sweep_level of include/tvf.h: one value of the swept variable of experiments.m:38-47."""
    _fields_ = [("noise", C.c_double), ("n", C.c_int32), ("reserved", C.c_int32), ("P", C.c_double * 36),
                ("calm", C.c_double * 27), ("Rt0_2", C.c_double * 12), ("Rt0_3", C.c_double * 12)]


METHOD_IDS = {"tft": 1, "f": 7, "optf": 8}      # numbering of experiments.m:51-59

# name -> (restype, argtypes); mirrors include/tvf.h one to one
_H = C.c_void_p
_D = c_double_p
_I = C.c_int
_L = C.c_int64
_S = c_int32_p
SIGNATURES = {
    "tvf_version": (_I, []),
    "tvf_device_count": (_I, []),
    "tvf_create": (_I, [C.POINTER(_H), _I]),
    "tvf_create_multi": (_I, [C.POINTER(_H), C.POINTER(C.c_int), _I]),
    "tvf_num_devices": (_I, [_H]),
    "tvf_set_host_register": (_I, [_H, _I]),
    "tvf_set_host_threads": (_I, [_H, _I]),
    "tvf_pose": (_I, [_H, _I, _D, _D, _I, _I, _L, C.POINTER(PoseOut)]),
    "tvf_pose_dev": (_I, [_H, _I, C.c_void_p, C.c_void_p, _I, _I, _L, C.POINTER(PoseOut)]),
    "tvf_destroy": (None, [_H]),
    "tvf_last_error": (C.c_char_p, [_H]),
    "tvf_device": (_I, [_H]),
    "tvf_set_chunk": (_I, [_H, _L]),
    "tvf_set_stream": (_I, [_H, C.c_void_p]),
    "tvf_use_own_stream": (_I, [_H]),
    "tvf_synchronize": (_I, [_H]),
    "tvf_host_alloc": (C.c_void_p, [C.c_size_t]),
    "tvf_host_free": (None, [C.c_void_p]),
    "tvf_linear_tft_pose": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, _D, _D, _D, _S]),
    "tvf_linear_f_pose": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, _D, _D, _D, _D, _D, _S]),
    "tvf_optim_f_pose": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, _D, _D, _D, _D, _D, _S, _S]),
    "tvf_optim_f_pose_dev": (_I, [_H, C.c_void_p, C.c_void_p, _I, _I, _L] + [C.c_void_p] * 9),
    "tvf_optim_f_max_n": (_I, []),
    "tvf_optim_f": (_I, [_H, _D, _D, _I, _I, _L, _D, _S, _S]),
    "tvf_linear_tft": (_I, [_H, _D, _D, _D, _I, _I, _L, _D, _D, _D, _S]),
    "tvf_linear_f": (_I, [_H, _D, _D, _I, _I, _L, _D, _S]),
    "tvf_normalize2d": (_I, [_H, _D, _I, _L, _D, _D]),
    "tvf_transform_tft": (_I, [_H, _D, _D, _D, _D, _I, _I, _L, _D]),
    "tvf_rt_from_tft": (_I, [_H, _D, _D, _I, _D, _I, _L, _D, _D, _S, _S]),
    "tvf_tft_from_p": (_I, [_H, _D, _D, _D, _L, _D]),
    "tvf_triangulate": (_I, [_H, _D, _I, _I, _D, _I, _I, _L, _D]),
    "tvf_repr_error": (_I, [_H, _D, _I, _I, _D, _I, _I, _L, _D, _I, _D]),
    "tvf_ang_error": (_I, [_H, _D, _I, _D, _L, _D, _D]),
    "tvf_project3d": (_I, [_H, _D, _D, _I, _I, _I, _L, _D]),
    "tvf_generate_sweep": (_I, [_H, _L, _L, _I, _D, _I, _D, C.c_double, C.c_double, _D]),
    "tvf_sweep_run": (_I, [_H, _I, _L, _L, _I, _D, _I, _D, C.c_double, C.c_double, _D, _D, _D, _D]),
    "tvf_sweep_run_levels": (_I, [_H, _I, _L, _L, C.POINTER(SweepLevel), _I, C.c_double, C.c_double, _D]),
    "tvf_sweep_run_levels_ba": (_I, [_H, _I, _L, _L, C.POINTER(SweepLevel), _I, C.c_double, C.c_double, _D]),
    "tvf_generate_sweep_dev": (_I, [_H, _L, _L, _I, _D, _I, _D, C.c_double, C.c_double, C.c_void_p]),
    "tvf_linear_tft_pose_dev": (_I, [_H, C.c_void_p, C.c_void_p, _I, _I, _L] + [C.c_void_p] * 6),
    "tvf_linear_f_pose_dev": (_I, [_H, C.c_void_p, C.c_void_p, _I, _I, _L] + [C.c_void_p] * 8),
    "tvf_bundle_adjust": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, _D, _D, _D, _D, _D, _S, _S]),
    "tvf_bundle_adjust_dev": (_I, [_H, C.c_void_p, C.c_void_p, _I, _I, _L] + [C.c_void_p] * 9),
    "tvf_ba_covariance": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, _D, _D, _D, _D, _S]),
    "tvf_ba_covariance_dev": (_I, [_H, C.c_void_p, C.c_void_p, _I, _I, _L] + [C.c_void_p] * 7),
    "tvf_consensus": (_I, [_H, _D, _D, _I, _I, _L, _D, _D, C.c_double, C.c_void_p, _S]),
    "tvf_ransac_pose": (_I, [_H, _I, _D, _D, _I, _I, _L, _I, C.c_double, C.c_void_p, _D, _D, C.c_void_p, _S, _S, _S]),
    "tvf_ransac_pose_dev": (_I, [_H, _I, C.c_void_p, C.c_void_p, _I, _I, _L, _I, C.c_double] + [C.c_void_p] * 7),
    "tvf_launch_count": (_L, [_H]),
    "tvf_profile_enable": (_I, [_H, _I]),
    "tvf_profile_reset": (_I, [_H]),
    "tvf_profile_read": (_I, [_H, _D, C.POINTER(C.c_int64)]),
    "tvf_kernel_name": (C.c_char_p, [_I]),
    "tvf_fp64_peak_tflops": (C.c_double, [_H]),
}
NUM_KERNELS = 14

_lib = None
_lock = threading.Lock()


class TvfError(RuntimeError):
    pass


def load():
    """Load libtvf.so and declare every prototype.  Raises if the library is absent."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise TvfError(
                "libtvf.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(tft_vs_fund_b200 has no CPU fallback)" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)          # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
        _lib = lib
        return lib


_handles = {}


def handle(device=None):
    """Process-wide handle per device (created on first use).  `device` may be a tuple/list of device ids: a group
    handle (tvf_create_multi) whose host-pointer pose calls shard the batch over those GPUs."""
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if lib.tvf_device_count() > 1 else 0
        device = device % max(1, lib.tvf_device_count())
    if isinstance(device, (list, tuple)):
        device = tuple(int(d) for d in device)
    key = (threading.get_ident(), device)
    h = _handles.get(key)
    if h is None:
        h = Handle(device)
        _handles[key] = h
    return h


class Handle:
    def __init__(self, device=0):
        self.lib = load()
        self._h = C.c_void_p()
        if isinstance(device, (list, tuple)):
            ids = (C.c_int * len(device))(*[int(d) for d in device])
            rc = self.lib.tvf_create_multi(C.byref(self._h), ids, len(device))
        else:
            rc = self.lib.tvf_create(C.byref(self._h), int(device))
        if rc != TVF_OK:
            msg = self.lib.tvf_last_error(None)
            raise TvfError("tvf_create(device=%s) failed (%d): %s" % (device, rc, msg.decode() if msg else ""))
        self.device = device

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            self.lib.tvf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def error(self):
        msg = self.lib.tvf_last_error(self._h)
        return msg.decode() if msg else ""

    def check(self, rc, what):
        if rc == TVF_ERR_TOO_FEW_POINTS:
            raise ValueError(LINEARF_ERRMSG)
        if rc < 0:
            raise TvfError("%s failed (%d): %s" % (what, rc, self.error()))
        return rc

    def call(self, name, *args):
        return self.check(getattr(self.lib, name)(self._h, *args), name)
