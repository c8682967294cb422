"""ctypes binding of liberirt_b200.so (include/erirt_b200.h).  No fallback: if the CUDA library is missing or
fails to load, importing the compute entry points raises."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ERIRT_B200_LIB", os.path.join(HERE, "liberirt_b200.so"))

ABI_VERSION = 1
MODELS = {"MlIrt": 0, "RtIrt": 1, "RtIrtNull": 2, "RtIrtCross": 3, "RtIrtCrossQr": 4, "RtIrtLatent": 5,
          "RtIrtLatentQr": 6, "RtIrtQuantile": 6}
F32, F64 = 0, 1
FIELDS = {"theta": 0, "zeta": 1, "a": 2, "b": 3, "lambda": 4, "sigma2": 5, "beta": 6, "rho": 7, "Sigma": 8, "nu": 9,
          "omega": 10}
TRACES = {"ra": 0, "rt": 1, "qr": 2, "logLike": 3}
ERROR_TYPES = {"tnorm": 0, "unit": 1, "norm": 2, "tail": 3, "skew": 4}
COMPAT_BETA_PRIOR_DIAG = 1
COMPAT_LATENTQR_SCALE_ELEMENTWISE = 2

EXPORTED = ["erirt_version", "erirt_last_error", "erirt_create", "erirt_create_batch", "erirt_destroy", "erirt_set_data",
            "erirt_set_data_device", "erirt_trim_pool", "erirt_generate_data", "erirt_get_data", "erirt_set_data_y8", "erirt_checkpoint_size", "erirt_checkpoint_save", "erirt_checkpoint_load", "erirt_set_state", "erirt_get_state", "erirt_sample", "erirt_get_trace",
            "erirt_trace_width", "erirt_get_moments", "erirt_trace_ess_rhat", "erirt_ess_rhat", "erirt_loglik_current", "erirt_get_stats", "erirt_debug_check_guards",
            "erirt_nccl_unique_id", "erirt_comm_init", "erirt_peer_export", "erirt_peer_attach", "erirt_peer_detach", "erirt_k_pg", "erirt_k_nu_person", "erirt_k_philox"]


class Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("model", C.c_int32), ("n_subj", C.c_int64), ("n_subj_total", C.c_int64),
                ("subj_offset", C.c_int64), ("n_item", C.c_int32), ("n_feat", C.c_int32), ("n_iter", C.c_int32),
                ("n_chain", C.c_int32), ("n_burnin", C.c_int32), ("q_rt", C.c_double), ("intercept", C.c_int32),
                ("itemtype_1pl", C.c_int32), ("cov2one", C.c_int32), ("dtype", C.c_int32), ("seed", C.c_uint64),
                ("chain", C.c_uint32), ("compat", C.c_int32), ("person_trace", C.c_int32), ("device", C.c_int32),
                ("use_graph", C.c_int32), ("time_kernels", C.c_int32), ("nu_cell_moments", C.c_int32), ("reserved", C.c_int32 * 6)]


class Stats(C.Structure):
    _fields_ = [("sweeps_done", C.c_int64), ("last_sample_ms", C.c_double), ("person_kernel_ms", C.c_double),
                ("bytes_per_sweep", C.c_int64), ("pg_deferred_frac", C.c_double), ("launches_per_sweep", C.c_int32),
                ("sm_count", C.c_int32)]


class ErirtError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"erirt_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load the shared library; raises if it has not been built (python -m ... build / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build the CUDA extension first (__graft_entry__.build()); "
                          "there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    dp, vp = C.POINTER(C.c_double), C.c_void_p
    L.erirt_version.restype = C.c_int
    L.erirt_last_error.restype = C.c_char_p
    L.erirt_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.erirt_create_batch.argtypes = [C.POINTER(Config), C.c_int32, C.POINTER(vp)]
    L.erirt_destroy.argtypes = [vp]
    L.erirt_trim_pool.argtypes = [C.c_int32]
    L.erirt_set_data.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64]
    L.erirt_set_data_device.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64]
    L.erirt_set_data_y8.argtypes = [vp, vp, C.c_int64, vp, C.c_int64, vp, C.c_int64]
    L.erirt_generate_data.argtypes = [vp, dp, dp, dp, dp, dp, dp, dp, dp, C.c_int64, C.c_int32, C.c_uint64]
    L.erirt_get_data.argtypes = [vp, dp, C.c_int64, dp, C.c_int64]
    L.erirt_checkpoint_size.argtypes = [vp]
    L.erirt_checkpoint_size.restype = C.c_int64
    L.erirt_checkpoint_save.argtypes = [vp, vp, C.c_int64]
    L.erirt_checkpoint_load.argtypes = [vp, vp, C.c_int64]
    L.erirt_set_state.argtypes = [vp, C.c_int32, dp, C.c_int64]
    L.erirt_get_state.argtypes = [vp, C.c_int32, dp, C.c_int64]
    L.erirt_sample.argtypes = [vp, C.c_int64]
    L.erirt_get_trace.argtypes = [vp, C.c_int32, C.c_int64, C.c_int64, dp]
    L.erirt_trace_width.argtypes = [vp, C.c_int32]
    L.erirt_trace_width.restype = C.c_int64
    L.erirt_get_moments.argtypes = [vp, C.c_int32, dp, dp, C.c_int64]
    L.erirt_trace_ess_rhat.argtypes = [vp, C.c_int32, C.c_int64, C.c_int64, C.c_int64, dp, dp]
    L.erirt_ess_rhat.argtypes = [dp, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_int32, dp, dp]
    L.erirt_loglik_current.argtypes = [vp, C.POINTER(C.c_double)]
    L.erirt_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.erirt_debug_check_guards.argtypes = [vp]
    L.erirt_debug_check_guards.restype = C.c_int64
    L.erirt_nccl_unique_id.argtypes = [vp]
    L.erirt_comm_init.argtypes = [vp, C.c_int32, C.c_int32, vp]
    L.erirt_peer_export.argtypes = [vp, vp]
    L.erirt_peer_attach.argtypes = [vp, vp]
    L.erirt_peer_detach.argtypes = [vp]
    L.erirt_k_pg.argtypes = [dp, C.c_int64, C.c_int32, C.c_int64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_int32,
                             C.c_int32, dp]
    L.erirt_k_nu_person.argtypes = [dp, C.c_double, C.c_int64, C.c_int64, C.c_uint64, C.c_uint32, C.c_uint32,
                                    C.c_int32, C.c_int32, dp]
    L.erirt_k_philox.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.c_int32, C.POINTER(C.c_uint32)]
    for name in EXPORTED:
        if name not in ("erirt_last_error", "erirt_trace_width", "erirt_version", "erirt_checkpoint_size", "erirt_debug_check_guards"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise ErirtError(rc, load().erirt_last_error().decode("utf-8", "replace"))
