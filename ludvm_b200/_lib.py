"""ctypes binding of libludvm_b200.so (C ABI declared in include/ludvm_b200.h).

There is no fallback of any kind: if the shared library is missing, or no CUDA device is present, the calls
raise.  The oracle under `oracle/` is test infrastructure and is never imported from here.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LUDVM_B200_LIB") or os.path.join(HERE, "libludvm_b200.so")   # (override: kernel experiments)

EXACT_F64, FAST_F64, FAST_F32, FAST12_F64 = 0, 1, 2, 3
PTR_HOST, PTR_DEVICE = 0, 1
MODES = {"exact": EXACT_F64, "fast": FAST_F64, "fp32": FAST_F32, "fast12": FAST12_F64}

c_dp = C.POINTER(C.c_double)
c_vp = C.c_void_p


class LudvmError(RuntimeError):
    pass


class SimParams(C.Structure):
    _fields_ = [("nt", C.c_int64), ("P", C.c_int64), ("Nc", C.c_int64), ("nfree", C.c_int64),
                ("method", C.c_int32), ("mode", C.c_int32), ("store_history", C.c_int32),
                ("steps_per_graph", C.c_int32),
                ("dt", C.c_double), ("Uinf", C.c_double), ("chord", C.c_double), ("rho", C.c_double),
                ("piv", C.c_double), ("lespcrit", C.c_double), ("vc4", C.c_double), ("ic", C.c_double), ("sum_free", C.c_double),
                ("a0_init", C.c_double), ("a1_init", C.c_double), ("maxerror", C.c_double),
                ("epsilon", C.c_double), ("maxiter", C.c_int64)]


TABLE_FIELDS = ("cos_a", "sin_a", "alpha_dot", "h_dot", "gp", "le", "te", "detadx_p", "eta_p", "x_p", "theta_p",
                "dtheta", "cos_tp", "sin_tp", "cosn", "sinn", "free_g", "free_xz")


class SimTables(C.Structure):
    _fields_ = [(n, c_dp) for n in TABLE_FIELDS]


FIELDS = dict(PATH_TEV=0, PATH_LEV=1, PATH_FREE=2, G_TEV=3, G_LEV=4, G_BOUND=5, G_AIRFOIL=6, GAMMA_AIRFOIL=7,
              GAMMA_INT_AIRFOIL=8, FOURIER=9, LESP=10, LESP_PREV=11, LEV_SHED=12, FN=13, FS=14, L=15, D=16, T=17,
              M=18, CUR_TEV=19, CUR_LEV=20, CUR_FREE=21, COUNTERS=22, RANGE_BAD=23, DP=24)

# name -> (restype, argtypes); every symbol include/ludvm_b200.h declares
SIGNATURES = {
    "ludvm_abi_version": (C.c_int, []),
    "ludvm_last_error": (C.c_char_p, []),
    "ludvm_ctx_create": (C.c_int, [C.c_int, c_vp, C.POINTER(c_vp)]),
    "ludvm_ctx_destroy": (C.c_int, [c_vp]),
    "ludvm_ctx_synchronize": (C.c_int, [c_vp]),
    "ludvm_ctx_launch_count": (C.c_int, [c_vp, C.POINTER(C.c_longlong)]),
    "ludvm_ctx_last_plan": (C.c_int, [c_vp, C.POINTER(C.c_int32)]),
    "ludvm_induced_velocity": (C.c_int, [c_vp, C.c_int, c_vp, C.c_long, c_vp, c_vp, c_vp, C.c_double, C.c_long,
                                         c_vp, c_vp, C.c_long, c_vp, c_vp, C.c_int]),
    "ludvm_selfconv_step": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_long, C.c_long,
                                      C.c_long, C.c_double, c_vp, c_vp, c_vp, c_vp]),
    "ludvm_selfconv_step_all": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_long, C.c_double,
                                          c_vp, c_vp, c_vp, c_vp]),
    "ludvm_selfconv_step_p2p": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_long, C.c_long,
                                          C.c_long, C.c_double, C.c_int, C.POINTER(c_vp), C.POINTER(c_vp)]),
    "ludvm_induced_velocity_tree": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_long, c_vp, c_vp, C.c_long, C.c_int,
                                              C.c_int, c_vp, c_vp, C.c_int, c_dp]),
    "ludvm_flowfield_velocity_tree": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_long, C.c_double, c_vp, C.c_long, c_vp, C.c_long,
                                                C.c_long, C.c_long, C.c_double, C.c_int, C.c_int, c_vp, c_vp, C.c_int, c_dp]),
    "ludvm_selfconv_step_tree": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_double, C.c_long, C.c_long, C.c_long, C.c_double,
                                           C.c_int, C.c_int, c_vp, c_vp, c_vp, c_vp, c_dp]),
    "ludvm_flowfield_velocity": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, C.c_long, c_vp, c_vp, c_vp, C.c_long,
                                           C.c_double, c_vp, C.c_long, c_vp, C.c_long, C.c_long, C.c_long,
                                           c_vp, c_vp, C.c_int]),
    "ludvm_flowfield": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp, C.c_long, c_vp, c_vp, c_vp, C.c_long, C.c_double, c_vp,
                                  C.c_long, c_vp, C.c_long, C.c_long, C.c_long, c_vp, c_vp, c_vp, C.c_int]),
    "ludvm_flowfield_vorticity": (C.c_int, [c_vp, c_vp, C.c_long, c_vp, C.c_long, c_vp, c_vp, C.c_long, c_vp,
                                            C.c_int]),
    "ludvm_sim_create": (C.c_int, [c_vp, C.POINTER(SimParams), C.POINTER(SimTables), C.POINTER(c_vp)]),
    "ludvm_sim_run": (C.c_int, [c_vp, C.c_long]),
    "ludvm_sim_steps_done": (C.c_int, [c_vp, C.POINTER(C.c_long)]),
    "ludvm_sim_profile_steps": (C.c_int, [c_vp, C.c_long, c_dp]),
    "ludvm_sim_enable_pressure": (C.c_int, [c_vp]),
    "ludvm_sim_enable_far_field": (C.c_int, [c_vp, C.c_int]),
    "ludvm_sim_far_field_info": (C.c_int, [c_vp, C.POINTER(C.c_int64)]),
    "ludvm_sim_fetch": (C.c_int, [c_vp, C.c_int, c_vp, C.c_size_t]),
    "ludvm_sim_fetch_many": (C.c_int, [c_vp, C.c_int, C.POINTER(C.c_int), C.POINTER(c_vp), C.POINTER(C.c_size_t)]),
    "ludvm_sim_field_bytes": (C.c_int, [c_vp, C.c_int, C.POINTER(C.c_size_t)]),
    "ludvm_sim_destroy": (C.c_int, [c_vp]),
    "ludvm_sweep_run": (C.c_int, [c_vp, C.c_long, C.POINTER(SimParams), C.POINTER(SimTables), c_vp, C.c_size_t]),
    "ludvm_sweep_run_pressure": (C.c_int, [c_vp, C.c_long, C.POINTER(SimParams), C.POINTER(SimTables), c_vp, C.c_size_t,
                                           c_vp, C.c_size_t]),
    "ludvm_measure_fp64_fma_rate": (C.c_int, [c_vp, C.c_double, C.POINTER(C.c_double)]),
    "ludvm_measure_fp32_fma_rate": (C.c_int, [c_vp, C.c_double, C.POINTER(C.c_double)]),
}

_lib = None


def load():
    """Load the shared library (raises if it has not been built: there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise LudvmError("libludvm_b200.so is not built (run `python -c 'import __graft_entry__ as g; "
                             "g.build()'`); ludvm_b200 has no CPU fallback")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise LudvmError("libludvm_b200 error %d: %s" % (rc, load().ludvm_last_error().decode()))


def f64(a):
    return np.ascontiguousarray(np.asarray(a, dtype=np.float64))


def ptr(a):
    """Device pointer of a torch CUDA tensor, host pointer of a numpy array, or None."""
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()


def _pair_slots(kernel, variant_word):
    """FP64-pipe slots per evaluated term: fast_sym shares 10 of the pair's 13 slots between the terms (i, j) and (j, i)."""
    if kernel == "fast_sym":
        return 8
    if kernel == "fast_fused" and variant_word == 1:
        return 12
    return 13 if kernel.startswith("fast_") else 0


class Context:
    """One device + stream + scratch.  `stream` is a raw cudaStream_t (int), e.g.
    `torch.cuda.current_stream().cuda_stream`; 0 means the legacy default stream (PyTorch's default stream);
    None lets the library create a private non-blocking stream."""

    CUDA_STREAM_LEGACY = 0x1

    def __init__(self, device=0, stream=None):
        self._h = c_vp()
        if stream is not None and int(stream) == 0:
            stream = self.CUDA_STREAM_LEGACY
        self.stream_handle = int(stream) if stream is not None else None   # None: the library's private stream
        check(load().ludvm_ctx_create(int(device), c_vp(stream) if stream is not None else None, C.byref(self._h)))
        self.device = int(device)

    @property
    def handle(self):
        return self._h

    def synchronize(self):
        check(load().ludvm_ctx_synchronize(self._h))

    def launch_count(self):
        n = C.c_longlong(0)
        check(load().ludvm_ctx_launch_count(self._h, C.byref(n)))
        return n.value

    KERNELS = ("none", "exact_rows", "exact_tiled", "fast_rows", "fast_tiled", "fast_tiled_tma", "fast32_tiled",
               "fast32x2_tiled", "fast_fused", "tree", "fast_sym")

    def last_plan(self):
        """The all-pairs kernel the last call chose: dict(kernel, rows_per_thread, fold, tma, cluster, variant)."""
        out = (C.c_int32 * 8)()
        check(load().ludvm_ctx_last_plan(self._h, out))
        k = self.KERNELS[out[0]]
        return dict(kernel=k, rows_per_thread=out[1], fold=out[2], tma=bool(out[3]), cluster=out[4], variant=out[5],
                    warps=out[6], range_bad=out[7] if k.startswith("exact") else 0,
                    pair_slots=_pair_slots(k, out[7]))

    def fp64_fma_rate(self, ms=200.0):
        r = C.c_double(0)
        check(load().ludvm_measure_fp64_fma_rate(self._h, float(ms), C.byref(r)))
        return r.value

    def fp32_fma_rate(self, ms=200.0):
        r = C.c_double(0)
        check(load().ludvm_measure_fp32_fma_rate(self._h, float(ms), C.byref(r)))
        return r.value

    def close(self):
        if self._h:
            load().ludvm_ctx_destroy(self._h)
            self._h = c_vp()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default_ctx = {}


def default_context(device=0):
    if device not in _default_ctx:
        _default_ctx[device] = Context(device)
    return _default_ctx[device]
