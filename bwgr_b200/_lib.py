"""ctypes binding of include/bwgr_b200.h (the same C ABI an Rcpp shim binds; see INTEGRATION.md).

No CPU path: if libbwgr_b200.so is missing or no B200 is visible, every call raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BWGR_LIB") or os.path.join(_HERE, "lib", "libbwgr_b200.so")  # BWGR_LIB: another build of the same library (A/B runs)

# every symbol include/bwgr_b200.h declares (tests check the shared object exports all of them)
SYMBOLS = [
    "bwgr_create", "bwgr_destroy", "bwgr_last_error", "bwgr_version", "bwgr_set_stream", "bwgr_set_tuning",
    "bwgr_fitted", "bwgr_fitted_sys", "bwgr_geno_load_f64", "bwgr_geno_load_f64_centred", "bwgr_geno_load_bed", "bwgr_geno_load_i8", "bwgr_geno_load_i8_device", "bwgr_geno_unpack_i8", "bwgr_geno_raw",
    "bwgr_geno_info", "bwgr_geno_stats", "bwgr_em_fit", "bwgr_em_begin", "bwgr_em_sweeps", "bwgr_em_end",
    "bwgr_gibbs_fit", "bwgr_gibbs_fit_sys", "bwgr_kmup_sweep", "bwgr_kmup2_sweep", "bwgr_wgr_fit_bag", "bwgr_gs_fit", "bwgr_wgr_fit", "bwgr_mrr3_fit", "bwgr_dist_unique_id", "bwgr_dist_init", "bwgr_dist_connect", "bwgr_launch_count", "bwgr_debug_gram", "bwgr_debug_gram_band", "bwgr_debug_narrow", "bwgr_trim", "bwgr_profile", "bwgr_profile_read",
]


class BwgrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("bwgr_b200 error %d: %s" % (code, msg))
        self.code = code


class EmParams(C.Structure):
    _fields_ = [("model", C.c_int), ("nsys", C.c_int), ("it", C.c_int), ("df", C.c_double), ("R2", C.c_double),
                ("Pi", C.c_double), ("alpha", C.c_double), ("row_mask", C.c_void_p), ("weights", C.c_void_p)]


class EmOut(C.Structure):
    _fields_ = [("mu", C.c_void_p), ("b", C.c_void_p), ("d", C.c_void_p), ("hat", C.c_void_p), ("vb", C.c_void_p),
                ("scal", C.c_void_p), ("its", C.c_void_p)]


class GibbsParams(C.Structure):
    _fields_ = [("model", C.c_int), ("nchains", C.c_int), ("it", C.c_int), ("bi", C.c_int), ("pi", C.c_double),
                ("df", C.c_double), ("R2", C.c_double), ("seed", C.c_uint64)]


class GibbsSysParams(C.Structure):
    _fields_ = [("base", GibbsParams), ("nsys", C.c_int), ("row_mask", C.c_void_p), ("chain0", C.c_int)]


class GibbsOut(C.Structure):
    _fields_ = [("mu", C.c_void_p), ("b", C.c_void_p), ("d", C.c_void_p), ("hat", C.c_void_p), ("vb", C.c_void_p),
                ("scal", C.c_void_p)]


_lib = None


def load():
    """Load the shared object (building is __graft_entry__.build()'s job, not an import side effect)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BwgrError(-2, "CUDA library %s not built (run `python -m bwgr_b200.build`); there is no CPU fallback" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        lib.bwgr_last_error.restype = C.c_char_p
        lib.bwgr_launch_count.restype = C.c_int64
        lib.bwgr_launch_count.argtypes = [C.c_void_p]
        lib.bwgr_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.bwgr_destroy.argtypes = [C.c_void_p]
        lib.bwgr_destroy.restype = None
        lib.bwgr_trim.restype = None
        lib.bwgr_trim.argtypes = []
        lib.bwgr_set_stream.argtypes = [C.c_void_p, C.c_void_p]
        lib.bwgr_set_tuning.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        for name in ("bwgr_geno_load_f64", "bwgr_geno_load_f64_centred", "bwgr_geno_load_i8", "bwgr_geno_load_i8_device"):
            getattr(lib, name).argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int]
        lib.bwgr_geno_load_bed.argtypes = [C.c_void_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p]
        lib.bwgr_geno_unpack_i8.argtypes = [C.c_void_p, C.c_void_p]
        lib.bwgr_geno_raw.argtypes = [C.c_void_p, C.c_void_p]
        lib.bwgr_geno_info.argtypes = [C.c_void_p] + [C.c_void_p] * 5
        lib.bwgr_geno_stats.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.bwgr_em_fit.argtypes = [C.c_void_p, C.POINTER(EmParams), C.c_void_p, C.POINTER(EmOut)]
        lib.bwgr_em_begin.argtypes = [C.c_void_p, C.POINTER(EmParams), C.c_void_p]
        lib.bwgr_em_sweeps.argtypes = [C.c_void_p, C.c_int]
        lib.bwgr_em_end.argtypes = [C.c_void_p, C.POINTER(EmOut)]
        lib.bwgr_gibbs_fit.argtypes = [C.c_void_p, C.POINTER(GibbsParams), C.c_void_p, C.POINTER(GibbsOut)]
        lib.bwgr_gibbs_fit_sys.argtypes = [C.c_void_p, C.POINTER(GibbsSysParams), C.c_void_p, C.POINTER(GibbsOut)]
        lib.bwgr_fitted.argtypes = [C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]
        lib.bwgr_fitted_sys.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.bwgr_kmup_sweep.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_double, C.c_double, C.c_uint64]
        lib.bwgr_kmup2_sweep.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_double, C.c_double, C.c_uint64]
        lib.bwgr_wgr_fit_bag.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_double,
                                         C.c_double, C.c_double, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p]
        lib.bwgr_gs_fit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int,
                                    C.c_void_p, C.c_void_p]
        lib.bwgr_wgr_fit.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_double,
                                     C.c_double, C.c_double, C.c_uint64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p]
        lib.bwgr_mrr3_fit.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 12
        lib.bwgr_dist_unique_id.argtypes = [C.c_void_p]
        lib.bwgr_dist_init.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
        lib.bwgr_dist_connect.argtypes = [C.c_void_p, C.c_void_p]
        lib.bwgr_profile.argtypes = [C.c_void_p, C.c_int]
        lib.bwgr_profile_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.bwgr_debug_gram_band.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.bwgr_debug_narrow.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.bwgr_debug_gram.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        _lib = lib
    return _lib


def check(rc):
    if rc != 0:
        raise BwgrError(rc, load().bwgr_last_error().decode("utf-8", "replace"))
