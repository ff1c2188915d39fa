"""ctypes binding of libbgmm.so (the C ABI declared in include/bgmm.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, "libbgmm.so")

# constants mirrored from include/bgmm.h (checked against bgmm_abi_version at load time)
ABI_VERSION = 6
F64, F32 = 0, 1
PASS_AUTO, PASS_SIMPLE, PASS_DMMA, PASS_F32, PASS_LARGE, PASS_DIRECT, PASS_TF32 = 0, 1, 2, 3, 4, 5, 6
SMALL_FEATURES, SMALL_ITERATE, SMALL_STATS = 0, 1, 2

OFF_NAMES = ("center", "alpha0", "kappa0", "nu0", "m0", "w0inv", "lnb0", "lnc0", "params0", "params1", "stats",
             "ns", "xbar", "smats", "vlk", "vlterms", "vlhist", "ctrl", "total", "stats_len", "params_len", "pitch", "shift")
STATS_ENTROPY, STATS_ROWS, STATS_FORMAT = 0, 1, 2       # tail slots of the statistics: stats[K * pitch + slot]
POFF_NAMES = ("alpha", "kappa", "nu", "m", "winv", "w", "elnpi", "elndet", "lnb", "coef", "acst", "linv")
CTRL_CUR, CTRL_ITER, CTRL_DONE, CTRL_CONVERGED, CTRL_TICKET, CTRL_PASS_TICKET, CTRL_ERROR, CTRL_SEQ, CTRL_ROBUST, CTRL_CRIT = range(10)
CTRL_COMM_LO, CTRL_COMM_HI = 10, 11
FORCE, FORCE_NO_PUBLISH = 1, 2
MAX_RANKS = 16
MAX_BATCH = 8
N_CTRL = 16
HMM_OFF_NAMES = ("zeta0", "lncz0", "set0", "set1", "set_zeta", "set_lna", "set_at", "set_misc", "ms", "g0", "sc", "vlx",
                 "total")
HMM_FULL, HMM_STATS_FROM_GAMMA, HMM_EMISSION_ONLY = 0, 1, 2

_lib = None


def load():
    """Load libbgmm.so once; raises RuntimeError (no CPU fallback) when it cannot be loaded."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA library is required (no CPU fallback). "
            "Build it with `python -m bayesml_b200.build`.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, f64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_double
    lib.bgmm_abi_version.restype = i32
    lib.bgmm_abi_version.argtypes = []
    lib.bgmm_last_error.restype = ctypes.c_char_p
    lib.bgmm_last_error.argtypes = []
    lib.bgmm_launch_count.restype = i64
    lib.bgmm_launch_count.argtypes = []
    lib.bgmm_robust_threshold.restype = f64
    lib.bgmm_robust_threshold.argtypes = []
    lib.bgmm_set_robust_threshold.restype = f64
    lib.bgmm_set_robust_threshold.argtypes = [f64]
    lib.bgmm_layout.restype = i32
    lib.bgmm_layout.argtypes = [i32, i32, i32, ctypes.POINTER(i64), ctypes.POINTER(i64)]
    lib.bgmm_workspace_doubles.restype = i64
    lib.bgmm_workspace_doubles.argtypes = [i32, i32]
    lib.bgmm_colsum.restype = i32
    lib.bgmm_colsum.argtypes = [vp, i64, i32, i32, vp, vp, vp]
    lib.bgmm_center.restype = i32
    lib.bgmm_center.argtypes = [vp, i32, vp, i32, i64, i32, vp, vp]
    lib.bgmm_pass.restype = i32
    lib.bgmm_pass.argtypes = [vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    lib.bgmm_pass_batched.restype = i32
    lib.bgmm_pass_batched.argtypes = [vp, i64, i32, i32, i32, ctypes.POINTER(vp), vp, vp, vp, vp]
    lib.bgmm_batch_capacity.restype = i32
    lib.bgmm_batch_capacity.argtypes = [i32, i32]
    lib.bgmm_pred_logdensity.restype = i32
    lib.bgmm_pred_logdensity.argtypes = [vp, i64, i32, vp, vp, vp, vp, vp, vp]
    lib.bgmm_dirichlet1.restype = i32
    lib.bgmm_dirichlet1.argtypes = [vp, i64, i32, ctypes.c_uint64, i64, vp]
    lib.bgmm_gen_sample.restype = i32
    lib.bgmm_gen_sample.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, ctypes.c_uint64, i64, vp]
    lib.bgmm_hmm_gen_workspace_bytes.restype = i64
    lib.bgmm_hmm_gen_workspace_bytes.argtypes = [i32, i64, i64, i64]
    lib.bgmm_hmm_gen_sample.restype = i32
    lib.bgmm_hmm_gen_sample.argtypes = [vp, vp, i64, i32, i32, vp, vp, vp, vp, i64, ctypes.c_uint64, i64, vp, vp]
    lib.bgmm_hmm_init_random_workspace_doubles.restype = i64
    lib.bgmm_hmm_init_random_workspace_doubles.argtypes = [i32, i64]
    lib.bgmm_hmm_init_random.restype = i32
    lib.bgmm_hmm_init_random.argtypes = [i64, i32, ctypes.c_uint64, vp, vp, i64, vp, vp, vp, vp]
    lib.bgmm_tc_selftest.restype = i32
    lib.bgmm_tc_selftest.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    lib.bgmm_tf32_workspace_doubles.restype = i64
    lib.bgmm_tf32_workspace_doubles.argtypes = [i32, i32, i64]
    lib.bgmm_pass_supported.restype = i32
    lib.bgmm_pass_supported.argtypes = [i32, i32, i32, i32]
    lib.bgmm_pass_resolve.restype = i32
    lib.bgmm_pass_resolve.argtypes = [i32, i32, i32, i32, i32]
    lib.bgmm_small.restype = i32
    lib.bgmm_small.argtypes = [i32, i32, vp, i32, i32, f64, i32, vp, vp]
    lib.bgmm_comm_block_doubles.restype = i64
    lib.bgmm_comm_block_doubles.argtypes = [i32, i32]
    lib.bgmm_comm_alloc.restype = i32
    lib.bgmm_comm_alloc.argtypes = [i64, ctypes.POINTER(vp), ctypes.c_char_p]
    lib.bgmm_comm_open.restype = i32
    lib.bgmm_comm_open.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
    lib.bgmm_comm_close.restype = i32
    lib.bgmm_comm_close.argtypes = [vp]
    lib.bgmm_comm_free.restype = i32
    lib.bgmm_comm_free.argtypes = [vp]
    lib.bgmm_hmm_layout.restype = i32
    lib.bgmm_hmm_layout.argtypes = [i32, ctypes.POINTER(i64)]
    lib.bgmm_hmm_supported.restype = i32
    lib.bgmm_hmm_supported.argtypes = [i32, i32]
    lib.bgmm_hmm_scan_workspace_doubles.restype = i64
    lib.bgmm_hmm_scan_workspace_doubles.argtypes = [i32, i64]
    lib.bgmm_hmm_pass.restype = i32
    lib.bgmm_hmm_pass.argtypes = [vp, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp]
    lib.bgmm_hmm_viterbi.restype = i32
    lib.bgmm_hmm_viterbi.argtypes = [i64, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.bgmm_hmm_seq_plan.restype = i64
    lib.bgmm_hmm_seq_plan.argtypes = [i64, i64, vp, vp, i64]
    lib.bgmm_hmm_seq_workspace_doubles.restype = i64
    lib.bgmm_hmm_seq_workspace_doubles.argtypes = [i32, i64, i64]
    lib.bgmm_hmm_pass_seqs.restype = i32
    lib.bgmm_hmm_pass_seqs.argtypes = [vp, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, vp, vp, vp]
    lib.bgmm_hmm_viterbi_seqs.restype = i32
    lib.bgmm_hmm_viterbi_seqs.argtypes = [i64, i32, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    lib.bgmm_hmm_small.restype = i32
    lib.bgmm_hmm_small.argtypes = [i32, i32, vp, vp, i32, i32, f64, i32, vp]
    if lib.bgmm_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libbgmm ABI {lib.bgmm_abi_version()} != binding ABI {ABI_VERSION}; rebuild the library")
    _lib = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().bgmm_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"{what} failed (code {rc}): {msg}")


def layout(K, D, hist_len):
    """Offsets (in doubles) of the device state block; see include/bgmm.h."""
    lib = load()
    off = (ctypes.c_int64 * len(OFF_NAMES))()
    poff = (ctypes.c_int64 * len(POFF_NAMES))()
    check(lib.bgmm_layout(K, D, hist_len, off, poff), "bgmm_layout")
    return dict(zip(OFF_NAMES, off)), dict(zip(POFF_NAMES, poff))


def hmm_layout(K):
    """Offsets (in doubles) of the hidden-Markov extension block; see include/bgmm.h."""
    lib = load()
    off = (ctypes.c_int64 * len(HMM_OFF_NAMES))()
    check(lib.bgmm_hmm_layout(K, off), "bgmm_hmm_layout")
    return dict(zip(HMM_OFF_NAMES, off))
