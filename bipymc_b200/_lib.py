"""ctypes binding of the C-ABI in include/bipymc_b200.h.

The shared library is built in-tree (bipymc_b200/lib/libbipymc_b200.so) by
``__graft_entry__.build()`` / ``python -m bipymc_b200.build``.  There is NO CPU fallback:
if the library is missing, or no CUDA device is present when a sampler is constructed,
the package raises instead of silently computing somewhere else.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# BIPYMC_B200_LIB: alternative build of the same library (A/B experiments of kernel variants)
LIB_PATH = os.environ.get("BIPYMC_B200_LIB") or os.path.join(_HERE, "lib", "libbipymc_b200.so")

BPM_ALGO_DEMC, BPM_ALGO_DREAM, BPM_ALGO_DEMC_SERIAL = 0, 1, 2
TARGET_EXTERNAL, TARGET_BANANA, TARGET_BIMODAL, TARGET_GAUSS, TARGET_LINEFIT, TARGET_EXPFIT, TARGET_JIT, \
    TARGET_JIT_SUM = 0, 1, 2, 3, 4, 5, 6, 7
BPM_MAX_PAIRS, BPM_MAX_CR, BPM_MAX_PEERS = 8, 16, 15


class Config(C.Structure):
    _fields_ = [("algo", C.c_int32), ("n_chains", C.c_int32), ("dim", C.c_int32), ("ld", C.c_int32),
                ("del_pairs", C.c_int32), ("n_cr", C.c_int32), ("burnin_gen", C.c_int32),
                ("n_cr_gen", C.c_int32), ("shuffle", C.c_int32), ("chain_lo", C.c_int32),
                ("chain_hi", C.c_int32), ("device", C.c_int32),
                ("gamma_scale", C.c_double), ("flip", C.c_double), ("epsilon", C.c_double),
                ("u_epsilon", C.c_double), ("gamma", C.c_double), ("seed", C.c_uint64)]


class State(C.Structure):
    _fields_ = [("X", C.c_void_p), ("lnl", C.c_void_p), ("mean", C.c_void_p), ("m2", C.c_void_p),
                ("history", C.c_void_p), ("hist_len", C.c_int64), ("mom_len", C.c_int64),
                ("pending", C.c_int64)]


class Replay(C.Structure):
    _fields_ = [("flip", C.c_int32), ("shuffle_idx", C.c_void_p), ("cr_idx", C.c_void_p),
                ("z", C.c_void_p), ("fallback_dim", C.c_void_p), ("pairs", C.c_void_p),
                ("gamma_u", C.c_void_p), ("e", C.c_void_p), ("nrm", C.c_void_p),
                ("accept_u", C.c_void_p)]


class TraceOut(C.Structure):
    _fields_ = [("accept", C.c_void_p), ("lnl_prop", C.c_void_p), ("prop", C.c_void_p)]


LNL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                     C.c_void_p)

# name -> (restype, argtypes); the CPU test-suite checks every symbol of the header is here
# and exported by the library.
SIGNATURES = {
    "bpm_last_error": (C.c_char_p, []),
    "bpm_version": (C.c_int, []),
    "bpm_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "bpm_destroy": (C.c_int, [C.c_void_p]),
    "bpm_set_run_params": (C.c_int, [C.c_void_p, C.c_double, C.c_int32, C.c_double, C.c_double,
                                     C.c_double]),
    "bpm_set_fused": (C.c_int, [C.c_void_p, C.c_int32]),
    "bpm_set_target": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(C.c_double), C.c_int64]),
    "bpm_set_batched_lnl": (C.c_int, [C.c_void_p, LNL_FN, C.c_void_p]),
    "bpm_jit_compile": (C.c_int, [C.c_char_p, C.c_int32, C.c_int64, C.c_int32, C.POINTER(C.c_int32), C.c_char_p,
                                  C.c_int64]),
    "bpm_set_jit_target": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.c_int64, C.c_int32,
                                     C.POINTER(C.c_int32), C.c_char_p, C.c_int64]),
    "bpm_jit_compile_sum": (C.c_int, [C.c_char_p, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                      C.c_char_p, C.c_int64]),
    "bpm_set_jit_sum_target": (C.c_int, [C.c_void_p, C.c_char_p, C.POINTER(C.c_double), C.c_int64, C.c_int32,
                                         C.c_int32, C.POINTER(C.c_int32), C.c_char_p, C.c_int64]),
    "bpm_eval_lnl": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "bpm_set_cr_state": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "bpm_get_cr_state": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double),
                                   C.POINTER(C.c_double)]),
    "bpm_cr_partials": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "bpm_apply_cr": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bpm_get_counters": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64),
                                   C.POINTER(C.c_int32)]),
    "bpm_reset_counters": (C.c_int, [C.c_void_p]),
    "bpm_step_generations": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int64, C.c_int32,
                                       C.c_void_p]),
    "bpm_step_generation_replay": (C.c_int, [C.c_void_p, C.POINTER(State), C.POINTER(Replay),
                                             C.c_int64, C.POINTER(TraceOut), C.c_void_p]),
    "bpm_dump_draws": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int64, C.POINTER(Replay),
                                 C.POINTER(C.c_int32), C.c_void_p]),
    "bpm_begin_generation": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int64, C.POINTER(Replay),
                                       C.c_void_p]),
    "bpm_propose": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int32, C.POINTER(C.c_void_p),
                              C.POINTER(C.c_int32), C.c_void_p]),
    "bpm_accept": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int32, C.c_void_p,
                             C.POINTER(TraceOut), C.c_void_p]),
    "bpm_end_generation": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p]),
    "bpm_phase": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int32, C.c_void_p]),
    "bpm_profile": (C.c_int, [C.c_void_p, C.c_int32]),
    "bpm_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "bpm_test_philox": (C.c_int, [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "bpm_test_permutation": (C.c_int, [C.c_uint64, C.c_uint64, C.c_int32, C.POINTER(C.c_int32)]),
    "bpm_generations_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                       C.c_int32]),
    "bpm_host_entry_restart": (C.c_int, [C.c_void_p]),
    "bpm_generations_host_sharded": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p, C.c_void_p, C.c_int64,
                                               C.c_int32, C.c_void_p]),
    "bpm_dev_alloc": (C.c_int, [C.c_int32, C.c_uint64, C.POINTER(C.c_void_p)]),
    "bpm_dev_free": (C.c_int, [C.c_int32, C.c_void_p]),
    "bpm_ipc_export": (C.c_int, [C.c_int32, C.c_void_p, C.c_char_p]),
    "bpm_ipc_open": (C.c_int, [C.c_int32, C.c_char_p, C.POINTER(C.c_void_p)]),
    "bpm_ipc_close": (C.c_int, [C.c_int32, C.c_void_p]),
    "bpm_set_peers": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32]),
    "bpm_peer_copy": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p]),
    "bpm_sync_bytes": (C.c_int, [C.POINTER(C.c_uint64)]),
    "bpm_set_sync": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_int32]),
    "bpm_peer_barrier": (C.c_int, [C.c_void_p, C.c_void_p]),
    "bpm_sync_error": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "bpm_last_d2h_bytes": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "bpm_moments_from_history": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p]),
    "bpm_flush": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p]),
    "bpm_omega_track": (C.c_int, [C.c_void_p, C.c_int32]),
    "bpm_omega": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "bpm_outlier_reset": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_void_p, C.c_void_p,
                                    C.POINTER(C.c_int32), C.POINTER(C.c_double), C.c_void_p]),
    "bpm_cov_track": (C.c_int, [C.c_void_p, C.c_int32]),
    "bpm_cov_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "bpm_rhat": (C.c_int, [C.c_void_p, C.POINTER(State), C.c_int64, C.c_void_p, C.c_void_p]),
}

_lib = None


class BpmError(RuntimeError):
    pass


def _nvrtc_default():
    """NVRTC for the run-time compiled likelihoods (bpm_jit_compile): the library looks at
    $BIPYMC_B200_NVRTC, then next to nvcc, then on the loader path.  Without a toolkit, point it at
    the copy torch ships (nvidia/cuda_nvrtc), when there is one."""
    if os.environ.get("BIPYMC_B200_NVRTC"):
        return
    for b in os.environ.get("PATH", "").split(os.pathsep) + ["/usr/local/cuda/bin"]:
        if b and os.access(os.path.join(b, "nvcc"), os.X_OK):
            if os.path.exists(os.path.join(b, "..", "lib64", "libnvrtc.so.12")):
                return
            break
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.cuda_nvrtc")
    except (ImportError, ValueError):
        return
    for d in (spec.submodule_search_locations or []) if spec else []:
        p = os.path.join(d, "lib", "libnvrtc.so.12")
        if os.path.exists(p):
            os.environ["BIPYMC_B200_NVRTC"] = p
            return


def load():
    """Load the CUDA library or fail loudly (no fallback of any kind)."""
    global _lib
    if _lib is not None:
        return _lib
    _nvrtc_default()
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "bipymc_b200: CUDA library %s is missing. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        msg = load().bpm_last_error()
        raise BpmError(msg.decode() if msg else "bipymc_b200 call failed")


def dptr(arr):
    """ctypes pointer to a float64 numpy array (host)."""
    return arr.ctypes.data_as(C.POINTER(C.c_double))
