"""ctypes binding of libldagpu.so (include/ldagpu.h).  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libldagpu.so")

# every entry point include/ldagpu.h declares (tests check that the library exports all of them)
SYMBOLS = [
    "ldagpu_version", "ldagpu_last_error", "ldagpu_device_count", "ldagpu_create", "ldagpu_destroy",
    "ldagpu_comm_unique_id", "ldagpu_comm_init", "ldagpu_get_exchange_mode", "ldagpu_init_z_java_random", "ldagpu_set_z",
    "ldagpu_get_z", "ldagpu_sweep", "ldagpu_sweep_get_z", "ldagpu_sample_z_given_phi", "ldagpu_next_iteration",
    "ldagpu_sample_theta", "ldagpu_sample_z", "ldagpu_rebuild_counts", "ldagpu_sample_phi",
    "ldagpu_get_iteration", "ldagpu_set_iteration", "ldagpu_get_type_topic_counts",
    "ldagpu_get_topic_totals", "ldagpu_get_doc_topic_counts", "ldagpu_get_phi", "ldagpu_set_phi",
    "ldagpu_set_phi_mean_schedule", "ldagpu_get_phi_mean", "ldagpu_get_theta", "ldagpu_set_theta",
    "ldagpu_log_likelihood", "ldagpu_log_posterior", "ldagpu_abort", "ldagpu_get_abort",
    "ldagpu_get_timers", "ldagpu_get_last_call_stats",
    "ldagpu_set_z16", "ldagpu_get_z16", "ldagpu_sweep_get_z16", "ldagpu_create_multi", "ldagpu_get_shards", "ldagpu_set_phi_sampler", "ldagpu_get_count_histograms", "ldagpu_set_alpha", "ldagpu_set_beta",
    "ldagpu_set_test_documents", "ldagpu_heldout_log_likelihood",
]


class LdaGpuError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Load the in-tree libldagpu.so (build it first with `python -m ldagroupedgibbssampler_b200.build`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise LdaGpuError(
            f"{SO_PATH} is missing: build it with `python -m ldagroupedgibbssampler_b200.build` "
            "(nvcc, sm_100a).  There is no CPU fallback.")
    L = C.CDLL(SO_PATH)
    i32, i64, u64, f64, vp = C.c_int32, C.c_int64, C.c_uint64, C.c_double, C.c_void_p
    pi32, pi64, pf64 = C.POINTER(C.c_int32), C.POINTER(C.c_int64), C.POINTER(C.c_double)

    def sig(name, res, *args):
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    sig("ldagpu_version", C.c_char_p)
    sig("ldagpu_last_error", C.c_char_p, vp)
    sig("ldagpu_device_count", C.c_int)
    sig("ldagpu_create", C.c_int, i32, i32, i64, vp, vp, vp, f64, u64, i32, i32, i64, i64, C.POINTER(vp))
    sig("ldagpu_create_multi", C.c_int, i32, i32, i64, vp, vp, vp, f64, u64, i32, i32, vp, C.POINTER(vp))
    sig("ldagpu_get_shards", C.c_int, vp, pi32, vp)
    sig("ldagpu_destroy", C.c_int, vp)
    sig("ldagpu_comm_unique_id", C.c_int, vp)
    sig("ldagpu_comm_init", C.c_int, vp, i32, i32, vp)
    sig("ldagpu_init_z_java_random", C.c_int, vp, i32)
    sig("ldagpu_set_z", C.c_int, vp, vp, i32)
    sig("ldagpu_get_z", C.c_int, vp, vp)
    sig("ldagpu_set_z16", C.c_int, vp, vp, i32)
    sig("ldagpu_get_z16", C.c_int, vp, vp)
    sig("ldagpu_sweep_get_z16", C.c_int, vp, i32, pi32, vp)
    sig("ldagpu_sweep", C.c_int, vp, i32, pi32)
    sig("ldagpu_sweep_get_z", C.c_int, vp, i32, pi32, vp)
    sig("ldagpu_sample_z_given_phi", C.c_int, vp, i32, pi32)
    for n in ("ldagpu_next_iteration", "ldagpu_sample_theta", "ldagpu_sample_z", "ldagpu_rebuild_counts",
              "ldagpu_sample_phi", "ldagpu_abort"):
        sig(n, C.c_int, vp)
    sig("ldagpu_get_iteration", C.c_int, vp, pi32)
    sig("ldagpu_get_exchange_mode", C.c_int, vp, pi32)
    sig("ldagpu_set_iteration", C.c_int, vp, i32)
    for n in ("ldagpu_get_type_topic_counts", "ldagpu_get_topic_totals", "ldagpu_get_doc_topic_counts",
              "ldagpu_get_phi", "ldagpu_set_phi", "ldagpu_get_theta", "ldagpu_set_theta"):
        sig(n, C.c_int, vp, vp)
    sig("ldagpu_set_phi_mean_schedule", C.c_int, vp, i32, i32)
    sig("ldagpu_set_phi_sampler", C.c_int, vp, i32, i32)
    sig("ldagpu_get_count_histograms", C.c_int, vp, i32, vp, i32, vp)
    sig("ldagpu_set_alpha", C.c_int, vp, vp)
    sig("ldagpu_set_beta", C.c_int, vp, f64)
    sig("ldagpu_set_test_documents", C.c_int, vp, i64, vp, vp, i64, i64)
    sig("ldagpu_heldout_log_likelihood", C.c_int, vp, i32, vp, pf64)
    sig("ldagpu_get_phi_mean", C.c_int, vp, vp, pi32)
    sig("ldagpu_log_likelihood", C.c_int, vp, pf64)
    sig("ldagpu_log_posterior", C.c_int, vp, pf64)
    sig("ldagpu_get_abort", C.c_int, vp, pi32)
    sig("ldagpu_get_timers", C.c_int, vp, pf64, pf64, pf64, pf64)
    sig("ldagpu_get_last_call_stats", C.c_int, vp, pf64, pf64, pi64, pi64)
    _lib = L
    return L


def ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


SYNTH_SO_PATH = os.path.join(_HERE, "libldasynth.so")
_synth = None


def load_synth() -> C.CDLL:
    """libldasynth.so (include/ldasynth.h): host-only corpus generator, separate from the product library."""
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_SO_PATH):
            raise LdaGpuError(f"{SYNTH_SO_PATH} is missing: build it with `python -m ldagroupedgibbssampler_b200.build`")
        S = C.CDLL(SYNTH_SO_PATH)
        S.ldasynth_corpus.restype = C.c_int
        S.ldasynth_corpus.argtypes = [C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_int32,
                                      C.c_uint64, C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]
        _synth = S
    return _synth


def synth_corpus(D: int, V: int, mean_len: float, seed: int = 20190529, K_gen: int = 50,
                 sigma_len: float = 0.6, max_len: int = 20000, doc_first: int = 0):
    """LDA-generative synthetic corpus of a given shape (SURVEY 8d).  Returns (doc_offsets, tokens)."""
    S = load_synth()
    off = np.zeros(D + 1, np.int64)
    n = C.c_int64(0)
    rc = S.ldasynth_corpus(D, doc_first, V, K_gen, mean_len, sigma_len, max_len, seed, ptr(off), None, 0, C.byref(n))
    if rc:
        raise LdaGpuError("ldasynth_corpus (sizing) failed")
    tokens = np.zeros(max(n.value, 1), np.int32)
    rc = S.ldasynth_corpus(D, doc_first, V, K_gen, mean_len, sigma_len, max_len, seed, ptr(off), ptr(tokens),
                           n.value, C.byref(n))
    if rc:
        raise LdaGpuError("ldasynth_corpus failed")
    return off, tokens[: n.value]
