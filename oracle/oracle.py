"""ctypes binding of the CPU oracle (oracle/lda_oracle.c) -- TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke(), bench.py's cpu_baseline / --impl reference legs and
tools/heldout_bench.py's CPU rate import this module.  The product package (ldagroupedgibbssampler_b200)
never does.

PARITY UNPINNED against a running reference (no JDK here; see lda_oracle.h).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liblda_oracle.so")

GGS, PCGS, SPALIAS, POLYAURN = 0, 1, 2, 3
STREAM_Z, STREAM_THETA, STREAM_PHI = 1, 2, 3


def build(force: bool = False) -> str:
    """Compile the oracle with the Makefile beside this file (gcc only)."""
    srcs = [os.path.join(_HERE, f) for f in ("lda_oracle.c", "lda_oracle_sparse.c", "lda_oracle.h",
                                             "contract_math.inc")]
    stale = (not os.path.exists(_SO)) or any(
        os.path.exists(s) and os.path.getmtime(s) > os.path.getmtime(_SO) for s in srcs)
    if force or stale:
        subprocess.check_call(["make", "-C", _HERE] + (["-B"] if force else []),
                              stdout=subprocess.DEVNULL)
    return _SO


_lib = None

_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is not None:
        return _lib
    build()
    L = C.CDLL(_SO)
    i32, i64, u32, u64, f32, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_double
    vp = C.c_void_p

    def sig(name, res, *args):
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = list(args)

    sig("oracle_philox4x32_10", None, _u32p, _u32p, _u32p)
    sig("oracle_java_random_next_ints", None, i64, i32, i64, _i32p)
    sig("oracle_java_random_raw_ints", None, i64, i64, _i32p)
    sig("oracle_rebuild_counts", C.c_int, i64, _i32p, _i32p, i32, i32, _i32p, _i32p)
    sig("oracle_doc_topic_counts", None, i64, _i64p, _i32p, i32, _i32p)
    sig("oracle_c_ln_f32", f32, f32)
    sig("oracle_c_ln_f64", f64, f64)
    sig("oracle_c_exp_neg_f32", f32, f32)
    sig("oracle_c_exp_neg_f64", f64, f64)
    sig("oracle_c_cos2pi_f32", f32, u32)
    sig("oracle_c_cos2pi_f64", f64, u32)
    sig("oracle_c_gamma_f32", f32, f32, u64, u64, u32, u32)
    sig("oracle_c_gamma_f64", f64, f64, u64, u64, u32, u32)
    sig("oracle_f_gamma", f64, f64, u64, u64, u32, u32, C.c_int)
    sig("oracle_draw_topic_contract", i32, _f32p, _f32p, i32, f32)
    sig("oracle_theta_contract", None, i64, _i64p, _i32p, i32, _f64p, u64, u32, i64, _f32p)
    sig("oracle_theta_faithful", None, i64, _i64p, _i32p, i32, _f64p, u64, u32, i64, _f64p)
    sig("oracle_z_ggs_contract", None, i64, _i64p, _i32p, _i32p, i32, _f32p, _f32p, u64, u32, i64)
    sig("oracle_z_pcgs_contract", None, i64, _i64p, _i32p, _i32p, i32, _f64p, _f32p, u64, u32, i64)
    sig("oracle_z_ggs_faithful", None, i64, _i64p, _i32p, _i32p, i32, _f64p, _f64p, u64, u32, i64)
    sig("oracle_z_pcgs_faithful", None, i64, _i64p, _i32p, _i32p, i32, _f64p, _f64p, u64, u32, i64)
    sig("oracle_phi_contract", None, i32, i32, _i32p, f64, u64, u32, _f32p)
    sig("oracle_phi_faithful", None, i32, i32, _i32p, f64, u64, u32, _f64p)
    sig("oracle_poisson", i32, f64, i32, i32, u64, u64, u32, C.c_int)
    sig("oracle_phi_polya_contract", None, i32, i32, _i32p, f64, i32, u64, u32, _f32p)
    sig("oracle_phi_polya_faithful", None, i32, i32, _i32p, f64, i32, u64, u32, _f64p)
    sig("oracle_log_gamma_stirling", f64, f64)
    sig("oracle_log_likelihood", f64, i64, _i64p, _i32p, i32, i32, _i32p, _i32p, _f64p, f64)
    sig("oracle_log_likelihood_lgamma", f64, i64, _i64p, _i32p, i32, i32, _i32p, _i32p, _f64p, f64)
    sig("oracle_log_posterior", f64, i64, _i64p, _i32p, _i32p, i32, i32, _f64p, _f64p, _f64p, f64)
    for mode in ("contract", "faithful"):
        sig("oracle_heldout_l2r_" + mode, f64, i64, _i64p, _i32p, i32, i32, _i32p, _i32p, _f64p, f64, u64, u32, i64, i32,
            _f64p)
    sig("oracle_sweeps_contract", None, C.c_int, i64, i32, i32, _i64p, _i32p, _i32p, _f64p, f64,
        u64, u32, i32, _f32p, vp, _i32p, _i32p)
    sig("oracle_sweeps_faithful", None, C.c_int, i64, i32, i32, _i64p, _i32p, _i32p, _f64p, f64,
        u64, u32, i32, _f64p, vp, _i32p, _i32p)
    sig("oracle_baseline_sweeps", None, C.c_int, i64, i32, i32, _i64p, _i32p, _i32p, _f64p, f64,
        u64, i32, i32, C.POINTER(f64), C.POINTER(f64))
    sig("oracle_max_threads", C.c_int)
    sig("oracle_set_num_threads", None, C.c_int)
    sig("oracle_alias_build_contract", None, i32, i32, _f64p, _f32p, _f32p, _i32p, _f32p)
    sig("oracle_alias_sample_contract", i32, _f32p, _i32p, i32, u32, u32)
    sig("oracle_z_spalias_contract", None, i64, _i64p, _i32p, _i32p, i32, _f32p, _f32p, _i32p, _f32p, u64, u32, i64)
    sig("oracle_z_spalias_faithful", None, i64, i32, _i64p, _i32p, _i32p, i32, _f64p, _f64p, u64, u32, i64)
    _lib = L
    return L


# --------------------------------------------------------------------------------------------
# thin numpy-level helpers
# --------------------------------------------------------------------------------------------
def set_num_threads(n: int):
    lib().oracle_set_num_threads(int(n))


def philox(ctr, key):
    out = np.zeros(4, np.uint32)
    lib().oracle_philox4x32_10(np.asarray(ctr, np.uint32), np.asarray(key, np.uint32), out)
    return out


def java_next_ints(seed: int, bound: int, n: int) -> np.ndarray:
    out = np.zeros(n, np.int32)
    lib().oracle_java_random_next_ints(seed, bound, n, out)
    return out


def java_raw_ints(seed: int, n: int) -> np.ndarray:
    out = np.zeros(n, np.int32)
    lib().oracle_java_random_raw_ints(seed, n, out)
    return out


def rebuild_counts(tokens, z, V, K):
    n_wk = np.zeros((V, K), np.int32)
    n_k = np.zeros(K, np.int32)
    rc = lib().oracle_rebuild_counts(len(tokens), np.ascontiguousarray(tokens, np.int32),
                                     np.ascontiguousarray(z, np.int32), V, K, n_wk, n_k)
    if rc:
        raise ValueError("topic or type out of range")
    return n_wk, n_k


def doc_topic_counts(doc_off, z, K):
    D = len(doc_off) - 1
    out = np.zeros((D, K), np.int32)
    lib().oracle_doc_topic_counts(D, np.ascontiguousarray(doc_off, np.int64),
                                  np.ascontiguousarray(z, np.int32), K, out)
    return out


def theta_contract(doc_off, z, K, alpha, seed, sweep, doc_base=0):
    D = len(doc_off) - 1
    th = np.zeros((D, K), np.float32)
    lib().oracle_theta_contract(D, np.ascontiguousarray(doc_off, np.int64),
                                np.ascontiguousarray(z, np.int32), K,
                                np.ascontiguousarray(alpha, np.float64), seed, sweep, doc_base, th)
    return th


def theta_faithful(doc_off, z, K, alpha, seed, sweep, doc_base=0):
    D = len(doc_off) - 1
    th = np.zeros((D, K), np.float64)
    lib().oracle_theta_faithful(D, np.ascontiguousarray(doc_off, np.int64),
                                np.ascontiguousarray(z, np.int32), K,
                                np.ascontiguousarray(alpha, np.float64), seed, sweep, doc_base, th)
    return th


def z_ggs_contract(doc_off, tokens, z, K, theta, phiT, seed, sweep, token_base=0):
    z = np.array(z, np.int32, copy=True)
    lib().oracle_z_ggs_contract(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
                                np.ascontiguousarray(tokens, np.int32), z, K,
                                np.ascontiguousarray(theta, np.float32),
                                np.ascontiguousarray(phiT, np.float32), seed, sweep, token_base)
    return z


def z_pcgs_contract(doc_off, tokens, z, K, alpha, phiT, seed, sweep, token_base=0):
    z = np.array(z, np.int32, copy=True)
    lib().oracle_z_pcgs_contract(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
                                 np.ascontiguousarray(tokens, np.int32), z, K,
                                 np.ascontiguousarray(alpha, np.float64),
                                 np.ascontiguousarray(phiT, np.float32), seed, sweep, token_base)
    return z


def z_ggs_faithful(doc_off, tokens, z, K, theta, phiT, seed, sweep, token_base=0):
    z = np.array(z, np.int32, copy=True)
    lib().oracle_z_ggs_faithful(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
                                np.ascontiguousarray(tokens, np.int32), z, K,
                                np.ascontiguousarray(theta, np.float64),
                                np.ascontiguousarray(phiT, np.float64), seed, sweep, token_base)
    return z


def z_pcgs_faithful(doc_off, tokens, z, K, alpha, phiT, seed, sweep, token_base=0):
    z = np.array(z, np.int32, copy=True)
    lib().oracle_z_pcgs_faithful(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
                                 np.ascontiguousarray(tokens, np.int32), z, K,
                                 np.ascontiguousarray(alpha, np.float64),
                                 np.ascontiguousarray(phiT, np.float64), seed, sweep, token_base)
    return z


def alias_build_contract(phiT, alpha):
    """Per-type alias tables over alpha_k * phi_kw: returns (ps float32[V][K], al int32[V][K], type_norm float32[V])."""
    V, K = phiT.shape
    ps, al, tn = np.zeros((V, K), np.float32), np.zeros((V, K), np.int32), np.zeros(V, np.float32)
    lib().oracle_alias_build_contract(V, K, np.ascontiguousarray(alpha, np.float64),
                                      np.ascontiguousarray(phiT, np.float32), ps, al, tn)
    return ps, al, tn


def z_spalias_contract(doc_off, tokens, z, K, alpha, phiT, seed, sweep, token_base=0, tables=None):
    z = np.array(z, np.int32, copy=True)
    phiT = np.ascontiguousarray(phiT, np.float32)
    ps, al, tn = tables if tables is not None else alias_build_contract(phiT, alpha)
    lib().oracle_z_spalias_contract(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
                                    np.ascontiguousarray(tokens, np.int32), z, K, phiT, ps, al, tn, seed, sweep,
                                    token_base)
    return z


def z_spalias_faithful(doc_off, tokens, z, K, alpha, phiT, seed, sweep, token_base=0):
    z = np.array(z, np.int32, copy=True)
    phiT = np.ascontiguousarray(phiT, np.float64)
    lib().oracle_z_spalias_faithful(len(doc_off) - 1, phiT.shape[0], np.ascontiguousarray(doc_off, np.int64),
                                    np.ascontiguousarray(tokens, np.int32), z, K,
                                    np.ascontiguousarray(alpha, np.float64), phiT, seed, sweep, token_base)
    return z


def phi_contract(n_wk, beta, seed, sweep):
    V, K = n_wk.shape
    out = np.zeros((V, K), np.float32)
    lib().oracle_phi_contract(V, K, np.ascontiguousarray(n_wk, np.int32), beta, seed, sweep, out)
    return out


def phi_faithful(n_wk, beta, seed, sweep):
    V, K = n_wk.shape
    out = np.zeros((V, K), np.float64)
    lib().oracle_phi_faithful(V, K, np.ascontiguousarray(n_wk, np.int32), beta, seed, sweep, out)
    return out


def phi_polya_contract(n_wk, beta, seed, sweep, L=100):
    V, K = n_wk.shape
    out = np.zeros((V, K), np.float32)
    lib().oracle_phi_polya_contract(V, K, np.ascontiguousarray(n_wk, np.int32), beta, L, seed, sweep, out)
    return out


def phi_polya_faithful(n_wk, beta, seed, sweep, L=100):
    V, K = n_wk.shape
    out = np.zeros((V, K), np.float64)
    lib().oracle_phi_polya_faithful(V, K, np.ascontiguousarray(n_wk, np.int32), beta, L, seed, sweep, out)
    return out


def poisson(beta, n, seed, cell, sweep, L=100, faithful=False):
    return lib().oracle_poisson(beta, n, L, seed, cell, sweep, 1 if faithful else 0)


def log_likelihood(doc_off, z, K, V, n_wk, n_k, alpha, beta, exact_lgamma=False):
    fn = lib().oracle_log_likelihood_lgamma if exact_lgamma else lib().oracle_log_likelihood
    return fn(len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
              np.ascontiguousarray(z, np.int32), K, V, np.ascontiguousarray(n_wk, np.int32),
              np.ascontiguousarray(n_k, np.int32), np.ascontiguousarray(alpha, np.float64), beta)


def log_posterior(doc_off, tokens, z, K, V, theta, phiT, alpha, beta):
    return lib().oracle_log_posterior(
        len(doc_off) - 1, np.ascontiguousarray(doc_off, np.int64),
        np.ascontiguousarray(tokens, np.int32), np.ascontiguousarray(z, np.int32), K, V,
        np.ascontiguousarray(theta, np.float64), np.ascontiguousarray(phiT, np.float64),
        np.ascontiguousarray(alpha, np.float64), beta)


def heldout_l2r(mode, doc_off, tokens, n_wk, n_k, alpha, beta, seed, iteration, R=10, token_base=0):
    """Held-out log-likelihood by the left-to-right estimator of the test set (doc_off, tokens) under the counts
    n_wk [V][K] / n_k [K]; mode "contract" (bit-exact with the kernels) or "faithful" (fp64, libm).
    Returns (total, per-document float64 array)."""
    V, K = n_wk.shape
    D = len(doc_off) - 1
    out = np.zeros(max(D, 1), np.float64)
    tok = np.ascontiguousarray(tokens, np.int32)
    total = getattr(lib(), "oracle_heldout_l2r_" + mode)(
        D, np.ascontiguousarray(doc_off, np.int64), tok if len(tok) else np.zeros(1, np.int32), V, K,
        np.ascontiguousarray(n_wk, np.int32), np.ascontiguousarray(n_k, np.int32), np.ascontiguousarray(alpha, np.float64),
        float(beta), int(seed) & 0xFFFFFFFFFFFFFFFF, int(iteration), int(token_base), int(R), out)
    return total, out[:D]


def sweeps(mode, scheme, doc_off, tokens, z, V, K, alpha, beta, seed, first_sweep, n_sweeps, phiT):
    """Run n_sweeps whole sweeps.  Returns dict(z, phiT, theta, n_wk, n_k)."""
    D = len(doc_off) - 1
    z = np.array(z, np.int32, copy=True)
    ft = np.float32 if mode == "contract" else np.float64
    phiT = np.array(phiT, ft, copy=True)
    theta = np.zeros((D, K), ft)
    n_wk = np.zeros((V, K), np.int32)
    n_k = np.zeros(K, np.int32)
    if scheme in (SPALIAS, POLYAURN):
        # same sweep as PCGS with the sparse z-step (the alias tables are rebuilt from every new Phi);
        # POLYAURN: the rows of Phi come from the Poisson Polya urn instead of the Gammas
        polya = scheme == POLYAURN
        for s in range(n_sweeps):
            it = first_sweep + s
            if mode == "contract":
                z = z_spalias_contract(doc_off, tokens, z, K, alpha, phiT, seed, it)
            else:
                z = z_spalias_faithful(doc_off, tokens, z, K, alpha, phiT, seed, it)
            n_wk, n_k = rebuild_counts(tokens, z, V, K)
            if polya:
                phiT = phi_polya_contract(n_wk, beta, seed, it) if mode == "contract" else phi_polya_faithful(n_wk, beta, seed, it)
            else:
                phiT = phi_contract(n_wk, beta, seed, it) if mode == "contract" else phi_faithful(n_wk, beta, seed, it)
        return dict(z=z, phiT=phiT, theta=theta, n_wk=n_wk, n_k=n_k)
    fn = lib().oracle_sweeps_contract if mode == "contract" else lib().oracle_sweeps_faithful
    fn(scheme, D, V, K, np.ascontiguousarray(doc_off, np.int64),
       np.ascontiguousarray(tokens, np.int32), z, np.ascontiguousarray(alpha, np.float64), beta,
       seed, first_sweep, n_sweeps, phiT, theta.ctypes.data, n_wk, n_k)
    return dict(z=z, phiT=phiT, theta=theta, n_wk=n_wk, n_k=n_k)


def baseline_sweeps(scheme, doc_off, tokens, z, V, K, alpha, beta, seed, n_sweeps, n_threads=0):
    """Faithful sweep with the reference's threading shape; returns (z_seconds, phi_seconds, threads)."""
    z = np.array(z, np.int32, copy=True)
    zs, ps = C.c_double(0), C.c_double(0)
    nt = n_threads or lib().oracle_max_threads()
    lib().oracle_baseline_sweeps(scheme, len(doc_off) - 1, V, K,
                                 np.ascontiguousarray(doc_off, np.int64),
                                 np.ascontiguousarray(tokens, np.int32), z,
                                 np.ascontiguousarray(alpha, np.float64), beta, seed, n_sweeps, nt,
                                 C.byref(zs), C.byref(ps))
    return zs.value, ps.value, nt
