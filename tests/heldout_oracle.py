"""ctypes binding of tests/heldout_oracle.c, the CPU restatement of the held-out log-likelihood (DESIGN.md 4.8) --
TEST INFRASTRUCTURE ONLY (tests/ and tools/heldout_bench.py's CPU rate).

The library is compiled on first use with the flags of oracle/Makefile into a directory under the system temporary
directory, keyed by a hash of its sources, so the repository tree is never written."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "heldout_oracle.c")
_INC = os.path.join(os.path.dirname(_HERE), "oracle", "contract_math.inc")
# oracle/Makefile's flags: the contract arithmetic must not be fused behind our back; fmaf() is explicit
CFLAGS = ["-O2", "-std=gnu11", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-mfma", "-mavx2", "-fopenmp",
          "-Wall", "-Wextra", "-Wno-unused-function", "-Wno-unknown-pragmas"]

_lib = None


def build() -> str:
    h = hashlib.sha256()
    for p in (_SRC, _INC):
        with open(p, "rb") as f:
            h.update(f.read())
    h.update(" ".join(CFLAGS).encode())
    out_dir = os.path.join(tempfile.gettempdir(), "ldagpu_heldout_oracle_" + h.hexdigest()[:16])
    so = os.path.join(out_dir, "libheldout_oracle.so")
    if not os.path.exists(so):
        os.makedirs(out_dir, exist_ok=True)
        cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
        tmp = so + ".%d.tmp" % os.getpid()
        subprocess.check_call([cc] + CFLAGS + ["-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)   # concurrent builders each write their own file; the rename is atomic
    return so


_i32p = np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
_f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(np.float64, flags="C_CONTIGUOUS")


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        i32, i64, u32, u64, f32, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_uint64, C.c_float, C.c_double
        for n in ("heldout_l2r_contract", "heldout_l2r_faithful"):
            fn = getattr(L, n)
            fn.restype = f64
            fn.argtypes = [i64, _i64p, _i32p, i32, i32, _i32p, _i32p, _f64p, f64, u64, u32, i64, i32, _f64p]
        L.heldout_philox4x32_10.restype = None
        L.heldout_philox4x32_10.argtypes = [_u32p, _u32p, _u32p]
        L.heldout_c_ln_f64.restype = f64
        L.heldout_c_ln_f64.argtypes = [f64]
        L.heldout_draw_lanes.restype = i32
        L.heldout_draw_lanes.argtypes = [_f32p, _f32p, i32, f32, C.POINTER(C.c_float)]
        _lib = L
    return _lib


def heldout_l2r(mode, doc_off, tokens, n_wk, n_k, alpha, beta, seed, iteration, R=10, token_base=0):
    """Held-out log-likelihood by the left-to-right estimator of the test set (doc_off, tokens) under the counts
    n_wk [V][K] / n_k [K]; mode "contract" (bit-exact with the kernels) or "faithful" (fp64, libm).
    Returns (total, per-document float64 array)."""
    V, K = n_wk.shape
    D = len(doc_off) - 1
    out = np.zeros(max(D, 1), np.float64)
    fn = lib().heldout_l2r_contract if mode == "contract" else lib().heldout_l2r_faithful
    tok = np.ascontiguousarray(tokens, np.int32)
    total = fn(D, np.ascontiguousarray(doc_off, np.int64), tok if len(tok) else np.zeros(1, np.int32), V, K,
               np.ascontiguousarray(n_wk, np.int32), np.ascontiguousarray(n_k, np.int32),
               np.ascontiguousarray(alpha, np.float64), float(beta), int(seed) & 0xFFFFFFFFFFFFFFFF, int(iteration),
               int(token_base), int(R), out)
    return total, out[:D]


def philox(ctr, key):
    out = np.zeros(4, np.uint32)
    lib().heldout_philox4x32_10(np.asarray(ctr, np.uint32), np.asarray(key, np.uint32), out)
    return out


def c_ln_f64(x: float) -> float:
    return lib().heldout_c_ln_f64(float(x))


def draw_lanes(a, phirow, K, U):
    """(topic, S) of the K <= 1024 contract draw"""
    S = C.c_float(0)
    k = lib().heldout_draw_lanes(np.ascontiguousarray(a, np.float32), np.ascontiguousarray(phirow, np.float32), K,
                                 float(U), C.byref(S))
    return k, S.value
