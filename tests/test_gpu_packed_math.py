"""Bit-exactness of the fp32 primitives the theta draw runs in packed FP32 or without the slow-path check
(ldagroupedgibbssampler_b200/csrc/contract_math.cuh), over every operand they can receive:

* div_ln, the division (m - 1) / (m + 1) of c_ln, against IEEE float32 division, for all 2^23 values of m in
  [sqrt(1/2), sqrt(2));
* sqrt_bm, the Box-Muller radius, against IEEE float32 square root, for all 2^23 arguments -2 ln(u), u a uniform23;
* the packed forms against the scalar ones: div_ln2 and sqrt_bm2 on the same operands, the packed logarithm on all
  2^23 uniform23 values, the packed cosine on all 2^26 (octant, fraction) inputs, and the packed squeeze attempt
  against gamma_attempt_squeeze<float> on Philox blocks at alpha in {1e-4, 0.05, 1, 200}.

Every packed call pairs input i (first half) with input (i + shift) mod n (second half), so each input is checked in
both halves and the halves of one call differ (octant, sine or cosine polynomial, boost or not).

A small harness that includes contract_math.cuh is compiled with the library's nvcc flags into a temporary directory
and loaded with ctypes."""
import ctypes as C
import subprocess

import numpy as np
import pytest

gpu = pytest.mark.gpu

HARNESS = r"""
#include <cuda_runtime.h>
#include "contract_math.cuh"
using namespace ldagpu;
typedef unsigned long long u64;

__device__ __forceinline__ uint32_t fbits(float x) { return __float_as_uint(x); }
__device__ __forceinline__ void miss(u64 *bad, bool differs) { if (differs) atomicAdd(bad, 1ull); }

__global__ void k_div(const float *a, const float *b, float *q, int n, int shift, u64 *bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = (i + shift) % n;
    const float qi = div_ln(a[i], b[i]), qj = div_ln(a[j], b[j]);
    q[i] = qi;
    const float2 p = div_ln2(make_float2(a[i], a[j]), make_float2(b[i], b[j]));
    miss(bad, fbits(p.x) != fbits(qi) || fbits(p.y) != fbits(qj));
}

__device__ __forceinline__ float radius_arg(int i) { return __fmul_rn(-2.0f, c_ln<float>(uniform23((uint32_t)i << 9))); }

__global__ void k_sqrt(float *x, float *y, int n, int shift, u64 *bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = (i + shift) % n;
    const float xi = radius_arg(i), xj = radius_arg(j);
    const float yi = sqrt_bm(xi), yj = sqrt_bm(xj);
    x[i] = xi;
    y[i] = yi;
    const float2 p = sqrt_bm2(make_float2(xi, xj));
    miss(bad, fbits(p.x) != fbits(yi) || fbits(p.y) != fbits(yj));
}

__global__ void k_ln(int n, int shift, u64 *bad)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = (i + shift) % n;
    const uint32_t wi = (uint32_t)i << 9, wj = (uint32_t)j << 9;
    const float2 u = uniform23_2(wi, wj);
    const float2 p = c_ln_normal2(u);
    miss(bad, fbits(u.x) != fbits(uniform23(wi)) || fbits(u.y) != fbits(uniform23(wj)) ||
              fbits(p.x) != fbits(c_ln<float>(uniform23(wi))) || fbits(p.y) != fbits(c_ln<float>(uniform23(wj))));
}

// input i of 2^26: octant i >> 23, 23-bit fraction i & (2^23 - 1) (c_cos2pi<float> reads bits 31..29 and 28..6)
__device__ __forceinline__ uint32_t angle_word(uint32_t i) { return ((i >> 23) << 29) | ((i & 0x7fffffu) << 6); }

__global__ void k_cos(uint32_t n, uint32_t shift, u64 *bad)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t wi = angle_word(i), wj = angle_word((i + shift) % n);
    const float2 p = c_cos2pi2(wi, wj);
    miss(bad, fbits(p.x) != fbits(c_cos2pi<float>(wi)) || fbits(p.y) != fbits(c_cos2pi<float>(wj)));
}

// pair i: cell 2i with alpha[i % na], cell 2i + 1 with alpha[(i / na) % na] -- every ordered pair of shapes
__global__ void k_attempt(const float *alpha, int na, int n, uint32_t k0, uint32_t k1, u64 *bad, u64 *accepted)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    bool b0, b1;
    float d0, c0, i0, d1, c1, i1;
    gamma_setup<float>(alpha[i % na], b0, d0, c0, i0);
    gamma_setup<float>(alpha[(i / na) % na], b1, d1, c1, i1);
    const uint4 r0 = philox4x32_10(2u * i, 0u, 7u, STREAM_THETA << 24, k0, k1);
    const uint4 r1 = philox4x32_10(2u * i + 1u, 0u, 7u, STREAM_THETA << 24, k0, k1);
    bool p0, p1;
    float2 g;
    gamma_attempt_squeeze2(make_float2(d0, d1), make_float2(c0, c1), make_float2(i0, i1), r0, r1, p0, p1, g);
    float g0 = 0.0f, g1 = 0.0f;
    const bool s0 = gamma_attempt_squeeze<float>(b0, d0, c0, i0, r0, g0);
    const bool s1 = gamma_attempt_squeeze<float>(b1, d1, c1, i1, r1, g1);
    miss(bad, p0 != s0 || p1 != s1 || (s0 && fbits(g.x) != fbits(g0)) || (s1 && fbits(g.y) != fbits(g1)));
    if (s0) atomicAdd(accepted, 1ull);
    if (s1) atomicAdd(accepted, 1ull);
}

static int grid(long long n) { return (int)((n + 255) / 256); }

struct Counters {
    u64 *d = nullptr;
    cudaError_t alloc() { cudaError_t e = cudaMalloc(&d, 2 * sizeof(u64)); return e ? e : cudaMemset(d, 0, 2 * sizeof(u64)); }
    cudaError_t fetch(u64 *out) { cudaError_t e = cudaMemcpy(out, d, 2 * sizeof(u64), cudaMemcpyDeviceToHost); cudaFree(d); return e; }
};

extern "C" int check_div(const float *a, const float *b, float *q, int n, int shift, u64 *counts)
{
    float *da, *db, *dq;
    Counters c;
    if (cudaMalloc(&da, n * 4) || cudaMalloc(&db, n * 4) || cudaMalloc(&dq, n * 4) || c.alloc()) return 1;
    cudaMemcpy(da, a, n * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(db, b, n * 4, cudaMemcpyHostToDevice);
    k_div<<<grid(n), 256>>>(da, db, dq, n, shift, c.d);
    cudaError_t e = cudaMemcpy(q, dq, n * 4, cudaMemcpyDeviceToHost);
    e = e ? e : c.fetch(counts);
    cudaFree(da); cudaFree(db); cudaFree(dq);
    return (int)e;
}

extern "C" int check_sqrt(float *x, float *y, int n, int shift, u64 *counts)
{
    float *dx, *dy;
    Counters c;
    if (cudaMalloc(&dx, n * 4) || cudaMalloc(&dy, n * 4) || c.alloc()) return 1;
    k_sqrt<<<grid(n), 256>>>(dx, dy, n, shift, c.d);
    cudaError_t e = cudaMemcpy(x, dx, n * 4, cudaMemcpyDeviceToHost);
    e = e ? e : cudaMemcpy(y, dy, n * 4, cudaMemcpyDeviceToHost);
    e = e ? e : c.fetch(counts);
    cudaFree(dx); cudaFree(dy);
    return (int)e;
}

extern "C" int check_ln(int n, int shift, u64 *counts)
{
    Counters c;
    if (c.alloc()) return 1;
    k_ln<<<grid(n), 256>>>(n, shift, c.d);
    return (int)c.fetch(counts);
}

extern "C" int check_cos(unsigned n, unsigned shift, u64 *counts)
{
    Counters c;
    if (c.alloc()) return 1;
    k_cos<<<grid(n), 256>>>(n, shift, c.d);
    return (int)c.fetch(counts);
}

extern "C" int check_attempt(const float *alpha, int na, int n, unsigned k0, unsigned k1, u64 *counts)
{
    float *dal;
    Counters c;
    if (cudaMalloc(&dal, na * 4) || c.alloc()) return 1;
    cudaMemcpy(dal, alpha, na * 4, cudaMemcpyHostToDevice);
    k_attempt<<<grid(n), 256>>>(dal, na, n, k0, k1, c.d, c.d + 1);
    cudaError_t e = c.fetch(counts);
    cudaFree(dal);
    return (int)e;
}
"""

N23 = 1 << 23
F32 = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
U64 = np.ctypeslib.ndpointer(np.uint64, flags="C_CONTIGUOUS")


@pytest.fixture(scope="module")
def H(tmp_path_factory):
    from ldagroupedgibbssampler_b200 import build as B
    d = tmp_path_factory.mktemp("packed_math")
    src, so = d / "harness.cu", d / "harness.so"
    src.write_text(HARNESS)
    cmd = [B.NVCC] + B.ARCH + B.NVFLAGS + ["-I", B.CSRC, "-shared", "-o", str(so), str(src)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    lib = C.CDLL(str(so))
    lib.check_div.argtypes = [F32, F32, F32, C.c_int, C.c_int, U64]
    lib.check_sqrt.argtypes = [F32, F32, C.c_int, C.c_int, U64]
    lib.check_ln.argtypes = [C.c_int, C.c_int, U64]
    lib.check_cos.argtypes = [C.c_uint, C.c_uint, U64]
    lib.check_attempt.argtypes = [F32, C.c_int, C.c_int, C.c_uint, C.c_uint, U64]
    return lib


def _bits(x):
    return np.asarray(x, np.float32).view(np.uint32)


@gpu
def test_div_ln_is_ieee_division_for_every_m(H):
    m = (np.arange(N23, dtype=np.uint32) + np.uint32(0x3F3504F3)).view(np.float32)   # c_ln's m, every value
    a, b = m - np.float32(1.0), m + np.float32(1.0)
    q = np.empty(N23, np.float32)
    counts = np.zeros(2, np.uint64)
    assert H.check_div(a, b, q, N23, 1234567, counts) == 0
    bad = np.flatnonzero(_bits(q) != _bits(a / b))
    assert bad.size == 0, f"{bad.size} quotients differ, first m = {m[bad[0]]!r}"
    assert counts[0] == 0, f"packed division differs from the scalar one on {counts[0]} pairs"


@gpu
def test_sqrt_bm_is_ieee_sqrt_for_every_radius_argument(H):
    x, y = np.empty(N23, np.float32), np.empty(N23, np.float32)
    counts = np.zeros(2, np.uint64)
    assert H.check_sqrt(x, y, N23, 1234567, counts) == 0
    assert 1.1e-7 < x.min() and x.max() < 33.4            # the range the fast path is specialised for
    bad = np.flatnonzero(_bits(y) != _bits(np.sqrt(x)))
    assert bad.size == 0, f"{bad.size} roots differ, first argument {x[bad[0]]!r}"
    assert counts[0] == 0, f"packed root differs from the scalar one on {counts[0]} pairs"


@gpu
def test_packed_ln_matches_scalar_for_every_uniform(H):
    counts = np.zeros(2, np.uint64)
    assert H.check_ln(N23, 1234567, counts) == 0
    assert counts[0] == 0, f"packed ln differs from c_ln<float> on {counts[0]} pairs"


@gpu
def test_packed_cos_matches_scalar_for_every_angle(H):
    n = 1 << 26
    counts = np.zeros(2, np.uint64)
    assert H.check_cos(n, 3 * N23 + 1234567, counts) == 0    # the halves of a call fall in different octants
    assert counts[0] == 0, f"packed cos differs from c_cos2pi<float> on {counts[0]} pairs"


@gpu
@pytest.mark.parametrize("seed", [2019, 0xDEADBEEF])
def test_packed_squeeze_attempt_matches_scalar(H, seed):
    alpha = np.array([1e-4, 0.05, 1.0, 200.0], np.float32)
    n = 1 << 22
    counts = np.zeros(2, np.uint64)
    assert H.check_attempt(alpha, len(alpha), n, seed & 0xFFFFFFFF, (seed * 2654435761) & 0xFFFFFFFF, counts) == 0
    assert counts[0] == 0, f"packed attempt differs from gamma_attempt_squeeze<float> on {counts[0]} pairs"
    assert counts[1] > n, counts                              # the squeeze accepts most candidates: g was compared
