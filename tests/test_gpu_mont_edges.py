"""Montgomery product and square of BLS12-381 Fr (the Bandersnatch base field) on the GPU at the edges of their reduction rows.

p = 1 - 2^32 (mod 2^64), so the lowest limb pair of every reduction row is formed from the row's column value by a borrow chain
(arith.cuh RedRows) instead of a multiply.  A row whose multiplier m is 0 takes a different path through that chain, and random
operands almost never reach it: the operands here are built limb by limb, by emulating the interleaved rows in Python, so that a
chosen row has m = 0.  Also: 0, 1, p - 1, R mod p and their products.  The kernels are compiled by the test from a small .cu that
includes arith.cuh; the results are checked against Python integers."""
import ctypes as C
import os
import random
import subprocess
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "ark_ec_vrfs_b200", "csrc")

P = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001
N = 8
M32 = (1 << 32) - 1
R = 1 << (32 * N)
RINV = pow(R, -1, P)

SRC = r"""
#include <cuda_runtime.h>
#include "arith.cuh"
#include "gen/field_consts.cuh"
using namespace vrfs;
typedef Fp<BlsFr> F;
__global__ void k_mul(uint32_t n, const F* a, const F* b, F* o) { uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) o[i] = a[i] * b[i]; }
__global__ void k_sqr(uint32_t n, const F* a, F* o) { uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) o[i] = sqr(a[i]); }
extern "C" int run(int op, uint32_t n, const uint32_t* a, const uint32_t* b, uint32_t* out) {
  F *da, *db, *dout;
  size_t bytes = (size_t)n * sizeof(F);
  if (cudaMalloc(&da, bytes) || cudaMalloc(&db, bytes) || cudaMalloc(&dout, bytes)) return 1;
  cudaMemcpy(da, a, bytes, cudaMemcpyHostToDevice);
  cudaMemcpy(db, b, bytes, cudaMemcpyHostToDevice);
  if (op == 0) k_mul<<<(n + 127) / 128, 128>>>(n, da, db, dout); else k_sqr<<<(n + 127) / 128, 128>>>(n, da, dout);
  int err = (int)cudaDeviceSynchronize();
  cudaMemcpy(out, dout, bytes, cudaMemcpyDeviceToHost);
  cudaFree(da); cudaFree(db); cudaFree(dout);
  return err;
}
"""


def limbs(x):
    return [(x >> (32 * i)) & M32 for i in range(N)]


def row_multipliers(a, b):
    """multipliers m_0..m_(N-1) of the interleaved Montgomery rows of a * b (the square reduces a^2 with the same m_i):
    m_i = limb i of -(a * (b mod 2^(32(i+1)))) / p mod 2^(32(i+1))"""
    out = []
    for i in range(N):
        mod = 1 << (32 * (i + 1))
        q = (-a * (b % mod) * pow(P, -1, mod)) % mod
        out.append(q >> (32 * i))
    return out


def sqr_row_multipliers(a):
    t = a * a
    return [((-t * pow(P, -1, 1 << (32 * (i + 1)))) % (1 << (32 * (i + 1)))) >> (32 * i) for i in range(N)]


def mul_with_zero_row(rng, row):
    """(a, b) < p whose product has m_row = 0: m_row is (const - a_0 b_row) mod 2^32 with p^-1 = 1 mod 2^32, a_0 odd"""
    while True:
        a = rng.randrange(P) | 1
        b = rng.randrange(P >> 32)           # top limb small: choosing limb `row` below keeps b < p
        b &= ~(M32 << (32 * row))
        c = row_multipliers(a, b)[row]
        b |= (c * pow(a & M32, -1, 1 << 32) % (1 << 32)) << (32 * row)
        if b < P and row_multipliers(a, b)[row] == 0:
            return a, b


def sqr_with_zero_row(rng, row):
    """a < p whose square has m_row = 0 (row 0: a_0 = 0 mod 2^16; later rows: m_row is linear in a_row with factor -2 a_0)"""
    while True:
        a = rng.randrange(P >> 32)
        if row == 0:
            a = (a & ~M32) | (rng.randrange(1 << 16) << 16)
        else:
            a |= 1
            a &= ~(M32 << (32 * row))
            c = sqr_row_multipliers(a)[row]
            if c & 1:
                continue
            k = (c >> 1) * pow(a & M32, -1, 1 << 31) % (1 << 31)
            a |= k << (32 * row)
        if a < P and sqr_row_multipliers(a)[row] == 0:
            return a


def cases():
    rng = random.Random(20261020)
    special = [0, 1, P - 1, R % P, P - (R % P), 2, (P - 1) // 2, R * R % P]
    pairs = [(x, y) for x in special for y in special]
    pairs += [mul_with_zero_row(rng, i) for i in range(N) for _ in range(4)]
    pairs += [(rng.randrange(P), rng.randrange(P)) for _ in range(256)]
    sq = special + [sqr_with_zero_row(rng, i) for i in range(N) for _ in range(4)] + [rng.randrange(P) for _ in range(256)]
    return pairs, sq


@pytest.fixture(scope="module")
def lib():
    from ark_ec_vrfs_b200 import build
    tmp = tempfile.mkdtemp(prefix="vrfs_mont_edges_")
    cu, so = os.path.join(tmp, "mont_edges.cu"), os.path.join(tmp, "libmont_edges.so")
    with open(cu, "w") as f:
        f.write(SRC)
    subprocess.run([build.nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                    "-shared", "-I", CSRC, "-o", so, cu], check=True)
    return C.CDLL(so)


def run(lib, op, xs, ys):
    a = np.array([limbs(x) for x in xs], dtype=np.uint32)
    b = np.array([limbs(y) for y in ys], dtype=np.uint32)
    out = np.zeros_like(a)
    p = lambda v: v.ctypes.data_as(C.c_void_p)
    assert lib.run(op, C.c_uint32(len(xs)), p(a), p(b), p(out)) == 0
    return [sum(int(w) << (32 * i) for i, w in enumerate(row)) for row in out]


def test_case_builders_reach_zero_rows():
    pairs, sq = cases()
    hit = {i for a, b in pairs for i, m in enumerate(row_multipliers(a, b)) if m == 0}
    assert set(range(N)) <= hit
    assert set(range(N)) <= {i for a in sq for i, m in enumerate(sqr_row_multipliers(a)) if m == 0}


@pytest.mark.gpu
def test_product_at_reduction_edges(lib):
    pairs, _ = cases()
    got = run(lib, 0, [a for a, _ in pairs], [b for _, b in pairs])
    for (a, b), g in zip(pairs, got):
        assert g == a * b * RINV % P, (hex(a), hex(b))


@pytest.mark.gpu
def test_square_at_reduction_edges(lib):
    _, sq = cases()
    got = run(lib, 1, sq, sq)
    for a, g in zip(sq, got):
        assert g == a * a * RINV % P, hex(a)
