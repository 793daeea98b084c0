"""CPU check of the G1 FFT (csrc/g1_fft.cuh, the per-thread pieces of the k_g1_fft_* kernels) compiled for the host: the twiddle
multiplication [w]P (GLV halves, one shared doubling chain) against the oracle's MSM with one base, the whole transform played stage by
stage against its definition (oracle MSM columns [w^(+-ij)]), and the per-block batch-affine store with identities."""
import ctypes as C
import hashlib
import os
import random
import subprocess

import numpy as np
import pytest

import oracle_lib as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
P_MOD = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
ROOT_OF_UNITY = 10238227357739495823651030575849232062558860180284477541189508159991286009131   # Fr::TWO_ADIC_ROOT_OF_UNITY
Z2 = 0xd201000000010000 ** 2                                        # z^2, z the BLS parameter (the GLV split k = k1 + q z^2)


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def domain_gen(logn):
    return pow(ROOT_OF_UNITY, 1 << (32 - logn), R)


def rand_fr(n, tag):
    return [int.from_bytes(hashlib.sha512(tag + b"%d" % i).digest(), "little") % R for i in range(n)]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostemu_g1_fft") / "libhostemu_g1_fft.so")
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-fno-strict-aliasing", "-std=c++17", "-fPIC", "-shared", "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "hostemu_g1_fft.cpp")], check=True)
    lib = C.CDLL(so)
    lib.hostemu_g1_mul.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    lib.hostemu_g1_fft.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_char_p]
    lib.hostemu_g1_batch_affine.argtypes = [C.c_uint32, C.c_char_p, C.c_char_p]
    return lib


def emu_mul(emu, p, w):
    out = C.create_string_buffer(96)
    emu.hostemu_g1_mul(p.tobytes(), int(w).to_bytes(32, "little"), out)
    return np.frombuffer(out.raw, np.uint8)


def emu_fft(emu, pts, inverse):
    pts = np.ascontiguousarray(pts, np.uint8).reshape(-1, 96)
    out = C.create_string_buffer(pts.size)
    emu.hostemu_g1_fft(len(pts).bit_length() - 1, int(inverse), pts.tobytes(), out)
    return np.frombuffer(out.raw, np.uint8).reshape(-1, 96)


def definition(pts, inverse):
    """the transform as n oracle MSM columns over the n points: column i holds [w^(+-ij)] (times 1/n for the inverse)"""
    n = len(pts); logn = n.bit_length() - 1
    w = domain_gen(logn) if not inverse else pow(domain_gen(logn), -1, R)
    s = pow(n, -1, R) if inverse else 1
    cols = [s * pow(w, i * j, R) % R for i in range(n) for j in range(n)]
    return O.msm_g1(pts, le32(cols), n)


def test_twiddle_multiplication_matches_the_oracle(emu):
    rnd = random.Random(5)
    pts = O.g1_mul_gen(le32([rnd.randrange(1, R) for _ in range(3)]))
    w4 = domain_gen(6) ** 16 % R                                    # w^(n/4) at n = 64: a square root of -1
    assert w4 * w4 % R == R - 1
    scalars = [1, R - 1, w4, 0, Z2, 3 * Z2, Z2 - 1, Z2 + 1, 12345, (1 << 128) - 1, R - Z2]   # k1 = 0 (w = q z^2), q = 0 (w < z^2)
    scalars += [rnd.randrange(R) for _ in range(8)] + [pow(domain_gen(11), j, R) for j in (1, 2, 511, 1023)]
    for p in pts:
        for w in scalars:
            assert np.array_equal(emu_mul(emu, p, w), O.msm_g1(p.reshape(1, 96), le32([w]))[0]), hex(w)
    # the identity stays the identity
    assert not emu_mul(emu, np.zeros(96, np.uint8), rnd.randrange(R)).any()


@pytest.mark.parametrize("logn", [0, 1, 2, 3, 6])
@pytest.mark.parametrize("inverse", [0, 1])
def test_transform_matches_its_definition(emu, logn, inverse):
    n = 1 << logn
    pts = O.g1_mul_gen(le32(rand_fr(n, b"g1fft%d" % logn)))
    if n >= 4:                                                      # identities and repeated points among random ones
        pts[1] = 0; pts[n - 1] = pts[2]; pts[n // 2] = 0
    assert np.array_equal(emu_fft(emu, pts, inverse), definition(pts, inverse))


def test_transform_edge_inputs(emu):
    n = 16
    g = O.g1_mul_gen(le32([7]))[0]
    neg = g.copy(); neg[48:] = np.frombuffer(((P_MOD - int.from_bytes(g[48:].tobytes(), "little")) % P_MOD).to_bytes(48, "little"), np.uint8)
    zero = np.zeros((n, 96), np.uint8)
    for inverse in (0, 1):
        assert not emu_fft(emu, zero, inverse).any()                # all identity
    one_hot = zero.copy(); one_hot[0] = g
    assert np.array_equal(emu_fft(emu, one_hot, 1), np.tile(O.g1_mul_gen(le32([7 * pow(n, -1, R) % R]))[0], (n, 1)))
    tiled = np.tile(g, (n, 1))                                      # a - t = 0 in every butterfly but the first column
    fwd = emu_fft(emu, tiled, 0)
    assert np.array_equal(fwd[0], O.g1_mul_gen(le32([7 * n]))[0]) and not fwd[1:].any()
    mixed = np.where(np.arange(n)[:, None] % 3 == 0, g, neg).astype(np.uint8)
    for inverse in (0, 1):
        assert np.array_equal(emu_fft(emu, mixed, inverse), definition(mixed, inverse))
        assert np.array_equal(emu_fft(emu, emu_fft(emu, mixed, inverse), 1 - inverse), mixed)


def test_batch_affine_store_with_identities(emu):
    """projective (lambda x : lambda y : lambda) with random lambda, identities (0 : y : 0) interleaved, one all-identity block and a
    short last block -> the affine points (zeros for the identity)"""
    bt = emu.hostemu_g1_fft_store_threads()
    rnd = random.Random(9)
    n = 2 * bt + bt + 5
    aff = O.g1_mul_gen(le32([rnd.randrange(1, R) for _ in range(n)]))
    ident = [i for i in range(n) if (bt <= i < 2 * bt) or i % 7 == 3 or i == n - 1]
    aff[ident] = 0
    proj = bytearray()
    for i in range(n):
        if i in ident:
            proj += bytes(48) + rnd.randrange(1, P_MOD).to_bytes(48, "little") + bytes(48)
            continue
        x = int.from_bytes(aff[i, :48].tobytes(), "little"); y = int.from_bytes(aff[i, 48:].tobytes(), "little")
        lam = rnd.randrange(1, P_MOD)
        proj += (x * lam % P_MOD).to_bytes(48, "little") + (y * lam % P_MOD).to_bytes(48, "little") + lam.to_bytes(48, "little")
    out = C.create_string_buffer(96 * n)
    emu.hostemu_g1_batch_affine(n, bytes(proj), out)
    assert np.array_equal(np.frombuffer(out.raw, np.uint8).reshape(n, 96), aff)
