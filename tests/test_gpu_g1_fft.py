"""GPU: the radix-2 FFT over BLS12-381 G1 (vrfs_g1_fft_batch, Engine.g1_fft) and the Lagrange-basis SRS it derives
(api.RingContext.from_powers).  Points with known logarithms pin the transform to the Fr FFT and to its definition; true-tau powers
pin the inverse transform to [L_i(tau)] G1; at 2^16 the round trips and the ring commitment over the derived basis against the
monomial one; edge inputs (identities, P and -P, a vector of one repeated point), in == out and the argument contract."""
import ctypes as C
import hashlib

import numpy as np
import pytest

import oracle_lib as O
import vectors as V

pytestmark = pytest.mark.gpu
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
P_MOD = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
ROOT_OF_UNITY = 10238227357739495823651030575849232062558860180284477541189508159991286009131   # Fr::TWO_ADIC_ROOT_OF_UNITY
TAU = int.from_bytes(hashlib.sha512(b"vrfs-b200-g1-fft-tau").digest(), "little") % R


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def domain_gen(logn):
    return pow(ROOT_OF_UNITY, 1 << (32 - logn), R)


def rand_fr(n, tag):
    return [int.from_bytes(hashlib.sha512(tag + b"%d" % i).digest(), "little") % R for i in range(n)]


def powers(n):
    """the monomial SRS [tau^j] G1, j < n"""
    return O.g1_mul_gen(le32([pow(TAU, j, R) for j in range(n)]))


def lagrange_scalars(logn):
    """L_i(tau) = (w^i / n)(tau^n - 1)/(tau - w^i), as tests/test_gpu_ring.py computes them"""
    n = 1 << logn; w = domain_gen(logn)
    zn = (pow(TAU, n, R) - 1) * pow(n, -1, R) % R
    wi = [pow(w, i, R) for i in range(n)]
    return [zn * x * pow((TAU - x) % R, -1, R) % R for x in wi]


def negate(p):
    q = p.copy()
    if p.any():
        q[48:] = np.frombuffer(((P_MOD - int.from_bytes(p[48:].tobytes(), "little")) % P_MOD).to_bytes(48, "little"), np.uint8)
    return q


def definition(pts, inverse):
    n = len(pts); logn = n.bit_length() - 1
    w = domain_gen(logn) if not inverse else pow(domain_gen(logn), -1, R)
    s = pow(n, -1, R) if inverse else 1
    return O.msm_g1(pts, le32([s * pow(w, i * j, R) % R for i in range(n) for j in range(n)]), n)


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


@pytest.mark.parametrize("logn", [0, 1, 2, 5, 8])
def test_transform_of_known_logarithms(eng, logn):
    """P_j = [a_j] G: the transform is [fr_fft(a)] G, forward and inverse"""
    n = 1 << logn
    a = le32(rand_fr(n, b"g1fft-a%d" % logn))
    pts = O.g1_mul_gen(a)
    for inverse in (False, True):
        got = eng.g1_fft(pts, inverse=inverse)
        assert np.array_equal(got, O.g1_mul_gen(eng.fr_fft(a, inverse=inverse))), inverse
        if logn == 5:                                               # independent of fr_fft: the DFT columns through the oracle MSM
            assert np.array_equal(got, definition(pts, inverse)), inverse
    if logn == 0:
        assert np.array_equal(eng.g1_fft(pts), pts) and np.array_equal(eng.g1_fft(pts, inverse=True), pts)


@pytest.mark.parametrize("logn", [11, 14])
def test_inverse_of_the_powers_is_the_lagrange_basis(eng, logn):
    mono = powers(1 << logn)
    lag = eng.g1_fft(mono, inverse=True)
    assert np.array_equal(lag, O.g1_mul_gen(le32(lagrange_scalars(logn))))
    assert np.array_equal(eng.g1_fft(lag), mono)


def test_round_trips_and_ring_commitment_at_2p16(eng):
    """true-tau SRS at 2^16: fft(ifft) = ifft(fft) = id; a half-full ring commits to the same points over the derived Lagrange basis
    (full and delta form) as over the monomial powers"""
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import api
    n = 1 << 16
    mono = powers(n)
    lag = eng.g1_fft(mono, inverse=True)
    assert np.array_equal(eng.g1_fft(lag), mono)
    fwd = eng.g1_fft(mono)
    assert np.array_equal(eng.g1_fft(fwd, inverse=True), mono)
    _, pk, inp, _ = V.make_keys_inputs(O.BANDERSNATCH, 1024)
    tail = inp[:255]
    suite = api.Suite(vrfs.BANDERSNATCH, eng)
    keys = np.tile(pk, (n // 2 // len(pk), 1))                       # half-full ring
    ctx_lag = api.RingContext(suite, lag, True, pk[0], tail)
    ctx_mono = api.RingContext(suite, mono, False, pk[0], tail)
    try:
        want = ctx_mono.verifier_key_commitment(keys)
        assert want.any()
        assert np.array_equal(ctx_lag.verifier_key_commitment(keys, incremental=False), want)
        assert np.array_equal(ctx_lag.verifier_key_commitment(keys, incremental=True), want)
    finally:
        ctx_lag.release(); ctx_mono.release()


def test_edge_inputs(eng):
    n = 64
    g = O.g1_mul_gen(le32([11]))[0]
    zero = np.zeros((n, 96), np.uint8)
    for inverse in (False, True):
        assert not eng.g1_fft(zero, inverse=inverse).any()
    one_hot = zero.copy(); one_hot[0] = g                           # [1/n] P everywhere under the inverse
    assert np.array_equal(eng.g1_fft(one_hot, inverse=True), np.tile(O.g1_mul_gen(le32([11 * pow(n, -1, R) % R]))[0], (n, 1)))
    fwd = eng.g1_fft(np.tile(g, (n, 1)))                            # [n] P at 0, the identity elsewhere
    assert np.array_equal(fwd[0], O.g1_mul_gen(le32([11 * n]))[0]) and not fwd[1:].any()
    m = 32
    h = O.g1_mul_gen(le32([5]))[0]
    mixed = np.stack([[g, negate(g), h, negate(h)][(j * 7) % 4] for j in range(m)])
    mixed[3] = 0
    for inverse in (False, True):
        assert np.array_equal(eng.g1_fft(mixed, inverse=inverse), definition(mixed, inverse)), inverse


def test_in_place_and_argument_contract(eng):
    from ark_ec_vrfs_b200 import _lib
    lib = eng._lib
    pts = O.g1_mul_gen(le32(rand_fr(256, b"g1fft-inplace")))
    for inverse in (0, 1):
        buf = pts.copy()
        assert lib.vrfs_g1_fft_batch(eng._ctx, 8, inverse, buf.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p)) == _lib.OK
        assert np.array_equal(buf, eng.g1_fft(pts, inverse=bool(inverse)))
    src = pts[:16].copy(); p_in = src.ctypes.data_as(C.c_void_p)
    out = np.full((16, 96), 0xA5, np.uint8); p_out = out.ctypes.data_as(C.c_void_p)
    for log_n, a, b in ((-1, p_in, p_out), (25, p_in, p_out), (4, None, p_out), (4, p_in, None), (4, None, None)):
        assert lib.vrfs_g1_fft_batch(eng._ctx, log_n, 0, a, b) == _lib.BAD_ARG, log_n
        assert (out == 0xA5).all(), log_n
    assert lib.vrfs_g1_fft_batch(None, 4, 0, p_in, p_out) == _lib.BAD_ARG
    with pytest.raises(ValueError):
        eng.g1_fft(pts[:12])
    # the context still works after the refusals
    assert np.array_equal(eng.g1_fft(src), O.g1_mul_gen(eng.fr_fft(le32(rand_fr(256, b"g1fft-inplace")[:16]))))


def test_ring_context_from_powers(eng):
    """RingContext.from_powers over a 3N + 1 powers vector at N = 2^8 commits like the monomial context and like big integers"""
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import api
    logn = 8; n = 1 << logn
    srs = powers(3 * n + 1)
    _, pk, inp, _ = V.make_keys_inputs(O.BANDERSNATCH, 150)
    tail, padding = inp[:50], pk[149]
    suite = api.Suite(vrfs.BANDERSNATCH, eng)
    ctx = api.RingContext.from_powers(suite, srs, n, padding, tail)
    mono = api.RingContext(suite, srs[:n], False, padding, tail)
    lag = lagrange_scalars(logn)
    try:
        assert ctx.lagrange and ctx.domain_size == n and ctx.keyset_part_size == mono.keyset_part_size
        part = ctx.keyset_part_size
        for nk in (0, 1, 100, part):
            keys = np.tile(pk[:149], (2, 1))[:nk]
            cols = eng.ring_fixed_columns(n, part, keys, padding, tail)
            direct = O.g1_mul_gen(le32([sum(int.from_bytes(c.tobytes(), "little") * l for c, l in zip(cols[k], lag)) % R for k in range(3)]))
            got = ctx.verifier_key_commitment(keys)
            assert np.array_equal(got, mono.verifier_key_commitment(keys)), nk
            assert np.array_equal(got, direct), nk
    finally:
        ctx.release(); mono.release()
    with pytest.raises(ValueError):
        api.RingContext.from_powers(suite, srs[:n - 1], n, padding, tail)
