"""GPU: aggregated KZG openings (vrfs_kzg_open_aggregated_batch, PreparedBases.kzg_open_aggregated) over a monomial SRS with a
public tau, in both modes of a prepared handle (multiples table and buckets): every p_i(z_g), P_g(z_g) and
W_g = [(P_g(tau) - P_g(z_g)) / (tau - z_g)] G1 for P_g = sum nu_i p_i against big integers; byte equality with vrfs_kzg_open_batch
on the host-aggregated polynomials and on each polynomial alone; the engine's batched KZG check over C_g = sum nu_i C_i; group
counts across the MSM's 32-column slices, empty groups, mixed lengths, edge values and the argument contract."""
import ctypes as C
import hashlib
import random

import numpy as np
import pytest

import oracle_lib as O
from oracle import pairing_ref as P

pytestmark = pytest.mark.gpu
R = P.R
N = 1 << 11
CH = 1024            # KZG_OPEN_CH of csrc/kzg_open.cuh (tests/test_host_emul_kzg_aggregated.py reads it from the compiled header)
TAU = int.from_bytes(hashlib.sha512(b"vrfs-b200-kzg-open-aggregated-tau").digest(), "little") % R


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def ints(a):
    return [int.from_bytes(r.tobytes(), "little") for r in np.asarray(a, np.uint8).reshape(-1, 32)]


def ev(coeffs, x):
    acc = 0
    for c in reversed(coeffs):
        acc = (acc * x + c) % R
    return acc


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


@pytest.fixture(scope="module")
def srs():
    return O.g1_mul_gen(le32([pow(TAU, j, R) for j in range(N)]))


@pytest.fixture(scope="module", params=["table", "buckets"])
def h(eng, srs, request):
    handle = eng.msm_g1_prepare(srs) if request.param == "table" else eng.msm_g1_prepare(srs, window_bits=10)
    yield handle
    handle.release()


@pytest.fixture(scope="module")
def vk():
    return np.frombuffer(P.g2_to_bytes(P.G2_GEN), np.uint8), np.frombuffer(P.g2_to_bytes(P.g2_mul(TAU, P.G2_GEN)), np.uint8)


def aggregate(groups, nus):
    """P_g = sum nu_i p_i as ints mod r, each of the length of its group's longest polynomial (inputs reduced first)"""
    out, i = [], 0
    for g in groups:
        agg = [0] * max([len(p) for p in g], default=0)
        for p in g:
            for j, c in enumerate(p):
                agg[j] = (agg[j] + nus[i] % R * (c % R)) % R
            i += 1
        out.append(agg)
    return out


def expected(groups, zs, nus):
    """(values, agg_values, proofs) from big integers"""
    vals = [ev([c % R for c in p], z % R) for g, z in zip(groups, zs) for p in g]
    aggs = aggregate(groups, nus)
    av = [ev(a, z % R) for a, z in zip(aggs, zs)]
    ws = [(ev(a, TAU) - v) * pow(TAU - z % R, -1, R) % R for a, z, v in zip(aggs, zs, av)]
    return le32(vals), le32(av), O.g1_mul_gen(le32(ws))


def open_agg(h, groups, zs, nus):
    return h.kzg_open_aggregated([le32(p) for g in groups for p in g], [len(g) for g in groups], le32(zs), le32(nus))


def padded(polys, length):
    a = np.zeros((len(polys), length, 32), np.uint8)
    for i, p in enumerate(polys):
        if p:
            a[i, :len(p)] = le32([c % R for c in p])
    return a


def commit(h, polys):
    cols = padded(polys, N)
    return np.concatenate([h.msm(cols[i:i + 32].reshape(-1, 32), min(32, len(polys) - i)) for i in range(0, len(polys), 32)])


def ring_shape(rnd, n=N):
    """a ring prover's opening round: 8 columns of length n and one of n - 3 at zeta with the transcript's nu, the linearisation
    polynomial alone at zeta omega with nu = 1"""
    groups = [[[rnd.randrange(R) for _ in range(n)] for _ in range(8)] + [[rnd.randrange(R) for _ in range(n - 3)]],
              [[rnd.randrange(R) for _ in range(n)]]]
    return groups, [rnd.randrange(R), rnd.randrange(R)], [rnd.randrange(R) for _ in range(9)] + [1]


def test_ring_prover_shape_matches_big_integers_and_verifies(eng, h, vk):
    rnd = random.Random(1)
    groups, zs, nus = ring_shape(rnd)
    values, agg, proofs = open_agg(h, groups, zs, nus)
    v_exp, a_exp, w_exp = expected(groups, zs, nus)
    assert np.array_equal(values, v_exp)
    assert np.array_equal(agg, a_exp)
    assert np.array_equal(proofs, w_exp)
    assert ints(agg) == [sum(n * v for n, v in zip(nus[:9], ints(values[:9]))) % R, ints(values[9:])[0]]
    # C_g = sum nu_i C_i from the commitments over the same handle, and [P_g(tau)] G1
    polys = [p for g in groups for p in g]
    C_i = commit(h, polys)
    C_g = np.concatenate([O.msm_g1(C_i[:9], le32(nus[:9])), C_i[9:]])
    assert np.array_equal(C_g, O.g1_mul_gen(le32([ev(a, TAU) for a in aggregate(groups, nus)])))
    g2, tau_g2 = vk
    rs = le32([rnd.randrange(R) for _ in range(2)])
    assert eng.kzg_batch_verify(C_g, le32(zs), agg, proofs, rs, g2, tau_g2) == 1
    bad_v = agg.copy(); bad_v[0] = le32([(ints(agg[:1])[0] + 1) % R])[0]
    assert eng.kzg_batch_verify(C_g, le32(zs), bad_v, proofs, rs, g2, tau_g2) == 0
    bad_w = proofs.copy(); bad_w[1] = O.g1_mul_gen(le32([777]))[0]
    assert eng.kzg_batch_verify(C_g, le32(zs), agg, bad_w, rs, g2, tau_g2) == 0


def test_equals_open_batch(eng, h):
    """byte equality with vrfs_kzg_open_batch on the host-aggregated polynomials and on every polynomial alone"""
    rnd = random.Random(2)
    groups, zs, nus = ring_shape(rnd, CH + 37)
    values, agg, proofs = open_agg(h, groups, zs, nus)
    aggs = aggregate(groups, nus)
    for g, (a, z) in enumerate(zip(aggs, zs)):
        v1, w1 = h.kzg_open(padded([a], len(a)), le32([z]))
        assert np.array_equal(v1[0], agg[g]) and np.array_equal(w1[0], proofs[g]), g
    polys = [p for g in groups for p in g]
    zi = [z for g, z in zip(groups, zs) for _ in g]
    v_all, _ = h.kzg_open(padded(polys, CH + 37), le32(zi))            # zero padding leaves p_i(z) as it is
    assert np.array_equal(v_all, values)


@pytest.mark.parametrize("n_groups", [1, 32, 33, 70])
def test_one_polynomial_per_group_with_nu_one_is_open_batch(eng, h, n_groups):
    rnd = random.Random(100 + n_groups)
    length = CH + 5
    polys = [[rnd.randrange(R) for _ in range(length)] for _ in range(n_groups)]
    zs = [rnd.randrange(R) for _ in range(n_groups)]
    values, agg, proofs = open_agg(h, [[p] for p in polys], zs, [1] * n_groups)
    v1, w1 = h.kzg_open(padded(polys, length), le32(zs))
    assert np.array_equal(values, v1) and np.array_equal(agg, v1) and np.array_equal(proofs, w1)


@pytest.mark.parametrize("n_groups", [1, 32, 33, 70])
def test_group_counts_across_msm_slices(eng, h, vk, n_groups):
    """groups of one to three polynomials of lengths that differ by group, so that slices of 32 groups have their own longest"""
    rnd = random.Random(200 + n_groups)
    groups = [[[rnd.randrange(R) for _ in range(rnd.choice([2, CH - 1, CH + 1, 300 + g]))] for _ in range(1 + g % 3)]
              for g in range(n_groups)]
    zs = [rnd.randrange(R) for _ in range(n_groups)]
    nus = [rnd.randrange(R) for _ in range(sum(len(g) for g in groups))]
    values, agg, proofs = open_agg(h, groups, zs, nus)
    v_exp, a_exp, w_exp = expected(groups, zs, nus)
    assert np.array_equal(values, v_exp) and np.array_equal(agg, a_exp) and np.array_equal(proofs, w_exp)
    assert len({p.tobytes() for p in proofs}) == n_groups
    g2, tau_g2 = vk
    C_g = O.g1_mul_gen(le32([ev(a, TAU) for a in aggregate(groups, nus)]))
    assert eng.kzg_batch_verify(C_g, le32(zs), agg, proofs, le32([rnd.randrange(R) for _ in range(n_groups)]), g2, tau_g2) == 1


def test_shapes_and_edge_values(eng, h):
    """empty groups, lengths 0, 1, CH +- 1 and n in one group, groups of constants only, nu = 0, z = 0 and z = 1"""
    rnd = random.Random(3)
    rp = lambda n: [rnd.randrange(R) for _ in range(n)]
    groups = [[], [rp(0), rp(1), rp(CH - 1), rp(CH + 1), rp(N)], [], [rp(1), rp(0), rp(1)], [rp(CH)], [rp(0)], [rp(CH + 1), rp(7)]]
    zs = [rnd.randrange(R), 0, 5, 1, rnd.randrange(R), 9, 1]
    n_polys = sum(len(g) for g in groups)
    nus = [rnd.randrange(R) for _ in range(n_polys)]
    nus[2] = 0                                                           # the CH - 1 polynomial contributes nothing
    nus[-1] = 0
    values, agg, proofs = open_agg(h, groups, zs, nus)
    v_exp, a_exp, w_exp = expected(groups, zs, nus)
    assert np.array_equal(values, v_exp) and np.array_equal(agg, a_exp) and np.array_equal(proofs, w_exp)
    assert not agg[0].any() and not proofs[0].any() and not agg[2].any() and not proofs[2].any()   # empty groups: 0, identity
    assert not proofs[3].any() and not proofs[5].any()                    # constants only, len 0 only: the identity
    assert not values[0].any() and not values[6].any() and not values[9].any()   # len 0: the value 0
    polys = [p for g in groups for p in g]
    assert ints(values[1:5]) == [p[0] for p in polys[1:5]]               # z = 0: the constant terms
    assert ints(values[10:11]) == [sum(polys[10]) % R]                   # z = 1: the sum of the coefficients


def test_inputs_at_or_above_r_are_reduced(eng, h):
    rnd = random.Random(4)
    lift = lambda x: x + R if x + R < 1 << 256 else x
    groups = [[[rnd.randrange(R) for _ in range(CH + 3)] for _ in range(3)], [[rnd.randrange(R) for _ in range(40)]]]
    zs = [rnd.randrange(R), rnd.randrange(R)]
    nus = [rnd.randrange(R) for _ in range(4)]
    red = open_agg(h, groups, zs, nus)
    raw_groups = [[[lift(c) for c in p] for p in g] for g in groups]
    raw_groups[0][2] = [(1 << 256) - 1] * (CH + 3)
    raw = open_agg(h, raw_groups, [lift(z) for z in zs], [lift(n) for n in nus[:3]] + [R])     # nu = R: 0
    exp = expected(raw_groups, [lift(z) for z in zs], [lift(n) for n in nus[:3]] + [R])
    for got, want in zip(raw, exp):
        assert np.array_equal(got, want)
    assert np.array_equal(raw[0][:2], red[0][:2]) and np.array_equal(raw[0][3], red[0][3])
    assert not raw[1][1].any() and not raw[2][1].any()                   # nu = r is 0: P_1 = 0


def test_argument_contract(eng, srs):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib
    h = eng.msm_g1_prepare(srs[:256])
    lib = eng._lib
    u64 = lambda xs: np.asarray(xs, np.uint64)
    coeffs = np.arange(32 * 600, dtype=np.uint32).astype(np.uint8)
    zs, nus = np.full(4 * 32, 3, np.uint8), np.full(4 * 32, 1, np.uint8)
    outs = [np.full(4 * 32, 0xAB, np.uint8), np.full(4 * 32, 0xAB, np.uint8), np.full(4 * 96, 0xAB, np.uint8)]
    P_ = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)

    def call(ctx=None, handle=None, n_groups=2, n_polys=3, group_off=u64([0, 2, 3]), coeff_off=u64([0, 5, 5, 9]), coeffs=coeffs, zs=zs,
             nus=nus, values=outs[0], agg=outs[1], proofs=outs[2]):
        return lib.vrfs_kzg_open_aggregated_batch(ctx or eng._ctx, handle or h.handle, C.c_size_t(n_groups), C.c_size_t(n_polys), P_(group_off),
                                                  P_(coeff_off), P_(coeffs), P_(zs), P_(nus), P_(values), P_(agg), P_(proofs))

    def untouched():
        return all((o == 0xAB).all() for o in outs)

    try:
        bad = [dict(coeffs=None), dict(nus=None), dict(values=None), dict(zs=None), dict(proofs=None), dict(group_off=None), dict(coeff_off=None),
               dict(group_off=u64([1, 2, 3])), dict(group_off=u64([0, 4, 3])), dict(group_off=u64([0, 2, 2])), dict(group_off=u64([0, 2, 4])),
               dict(coeff_off=u64([1, 5, 5, 9])), dict(coeff_off=u64([0, 5, 4, 9])), dict(coeff_off=u64([0, 5, 5, 257 + 5])),
               dict(n_groups=1 + (1 << 16), n_polys=3), dict(n_groups=2, n_polys=1 + (1 << 16)), dict(n_groups=0, n_polys=3)]
        for kw in bad:
            assert call(**kw) == _lib.BAD_ARG, kw
            assert untouched(), kw
        # more than 2^26 coefficients in all, each polynomial within the SRS: 2^16 polynomials of 2^11 over the full SRS
        h_full = eng.msm_g1_prepare(srs)
        try:
            assert call(handle=h_full.handle, n_groups=1, n_polys=1 << 16, group_off=u64([0, 1 << 16]),
                        coeff_off=np.arange((1 << 16) + 1, dtype=np.uint64) * N) == _lib.BAD_ARG
        finally:
            h_full.release()
        assert untouched()
        with vrfs.Engine(0) as other:                                    # a handle of another context
            assert call(ctx=other._ctx) == _lib.BAD_ARG
        assert untouched()
        # n_groups = 0: OK, nothing written, nothing read
        assert call(n_groups=0, n_polys=0, group_off=None, coeff_off=None, coeffs=None, zs=None, nus=None, values=None, agg=None, proofs=None) == _lib.OK
        v, a, w = h.kzg_open_aggregated([], [], np.zeros((0, 32), np.uint8), np.zeros((0, 32), np.uint8))
        assert v.shape == (0, 32) and a.shape == (0, 32) and w.shape == (0, 96)
        with pytest.raises(ValueError):
            h.kzg_open_aggregated([le32([1])], [2], le32([1]), le32([1]))
        with pytest.raises(vrfs.VrfsError) as e:
            h.kzg_open_aggregated([np.zeros((257, 32), np.uint8)], [1], le32([1]), le32([1]))   # longer than the SRS
        assert e.value.status == _lib.BAD_ARG
        # out_agg_values may be NULL; the context still works after the refusals: p_0 = 3 + 4X at 5, nu_0 = 2
        assert call(n_groups=1, n_polys=1, group_off=u64([0, 1]), coeff_off=u64([0, 2]), coeffs=le32([3, 4]), zs=le32([5]), nus=le32([2]),
                    agg=None) == _lib.OK
        assert ints(outs[0][:32]) == [23] and np.array_equal(outs[2][:96], O.g1_mul_gen(le32([8]))[0])
        v, a, w = h.kzg_open_aggregated([le32([3, 4])], [1], le32([5]), le32([2]))
        assert ints(v) == [23] and ints(a) == [46] and np.array_equal(w, O.g1_mul_gen(le32([8])))
    finally:
        h.release()
