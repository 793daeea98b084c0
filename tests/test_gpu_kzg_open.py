"""GPU: KZG opening proofs (vrfs_kzg_open_batch, PreparedBases.kzg_open) over a monomial SRS with a public tau, in both modes of a
prepared handle (multiples table and buckets): v = p(z) and W = [(p(tau) - v) / (tau - z)] G1 against big integers, commitments
through the same handle, the engine's own batched KZG check, batch shapes around the chunk and the MSM's 32-column groups,
edge values and the argument contract."""
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
CH = 1024            # KZG_OPEN_CH of csrc/kzg_open.cuh (tests/test_host_emul_kzg.py reads it from the compiled header)
TAU = int.from_bytes(hashlib.sha512(b"vrfs-b200-kzg-open-tau").digest(), "little") % R


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


def expected(polys, zs):
    """v_i = p_i(z_i) and W_i = [(p_i(tau) - v_i) / (tau - z_i)] G1 (canonical bytes), polys as ints mod r"""
    vs = [ev(p, z) for p, z in zip(polys, zs)]
    ws = [(ev(p, TAU) - v) * pow(TAU - z, -1, R) % R for p, z, v in zip(polys, zs, vs)]
    return le32(vs), O.g1_mul_gen(le32(ws))


def commit(h, polys):
    cols = np.zeros((len(polys), N, 32), np.uint8)
    for i, p in enumerate(polys):
        if p:
            cols[i, :len(p)] = le32(p)
    return np.concatenate([h.msm(cols[i:i + 32].reshape(-1, 32), min(32, len(polys) - i)) for i in range(0, len(polys), 32)])


def rand_polys(rnd, k, length):
    return [[rnd.randrange(R) for _ in range(length)] for _ in range(k)]


def coeff_array(polys, length):
    return np.stack([le32(p) for p in polys]).reshape(len(polys), length, 32)


@pytest.mark.parametrize("length", [0, 1, 2, CH - 1, CH, CH + 1, N])
def test_openings_match_big_integers_and_verify(eng, h, vk, length):
    rnd = random.Random(length)
    k = 3
    polys = rand_polys(rnd, k, length)
    zs = [rnd.randrange(R) for _ in range(k)]
    values, proofs = h.kzg_open(coeff_array(polys, length), le32(zs))
    v_exp, w_exp = expected(polys, zs)
    assert np.array_equal(values, v_exp)
    assert np.array_equal(proofs, w_exp)
    if length <= 1:
        assert not proofs.any()                                       # the identity
    C_ = commit(h, polys)
    assert np.array_equal(C_, O.g1_mul_gen(le32([ev(p, TAU) for p in polys])))
    rs = le32([rnd.randrange(R) for _ in range(k)])
    g2, tau_g2 = vk
    assert eng.kzg_batch_verify(C_, le32(zs), values, proofs, rs, g2, tau_g2) == 1
    bad_v = values.copy(); bad_v[1] = le32([(ints(values[1:2])[0] + 1) % R])[0]
    assert eng.kzg_batch_verify(C_, le32(zs), bad_v, proofs, rs, g2, tau_g2) == 0
    bad_w = proofs.copy(); bad_w[2] = O.g1_mul_gen(le32([12345]))[0]
    assert eng.kzg_batch_verify(C_, le32(zs), values, bad_w, rs, g2, tau_g2) == 0


@pytest.mark.parametrize("k", [1, 32, 33, 70])
def test_batches_equal_single_calls(eng, h, vk, k):
    """every polynomial of a batch different; groups of 32 columns for the MSM, so 33 and 70 take two and three groups"""
    rnd = random.Random(1000 + k)
    length = CH + 37
    polys = rand_polys(rnd, k, length)
    zs = [rnd.randrange(R) for _ in range(k)]
    a, z = coeff_array(polys, length), le32(zs)
    values, proofs = h.kzg_open(a, z)
    v_exp, w_exp = expected(polys, zs)
    assert np.array_equal(values, v_exp) and np.array_equal(proofs, w_exp)
    assert len({p.tobytes() for p in proofs}) == k
    for i in range(k):
        v1, w1 = h.kzg_open(a[i:i + 1], z[i:i + 1])
        assert np.array_equal(v1[0], values[i]) and np.array_equal(w1[0], proofs[i]), i
    g2, tau_g2 = vk
    assert eng.kzg_batch_verify(commit(h, polys), z, values, proofs, le32([rnd.randrange(R) for _ in range(k)]), g2, tau_g2) == 1


def test_edge_values(eng, h):
    rnd = random.Random(5)
    length = CH + 3
    p = [rnd.randrange(R) for _ in range(length)]
    root = rnd.randrange(R)
    p_root = [(p[0] - ev(p, root)) % R] + p[1:]                       # p_root(root) = 0
    polys = [p, p, p_root, [0] * length]
    zs = [0, R - 1, root, rnd.randrange(R)]
    values, proofs = h.kzg_open(coeff_array(polys, length), le32(zs))
    v_exp, w_exp = expected(polys, zs)
    assert np.array_equal(values, v_exp) and np.array_equal(proofs, w_exp)
    assert ints(values[:1]) == [p[0]] and ints(values[2:])[0] == 0
    assert not values[3].any() and not proofs[3].any()                # the zero polynomial: v = 0, W = identity
    # coefficients and points >= r: the same openings as their residues
    raw = [[x + R if x + R < 1 << 256 else x for x in q] for q in polys[:2]] + [[(1 << 256) - 1] * length]
    raw_z = [R, (1 << 256) - 1, root + R if root + R < 1 << 256 else root]
    v_raw, w_raw = h.kzg_open(coeff_array(raw, length), le32(raw_z))
    red = [[x % R for x in q] for q in raw]
    v_red, w_red = h.kzg_open(coeff_array(red, length), le32([x % R for x in raw_z]))
    assert np.array_equal(v_raw, v_red) and np.array_equal(w_raw, w_red)
    assert np.array_equal(v_red, expected(red, [x % R for x in raw_z])[0])


def test_argument_contract(eng, srs):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib
    h = eng.msm_g1_prepare(srs[:256])
    try:
        with pytest.raises(vrfs.VrfsError) as e:
            h.kzg_open(np.zeros((1, 257, 32), np.uint8), np.zeros((1, 32), np.uint8))   # longer than the SRS
        assert e.value.status == _lib.BAD_ARG
        v, w = h.kzg_open(np.zeros((0, 5, 32), np.uint8), np.zeros((0, 32), np.uint8))
        assert v.shape == (0, 32) and w.shape == (0, 96)
        lib = eng._lib
        buf = np.zeros(4096, np.uint8); p = buf.ctypes.data_as(C.c_void_p)
        assert lib.vrfs_kzg_open_batch(eng._ctx, h.handle, C.c_size_t(0), C.c_size_t(4), None, None, None, None) == _lib.OK
        for nulls in range(4):
            args = [p] * 4
            args[nulls] = None
            assert lib.vrfs_kzg_open_batch(eng._ctx, h.handle, C.c_size_t(1), C.c_size_t(4), *args) == _lib.BAD_ARG
        assert lib.vrfs_kzg_open_batch(eng._ctx, h.handle, C.c_size_t(1 << 20), C.c_size_t(128), p, p, p, p) == _lib.BAD_ARG  # 2^27 coefficients
        with vrfs.Engine(0) as other:                                 # a handle of another context
            assert lib.vrfs_kzg_open_batch(other._ctx, h.handle, C.c_size_t(1), C.c_size_t(4), p, p, p, p) == _lib.BAD_ARG
        # the context still works after the refusals
        v, w = h.kzg_open(np.stack([le32([3, 4])]), le32([5]))
        assert ints(v) == [23] and np.array_equal(w, O.g1_mul_gen(le32([4])))
    finally:
        h.release()
