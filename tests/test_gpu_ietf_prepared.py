"""IETF verify against prepared public keys (vrfs_public_keys_prepare / vrfs_ietf_verify_prepared_batch[_dev]).

The reference in every case is vrfs_ietf_verify_batch run on the gathered keys pks[key_index]: ok flags and statuses must be
identical item by item.  Proofs come from the engine's prover (the oracle is too slow for 2^16 items); the CPU oracle is added
at small sizes."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

SUITES = [O.BANDERSNATCH, O.ED25519, O.P256, O.BANDERSNATCH_SW, O.JUBJUB, O.BABYJUBJUB]
# base field moduli, to write a non-canonical coordinate x + p
FIELD_P = {O.BANDERSNATCH: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.BANDERSNATCH_SW: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.JUBJUB: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.ED25519: 2 ** 255 - 19,
           O.P256: 0xffffffff00000001000000000000000000000000ffffffffffffffffffffffff,
           O.BABYJUBJUB: 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001}
N_MAX = 1 << 16


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def workload(eng, suite, n, n_keys, seed, with_ad=True):
    """n honest proofs by n_keys signers (random key index per item) -> dict(pks, idx, inp, out, c, s, ads)"""
    rng = np.random.default_rng(seed)
    sk_all, pks = eng.secret_from_seed(suite, [b"prepared-%d-%d-%d" % (suite, seed, k) for k in range(n_keys)])
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    data = rng.integers(0, 256, n * 8, dtype=np.uint8)
    inp, ok = eng.data_to_point(suite, (data, np.arange(n + 1, dtype=np.uint64) * 8))
    assert ok.all()
    sk = np.ascontiguousarray(sk_all[idx])
    out = eng.output(suite, sk, inp)
    ads = [rng.integers(0, 256, int(rng.integers(0, 80)), dtype=np.uint8).tobytes() for _ in range(n)] if with_ad else None
    c, s = eng.ietf_prove(suite, sk, inp, out, ads)
    return dict(pks=pks, idx=idx, inp=inp, out=out, c=c, s=s, ads=ads)


def damage(w, rng, frac=8):
    """every frac-th item (random) gets one fault: c, s, O, I, ad or a valid but wrong key index"""
    w = {k: (v.copy() if isinstance(v, np.ndarray) else (list(v) if isinstance(v, list) else v)) for k, v in w.items()}
    n, n_keys = len(w["idx"]), len(w["pks"])
    for i in rng.choice(n, max(1, n // frac), replace=False):
        kind = int(rng.integers(0, 6 if n_keys > 1 else 5))
        if kind == 0:
            w["c"][i, int(rng.integers(0, 16))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:
            w["s"][i, int(rng.integers(0, 31))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 2:
            w["out"][i] = w["out"][(i + 1) % n]
        elif kind == 3:
            w["inp"][i, 5] ^= 0x10
        elif kind == 4 and w["ads"] is not None:
            w["ads"][i] = w["ads"][i] + b"\x01"
        else:
            w["idx"][i] = (w["idx"][i] + 1) % n_keys
    return w


def reference(eng, suite, w, n=None):
    n = len(w["idx"]) if n is None else n
    ads = None if w["ads"] is None else w["ads"][:n]
    return eng.ietf_verify(suite, w["pks"][w["idx"][:n]], w["inp"][:n], w["out"][:n], w["c"][:n], w["s"][:n], ads, status=True)


def prepared(p, w, n=None):
    n = len(w["idx"]) if n is None else n
    ads = None if w["ads"] is None else w["ads"][:n]
    return p.verify(w["idx"][:n], w["inp"][:n], w["out"][:n], w["c"][:n], w["s"][:n], ads, status=True)


@pytest.mark.parametrize("suite", SUITES)
@pytest.mark.parametrize("n_keys", [1, 7, 1023])
def test_parity_with_gathered_keys(eng, suite, n_keys):
    rng = np.random.default_rng(suite * 7919 + n_keys)
    w = damage(workload(eng, suite, N_MAX, n_keys, seed=n_keys), rng)
    with eng.public_keys_prepare(suite, w["pks"]) as p:
        assert p.key_ok.all() and p.n_keys == n_keys
        for n in (1, 31, 33, 4097, N_MAX):
            ok, st = prepared(p, w, n)
            ok_r, st_r = reference(eng, suite, w, n)
            assert np.array_equal(ok, ok_r) and np.array_equal(st, st_r), (suite, n_keys, n)
            if n == N_MAX:
                assert 0 < ok.sum() < n and (st == 2).any() and (st == 1).any()
            if n == 33:          # the CPU oracle on the gathered keys
                exp = O.ietf_verify(suite, w["pks"][w["idx"][:n]], w["inp"][:n], w["out"][:n], w["c"][:n], w["s"][:n], w["ads"][:n])
                assert np.array_equal(ok, exp)


@pytest.mark.parametrize("suite", SUITES)
def test_single_faults_first_middle_last(eng, suite):
    n, n_keys = 1001, 7
    w = workload(eng, suite, n, n_keys, seed=3)
    with eng.public_keys_prepare(suite, w["pks"]) as p:
        assert prepared(p, w)[0].all()
        for kind in ("c", "s", "out", "inp", "ad", "key"):
            for i in (0, n // 2, n - 1):
                d = {k: (v.copy() if isinstance(v, np.ndarray) else list(v)) for k, v in w.items()}
                if kind in ("c", "s"):
                    d[kind][i, 3] ^= 0x40
                elif kind == "out":
                    d["out"][i] = d["out"][(i + 1) % n]
                elif kind == "inp":
                    d["inp"][i] = d["inp"][(i + 1) % n]
                elif kind == "ad":
                    d["ads"][i] = d["ads"][i] + b"x"
                else:
                    d["idx"][i] = (d["idx"][i] + 1) % n_keys
                ok, st = prepared(p, d)
                ok_r, st_r = reference(eng, suite, d)
                assert np.array_equal(ok, ok_r) and np.array_equal(st, st_r), (kind, i)
                assert ok[i] == 0 and ok.sum() == n - 1, (kind, i)


@pytest.mark.parametrize("suite", SUITES)
def test_invalid_keys_and_indices(eng, suite):
    n, n_good = 400, 4
    w = workload(eng, suite, n, n_good, seed=5)
    pks = list(w["pks"])
    p_mod = FIELD_P[suite]
    bad = pks[0].copy()                                           # non-canonical x: x + p (or p itself when that overflows)
    x = int.from_bytes(bad[:32].tobytes(), "little")
    bad[:32] = np.frombuffer((x + p_mod if x + p_mod < 2 ** 256 else p_mod).to_bytes(32, "little"), np.uint8)
    off = pks[1].copy(); off[40] ^= 0x04                          # off the curve
    zero = np.zeros(64, np.uint8)                                 # the short-Weierstrass identity; off the curve for the others
    pks = np.stack(pks + [bad, off, zero])
    with eng.public_keys_prepare(suite, pks) as p:
        assert p.key_ok.tolist() == [1] * n_good + [0, 0, 0]
        idx = w["idx"].copy()
        idx[10], idx[20], idx[30] = n_good, n_good + 1, n_good + 2
        idx[40], idx[50] = len(pks), 0xFFFFFFFF                   # out of range
        d = dict(w, idx=idx)
        ok, st = prepared(p, d)
        gathered = dict(d, pks=pks, idx=np.where(idx < len(pks), idx, 0).astype(np.uint32))
        ok_r, st_r = reference(eng, suite, gathered)
        inval = [10, 20, 30, 40, 50]
        for i in inval:
            assert ok[i] == 0 and st[i] == 2, i
        for i in (10, 20, 30):
            assert ok_r[i] == 0 and st_r[i] == 2, i
        rest = np.setdiff1d(np.arange(n), inval)
        assert np.array_equal(ok[rest], ok_r[rest]) and np.array_equal(st[rest], st_r[rest]) and ok[rest].all()


@pytest.mark.parametrize("suite", [O.BANDERSNATCH, O.ED25519, O.JUBJUB, O.BABYJUBJUB])
def test_key_with_a_torsion_component(eng, suite):
    """Y + (0, -1) = (-x, -y): on the curve but outside the prime-order subgroup, so no typed Public.  It is prepared as a valid
    key, and the proofs made for Y fail under it in both calls (its encoding enters the challenge)."""
    n, n_good = 300, 3
    w = workload(eng, suite, n, n_good, seed=21)
    p_mod = FIELD_P[suite]
    tors = w["pks"][0].copy()
    for h in (0, 32):
        v = int.from_bytes(tors[h:h + 32].tobytes(), "little")
        tors[h:h + 32] = np.frombuffer(((p_mod - v) % p_mod).to_bytes(32, "little"), np.uint8)
    pks = np.concatenate([w["pks"], tors[None]])
    with eng.public_keys_prepare(suite, pks) as p:
        assert p.key_ok.all()
        idx = np.where(w["idx"] == 0, n_good, w["idx"]).astype(np.uint32)      # every item of key 0 names its torsion twin
        d = dict(w, pks=pks, idx=idx)
        ok, st = prepared(p, d)
        ok_r, st_r = reference(eng, suite, d)
        assert np.array_equal(ok, ok_r) and np.array_equal(st, st_r)
        assert (idx == n_good).any() and (st[idx == n_good] == 1).all() and ok[idx != n_good].all()


def test_device_form_matches_host_form(eng):
    torch = pytest.importorskip("torch")
    suite = O.BANDERSNATCH
    w = damage(workload(eng, suite, 5000, 31, seed=9, with_ad=False), np.random.default_rng(1))
    w["idx"][7] = 31                                              # out of range
    with eng.public_keys_prepare(suite, w["pks"]) as p:
        ok_h, st_h = prepared(p, w)
        dev = {k: torch.from_numpy(np.ascontiguousarray(w[k])).cuda() for k in ("inp", "out", "c", "s")}
        idx = torch.from_numpy(w["idx"].view(np.int32)).cuda()
        ok = torch.zeros(len(idx), dtype=torch.uint8, device="cuda"); st = torch.zeros_like(ok)
        torch.cuda.synchronize()
        p.verify_dev(len(idx), idx, dev["inp"], dev["out"], dev["c"], dev["s"], ok, d_status=st)
        eng.sync()
        assert np.array_equal(ok.cpu().numpy(), ok_h) and np.array_equal(st.cpu().numpy(), st_h)
        assert st_h[7] == 2 and 0 < ok_h.sum() < len(ok_h)


def test_handles_and_arguments(eng):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib as L
    lib = eng._lib
    suite = O.ED25519
    w = workload(eng, suite, 4, 2, seed=11, with_ad=False)
    p = eng.public_keys_prepare(suite, w["pks"])
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    ok = np.zeros(4, np.uint8)
    args = (C.c_size_t(4), ptr(w["idx"]), ptr(w["inp"]), ptr(w["out"]), ptr(w["c"]), ptr(w["s"]), None, None, ptr(ok), None)
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, p.handle, *args) == L.OK and ok.all()
    # a handle with another context
    other = vrfs.Engine(0)
    try:
        assert lib.vrfs_ietf_verify_prepared_batch(other._ctx, p.handle, *args) == L.BAD_ARG
        assert lib.vrfs_ietf_verify_prepared_batch_dev(other._ctx, p.handle, *args) == L.BAD_ARG
    finally:
        other.close()
    # n = 0, null buffers, no handle
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, p.handle, C.c_size_t(0), None, None, None, None, None, None, None, None, None) == L.OK
    assert lib.vrfs_ietf_verify_prepared_batch_dev(eng._ctx, p.handle, C.c_size_t(0), None, None, None, None, None, None, None, None, None) == L.OK
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, p.handle, C.c_size_t(4), None, *args[2:]) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, p.handle, *args[:-2], None, None) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, None, *args) == L.BAD_ARG
    # n_keys out of 1..65536, null keys, unknown suite
    h = C.c_void_p()
    many = np.zeros((65537, 64), np.uint8)
    assert lib.vrfs_public_keys_prepare(eng._ctx, suite, C.c_size_t(0), ptr(many), None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare(eng._ctx, suite, C.c_size_t(65537), ptr(many), None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare(eng._ctx, suite, C.c_size_t(1), None, None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare(eng._ctx, 99, C.c_size_t(1), ptr(many), None, C.byref(h)) == L.BAD_ARG
    assert not h.value
    p.release()
    lib.vrfs_public_keys_release(None)
    # released after its context was destroyed
    e3 = vrfs.Engine(0)
    q = e3.public_keys_prepare(suite, w["pks"])
    e3._prepared.remove(q)
    e3.close()
    q.release()
    assert eng.ietf_verify(suite, w["pks"][w["idx"]], w["inp"], w["out"], w["c"], w["s"]).all()


def test_large_batch_one_damaged_item(eng):
    suite = O.BANDERSNATCH
    n = 1 << 20
    w = workload(eng, suite, n, 1023, seed=13, with_ad=False)
    with eng.public_keys_prepare(suite, w["pks"]) as p:
        assert prepared(p, w)[0].all()
        j = 777_777
        w["s"][j, 0] ^= 1
        ok, st = prepared(p, w)
        assert ok.sum() == n - 1 and ok[j] == 0 and st[j] == 1


def test_kernel_timings_name_the_new_kernels(eng):
    suite = O.BANDERSNATCH
    w = workload(eng, suite, 300, 5, seed=17, with_ad=False)
    eng.enable_kernel_timing(True)
    try:
        p = eng.public_keys_prepare(suite, w["pks"])
        names = [k for k, _ in eng.kernel_timings()]
        assert "key_table_powers" in names and "key_table_windows" in names
        assert prepared(p, w)[0].all()
        names = [k for k, _ in eng.kernel_timings()]
        for k in ("gather_keys", "lincomb_keyed", "lincomb<2,0>", "ietf_verify_finish"):
            assert k in names, names
        p.release()
    finally:
        eng.enable_kernel_timing(False)


def test_api_public_prepare():
    from ark_ec_vrfs_b200 import api
    s = api.Suite.bandersnatch()
    sec = api.Secret.from_seed(s, [b"api-%d" % k for k in range(3)])
    idx = np.array([0, 2, 1, 2, 0], np.uint32)
    signer = api.Secret(s, np.ascontiguousarray(sec.scalars[idx]), np.ascontiguousarray(sec.public_points[idx]))
    inp, ok = api.Input.new(s, [b"m%d" % i for i in range(5)])
    assert ok.all()
    out = signer.output(inp)
    ad = [b"", b"a", b"bb", b"", b"c"]
    proof = signer.prove(inp, out, ad)
    with sec.public().prepare() as pp:
        assert pp.key_ok.all()
        got, st = pp.verify(idx, inp, out, ad, proof, status=True)
        exp, st_e = signer.public().verify(inp, out, ad, proof, status=True)
        assert got.all() and np.array_equal(got, exp) and np.array_equal(st, st_e)
    s.engine.close()
