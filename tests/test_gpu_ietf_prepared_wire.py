"""Serialised IETF signatures verified against keys prepared from their encodings (vrfs_public_keys_prepare_encoded /
vrfs_ietf_verify_prepared_wire_batch).

The reference in every case is vrfs_ietf_verify_wire_batch on the gathered encodings enc[key_index]: ok flags, hashes and statuses
must be identical item by item.  Signatures come from the engine's signer (the oracle is too slow for 2^16 items); the CPU oracle
is added at small sizes."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
SUITES = [O.BANDERSNATCH, O.ED25519, O.P256, O.BANDERSNATCH_SW, O.JUBJUB, O.BABYJUBJUB]
TE_SUITES = [O.BANDERSNATCH, O.ED25519, O.JUBJUB, O.BABYJUBJUB]     # (x, y) + (0, -1) = (-x, -y) is their affine 2-torsion shift
FIELD_P = {O.BANDERSNATCH: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.BANDERSNATCH_SW: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.JUBJUB: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.ED25519: 2 ** 255 - 19,
           O.P256: 0xffffffff00000001000000000000000000000000ffffffffffffffffffffffff,
           O.BABYJUBJUB: 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001}
N_MAX = 1 << 16
DAMAGE = ("out_noncanonical", "out_offcurve", "out_torsion", "c", "s", "s_ge_r", "data", "ad", "key")


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def workload(eng, suite, n, n_keys, seed, with_ad=True):
    """n honest signatures by n_keys signers (random key index per item) -> dict(enc, idx, data, off, sig, ads)"""
    rng = np.random.default_rng(seed)
    sk_all, pks = eng.secret_from_seed(suite, [b"prepared-wire-%d-%d-%d" % (suite, seed, k) for k in range(n_keys)])
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    data = rng.integers(0, 256, n * 8, dtype=np.uint8)
    off = np.arange(n + 1, dtype=np.uint64) * 8
    ads = [rng.integers(0, 256, int(rng.integers(0, 80)), dtype=np.uint8).tobytes() for _ in range(n)] if with_ad else None
    sig, ok = eng.ietf_sign_wire(suite, np.ascontiguousarray(sk_all[idx]), (data, off), ads)
    assert ok.all()
    return dict(enc=eng.point_encode(suite, pks), idx=idx, data=data, off=off, sig=sig, ads=ads)


def copy(w):
    return {k: (v.copy() if isinstance(v, np.ndarray) else (list(v) if isinstance(v, list) else v)) for k, v in w.items()}


def torsion_shift(suite, pt):
    """(x, y) -> (-x, -y) = (x, y) + (0, -1) on a twisted-Edwards curve"""
    p = FIELD_P[suite]
    out = pt.copy()
    for h in (0, 32):
        v = int.from_bytes(pt[h:h + 32].tobytes(), "little")
        out[h:h + 32] = np.frombuffer(((p - v) % p).to_bytes(32, "little"), np.uint8)
    return out


def damage_item(eng, suite, w, i, kind, rng):
    """one fault of the given kind in item i of w (in place)"""
    L, cl, n_keys = eng.point_enc_len(suite), eng.challenge_len(suite), len(w["enc"])
    if kind == "out_noncanonical":
        w["sig"][i, :L] = 0xFF                         # y >= p (twisted Edwards, arkworks SW) / no SEC1 prefix
    elif kind == "out_offcurve":
        w["sig"][i, 1 + int(rng.integers(0, L - 2))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "out_torsion" and suite in TE_SUITES:
        pt, ok = eng.point_decode_checked(suite, w["sig"][i, :L])
        assert ok[0]
        w["sig"][i, :L] = eng.point_encode(suite, torsion_shift(suite, pt[0]))[0]
    elif kind == "c":
        w["sig"][i, L + int(rng.integers(0, cl))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "s":
        w["sig"][i, L + cl + int(rng.integers(0, 31))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "s_ge_r":
        w["sig"][i, L + cl:] = 0xFF
    elif kind == "data":
        w["data"][int(w["off"][i])] ^= 0x10
    elif kind == "ad" and w["ads"] is not None:
        w["ads"][i] = w["ads"][i] + b"\x01"
    elif kind == "key" and n_keys > 1:
        w["idx"][i] = (w["idx"][i] + 1) % n_keys
    else:
        w["sig"][i, L] ^= 1                           # kinds the suite or workload cannot take: a flipped challenge byte


def damage(eng, suite, w, rng, frac=8):
    w = copy(w)
    n = len(w["idx"])
    for i in rng.choice(n, max(1, n // frac), replace=False):
        damage_item(eng, suite, w, i, DAMAGE[int(rng.integers(0, len(DAMAGE)))], rng)
    return w


def sliced(w, n):
    return (w["data"], w["off"][:n + 1]), w["sig"][:n], None if w["ads"] is None else w["ads"][:n]


def reference(eng, suite, w, n=None, enc=None):
    n = len(w["idx"]) if n is None else n
    datas, sig, ads = sliced(w, n)
    enc = w["enc"] if enc is None else enc
    return eng.ietf_verify_wire(suite, enc[w["idx"][:n]], datas, sig, ads, status=True)


def prepared(p, w, n=None, want_hash=True):
    n = len(w["idx"]) if n is None else n
    datas, sig, ads = sliced(w, n)
    return p.verify_wire(w["idx"][:n], datas, sig, ads, want_hash=want_hash, status=True)


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("suite", SUITES)
@pytest.mark.parametrize("n_keys", [1, 7, 1023])
def test_parity_with_wire_call(eng, suite, n_keys):
    rng = np.random.default_rng(suite * 7919 + n_keys)
    w = damage(eng, suite, workload(eng, suite, N_MAX, n_keys, seed=n_keys), rng)
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p:
        assert p.key_ok.all() and p.n_keys == n_keys and p.from_encodings
        for n in (1, 31, 33, 4097, N_MAX):
            got = prepared(p, w, n)
            exp = reference(eng, suite, w, n)
            assert same(got, exp), (suite, n_keys, n)
            if n == N_MAX:
                st = got[2]
                assert (st == 0).any() and (st == 1).any() and (st == 2).any()
            if n == 33:          # the CPU oracle on the gathered encodings
                datas = [w["data"][int(w["off"][i]):int(w["off"][i + 1])].tobytes() for i in range(n)]
                ok_o, h_o, st_o = O.ietf_verify_wire(suite, w["enc"][w["idx"][:n]], datas, w["sig"][:n], w["ads"][:n], status=True)
                assert same(got, (ok_o, h_o, st_o)), (suite, n_keys)


@pytest.mark.parametrize("suite", SUITES)
def test_single_faults_first_middle_last(eng, suite):
    n, n_keys = 1001, 7
    w = workload(eng, suite, n, n_keys, seed=3)
    rng = np.random.default_rng(suite)
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p:
        ok, h, st = prepared(p, w)
        assert ok.all() and (st == 0).all() and h.any(axis=1).all()
        for kind in DAMAGE + ("index_out_of_range",):
            for i in (0, n // 2, n - 1):
                d = copy(w)
                if kind == "index_out_of_range":
                    d["idx"][i] = n_keys + i
                    got = prepared(p, d)
                    exp = list(reference(eng, suite, dict(d, idx=np.where(d["idx"] < n_keys, d["idx"], 0).astype(np.uint32))))
                    exp[0][i], exp[1][i], exp[2][i] = 0, 0, 2          # InvalidData, zero hash
                else:
                    damage_item(eng, suite, d, i, kind, rng)
                    got = prepared(p, d)
                    exp = reference(eng, suite, d)
                assert same(got, exp), (kind, i)
                assert got[0][i] == 0 and got[0].sum() == n - 1 and not got[1][i].any(), (kind, i)


def bad_key_encodings(eng, suite, good_enc, good_pts):
    """encodings that must not become keys: non-canonical, off the curve, outside the subgroup (twisted Edwards), the
    short-Weierstrass identity"""
    L = eng.point_enc_len(suite)
    out = [np.full(L, 0xFF, np.uint8)]
    plain_ok = 1
    e = good_enc[0].copy()
    for j in range(256):                               # a one-byte change that no longer decodes to a curve point
        e = good_enc[0].copy(); e[1 + j % (L - 2)] ^= 1 + j // (L - 2)
        _, plain_ok = O.point_decode(suite, e)
        if not plain_ok[0]:
            break
    assert not plain_ok[0]
    out.append(e)
    if suite in TE_SUITES:
        out.append(eng.point_encode(suite, torsion_shift(suite, good_pts[1]))[0])
    if suite in (O.P256, O.BANDERSNATCH_SW):
        out.append(eng.point_encode(suite, np.zeros(64, np.uint8))[0])
    return np.stack(out)


@pytest.mark.parametrize("suite", SUITES)
def test_invalid_key_encodings(eng, suite):
    n, n_good = 400, 4
    w = workload(eng, suite, n, n_good, seed=5)
    good_pts, ok = eng.point_decode_checked(suite, w["enc"])
    assert ok.all()
    bad = bad_key_encodings(eng, suite, w["enc"], good_pts)
    enc = np.concatenate([w["enc"], bad])
    with eng.public_keys_prepare_encoded(suite, enc) as p:
        pts, dec_ok = eng.point_decode_checked(suite, enc)
        with eng.public_keys_prepare(suite, pts) as q:
            assert np.array_equal(p.key_ok, dec_ok & q.key_ok)
        assert p.key_ok.tolist() == [1] * n_good + [0] * len(bad)
        idx = w["idx"].copy()
        named = list(range(10, 10 + 10 * len(bad), 10))
        for j, i in enumerate(named):
            idx[i] = n_good + j
        d = dict(w, idx=idx)
        got = prepared(p, d)
        exp = reference(eng, suite, d, enc=enc)
        assert same(got, exp)
        assert all(got[2][i] == 2 and got[0][i] == 0 and not got[1][i].any() for i in named)
        rest = np.setdiff1d(np.arange(n), named)
        assert got[0][rest].all()


@pytest.mark.parametrize("suite", TE_SUITES)
def test_torsion_key_is_not_a_key(eng, suite):
    """Y + (0, -1), encoded: on the curve, outside the prime-order subgroup.  The affine prepare accepts it as a key; prepared from
    its encoding it is rejected like the wire call rejects it, so no item can reach the table's c*Y with it."""
    w = workload(eng, suite, 200, 3, seed=21)
    pts, _ = eng.point_decode_checked(suite, w["enc"])
    tors = torsion_shift(suite, pts[0])
    enc = np.concatenate([w["enc"], eng.point_encode(suite, tors)])
    with eng.public_keys_prepare_encoded(suite, enc) as p:
        assert p.key_ok.tolist() == [1, 1, 1, 0]
        idx = np.where(w["idx"] == 0, 3, w["idx"]).astype(np.uint32)
        d = dict(w, idx=idx)
        got = prepared(p, d)
        assert same(got, reference(eng, suite, d, enc=enc))
        assert (got[2][idx == 3] == 2).all() and got[0][idx != 3].all()
    with eng.public_keys_prepare(suite, tors[None]) as q:
        assert q.key_ok.all()


def test_golden_vectors(eng):
    g = json.load(open(os.path.join(GOLDEN, "bandersnatch_upstream.json")))
    v = g["ietf"][0]
    data = bytes.fromhex(v["salt"]) + bytes.fromhex(v["alpha"])
    sig = np.frombuffer(bytes.fromhex(v["gamma"] + v["proof_c"] + v["proof_s"]), np.uint8)
    with eng.public_keys_prepare_encoded(O.BANDERSNATCH, np.frombuffer(bytes.fromhex(v["pk"]), np.uint8)) as p:
        ok, beta, st = p.verify_wire([0], [data], sig, [bytes.fromhex(v["ad"])], status=True)
        assert ok[0] and st[0] == 0 and beta[0].tobytes().hex() == v["beta"]
    g = json.load(open(os.path.join(GOLDEN, "p256_rfc9381.json")))
    for v in g["ietf"]:
        pk = bytes.fromhex(v["pk"]); pi = bytes.fromhex(v["pi"])
        beta_exp = hashlib.sha256(b"\x01\x03" + pi[:33] + b"\x00").digest()     # RFC 9381 5.2, suite 0x01, cofactor 1
        with eng.public_keys_prepare_encoded(O.P256, np.frombuffer(pk, np.uint8)) as p:
            ok, beta = p.verify_wire([0], [pk + bytes.fromhex(v["alpha"])], np.frombuffer(pi, np.uint8))
            assert ok[0] and beta[0].tobytes() == beta_exp


@pytest.mark.parametrize("suite", [O.BANDERSNATCH, O.ED25519, O.P256])
def test_encoded_handle_on_typed_calls(eng, suite):
    torch = pytest.importorskip("torch")
    n, n_keys = 3000, 31
    w = workload(eng, suite, n, n_keys, seed=9, with_ad=False)
    L = eng.point_enc_len(suite)
    pts, _ = eng.point_decode_checked(suite, w["enc"])
    out, ok_o = eng.point_decode_checked(suite, w["sig"][:, :L])
    inp, ok_i = eng.data_to_point(suite, (w["data"], w["off"]))
    assert ok_o.all() and ok_i.all()
    cl = eng.challenge_len(suite)
    c = np.zeros((n, 32), np.uint8); s = np.zeros((n, 32), np.uint8)
    be = suite == O.P256                             # SEC1 suites carry big-endian scalars on the wire
    c[:, :cl] = w["sig"][:, L:L + cl][:, ::-1] if be else w["sig"][:, L:L + cl]
    s[:] = w["sig"][:, L + cl:][:, ::-1] if be else w["sig"][:, L + cl:]
    c[5, 0] ^= 1; s[6, 1] ^= 1; w["idx"][7] = (w["idx"][7] + 1) % n_keys
    ok_r, st_r = eng.ietf_verify(suite, pts[w["idx"]], inp, out, c, s, status=True)
    assert ok_r.sum() == n - 3
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p:
        ok, st = p.verify(w["idx"], inp, out, c, s, status=True)
        assert np.array_equal(ok, ok_r) and np.array_equal(st, st_r)
        dev = {k: torch.from_numpy(np.ascontiguousarray(a)).cuda() for k, a in (("inp", inp), ("out", out), ("c", c), ("s", s))}
        idx = torch.from_numpy(w["idx"].view(np.int32)).cuda()
        d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda"); d_st = torch.zeros_like(d_ok)
        torch.cuda.synchronize()
        p.verify_dev(n, idx, dev["inp"], dev["out"], dev["c"], dev["s"], d_ok, d_status=d_st)
        eng.sync()
        assert np.array_equal(d_ok.cpu().numpy(), ok_r) and np.array_equal(d_st.cpu().numpy(), st_r)


def test_handles_and_arguments(eng):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib as L
    lib = eng._lib
    suite = O.ED25519
    w = workload(eng, suite, 4, 2, seed=11, with_ad=False)
    p = eng.public_keys_prepare_encoded(suite, w["enc"])
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    ok = np.zeros(4, np.uint8); h = np.zeros((4, 64), np.uint8); st = np.zeros(4, np.uint8)
    args = (C.c_size_t(4), ptr(w["idx"]), ptr(w["data"]), ptr(w["off"]), ptr(w["sig"]), None, None, ptr(ok), ptr(h), ptr(st))
    assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, p.handle, *args) == L.OK and ok.all()
    # out_hash NULL changes neither ok nor status
    ok2 = np.zeros(4, np.uint8); st2 = np.full(4, 9, np.uint8)
    assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, p.handle, *args[:7], ptr(ok2), None, ptr(st2)) == L.OK
    assert np.array_equal(ok2, ok) and np.array_equal(st2, st)
    d = damage(eng, suite, w, np.random.default_rng(2), frac=2)
    a_h, b_h = prepared(p, d), prepared(p, d, want_hash=False)
    assert np.array_equal(a_h[0], b_h[0]) and np.array_equal(a_h[2], b_h[1]) and not a_h[0].all()
    # an affine handle is refused
    with eng.public_keys_prepare(suite, eng.point_decode_checked(suite, w["enc"])[0]) as q:
        assert not q.from_encodings
        assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, q.handle, *args) == L.BAD_ARG
        assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, q.handle, C.c_size_t(0), *([None] * 9)) == L.BAD_ARG
    # a handle with another context
    other = vrfs.Engine(0)
    try:
        assert lib.vrfs_ietf_verify_prepared_wire_batch(other._ctx, p.handle, *args) == L.BAD_ARG
    finally:
        other.close()
    # n = 0, null buffers, no handle
    assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, p.handle, C.c_size_t(0), *([None] * 9)) == L.OK
    for j in (1, 3, 4, 7):                             # key_index, data_off, sig, out_ok
        a = list(args); a[j] = None
        assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, p.handle, *a) == L.BAD_ARG, j
    assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, None, *args) == L.BAD_ARG
    # n_keys out of 1..65536, null keys, unknown suite
    hh = C.c_void_p()
    many = np.zeros((65537, 33), np.uint8)
    assert lib.vrfs_public_keys_prepare_encoded(eng._ctx, suite, C.c_size_t(0), ptr(many), None, C.byref(hh)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare_encoded(eng._ctx, suite, C.c_size_t(65537), ptr(many), None, C.byref(hh)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare_encoded(eng._ctx, suite, C.c_size_t(1), None, None, C.byref(hh)) == L.BAD_ARG
    assert lib.vrfs_public_keys_prepare_encoded(eng._ctx, 99, C.c_size_t(1), ptr(many), None, C.byref(hh)) == L.BAD_ARG
    assert b"unknown suite" in lib.vrfs_last_error(eng._ctx)
    assert not hh.value
    p.release()
    # a destroyed context's handle, released after its context
    e3 = vrfs.Engine(0)
    q = e3.public_keys_prepare_encoded(suite, w["enc"])
    e3._prepared.remove(q)
    e3.close()
    assert lib.vrfs_ietf_verify_prepared_wire_batch(eng._ctx, q.handle, *args) == L.BAD_ARG
    q.release()
    assert eng.ietf_verify_wire(suite, w["enc"][w["idx"]], (w["data"], w["off"]), w["sig"])[0].all()


def test_large_batch_one_damaged_item(eng):
    suite = O.BANDERSNATCH
    n = 1 << 20
    w = workload(eng, suite, n, 1023, seed=13, with_ad=False)
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p:
        ok, h, st = prepared(p, w)
        assert ok.all() and (st == 0).all()
        j = 777_777
        w["sig"][j, 70] ^= 1                           # s
        ok2, h2, st2 = prepared(p, w)
        assert ok2.sum() == n - 1 and ok2[j] == 0 and st2[j] == 1 and not h2[j].any()
        keep = np.arange(n) != j
        assert np.array_equal(h2[keep], h[keep])
        sub = np.arange(0, n, 4099)                    # the wire call on a spread of items
        d = dict(w, idx=w["idx"][sub], sig=w["sig"][sub], data=np.concatenate([w["data"][i * 8:i * 8 + 8] for i in sub]),
                 off=np.arange(len(sub) + 1, dtype=np.uint64) * 8)
        ok_r, h_r, st_r = reference(eng, suite, d)
        assert np.array_equal(ok_r, ok2[sub]) and np.array_equal(h_r, h2[sub]) and np.array_equal(st_r, st2[sub])


def test_kernel_timings_name_the_new_kernels(eng):
    suite = O.BANDERSNATCH
    w = workload(eng, suite, 300, 5, seed=17, with_ad=False)
    eng.enable_kernel_timing(True)
    try:
        p = eng.public_keys_prepare_encoded(suite, w["enc"])
        names = [k for k, _ in eng.kernel_timings()]
        for k in ("decode_checked", "key_table_powers", "key_table_windows", "merge_flags"):
            assert k in names, names
        assert prepared(p, w)[0].all()
        names = [k for k, _ in eng.kernel_timings()]
        for k in ("wire_prepared_unpack", "data_to_point", "lincomb_keyed", "lincomb<2,0>", "ietf_verify_finish", "point_to_hash", "merge_flags"):
            assert k in names, names
        for k in ("decode_checked", "wire_parse_proof", "gather_keys"):
            assert k not in names, names
        p.release()
    finally:
        eng.enable_kernel_timing(False)


def test_api_prepare_compressed():
    from ark_ec_vrfs_b200 import api
    s = api.Suite.bandersnatch()
    sec = api.Secret.from_seed(s, [b"api-wire-%d" % k for k in range(3)])
    idx = np.array([0, 2, 1, 2, 0], np.uint32)
    eng = s.engine
    datas = [b"m%d" % i for i in range(5)]
    ad = [b"", b"a", b"bb", b"", b"c"]
    sig, ok = eng.ietf_sign_wire(s.suite_id, np.ascontiguousarray(sec.scalars[idx]), datas, ad)
    assert ok.all()
    enc = sec.public().encode()
    with api.Public.prepare_compressed(s, enc) as pp:
        assert pp.key_ok.all()
        got, beta, st = pp.verify_signatures(idx, datas, sig, ad, status=True)
        exp, beta_e, st_e = api.Public.verify_signatures(s, enc[idx], datas, sig, ad, status=True)
        assert got.all() and np.array_equal(got, exp) and np.array_equal(beta, beta_e) and np.array_equal(st, st_e)
        got2, beta2 = pp.verify_signatures(idx, datas, sig, ad)
        assert np.array_equal(got2, got) and np.array_equal(beta2, beta)
    s.engine.close()
