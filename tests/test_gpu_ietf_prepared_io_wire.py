"""Serialised IETF signatures verified against prepared keys and prepared VRF inputs, both by index
(vrfs_ietf_verify_prepared_io_wire_batch).

The references are vrfs_ietf_verify_prepared_wire_batch and vrfs_ietf_verify_wire_batch on the gathered encodings and data: ok
flags, hashes and statuses must be identical item by item.  Signatures come from the engine's signer."""
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
N_MAX = 1 << 16
DAMAGE = ("out_noncanonical", "out_offcurve", "c", "s", "s_ge_r", "ad", "key", "input")


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def workload(eng, suite, n, n_keys, n_inputs, seed, with_ad=True):
    """n honest signatures by n_keys signers over n_inputs inputs -> dict(enc, idx, datas, jdx, sig, ads)"""
    rng = np.random.default_rng(seed)
    sk_all, pks = eng.secret_from_seed(suite, [b"prepared-io-wire-%d-%d-%d" % (suite, seed, k) for k in range(n_keys)])
    datas = [b"io-wire-round-%d-%d" % (suite, j) + rng.integers(0, 256, int(rng.integers(0, 70)), dtype=np.uint8).tobytes()
             for j in range(n_inputs)]
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    jdx = rng.integers(0, n_inputs, n).astype(np.uint32)
    ads = [rng.integers(0, 256, int(rng.integers(0, 300)), dtype=np.uint8).tobytes() for _ in range(n)] if with_ad else None
    sig, ok = eng.ietf_sign_wire(suite, np.ascontiguousarray(sk_all[idx]), [datas[j] for j in jdx], ads)
    assert ok.all()
    return dict(enc=eng.point_encode(suite, pks), idx=idx, datas=datas, jdx=jdx, sig=sig, ads=ads)


def copy(w):
    return {k: (v.copy() if isinstance(v, np.ndarray) else (list(v) if isinstance(v, list) else v)) for k, v in w.items()}


def damage_item(eng, suite, w, i, kind, rng):
    L, cl = eng.point_enc_len(suite), eng.challenge_len(suite)
    if kind == "out_noncanonical":
        w["sig"][i, :L] = 0xFF
    elif kind == "out_offcurve":
        w["sig"][i, 1 + int(rng.integers(0, L - 2))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "c":
        w["sig"][i, L + int(rng.integers(0, cl))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "s":
        w["sig"][i, L + cl + int(rng.integers(0, 31))] ^= 1 << int(rng.integers(0, 8))
    elif kind == "s_ge_r":
        w["sig"][i, L + cl:] = 0xFF
    elif kind == "ad" and w["ads"] is not None:
        w["ads"][i] = w["ads"][i] + b"\x01"
    elif kind == "key" and len(w["enc"]) > 1:
        w["idx"][i] = (w["idx"][i] + 1) % len(w["enc"])
    elif kind == "input" and len(w["datas"]) > 1:
        w["jdx"][i] = (w["jdx"][i] + 1) % len(w["datas"])
    else:
        w["sig"][i, L] ^= 1


def damage(eng, suite, w, rng, frac=64):
    w = copy(w)
    n = len(w["idx"])
    for i in rng.choice(n, max(1, n // frac), replace=False):
        damage_item(eng, suite, w, i, DAMAGE[int(rng.integers(0, len(DAMAGE)))], rng)
    return w


def ads_of(w, n):
    return None if w["ads"] is None else w["ads"][:n]


def io_wire(p, q, w, n=None):
    n = len(w["idx"]) if n is None else n
    return p.verify_io_wire(q, w["idx"][:n], w["jdx"][:n], w["sig"][:n], ads_of(w, n), status=True)


def gathered_data(w, n):
    return [w["datas"][j] if j < len(w["datas"]) else b"" for j in w["jdx"][:n]]


def by_prepared_wire(p, w, n=None):
    n = len(w["idx"]) if n is None else n
    return p.verify_wire(w["idx"][:n], gathered_data(w, n), w["sig"][:n], ads_of(w, n), status=True)


def by_wire(eng, suite, w, n=None, enc=None):
    n = len(w["idx"]) if n is None else n
    enc = w["enc"] if enc is None else enc
    return eng.ietf_verify_wire(suite, enc[w["idx"][:n]], gathered_data(w, n), w["sig"][:n], ads_of(w, n), status=True)


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("suite", SUITES)
@pytest.mark.parametrize("n_inputs", [1, 3, 300])
def test_parity_with_wire_calls(eng, suite, n_inputs):
    n_keys = 1023 if n_inputs == 300 else 7
    rng = np.random.default_rng(suite * 7919 + n_inputs)
    w = damage(eng, suite, workload(eng, suite, N_MAX, n_keys, n_inputs, seed=n_inputs), rng)
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        assert p.key_ok.all() and q.input_ok.all()
        for n in (1, 33, 4097, N_MAX):
            got = io_wire(p, q, w, n)
            assert same(got, by_prepared_wire(p, w, n)), (suite, n_inputs, n)
            assert same(got, by_wire(eng, suite, w, n)), (suite, n_inputs, n)
            if n == N_MAX:
                st = got[2]
                assert (st == 0).any() and (st == 1).any() and (st == 2).any()


@pytest.mark.parametrize("suite", SUITES)
def test_bad_keys_and_indices(eng, suite):
    """a key encoding that is rejected (key_ok = 0), key and input indices out of range"""
    n, n_good = 400, 4
    w = workload(eng, suite, n, n_good, 2, seed=5)
    enc = np.concatenate([w["enc"], np.full((1, eng.point_enc_len(suite)), 0xFF, np.uint8)])
    with eng.public_keys_prepare_encoded(suite, enc) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        assert p.key_ok.tolist() == [1] * n_good + [0]
        d = copy(w)
        d["idx"][10] = n_good                           # a key with key_ok = 0: the wire call's verdict on its encoding
        got = io_wire(p, q, d)
        assert same(got, by_wire(eng, suite, d, enc=enc)) and got[2][10] == 2
        d["idx"][20] = len(enc)                         # key index out of range
        d["jdx"][30], d["jdx"][40] = 2, 0xFFFFFFFF      # input indices out of range
        got = io_wire(p, q, d)
        for i in (10, 20, 30, 40):
            assert got[0][i] == 0 and got[2][i] == 2 and not got[1][i].any(), i
        rest = np.setdiff1d(np.arange(n), [10, 20, 30, 40])
        assert got[0][rest].all() and (got[2][rest] == 0).all()
        d2 = dict(d, idx=np.where(d["idx"] < len(enc), d["idx"], 0).astype(np.uint32))
        exp = by_wire(eng, suite, d2, enc=enc)
        assert all(np.array_equal(g[rest], e[rest]) for g, e in zip(got, exp))


def test_golden_vectors(eng):
    g = json.load(open(os.path.join(GOLDEN, "bandersnatch_upstream.json")))
    v = g["ietf"][0]
    data = bytes.fromhex(v["salt"]) + bytes.fromhex(v["alpha"])
    sig = np.frombuffer(bytes.fromhex(v["gamma"] + v["proof_c"] + v["proof_s"]), np.uint8)
    with eng.public_keys_prepare_encoded(O.BANDERSNATCH, np.frombuffer(bytes.fromhex(v["pk"]), np.uint8)) as p, \
            eng.inputs_prepare(O.BANDERSNATCH, [b"another input", data]) as q:
        ok, beta, st = p.verify_io_wire(q, [0], [1], sig, [bytes.fromhex(v["ad"])], status=True)
        assert ok[0] and st[0] == 0 and beta[0].tobytes().hex() == v["beta"]
        ok, beta, st = p.verify_io_wire(q, [0], [0], sig, [bytes.fromhex(v["ad"])], status=True)
        assert not ok[0] and st[0] == 1
    g = json.load(open(os.path.join(GOLDEN, "p256_rfc9381.json")))
    for v in g["ietf"]:
        pk = bytes.fromhex(v["pk"]); pi = bytes.fromhex(v["pi"])
        beta_exp = hashlib.sha256(b"\x01\x03" + pi[:33] + b"\x00").digest()     # RFC 9381 5.2, suite 0x01, cofactor 1
        with eng.public_keys_prepare_encoded(O.P256, np.frombuffer(pk, np.uint8)) as p, \
                eng.inputs_prepare(O.P256, [pk + bytes.fromhex(v["alpha"])]) as q:
            ok, beta = p.verify_io_wire(q, [0], [0], np.frombuffer(pi, np.uint8))
            assert ok[0] and beta[0].tobytes() == beta_exp


def test_handles_and_arguments(eng):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib as L
    lib = eng._lib
    suite = O.ED25519
    w = workload(eng, suite, 4, 2, 2, seed=11, with_ad=False)
    p = eng.public_keys_prepare_encoded(suite, w["enc"])
    q = eng.inputs_prepare(suite, w["datas"])
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    ok = np.zeros(4, np.uint8); h = np.zeros((4, 64), np.uint8); st = np.zeros(4, np.uint8)
    args = (C.c_size_t(4), ptr(w["idx"]), ptr(w["jdx"]), ptr(w["sig"]), None, None, ptr(ok), ptr(h), ptr(st))
    fn = lib.vrfs_ietf_verify_prepared_io_wire_batch
    assert fn(eng._ctx, p.handle, q.handle, *args) == L.OK and ok.all() and (st == 0).all()
    # out_hash and out_status may be NULL
    ok2 = np.zeros(4, np.uint8)
    assert fn(eng._ctx, p.handle, q.handle, *args[:6], ptr(ok2), None, None) == L.OK and ok2.all()
    # an affine key handle is refused, with n = 0 too
    with eng.public_keys_prepare(suite, eng.point_decode_checked(suite, w["enc"])[0]) as a:
        assert fn(eng._ctx, a.handle, q.handle, *args) == L.BAD_ARG
        assert fn(eng._ctx, a.handle, q.handle, C.c_size_t(0), *([None] * 8)) == L.BAD_ARG
    # other context, suite mismatch, swapped handles
    other = vrfs.Engine(0)
    try:
        assert fn(other._ctx, p.handle, q.handle, *args) == L.BAD_ARG
    finally:
        other.close()
    with eng.inputs_prepare(O.P256, w["datas"]) as qp:
        assert fn(eng._ctx, p.handle, qp.handle, *args) == L.BAD_ARG
    assert fn(eng._ctx, q.handle, p.handle, *args) == L.BAD_ARG
    # n = 0, null buffers, no handle
    assert fn(eng._ctx, p.handle, q.handle, C.c_size_t(0), *([None] * 8)) == L.OK
    for j in (1, 2, 3, 6):                             # key_index, input_index, sig, out_ok
        a = list(args); a[j] = None
        assert fn(eng._ctx, p.handle, q.handle, *a) == L.BAD_ARG, j
    assert fn(eng._ctx, p.handle, None, *args) == L.BAD_ARG
    q.release(); p.release()
    # handles of a destroyed context
    e3 = vrfs.Engine(0)
    p3 = e3.public_keys_prepare_encoded(suite, w["enc"]); q3 = e3.inputs_prepare(suite, w["datas"])
    e3._prepared.remove(p3); e3._prepared.remove(q3)
    e3.close()
    assert fn(eng._ctx, p3.handle, q3.handle, *args) == L.BAD_ARG
    q3.release(); p3.release()


def test_kernel_timings_name_the_new_kernels(eng):
    suite = O.BANDERSNATCH
    w = workload(eng, suite, 300, 5, 2, seed=17, with_ad=False)
    with eng.public_keys_prepare_encoded(suite, w["enc"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        eng.enable_kernel_timing(True)
        try:
            assert io_wire(p, q, w)[0].all()
            names = [k for k, _ in eng.kernel_timings()]
        finally:
            eng.enable_kernel_timing(False)
    for k in ("wire_prepared_unpack", "gather_inputs", "lincomb_keyed", "lincomb_io", "ietf_verify_finish", "point_to_hash", "merge_flags"):
        assert k in names, names
    for k in ("data_to_point", "lincomb<2,0>", "decode_checked", "gather_keys"):
        assert k not in names, names


def test_api_verify_signatures_prepared_input():
    from ark_ec_vrfs_b200 import api
    s = api.Suite.bandersnatch()
    eng = s.engine
    sec = api.Secret.from_seed(s, [b"api-io-wire-%d" % k for k in range(3)])
    idx = np.array([0, 2, 1, 2, 0], np.uint32)
    jdx = np.array([1, 0, 0, 1, 1], np.uint32)
    rounds = [b"epoch-entropy-0", b"epoch-entropy-1"]
    ad = [b"header-%d" % i for i in range(5)]
    sig, ok = eng.ietf_sign_wire(s.suite_id, np.ascontiguousarray(sec.scalars[idx]), [rounds[j] for j in jdx], ad)
    assert ok.all()
    enc = sec.public().encode()
    with api.Public.prepare_compressed(s, enc) as pp, api.Input.prepare(s, rounds) as pi:
        got, beta, st = pp.verify_signatures_prepared_input(idx, pi, jdx, sig, ad, status=True)
        exp, beta_e, st_e = api.Public.verify_signatures(s, enc[idx], [rounds[j] for j in jdx], sig, ad, status=True)
        assert got.all() and np.array_equal(got, exp) and np.array_equal(beta, beta_e) and np.array_equal(st, st_e)
    s.engine.close()
