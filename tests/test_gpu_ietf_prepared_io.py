"""IETF verify against prepared keys AND prepared VRF inputs (vrfs_inputs_prepare / vrfs_ietf_verify_prepared_io_batch[_dev]).

The references are vrfs_ietf_verify_prepared_batch with the gathered input points, and vrfs_ietf_verify_batch with the gathered
keys and input points: ok flags and statuses must be identical item by item.  Proofs come from the engine's prover (the oracle
is too slow for 2^16 items); the CPU oracle is added at small sizes."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O

pytestmark = pytest.mark.gpu

SUITES = [O.BANDERSNATCH, O.ED25519, O.P256, O.BANDERSNATCH_SW, O.JUBJUB, O.BABYJUBJUB]
TE_SUITES = [O.BANDERSNATCH, O.ED25519, O.JUBJUB, O.BABYJUBJUB]
FIELD_P = {O.BANDERSNATCH: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.ED25519: 2 ** 255 - 19,
           O.JUBJUB: 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001,
           O.BABYJUBJUB: 0x30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001}
N_MAX = 1 << 16


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def input_datas(suite, seed, n_inputs):
    """round inputs of a lottery: a context string, the round's entropy and an attempt number, of ragged lengths"""
    rng = np.random.default_rng(seed)
    return [b"io-round-%d-%d" % (suite, j) + rng.integers(0, 256, int(rng.integers(0, 70)), dtype=np.uint8).tobytes() for j in range(n_inputs)]


def workload(eng, suite, n, n_keys, n_inputs, seed, with_ad=True):
    """n honest proofs by n_keys signers over n_inputs inputs (random key and input index per item)
    -> dict(pks, idx, datas, pts, jdx, inp, out, c, s, ads)"""
    rng = np.random.default_rng(seed)
    sk_all, pks = eng.secret_from_seed(suite, [b"prepared-io-%d-%d-%d" % (suite, seed, k) for k in range(n_keys)])
    datas = input_datas(suite, seed, n_inputs)
    pts, ok = eng.data_to_point(suite, datas)
    assert ok.all()
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    jdx = rng.integers(0, n_inputs, n).astype(np.uint32)
    sk = np.ascontiguousarray(sk_all[idx]); inp = np.ascontiguousarray(pts[jdx])
    out = eng.output(suite, sk, inp)
    # ragged ad across the SHA-512 / SHA-256 block boundaries of the challenge hash
    ads = [rng.integers(0, 256, int(rng.integers(0, 300)), dtype=np.uint8).tobytes() for _ in range(n)] if with_ad else None
    c, s = eng.ietf_prove(suite, sk, inp, out, ads)
    return dict(pks=pks, idx=idx, datas=datas, pts=pts, jdx=jdx, inp=inp, out=out, c=c, s=s, ads=ads)


def copy(w):
    return {k: (v.copy() if isinstance(v, np.ndarray) else (list(v) if isinstance(v, list) else v)) for k, v in w.items()}


def damage(w, rng, frac=64):
    """every frac-th item (random) gets one fault: c, s or O"""
    w = copy(w)
    n = len(w["idx"])
    for i in rng.choice(n, max(1, n // frac), replace=False):
        kind = int(rng.integers(0, 3))
        if kind == 0:
            w["c"][i, int(rng.integers(0, 16))] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:
            w["s"][i, int(rng.integers(0, 31))] ^= 1 << int(rng.integers(0, 8))
        else:
            w["out"][i] = w["out"][(i + 1) % n]
    return w


def ads_of(w, n):
    return None if w["ads"] is None else w["ads"][:n]


def io(p, q, w, n=None):
    n = len(w["idx"]) if n is None else n
    return p.verify_io(q, w["idx"][:n], w["jdx"][:n], w["out"][:n], w["c"][:n], w["s"][:n], ads_of(w, n), status=True)


def by_prepared_keys(p, w, n=None):
    n = len(w["idx"]) if n is None else n
    inp = w["pts"][np.where(w["jdx"][:n] < len(w["pts"]), w["jdx"][:n], 0)]
    return p.verify(w["idx"][:n], inp, w["out"][:n], w["c"][:n], w["s"][:n], ads_of(w, n), status=True)


def by_gathered(eng, suite, w, n=None):
    n = len(w["idx"]) if n is None else n
    return eng.ietf_verify(suite, w["pks"][w["idx"][:n]], w["pts"][w["jdx"][:n]], w["out"][:n], w["c"][:n], w["s"][:n], ads_of(w, n), status=True)


def same(a, b):
    return all(np.array_equal(x, y) for x, y in zip(a, b))


@pytest.mark.parametrize("suite", SUITES)
@pytest.mark.parametrize("n_inputs", [1, 3, 300])
def test_parity_with_prepared_and_gathered_calls(eng, suite, n_inputs):
    n_keys = 1023 if n_inputs == 300 else 7
    rng = np.random.default_rng(suite * 7919 + n_inputs)
    w = damage(workload(eng, suite, N_MAX, n_keys, n_inputs, seed=n_inputs), rng)
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        pts, ok = eng.data_to_point(suite, w["datas"])
        assert np.array_equal(q.input_ok, ok) and np.array_equal(q.points, pts) and q.n_inputs == n_inputs
        for n in (1, 31, 33, 4097, N_MAX):
            got = io(p, q, w, n)
            assert same(got, by_prepared_keys(p, w, n)), (suite, n_inputs, n)
            assert same(got, by_gathered(eng, suite, w, n)), (suite, n_inputs, n)
            if n == N_MAX:
                assert 0 < got[0].sum() < n and (got[1] == 1).any()
            if n == 33:          # the CPU oracle on the gathered keys and inputs
                exp = O.ietf_verify(suite, w["pks"][w["idx"][:n]], w["pts"][w["jdx"][:n]], w["out"][:n], w["c"][:n], w["s"][:n], w["ads"][:n])
                assert np.array_equal(got[0], exp)


@pytest.mark.parametrize("suite", SUITES)
def test_input_indices_out_of_range_and_faults(eng, suite):
    n, n_inputs = 1001, 3
    w = workload(eng, suite, n, 5, n_inputs, seed=3)
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        assert io(p, q, w)[0].all()
        for i in (0, n // 2, n - 1):
            d = copy(w)
            d["jdx"][i] = (d["jdx"][i] + 1) % n_inputs              # a valid but wrong input
            ok, st = io(p, q, d)
            assert same((ok, st), by_gathered(eng, suite, d)) and ok[i] == 0 and st[i] == 1 and ok.sum() == n - 1
            d["jdx"][i] = n_inputs + i if i else 0xFFFFFFFF          # out of range
            d["idx"][(i + 1) % n] = 5                                # and a key index out of range
            ok, st = io(p, q, d)
            assert ok[i] == 0 and st[i] == 2 and ok[(i + 1) % n] == 0 and st[(i + 1) % n] == 2, i
            rest = np.arange(n) != i                                 # the reference has no point for item i: it reads input 0
            ok_r, st_r = by_prepared_keys(p, d)
            assert np.array_equal(ok[rest], ok_r[rest]) and np.array_equal(st[rest], st_r[rest]), i
            assert ok.sum() == n - 2


@pytest.mark.parametrize("suite", TE_SUITES)
def test_output_with_a_torsion_component(eng, suite):
    """O + (0, -1) = (-x, -y): on the curve, outside the prime-order subgroup.  c*O goes through the same variable-base path as in
    the other calls, so every verdict is theirs."""
    n = 500
    w = workload(eng, suite, n, 3, 2, seed=21)
    p_mod = FIELD_P[suite]
    d = copy(w)
    for i in range(0, n, 3):
        for h in (0, 32):
            v = int.from_bytes(d["out"][i, h:h + 32].tobytes(), "little")
            d["out"][i, h:h + 32] = np.frombuffer(((p_mod - v) % p_mod).to_bytes(32, "little"), np.uint8)
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        got = io(p, q, d)
        assert same(got, by_prepared_keys(p, d)) and same(got, by_gathered(eng, suite, d))
        assert (got[1][::3] != 0).all() and got[0][np.arange(n) % 3 != 0].all()


def test_device_form_matches_host_form(eng):
    torch = pytest.importorskip("torch")
    suite = O.BANDERSNATCH
    w = damage(workload(eng, suite, 5000, 31, 3, seed=9, with_ad=False), np.random.default_rng(1), frac=8)
    w["jdx"][7] = 3                                                  # out of range
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        ok_h, st_h = io(p, q, w)
        dev = {k: torch.from_numpy(np.ascontiguousarray(w[k])).cuda() for k in ("out", "c", "s")}
        idx = torch.from_numpy(w["idx"].view(np.int32)).cuda(); jdx = torch.from_numpy(w["jdx"].view(np.int32)).cuda()
        ok = torch.zeros(len(idx), dtype=torch.uint8, device="cuda"); st = torch.zeros_like(ok)
        torch.cuda.synchronize()
        p.verify_io_dev(q, len(idx), idx, jdx, dev["out"], dev["c"], dev["s"], ok, d_status=st)
        eng.sync()
        assert np.array_equal(ok.cpu().numpy(), ok_h) and np.array_equal(st.cpu().numpy(), st_h)
        assert st_h[7] == 2 and 0 < ok_h.sum() < len(ok_h)


def test_piecewise_host_call_equals_small_calls(eng):
    """250 000 items: the host call stages them in pieces; item by item it equals calls of 25 000"""
    suite = O.BANDERSNATCH
    n, step = 250_000, 25_000
    w = damage(workload(eng, suite, n, 63, 3, seed=23), np.random.default_rng(23))
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        ok, st = io(p, q, w)
        for lo in range(0, n, step):
            part = {k: (v[lo:lo + step] if k in ("idx", "jdx", "out", "c", "s", "ads") else v) for k, v in w.items()}
            ok_p, st_p = io(p, q, part)
            assert np.array_equal(ok_p, ok[lo:lo + step]) and np.array_equal(st_p, st[lo:lo + step]), lo
        assert 0 < ok.sum() < n


def test_large_batch_honest(eng):
    suite = O.BANDERSNATCH
    n = 1 << 20
    w = workload(eng, suite, n, 1023, 3, seed=13, with_ad=False)
    with eng.public_keys_prepare(suite, w["pks"]) as p, eng.inputs_prepare(suite, w["datas"]) as q:
        ok, st = io(p, q, w)
        assert ok.all() and (st == 0).all()


def test_handles_and_arguments(eng):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib as L
    lib = eng._lib
    suite = O.ED25519
    w = workload(eng, suite, 4, 2, 2, seed=11, with_ad=False)
    p = eng.public_keys_prepare(suite, w["pks"])
    q = eng.inputs_prepare(suite, w["datas"])
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    ok = np.zeros(4, np.uint8)
    args = (C.c_size_t(4), ptr(w["idx"]), ptr(w["jdx"]), ptr(w["out"]), ptr(w["c"]), ptr(w["s"]), None, None, ptr(ok), None)
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, q.handle, *args) == L.OK and ok.all()
    # handles of another context
    other = vrfs.Engine(0)
    try:
        for fn in ("vrfs_ietf_verify_prepared_io_batch", "vrfs_ietf_verify_prepared_io_batch_dev"):
            assert getattr(lib, fn)(other._ctx, p.handle, q.handle, *args) == L.BAD_ARG
        q2 = other.inputs_prepare(suite, w["datas"])
        assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, q2.handle, *args) == L.BAD_ARG
        q2.release()
    finally:
        other.close()
    # suite mismatch; a keys handle where the inputs handle goes, and the other way round
    with eng.inputs_prepare(O.BANDERSNATCH, w["datas"]) as qb:
        assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, qb.handle, *args) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, p.handle, *args) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, q.handle, q.handle, *args) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_batch(eng._ctx, q.handle, C.c_size_t(4), ptr(w["idx"]), ptr(w["inp"]), ptr(w["out"]), ptr(w["c"]),
                                               ptr(w["s"]), None, None, ptr(ok), None) == L.BAD_ARG
    # n = 0, null buffers, no handle
    for fn in ("vrfs_ietf_verify_prepared_io_batch", "vrfs_ietf_verify_prepared_io_batch_dev"):
        assert getattr(lib, fn)(eng._ctx, p.handle, q.handle, C.c_size_t(0), *([None] * 9)) == L.OK
    for j in (1, 2, 3, 4, 5, 8):                                     # key_index, input_index, output, c, s, out_ok
        a = list(args); a[j] = None
        assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, q.handle, *a) == L.BAD_ARG, j
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p.handle, None, *args) == L.BAD_ARG
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, None, q.handle, *args) == L.BAD_ARG
    # n_inputs out of 1..65536, null offsets, unknown suite
    h = C.c_void_p()
    off = np.zeros(65538, np.uint64); data = np.zeros(16, np.uint8)
    assert lib.vrfs_inputs_prepare(eng._ctx, suite, C.c_size_t(0), ptr(data), ptr(off), None, None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_inputs_prepare(eng._ctx, suite, C.c_size_t(65537), ptr(data), ptr(off), None, None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_inputs_prepare(eng._ctx, suite, C.c_size_t(1), ptr(data), None, None, None, C.byref(h)) == L.BAD_ARG
    assert lib.vrfs_inputs_prepare(eng._ctx, 99, C.c_size_t(1), ptr(data), ptr(off), None, None, C.byref(h)) == L.BAD_ARG
    assert b"unknown suite" in lib.vrfs_last_error(eng._ctx)
    assert not h.value
    # 65536 empty inputs are accepted; NULL out_input_ok / out_points are allowed
    assert lib.vrfs_inputs_prepare(eng._ctx, suite, C.c_size_t(65536), ptr(data), ptr(off), None, None, C.byref(h)) == L.OK and h.value
    lib.vrfs_inputs_release(h)
    q.release(); p.release()
    lib.vrfs_inputs_release(None)
    # a released handle; a destroyed context's handle, released after its context
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, None, None, *args) == L.BAD_ARG
    e3 = vrfs.Engine(0)
    p3 = e3.public_keys_prepare(suite, w["pks"]); q3 = e3.inputs_prepare(suite, w["datas"])
    e3._prepared.remove(p3); e3._prepared.remove(q3)
    e3.close()
    assert lib.vrfs_ietf_verify_prepared_io_batch(eng._ctx, p3.handle, q3.handle, *args) == L.BAD_ARG
    q3.release(); p3.release()
    assert eng.ietf_verify(suite, w["pks"][w["idx"]], w["inp"], w["out"], w["c"], w["s"]).all()


def test_kernel_timings_name_the_new_kernels(eng):
    suite = O.BANDERSNATCH
    w = workload(eng, suite, 300, 5, 2, seed=17, with_ad=False)
    eng.enable_kernel_timing(True)
    try:
        p = eng.public_keys_prepare(suite, w["pks"])
        q = eng.inputs_prepare(suite, w["datas"])
        names = [k for k, _ in eng.kernel_timings()]
        for k in ("data_to_point", "key_table_powers", "key_table_windows", "merge_flags"):
            assert k in names, names
        assert io(p, q, w)[0].all()
        names = [k for k, _ in eng.kernel_timings()]
        for k in ("gather_keys", "gather_inputs", "lincomb_keyed", "lincomb_io", "ietf_verify_finish"):
            assert k in names, names
        assert "lincomb<2,0>" not in names and "data_to_point" not in names, names
        q.release(); p.release()
    finally:
        eng.enable_kernel_timing(False)


def test_api_input_prepare():
    from ark_ec_vrfs_b200 import api
    s = api.Suite.bandersnatch()
    sec = api.Secret.from_seed(s, [b"api-io-%d" % k for k in range(3)])
    idx = np.array([0, 2, 1, 2, 0], np.uint32)
    jdx = np.array([1, 1, 0, 1, 0], np.uint32)
    signer = api.Secret(s, np.ascontiguousarray(sec.scalars[idx]), np.ascontiguousarray(sec.public_points[idx]))
    rounds = [b"round-0", b"round-1"]
    inp, ok = api.Input.new(s, [rounds[j] for j in jdx])
    assert ok.all()
    out = signer.output(inp)
    ad = [b"", b"a", b"bb", b"", b"c"]
    proof = signer.prove(inp, out, ad)
    with sec.public().prepare() as pp, api.Input.prepare(s, rounds) as pi:
        assert pi.input_ok.all() and np.array_equal(pi.points[jdx], inp.points)
        got, st = pp.verify_prepared_input(idx, pi, jdx, out, ad, proof, status=True)
        exp, st_e = signer.public().verify(inp, out, ad, proof, status=True)
        assert got.all() and np.array_equal(got, exp) and np.array_equal(st, st_e)
    s.engine.close()
