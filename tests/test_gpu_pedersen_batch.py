"""GPU: vrfs_pedersen_batch_verify / vrfs_pedersen_batch_verify_wire - a batch of Bandersnatch Pedersen proofs checked by one
random linear combination - against the per-item verifier (vrfs_pedersen_verify_batch, vrfs_pedersen_verify_wire_batch) and the
CPU oracle.  Proofs come from the engine's prover."""
import ctypes as C
import hashlib
import json
import os

import numpy as np
import pytest

import oracle_lib as O
import vectors as V

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
B = O.BANDERSNATCH
FQ = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
FR = 0x1cfb69d4ca675f520cce760202687600ff8f87007419047174fd06b52876e7e1
T2 = (0, FQ - 1)                      # the affine 2-torsion point


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def make_batch(eng, n, ad_kind="ragged", tag=b"ped-batch"):
    seeds = [hashlib.sha256(tag + b"-sk-%d" % i).digest() for i in range(n)]
    sk, _ = eng.secret_from_seed(B, seeds)
    alphas = [tag + b"-alpha-" + i.to_bytes(8, "little") for i in range(n)]
    inp, ok = eng.data_to_point(B, alphas)
    assert ok.all()
    out = eng.output(B, sk, inp)
    ads = V.make_ads(n, ad_kind)
    proof, _ = eng.pedersen_prove(B, sk, inp, out, ads)
    return dict(sk=sk, alphas=alphas, inp=inp, out=out, proof=proof.copy(), ads=ads)


def pt(P):
    return np.frombuffer(P[0].to_bytes(32, "little") + P[1].to_bytes(32, "little"), np.uint8)


def xy(a):
    return int.from_bytes(a[:32].tobytes(), "little"), int.from_bytes(a[32:].tobytes(), "little")


def check(eng, inp, out, proof, ads, seed=None, oracle=True, all_matches=True):
    """batch verdict and fallback against the per-item verifier (and the oracle); returns (all_ok, per-item ok)"""
    ok_ref, st_ref = eng.pedersen_verify(B, inp, out, proof, ads, status=True)
    if oracle:
        ok_o, st_o = O.pedersen_verify(B, inp, out, proof, ads, status=True)
        assert np.array_equal(ok_o, ok_ref) and np.array_equal(st_o, st_ref)
    all_ok, ok, st = eng.pedersen_batch_verify(B, inp, out, proof, ads, seed=seed, per_item=True, status=True)
    if all_matches:
        assert all_ok == bool(ok_ref.all())
    assert np.array_equal(ok, ok_ref) and np.array_equal(st, st_ref)
    return all_ok, ok_ref


@pytest.mark.parametrize("n", [1, 2, 33, 4097, 1 << 16])
def test_honest_batches_accept(eng, n):
    d = make_batch(eng, n)
    assert check(eng, d["inp"], d["out"], d["proof"], d["ads"], oracle=n <= 4097)[0] is True
    assert eng.pedersen_batch_verify(B, d["inp"], d["out"], d["proof"], d["ads"]) is True


def test_upstream_pedersen_vector(eng):
    with open(os.path.join(GOLDEN, "bandersnatch_upstream.json")) as f:
        vec = json.load(f)["pedersen"][0]
    dec = lambda h: O.point_decode(0, bytes.fromhex(h))
    (inp, a), (out, b), (yb, c), (r, d), (okp, e) = (dec(vec[k]) for k in ("h", "gamma", "proof_pk_com", "proof_r", "proof_ok"))
    assert a.all() and b.all() and c.all() and d.all() and e.all()
    proof = np.concatenate([yb, r, okp, np.frombuffer(bytes.fromhex(vec["proof_s"]), np.uint8).reshape(1, 32),
                            np.frombuffer(bytes.fromhex(vec["proof_sb"]), np.uint8).reshape(1, 32)], axis=1)
    ad = [bytes.fromhex(vec["ad"])]
    assert eng.pedersen_verify(B, inp, out, proof, ad).tolist() == [1]
    assert eng.pedersen_batch_verify(B, inp, out, proof, ad) is True


FIELDS = ["s", "sb", "Ok", "R", "Yb", "O", "I", "ad"]


@pytest.mark.parametrize("field", FIELDS)
@pytest.mark.parametrize("where", ["first", "middle", "last"])
def test_single_fault_rejected_and_fallback_exact(eng, field, where):
    n = 65
    d = make_batch(eng, n)
    j = {"first": 0, "middle": n // 2, "last": n - 1}[where]
    inp, out, proof, ads = d["inp"].copy(), d["out"].copy(), d["proof"].copy(), list(d["ads"])
    k = (j + 1) % n
    if field == "s":
        proof[j, 192 + 3] ^= 0x10
    elif field == "sb":
        proof[j, 224 + 7] ^= 0x01
    elif field == "Ok":
        proof[j, 128:192] = proof[k, 128:192]
    elif field == "R":
        proof[j, 64:128] = proof[k, 64:128]
    elif field == "Yb":
        proof[j, 0:64] = proof[k, 0:64]
    elif field == "O":
        out[j] = out[k]
    elif field == "I":
        inp[j] = inp[k]
    else:
        ads[j] = ads[j] + b"\x00" if not ads[j] else bytes([ads[j][0] ^ 1]) + ads[j][1:]
    all_ok, ok = check(eng, inp, out, proof, ads)
    assert all_ok is False and ok[j] == 0 and ok.sum() == n - 1


def test_invalid_data_and_scalar_reduction(eng):
    n = 16
    d = make_batch(eng, n, "fixed32")
    inp, out, proof, ads = d["inp"].copy(), d["out"].copy(), d["proof"].copy(), d["ads"]
    cases = []
    j = next(i for i in range(n) if xy(out[i])[0] + FQ < 2 ** 256)
    x, y = xy(out[j])                                       # non-canonical x of O: x + p
    o2 = out.copy(); o2[j, :32] = np.frombuffer((x + FQ).to_bytes(32, "little"), np.uint8); cases.append((inp, o2, proof))
    p2 = proof.copy(); p2[3, 64 + 40] ^= 0x04; cases.append((inp, out, p2))          # R off the curve
    i2 = inp.copy(); i2[5] = pt((0, 1)); cases.append((i2, out, proof))             # the identity as input: on the curve, in the subgroup
    p3 = proof.copy(); p3[7, 128:192] = pt((0, 1)); cases.append((inp, out, p3))    # the identity as Ok
    for a, b, c in cases:
        all_ok, _ = check(eng, a, b, c, ads)
        assert all_ok is False
    # s + r in place of s: scalars are reduced on load, so both paths accept
    p4 = proof.copy()
    s = int.from_bytes(p4[2, 192:224].tobytes(), "little")
    p4[2, 192:224] = np.frombuffer((s + FR).to_bytes(32, "little"), np.uint8)
    assert check(eng, inp, out, p4, ads)[0] is True


@pytest.mark.parametrize("target", ["Ok", "O"])
def test_torsion_component_is_rejected_for_every_seed(eng, target):
    """(0, -1) added to one point: the per-item verifier sees it in E_j, a combination with an even rho_j would not - the
    subgroup test must catch it whatever the seed"""
    from oracle import pyref as R
    Cv = R.BANDERSNATCH
    n = 8
    d = make_batch(eng, n, "fixed32")
    inp, out, proof = d["inp"], d["out"].copy(), d["proof"].copy()
    j = 3
    if target == "Ok":
        proof[j, 128:192] = pt(Cv.add(xy(proof[j, 128:192]), T2))
    else:
        out[j] = pt(Cv.add(xy(out[j]), T2))
    for t in range(32):
        seed = hashlib.sha256(b"torsion-seed-%d" % t).digest()
        all_ok, ok = check(eng, inp, out, proof, d["ads"], seed=seed, oracle=t == 0, all_matches=False)
        assert all_ok is False
        if target == "Ok":
            assert ok[j] == 0


def test_cancelling_forgeries_rejected(eng):
    from oracle import pyref as R
    Cv = R.BANDERSNATCH
    n = 8
    d = make_batch(eng, n, "fixed32")
    D = Cv.mul(123456789, Cv.G)
    # Ok_1 + D and Ok_2 - D: a plain sum (every rho = 1) would accept
    p = d["proof"].copy()
    p[1, 128:192] = pt(Cv.add(xy(p[1, 128:192]), D))
    p[2, 128:192] = pt(Cv.add(xy(p[2, 128:192]), Cv.neg(D)))
    all_ok, ok = check(eng, d["inp"], d["out"], p, d["ads"])
    assert all_ok is False and ok[1] == 0 and ok[2] == 0
    # Ok_j + D and R_j - D: accepted if rho_j = sigma_j
    p = d["proof"].copy()
    p[4, 128:192] = pt(Cv.add(xy(p[4, 128:192]), D))
    p[4, 64:128] = pt(Cv.add(xy(p[4, 64:128]), Cv.neg(D)))
    all_ok, ok = check(eng, d["inp"], d["out"], p, d["ads"])
    assert all_ok is False and ok[4] == 0


def test_seed_behaviour(eng):
    d = make_batch(eng, 40)
    bad = d["proof"].copy(); bad[9, 200] ^= 1
    seed = bytes(range(32))
    for _ in range(3):
        assert eng.pedersen_batch_verify(B, d["inp"], d["out"], d["proof"], d["ads"], seed=seed) is True
        assert eng.pedersen_batch_verify(B, d["inp"], d["out"], bad, d["ads"], seed=seed) is False
    for t in range(8):
        assert eng.pedersen_batch_verify(B, d["inp"], d["out"], d["proof"], d["ads"], seed=hashlib.sha256(b"%d" % t).digest()) is True


def test_arguments(eng):
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import _lib
    d = make_batch(eng, 4, "fixed32")
    for suite in (1, 2, 3, 4, 5):
        with pytest.raises(vrfs.VrfsError) as ei:
            eng.pedersen_batch_verify(suite, d["inp"], d["out"], d["proof"], d["ads"])
        assert ei.value.status == _lib.UNSUPPORTED and "Bandersnatch" in str(ei.value)
    for suite in (6, 99):
        with pytest.raises(vrfs.VrfsError) as ei:
            eng.pedersen_batch_verify(suite, d["inp"], d["out"], d["proof"], d["ads"])
        assert ei.value.status == _lib.BAD_ARG and "unknown suite %d" % suite in str(ei.value)
    assert eng.pedersen_batch_verify(B, np.zeros((0, 64), np.uint8), np.zeros((0, 64), np.uint8), np.zeros((0, 256), np.uint8)) is True
    lib, ctx = eng._lib, eng._ctx
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    all_ok = np.full(1, 7, np.uint8); seed = np.zeros(32, np.uint8)
    assert lib.vrfs_pedersen_batch_verify(ctx, B, C.c_size_t(0), None, None, None, None, None, p(seed), p(all_ok), None, None) == _lib.OK and all_ok[0] == 1
    assert lib.vrfs_pedersen_batch_verify_wire(ctx, B, C.c_size_t(0), None, None, None, None, None, p(seed), p(all_ok), None, None) == _lib.OK and all_ok[0] == 1
    args = [p(d["inp"]), p(d["out"]), p(d["proof"])]
    for k in range(3):
        a = list(args); a[k] = None
        assert lib.vrfs_pedersen_batch_verify(ctx, B, C.c_size_t(4), *a, None, None, p(seed), p(all_ok), None, None) == _lib.BAD_ARG
        assert "null buffer" in lib.vrfs_last_error(ctx).decode()
    assert lib.vrfs_pedersen_batch_verify(ctx, B, C.c_size_t(4), *args, None, None, None, p(all_ok), None, None) == _lib.BAD_ARG
    assert lib.vrfs_pedersen_batch_verify(ctx, B, C.c_size_t(4), *args, None, None, p(seed), None, None, None) == _lib.BAD_ARG
    assert lib.vrfs_pedersen_batch_verify_wire(ctx, B, C.c_size_t(4), None, None, None, None, None, p(seed), p(all_ok), None, None) == _lib.BAD_ARG
    assert "null buffer" in lib.vrfs_last_error(ctx).decode()


def test_large_batches(eng):
    n = 1 << 20
    d = make_batch(eng, n, "empty", tag=b"ped-batch-large")
    all_ok, ok, st = eng.pedersen_batch_verify(B, d["inp"], d["out"], d["proof"], None, per_item=True, status=True)
    assert all_ok is True and ok.all() and not st.any()
    j = 777_777
    p = d["proof"].copy(); p[j, 230] ^= 0x20
    all_ok, ok, st = eng.pedersen_batch_verify(B, d["inp"], d["out"], p, None, per_item=True, status=True)
    assert all_ok is False and np.flatnonzero(ok == 0).tolist() == [j] and st[j] == 1       # VRFS_ITEM_VERIFICATION_FAILURE


def test_wire_form(eng):
    from oracle import pyref as R
    Cv = R.BANDERSNATCH
    n = 33
    d = make_batch(eng, n)
    sig, _, sok = eng.pedersen_sign_wire(B, d["sk"], d["alphas"], d["ads"])
    assert sok.all()

    def wcheck(s, datas, ads):
        ok_ref, st_ref = eng.pedersen_verify_wire(B, datas, s, ads, status=True)
        ok_o, st_o = O.pedersen_verify_wire(B, datas, s, ads, status=True)
        assert np.array_equal(ok_o, ok_ref) and np.array_equal(st_o, st_ref)
        all_ok, ok, st = eng.pedersen_batch_verify_wire(B, datas, s, ads, per_item=True, status=True)
        assert all_ok == bool(ok_ref.all()) and np.array_equal(ok, ok_ref) and np.array_equal(st, st_ref)
        return all_ok, ok_ref

    assert wcheck(sig, d["alphas"], d["ads"])[0] is True
    L = 32
    s2 = sig.copy(); s2[n // 2, 4 * L + 5] ^= 0x08                                  # s corrupted
    assert wcheck(s2, d["alphas"], d["ads"])[0] is False
    s3 = sig.copy(); s3[0, 4 * L + 63] = 0xff                                       # sb not canonical -> InvalidData
    assert wcheck(s3, d["alphas"], d["ads"])[0] is False
    s4 = sig.copy(); s4[n - 1, 2 * L + 3] ^= 0x40                                   # R's encoding damaged
    assert wcheck(s4, d["alphas"], d["ads"])[0] is False
    datas = list(d["alphas"]); datas[5] = datas[5] + b"x"                           # another input
    assert wcheck(sig, datas, d["ads"])[0] is False
    # a torsion point inside an encoded signature: Ok + (0, -1) is rejected by the decoder's subgroup test
    s5 = sig.copy()
    Ok = O.point_decode(0, bytes(s5[7, 3 * L:4 * L]))[0][0]
    s5[7, 3 * L:4 * L] = O.point_encode(0, pt(Cv.add(xy(Ok), T2)).reshape(1, 64))[0]
    all_ok, ok = wcheck(s5, d["alphas"], d["ads"])
    assert all_ok is False and ok[7] == 0


def test_kernel_timings_name_the_new_kernels(eng):
    d = make_batch(eng, 300)
    eng.enable_kernel_timing(True)
    try:
        assert eng.pedersen_batch_verify(B, d["inp"], d["out"], d["proof"], d["ads"]) is True
        names = {k for k, _ in eng.kernel_timings()}
        sig, _, _ = eng.pedersen_sign_wire(B, d["sk"], d["alphas"], d["ads"])
        assert eng.pedersen_batch_verify_wire(B, d["alphas"], sig, d["ads"]) is True
        wnames = {k for k, _ in eng.kernel_timings()}
    finally:
        eng.enable_kernel_timing(False)
    new = {"pedersen_batch_sum", "te_msm_histogram", "te_msm_scan", "te_msm_scatter", "te_msm_accumulate", "te_msm_chunks", "te_msm_window_sum", "te_msm_final"}
    assert new | {"pedersen_batch_prep"} <= names
    assert new | {"pedersen_batch_prep_wire", "decode_checked"} <= wnames
