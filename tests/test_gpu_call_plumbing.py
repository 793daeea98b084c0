"""GPU tests of the host plumbing shared by the batch entry points: kernel-timing names, the timings of a host-buffer verify
that runs in two pieces, and the suite check of every entry point that takes a suite."""
import ctypes as C

import numpy as np
import pytest

import oracle_lib as O
import vectors as V


@pytest.fixture(scope="module")
def eng():
    import ark_ec_vrfs_b200 as vrfs
    e = vrfs.Engine(0)
    yield e
    e.close()


def _timed(eng, call):
    eng.enable_kernel_timing(True)
    try:
        return call(), [name for name, _ in eng.kernel_timings()]
    finally:
        eng.enable_kernel_timing(False)


@pytest.mark.gpu
def test_pedersen_verify_timings_name_each_linear_combination(eng):
    """T1 = s*I - c*O is lincomb<2,0> and T2 = s*G + sb*B - c*Yb is lincomb<1,2>; no one-variable-base lincomb<1,0> runs"""
    sk, _, inp, out = V.make_keys_inputs(O.BANDERSNATCH, 64)
    proof, _ = eng.pedersen_prove(O.BANDERSNATCH, sk, inp, out)
    ok, names = _timed(eng, lambda: eng.pedersen_verify(O.BANDERSNATCH, inp, out, proof))
    assert ok.all() and "lincomb<2,0>" in names and "lincomb<1,2>" in names and "lincomb<1,0>" not in names


@pytest.mark.gpu
def test_piecewise_host_verify_times_every_piece(eng):
    """above three resident waves of the lincomb grid (SMs x 2 x 256 items each) a host-buffer verify runs in two pieces"""
    import torch
    import ark_ec_vrfs_b200 as vrfs
    base, n = 512, 3 * torch.cuda.get_device_properties(0).multi_processor_count * 2 * 256 + 1
    sk0, pk0, inp0, out0 = V.make_keys_inputs(O.BANDERSNATCH, base)
    c0, s0 = eng.ietf_prove(O.BANDERSNATCH, sk0, inp0, out0)
    pk, inp, out, c, s = (vrfs.host_copy(a[np.arange(n) % base]) for a in (pk0, inp0, out0, c0, s0))
    ok, names = _timed(eng, lambda: eng.ietf_verify(O.BANDERSNATCH, pk, inp, out, c, s))
    assert ok.all() and names.count("ietf_verify_finish") == 2


# every entry point that takes a suite, with the number of buffer arguments after (ctx, suite, n)
SUITE_CALLS = {
    "vrfs_secret_from_seed_batch": 4, "vrfs_data_to_point_batch": 4, "vrfs_output_batch": 3, "vrfs_point_to_hash_batch": 2,
    "vrfs_point_encode_batch": 2, "vrfs_point_decode_batch": 3, "vrfs_nonce_batch": 3, "vrfs_ietf_prove_batch": 7,
    "vrfs_ietf_verify_batch": 9, "vrfs_ietf_verify_batch_dev": 9, "vrfs_pedersen_prove_batch": 7, "vrfs_pedersen_verify_batch": 7,
    "vrfs_pedersen_prove_compressed_batch": 7, "vrfs_pedersen_verify_compressed_batch": 7, "vrfs_point_decode_checked_batch": 3,
    "vrfs_subgroup_check_batch": 2, "vrfs_ietf_sign_wire_batch": 7, "vrfs_ietf_verify_wire_batch": 9,
    "vrfs_pedersen_sign_wire_batch": 8, "vrfs_pedersen_verify_wire_batch": 7,
}


@pytest.mark.gpu
@pytest.mark.parametrize("fn", sorted(SUITE_CALLS))
def test_unknown_suite_is_a_bad_argument(eng, fn):
    """a suite value outside vrfs_suite, with buffers that are otherwise accepted (zeros: empty variable-length items)"""
    import torch
    from ark_ec_vrfs_b200 import _lib
    buf = torch.zeros(1 << 14, dtype=torch.uint8, device="cuda" if fn.endswith("_dev") else "cpu")
    lib = _lib.load()
    for suite in (6, 0x7fffffff, -1):                                 # 6 = VRFS_SUITE_COUNT
        st = getattr(lib, fn)(eng._ctx, C.c_int(suite), C.c_size_t(4), *[C.c_void_p(buf.data_ptr())] * SUITE_CALLS[fn])
        assert st == _lib.BAD_ARG and "unknown suite %d" % suite in lib.vrfs_last_error(eng._ctx).decode()
