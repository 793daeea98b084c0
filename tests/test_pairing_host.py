"""CPU: the engine's BLS12-381 pairing code (csrc/pairing.cuh, compiled for the host by tests/host_emul) against the naive
big-integer oracle (oracle/pairing_ref.py): every tower operation, the Miller loop + final exponentiation, bilinearity, and
malformed inputs.  The same header is what the CUDA kernels execute (tests/test_gpu_pairing.py)."""
import ctypes as C
import os
import random
import subprocess
import sys

import pytest

from oracle import pairing_ref as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emu():
    subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "tests", "host_emul")], check=True)
    lib = C.CDLL(os.path.join(ROOT, "tests", "host_emul", "libhostemu.so"))
    lib.hostemu_pairing_product.restype = C.c_int
    return lib


def rand_f12(rnd):
    f2 = lambda: (rnd.randrange(P.Q), rnd.randrange(P.Q))
    f6 = lambda: (f2(), f2(), f2())
    return (f6(), f6())


def op(emu, o, a, b=None):
    out = C.create_string_buffer(576)
    emu.hostemu_f12_op(o, P.f12_to_bytes(a), P.f12_to_bytes(b if b is not None else P.F12_ONE), out)
    return P.f12_from_bytes(out.raw)


def test_tower_operations(emu):
    rnd = random.Random(12)
    for _ in range(20):
        a, b = rand_f12(rnd), rand_f12(rnd)
        assert op(emu, 0, a, b) == P.f12_mul(a, b)
        assert op(emu, 1, a) == P.f12_sqr(a)
        assert op(emu, 2, a) == P.f12_inv(a)
        assert op(emu, 3, a) == P.f12_pow(a, P.Q)
        assert op(emu, 4, a) == P.f12_pow(a, P.Q ** 2)
        assert op(emu, 7, a) == P.f12_conj(a)
        sparse = ((b[0][0], b[0][1], P.F2_ZERO), (P.F2_ZERO, b[1][1], P.F2_ZERO))
        assert op(emu, 6, a, b) == P.f12_mul(a, sparse)
    edge = [P.F12_ONE, P.f12_from_fq(P.Q - 1), ((P.F2_ZERO,) * 3, ((1, 0), P.F2_ZERO, P.F2_ZERO))]
    for a in edge:
        assert op(emu, 1, a) == P.f12_sqr(a) and op(emu, 2, a) == P.f12_inv(a)


def test_cyclotomic_operations_and_final_exponentiation(emu):
    rnd = random.Random(13)
    for _ in range(3):
        a = rand_f12(rnd)
        easy = P.f12_mul(P.f12_conj(a), P.f12_inv(a))
        m = P.f12_mul(P.f12_pow(easy, P.Q ** 2), easy)                    # an element of the cyclotomic subgroup
        assert op(emu, 5, m) == P.f12_sqr(m)
        assert op(emu, 8, m) == P.f12_conj(P.f12_pow(m, P.X_ABS))          # m^x, x = -X_ABS
        assert op(emu, 9, a) == P.gt_cubed(P.final_exponentiation(a))


def g1b(p): return P.g1_to_bytes(p)
def g2b(p): return P.g2_to_bytes(p)


def test_pairing_matches_oracle_and_is_bilinear(emu):
    rnd = random.Random(14)
    out = C.create_string_buffer(576)
    for _ in range(3):
        a, b = rnd.randrange(1, P.R), rnd.randrange(1, P.R)
        p, q = P.g1_mul(a, P.G1_GEN), P.g2_mul(b, P.G2_GEN)
        assert emu.hostemu_pairing_product(1, g1b(p), g2b(q), 0, out) == 0
        assert P.f12_from_bytes(out.raw) == P.gt_cubed(P.pairing(p, q))
        # e(aG1, bG2) * e(-(ab)G1, G2) = 1, through the negate mask and through an explicitly negated point
        ab = P.g1_mul(a * b, P.G1_GEN)
        assert emu.hostemu_pairing_product(2, g1b(p) + g1b(ab), g2b(q) + g2b(P.G2_GEN), 2, None) == 1
        assert emu.hostemu_pairing_product(2, g1b(p) + g1b(P.g1_neg(ab)), g2b(q) + g2b(P.G2_GEN), 0, None) == 1
        assert emu.hostemu_pairing_product(2, g1b(p) + g1b(ab), g2b(q) + g2b(P.G2_GEN), 0, None) == 0
        # three pairs: e(aG, Q) e(bG, Q) e(-(a+b)G, Q) = 1
        s = P.g1_mul(a + b, P.G1_GEN)
        assert emu.hostemu_pairing_product(3, g1b(p) + g1b(P.g1_mul(b, P.G1_GEN)) + g1b(s), g2b(q) * 3, 4, None) == 1


def test_lane_programs_match_oracle(emu):
    """the warp-cooperative form (csrc/pairing_coop.cuh + the tables of tools/gen_pairing_prog.py), all lanes played on the host"""
    rnd = random.Random(16)
    emu.hostemu_pairing_product_lanes.restype = C.c_int
    out, out1 = C.create_string_buffer(576), C.create_string_buffer(576)
    for trial in range(3):
        a, b, c, d = (rnd.randrange(1, P.R) for _ in range(4))
        p1, q1, p2, q2 = P.g1_mul(a, P.G1_GEN), P.g2_mul(b, P.G2_GEN), P.g1_mul(c, P.G1_GEN), P.g2_mul(d, P.G2_GEN)
        g1, g2 = g1b(p1) + g1b(p2), g2b(q1) + g2b(q2)
        assert emu.hostemu_pairing_product_lanes(g1, g2, trial, out) == 0
        e2 = P.pairing(P.g1_neg(p2) if trial & 2 else p2, q2)
        e1 = P.pairing(P.g1_neg(p1) if trial & 1 else p1, q1)
        assert P.f12_from_bytes(out.raw) == P.gt_cubed(P.f12_mul(e1, e2))
        assert emu.hostemu_pairing_product(2, g1, g2, trial, out1) == 0 and out1.raw == out.raw
        ab = P.g1_mul(a * b, P.G1_GEN)
        assert emu.hostemu_pairing_product_lanes(g1b(p1) + g1b(ab), g2b(q1) + g2b(P.G2_GEN), 2, out) == 1
        assert P.f12_from_bytes(out.raw) == P.F12_ONE
    # an identity in the product and malformed points fall back to / agree with the one-thread form
    assert emu.hostemu_pairing_product_lanes(bytes(96) + g1b(p2), g2b(q1) + g2b(q2), 0, out) == 0
    assert P.f12_from_bytes(out.raw) == P.gt_cubed(P.pairing(p2, q2))
    bad = bytearray(g1b(p1) + g1b(p2)); bad[99] ^= 1
    assert emu.hostemu_pairing_product_lanes(bytes(bad), g2b(q1) + g2b(q2), 0, None) == 2


def test_lane_program_generator_self_check():
    """the generator's own model run of the emitted tables (twin and oracle equality) passes, and the committed tables are current"""
    subprocess.run([sys.executable, os.path.join(ROOT, "tools", "gen_pairing_prog.py"), "--check"], check=True, capture_output=True)


def test_pairing_identity_and_malformed_inputs(emu):
    q = P.g2_mul(7, P.G2_GEN)
    out = C.create_string_buffer(576)
    assert emu.hostemu_pairing_product(1, bytes(96), g2b(q), 0, out) == 1 and P.f12_from_bytes(out.raw) == P.F12_ONE    # e(O, Q) = 1
    assert emu.hostemu_pairing_product(1, g1b(P.G1_GEN), bytes(192), 0, None) == 1
    bad = bytearray(g1b(P.G1_GEN)); bad[3] ^= 1
    assert emu.hostemu_pairing_product(1, bytes(bad), g2b(q), 0, None) == 2                       # off the curve
    bad2 = bytearray(g2b(q)); bad2[100] ^= 1
    assert emu.hostemu_pairing_product(1, g1b(P.G1_GEN), bytes(bad2), 0, None) == 2
    assert emu.hostemu_pairing_product(1, b"\xff" * 96, g2b(q), 0, None) == 2                      # non-canonical


def test_kzg_batch_check_model():
    """the oracle's aggregated KZG check accepts honest openings under a public tau and rejects forged ones"""
    rnd = random.Random(15)
    tau = rnd.randrange(1, P.R)
    tau_g2 = P.g2_mul(tau, P.G2_GEN)
    polys = [[rnd.randrange(P.R) for _ in range(5)] for _ in range(4)]
    zs = [rnd.randrange(P.R) for _ in polys]
    rs = [rnd.randrange(P.R) for _ in polys]
    Cs = [P.kzg_commit(c, tau) for c in polys]
    vs, Ws = zip(*(P.kzg_open(c, z, tau) for c, z in zip(polys, zs)))
    assert P.kzg_batch_verify(Cs, zs, list(vs), list(Ws), rs, P.G2_GEN, tau_g2)
    bad = list(vs); bad[2] = (bad[2] + 1) % P.R
    assert not P.kzg_batch_verify(Cs, zs, bad, list(Ws), rs, P.G2_GEN, tau_g2)
    badW = list(Ws); badW[0] = P.g1_add(badW[0], P.G1_GEN)
    assert not P.kzg_batch_verify(Cs, zs, list(vs), badW, rs, P.G2_GEN, tau_g2)
