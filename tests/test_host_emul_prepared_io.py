"""CPU check of the prepared-input linear combination V = s*I_j - c*O (lincomb.cuh lincomb_io_item, the item function of the
k_lincomb_io kernel): compiled for the host with the input tables built by the GPU's table functions, and compared with the
Python curve model for the three pinned suites - neg masks, scalars 0, 1, r - 1 and random, and 16-byte challenges."""
import ctypes as C
import os
import random
import subprocess

import pytest

from oracle import pyref as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def emu_io(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostemu_io") / "libhostemu_io.so")
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-fno-strict-aliasing", "-std=c++17", "-fPIC", "-shared", "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "hostemu_io.cpp")], check=True)
    lib = C.CDLL(so)
    lib.hostemu_lincomb_io.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_uint32, C.c_char_p, C.c_char_p, C.c_char_p, C.c_uint32, C.c_int, C.c_char_p]
    return lib


def le(x):
    return x.to_bytes(32, "little")


def pt(P):
    return bytes(64) if P is None else le(P[0]) + le(P[1])      # short-Weierstrass identity = 64 zero bytes


@pytest.mark.parametrize("suite,cv", [(0, R.BANDERSNATCH), (1, R.ED25519), (2, R.P256)], ids=["bandersnatch", "ed25519", "p256"])
def test_lincomb_io_item_matches_curve_model(emu_io, suite, cv):
    r = cv.r
    rnd = random.Random(100 + suite)
    inputs = [cv.mul(rnd.randrange(1, r), cv.G) for _ in range(3)]
    ins = b"".join(pt(P) for P in inputs)
    cases = 0
    for t in range(24):
        j = t % 3
        O = cv.mul(rnd.randrange(1, r), cv.G)
        s = [0, 1, r - 1][t % 3] if t < 6 else rnd.randrange(r)
        short = t % 2 == 1                                          # a 16-byte challenge, its empty windows skipped
        c = rnd.randrange(1 << 128) if short else ([r - 1, 0, 1][t % 3] if t < 6 else rnd.randrange(r))
        if t in (7, 9):
            c = (1 << 128) - 1                                      # every bit of the short window set
        c_bits = 128 if short else 0
        neg = t % 4
        out = C.create_string_buffer(64)
        flags = emu_io.hostemu_lincomb_io(suite, 3, ins, j, le(s), pt(O), le(c), c_bits, neg, out)
        assert flags == 0b1111, (suite, t, flags)                   # O valid, all three input tables valid
        E = cv.add(cv.mul((-c if neg & 1 else c) % r, O), cv.mul((-s if neg & 2 else s) % r, inputs[j]))
        assert out.raw == pt(E), (suite, t, j, neg)
        cases += 1
    assert cases == 24


@pytest.mark.parametrize("suite,cv", [(0, R.BANDERSNATCH), (1, R.ED25519), (2, R.P256)], ids=["bandersnatch", "ed25519", "p256"])
def test_lincomb_io_item_flags_an_invalid_output_point(emu_io, suite, cv):
    """O off the curve clears the item's flag, as lincomb_item does for the variable bases of the gathered-input call"""
    r = cv.r
    I = cv.mul(12345, cv.G)
    O = cv.mul(777, cv.G)
    bad = le(O[0]) + le((O[1] + 1) % cv.p)
    out = C.create_string_buffer(64)
    flags = emu_io.hostemu_lincomb_io(suite, 1, pt(I), 0, le(5), bad, le(3), 0, 1, out)
    assert flags == 0b10, flags
    # an index out of range reads the table of input 0 (the gather kernel rejects the item)
    flags = emu_io.hostemu_lincomb_io(suite, 1, pt(I), 7, le(5), pt(O), le(3), 0, 1, out)
    assert flags == 0b11 and out.raw == pt(cv.add(cv.mul(5, I), cv.mul((-3) % r, O)))
