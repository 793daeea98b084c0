"""CPU check of the KZG opening quotient q = (p - p(z)) / (X - z) and v = p(z) (csrc/kzg_open.cuh, the per-thread pieces of the
k_kzg_quotient_* kernels): compiled for the host, run through the kernels' three phases for one polynomial and compared with the
big-integer recurrence at lengths around the chunk boundaries, z in {0, 1, r - 1, random} and coefficients 2^256 - 1."""
import ctypes as C
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def open_ref(a, z):                  # a: ints mod r, low to high
    q, acc = [0] * max(len(a) - 1, 0), 0
    for j in range(len(a) - 1, 0, -1):
        acc = (acc * z + a[j]) % R; q[j - 1] = acc
    return ((acc * z + a[0]) % R if a else 0), q


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostemu_kzg") / "libhostemu_kzg.so")
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-fno-strict-aliasing", "-std=c++17", "-fPIC", "-shared", "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "hostemu_kzg.cpp")], check=True)
    lib = C.CDLL(so)
    lib.hostemu_kzg_open.argtypes = [C.c_uint32, C.c_uint32, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p]
    return lib


def open_emu(emu, raw, z, n):
    """the emulated kernels on raw 256-bit coefficients: (v, the n rows of the quotient column)"""
    v, q = C.create_string_buffer(32), C.create_string_buffer(32 * max(n, 1))
    emu.hostemu_kzg_open(len(raw), n, b"".join(x.to_bytes(32, "little") for x in raw), z.to_bytes(32, "little"), v, q)
    return int.from_bytes(v.raw, "little"), [int.from_bytes(q.raw[32 * i:32 * i + 32], "little") for i in range(n)]


def test_chunk_is_a_power_of_two_of_whole_segments(emu):
    ch = emu.hostemu_kzg_chunk()
    assert ch >= 256 and ch & (ch - 1) == 0


@pytest.mark.parametrize("z_kind", ["zero", "one", "r-1", "random"])
def test_quotient_matches_the_recurrence(emu, z_kind):
    ch = emu.hostemu_kzg_chunk()
    rnd = random.Random(z_kind)
    z = {"zero": 0, "one": 1, "r-1": R - 1, "random": rnd.randrange(R)}[z_kind]
    for length in (0, 1, 2, 8, 9, ch - 1, ch, ch + 1, 3 * ch + 5):
        for fill in ("max", "random"):
            raw = [(1 << 256) - 1] * length if fill == "max" else [rnd.randrange(1 << 256) for _ in range(length)]
            n = length + (ch + 3 if length % 2 else 1)               # rows above the polynomial, whole chunks of them for odd lengths
            v, q = open_emu(emu, raw, z, n)
            v_ref, q_ref = open_ref([x % R for x in raw], z)
            assert v == v_ref, (length, fill)
            assert q == q_ref + [0] * (n - len(q_ref)), (length, fill)


def test_opening_identity_holds(emu):
    """p(X) - p(z) = q(X) (X - z) at a random X: the quotient is the one KZG commits to"""
    ch = emu.hostemu_kzg_chunk()
    rnd = random.Random(7)
    a = [rnd.randrange(R) for _ in range(2 * ch + 17)]
    z, x = rnd.randrange(R), rnd.randrange(R)
    v, q = open_emu(emu, a, z, len(a))
    ev = lambda c, t: sum(ci * pow(t, j, R) for j, ci in enumerate(c)) % R
    assert (ev(a, x) - v) % R == ev(q, x) * (x - z) % R
    # z a root of p: v = 0
    a[0] = (a[0] - ev(a, z)) % R
    assert open_emu(emu, a, z, len(a))[0] == 0
