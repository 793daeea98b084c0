"""CPU check of the evaluation and aggregation of vrfs_kzg_open_aggregated_batch (csrc/kzg_open.cuh, the per-thread pieces of
k_kzg_eval_chunks, k_kzg_eval_finish and k_kzg_aggregate): compiled for the host, run the way the kernels run them (the ordered
span reduction lane by lane, Horner over the chunk values, the aggregation per segment) and compared with big integers at lengths
around the chunk boundaries, in groups of mixed lengths, with coefficients, points and nu >= r."""
import ctypes as C
import os
import random
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def ev(a, z):
    acc = 0
    for c in reversed(a):
        acc = (acc * z + c) % R
    return acc


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("hostemu_kzg_agg") / "libhostemu_kzg_agg.so")
    subprocess.run([os.environ.get("CXX", "g++"), "-O2", "-fno-strict-aliasing", "-std=c++17", "-fPIC", "-shared", "-o", so,
                    os.path.join(ROOT, "tests", "host_emul", "hostemu_kzg_agg.cpp")], check=True)
    lib = C.CDLL(so)
    lib.hostemu_kzg_agg.argtypes = [C.c_uint32, C.c_uint32, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p,
                                    C.c_char_p, C.c_char_p]
    return lib


def u64s(xs):
    return b"".join(int(x).to_bytes(8, "little") for x in xs)


def le(xs):
    return b"".join(int(x).to_bytes(32, "little") for x in xs)


def run(emu, groups, zs, nus):
    """groups: lists of raw 256-bit coefficient lists; zs one raw point per group, nus one raw nu per polynomial ->
    (values per polynomial, aggregated rows per group), as ints"""
    polys = [p for g in groups for p in g]
    group_off, coeff_off, row_off = [0], [0], [0]
    for g in groups:
        group_off.append(group_off[-1] + len(g))
        row_off.append(row_off[-1] + max([len(p) for p in g], default=0))
    for p in polys:
        coeff_off.append(coeff_off[-1] + len(p))
    vals = C.create_string_buffer(32 * max(len(polys), 1))
    rows = C.create_string_buffer(32 * max(row_off[-1], 1))
    emu.hostemu_kzg_agg(len(groups), len(polys), u64s(group_off), u64s(coeff_off), le([c for p in polys for c in p]) or b"\0" * 32,
                        le(zs), le(nus) or b"\0" * 32, vals, u64s(row_off), rows)
    ints = lambda b, k: [int.from_bytes(b[32 * i:32 * i + 32], "little") for i in range(k)]
    r = ints(rows.raw, row_off[-1])
    return ints(vals.raw, len(polys)), [r[row_off[g]:row_off[g + 1]] for g in range(len(groups))]


def expect(groups, zs, nus):
    vals, rows, i = [], [], 0
    for g, z in zip(groups, zs):
        width = max([len(p) for p in g], default=0)
        agg = [0] * width
        for p in g:
            vals.append(ev([c % R for c in p], z % R))
            for j, c in enumerate(p):
                agg[j] = (agg[j] + nus[i] % R * (c % R)) % R
            i += 1
        rows.append(agg)
    return vals, rows


def test_chunk_is_a_power_of_two_of_whole_segments(emu):
    ch = emu.hostemu_kzg_agg_chunk()
    assert ch >= 256 and ch & (ch - 1) == 0


@pytest.mark.parametrize("z_kind", ["zero", "one", "r-1", "random"])
def test_single_lengths(emu, z_kind):
    """one polynomial per group at every length around the chunk boundaries, nu = 1: the values are p(z), the rows p itself"""
    ch = emu.hostemu_kzg_agg_chunk()
    rnd = random.Random(z_kind)
    for length in (0, 1, 2, ch - 1, ch, ch + 1, 3 * ch + 5):
        z = {"zero": 0, "one": 1, "r-1": R - 1, "random": rnd.randrange(R)}[z_kind]
        p = [rnd.randrange(R) for _ in range(length)]
        vals, rows = run(emu, [[p]], [z], [1])
        assert vals == [ev(p, z)], length
        assert rows == [p], length


def test_mixed_groups(emu):
    """groups of mixed lengths (empty groups and polynomials among them), raw inputs >= r, nu = 0 and r - 1"""
    ch = emu.hostemu_kzg_agg_chunk()
    rnd = random.Random(11)
    raw = lambda: rnd.choice([rnd.randrange(1 << 256), (1 << 256) - 1, R, rnd.randrange(R)])
    shapes = [[ch, ch - 1, ch + 1, 0, 1, 3 * ch + 5], [], [0], [1, 1], [2 * ch, 17, 3 * ch + 5, ch], [ch + 1]]
    groups = [[[raw() for _ in range(n)] for n in g] for g in shapes]
    zs = [raw() for _ in groups]
    n_polys = sum(len(g) for g in groups)
    nus = [raw() for _ in range(n_polys)]
    nus[1], nus[2] = 0, R - 1
    assert run(emu, groups, zs, nus) == expect(groups, zs, nus)


def test_ring_prover_shape(emu):
    """8 columns of length n and one of n - 3 at zeta, the linearisation polynomial alone at zeta omega with nu = 1"""
    ch = emu.hostemu_kzg_agg_chunk()
    n = 2 * ch
    rnd = random.Random(3)
    groups = [[[rnd.randrange(R) for _ in range(n)] for _ in range(8)] + [[rnd.randrange(R) for _ in range(n - 3)]],
              [[rnd.randrange(R) for _ in range(n)]]]
    zs = [rnd.randrange(R), rnd.randrange(R)]
    nus = [rnd.randrange(R) for _ in range(9)] + [1]
    vals, rows = run(emu, groups, zs, nus)
    assert (vals, rows) == expect(groups, zs, nus)
    # the aggregated value the quotient pass yields, P_g(z_g), is sum nu_i v_i
    for g, (rows_g, z) in enumerate(zip(rows, zs)):
        lo = sum(len(x) for x in groups[:g])
        assert ev(rows_g, z) == sum(nus[lo + i] * vals[lo + i] for i in range(len(groups[g]))) % R
