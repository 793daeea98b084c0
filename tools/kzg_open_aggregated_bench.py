"""Aggregated KZG openings (vrfs_kzg_open_aggregated_batch) in the shape of a ring prover's opening round, against the two ways
of getting the same openings from vrfs_kzg_open_batch over the same handle:

  aggregated  one call: group 0 = 8 columns of length n and one of n - 3 at zeta with nu_0..nu_8, group 1 = one polynomial of
              length n at zeta omega with nu = 1 -> 10 values, 2 aggregated values, 2 proofs;
  k2          P_0 = sum nu_i p_i aggregated on the host (Python integers, timed apart, once per size), then vrfs_kzg_open_batch
              of k = 2 (P_0 at zeta, the linearisation polynomial at zeta omega);
  k10         vrfs_kzg_open_batch of k = 10, every polynomial opened on its own (zero-padded to n).

Before any timing, per size: the aggregated call's values, aggregated values and proofs equal k2's byte for byte, its values
equal k10's, and its aggregated value of group 0 is sum nu_i v_i.  Then the wall time of each call from page-locked buffers, the
three alternated after a warm-up of every shape, and in separate timed runs the device time per kernel name from the
kernel-timing API.  The timed SRS is a tile of 1024 distinct points (the MSM's cost does not depend on the points); handles use
the default plan (the multiples table up to 2^14, the buckets above).  The GPU's name and power limit are read in the same run.
Writes JSON.

    python tools/kzg_open_aggregated_bench.py --log2 12,14,16,17 --out profiles/r3_kzg_open_aggregated_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ark_ec_vrfs_b200 as vrfs  # noqa: E402
import oracle_lib as O  # noqa: E402
from oracle import pairing_ref as P  # noqa: E402

R = P.R


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [x.strip() for x in out.splitlines()[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:            # the numbers are still recorded, marked as lacking their context
        return dict(gpu="unknown (%s)" % e)


def ints(a):
    return [int.from_bytes(r.tobytes(), "little") for r in np.asarray(a, np.uint8).reshape(-1, 32)]


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def rand_fr(rng, shape):
    a = rng.integers(0, 256, size=shape + (32,), dtype=np.uint8)
    a[..., 31] &= 0x3F                                                   # < 2^254 < r
    return a


def host_aggregate(cols, nus):
    """sum nu_i p_i over the host's big integers, (n, 32) canonical"""
    acc = [0] * cols.shape[1]
    for col, nu in zip(cols, ints(nus)):
        for j, c in enumerate(ints(col)):
            acc[j] = (acc[j] + nu * c) % R
    return le32(acc)


def timed(eng, call):
    eng.enable_kernel_timing(True)
    call()
    kernels = eng.kernel_timings()
    eng.enable_kernel_timing(False)
    split = {}
    for name, ms in kernels:
        split[name] = split.get(name, 0.0) + ms
    return split


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", default="12,14,16,17")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_kzg_open_aggregated_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), cases=[])
    with vrfs.Engine(0) as eng:
        tile = O.g1_mul_gen(rand_fr(np.random.default_rng(99), (1024,)))
        for lg in [int(x) for x in a.log2.split(",")]:
            n = 1 << lg
            h = eng.msm_g1_prepare(np.tile(tile, (n // 1024, 1)))
            rng = np.random.default_rng(lg)
            # ten polynomials zero-padded to n (the ninth is n - 3 long), points zeta and zeta omega, nu_9 = 1
            cols = rand_fr(rng, (10, n))
            cols[8, n - 3:] = 0
            zs = rand_fr(rng, (2,))
            nus = rand_fr(rng, (10,))
            nus[9] = le32([1])[0]
            lens = [n] * 8 + [n - 3, n]
            coeff_off = np.zeros(11, np.uint64); coeff_off[1:] = np.cumsum(lens)
            group_off = np.array([0, 9, 10], np.uint64)
            # page-locked inputs and outputs of every call
            flat = vrfs.host_copy(np.concatenate([cols[i, :lens[i]] for i in range(10)]))
            z_pin, nu_pin = vrfs.host_copy(zs), vrfs.host_copy(nus)
            vals, aggv, proofs = vrfs.host_copy(np.zeros((10, 32), np.uint8)), vrfs.host_copy(np.zeros((2, 32), np.uint8)), vrfs.host_copy(np.zeros((2, 96), np.uint8))
            t0 = time.perf_counter()
            p0 = host_aggregate(cols[:9], nus[:9])
            host_agg_ms = (time.perf_counter() - t0) * 1e3
            k2_coeffs = vrfs.host_copy(np.stack([p0, cols[9]]))
            k10_coeffs = vrfs.host_copy(cols)
            k10_zs = vrfs.host_copy(zs[[0] * 9 + [1]])
            p = lambda x: x.ctypes.data_as(C.c_void_p)

            def aggregated():
                eng._call("vrfs_kzg_open_aggregated_batch", h.handle, C.c_size_t(2), C.c_size_t(10), p(group_off), p(coeff_off), p(flat), p(z_pin),
                          p(nu_pin), p(vals), p(aggv), p(proofs))
            calls = dict(aggregated=aggregated, k2=lambda: h.kzg_open(k2_coeffs, z_pin), k10=lambda: h.kzg_open(k10_coeffs, k10_zs))
            # correctness before timing
            aggregated()
            v2, w2 = calls["k2"]()
            v10, _ = calls["k10"]()
            assert np.array_equal(aggv, v2) and np.array_equal(proofs, w2), n
            assert np.array_equal(vals, v10), n
            assert ints(aggv[:1])[0] == sum(x * y for x, y in zip(ints(nus[:9]), ints(vals[:9]))) % R, n
            for _ in range(a.warmup):
                for call in calls.values():
                    call()
            wall = {kind: [] for kind in calls}
            for _ in range(a.repeats):
                for kind, call in calls.items():
                    t0 = time.perf_counter()
                    call()                                               # returns after the call's stream synchronise
                    wall[kind].append(time.perf_counter() - t0)
            kern = {kind: [timed(eng, call) for _ in range(3)] for kind, call in calls.items()}
            med = lambda xs: float(np.median(xs))
            part = lambda kind, pre: med([sum(v for name, v in s.items() if name.startswith(pre)) for s in kern[kind]])
            case = dict(n=n, mode="table" if n <= 16384 else "buckets", host_aggregate_ms=host_agg_ms,
                        **{f"{kind}_wall_ms": med(wall[kind]) * 1e3 for kind in calls},
                        **{f"{kind}_device_ms": part(kind, "") for kind in calls},
                        aggregated_eval_ms=part("aggregated", "kzg_eval"), aggregated_aggregate_ms=part("aggregated", "kzg_aggregate"),
                        aggregated_quotient_ms=part("aggregated", "kzg_quotient"), aggregated_msm_ms=part("aggregated", "msm_"),
                        k2_quotient_ms=part("k2", "kzg_quotient"), k2_msm_ms=part("k2", "msm_"),
                        k10_quotient_ms=part("k10", "kzg_quotient"), k10_msm_ms=part("k10", "msm_"),
                        wall_ms_all={kind: [w * 1e3 for w in wall[kind]] for kind in calls},
                        kernels_ms={kind: kern[kind][-1] for kind in calls})
            res["cases"].append(case)
            print(json.dumps({key: (round(v, 4) if isinstance(v, float) else v) for key, v in case.items()
                              if key not in ("wall_ms_all", "kernels_ms")}), flush=True)
            h.release()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
