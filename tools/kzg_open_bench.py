"""KZG opening proofs (vrfs_kzg_open_batch, PreparedBases.kzg_open) against their floor, the prepared MSM of the same k columns
(PreparedBases.msm) over the same handle.

Correctness first, on true-tau monomial SRS of 2^11 and 2^14 points: values against big integers, and the openings with the
commitments of the same handle accepted by the engine's batched KZG check (a changed value rejected).  Then per (n, k): the wall
time of each call from page-locked buffers, the two calls alternated after a warm-up of every shape, and in separate timed runs the
device time of the quotient kernels (kzg_quotient_*) and of the MSM kernels (msm_*) from the kernel-timing API.  The timed SRS is a
tile of 1024 distinct points (the MSM's cost does not depend on the points); handles are prepared with the default plan (the
multiples table up to 2^14, the buckets above).  The GPU's name and power limit are read in the same run.  Writes JSON.

    python tools/kzg_open_bench.py --log2 11,14,16,17 --k 1,3,32 --out profiles/r3_kzg_open_bench.json
"""
import argparse
import hashlib
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


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def ints(a):
    return [int.from_bytes(r.tobytes(), "little") for r in np.asarray(a, np.uint8).reshape(-1, 32)]


def rand_fr(rng, shape):
    a = rng.integers(0, 256, size=shape + (32,), dtype=np.uint8)
    a[..., 31] &= 0x3F                                                   # < 2^254 < r
    return a


def check(eng, lg, k=3):
    """true-tau SRS of 2^lg points: k openings of full-length polynomials verified by vrfs_kzg_batch_verify"""
    n = 1 << lg
    tau = int.from_bytes(hashlib.sha512(b"kzg-open-bench-tau").digest(), "little") % R
    h = eng.msm_g1_prepare(O.g1_mul_gen(le32([pow(tau, j, R) for j in range(n)])))
    rng = np.random.default_rng(lg)
    a, z = rand_fr(rng, (k, n)), rand_fr(rng, (k,))
    values, proofs = h.kzg_open(a, z)
    for i in range(k):
        acc, zi = 0, ints(z[i:i + 1])[0]
        for c in reversed(ints(a[i])):
            acc = (acc * zi + c) % R
        assert ints(values[i:i + 1])[0] == acc, (lg, i)
    C = h.msm(a.reshape(-1, 32), k)
    rs = rand_fr(rng, (k,))
    g2, tau_g2 = np.frombuffer(P.g2_to_bytes(P.G2_GEN), np.uint8), np.frombuffer(P.g2_to_bytes(P.g2_mul(tau, P.G2_GEN)), np.uint8)
    ok = eng.kzg_batch_verify(C, z, values, proofs, rs, g2, tau_g2)
    bad = values.copy(); bad[0, 0] ^= 1
    rejected = eng.kzg_batch_verify(C, z, bad, proofs, rs, g2, tau_g2)
    h.release()
    assert ok == 1 and rejected == 0, (lg, ok, rejected)
    return dict(n=n, k=k, accepted=ok, tampered_value_accepted=rejected)


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
    ap.add_argument("--log2", default="11,14,16,17")
    ap.add_argument("--k", default="1,3,32")
    ap.add_argument("--check-log2", default="11,14")
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_kzg_open_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), checks=[], cases=[])
    with vrfs.Engine(0) as eng:
        for lg in [int(x) for x in a.check_log2.split(",") if x]:
            res["checks"].append(check(eng, lg))
            print(json.dumps(res["checks"][-1]), flush=True)
        tile = O.g1_mul_gen(rand_fr(np.random.default_rng(99), (1024,)))
        for lg in [int(x) for x in a.log2.split(",")]:
            n = 1 << lg
            h = eng.msm_g1_prepare(np.tile(tile, (n // 1024, 1)))
            for k in [int(x) for x in a.k.split(",")]:
                rng = np.random.default_rng(1000 * lg + k)
                coeffs, zs = vrfs.host_copy(rand_fr(rng, (k, n))), vrfs.host_copy(rand_fr(rng, (k,)))
                cols = coeffs.reshape(-1, 32)
                calls = dict(open=lambda: h.kzg_open(coeffs, zs), msm=lambda: h.msm(cols, k))
                for _ in range(a.warmup):
                    for call in calls.values():
                        call()
                wall = {kind: [] for kind in calls}
                for _ in range(a.repeats):
                    for kind, call in calls.items():
                        t0 = time.perf_counter()
                        call()                                           # returns after the call's stream synchronise
                        wall[kind].append(time.perf_counter() - t0)
                kern = {kind: [timed(eng, call) for _ in range(3)] for kind, call in calls.items()}
                med = lambda xs: float(np.median(xs))
                quot = med([sum(v for name, v in s.items() if name.startswith("kzg_quotient")) for s in kern["open"]])
                msm_in_open = med([sum(v for name, v in s.items() if name.startswith("msm_")) for s in kern["open"]])
                msm_floor = med([sum(v for name, v in s.items() if name.startswith("msm_")) for s in kern["msm"]])
                case = dict(n=n, k=k, mode="table" if n <= 16384 else "buckets",
                            open_wall_ms=med(wall["open"]) * 1e3, msm_wall_ms=med(wall["msm"]) * 1e3,
                            open_wall_ms_all=[w * 1e3 for w in wall["open"]], msm_wall_ms_all=[w * 1e3 for w in wall["msm"]],
                            quotient_kernels_ms=quot, msm_kernels_in_open_ms=msm_in_open, msm_floor_kernels_ms=msm_floor,
                            quotient_share=quot / (quot + msm_in_open) if quot + msm_in_open else None,
                            open_kernels_ms=kern["open"][-1], msm_kernels_ms=kern["msm"][-1])
                res["cases"].append(case)
                print(json.dumps({key: (round(v, 4) if isinstance(v, float) else v) for key, v in case.items()
                                  if not key.endswith("_all") and key not in ("open_kernels_ms", "msm_kernels_ms")}), flush=True)
            h.release()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
