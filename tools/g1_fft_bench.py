"""The G1 FFT (vrfs_g1_fft_batch, Engine.g1_fft): the inverse transform of a true-tau monomial SRS [tau^j] G1 into its Lagrange
basis, the ring-setup step of ring-proof's `RingBuilderKey::from_srs`.

Every timed output is checked before it counts: at 2^11 and 2^14 against [L_i(tau)] G1 from big integers; at every size by the round
trip (the forward transform gives the powers back) and by the commitment of a half-full ring, equal over a handle of the derived basis
(lagrange=True) and over the monomial handle (lagrange=False).  tau is seeded; the powers come from the CPU oracle.  Then per size,
after a warm-up: the wall time of the inverse call from page-locked buffers (median of --repeats), and in separate runs the device
time per launch name from the kernel-timing API (g1_fft_stage summed over the stages, and listed per stage), for the inverse and the
forward transform (their store kernels differ by the [1/n] scaling).  The GPU's name and power limit are read in the same run.

    python tools/g1_fft_bench.py --log2 11,14,16,17 --out profiles/r3_g1_fft_bench.json
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
import vectors as V  # noqa: E402
from ark_ec_vrfs_b200 import api  # noqa: E402
from ark_ec_vrfs_b200.engine import _p  # noqa: E402

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
ROOT_OF_UNITY = 10238227357739495823651030575849232062558860180284477541189508159991286009131   # Fr::TWO_ADIC_ROOT_OF_UNITY
TAU = int.from_bytes(hashlib.sha512(b"vrfs-b200-g1-fft-bench-tau").digest(), "little") % R


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [x.strip() for x in out.splitlines()[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:            # the numbers are still recorded, marked as lacking their context
        return dict(gpu="unknown (%s)" % e)


def le32(vals):
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), np.uint8).reshape(-1, 32).copy()


def lagrange_scalars(lg):
    n = 1 << lg; w = pow(ROOT_OF_UNITY, 1 << (32 - lg), R)
    zn = (pow(TAU, n, R) - 1) * pow(n, -1, R) % R
    return [zn * x * pow((TAU - x) % R, -1, R) % R for x in (pow(w, i, R) for i in range(n))]


def scalar_mults(lg):
    """twiddle multiplications of the network (butterflies with w != 1: sum_s n/2 - n/2^s) plus the n of the [1/n] scaling"""
    n = 1 << lg
    return (n // 2) * lg - n + 1 + n


def check(eng, suite, lg, mono, lag, keys, tail):
    res = dict(n=1 << lg)
    if lg <= 14:
        assert np.array_equal(lag, O.g1_mul_gen(le32(lagrange_scalars(lg)))), lg
        res["big_integer_lagrange_basis"] = True
    assert np.array_equal(eng.g1_fft(lag), mono), lg
    res["round_trip"] = True
    ring = keys[:(1 << lg) // 2]
    c_lag = api.RingContext(suite, lag, True, keys[0], tail)
    c_mono = api.RingContext(suite, mono, False, keys[0], tail)
    try:
        want = c_mono.verifier_key_commitment(ring)
        assert want.any()
        assert np.array_equal(c_lag.verifier_key_commitment(ring, incremental=False), want), lg
        assert np.array_equal(c_lag.verifier_key_commitment(ring, incremental=True), want), lg
    finally:
        c_lag.release(); c_mono.release()
    res["ring_commitment_equal"] = dict(ring_size=len(ring), full=True, delta=True)
    return res


def timed(eng, call):
    eng.enable_kernel_timing(True)
    call()
    kernels = eng.kernel_timings()
    eng.enable_kernel_timing(False)
    split, stages = {}, []
    for name, ms in kernels:
        split[name] = split.get(name, 0.0) + ms
        if name == "g1_fft_stage":
            stages.append(ms)
    return split, stages


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", default="11,14,16,17")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_g1_fft_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), tau_seed="sha512(b'vrfs-b200-g1-fft-bench-tau') mod r", cases=[])
    sizes = [int(x) for x in a.log2.split(",")]
    _, pk, inp, _ = V.make_keys_inputs(O.BANDERSNATCH, 1024)
    keys, tail = np.tile(pk, ((1 << max(sizes)) // 2 // 1024 + 1, 1)), inp[:255]
    med = lambda xs: float(np.median(xs))
    with vrfs.Engine(0) as eng:
        suite = api.Suite(vrfs.BANDERSNATCH, eng)
        for lg in sizes:
            n = 1 << lg
            t0 = time.perf_counter()
            mono = O.g1_mul_gen(le32([pow(TAU, j, R) for j in range(n)]))
            oracle_s = time.perf_counter() - t0
            src, out = vrfs.host_copy(mono), vrfs.host_buffer((n, 96))
            call = lambda inverse: eng._call("vrfs_g1_fft_batch", lg, inverse, _p(src), _p(out))
            for _ in range(a.warmup):
                call(1)
            wall = []
            for _ in range(a.repeats):
                out[:] = 0
                t0 = time.perf_counter()
                call(1)                                                  # returns after the call's stream synchronise
                wall.append(time.perf_counter() - t0)
            lag = np.array(out)
            chk = check(eng, suite, lg, mono, lag, keys, tail)            # the timed output, checked before it counts
            inv_runs = [timed(eng, lambda: call(1)) for _ in range(3)]
            assert np.array_equal(np.array(out), lag)
            call(0)
            fwd_runs = [timed(eng, lambda: call(0)) for _ in range(3)]
            assert np.array_equal(eng.g1_fft(np.array(out), inverse=True), mono)   # the timed forward output, checked
            split = lambda runs, name: med([s.get(name, 0.0) for s, _ in runs])
            device = {name: split(inv_runs, name) for name in ("ntt_twiddles", "g1_fft_load", "g1_fft_stage", "g1_fft_store")}
            total = sum(device.values())
            case = dict(n=n, check=chk, oracle_powers_s=oracle_s,
                        inverse_wall_ms=med(wall) * 1e3, inverse_wall_ms_all=[w * 1e3 for w in wall],
                        inverse_device_ms=device, inverse_device_total_ms=total,
                        inverse_stage_ms=[float(np.median(x)) for x in zip(*[st for _, st in inv_runs])],
                        forward_device_ms={name: split(fwd_runs, name) for name in ("ntt_twiddles", "g1_fft_load", "g1_fft_stage", "g1_fft_store")},
                        scalar_mults=scalar_mults(lg), scalar_mults_per_s=scalar_mults(lg) / (total * 1e-3) if total else None)
            res["cases"].append(case)
            print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in case.items() if k not in ("inverse_wall_ms_all", "inverse_stage_ms")}), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
