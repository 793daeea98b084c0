"""Serialised signatures verified against keys prepared from their encodings (vrfs_ietf_verify_prepared_wire_batch) against
vrfs_ietf_verify_wire_batch on the gathered encodings, on the same distinct signatures from the engine's signer: n signatures by K
signers, a random signer per signature, 8 bytes of VRF input data each, no ad.

Per (suite, K, n): device time (the sum of kernel_timings()) and end-to-end wall time of both calls from page-locked buffers
(vrfs.host_copy, results into page-locked arrays too), alternated after a warm-up; every run is checked to give the same ok flags,
hashes and statuses as the first wire call; the per-kernel split of one timed call of each; the prepare time (wall, and the device
time of its kernels).  Batches of at most 256 items per SM run U on the side stream, so for them the sum of kernel_timings() is not
device time: report their end-to-end times.  The GPU's name and power limit are read (never set) in the same run.  Writes JSON.

    python tools/ietf_prepared_wire_bench.py --suites 0,1,2 --keys 1,1023,16384 --log2 16,20 --out profiles/r3_ietf_prepared_wire_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ark_ec_vrfs_b200 as vrfs  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [x.strip() for x in out.splitlines()[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:            # the numbers are still recorded, marked as lacking their context
        return dict(gpu="unknown (%s)" % e)


def make_signatures(eng, suite, n, n_keys, seed=1):
    rng = np.random.default_rng(seed)
    sk_keys, pks = eng.secret_from_seed(suite, [b"prepared-wire-bench-%d-%d" % (suite, k) for k in range(n_keys)])
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    data, off = rng.integers(0, 256, 8 * n, dtype=np.uint8), np.arange(n + 1, dtype=np.uint64) * 8
    sig, ok = eng.ietf_sign_wire(suite, np.ascontiguousarray(sk_keys[idx]), (data, off))
    assert ok.all()
    enc = eng.point_encode(suite, pks)
    h = vrfs.host_copy
    return enc, h(idx), h(enc[idx]), (h(data), h(off)), h(sig)


def split(kernels):
    d = {}
    for k, ms in kernels:
        d[k] = d.get(k, 0.0) + ms
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--suites", default="0,1,2")
    ap.add_argument("--keys", default="1,1023,16384")
    ap.add_argument("--log2", default="16,20")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_ietf_prepared_wire_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), cases=[])
    with vrfs.Engine(0) as eng:
        for suite in [int(x) for x in a.suites.split(",")]:
            hl = eng.hash_len(suite)
            for n_keys in [int(x) for x in a.keys.split(",")]:
                for lg in [int(x) for x in a.log2.split(",")]:
                    n = 1 << lg
                    enc, idx, pk_enc, datas, sig = make_signatures(eng, suite, n, n_keys)
                    eng.enable_kernel_timing(True)
                    t0 = time.perf_counter()
                    p = eng.public_keys_prepare_encoded(suite, enc)
                    prep_wall = time.perf_counter() - t0
                    prep_kernels = split(eng.kernel_timings())
                    eng.enable_kernel_timing(False)
                    assert p.key_ok.all()
                    outs = {k: (vrfs.host_buffer(n), vrfs.host_buffer((n, hl))) for k in ("wire", "prepared")}
                    calls = dict(wire=lambda: eng.ietf_verify_wire(suite, pk_enc, datas, sig, status=True, out_ok=outs["wire"][0], out_hash=outs["wire"][1]),
                                 prepared=lambda: p.verify_wire(idx, datas, sig, status=True, out_ok=outs["prepared"][0], out_hash=outs["prepared"][1]))
                    truth = [x.copy() for x in calls["wire"]()]
                    assert truth[0].all(), (suite, n_keys, n)
                    for _ in range(a.warmup):
                        for call in calls.values():
                            call()
                    rec = {k: dict(wall_s=[], device_ms=[]) for k in calls}
                    for _ in range(a.repeats):
                        for kind, call in calls.items():
                            for timed in (False, True):
                                eng.enable_kernel_timing(timed)
                                t0 = time.perf_counter()
                                got = call()
                                wall = time.perf_counter() - t0
                                kernels = eng.kernel_timings() if timed else None
                                eng.enable_kernel_timing(False)
                                assert all(np.array_equal(x, y) for x, y in zip(got, truth)), (kind, suite, n_keys, n)
                                if timed:
                                    rec[kind]["device_ms"].append(sum(ms for _, ms in kernels))
                                    rec[kind]["kernels_ms"] = split(kernels)
                                else:
                                    rec[kind]["wall_s"].append(wall)
                    for r in rec.values():
                        r["device_ms_median"] = float(np.median(r["device_ms"]))
                        r["wall_ms_median"] = float(np.median(r["wall_s"]) * 1e3)
                        r["device_M_per_s"] = n / r["device_ms_median"] / 1e3
                        r["e2e_M_per_s"] = n / r["wall_ms_median"] / 1e3
                    case = dict(suite=vrfs.engine.SUITE_NAMES[suite], n=n, n_keys=n_keys, **rec,
                                device_speedup=rec["wire"]["device_ms_median"] / rec["prepared"]["device_ms_median"],
                                e2e_speedup=rec["wire"]["wall_ms_median"] / rec["prepared"]["wall_ms_median"],
                                prepare=dict(wall_ms=prep_wall * 1e3, kernels_ms=prep_kernels))
                    res["cases"].append(case)
                    p.release()
                    print(json.dumps(dict(suite=suite, n=n, n_keys=n_keys, wire_dev_ms=round(rec["wire"]["device_ms_median"], 3),
                                          prepared_dev_ms=round(rec["prepared"]["device_ms_median"], 3), wire_e2e_ms=round(rec["wire"]["wall_ms_median"], 3),
                                          prepared_e2e_ms=round(rec["prepared"]["wall_ms_median"], 3), device_speedup=round(case["device_speedup"], 3),
                                          e2e_speedup=round(case["e2e_speedup"], 3), prepare_ms=round(prep_wall * 1e3, 2),
                                          kernels_ms={k: round(v, 3) for k, v in rec["prepared"]["kernels_ms"].items()},
                                          wire_kernels_ms={k: round(v, 3) for k, v in rec["wire"]["kernels_ms"].items()})), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
