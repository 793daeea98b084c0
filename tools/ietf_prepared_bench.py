"""IETF verify against prepared public keys (vrfs_ietf_verify_prepared_batch) against vrfs_ietf_verify_batch on the gathered keys,
on the same distinct proofs from the engine's prover: n proofs by K signers, a random signer per proof.

Per (suite, K, n): device time (the sum of kernel_timings()) and end-to-end wall time from page-locked buffers (vrfs.host_copy) of both
calls, alternated after a warm-up, every run checked to give identical verdicts; the per-kernel split of one timed call of each; the
prepare time (wall, and the device time of its kernels) and the bytes of the key tables (computed from their layout).  The sum of
kernel_timings() is device time only when every kernel runs on the main stream: batches of at most 256 items per SM run U on the side
stream (both calls), so report their end-to-end times, not that sum.  The GPU's name
and power limit are read in the same run.  Writes JSON (default profiles/).

    python tools/ietf_prepared_bench.py --suites 0,1,2 --keys 1,1023,16384 --log2 20 --out profiles/r3_ietf_prepared_bench.json
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

SW_SUITES = (vrfs.P256, vrfs.BANDERSNATCH_SW)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [x.strip() for x in out.splitlines()[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:            # the numbers are still recorded, marked as lacking their context
        return dict(gpu="unknown (%s)" % e)


def table_bytes(suite, n_keys):
    windows = 33 if suite in SW_SUITES else 32          # 8-bit windows (+ the carry window of the short-Weierstrass suites)
    return n_keys * (windows * 129 * 96 + 64 + 1)       # tables + key rows + key_ok


def make_proofs(eng, suite, n, n_keys, seed=1):
    rng = np.random.default_rng(seed)
    sk_keys, pks = eng.secret_from_seed(suite, [b"prepared-bench-%d-%d" % (suite, k) for k in range(n_keys)])
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    inp, ok = eng.data_to_point(suite, (rng.integers(0, 256, 8 * n, dtype=np.uint8), np.arange(n + 1, dtype=np.uint64) * 8))
    assert ok.all()
    sk = np.ascontiguousarray(sk_keys[idx])
    out = eng.output(suite, sk, inp)
    c, s = eng.ietf_prove(suite, sk, inp, out, None)
    h = vrfs.host_copy
    return pks, h(idx), h(pks[idx]), h(inp), h(out), h(c), h(s)


def run(eng, call, timed_kernels):
    eng.enable_kernel_timing(timed_kernels)
    t0 = time.perf_counter()
    ok = call()
    wall = time.perf_counter() - t0
    kernels = eng.kernel_timings() if timed_kernels else None
    eng.enable_kernel_timing(False)
    return ok, wall, kernels


def split(kernels):
    d = {}
    for k, ms in kernels:
        d[k] = d.get(k, 0.0) + ms
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--suites", default="0,1,2")
    ap.add_argument("--keys", default="1,1023,16384")
    ap.add_argument("--log2", default="20")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_ietf_prepared_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), cases=[])
    with vrfs.Engine(0) as eng:
        for suite in [int(x) for x in a.suites.split(",")]:
            for n_keys in [int(x) for x in a.keys.split(",")]:
                for lg in [int(x) for x in a.log2.split(",")]:
                    n = 1 << lg
                    pks, idx, pk, inp, out, c, s = make_proofs(eng, suite, n, n_keys)
                    eng.enable_kernel_timing(True)
                    t0 = time.perf_counter()
                    p = eng.public_keys_prepare(suite, pks)
                    prep_wall = time.perf_counter() - t0
                    prep_kernels = split(eng.kernel_timings())
                    eng.enable_kernel_timing(False)
                    assert p.key_ok.all()
                    calls = dict(gathered=lambda: eng.ietf_verify(suite, pk, inp, out, c, s), prepared=lambda: p.verify(idx, inp, out, c, s))
                    truth = calls["gathered"]()
                    assert truth.all(), (suite, n_keys, n)
                    for _ in range(a.warmup):
                        for call in calls.values():
                            call()
                    rec = {k: dict(wall_s=[], device_ms=[]) for k in calls}
                    for _ in range(a.repeats):
                        for kind, call in calls.items():
                            for timed in (False, True):
                                ok, wall, kernels = run(eng, call, timed)
                                assert np.array_equal(ok, truth), (kind, suite, n_keys, n)
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
                                device_speedup=rec["gathered"]["device_ms_median"] / rec["prepared"]["device_ms_median"],
                                e2e_speedup=rec["gathered"]["wall_ms_median"] / rec["prepared"]["wall_ms_median"],
                                prepare=dict(wall_ms=prep_wall * 1e3, kernels_ms=prep_kernels, table_bytes=table_bytes(suite, n_keys)))
                    res["cases"].append(case)
                    p.release()
                    print(json.dumps(dict(suite=suite, n=n, n_keys=n_keys, gathered_dev_ms=round(rec["gathered"]["device_ms_median"], 3),
                                          prepared_dev_ms=round(rec["prepared"]["device_ms_median"], 3), gathered_e2e_ms=round(rec["gathered"]["wall_ms_median"], 3),
                                          prepared_e2e_ms=round(rec["prepared"]["wall_ms_median"], 3), device_speedup=round(case["device_speedup"], 3),
                                          e2e_speedup=round(case["e2e_speedup"], 3), prepare_ms=round(prep_wall * 1e3, 2),
                                          table_MB=round(table_bytes(suite, n_keys) / 1e6, 1),
                                          kernels_ms={k: round(v, 3) for k, v in rec["prepared"]["kernels_ms"].items()},
                                          gathered_kernels_ms={k: round(v, 3) for k, v in rec["gathered"]["kernels_ms"].items()})), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
