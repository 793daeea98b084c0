"""Pedersen batch verification (vrfs_pedersen_batch_verify: one random linear combination, one MSM) against the per-item verifier
(vrfs_pedersen_verify_batch) on the same distinct Bandersnatch proofs from the engine's prover.

Per size: device time (the sum of kernel_timings()) and end-to-end wall time from page-locked buffers (vrfs.host_copy), the two
calls alternated after a warm-up; the failure path (batch + per-item fallback, one corrupted item); every run checks that the batch
verdict equals all(per-item verdicts).  The GPU's name and power limit are read in the same run.  Writes JSON (default profiles/).

    python tools/pedersen_batch_bench.py --log2 16,18,20 --repeats 3 --out profiles/pedersen_batch_bench.json
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
import ark_ec_vrfs_b200 as vrfs  # noqa: E402

B = vrfs.BANDERSNATCH


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=60).stdout
        name, power, clk = [x.strip() for x in out.splitlines()[0].split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:            # the numbers are still recorded, marked as lacking their context
        return dict(gpu="unknown (%s)" % e)


def make_proofs(eng, n, tag=b"ped-batch-bench"):
    seeds = [hashlib.sha256(tag + b"-%d" % i).digest() for i in range(n)]
    sk, _ = eng.secret_from_seed(B, seeds)
    inp, ok = eng.data_to_point(B, [tag + i.to_bytes(8, "little") for i in range(n)])
    assert ok.all()
    out = eng.output(B, sk, inp)
    proof, _ = eng.pedersen_prove(B, sk, inp, out, None)
    return vrfs.host_copy(inp), vrfs.host_copy(out), vrfs.host_copy(proof)


def run(eng, kind, inp, out, proof, timed_kernels):
    """one call; returns (all_ok, per-item ok or None, wall seconds, device ms or None)"""
    eng.enable_kernel_timing(timed_kernels)
    t0 = time.perf_counter()
    if kind == "per_item":
        ok = eng.pedersen_verify(B, inp, out, proof)
        res = (bool(ok.all()), ok)
    elif kind == "batch":
        res = (eng.pedersen_batch_verify(B, inp, out, proof), None)
    else:                              # failure path: batch + per-item fallback
        a, ok = eng.pedersen_batch_verify(B, inp, out, proof, per_item=True)
        res = (a, ok)
    wall = time.perf_counter() - t0
    dev = sum(ms for _, ms in eng.kernel_timings()) if timed_kernels else None
    eng.enable_kernel_timing(False)
    return res[0], res[1], wall, dev


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2", default="16,18,20")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "pedersen_batch_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), sizes=[])
    with vrfs.Engine(0) as eng:
        for lg in [int(x) for x in a.log2.split(",")]:
            n = 1 << lg
            inp, out, proof = make_proofs(eng, n)
            bad = vrfs.host_copy(proof); bad[n // 3, 200] ^= 1
            truth = eng.pedersen_verify(B, inp, out, proof)
            truth_bad = eng.pedersen_verify(B, inp, out, bad)
            assert truth.all() and truth_bad.sum() == n - 1
            for _ in range(a.warmup):
                for kind in ("per_item", "batch"):
                    run(eng, kind, inp, out, proof, False)
                run(eng, "failure", inp, out, bad, False)
            rec = {k: dict(wall_s=[], device_ms=[]) for k in ("per_item", "batch", "failure")}
            for _ in range(a.repeats):
                for kind in ("per_item", "batch", "failure"):
                    p = bad if kind == "failure" else proof
                    for timed in (False, True):
                        all_ok, ok, wall, dev = run(eng, kind, inp, out, p, timed)
                        expect = truth_bad if kind == "failure" else truth
                        assert all_ok == bool(expect.all()), (kind, n)
                        if ok is not None:
                            assert np.array_equal(ok, expect), (kind, n)
                        rec[kind]["device_ms" if timed else "wall_s"].append(dev if timed else wall)
            for kind, r in rec.items():
                r["device_ms_median"] = float(np.median(r["device_ms"]))
                r["wall_ms_median"] = float(np.median(r["wall_s"]) * 1e3)
                r["device_M_per_s"] = n / r["device_ms_median"] / 1e3
                r["e2e_M_per_s"] = n / r["wall_ms_median"] / 1e3
            eng.enable_kernel_timing(True)
            eng.pedersen_batch_verify(B, inp, out, proof)
            kernels = {}
            for k, ms in eng.kernel_timings():
                kernels[k] = kernels.get(k, 0.0) + ms
            eng.enable_kernel_timing(False)
            rec["batch"]["kernels_ms"] = kernels
            rec["device_speedup"] = rec["per_item"]["device_ms_median"] / rec["batch"]["device_ms_median"]
            rec["e2e_speedup"] = rec["per_item"]["wall_ms_median"] / rec["batch"]["wall_ms_median"]
            res["sizes"].append(dict(n=n, **rec))
            print(json.dumps(dict(n=n, per_item_dev_ms=rec["per_item"]["device_ms_median"], batch_dev_ms=rec["batch"]["device_ms_median"],
                                  per_item_e2e_ms=rec["per_item"]["wall_ms_median"], batch_e2e_ms=rec["batch"]["wall_ms_median"],
                                  failure_e2e_ms=rec["failure"]["wall_ms_median"], device_speedup=round(rec["device_speedup"], 2),
                                  kernels_ms={k: round(v, 3) for k, v in kernels.items()})), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
