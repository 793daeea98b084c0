"""Proofs verified against prepared keys AND prepared VRF inputs, both by index, against the same calls with the input points
(typed) or the input data (wire) gathered per item, on the same proofs:

    typed  vrfs_ietf_verify_prepared_io_batch       vs  vrfs_ietf_verify_prepared_batch       (inputs = points[input_index])
    wire   vrfs_ietf_verify_prepared_io_wire_batch  vs  vrfs_ietf_verify_prepared_wire_batch  (data = datas[input_index])

n proofs by K signers over M inputs, a random signer and input per proof, no ad; the keys are prepared from their encodings (such
a handle serves both forms).  Per (suite, M, n): device time (the sum of kernel_timings()) and end-to-end wall time of all four
calls from page-locked buffers (vrfs.host_copy), alternated after a warm-up; every run is checked to give the same ok flags
(hashes, statuses) as its reference call's first run; the per-kernel split of one timed call of each; the prepare time of the inputs (wall, and the device time of its kernels) and the device memory it takes.  Batches of at
most 256 items per SM run U on the side stream, so for them the sum of kernel_timings() is not device time: use their end-to-end
times.  The GPU's name and power limit are read (never set) in the same run.  Writes JSON.

    python tools/ietf_prepared_io_bench.py --suites 0,1,2 --inputs 1,3,1024 --log2 16,20 --out profiles/r3_ietf_prepared_io_bench.json
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


def free_device_bytes():
    try:
        import torch
        return torch.cuda.mem_get_info(0)[0]
    except Exception:
        return None


def make_proofs(eng, suite, n, sk_keys, datas, pts, seed=1):
    """the same n proofs twice: typed (out, c, s) and serialised; a random key and input per proof"""
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, len(sk_keys), n).astype(np.uint32)
    jdx = rng.integers(0, len(datas), n).astype(np.uint32)
    sk = np.ascontiguousarray(sk_keys[idx]); inp = np.ascontiguousarray(pts[jdx])
    out = eng.output(suite, sk, inp)
    c, s = eng.ietf_prove(suite, sk, inp, out)
    data = np.concatenate([np.frombuffer(d, np.uint8) for d in datas])
    doff = np.concatenate([[0], np.cumsum([len(d) for d in datas])]).astype(np.uint64)
    g_off = np.concatenate([[0], np.cumsum(doff[jdx + 1] - doff[jdx])]).astype(np.uint64)
    g_data = np.concatenate([data[int(doff[j]):int(doff[j + 1])] for j in jdx]) if g_off[-1] else np.zeros(16, np.uint8)
    sig, ok = eng.ietf_sign_wire(suite, sk, (g_data, g_off))
    assert ok.all()
    h = vrfs.host_copy
    return h(idx), h(jdx), h(inp), h(out), h(c), h(s), (h(g_data), h(g_off)), h(sig)


def split(kernels):
    d = {}
    for k, ms in kernels:
        d[k] = d.get(k, 0.0) + ms
    return d


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--suites", default="0,1,2")
    ap.add_argument("--keys", type=int, default=1023)
    ap.add_argument("--inputs", default="1,3,1024")
    ap.add_argument("--log2", default="16,20")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_ietf_prepared_io_bench.json"))
    a = ap.parse_args()
    res = dict(info=gpu_info(), n_keys=a.keys, cases=[])
    with vrfs.Engine(0) as eng:
        for suite in [int(x) for x in a.suites.split(",")]:
            sk_keys, pks = eng.secret_from_seed(suite, [b"prepared-io-bench-%d-%d" % (suite, k) for k in range(a.keys)])
            keys = eng.public_keys_prepare_encoded(suite, eng.point_encode(suite, pks))
            assert keys.key_ok.all()
            for n_inputs in [int(x) for x in a.inputs.split(",")]:
                datas = [b"bench-round-%d-%d" % (suite, j) + bytes(32) for j in range(n_inputs)]
                free0 = free_device_bytes()
                eng.enable_kernel_timing(True)
                t0 = time.perf_counter()
                q = eng.inputs_prepare(suite, datas)
                prep_wall = time.perf_counter() - t0
                prep_kernels = split(eng.kernel_timings())
                eng.enable_kernel_timing(False)
                free1 = free_device_bytes()
                assert q.input_ok.all()
                for lg in [int(x) for x in a.log2.split(",")]:
                    n = 1 << lg
                    idx, jdx, inp, out, c, s, g_datas, sig = make_proofs(eng, suite, n, sk_keys, datas, q.points)
                    calls = dict(typed=lambda: keys.verify(idx, inp, out, c, s, status=True),
                                 typed_io=lambda: keys.verify_io(q, idx, jdx, out, c, s, status=True),
                                 wire=lambda: keys.verify_wire(idx, g_datas, sig, status=True),
                                 wire_io=lambda: keys.verify_io_wire(q, idx, jdx, sig, status=True))
                    truth = {k: [x.copy() for x in calls[k]()] for k in ("typed", "wire")}
                    assert truth["typed"][0].all() and truth["wire"][0].all(), (suite, n_inputs, n)
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
                                ref = truth[kind.split("_")[0]]
                                assert all(np.array_equal(x, y) for x, y in zip(got, ref)), (kind, suite, n_inputs, n)
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
                    sp = lambda a_, b_, f: rec[a_][f] / rec[b_][f]
                    case = dict(suite=vrfs.engine.SUITE_NAMES[suite], n=n, n_inputs=n_inputs, **rec,
                                typed_device_speedup=sp("typed", "typed_io", "device_ms_median"), typed_e2e_speedup=sp("typed", "typed_io", "wall_ms_median"),
                                wire_device_speedup=sp("wire", "wire_io", "device_ms_median"), wire_e2e_speedup=sp("wire", "wire_io", "wall_ms_median"),
                                prepare=dict(wall_ms=prep_wall * 1e3, kernels_ms=prep_kernels,
                                             device_bytes=(free0 - free1) if free0 is not None and free1 is not None else None))
                    res["cases"].append(case)
                    r2 = lambda x: round(x, 3)
                    print(json.dumps(dict(suite=suite, n=n, n_inputs=n_inputs,
                                          dev_ms={k: r2(v["device_ms_median"]) for k, v in rec.items()},
                                          e2e_ms={k: r2(v["wall_ms_median"]) for k, v in rec.items()},
                                          speedup=dict(typed_dev=r2(case["typed_device_speedup"]), typed_e2e=r2(case["typed_e2e_speedup"]),
                                                       wire_dev=r2(case["wire_device_speedup"]), wire_e2e=r2(case["wire_e2e_speedup"])),
                                          prepare_ms=r2(prep_wall * 1e3), kernels_ms={k: {kk: r2(vv) for kk, vv in v["kernels_ms"].items()} for k, v in rec.items()})),
                          flush=True)
                q.release()
            keys.release()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res["info"]))


if __name__ == "__main__":
    main()
