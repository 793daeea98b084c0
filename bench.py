#!/usr/bin/env python3
"""bench.py - headline benchmark: Bandersnatch IETF VRF batch verify (BASELINE.json configs[1]) plus, in the same driver-run
line, every other BASELINE config and the multi-GPU commitment MSM.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--logn 20] [--dump-outputs DIR]

A step = one pass of `ietf::Verifier::verify` over one batch of 2^logn synthetic proofs per GPU.
Workload (SURVEY.md 8d): 2^logn DISTINCT items per GPU - sk_i = Secret::from_seed("vrfs-b200-bench-sk" || u64le(i)),
alpha_i = u64le(i) || 24 x 0x00, proofs produced by the engine's own prover and cross-checked against the CPU oracle on a
2^12 subsample (prover output AND verdicts); 1/64 of the items corrupted (bit flip in c, s or O, position i mod 3).
  value : verifies/s, whole job, inputs resident in HBM (vrfs_ietf_verify_batch_dev), CUDA-event timed on the engine's
          stream, max over ranks.
  e2e   : the same through the host-buffer C ABI call (vrfs_ietf_verify_batch) from pinned host memory, H2D + D2H inside.
  roofline : integer-pipe (32x32+64 multiply-accumulate) roofline of the dominant kernel, plus its HBM view.
  cpu_baseline : the CPU oracle (restatement of the reference algorithm, NOT the arkworks binary - the mounted reference is a
          deprecation stub and no Rust toolchain exists) on a bounded sample, all host threads.
  configs : with_ad32 (the headline with 32-byte additional data), strong_scaling (ONE 2^logn batch over the N GPUs),
          ietf_prove (Ed25519, secp256r1; BASELINE configs[2]), pedersen (Bandersnatch prove + verify; configs[3]),
          ring_kzg_msm_ms (3-column commitment MSM for the domains 2^11..2^17; configs[4]) - at N > 1 the point-range-split
          form whose partial sums are exchanged by the MSM's last kernel over NVLink (no NCCL on the data path).
--impl reference times the CPU oracle as the reference arm.
--dump-outputs DIR writes the verdicts of the last timed headline step as DIR/ietf_verify_ok.npy (float32, one per item; the
inputs are the same on every run with the same arguments), so that two builds can be compared output for output.
Only the cross-checks, the cpu_baseline leg and --impl reference touch oracle/ (tests/oracle_lib.py).
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import traceback

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the benchmark may run from a read-only tree and writes nothing into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "bandersnatch_ietf_vrf_verifies_per_sec"
UNIT = "verifies/s"
MAC_PER_MUL = 136          # one 8-limb Montgomery product = 2 n^2 + n multiply-accumulates (SURVEY.md 8d)
R_BLS = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
SUITE_NAMES = {0: "Bandersnatch_SHA-512_ELL2", 1: "Ed25519_SHA-512_TAI", 2: "secp256r1_SHA-256_TAI"}


# MAC32 per field product of each suite's base field (csrc/arith.cuh): an 8-limb Montgomery product is 2 n^2 + n = 136; the
# pseudo-Mersenne prime 2^255 - 19 needs the 64 schoolbook products + 8 for the fold; the P-256 Solinas reduction uses no multiplier
MAC_PER_MUL_SUITE = {0: 136, 1: 72, 2: 64}


def kernel_muls(suite, kernel):
    """algorithmic field products per item of one kernel.  Bandersnatch: the figures of SURVEY.md Appendix D (squarings = products;
    additions and small-constant multiplications free) - 2 110 for the joint 4-way GLV combination, 1 820 for fixed + variable,
    1 560 for one variable base, 275 for two points to affine with a shared inversion; a fixed-base multiplication is the 16
    mixed additions of 8 products the engine executes (16-bit windows; the survey's 8-bit model has 32).  The engine executes ~7 %
    MORE than the survey's model on the headline kernel (fixed radix-16 windows instead of wNAF: 124 doublings of 4S + 3..4M,
    128 cached additions of 9M, four 8-entry tables, two endomorphisms ~ 2 255 product-equivalents), so the fraction reported from
    the model is a lower bound of the multiplier's actual load.  Ed25519 / secp256r1 (not in the survey): the same style of count
    for what the kernels do - no GLV, 64 / 65 radix-16 windows."""
    if suite == 0:
        t = {"lincomb<2,0>": 2110, "lincomb<1,1>": 1820, "lincomb<1,0>": 1560, "lincomb<0,1>": 128, "lincomb<0,2>": 256, "lincomb<1,2>": 1560 + 256,
             "ietf_verify_finish": 275, "zinv": 45}
    elif suite == 1:     # 252 doublings (4S + 3..4M), 64 cached additions (a = -1 entry form: 8M; 7M against the affine fixed-base entries), one 8-entry table
        var = 252 * 7.25 + 64 * 8 + 68
        t = {"lincomb<2,0>": 252 * 7.25 + 2 * (64 * 8 + 68), "lincomb<1,1>": var + 112, "lincomb<1,0>": var, "lincomb<0,1>": 112, "lincomb<0,2>": 224, "lincomb<1,2>": var + 224}
    else:                # 64 quadruple doublings of 16M + 22S (a squaring is 36 of a product's 64 wide multiplies: counted as 0.5625),
                         # 65 complete additions of 12, one table; fixed base: 17 complete additions
        var = 64 * (16 + 22 * 0.5625) + 65 * 12 + 84
        t = {"lincomb<2,0>": 64 * (16 + 22 * 0.5625) + 2 * (65 * 12 + 84), "lincomb<1,1>": var + 17 * 12, "lincomb<1,0>": var, "lincomb<0,1>": 17 * 12, "lincomb<0,2>": 34 * 12, "lincomb<1,2>": var + 34 * 12}
    return t.get(kernel)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--logn", type=int, default=20, help="log2 of the per-GPU batch")
    ap.add_argument("--ref-logn", type=int, default=14, help="log2 of the reference arm's per-step sample")
    ap.add_argument("--cpu-sample-logn", type=int, default=18)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--headline-only", action="store_true", help="skip the secondary configs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the verdicts of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


DUMP_MAX_ITEMS = 1 << 22        # 16 MiB of float32 verdicts (+ 32 MiB of float64 indices when sampled): under 64 MB in all


def dump_outputs(path, arrays):
    """each array as path/<name>.npy in float32.  An array longer than DUMP_MAX_ITEMS is reduced to a sample of items drawn
    with a fixed seed (the same for every run of the same size), and the sampled item indices go to path/<name>_index.npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, arr in arrays.items():
        arr = np.asarray(arr)
        if len(arr) > DUMP_MAX_ITEMS:
            idx = np.sort(np.random.default_rng(0).choice(len(arr), DUMP_MAX_ITEMS, replace=False))
            np.save(os.path.join(path, name + "_index.npy"), idx.astype(np.float64))
            arr = arr[idx]
        np.save(os.path.join(path, name + ".npy"), arr.astype(np.float32))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], None, [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx = float(f[2]); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "power_w": statistics.median(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            for k in ("hbm_gbs", "hbm_gb_s", "hbm_GBps"):
                if k in d:
                    return float(d[k]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def ncu_record(kernel, key, n):
    """figures of the committed ncu capture of the dominant kernel (profiles/traffic.json); byte counts scaled to n items"""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
        v = d[key][kernel]
        return v / d["items_per_launch"] * n if key == "dram_bytes_per_launch" else v
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------------------------------
# workload generation (on the GPU, by the engine's own prover; the oracle only cross-checks a subsample)
# ---------------------------------------------------------------------------------------------------------------------------
def packed_counter(prefix, base, n, pad=0):
    """n items prefix || u64le(base + i) || pad zero bytes, as (data, offsets) for the engine"""
    import numpy as np
    L = len(prefix) + 8 + pad
    d = np.zeros((n, L), np.uint8)
    if prefix:
        d[:, :len(prefix)] = np.frombuffer(prefix, np.uint8)
    d[:, len(prefix):len(prefix) + 8] = np.arange(base, base + n, dtype=np.uint64).view(np.uint8).reshape(n, 8)
    return d.reshape(-1), np.arange(n + 1, dtype=np.uint64) * L


def ad32(base, n):
    import numpy as np
    raw = b"".join(hashlib.sha256((base + i).to_bytes(8, "little")).digest() for i in range(n))
    return np.frombuffer(raw, np.uint8).copy(), np.arange(n + 1, dtype=np.uint64) * 32


def slice_var(v, idx):
    data, off = v
    return [data[int(off[i]):int(off[i + 1])].tobytes() for i in idx]


def make_keys(eng, suite, base, n):
    seeds = packed_counter(b"vrfs-b200-bench-sk", base, n)
    alphas = packed_counter(b"", base, n, pad=24)
    sk, pk = eng.secret_from_seed(suite, seeds)
    inp, ok = eng.data_to_point(suite, alphas)
    assert ok.all()
    out = eng.output(suite, sk, inp)
    return dict(seeds=seeds, alphas=alphas, sk=sk, pk=pk, inp=inp, out=out)


def make_verify_workload(eng, suite, base, n, with_ad, oracle_threads):
    """2^logn distinct proofs by the GPU prover; 1/64 corrupted; prover output and verdicts oracle-checked on a 2^12 subsample"""
    import numpy as np
    import oracle_lib as O
    w = make_keys(eng, suite, base, n)
    w["ads"] = ad32(base, n) if with_ad else None
    c, s = eng.ietf_prove(suite, w["sk"], w["inp"], w["out"], w["ads"])
    expect = np.ones(n, np.uint8)
    bad = np.arange(0, n, 64)
    out = w["out"].copy()
    for kind, arr in ((0, c), (1, s), (2, out)):
        rows = bad[bad % 3 == kind]
        arr[rows, (rows // 64) % 16] ^= 1 << 3
    w["out_good"] = w["out"]; w["out"] = out
    expect[bad] = 0
    w["c"], w["s"], w["expect"] = c, s, expect
    sub = np.arange(0, n, max(1, n // 4096))
    adsub = slice_var(w["ads"], sub) if with_ad else None
    sk_o, pk_o = O.secret_from_seed(suite, slice_var(w["seeds"], sub), nthreads=oracle_threads)
    inp_o, _ = O.data_to_point(suite, slice_var(w["alphas"], sub), nthreads=oracle_threads)
    assert np.array_equal(sk_o, w["sk"][sub]) and np.array_equal(pk_o, w["pk"][sub]) and np.array_equal(inp_o, w["inp"][sub]), "keys / inputs differ from the oracle"
    c_o, s_o = O.ietf_prove(suite, sk_o, inp_o, w["out_good"][sub], adsub, nthreads=oracle_threads)
    good = expect[sub] == 1
    assert np.array_equal(c_o[good], c[sub][good]) and np.array_equal(s_o[good], s[sub][good]), "GPU prover differs from the oracle"
    v_o = O.ietf_verify(suite, w["pk"][sub], w["inp"][sub], out[sub], c[sub], s[sub], adsub, nthreads=oracle_threads)
    assert np.array_equal(v_o, expect[sub]), "expected verdicts differ from the oracle"
    w["oracle_checked_items"] = int(len(sub))
    return w


# ---------------------------------------------------------------------------------------------------------------------------
# secondary configs (host-buffer calls; every rank runs them on its own 2^logn items, rank 0 aggregates)
# ---------------------------------------------------------------------------------------------------------------------------
def pinned(a):
    """the same array in page-locked host memory (the C ABI copies straight from / into the caller's buffers: pageable memory makes
    every copy a staged, synchronous one)"""
    import numpy as np
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    _PINNED.append(t)                       # keeps the page-locked allocation alive behind the numpy view
    return t.numpy()


_PINNED = []


def pinned_zeros(shape):
    import torch
    t = torch.zeros(shape, dtype=torch.uint8).pin_memory()
    _PINNED.append(t)
    return t.numpy()


def timed_host_call(eng, fn, steps):
    """(seconds per call by wall clock, {kernel: ms} of one call by CUDA events on the engine's stream)"""
    fn()
    t0 = time.perf_counter()
    for _ in range(steps):
        fn()
    wall = (time.perf_counter() - t0) / steps
    eng.enable_kernel_timing(True)
    fn()
    kt = {}
    for name, ms in eng.kernel_timings():
        kt[name] = kt.get(name, 0.0) + ms
    eng.enable_kernel_timing(False)
    return wall, kt


def roofline_of(kt, suite, n, peak_mac):
    dom = max(kt, key=kt.get)
    muls = kernel_muls(suite, dom)
    r = {"kernel": dom, "kernel_ms": {k: round(v, 3) for k, v in kt.items()}, "share_of_device_time": kt[dom] / sum(kt.values())}
    if muls:
        ach = n * muls * MAC_PER_MUL_SUITE[suite] / (kt[dom] * 1e-3)
        r.update({"field_muls_per_item": muls, "mac32_per_mul": MAC_PER_MUL_SUITE[suite], "achieved_tmac32": ach / 1e12,
                  "frac_of_mac32_peak": ach / peak_mac if peak_mac else None})
    return r


def config_ietf_prove(eng, suite, base, n, steps, peak_mac, oracle_threads):
    """BASELINE configs[2]: batch IETF prove with deterministic nonces; inputs in host memory, c and s back to host"""
    import numpy as np
    import oracle_lib as O
    w = make_keys(eng, suite, base, n)
    res = {}
    sk_p, inp_p, out_p = pinned(w["sk"]), pinned(w["inp"]), pinned(w["out"])
    outs = (pinned_zeros((n, 32)), pinned_zeros((n, 32)))
    fn = lambda: eng.ietf_prove(suite, sk_p, inp_p, out_p, None, out=outs)
    wall, kt = timed_host_call(eng, fn, steps)
    c, s = fn()
    sub = np.arange(0, n, max(1, n // 1024))
    c_o, s_o = O.ietf_prove(suite, w["sk"][sub], w["inp"][sub], w["out"][sub], None, nthreads=oracle_threads)
    assert np.array_equal(c_o, c[sub]) and np.array_equal(s_o, s[sub]), "prove differs from the oracle"
    assert eng.ietf_verify(suite, w["pk"], w["inp"], w["out"], c, s).all()
    dev_ms = sum(kt.values())
    res = {"items": n, "e2e_per_s": n / wall, "device_per_s": n / (dev_ms * 1e-3), "e2e_ms": wall * 1e3, "device_ms": dev_ms,
           "h2d_bytes": n * 160, "d2h_bytes": n * 64, "oracle_checked_items": int(len(sub)), "roofline": roofline_of(kt, suite, n, peak_mac)}
    return res


def config_pedersen(eng, base, n, steps, peak_mac, oracle_threads):
    """BASELINE configs[3]: Pedersen prove + verify over Bandersnatch"""
    import numpy as np
    import oracle_lib as O
    suite = 0
    w = make_keys(eng, suite, base, n)
    sk_p, inp_p, out_p = pinned(w["sk"]), pinned(w["inp"]), pinned(w["out"])
    outs = (pinned_zeros((n, 256)), pinned_zeros((n, 32)))
    fnp = lambda: eng.pedersen_prove(suite, sk_p, inp_p, out_p, None, out=outs)
    wall_p, kt_p = timed_host_call(eng, fnp, steps)
    proof, bl = fnp()
    sub = np.arange(0, n, max(1, n // 1024))
    p_o, b_o = O.pedersen_prove(suite, w["sk"][sub], w["inp"][sub], w["out"][sub], None, nthreads=oracle_threads)
    assert np.array_equal(p_o, proof[sub]) and np.array_equal(b_o, bl[sub]), "pedersen prove differs from the oracle"
    bad = np.arange(0, n, 64)
    proof[bad, 192 + (bad // 64) % 30] ^= 4
    fnv = lambda: eng.pedersen_verify(suite, inp_p, out_p, proof, None)
    wall_v, kt_v = timed_host_call(eng, fnv, steps)
    ok = fnv()
    expect = np.ones(n, np.uint8); expect[bad] = 0
    assert np.array_equal(ok, expect), "pedersen verdicts"
    assert np.array_equal(O.pedersen_verify(suite, w["inp"][sub], w["out"][sub], proof[sub], None, nthreads=oracle_threads), expect[sub])
    dp, dv = sum(kt_p.values()), sum(kt_v.values())
    return {"items": n,
            "prove": {"e2e_per_s": n / wall_p, "device_per_s": n / (dp * 1e-3), "e2e_ms": wall_p * 1e3, "device_ms": dp, "h2d_bytes": n * 160, "d2h_bytes": n * 288,
                      "roofline": roofline_of(kt_p, suite, n, peak_mac)},
            "verify": {"e2e_per_s": n / wall_v, "device_per_s": n / (dv * 1e-3), "e2e_ms": wall_v * 1e3, "device_ms": dv, "h2d_bytes": n * 384, "d2h_bytes": n,
                       "invalid_fraction": 1 / 64, "roofline": roofline_of(kt_v, suite, n, peak_mac)},
            "oracle_checked_items": int(len(sub))}


def bench_srs(eng, nmax):
    """test-only SRS [tau^j]G1 with the PUBLIC tau = LE(SHA-512("vrfs-b200-bench-tau")) mod r (SURVEY 8d), produced by the engine"""
    import numpy as np
    tau = int.from_bytes(hashlib.sha512(b"vrfs-b200-bench-tau").digest(), "little") % R_BLS
    pw = np.zeros((nmax, 32), np.uint8); t = 1
    for j in range(nmax):
        pw[j] = np.frombuffer(t.to_bytes(32, "little"), np.uint8); t = t * tau % R_BLS
    gen = np.zeros((1, 96), np.uint8)
    gx = 0x17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb
    gy = 0x08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1
    gen[0, :48] = np.frombuffer(gx.to_bytes(48, "little"), np.uint8); gen[0, 48:] = np.frombuffer(gy.to_bytes(48, "little"), np.uint8)
    h1 = eng.msm_g1_prepare(gen)
    srs = np.concatenate([h1.msm(pw[i:i + 32], 32) for i in range(0, nmax, 32)])
    h1.release()
    return srs


def bench_scalars(m):
    """uniform field elements (what ring columns and polynomial coefficients look like), deterministic"""
    import numpy as np
    rng = np.random.default_rng(20261017)
    raw = rng.integers(0, 256, size=(m, 40), dtype=np.uint8)
    return np.frombuffer(b"".join((int.from_bytes(r.tobytes(), "little") % R_BLS).to_bytes(32, "little") for r in raw), np.uint8).reshape(m, 32).copy()


def msm_window(logn):
    return 8 if logn <= 9 else 10 if logn <= 12 else 13 if logn <= 16 else 16      # msm_plan's prepared-mode table (csrc/msm.cuh)


def config_msm(eng, rank, world, peak_mac, hbm_peak, sizes, steps=5):
    """BASELINE configs[4]: 3-column KZG commitment MSM over BLS12-381 G1, prepared SRS, for every domain size; plus the commitment
    of an actual ring (fixed columns built on the device).  world > 1: the SRS is split by point range over the ranks and the
    partials are exchanged by the MSM's last kernel over NVLink (vrfs_msm_g1_prepared_allgather / vrfs_ring_commit_rows_allgather);
    every rank checks the collective result against its own single-GPU computation."""
    import numpy as np
    import ark_ec_vrfs_b200 as vrfs
    from ark_ec_vrfs_b200 import dist as D
    nmax = 1 << max(sizes)
    srs = bench_srs(eng, nmax)
    pool = bench_scalars(3 * nmax).reshape(3, nmax, 32)
    _, allkeys = eng.secret_from_seed(vrfs.BANDERSNATCH, packed_counter(b"bench-ring-key-", 0, nmax // 2 + 254))
    out = {}
    device_exchange = world > 1 and eng.peer_world == world      # main() connected the peer group (a collective of its own)
    out["exchange"] = ("device-side: partials stored into the peers' mailboxes by k_msm_final2 over NVLink (CUDA IPC), flags + fold in the same kernel"
                       if device_exchange else ("single GPU" if world == 1 else "host all-gather fallback (no peer access)"))
    for logn in sizes:
        n = 1 << logn
        sc = np.ascontiguousarray(pool[:, :n]).reshape(-1, 32)
        h = eng.msm_g1_prepare(srs[:n])
        ref = h.msm(sc, 3)
        wall1, kt1 = timed_host_call(eng, lambda: h.msm(sc, 3), steps)
        r = {"single_gpu": {"device_ms": sum(kt1.values()), "e2e_ms": wall1 * 1e3, "kernel_ms": {k: round(v, 4) for k, v in kt1.items()},
                            "mode": "table (128 multiples of every 2^(8w) P_i, no buckets)" if "msm_table_sum" in kt1 else "buckets"}}
        # the stateless entry point (the literal VariableBaseMSM::msm signature: bases uploaded and converted per call, GLV halves, Horner over the windows)
        assert np.array_equal(eng.msm_g1(srs[:n], sc, 3), ref), "stateless MSM differs from the prepared one at 2^%d" % logn
        walls, kts = timed_host_call(eng, lambda: eng.msm_g1(srs[:n], sc, 3), steps)
        r["single_gpu"]["stateless_device_ms"] = sum(kts.values()); r["single_gpu"]["stateless_e2e_ms"] = walls * 1e3
        c = msm_window(logn)
        entries = 3 * n * ((255 + c) // c)
        acc_ms = kt1.get("msm_accumulate")
        if acc_ms:
            # every non-zero signed digit is one XYZZ mixed addition = 10 products of 12 limbs = 10 x 300 MAC32, one 96-byte table record + 4-byte list entry
            rl = {"kernel": "k_msm_accumulate", "ms": acc_ms, "share_of_call": acc_ms / sum(kt1.values()), "mixed_additions": entries,
                  "achieved_tmac32": entries * 3000 / (acc_ms * 1e-3) / 1e12, "hbm_gbps": entries * 100 / (acc_ms * 1e-3) / 1e9}
            if peak_mac:
                rl["frac_of_mac32_peak"] = rl["achieved_tmac32"] * 1e12 / peak_mac
                r["single_gpu"]["whole_call_frac_of_mac32_peak"] = entries * 3000 / (sum(kt1.values()) * 1e-3) / peak_mac
            if hbm_peak:
                rl["frac_of_hbm_peak"] = rl["hbm_gbps"] / hbm_peak
            r["single_gpu"]["roofline"] = rl
        tab_ms = kt1.get("msm_table_sum")
        if tab_ms:
            # table mode: every non-zero signed radix-256 digit is one XYZZ mixed addition (10 x 300 MAC32) over a random 96-byte table record
            ent = 3 * n * 32
            rl = {"kernel": "k_msm_table_sum", "ms": tab_ms, "share_of_call": tab_ms / sum(kt1.values()), "mixed_additions": ent,
                  "achieved_tmac32": ent * 3000 / (tab_ms * 1e-3) / 1e12, "hbm_gbps": ent * 96 / (tab_ms * 1e-3) / 1e9}
            if peak_mac:
                rl["frac_of_mac32_peak"] = rl["achieved_tmac32"] * 1e12 / peak_mac
                r["single_gpu"]["whole_call_frac_of_mac32_peak"] = ent * 3000 / (sum(kt1.values()) * 1e-3) / peak_mac
            if hbm_peak:
                rl["frac_of_hbm_peak"] = rl["hbm_gbps"] / hbm_peak
            r["single_gpu"]["roofline"] = rl
        # the commitment of an actual ring (SURVEY 8f-2): N/2 distinct keys, the remaining key slots padded, 253-row tail, Lagrange-basis SRS
        tail, padding, keys = allkeys[n // 2 + 1:n // 2 + 254], allkeys[n // 2], allkeys[:n // 2]
        part = n - 3 - len(tail) - 1
        ring_ref = h.ring_commit(keys, part, padding, tail, lagrange=True)
        wr, ktr = timed_host_call(eng, lambda: h.ring_commit(keys, part, padding, tail, lagrange=True), steps)
        r["single_gpu"]["ring_commit_device_ms"] = sum(ktr.values()); r["single_gpu"]["ring_commit_e2e_ms"] = wr * 1e3
        wd, ktd = timed_host_call(eng, lambda: h.ring_commit_delta(keys, padding), steps)
        r["single_gpu"]["ring_commit_incremental_device_ms"] = sum(ktd.values())
        h.release()
        if world > 1:
            sh = D.ShardedPreparedBases(eng, srs[:n])
            loc = sh.local_scalars(sc, 3)
            got = sh.msm_local(loc, 3)
            assert np.array_equal(got, ref), "sharded MSM differs from the single-GPU result at 2^%d" % logn
            wall, kt = timed_host_call(eng, lambda: sh.msm_local(loc, 3), steps)
            rc = D.ShardedRingContext(eng, srs[:n], part, padding, tail)
            assert np.array_equal(rc.verifier_key_commitment(keys), ring_ref), "sharded ring commitment differs at 2^%d" % logn
            wallr, ktrr = timed_host_call(eng, lambda: rc.verifier_key_commitment(keys), steps)
            r["sharded"] = {"device_ms": sum(kt.values()), "e2e_ms": wall * 1e3, "ring_commit_device_ms": sum(ktrr.values()), "ring_commit_e2e_ms": wallr * 1e3,
                            "kernel_ms": {k: round(v, 4) for k, v in kt.items()}, "points_per_rank": n // world}
            rc.release(); sh.release()
        out["2^%d" % logn] = r
    return out


def config_kzg(eng, sizes, steps=3):
    """BASELINE configs[4], second half ("plus batched ring-proof verify"): k KZG openings checked at once - the 2-column MSM over
    2k + 1 points and the product of two BLS12-381 pairings a ring-proof verifier ends in (transcript coefficients as inputs).
    Honest openings under the bench's public tau; every size must accept, and reject with one forged value."""
    import numpy as np
    tau = int.from_bytes(hashlib.sha512(b"vrfs-b200-bench-tau").digest(), "little") % R_BLS
    kmax = 1 << max(sizes)
    rng = np.random.default_rng(4242)
    def fr(m):
        raw = rng.integers(0, 256, size=(m, 40), dtype=np.uint8)
        return [int.from_bytes(r.tobytes(), "little") % R_BLS for r in raw]
    pt, z, r = fr(kmax), fr(kmax), fr(kmax)                  # p_i(tau), z_i, r_i; the polynomial is p_i(X) = pt_i + a_i (X - tau) with a_i = z_i + 1
    v = [(p + (zz + 1) * (zz - tau)) % R_BLS for p, zz in zip(pt, z)]
    w = [(zz + 1) % R_BLS for zz in z]                       # (p(tau) - p(z)) / (tau - z) = a_i
    sc = lambda xs: np.frombuffer(b"".join(x.to_bytes(32, "little") for x in xs), np.uint8).reshape(-1, 32).copy()
    gen = np.zeros((1, 96), np.uint8)
    gx = 0x17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb
    gy = 0x08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1
    gen[0, :48] = np.frombuffer(gx.to_bytes(48, "little"), np.uint8); gen[0, 48:] = np.frombuffer(gy.to_bytes(48, "little"), np.uint8)
    h1 = eng.msm_g1_prepare(gen)
    mults = lambda s: np.concatenate([h1.msm(s[i:i + 32], 32) for i in range(0, len(s), 32)])
    C, W = mults(sc(pt)), mults(sc(w))
    h1.release()
    # the verifier key's [tau] G2: one scalar multiplication on the host (affine big-integer arithmetic, not timed)
    from oracle import pairing_ref as PR
    g2 = np.frombuffer(PR.g2_to_bytes(PR.G2_GEN), np.uint8); tau_g2 = np.frombuffer(PR.g2_to_bytes(PR.g2_mul(tau, PR.G2_GEN)), np.uint8)
    Z, V, Rr = sc(z), sc(v), sc(r)
    out = {}
    for logk in sizes:
        k = 1 << logk
        args = (C[:k], Z[:k], V[:k], W[:k], Rr[:k], g2, tau_g2)
        assert eng.kzg_batch_verify(*args, check_points=0) == 1, "honest openings rejected at 2^%d" % logk
        bad = V[:k].copy(); bad[k // 3, 1] ^= 4
        assert eng.kzg_batch_verify(C[:k], Z[:k], bad, W[:k], Rr[:k], g2, tau_g2, check_points=0) == 0, "forged opening accepted at 2^%d" % logk
        wall, kt = timed_host_call(eng, lambda: eng.kzg_batch_verify(*args, check_points=0), steps)
        wall2, kt2 = timed_host_call(eng, lambda: eng.kzg_batch_verify(*args, check_points=2), steps)
        msm_ms = sum(ms for name, ms in kt.items() if name.startswith("msm_"))
        out["2^%d" % logk] = {"device_ms": sum(kt.values()), "e2e_ms": wall * 1e3, "msm_ms": msm_ms, "pairing_ms": kt.get("kzg_pairing"),
                              "with_subgroup_checks_device_ms": sum(kt2.values()), "g1_validate_ms": kt2.get("g1_validate"),
                              "openings_per_s": k / (sum(kt.values()) * 1e-3)}
    return out


def config_wire(eng, n):
    """SURVEY 8f-1: verification straight off the wire - serialised 32-byte keys, 8-byte VRF input data and 96-byte signatures
    (Output || c || s) in HOST memory -> verdicts + Output::hash, one C-ABI call (deserialisation with subgroup checks, Elligator2,
    verify, hash).  Signatures by the engine's own signer (bit-exact vs the oracle in tests)."""
    import numpy as np
    import ark_ec_vrfs_b200 as vrfs
    sk256, pk256 = eng.secret_from_seed(vrfs.BANDERSNATCH, [b"bench-wire-%d" % i for i in range(256)])
    sk = np.tile(sk256, (n // 256, 1)); pk_enc = np.tile(eng.point_encode(vrfs.BANDERSNATCH, pk256), (n // 256, 1))
    datas = (np.arange(n, dtype=np.uint64).view(np.uint8).copy(), np.arange(n + 1, dtype=np.uint64) * 8)
    sig, ok = eng.ietf_sign_wire(vrfs.BANDERSNATCH, sk, datas)
    assert ok.all()
    sig[::64, 40] ^= 1
    # page-locked host buffers in and out (as the headline's e2e leg): pageable ones make every copy a staged, synchronous one
    pk_enc, sig = pinned(pk_enc), pinned(sig)
    datas = (pinned(datas[0]), pinned(datas[1].view(np.uint8)).view(np.uint64))
    out_ok, out_hash = pinned_zeros((n,)), pinned_zeros((n, 64))
    best = None
    for _ in range(3):
        t0 = time.perf_counter(); okv, beta = eng.ietf_verify_wire(vrfs.BANDERSNATCH, pk_enc, datas, sig, out_ok=out_ok, out_hash=out_hash); dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    assert int(okv.sum()) == n - n // 64
    return {"what": "Bandersnatch: serialised keys + input data + 96-byte signatures (host) -> verdicts + 64-byte VRF outputs, %d items, 1/64 corrupted" % n,
            "verifies_per_s": n / best, "bytes_in_per_item": 32 + 8 + 96, "bytes_out_per_item": 65}


# ---------------------------------------------------------------------------------------------------------------------------
def run_reference(a, rank, world):
    """reference arm: the CPU oracle's ietf verify, all host threads, bounded sample per step (rank 0 only)"""
    if rank != 0:
        return
    import numpy as np
    import oracle_lib as O
    import vectors as V
    n = 1 << a.ref_logn
    w = V.make_ietf_proofs(O.BANDERSNATCH, n, "empty")
    cores = os.cpu_count() or 1
    for _ in range(a.warmup):
        O.ietf_verify(O.BANDERSNATCH, w["pk"], w["inp"], w["out"], w["c"], w["s"], None, nthreads=cores)
    t0 = time.perf_counter()
    for _ in range(a.steps):
        got = O.ietf_verify(O.BANDERSNATCH, w["pk"], w["inp"], w["out"], w["c"], w["s"], None, nthreads=cores)
    dt = time.perf_counter() - t0
    assert np.array_equal(got, w["expect"])
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, {"ietf_verify_ok": got})
    v = n * a.steps / dt
    sample = f"2^{a.ref_logn} distinct proofs per step (oracle-generated, same suite / ad as the GPU workload), {cores} pthreads"
    emit({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": dt / a.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (u64 on CPU)",
        "data": "synthetic", "config": {"workload": f"Bandersnatch IETF VRF batch verify, sample of 2^{a.ref_logn} per step on host CPU",
                                        "suite": "Bandersnatch_SHA-512_ELL2", "ad": "empty"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "note": "CPU restatement of the reference algorithm (oracle/vrf_oracle.c), not the arkworks binary"},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


_REAL_STDOUT = None


def quiet_stdout():
    """Everything any library prints on stdout (NCCL's version banner, ...) goes to stderr; the ONE JSON line is written to the
    real stdout by emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        os.write(1, line)
    else:
        os.write(_REAL_STDOUT, line)


def main():
    a = parse()
    quiet_stdout()
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    import numpy as np
    import torch
    import torch.distributed as dist
    import ark_ec_vrfs_b200 as vrfs

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        host_group = dist.new_group(backend="gloo")      # CPU-side barrier for the phase in which rank 0 drives every GPU by itself
    eng = vrfs.Engine(local)
    n = 1 << a.logn
    cores = os.cpu_count() or 1
    oracle_threads = max(1, cores // world)
    base = rank * n                                  # every rank proves and verifies its own index range: all items of the job are distinct
    w = make_verify_workload(eng, vrfs.BANDERSNATCH, base, n, False, oracle_threads)
    names = ("pk", "inp", "out", "c", "s")
    host = {k: torch.from_numpy(w[k]).pin_memory() for k in names}
    dev = {k: host[k].cuda(non_blocking=False) for k in names}
    d_ok = torch.zeros(n, dtype=torch.uint8, device="cuda")
    h_ok = torch.zeros(n, dtype=torch.uint8).pin_memory()
    expect = w["expect"]
    stream = torch.cuda.ExternalStream(eng.stream)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def gather(obj):
        """every rank's object on rank 0 (None elsewhere); ALWAYS called by all ranks, whatever happened inside a section"""
        if world == 1:
            return [obj]
        objs = [None] * world
        dist.all_gather_object(objs, obj)
        return objs

    def section(fn):
        """run a per-rank measurement; a failure on any rank becomes an error entry instead of a hang or a lost headline"""
        try:
            r = fn()
        except Exception as ex:   # noqa: BLE001
            r = {"error": repr(ex), "trace": traceback.format_exc(limit=3)}
        return gather(r)

    def step_dev(d=dev, ad=None, off=None):
        eng.ietf_verify_dev(vrfs.BANDERSNATCH, n, d["pk"].data_ptr(), d["inp"].data_ptr(), d["out"].data_ptr(),
                            d["c"].data_ptr(), d["s"].data_ptr(), d_ok.data_ptr(), ad, off)

    def step_host(h=host, m=n, ad=None, off=None):
        eng.ietf_verify_host_ptrs(vrfs.BANDERSNATCH, m, h["pk"].data_ptr(), h["inp"].data_ptr(), h["out"].data_ptr(),
                                  h["c"].data_ptr(), h["s"].data_ptr(), h_ok.data_ptr(), ad, off)

    # ---- integer-pipe peak, measured live (the roofline denominator of this path): the best sustained rate of any
    # 32x32->64-bit multiply(-accumulate) instruction form, each with data-dependent operands
    peak_probe = {"IMAD.WIDE.U32": eng.measure_mac32_peak(0)[0], "IMAD.HI.U32": eng.measure_mac32_peak(4)[0],
                  "IMAD.WIDE.U32.X carry rows": eng.measure_mac32_peak(5)[0]}
    peak_mac = max(peak_probe.values())

    # ---- device-resident timing
    for _ in range(max(a.warmup, 3)):
        step_dev()
    eng.sync()
    assert np.array_equal(d_ok.cpu().numpy(), expect), "GPU verdicts differ from the expected ones"
    eng.enable_kernel_timing(True)
    ktimes = {}
    sampler = ClockSampler(local); sampler.start()
    barrier()
    launches0 = eng.launch_count
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for _ in range(a.steps):
            step_dev()
            for name, ms in eng.kernel_timings():
                ktimes.setdefault(name, []).append(ms)
        ev1.record(stream)
    barrier()
    launches = eng.launch_count - launches0
    ms_total = ev0.elapsed_time(ev1)
    clocks = sampler.stop()
    eng.enable_kernel_timing(False)
    verdicts = d_ok.cpu().numpy()
    assert np.array_equal(verdicts, expect)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, {"ietf_verify_ok": verdicts})

    # ---- end to end through the host-buffer ABI (pinned host memory; H2D/D2H inside)
    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step_host()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert np.array_equal(h_ok.numpy(), expect)

    # ---- strong scaling: ONE batch of 2^logn items over the N GPUs (rank g takes the g-th index range), host buffers, max over ranks
    lo, hi = (n * rank) // world, (n * (rank + 1)) // world
    hs = {k: host[k][lo:hi] for k in names}
    for _ in range(2):
        step_host(hs, hi - lo)
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.steps):
        step_host(hs, hi - lo)
    torch.cuda.synchronize()
    strong_s = time.perf_counter() - t0
    assert np.array_equal(h_ok.numpy()[:hi - lo], expect[lo:hi])

    t = torch.tensor([ms_total, e2e_s * 1e3, strong_s * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, strong_ms = float(t[0]), float(t[1]), float(t[2])
    value = n * world * a.steps / (ms_total * 1e-3)
    e2e_value = n * world * a.steps / (e2e_ms * 1e-3)

    # ---- secondary configs (all ranks; results gathered on rank 0)
    extras = {}
    if world > 1 and not a.headline_only:
        # the peer group of the MSM exchange: one host-side all-gather of the 64-byte mailbox handles.  Generous timeout: the ranks
        # reach the collective MSM calls seconds apart (their CPU-side preparation differs); a lost peer still cannot hang a GPU.
        from ark_ec_vrfs_b200 import dist as D
        if D.connect_peers(eng):
            eng.peer_set_timeout_ms(30000)
    if not a.headline_only:
        ksteps = max(2, min(a.steps, 5))

        def with_ad():
            wa = make_verify_workload(eng, vrfs.BANDERSNATCH, base, n, True, oracle_threads)
            ha = {k: torch.from_numpy(wa[k]).pin_memory() for k in names}
            da = {k: ha[k].cuda() for k in names}
            adh, offh = torch.from_numpy(wa["ads"][0]).pin_memory(), torch.from_numpy(wa["ads"][1].view(np.int64)).pin_memory()
            add, offd = adh.cuda(), offh.cuda()
            for _ in range(2):
                step_dev(da, add.data_ptr(), offd.data_ptr())
            eng.sync()
            assert np.array_equal(d_ok.cpu().numpy(), wa["expect"])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                e0.record(stream)
                for _ in range(ksteps):
                    step_dev(da, add.data_ptr(), offd.data_ptr())
                e1.record(stream)
            eng.sync()
            dms = e0.elapsed_time(e1) / ksteps
            step_host(ha, n, adh.data_ptr(), offh.data_ptr())
            t0 = time.perf_counter()
            for _ in range(ksteps):
                step_host(ha, n, adh.data_ptr(), offh.data_ptr())
            wall = (time.perf_counter() - t0) / ksteps
            assert np.array_equal(h_ok.numpy(), wa["expect"])
            return {"device_ms": dms, "e2e_ms": wall * 1e3, "oracle_checked_items": wa["oracle_checked_items"]}

        extras["with_ad32"] = section(with_ad)
        extras["ietf_prove_ed25519"] = section(lambda: config_ietf_prove(eng, vrfs.ED25519, base, n, ksteps, peak_mac, oracle_threads))
        extras["ietf_prove_secp256r1"] = section(lambda: config_ietf_prove(eng, vrfs.P256, base, n, ksteps, peak_mac, oracle_threads))
        extras["pedersen_bandersnatch"] = section(lambda: config_pedersen(eng, base, n, ksteps, peak_mac, oracle_threads))
        hbm_peak_, _ = measured_peaks()
        extras["ring_kzg_msm_ms"] = section(lambda: config_msm(eng, rank, world, peak_mac, hbm_peak_, list(range(11, 18))))
        if world == 1:
            extras["kzg_batch_verify_ms"] = section(lambda: config_kzg(eng, list(range(10, 17))))
            extras["ietf_verify_wire"] = section(lambda: config_wire(eng, min(n, 1 << 20)))

    # ---- one caller, all GPUs (vrfs_ctx_create_multi): rank 0 drives every device of the job with ONE host call per step while the
    # other ranks idle at the barrier
    multi = None
    if world > 1 and not a.headline_only:
        barrier()
        # the other ranks must wait on the HOST: an NCCL barrier would park a spinning kernel on the GPUs rank 0 is about to use
        if rank == 0:
            try:
                with vrfs.MultiEngine(list(range(world))) as me:
                    for _ in range(2):
                        me.ietf_verify_host_ptrs(vrfs.BANDERSNATCH, n, host["pk"].data_ptr(), host["inp"].data_ptr(), host["out"].data_ptr(),
                                                 host["c"].data_ptr(), host["s"].data_ptr(), h_ok.data_ptr())
                    t0 = time.perf_counter()
                    for _ in range(a.steps):
                        me.ietf_verify_host_ptrs(vrfs.BANDERSNATCH, n, host["pk"].data_ptr(), host["inp"].data_ptr(), host["out"].data_ptr(),
                                                 host["c"].data_ptr(), host["s"].data_ptr(), h_ok.data_ptr())
                    dt = (time.perf_counter() - t0) / a.steps
                    assert np.array_equal(h_ok.numpy(), expect)
                    multi = {"what": "vrfs_multi_ietf_verify_batch: one process, one call per step, 2^%d host items sharded over %d GPUs" % (a.logn, world),
                             "verifies_per_s": n / dt, "ms_per_step": dt * 1e3}
            except Exception as ex:   # noqa: BLE001
                multi = {"error": repr(ex)}
        dist.barrier(group=host_group)
        barrier()

    if rank == 0:
        kavg = {k: sum(v) / len(v) for k, v in ktimes.items()}
        dom = max(kavg, key=kavg.get)
        dom_s = kavg[dom] * 1e-3
        muls = kernel_muls(0, dom) or 0
        achieved = n * muls * MAC_PER_MUL / dom_s
        executed = {"lincomb<2,0>": 2255, "lincomb<1,1>": 1750}.get(dom)
        hbm_peak, hbm_src = measured_peaks()
        bytes_per_item = {"lincomb<2,0>": 64 + 64 + 32 + 32 + 96, "lincomb<1,1>": 64 + 32 + 32 + 96, "ietf_verify_finish": 3 * 64 + 32 + 2 * 96 + 2}.get(dom, 0)
        hbm_ach = n * bytes_per_item / dom_s / 1e9
        total_k = sum(kavg.values())
        traffic = ncu_record(dom, "dram_bytes_per_launch", n)
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_total / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32 limbs (256-bit Montgomery, integer)", "data": "synthetic",
            "config": {"workload": f"Bandersnatch IETF VRF batch verify, 2^{a.logn} distinct proofs per GPU (BASELINE configs[1])",
                       "suite": "Bandersnatch_SHA-512_ELL2", "ad": "empty", "batch_per_gpu": n, "invalid_fraction": float(1 - expect.mean()),
                       "distinct_items": int(n * world), "generator": "engine prover on the GPU (Secret::from_seed, Input::new, Secret::output, ietf prove); keys, inputs, proofs and verdicts oracle-checked on a 2^12 subsample per rank",
                       "oracle_checked_items_per_rank": w["oracle_checked_items"],
                       "l2": "inputs (256 B/item = %.0f MB) exceed the 126 MB L2; no flush needed" % (n * 256 / 1e6),
                       "parallelism": f"batch sharded by index range over {world} GPU(s), no collective"},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n * 256, "d2h_bytes_per_step": n, "ms_per_step": e2e_ms / a.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "int32-mac (IMAD pipe; no tensor-core or HBM-bound stage on this path)", "kernel": dom,
                         "achieved": achieved / 1e12, "peak": peak_mac / 1e12, "unit": "TMAC32/s", "frac": achieved / peak_mac,
                         "peak_source": "measured live: max over 64-bit-product instruction microbenchmarks (vrfs_measure_mac32_peak)",
                         "peak_probe_tmac32": {k: v / 1e12 for k, v in peak_probe.items()},
                         "algorithmic_per_item": {"field_muls": muls, "mac32_per_mul": MAC_PER_MUL, "source": "SURVEY.md Appendix D",
                                                  "executed_product_equivalents_estimate": executed},
                         "kernel_ms": kavg, "kernel_share": {k: v / total_k for k, v in kavg.items()},
                         "traffic": traffic,
                         "traffic_unit": "bytes/launch (dram read+write of the dominant kernel, ncu --set full capture under profiles/)",
                         "fmaheavy_pipe_active_pct_ncu": ncu_record(dom, "fmaheavy_pipe_active_pct", n),
                         "hbm": {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak, "peak_source": hbm_src,
                                 "bytes_per_item": bytes_per_item}},
            "strong_scaling": {"what": f"ONE batch of 2^{a.logn} host items over {world} GPU(s): rank g verifies the g-th index range, H2D/D2H inside, max over ranks",
                               "value": n * a.steps / (strong_ms * 1e-3), "unit": UNIT, "ms_per_step": strong_ms / a.steps, "items_per_gpu": n // world},
        }
        if multi:
            out["one_caller_multi_gpu"] = multi
        if world == 1 and not a.no_cpu_baseline:
            import oracle_lib as O
            m = min(n, 1 << a.cpu_sample_logn)
            t0 = time.perf_counter()
            got = O.ietf_verify(O.BANDERSNATCH, w["pk"][:m], w["inp"][:m], w["out"][:m], w["c"][:m], w["s"][:m], None, nthreads=cores)
            dt = time.perf_counter() - t0
            assert np.array_equal(got, expect[:m])
            out["cpu_baseline"] = {"value": m / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                   "sample": f"first 2^{a.cpu_sample_logn} proofs of the same workload, {cores} pthreads, {dt:.1f} s",
                                   "note": "CPU restatement of the reference algorithm (oracle/vrf_oracle.c), not the arkworks binary"}
        # ---- aggregate the per-rank sections: rates add up over ranks, times take the slowest rank
        def agg(rs, path, how):
            vals = []
            for r in rs:
                x = r
                for k in path:
                    x = x.get(k) if isinstance(x, dict) else None
                if x is None:
                    return None
                vals.append(x)
            return sum(vals) if how == "sum" else max(vals)

        def errors(rs):
            e = [r["error"] for r in rs if isinstance(r, dict) and "error" in r]
            return e or None

        if "with_ad32" in extras:
            rs = extras["with_ad32"]
            if errors(rs):
                out["with_ad32"] = {"error": errors(rs)}
            else:
                dms, ems = agg(rs, ["device_ms"], "max"), agg(rs, ["e2e_ms"], "max")
                out["with_ad32"] = {"what": "the headline with 32-byte additional data per item (SHA-256(u64le(i))), distinct proofs made with that ad",
                                    "value": n * world / (dms * 1e-3), "e2e": n * world / (ems * 1e-3), "unit": UNIT, "device_ms_per_step": dms, "e2e_ms_per_step": ems}
        for key, label in (("ietf_prove_ed25519", "Ed25519_SHA-512_TAI"), ("ietf_prove_secp256r1", "secp256r1 (RFC 9381 suite 0x01)")):
            if key in extras:
                rs = extras[key]
                if errors(rs):
                    out[key] = {"error": errors(rs)}
                else:
                    out[key] = {"what": f"BASELINE configs[2]: {label} IETF prove of 2^{a.logn} items per GPU with deterministic nonces, host buffers in and out",
                                "unit": "proves/s", "e2e": agg(rs, ["e2e_per_s"], "sum"), "device": agg(rs, ["device_per_s"], "sum"),
                                "e2e_ms_per_step": agg(rs, ["e2e_ms"], "max"), "device_ms_per_step": agg(rs, ["device_ms"], "max"),
                                "h2d_bytes_per_step": rs[0]["h2d_bytes"], "d2h_bytes_per_step": rs[0]["d2h_bytes"],
                                "oracle_checked_items_per_rank": rs[0]["oracle_checked_items"], "roofline": rs[0]["roofline"]}
        if "pedersen_bandersnatch" in extras:
            rs = extras["pedersen_bandersnatch"]
            if errors(rs):
                out["pedersen_bandersnatch"] = {"error": errors(rs)}
            else:
                o = {"what": f"BASELINE configs[3]: Pedersen VRF prove and verify of 2^{a.logn} items per GPU over Bandersnatch, host buffers in and out",
                     "oracle_checked_items_per_rank": rs[0]["oracle_checked_items"]}
                for leg, unit in (("prove", "proves/s"), ("verify", "verifies/s")):
                    o[leg] = {"unit": unit, "e2e": agg(rs, [leg, "e2e_per_s"], "sum"), "device": agg(rs, [leg, "device_per_s"], "sum"),
                              "e2e_ms_per_step": agg(rs, [leg, "e2e_ms"], "max"), "device_ms_per_step": agg(rs, [leg, "device_ms"], "max"),
                              "h2d_bytes_per_step": rs[0][leg]["h2d_bytes"], "d2h_bytes_per_step": rs[0][leg]["d2h_bytes"], "roofline": rs[0][leg]["roofline"]}
                out["pedersen_bandersnatch"] = o
        if "ring_kzg_msm_ms" in extras:
            rs = extras["ring_kzg_msm_ms"]
            if errors(rs):
                out["ring_kzg_msm_ms"] = {"error": errors(rs)}
            else:
                o = {"what": "BASELINE configs[4]: 3-column commitment MSM over BLS12-381 G1 with a prepared SRS, domain size N (ring size N/2), uniform field elements; ring_commit: the fixed columns of a ring of N/2 keys built on the device and committed in one call over a Lagrange-basis SRS; single_gpu = every rank alone, sharded = the SRS split by point range over all ranks (times: slowest rank)",
                     "exchange": rs[0]["exchange"], "n_gpus": world}
                for key in [k for k in rs[0] if k.startswith("2^")]:
                    e = {"single_gpu": rs[0][key]["single_gpu"]}
                    if "sharded" in rs[0][key]:
                        e["sharded"] = {f: agg(rs, [key, "sharded", f], "max") for f in ("device_ms", "e2e_ms", "ring_commit_device_ms", "ring_commit_e2e_ms")}
                        e["sharded"]["points_per_rank"] = rs[0][key]["sharded"]["points_per_rank"]
                        e["sharded"]["kernel_ms_rank0"] = rs[0][key]["sharded"]["kernel_ms"]
                    o[key] = e
                out["ring_kzg_msm_ms"] = o
        if "kzg_batch_verify_ms" in extras:
            out["kzg_batch_verify_ms"] = {"what": "BASELINE configs[4] 'plus batched ring-proof verify' (SURVEY 8f-3): k KZG openings (commitment, point, value, proof, transcript coefficient) checked at once = one 2-column MSM over 2k+1 G1 points + one product of two BLS12-381 pairings; every size accepts honest openings and rejects one forged value",
                                          **extras["kzg_batch_verify_ms"][0]}
        if "ietf_verify_wire" in extras:
            out["ietf_verify_wire"] = extras["ietf_verify_wire"][0]
        emit(out)
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
