#!/usr/bin/env python3
"""Public-key recovery measurements (writes one JSON object, default profiles/r3_recover.json).

Workload: sv_synth_device(SV_KIND_ECDSA33) signatures; the timed passes use recid 0, and an untimed second call with
recid 1 on the items whose key did not come back must account for every remaining item, so that every key is proven
equal to its signer's.
  * throughput at 1 M items: sv_recover_host end to end (host buffers, pinned; profiler off) and the kernels' span in a
    torch.profiler trace of one call (a 1 M call runs as several slices on two streams, so the engine's profiling events
    would time only the last slice), next to plain-flow compressed-key verification (sv_set_nosqrt(0)) of the same
    items in the same run;
  * latency (small-batch kernel) at n = 1, 4, 32, 483, 4096, 8192: wall clock of the synchronous call, median;
  * libsecp256k1's parse_compact + secp256k1_ecdsa_recover on one and on all host cores (oracle/_ref, one ctypes call
    sequence per item from Python threads, so slightly below what a C loop reaches), on a sample;
  * the card's name and power limit, read in the same run.
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
import lightning_b200 as L  # noqa: E402
from tests import recovery  # noqa: E402


def card():
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_recover.json"))
    ap.add_argument("-n", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    n = a.n
    eng = L.SigVerifier(0)
    out = {"card": card(), "n": n}
    msg = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    key = torch.empty((n, 33), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    eng.synth_device(L.KIND_ECDSA33, 4242, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr())
    eng.sync()

    def pin(t):
        x = t.cpu().numpy()
        b = eng.host_alloc(x.nbytes)
        b[:] = x.reshape(-1)
        return b.reshape(x.shape)
    m, k, s = pin(msg), pin(key), pin(sig)
    r0 = pin(torch.zeros(n, dtype=torch.uint8))

    def kernel_span(fn):
        """(sum of kernel durations, first kernel start to last kernel end) in ms of one call, from a torch.profiler trace:
        a 1 M call runs as several slices on two streams, so the engine's own events would time only the last slice"""
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        ks = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "k_" in e.name]
        names = sorted({e.name.split("(")[0] for e in ks})
        t0, t1 = min(e.time_range.start for e in ks), max(e.time_range.end for e in ks)
        return sum(e.time_range.elapsed_us() for e in ks) * 1e-3, (t1 - t0) * 1e-3, names

    def timed(fn, reps):
        fn()  # warm-up of the same shape
        walls = []
        for _ in range(reps):
            t0 = time.perf_counter()
            r = fn()
            walls.append(time.perf_counter() - t0)
        return r, float(np.median(walls))

    # ---- throughput, recovery and plain-flow verification alternated in one run (profiler off while timing) ----
    eng.set_nosqrt(False)
    rec, verif = [], []
    for _ in range(2):
        (xy, st), wall = timed(lambda: eng.recover(m, s, r0), a.reps)
        rec.append(wall)
        v, vwall = timed(lambda: eng.verify(L.KIND_ECDSA33, m, k, s), a.reps)
        verif.append(vwall)
    assert v.all()
    wall, vwall = min(rec), min(verif)
    out["recover_1M"] = {"e2e_ms": wall * 1e3, "e2e_per_s": n / wall}
    out["verify_ecdsa33_plain_flow_1M"] = {"e2e_ms": vwall * 1e3, "e2e_per_s": n / vwall}
    try:
        for name, fn in (("recover_1M", lambda: eng.recover(m, s, r0)),
                         ("verify_ecdsa33_plain_flow_1M", lambda: eng.verify(L.KIND_ECDSA33, m, k, s))):
            spans = [kernel_span(fn) for _ in range(3)]
            busy, span, names = min(spans, key=lambda t: t[1])
            out[name].update(kernel_span_ms=span, kernel_per_s=n / (span * 1e-3), kernel_busy_ms=busy, kernels=names)
        out["recover_over_verify_kernel"] = out["recover_1M"]["kernel_per_s"] / out["verify_ecdsa33_plain_flow_1M"]["kernel_per_s"]
    except Exception as e:  # noqa: BLE001 - the trace is an extra; the wall-clock numbers above stand without it
        out["kernel_time"] = f"not measured: {type(e).__name__}: {e}"
    eng.set_nosqrt(True)

    # ---- every key proven: recid 0 (timed above), recid 1 for the rest (untimed) ----
    def hits(xy, st, kk):
        return (st == 1) & ((xy[:, 63] & 1) == kk[:, 0] - 2) & (xy[:, :32] == kk[:, 1:]).all(axis=1)
    h0 = hits(xy, st, k)
    miss = np.nonzero(~h0)[0]
    xy1, st1 = eng.recover(np.ascontiguousarray(m[miss]), np.ascontiguousarray(s[miss]), np.ones(miss.size, np.uint8))
    h1 = hits(xy1, st1, k[miss])
    assert h1.all(), f"{int((~h1).sum())} keys not recovered"
    out["keys_checked"] = {"recid0": int(h0.sum()), "recid1": int(h1.sum()), "all_signers": True}

    # ---- latency on the small-batch kernel ----
    lat = {}
    for cnt in (1, 4, 32, 483, 4096, 8192):
        mm, ss, rr = (np.ascontiguousarray(x[:cnt]) for x in (m, s, r0))
        eng.recover(mm, ss, rr)
        walls = []
        for _ in range(max(20, a.reps)):
            t0 = time.perf_counter()
            eng.recover(mm, ss, rr)
            walls.append(time.perf_counter() - t0)
        lat[str(cnt)] = {"median_us": float(np.median(walls)) * 1e6, "min_us": float(np.min(walls)) * 1e6}
    out["latency_small_path"] = lat

    # ---- the reference on the host ----
    try:
        live = recovery.LiveReference()
        cnt = 20000
        w = {"msg": m[:cnt], "sig": s[:cnt], "recid": r0[:cnt]}
        cores = os.cpu_count()
        res = {}
        for th in (1, cores):
            t0 = time.perf_counter()
            xy, stv = live.recover(w, threads=th)
            dt = time.perf_counter() - t0
            res[f"threads_{th}"] = {"per_s": cnt / dt}
        gx, gs = eng.recover(*(np.ascontiguousarray(w[k]) for k in ("msg", "sig", "recid")))
        assert np.array_equal(gs, stv) and np.array_equal(gx, xy)
        out["libsecp256k1_recover"] = dict(res, sample=cnt, host_cores=cores, bit_exact_vs_engine=True)
    except RuntimeError as e:
        out["libsecp256k1_recover"] = f"not measured: {e}"
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out, indent=1))
    eng.close()


if __name__ == "__main__":
    main()
