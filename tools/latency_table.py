#!/usr/bin/env python3
"""Wall-clock latency of the small-batch entry points (VERDICT r1 item 4): median and p90 over repeated synchronous calls
through the C ABI with host buffers, n = 1, 4, 32, 483, 4096, all three kinds, plus the one-call drop-ins.
Prints one JSON object (committed under profiles/)."""
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import lightning_b200 as L  # noqa: E402
from tests import util  # noqa: E402


def timed(fn, reps):
    for _ in range(5):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e6)
    ts.sort()
    return {"median_us": round(ts[len(ts) // 2], 1), "p90_us": round(ts[int(len(ts) * 0.9)], 1), "min_us": round(ts[0], 1)}


def main():
    eng = L.SigVerifier(0)
    ref = util.load_ref()
    sizes = tuple(int(x) for x in os.environ.get("SV_LATENCY_SIZES", "1,4,32,483,4096").split(","))
    w = util.make_signed(max(4096, max(sizes)), seed=7)
    out = {"small_max": eng.small_max(), "sizes": {}, "note": "synchronous sv_verify_host calls, pageable numpy host buffers, perf_counter around the call"}
    kinds = (("ecdsa33", 0, "pub33", "sig"), ("ecdsa_xy", 1, "pubxy", "sig"), ("schnorr", 2, "xonly", "ssig"))
    for n in sizes:
        row = {}
        for name, kind, kk, ss in kinds:
            m, k, s = (np.ascontiguousarray(w[x][:n]) for x in ("msg", kk, ss))
            v = np.zeros(n, np.uint8)
            fn = lambda: eng.lib.sv_verify_host(eng._ctx, kind, m.ctypes.data, k.ctypes.data, s.ctypes.data, n, v.ctypes.data)
            row[name] = timed(fn, 300 if n <= 483 else 100)
            assert v.all()
        # the reference's CPU path on the same n (one thread, as CLN's daemons run it)
        m, k, s = (np.ascontiguousarray(w[x][:n]) for x in ("msg", "pub33", "sig"))
        row["cpu_reference_1thread"] = timed(lambda: util.ref_verify(ref, 0, m, k, s, 1), 20 if n > 483 else 100)
        if n == 483:
            key = np.ascontiguousarray(w["pub33"][0])
            sk_msgs = np.ascontiguousarray(w["msg"][:n])
            # same-key entry point needs signatures by one key: reuse timing only (verdicts are mostly 0)
            sig = np.ascontiguousarray(w["sig"][:n])
            v = np.zeros(n, np.uint8)
            row["samekey_ecdsa33"] = timed(lambda: eng.lib.sv_verify_samekey_host(eng._ctx, 0, key.ctypes.data, sk_msgs.ctypes.data, sig.ctypes.data, n, v.ctypes.data), 200)
        out["sizes"][str(n)] = row
    # single-warp dependent-chain latency of the field primitives (cycles at the measured clock come from the probe)
    try:
        out["probe_single_warp_fe_mul_per_s"] = eng.probe(9)
        out["probe_single_warp_fe_sqr_per_s"] = eng.probe(10)
    except Exception as ex:
        out["probe_single_warp"] = repr(ex)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
