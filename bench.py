#!/usr/bin/env python3
"""bench.py — secp256k1 verifies/sec on N B200s (BASELINE.json metric), one JSON line on rank 0.

  python bench.py [--gpus N] [--steps K] [--warmup W]          engine arm (CUDA, this repo)
  python bench.py --impl reference [...]                       the reference's own CPU path (oracle/_ref)
  python bench.py --dump-outputs DIR [...]                     also write the last timed step's verdicts to DIR

Workload (config.workload): BASELINE.json configs[1] — "1M ECDSA verifies, single B200": per GPU and per
step one batch of 1,000,000 (msg32, pub33, sig64) triples, random distinct keys, 90 % valid + 10 % corrupted
(SURVEY.md §8(d) classes).  A "step" is one pass of the hot path (scalar-side kernel + curve-side kernel)
over one batch.  Two alternating batches are kept resident (2 x (129 MB inputs + 128 MB work records)
+ 58 MB per-thread tables > 126 MB L2), so no step finds its inputs in L2.

  value     whole-job verifies/s, inputs resident in HBM when the timed region starts
  e2e       same metric through the public host-buffer API (sv_verify_host): pinned host inputs -> H2D ->
            kernels -> D2H verdict bytes, all inside the timed region
  roofline  integer-pipe roofline of the curve-side kernel: algorithmic 32x32->64 multiply-accumulates
            (125,440 per ECDSA verify from a 33-byte key, SURVEY.md §8(d)) / CUDA-event time of that kernel,
            against the IMAD.WIDE.U32 peak MEASURED live by the engine's probe kernel.  The path is
            integer-compute bound, not HBM bound; the HBM view is reported beside it (roofline_hbm).
  cpu_baseline  oracle/_ref (unmodified libsecp256k1) on all host cores over a bounded sample of the same
            batch, verdicts compared bit for bit with the GPU's.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ORDER = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
BATCH = 1_000_000
IMAD_PER_VERIFY = 125_440  # 1,960 field mults x 64 (SURVEY.md §8(d))
BYTES_PER_VERIFY = 129.125
# dram__bytes_read.sum + dram__bytes_write.sum of ONE curve-kernel launch over 1,000,000 verifications, from `ncu --set full`
# (round 2: 724.9 MB + 311.6 MB; round 1 was 766.8 + 562.9 MB).  Algorithmic traffic is 0.32 GB (161 B of input, the 128-byte
# work record in and out, the verdict); the rest are the comb's random 64-byte reads out of a 34 MiB table and the part of
# the per-thread Q-table slabs that the L2 access-policy window cannot hold.
NCU_DRAM_BYTES_PER_1M_LAUNCH = 724_892_672 + 311_600_384  # dram__bytes_read + _write, profiles/r2_k_main_nosqrt_ncu_summary.md
# IMAD.WIDE.U32 the shipped curve kernel EXECUTES per verification (ncu, profiles/r2_k_main_nosqrt_dynamic_opmix.txt:
# 3,571,030,146 warp instructions x 32 lanes / 1,000,000): the flow without the square root does less than SURVEY's 125,440
EXECUTED_IMAD_PER_VERIFY = 114_273
METRIC = "secp256k1 verifies/sec"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# --------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi, during the timed region)
# --------------------------------------------------------------------------------------------------
class ClockSampler:
    """One streaming `nvidia-smi -lms 100` process for the duration of the timed regions."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.samples = []
        self._proc = None
        self._th = None

    def _run(self):
        for line in self._proc.stdout:
            parts = [p.strip() for p in line.strip().split(",")]
            if len(parts) >= 8:
                self.samples.append(parts)

    def start(self):
        try:
            self._proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.FIELDS,
                                           "--format=csv,noheader,nounits", "-lms", "100"],
                                          stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()
        except Exception:
            self._proc = None

    def stop(self):
        if self._proc:
            self._proc.terminate()
            try:
                self._proc.wait(timeout=5)
            except Exception:
                self._proc.kill()
        if self._th:
            self._th.join(timeout=5)
        sm = sorted(int(float(s[1])) for s in self.samples if s[1].replace(".", "").isdigit())
        mx = [int(float(s[2])) for s in self.samples if s[2].replace(".", "").isdigit()]
        pw = [float(s[3]) for s in self.samples if s[3].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation (oracle/_ref), all host threads
# --------------------------------------------------------------------------------------------------
def load_ref():
    path = os.path.join(ROOT, "oracle", "_ref", "libsecp_ref.so")
    kind = "reference"
    if not os.path.exists(path):
        if os.path.isdir("/root/reference"):
            subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "ref"])
    if os.path.exists(path):
        return ctypes.CDLL(path), kind
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"])
    return ctypes.CDLL(os.path.join(ROOT, "oracle", "libsecp_port.so")), "port"


def cpu_verify(lib, kind, msg, pub, sig, threads):
    n = msg.shape[0]
    out = np.zeros(n, np.uint8)
    fn = lib.ref_ecdsa_verify_batch if kind == "reference" else lib.port_ecdsa_verify_batch
    p8 = ctypes.POINTER(ctypes.c_uint8)
    fn(msg.ctypes.data_as(p8), pub.ctypes.data_as(p8), sig.ctypes.data_as(p8), ctypes.c_size_t(n),
       out.ctypes.data_as(p8), int(threads))
    return out


def host_cores():
    """(threads to use, logical CPUs visible, cgroup CPU limit or None).  A container lease can see every logical CPU of
    the host through sched_getaffinity and still be held to a CPU-time quota by its cgroup (cpu.max); the number of
    cores the reference can actually use is the smaller of the two, and that is what `cores` reports."""
    try:
        logical = max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        logical = max(1, os.cpu_count() or 1)
    limit = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            limit = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                limit = q / per
        except Exception:
            pass
    threads = logical if limit is None else max(1, min(logical, int(limit + 0.999)))
    return threads, logical, limit


def host_threads():
    return host_cores()[0]


def cores_note():
    t, logical, limit = host_cores()
    return {"cores": t, "logical_cpus": logical, "cgroup_cpu_limit": limit}


BENCH_SEED = 20260922
WORKLOAD = ("1M random-key ECDSA (msg32,pub33,sig64) verifies per GPU per step [BASELINE configs[1]]; triples from the "
            "reference signer (secp256k1_ecdsa_sign, RFC6979) over SplitMix64 keys/hashes, seed 20260922, 90% valid / 10% "
            "corrupted in 7 classes")


def bench_config(world):
    """`config` of the JSON line — the SAME object in both arms (the arms differ in `impl`, not in workload)."""
    return {"workload": WORKLOAD, "batch_per_gpu": BATCH, "valid_fraction": 0.9, "kind": "ecdsa33",
            "l2": "two alternating resident batches; inputs+work records+tables per step exceed the 126 MB L2",
            "parallelism": f"dp{world} (independent shards; NCCL all_gather of the verdict bitmap)" if world > 1 else "dp1"}


def make_reference_batch(lib, seed, n, threads):
    """(msg, pub33, sig) numpy arrays: n triples signed by the UNMODIFIED reference (oracle/_ref ref_make_ecdsa_batch:
    SplitMix64 keys and hashes from (seed, i), secp256k1_ecdsa_sign, every 10th item corrupted round-robin over the 7
    classes of SURVEY.md 8(d)).  Input generation only: nothing here is on a timed path."""
    p8 = ctypes.POINTER(ctypes.c_uint8)
    msg = np.zeros((n, 32), np.uint8)
    pub = np.zeros((n, 33), np.uint8)
    sig = np.zeros((n, 64), np.uint8)
    lib.ref_make_ecdsa_batch(ctypes.c_uint64(seed), ctypes.c_size_t(n), msg.ctypes.data_as(p8), pub.ctypes.data_as(p8),
                             sig.ctypes.data_as(p8), int(threads))
    return msg, pub, sig


def run_reference(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    lib, kind = load_ref()
    threads = host_threads()
    if kind != "reference":
        # cannot happen while oracle/_ref travels with the snapshot; keep the driver's contract anyway
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libsecp_ref.so is missing (the port has no signer)"}))
        return 0
    # the SAME bytes the engine arm verifies (rank 0's first batch); each step verifies a bounded sample of it, sized so
    # that the whole --steps/--warmup run is ~60 s of all-core work at ~20k verifies/s/core (at most one batch per step)
    budget = 60.0 * 20_000 * threads
    sample = int(min(BATCH, max(2_000 * threads, budget / (args.steps + args.warmup))))
    msg, pub, sig = make_reference_batch(lib, BENCH_SEED, BATCH, threads)
    msg, pub, sig = (np.ascontiguousarray(a[:sample]) for a in (msg, pub, sig))
    for _ in range(args.warmup):
        cpu_verify(lib, kind, msg, pub, sig, threads)
    t0 = time.perf_counter()
    valid = 0
    for _ in range(args.steps):
        valid = int(cpu_verify(lib, kind, msg, pub, sig, threads).sum())
    dt = time.perf_counter() - t0
    value = sample * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "verifies/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u64 limbs (libsecp256k1 5x52 field / 4x64 scalar)",
        "data": "synthetic",
        "config": bench_config(max(1, args.gpus)),
        "reference": {"sample_per_step": sample, "valid_in_sample": valid,
                      "note": "each step verifies the first sample_per_step triples of the engine arm's batch (same bytes)"},
        "cpu_baseline": dict({"value": value, "unit": "verifies/s", "kind": kind,
                              "sample": f"first {sample} triples of the bench batch x {args.steps} steps, ec_pubkey_parse + signature_parse_compact + ecdsa_verify per item"},
                             **cores_note()),
        "e2e": {"value": value, "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------------
# engine arm
# --------------------------------------------------------------------------------------------------
def corrupt_on_device(torch, msg, key, sig):
    """Every 10th item gets one of the 7 SURVEY §8(d) corruption classes (round-robin).  Returns the
    expected-invalid index tensor.  msg (n,32), key (n,33), sig (n,64) uint8 CUDA tensors, all valid."""
    n = msg.shape[0]
    idx = torch.arange(0, n, 10, device=msg.device)
    cls = torch.arange(idx.numel(), device=msg.device) % 7
    sel = lambda c: idx[cls == c]
    msg[sel(0), 5] ^= 4
    sig[sel(1), 7] ^= 1
    sig[sel(2), 40] ^= 1
    hs = sel(3)  # s <- n - s (host big-int on the ~1.4 % affected rows)
    rows = sig[hs, 32:].cpu().numpy()
    for r in range(rows.shape[0]):
        s = int.from_bytes(rows[r].tobytes(), "big")
        rows[r] = np.frombuffer((N_ORDER - s).to_bytes(32, "big"), dtype=np.uint8)
    sig[hs, 32:] = torch.from_numpy(rows).to(sig.device)
    nb = sel(4)
    key[nb] = key[(nb + 1) % n].clone()
    nr = sel(5)  # x = 5 is not on the curve (5^3 + 7 is a non-residue)
    key[nr, 1:] = 0
    key[nr, 32] = 5
    key[sel(6), 0] = 4
    return idx


def dump_outputs(out_dir, verdict, bitmap, gathered):
    """What a caller of the timed path receives from one step, as float64 .npy files in out_dir: the verdict bytes, the
    verdict bitmap's 32-bit words and, with N > 1, the bitmap gathered from every rank (8.3 MB, plus 0.25 MB per rank)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"verdicts": verdict, "bitmap": bitmap}
    if gathered is not None:
        arrays["gathered_bitmap"] = gathered
    for name, t in arrays.items():
        a = t.cpu().numpy()
        if a.dtype == np.int32:
            a = a.view(np.uint32)
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


def run_engine(args):
    import torch
    import lightning_b200 as L

    world = env_int("WORLD_SIZE", 1)
    rank = env_int("RANK", 0)
    local = env_int("LOCAL_RANK", 0)
    dist = None
    # keep stdout to the one JSON line: NCCL prints its version banner there when NCCL_DEBUG=VERSION
    # (NCCL writes its debug output, including that banner, to stdout unless told otherwise)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        os.environ.pop("NCCL_DEBUG")
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        # the only collective is a 125 KB-per-rank gather: two channels (= two CTAs, the slots SV_MAIN_GRID_RESERVE leaves
        # free beside the persistent curve grid) are plenty, and more could not be placed anyway
        os.environ.setdefault("NCCL_MAX_NCHANNELS", "2")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # leave two CTA slots of the persistent curve kernel free for NCCL's gather kernel: with the full grid resident it
        # only gets an SM when a curve CTA retires and then delays a CTA of the next launch (measured at N = 2: 103.6 ->
        # 105.4 M verifies/s, profiles/r2_n2_grid_reserve.txt; costs 0.7 % of a lone GPU, so not the N = 1 default)
        os.environ.setdefault("SV_MAIN_GRID_RESERVE", "2")
    eng = L.SigVerifier(local)  # raises if the CUDA library or the GPU is missing: no CPU path
    eng.set_profiling(True)
    kind = L.KIND_ECDSA33
    n = BATCH
    # Two launch streams, used alternately by consecutive steps: the engine gives each in-flight launch pair its own
    # slot (work records + table slab), so the thinly filled last wave of one batch's curve kernel (1,000,000 items are
    # 13.2 waves of the persistent grid) overlaps the next batch's kernels instead of idling most of the SMs.
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    if os.environ.get("SV_BENCH_ONE_STREAM"):
        streams[1] = streams[0]
    stream = streams[0]
    sh = stream.cuda_stream

    # two resident batches per rank.  Triples come from the reference signer (the bytes the reference arm verifies:
    # rank 0's first batch is seed BENCH_SEED); where oracle/_ref did not travel, the engine's own device-side signer
    # (k_synth) stands in and `data` says so.
    batches = []
    host_batches = []
    try:
        ref_lib, ref_kind = load_ref()
    except Exception:
        ref_lib, ref_kind = None, "unavailable"
    data_note = "synthetic"
    for b in range(2):
        if ref_kind == "reference":
            hm, hk, hs = make_reference_batch(ref_lib, BENCH_SEED + 1000 * rank + b, n, host_threads())
            msg, key, sig = (torch.from_numpy(a).to(dev) for a in (hm, hk, hs))
            bad = torch.arange(0, n, 10, device=dev)
            host_batches.append((hm, hk, hs))
        else:
            data_note = "synthetic (oracle/_ref absent: triples from the engine's device-side signer k_synth)"
            msg = torch.empty((n, 32), dtype=torch.uint8, device=dev)
            key = torch.empty((n, 33), dtype=torch.uint8, device=dev)
            sig = torch.empty((n, 64), dtype=torch.uint8, device=dev)
            eng.synth_device(kind, 0x9E3779B97F4A7C15 + 1000 * rank + b, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr(), sh)
            eng.sync(sh)
            bad = corrupt_on_device(torch, msg, key, sig)
        batches.append((msg, key, sig, bad))
    # Output sets (verdict bytes, bitmap, gathered bitmap), NOUT deep.  Two steps may be computing, and with N > 1 the
    # gather of a finished step must not hold up the launch streams: the NCCL kernel only gets an SM when a CTA of the
    # persistent curve kernel retires, so a launch stream that waited for "its" gather would idle through most of the other
    # stream's batch (measured at N = 2: 49.9 M/s per GPU instead of 53).  The gather therefore runs on a stream of its own
    # behind an event, and a launch stream only waits for the gather that read its output set NOUT steps earlier.
    NOUT = 4
    verdicts = [torch.zeros(n, dtype=torch.uint8, device=dev) for _ in range(NOUT)]
    bitmaps = [torch.zeros((n + 31) // 32, dtype=torch.int32, device=dev) for _ in range(NOUT)]
    gathereds = [torch.zeros(world * bitmaps[0].numel(), dtype=torch.int32, device=dev) if world > 1 else None for _ in range(NOUT)]
    comm = torch.cuda.Stream(device=dev) if world > 1 else None
    gathered_ev = [None] * NOUT
    verdict, bitmap = verdicts[0], bitmaps[0]
    torch.cuda.synchronize()

    def step(i, single=False):
        j = 0 if single else (i & 1)
        o = 0 if single else (i % NOUT)
        st = streams[j]
        msg, key, sig, _ = batches[i & 1]
        if world > 1 and gathered_ev[o] is not None:
            st.wait_event(gathered_ev[o])  # bitmaps[o] is about to be overwritten
        eng.verify_device(kind, msg.data_ptr(), key.data_ptr(), sig.data_ptr(), n, verdicts[o].data_ptr(),
                          bitmaps[o].data_ptr(), st.cuda_stream)
        if world > 1:  # the only exchange step of the path: gather the verdict bitmap over NVLink
            ev = torch.cuda.Event()
            ev.record(st)
            comm.wait_event(ev)
            with torch.cuda.stream(comm):
                dist.all_gather_into_tensor(gathereds[o], bitmaps[o])
            gathered_ev[o] = torch.cuda.Event()
            gathered_ev[o].record(comm)

    def join_streams():
        """make streams[0] wait for everything queued on streams[1] and on the gather stream"""
        for other in ([streams[1]] if streams[1] is not streams[0] else []) + ([comm] if comm is not None else []):
            ev = torch.cuda.Event()
            ev.record(other)
            streams[0].wait_event(ev)

    def fork_streams():
        """nothing on streams[1] may start before this point of streams[0]"""
        if streams[1] is not streams[0]:
            ev = torch.cuda.Event()
            ev.record(streams[0])
            streams[1].wait_event(ev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step(i)
    barrier()
    launches0 = eng.info()["launches"]
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    main_ms, prep_ms = [], []
    barrier()
    e0.record(stream)
    fork_streams()
    for i in range(args.steps):
        step(i)
    join_streams()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    launches = eng.info()["launches"] - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, verdicts[(args.steps - 1) % NOUT], bitmaps[(args.steps - 1) % NOUT],
                     gathereds[(args.steps - 1) % NOUT])
    # the same K steps again with the clock sampler still running (reported separately as `sustained`)
    quick = bool(os.environ.get("SV_BENCH_QUICK"))  # variant sweeps (tools/variants.py): only the K timed steps + kernel timing
    sus_steps = args.steps
    s0 = torch.cuda.Event(enable_timing=True)
    s1 = torch.cuda.Event(enable_timing=True)
    barrier()
    s0.record(stream)
    fork_streams()
    for i in range(sus_steps):
        step(i)
    join_streams()
    s1.record(stream)
    barrier()
    sus_ms = s0.elapsed_time(s1)
    # per-kernel device time (events recorded by the engine on the launch stream), a few extra steps
    for i in range(3):
        step(i, single=True)
        eng.sync(sh)
        p, m = eng.last_timing()
        prep_ms.append(p)
        main_ms.append(m)
    # verdicts of the last step, checked by construction: valid everywhere except the corrupted indices
    step(args.steps - 1 if args.steps else 0, single=True)
    eng.sync(sh)
    torch.cuda.synchronize()
    bad = batches[(args.steps - 1) & 1 if args.steps else 0][3]
    expect = torch.ones(n, dtype=torch.uint8, device=dev)
    expect[bad] = 0
    construct_ok = bool(torch.equal(verdict, expect))
    bits = (bitmap.view(torch.int32).cpu().numpy().view(np.uint32)[:, None] >> np.arange(32, dtype=np.uint32)) & 1
    bitmap_ok = bool(np.array_equal(bits.reshape(-1)[:n].astype(np.uint8), verdict.cpu().numpy()))

    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms_max = float(t_ms.item())
    value = world * n * args.steps / (ms_max * 1e-3)
    t_sus = torch.tensor([sus_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_sus, op=dist.ReduceOp.MAX)
    sustained = {"steps": sus_steps, "seconds": float(t_sus.item()) * 1e-3, "value": world * n * sus_steps / (float(t_sus.item()) * 1e-3),
                 "unit": "verifies/s"}

    # ---- e2e: host pinned buffers through sv_verify_host (H2D + kernels + D2H inside the timed region) ----
    msg, key, sig, _ = batches[0]
    h_msg = eng.host_alloc(n * 32)
    h_key = eng.host_alloc(n * 33)
    h_sig = eng.host_alloc(n * 64)
    h_out = eng.host_alloc(n)
    h_msg[:] = msg.cpu().numpy().reshape(-1)
    h_key[:] = key.cpu().numpy().reshape(-1)
    h_sig[:] = sig.cpu().numpy().reshape(-1)
    e2e_steps = 3 if quick else args.steps
    for _ in range(2):
        rc = eng.lib.sv_verify_host(eng._ctx, kind, h_msg.ctypes.data, h_key.ctypes.data, h_sig.ctypes.data, n, h_out.ctypes.data)
        assert rc == 0
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        rc = eng.lib.sv_verify_host(eng._ctx, kind, h_msg.ctypes.data, h_key.ctypes.data, h_sig.ctypes.data, n, h_out.ctypes.data)
        assert rc == 0
    dt = time.perf_counter() - t0
    t_e = torch.tensor([dt], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e, op=dist.ReduceOp.MAX)
    e2e_value = world * n * e2e_steps / float(t_e.item())
    e2e_expect = (torch.ones(n, dtype=torch.uint8).index_fill_(0, batches[0][3].cpu(), 0)).numpy()
    e2e_matches = bool(np.array_equal(np.asarray(h_out), e2e_expect))
    # The synchronous call above drains the GPU at every return (the thin last wave of a batch has nothing to overlap with).
    # A host that keeps two calls in flight — two threads, each with its own context, as two CLN daemons sharing the GPU
    # would — gets that overlap back.  Both numbers are reported: `e2e.value` is the two-caller one (what the GPU sustains
    # when its host keeps it fed through the same synchronous C ABI; every step's H2D and D2H inside the timed region),
    # `e2e.single_caller` the strictly sequential loop.
    e2e_two = None
    if not quick:
        import threading
        eng2 = L.SigVerifier(local)
        h_out2 = eng2.host_alloc(n)
        half = max(1, e2e_steps // 2)

        def caller(e, out, k):
            torch.cuda.set_device(local)  # a new host thread starts on device 0: without this, every call on rank r > 0 switches devices
            for _ in range(k):
                r = e.lib.sv_verify_host(e._ctx, kind, h_msg.ctypes.data, h_key.ctypes.data, h_sig.ctypes.data, n, out.ctypes.data)
                assert r == 0
        caller(eng2, h_out2, 2)
        barrier()
        th = [threading.Thread(target=caller, args=(eng, h_out, half)), threading.Thread(target=caller, args=(eng2, h_out2, half))]
        t0 = time.perf_counter()
        for t in th:
            t.start()
        for t in th:
            t.join()
        dt2 = time.perf_counter() - t0
        t_2 = torch.tensor([dt2], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t_2, op=dist.ReduceOp.MAX)
        dt2 = float(t_2.item())
        same2 = bool(np.array_equal(np.asarray(h_out2), e2e_expect)) and bool(np.array_equal(np.asarray(h_out), e2e_expect))
        e2e_two = {"value": world * 2 * half * n / dt2, "steps": 2 * half, "seconds": dt2, "verdicts_as_constructed": same2}
        e2e_matches = e2e_matches and same2
        eng2.close()
    clocks = sampler.stop() if rank == 0 else None  # sampled across the timed regions

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel (curve side), measured live ----
    peak_imad = eng.probe(0)  # IMAD.WIDE.U32 multiply-accumulates/s on this device, measured now
    main_avg = sum(main_ms) / len(main_ms)
    prep_avg = sum(prep_ms) / len(prep_ms)
    achieved = n * IMAD_PER_VERIFY / (main_avg * 1e-3)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_ach = n * BYTES_PER_VERIFY / (main_avg * 1e-3) / 1e9

    # ---- CPU baseline on a bounded sample of THIS workload, verdicts compared bit for bit ----
    cpu = None
    try:
        if world > 1:
            raise RuntimeError("reported at N=1 only")
        if quick:
            raise RuntimeError("SV_BENCH_QUICK")
        lib, ckind = load_ref()
        threads = host_threads()
        m = int(min(n, max(20_000, 30_000 * threads)))
        hm = np.ascontiguousarray(np.asarray(h_msg).reshape(n, 32)[:m])
        hk = np.ascontiguousarray(np.asarray(h_key).reshape(n, 33)[:m])
        hs = np.ascontiguousarray(np.asarray(h_sig).reshape(n, 64)[:m])
        cpu_verify(lib, ckind, hm[:2000], hk[:2000], hs[:2000], threads)
        t0 = time.perf_counter()
        passes = 0
        while True:
            want = cpu_verify(lib, ckind, hm, hk, hs, threads)
            passes += 1
            if time.perf_counter() - t0 > 8.0 or passes >= 20:
                break
        cdt = time.perf_counter() - t0
        same = bool(np.array_equal(want, np.asarray(h_out)[:m]))
        t1 = time.perf_counter()
        cpu_verify(lib, ckind, hm[:20000], hk[:20000], hs[:20000], 1)
        one = 20000 / (time.perf_counter() - t1)
        cpu = dict({"value": m * passes / cdt, "unit": "verifies/s", "kind": ckind,
                    "sample": f"first {m} triples of the bench batch x {passes} passes, {threads} threads; 1 thread: {one:.0f}/s",
                    "verdicts_bit_exact_vs_gpu": same}, **cores_note())
    except Exception as ex:  # the baseline is a reported number, never a dependency of the product path
        cpu = {"value": None, "unit": "verifies/s", "cores": 0, "kind": "unavailable", "sample": repr(ex),
               "verdicts_bit_exact_vs_gpu": None}

    info = eng.info()
    line = {
        "metric": METRIC, "value": value, "unit": "verifies/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_max / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32 (8x32-bit limbs, IMAD.WIDE.U32 carry chains)", "data": data_note,
        "config": bench_config(world),
        "engine": {"main_grid": info["main_grid"], "main_block": info["main_block"], "main_regs": info["main_regs"],
                   "launch_streams": 1 if streams[1] is streams[0] else 2, "l2_persist_bytes": info.get("l2_persist_bytes"), "l2_max_persist_bytes": info.get("l2_max_persist_bytes")},
        "e2e": {"value": e2e_two["value"] if e2e_two else e2e_value, "unit": "verifies/s",
                "h2d_bytes_per_step": n * 129, "d2h_bytes_per_step": n,
                "steps": e2e_two["steps"] if e2e_two else e2e_steps, "seconds": e2e_two["seconds"] if e2e_two else float(t_e.item()),
                "callers_per_gpu": 2 if e2e_two else 1,
                "how": "sv_verify_host (synchronous C ABI) on pinned host buffers; per step 129 MB H2D + kernels + 1 MB D2H, all inside the "
                       "timed region" + ("; two host threads per GPU, each with its own sv_ctx, keep two calls in flight" if e2e_two else ""),
                "single_caller": {"value": e2e_value, "steps": e2e_steps, "seconds": float(t_e.item())},
                "verdicts_as_constructed": e2e_matches},
        "sustained": sustained,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "integer (IMAD.WIDE.U32 issue)", "achieved": achieved / 1e9, "peak": peak_imad / 1e9,
                     "unit": "GIMAD/s", "frac": achieved / peak_imad,
                     "traffic": NCU_DRAM_BYTES_PER_1M_LAUNCH if n == 1_000_000 else None, "traffic_unit": "bytes/launch (ncu, profiles/r2_k_main_nosqrt_ncu_raw.csv)",
                     "kernel": "k_main<3> + k_final_ecdsa33 (compressed keys, no square root)", "kernel_ms": main_avg, "prep_kernel_ms": prep_avg,
                     "algorithmic_imad_per_verify": IMAD_PER_VERIFY,
                     "executed_imad_per_verify": EXECUTED_IMAD_PER_VERIFY if os.environ.get("SV_NOSQRT", "1") != "0" else IMAD_PER_VERIFY,
                     "pipe_frac": n * (EXECUTED_IMAD_PER_VERIFY if os.environ.get("SV_NOSQRT", "1") != "0" else IMAD_PER_VERIFY) / (main_avg * 1e-3) / peak_imad,
                     "note": "frac = SURVEY 8(d)'s algorithmic 125,440 IMAD/verify over the kernel time; pipe_frac = multiplies actually issued (the shipped flow skips the key's square root)",
                     "peak_source": "measured live: engine probe k_probe_imad_wide (independent IMAD.WIDE.U32 chains)"},
        "roofline_hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s",
                         "frac": hbm_ach / hbm_peak, "traffic": NCU_DRAM_BYTES_PER_1M_LAUNCH if n == 1_000_000 else None,
                         "achieved_incl_scratch": (NCU_DRAM_BYTES_PER_1M_LAUNCH / (main_avg * 1e-3) / 1e9) if n == 1_000_000 else None,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks else "fallback 6650",
                         "note": "algorithmic bytes only (129.125 B/verify); the path is integer-compute bound"},
        "cpu_baseline": cpu,
        "checks": {"verdicts_as_constructed": construct_ok, "bitmap_matches_bytes": bitmap_ok},
    }
    # a throughput number for wrong verdicts is worthless: a failed check nulls the headline and fails the run
    failed = [k for k, ok in (("verdicts_as_constructed", construct_ok), ("bitmap_matches_bytes", bitmap_ok),
                              ("e2e_verdicts_as_constructed", e2e_matches),
                              ("verdicts_bit_exact_vs_reference", cpu.get("verdicts_bit_exact_vs_gpu") is not False)) if not ok]
    if world == 1 and cpu.get("kind") == "unavailable" and not quick:
        failed.append("cpu_baseline_unavailable: " + str(cpu.get("sample")))
    if failed:
        line["value"] = None
        line["e2e"]["value"] = None
        line["failed_checks"] = failed
    print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 1 if failed else 0


# --------------------------------------------------------------------------------------------------
# the other BASELINE configs (parity cases first, measured here so that they are driver-visible): --config c3|c4|c5
# --------------------------------------------------------------------------------------------------
def _events_ms(torch, fn, stream, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_c3(args):
    """configs[2]: 1M mixed ECDSA + BIP-340, interleaved by a seeded shuffle with a 1-byte kind tag per item, through
    sv_verify_mixed_device / _host; every verdict compared with the reference."""
    import torch
    import lightning_b200 as L
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    eng = L.SigVerifier(0)
    lib, kind = load_ref()
    assert kind == "reference", "config c3 needs oracle/_ref (the reference signer)"
    n, half, threads = BATCH, BATCH // 2, host_threads()
    p8 = ctypes.POINTER(ctypes.c_uint8)
    em, ek, es = make_reference_batch(lib, BENCH_SEED + 3, half, threads)
    sm, sx, ss = np.zeros((half, 32), np.uint8), np.zeros((half, 32), np.uint8), np.zeros((half, 64), np.uint8)
    lib.ref_make_schnorr_batch(ctypes.c_uint64(BENCH_SEED + 4), ctypes.c_size_t(half), sm.ctypes.data_as(p8), sx.ctypes.data_as(p8),
                               ss.ctypes.data_as(p8), int(threads))
    rng = np.random.default_rng(BENCH_SEED)
    perm = rng.permutation(n)
    kinds = np.zeros(n, np.uint8)
    msg, key, sig = np.zeros((n, 32), np.uint8), np.zeros((n, 64), np.uint8), np.zeros((n, 64), np.uint8)
    pe, ps = perm[:half], perm[half:]
    kinds[ps] = 2
    msg[pe], msg[ps] = em, sm
    key[pe, :33], key[ps, :32] = ek, sx
    sig[pe], sig[ps] = es, ss
    d = [torch.from_numpy(a).to(dev) for a in (kinds, msg, key, sig)]
    out = torch.zeros(n, dtype=torch.uint8, device=dev)
    st = torch.cuda.Stream(device=dev)
    call = lambda: eng._check(eng.lib.sv_verify_mixed_device(eng._ctx, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(),
                                                             n, out.data_ptr(), st.cuda_stream), "sv_verify_mixed_device")
    for _ in range(args.warmup):
        call()
    launches0 = eng.info()["launches"]
    ms = _events_ms(torch, call, st, args.steps)
    launches = eng.info()["launches"] - launches0
    got = out.cpu().numpy()
    h = [eng.host_alloc(a.nbytes) for a in (kinds, msg, key, sig)]
    for hb, a in zip(h, (kinds, msg, key, sig)):
        hb[:] = a.reshape(-1)
    hout = eng.host_alloc(n)
    hcall = lambda: eng._check(eng.lib.sv_verify_mixed_host(eng._ctx, h[0].ctypes.data, h[1].ctypes.data, h[2].ctypes.data, h[3].ctypes.data, n,
                                                            hout.ctypes.data), "sv_verify_mixed_host")
    hcall()
    e2e_steps = max(3, min(args.steps, 20))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        hcall()
    e2e = n * e2e_steps / (time.perf_counter() - t0)
    # reference verdicts for ALL items (the two halves on all host threads), timed as the CPU baseline
    t0 = time.perf_counter()
    want = np.zeros(n, np.uint8)
    want[pe] = cpu_verify(lib, "reference", em, ek, es, threads)
    ws = np.zeros(half, np.uint8)
    lib.ref_schnorr_verify_batch(sm.ctypes.data_as(p8), sx.ctypes.data_as(p8), ss.ctypes.data_as(p8), ctypes.c_size_t(half), ws.ctypes.data_as(p8), int(threads))
    want[ps] = ws
    cpu_s = time.perf_counter() - t0
    same = bool(np.array_equal(got, want)) and bool(np.array_equal(np.asarray(hout), want))
    peak = eng.probe(0)
    work = half * IMAD_PER_VERIFY + half * 2230 * 64  # SURVEY 8(d): ECDSA33 1,960 fmul, BIP-340 2,230 fmul-equivalents
    line = {"metric": METRIC, "value": n / (ms * 1e-3), "unit": "verifies/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs", "data": "synthetic",
            "config": {"workload": "1M mixed: 500k ECDSA (33-byte keys) + 500k BIP-340, reference-signed, 10% corrupted per kind, interleaved "
                                   "by a seeded shuffle, 1-byte kind tag per item, keys in 64-byte slots [BASELINE configs[2]]",
                       "batch_per_gpu": n, "l2": "161 MB of inputs + index lists + staging per step exceed the 126 MB L2"},
            "e2e": {"value": e2e, "unit": "verifies/s", "h2d_bytes_per_step": n * 161, "d2h_bytes_per_step": n, "steps": e2e_steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "integer (IMAD.WIDE.U32 issue)", "achieved": work / (ms * 1e-3) / 1e9, "peak": peak / 1e9, "unit": "GIMAD/s",
                         "frac": work / (ms * 1e-3) / peak, "traffic": None,
                         "note": "whole step (split + both kinds' kernels + scatter) against the live IMAD.WIDE probe"},
            "cpu_baseline": dict({"value": n / cpu_s, "unit": "verifies/s", "kind": "reference", "sample": "all 1M items, both kinds",
                                  "verdicts_bit_exact_vs_gpu": same}, **cores_note()),
            "checks": {"valid_fraction": float(want.mean())}}
    if not same:
        line["value"] = None
        line["failed_checks"] = ["verdicts_bit_exact_vs_reference"]
    print(json.dumps(line))
    return 0 if same else 1


def load_gossip_store():
    """tests/golden/routing_gossip_store (the reference's tests/data fixture; format common/gossip_store.h:15-51):
    -> list of raw wire messages of types 256/257/258"""
    path = os.path.join(ROOT, "tests", "golden", "routing_gossip_store")
    data = open(path, "rb").read()
    pos, msgs = 1, []
    while pos + 12 <= len(data):
        ln = int.from_bytes(data[pos + 2:pos + 4], "big")
        m = data[pos + 12:pos + 12 + ln]
        pos += 12 + ln
        if len(m) >= 2 and m[0] == 1 and m[1] in (0, 1, 2):
            msgs.append(m)
    return msgs


def run_c4(args):
    """configs[3]: gossip-sync replay — the WHOLE routing_gossip_store (11,796 channel_announcements, 2,175
    node_announcements, 9,703 channel_updates = 59,062 signatures) tiled x7, >= 1% of the messages bit-flipped, raw wire
    bytes handed to sv_verify_gossip_host (the device slices, hashes and verifies); per-message status compared with
    CLN's own gossipd/sigcheck.c (oracle/_ref/libcln_ref.so)."""
    import struct
    import lightning_b200 as L
    from concurrent.futures import ThreadPoolExecutor
    eng = L.SigVerifier(0)
    eng.set_profiling(True)
    if os.environ.get("SV_BENCH_NODEDUP"):  # measurement aid: every signature decodes its own key
        eng.set_dedup(False)
    base = load_gossip_store()
    chans = {}
    for m in base:
        if m[1] == 0:
            flen = struct.unpack(">H", m[258:260])[0]
            p = 260 + flen + 32
            chans[m[p:p + 8]] = (m[p + 8:p + 41], m[p + 41:p + 74])
    msgs = [bytearray(m) for m in base * 7]
    rng = np.random.default_rng(BENCH_SEED)
    flipped = rng.choice(len(msgs), size=len(msgs) // 80, replace=False)
    for mi in flipped:
        pos = int(rng.integers(2, len(msgs[mi])))
        msgs[mi][pos] ^= 1 << int(rng.integers(0, 8))
    msgs = [bytes(m) for m in msgs]
    signers = np.zeros((len(msgs), 33), np.uint8)
    for i, m in enumerate(msgs):
        if m[1] == 2 and len(m) >= 112:  # signer by direction bit, as gossipd/gossmap_manage.c:920-922 selects it
            ends = chans.get(bytes(m[98:106]))
            if ends:
                signers[i] = np.frombuffer(ends[m[111] & 1], dtype=np.uint8)
    n_msgs = len(msgs)
    sigs = sum(4 if m[1] == 0 else 1 for m in msgs)
    lens = np.array([len(m) for m in msgs], dtype=np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64)
    blob = np.frombuffer(b"".join(msgs), dtype=np.uint8)
    hb, ho, hl, hs = (eng.host_alloc(a.nbytes) for a in (blob, offs, lens, signers))
    hb[:] = blob
    ho[:] = offs.view(np.uint8)
    hl[:] = lens.view(np.uint8)
    hs[:] = signers.reshape(-1)
    status = np.zeros(n_msgs, np.int32)
    call = lambda: eng._check(eng.lib.sv_verify_gossip_host(eng._ctx, hb.ctypes.data, blob.size, ho.ctypes.data, hl.ctypes.data, n_msgs,
                                                            hs.ctypes.data, status.ctypes.data), "sv_verify_gossip_host")
    for _ in range(max(args.warmup, 2)):
        call()
    launches0 = eng.info()["launches"]
    steps = max(args.steps, 5)
    t0 = time.perf_counter()
    kern = []
    for _ in range(steps):
        call()
        kern.append(sum(eng.last_timing()))
    dt = (time.perf_counter() - t0) / steps
    launches = (eng.info()["launches"] - launches0) // steps
    kern_ms = sum(kern) / len(kern)
    # reference: CLN's own sigcheck on every message (thread pool: ctypes releases the GIL)
    from tests import util as tutil
    cln = tutil.load_cln()
    cln.cln_sigcheck_channel_announcement(msgs[0], ctypes.c_size_t(len(msgs[0])))  # one-time setup before the threads start
    p8 = ctypes.POINTER(ctypes.c_uint8)

    def ref_one(i):
        m = msgs[i]
        if m[1] == 0:
            return cln.cln_sigcheck_channel_announcement(m, ctypes.c_size_t(len(m)))
        if m[1] == 1:
            return cln.cln_sigcheck_node_announcement(m, ctypes.c_size_t(len(m)))
        return cln.cln_sigcheck_channel_update(m, ctypes.c_size_t(len(m)), signers[i].ctypes.data_as(p8))
    t0 = time.perf_counter()
    want = np.array([ref_one(i) for i in range(n_msgs)], np.int32)  # the harness keeps one tal context: single thread
    cpu_s = time.perf_counter() - t0
    same = bool(np.array_equal(status, want))
    peak = eng.probe(0)
    line = {"metric": METRIC, "value": sigs / (kern_ms * 1e-3), "unit": "verifies/s", "n_gpus": 1, "steps": steps, "warmup": max(args.warmup, 2),
            "ms_per_step": kern_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs", "data": "real mainnet gossip (reference fixture), tiled x7, 1.25% of the messages bit-flipped",
            "config": {"workload": "gossip-sync replay: whole tests/data/routing_gossip_store x7 = 82,572 channel_announcements (4 sigs each) + 15,225 "
                                   "node_announcements + 67,921 channel_updates; device-side slicing + SHA-256d + verification, per-message status "
                                   "[BASELINE configs[3]]",
                       "messages": n_msgs, "signatures": sigs, "blob_bytes": int(blob.size)},
            "e2e": {"value": sigs / dt, "unit": "verifies/s", "messages_per_s": n_msgs / dt, "h2d_bytes_per_step": int(blob.size + 12 * n_msgs + 4 * n_msgs + 33 * n_msgs),
                    "d2h_bytes_per_step": 4 * n_msgs, "steps": steps},
            "gpu_launches": int(launches),
            "roofline": {"bound": "integer (IMAD.WIDE.U32 issue)", "achieved": sigs * IMAD_PER_VERIFY / (kern_ms * 1e-3) / 1e9, "peak": peak / 1e9,
                         "unit": "GIMAD/s", "frac": sigs * IMAD_PER_VERIFY / (kern_ms * 1e-3) / peak, "traffic": None,
                         "note": "scalar-side + curve-side kernels (CUDA events); slicing, hashing and status kernels are in e2e"},
            "cpu_baseline": dict({"value": sigs / cpu_s, "unit": "verifies/s", "kind": "reference", "cores": 1,
                                  "sample": "every message through CLN's own sigcheck_* (gossipd/sigcheck.c, unmodified), one thread as gossipd runs it",
                                  "status_bit_exact_vs_gpu": same}),
            "checks": {"status_ok": int((want == 0).sum()), "status_bad_sig": int((want > 0).sum()), "status_malformed": int((want < 0).sum())}}
    if not same:
        bad = np.nonzero(status != want)[0]
        line["value"] = None
        line["failed_checks"] = [f"status differs from gossipd at {bad.size} messages, first {int(bad[0])}: got {int(status[bad[0]])} want {int(want[bad[0]])}"]
    print(json.dumps(line))
    return 0 if same else 1


def run_c5(args):
    """configs[4]: 100M-signature synthetic batch over 8 B200s = 12.5M per GPU (weak scaling: N GPUs hold N x 12.5M).  Rank 0
    holds ALL triples in pinned host memory (the 1M reference-signed set replicated, each replica with its own deterministic
    corruption mask); inside the timed region it pushes every rank's share to the device chunk by chunk and scatters it
    with NCCL send/recv over NVLink, every rank verifies its chunks as they arrive (two launch streams), and the verdict
    bitmaps are gathered back to rank 0 and copied to the host."""
    import torch
    import lightning_b200 as L
    world, rank, local = env_int("WORLD_SIZE", 1), env_int("RANK", 0), env_int("LOCAL_RANK", 0)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "WARN"):
        os.environ.pop("NCCL_DEBUG")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    if world > 1:
        os.environ.setdefault("SV_MAIN_GRID_RESERVE", "2")  # room for NCCL's send/recv kernels beside the persistent curve grid
    eng = L.SigVerifier(local)
    per_rank = int(os.environ.get("SV_C5_PER_RANK", 12_500_000))
    nchunk = int(os.environ.get("SV_C5_CHUNKS", 25))  # 12.5M = 2^5 x 5^8: 25 chunks of 500,000 keep every chunk a multiple of 32
    c = per_rank // nchunk
    assert c * nchunk == per_rank and c % 32 == 0
    rec = 129 * c  # packed chunk: [msg c x 32 | key c x 33 | sig c x 64]
    total = per_rank * world
    pool = expect = None
    if rank == 0:
        lib, kind = load_ref()
        assert kind == "reference"
        bm, bk, bs = make_reference_batch(lib, BENCH_SEED, BATCH, host_threads())
        base_ok = np.ones(BATCH, np.uint8)
        base_ok[::10] = 0
        pool = torch.empty(total * 129, dtype=torch.uint8, pin_memory=True)
        pv = pool.numpy()
        expect = np.zeros(total, np.uint8)
        for g in range(world * nchunk):  # global chunk g = (rank g // nchunk, chunk g % nchunk)
            idx = (np.arange(c, dtype=np.int64) + g * c) % BATCH
            m = bm[idx].copy()
            ok = base_ok[idx].copy()
            hit = np.nonzero((idx * 2654435761 + g * 40503) % 1009 == 0)[0]  # this replica's corruption mask
            m[hit, g % 32] ^= 1 << (g % 8)
            ok[hit] = 0
            o = g * rec
            pv[o:o + 32 * c] = m.reshape(-1)
            pv[o + 32 * c:o + 65 * c] = bk[idx].reshape(-1)
            pv[o + 65 * c:o + rec] = bs[idx].reshape(-1)
            expect[g * c:(g + 1) * c] = ok
    inbuf = [torch.empty(rec, dtype=torch.uint8, device=dev) for _ in range(nchunk)]
    NST = 4  # staging ring on rank 0: the H2D copy of one peer's chunk runs while the previous one is on the wire
    stage = [torch.empty(rec, dtype=torch.uint8, device=dev) for _ in range(NST)] if (rank == 0 and world > 1) else None
    verdict = torch.zeros(per_rank, dtype=torch.uint8, device=dev)
    bitmap = torch.zeros(per_rank // 32, dtype=torch.int32, device=dev)
    gathered = torch.zeros(world * bitmap.numel(), dtype=torch.int32, device=dev) if world > 1 else bitmap
    host_bits = torch.empty(world * bitmap.numel(), dtype=torch.int32, pin_memory=True) if rank == 0 else None
    streams = [torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)]
    comm = torch.cuda.Stream(device=dev)   # NCCL send / recv / all_gather
    h2d = torch.cuda.Stream(device=dev)    # rank 0: host -> device copies (copy engine), one step ahead of the sends
    state = {"slot": 0, "sent": [None] * NST, "pass_done": None}

    def one_pass():
        evs = []
        if state["pass_done"] is not None:
            h2d.wait_event(state["pass_done"])  # the chunk buffers are reused: the previous pass must be through with them
        for k in range(nchunk):
            if rank == 0:
                with torch.cuda.stream(h2d):
                    inbuf[k].copy_(pool[(0 * nchunk + k) * rec:(0 * nchunk + k + 1) * rec], non_blocking=True)
                    ev = torch.cuda.Event()
                    ev.record(h2d)
                for r in range(1, world):
                    sl = state["slot"]
                    sb = stage[sl]
                    g = r * nchunk + k
                    with torch.cuda.stream(h2d):
                        if state["sent"][sl] is not None:
                            h2d.wait_event(state["sent"][sl])
                        sb.copy_(pool[g * rec:(g + 1) * rec], non_blocking=True)
                        staged = torch.cuda.Event()
                        staged.record(h2d)
                    comm.wait_event(staged)
                    with torch.cuda.stream(comm):
                        dist.send(sb, dst=r)
                        se = torch.cuda.Event()
                        se.record(comm)
                    state["sent"][sl] = se
                    state["slot"] = (sl + 1) % NST
            else:
                with torch.cuda.stream(comm):
                    dist.recv(inbuf[k], src=0)
                    ev = torch.cuda.Event()
                    ev.record(comm)
            st = streams[k & 1]
            st.wait_event(ev)
            b = inbuf[k]
            eng.verify_device(L.KIND_ECDSA33, b.data_ptr(), b.data_ptr() + 32 * c, b.data_ptr() + 65 * c, c,
                              verdict.data_ptr() + k * c, bitmap.data_ptr() + 4 * (k * c // 32), st.cuda_stream)
            e2 = torch.cuda.Event()
            e2.record(st)
            evs.append(e2)
        for e2 in evs:
            comm.wait_event(e2)
        with torch.cuda.stream(comm):
            if world > 1:
                dist.all_gather_into_tensor(gathered, bitmap)
            if rank == 0:
                host_bits.copy_(gathered, non_blocking=True)
            state["pass_done"] = torch.cuda.Event()
            state["pass_done"].record(comm)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    for _ in range(max(1, min(args.warmup, 2))):
        one_pass()
    barrier()
    steps = max(1, min(args.steps, 5))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = eng.info()["launches"]
    barrier()
    e0.record(comm)
    for _ in range(steps):
        one_pass()
    e1.record(comm)
    barrier()
    ms = e0.elapsed_time(e1) / steps
    t_ms = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_ms, op=dist.ReduceOp.MAX)
    ms = float(t_ms.item())
    launches = (eng.info()["launches"] - launches0) // steps
    rc = 0
    if rank == 0:
        bits = (host_bits.numpy().view(np.uint32)[:, None] >> np.arange(32, dtype=np.uint32)) & 1
        got = bits.reshape(-1)[:total].astype(np.uint8)
        same = bool(np.array_equal(got, expect))
        line = {"metric": METRIC, "value": total / (ms * 1e-3), "unit": "verifies/s", "n_gpus": world, "steps": steps, "warmup": max(1, min(args.warmup, 2)),
                "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs", "data": "synthetic",
                "config": {"workload": f"{total} ECDSA triples = {per_rank} per GPU [BASELINE configs[4]: 100M over 8 GPUs]: the 1M reference-signed set "
                                       "replicated with a per-replica corruption mask, ALL held by rank 0 in pinned host memory; H2D + NCCL "
                                       "send/recv scatter of 129 B/triple, verification and the all_gather + D2H of the 1-bit verdicts are all inside the timed region",
                           "per_gpu": per_rank, "chunks_per_gpu": nchunk, "parallelism": f"dp{world}: NCCL scatter of triples from rank 0, gather of the verdict bitmap"},
                "e2e": {"value": total / (ms * 1e-3), "unit": "verifies/s", "h2d_bytes_per_step": total * 129, "d2h_bytes_per_step": total // 8,
                        "note": "this config IS end to end: inputs start in rank 0's host memory, verdict bits end there"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "host feed (one PCIe link carries every rank's triples)", "achieved": total * 129 / (ms * 1e-3) / 1e9, "peak": None,
                             "unit": "GB/s", "frac": None, "traffic": None},
                "checks": {"verdict_bits_as_constructed": same, "valid_fraction": float(expect.mean())}}
        if not same:
            line["value"] = None
            line["failed_checks"] = ["verdict_bits_as_constructed"]
            rc = 1
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=240)  # ~5.2 s timed at ~21.6 ms/step
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (engine arm, config c2)")
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--config", default="c2", choices=["c2", "c3", "c4", "c5"],
                    help="BASELINE config: c2 (default, the headline: 1M ECDSA), c3 mixed ECDSA+BIP-340, c4 gossip replay, c5 100M over N GPUs with NCCL scatter")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "engine" or args.config != "c2" or args.steps < 1):
        ap.error("--dump-outputs is for the engine arm of config c2, with at least one timed step")
    if args.impl == "engine" and args.config == "c3":
        return run_c3(args)
    if args.impl == "engine" and args.config == "c4":
        return run_c4(args)
    if args.impl == "engine" and args.config == "c5":
        return run_c5(args)
    args.warmup = max(args.warmup, 3) if args.impl == "engine" else max(args.warmup, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_engine(args)


if __name__ == "__main__":
    sys.exit(main())
