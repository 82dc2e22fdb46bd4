"""GPU parity: the CUDA engine (through the C ABI) vs the unmodified reference on identical inputs."""
import ctypes

import numpy as np
import pytest

from tests import util

pytestmark = pytest.mark.gpu

K33, KXY, KSCH = 0, 1, 2


@pytest.fixture(scope="module")
def workload(ref):
    w = util.make_signed(6000, seed=20260922)
    return util.corrupt(w, every=7)


def _cmp(engine, ref, kind, msg, key, sig):
    got = engine.verify(kind, msg, key, sig)
    want = util.ref_verify(ref, kind, msg, key, sig)
    bad = np.nonzero(got != want)[0]
    assert bad.size == 0, f"kind {kind}: {bad.size} verdict mismatches, first at {bad[:5]}, want {want[bad[:5]]}"
    return want


def test_ecdsa33_random_and_corrupted(engine, ref, workload):
    want = _cmp(engine, ref, K33, workload["msg"], workload["pub33"], workload["sig"])
    assert 0 < want.sum() < want.size


def test_ecdsa_xy_random_and_corrupted(engine, ref, workload):
    want = _cmp(engine, ref, KXY, workload["msg"], workload["pubxy"], workload["sig"])
    assert 0 < want.sum() < want.size


def test_schnorr_random_and_corrupted(engine, ref, workload):
    want = _cmp(engine, ref, KSCH, workload["msg"], workload["xonly"], workload["ssig"])
    assert 0 < want.sum() < want.size


def test_ragged_sizes(engine, ref, workload):
    """batch sizes around the prep batch (16), the warp (32) and the CTA (128/256/512), every kind; lanes past
    the end of a batch must not disturb live records (regression: idle lanes once aliased record 0, which the
    BIP-340 path overwrites with the parked R)."""
    for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
        for n in (0, 1, 2, 15, 16, 17, 31, 33, 127, 129, 255, 257, 511, 513, 1000):
            for rep in range(3 if n < 40 else 1):
                o = rep * 40
                m, kk, ss = workload["msg"][o:o + n], workload[k][o:o + n], workload[s][o:o + n]
                got = engine.verify(kind, m, kk, ss)
                want = util.ref_verify(ref, kind, m, kk, ss) if n else np.zeros(0, np.uint8)
                assert np.array_equal(got, want), (kind, n, rep)


def test_sha256d_spans(engine, ref):
    rng = np.random.default_rng(5)
    data = rng.integers(0, 256, size=70000, dtype=np.uint8)
    lens = np.array([0, 1, 31, 32, 55, 56, 63, 64, 65, 119, 120, 127, 128, 174, 300, 1000, 6771] + list(rng.integers(0, 700, size=200)), dtype=np.uint32)
    offs = rng.integers(0, data.size - 7000, size=lens.size).astype(np.uint64)
    got = engine.sha256_double(data, offs, lens)
    for i in range(lens.size):
        want = np.zeros(32, np.uint8)
        seg = np.ascontiguousarray(data[int(offs[i]):int(offs[i]) + int(lens[i])])
        ref.ref_sha256d(util.P(seg) if seg.size else None, ctypes.c_size_t(int(lens[i])), util.P(want))
        assert np.array_equal(got[i], want), (i, lens[i])


def test_verify_raw_matches_hash_then_verify(engine, ref, workload):
    # sign SHA256d(span) with the reference, then let the device hash the span itself
    rng = np.random.default_rng(9)
    n = 300
    data = rng.integers(0, 256, size=n * 200, dtype=np.uint8)
    offs = (np.arange(n) * 200).astype(np.uint64)
    lens = rng.integers(1, 200, size=n).astype(np.uint32)
    sk = rng.integers(1, 256, size=(n, 32), dtype=np.uint8)
    pub = np.zeros((n, 33), np.uint8)
    sig = np.zeros((n, 64), np.uint8)
    for i in range(n):
        h = np.zeros(32, np.uint8)
        seg = np.ascontiguousarray(data[int(offs[i]):int(offs[i]) + int(lens[i])])
        ref.ref_sha256d(util.P(seg), ctypes.c_size_t(int(lens[i])), util.P(h))
        assert ref.ref_pubkey_create(util.P(sk[i]), util.P(pub[i]), None)
        assert ref.ref_ecdsa_sign(util.P(sk[i]), util.P(h), util.P(sig[i]))
    data[int(offs[7]) + 0] ^= 1  # corrupt one message
    got = engine.verify_raw(K33, data, offs, lens, pub, sig)
    assert got[7] == 0 and got.sum() == n - 1


def test_pubkey_parse(engine, ref, workload):
    xy, ok = engine.pubkey_parse(workload["pub33"])
    n = ok.size
    for i in range(n):
        o33 = np.zeros(33, np.uint8)
        oxy = np.zeros(64, np.uint8)
        r = ref.ref_pubkey_convert(util.P(np.ascontiguousarray(workload["pub33"][i])), ctypes.c_size_t(33), util.P(o33), util.P(oxy))
        assert bool(r) == bool(ok[i]), i
        if r:
            assert np.array_equal(xy[i], oxy), i


def test_queue_mixed_kinds(engine, ref, workload):
    want = []
    for i in range(200):
        kind = i % 3
        key = [workload["pub33"], workload["pubxy"], workload["xonly"]][kind][i]
        sig = [workload["sig"], workload["sig"], workload["ssig"]][kind][i]
        engine.enqueue(kind, workload["msg"][i], key, sig)
        want.append(util.ref_verify(ref, kind, workload["msg"][i:i + 1], key.reshape(1, -1), sig.reshape(1, -1))[0])
    assert engine.pending() == 200
    got = engine.flush()
    assert engine.pending() == 0
    assert np.array_equal(got, np.array(want, np.uint8))


def test_synth_generator_is_valid_under_reference(engine, ref):
    import torch
    n = 3000
    for kind in (K33, KXY, KSCH):
        ks = [33, 64, 32][kind]
        msg = torch.empty(n * 32, dtype=torch.uint8, device="cuda")
        key = torch.empty(n * ks, dtype=torch.uint8, device="cuda")
        sig = torch.empty(n * 64, dtype=torch.uint8, device="cuda")
        ver = torch.empty(n, dtype=torch.uint8, device="cuda")
        bits = torch.zeros((n + 31) // 32, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        engine.synth_device(kind, 1234 + kind, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr())
        engine.verify_device(kind, msg.data_ptr(), key.data_ptr(), sig.data_ptr(), n, ver.data_ptr(), bits.data_ptr())
        engine.sync()
        m = msg.cpu().numpy().reshape(n, 32)
        k = key.cpu().numpy().reshape(n, ks)
        s = sig.cpu().numpy().reshape(n, 64)
        want = util.ref_verify(ref, kind, m, k, s)
        assert want.all(), f"kind {kind}: generator produced {n - want.sum()} signatures the reference rejects"
        got = ver.cpu().numpy()
        assert np.array_equal(got, want)
        b = bits.cpu().numpy().view(np.uint32)
        unpacked = ((b[:, None] >> np.arange(32, dtype=np.uint32)[None, :]) & 1).reshape(-1)[:n].astype(np.uint8)
        assert np.array_equal(unpacked, got)


def test_mutation_differential(engine, ref):
    """20,000 structured mutations (boundary r/s/x/m values, negated or swapped fields, random flips): GPU vs reference."""
    from tests import mutations
    w = util.make_signed(20000, seed=321)
    cls = mutations.mutate(w, seed=10)
    for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s], threads=8)
        got = engine.verify(kind, w["msg"], w[k], w[s])
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (kind, bad[:5], cls[bad[:5]], want[bad[:5]])
