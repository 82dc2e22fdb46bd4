"""GPU: the small-batch (latency) path k_small against the reference AND against the throughput kernels.

Every vector set the throughput path is held to is pushed through both paths (sv_set_small_max switches): random and
corrupted triples of all three kinds at ragged sizes around the CTA width (32) and the dispatch threshold, structured
mutations, adversarial scalars (partial sums that collide, cancel or vanish), Wycheproof, BIP-340, the tests.c edge
cases; then the composite entry points (gossip slicing, device-side BIP143, same-key batches, the deferral queue) with the
small path on and off."""
import json
import os

import numpy as np
import pytest

from tests import adversarial, mutations, util

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
KINDS = [("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]


@pytest.fixture()
def both(engine):
    """run fn(engine) with the small path enabled (every batch up to 8192) and disabled; restore the default"""
    default = engine.small_max()

    def run(fn):
        engine.set_small_max(8192)
        a = fn()
        engine.set_small_max(0)
        b = fn()
        engine.set_small_max(default)
        return a, b
    yield run
    engine.set_small_max(default)


def test_small_path_random_corrupted_ragged(engine, ref, both):
    w = util.corrupt(util.make_signed(8200, seed=77), every=5)
    for kind, (k, s) in enumerate(KINDS):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s], threads=4)
        for n in (1, 2, 3, 4, 5, 31, 32, 33, 63, 64, 65, 95, 96, 97, 483, 1000, 2047, 2048, 2049, 2600, 8191, 8192, 8193, 8200):
            a, b = both(lambda: engine.verify(kind, w["msg"][:n], w[k][:n], w[s][:n]))
            assert np.array_equal(a, want[:n]), (kind, n, "small")
            assert np.array_equal(b, want[:n]), (kind, n, "throughput")
        o = 1234  # a window that does not start at item 0
        a, b = both(lambda: engine.verify(kind, w["msg"][o:o + 40], w[k][o:o + 40], w[s][o:o + 40]))
        assert np.array_equal(a, want[o:o + 40]) and np.array_equal(b, want[o:o + 40])
    assert engine.small_max() == 8192


def test_small_path_mutations_adversarial_golden(engine, ref, both):
    w = util.make_signed(3000, seed=123)
    mutations.mutate(w, seed=9)
    for kind, (k, s) in enumerate(KINDS):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s], threads=4)
        a, b = both(lambda: engine.verify(kind, w["msg"], w[k], w[s]))
        assert np.array_equal(a, want) and np.array_equal(b, want), kind
    msg, pub33, pubxy, sig = adversarial.load()
    a, b = both(lambda: (engine.verify(0, msg, pub33, sig), engine.verify(1, msg, pubxy, sig)))
    assert all(x.all() for x in a + b), "crafted (valid) signatures must verify on both paths"
    msg2 = msg.copy()
    msg2[:, 31] ^= 1
    want = util.ref_verify(ref, 0, msg2, pub33, sig, threads=4)
    a, b = both(lambda: engine.verify(0, msg2, pub33, sig))
    assert np.array_equal(a, want) and np.array_equal(b, want)
    H = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()
    vec = [v for v in json.load(open(os.path.join(GOLD, "wycheproof_ecdsa.json"))) if v["sig64"]]
    m, k, s = (np.concatenate([H(v[x], n) for v in vec]) for x, n in (("msg32", 32), ("pub33", 33), ("sig64", 64)))
    want = np.array([v["expected"] for v in vec], np.uint8)
    a, b = both(lambda: engine.verify(0, m, k, s))
    assert np.array_equal(a, want) and np.array_equal(b, want)
    for i in range(0, len(vec), 7):  # one call per signature, as CLN's synchronous callers make them
        assert engine.verify(0, m[i:i + 1], k[i:i + 1], s[i:i + 1])[0] == want[i], vec[i]["tcId"]
    vec = json.load(open(os.path.join(GOLD, "bip340.json")))
    m, k, s = (np.concatenate([H(v[x], n) for v in vec]) for x, n in (("msg32", 32), ("xonly", 32), ("sig64", 64)))
    want = np.array([v["expected"] for v in vec], np.uint8)
    a, b = both(lambda: engine.verify(2, m, k, s))
    assert np.array_equal(a, want) and np.array_equal(b, want)
    vec = json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json")))
    m, k, s = (np.concatenate([H(v[x], n) for v in vec]) for x, n in (("msg32", 32), ("pub33", 33), ("sig64", 64)))
    want = np.array([v["expected"] for v in vec], np.uint8)
    a, b = both(lambda: engine.verify(0, m, k, s))
    assert np.array_equal(a, want) and np.array_equal(b, want)


def test_small_path_composite_entry_points(engine, ref, cln, both):
    """gossip slicing, device BIP143, same-key batches and the mixed deferral queue agree between the two paths"""
    from tests import gossip
    msgs = gossip.load_subset()
    sel = [m for m in msgs if m[:2] == b"\x01\x00"][:150] + [m for m in msgs if m[:2] == b"\x01\x01"][:100]
    rng = np.random.default_rng(3)
    batch = []
    for m in sel:
        b = bytearray(m)
        if rng.random() < 0.2:
            b[int(rng.integers(2, 66))] ^= 1 << int(rng.integers(0, 8))
        batch.append(bytes(b))
    a, b = both(lambda: engine.verify_gossip(batch).copy())
    assert np.array_equal(a, b) and (a == 0).sum() > 150 and (a != 0).sum() > 20
    # one channel_announcement at a time (what gossipd's synchronous path hands over), vs gossipd/sigcheck.c
    import ctypes
    for m in batch[:12]:
        want = cln.cln_sigcheck_channel_announcement(m, ctypes.c_size_t(len(m)))
        assert engine.verify_gossip([m])[0] == want
    n = 483
    txs, blob = util.make_htlc_txs(np.random.default_rng(77), n)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(util.P(sk), util.P(pub33), util.P(pubxy))
    sig = np.zeros((n, 64), np.uint8)
    hs = np.zeros((n, 32), np.uint8)
    for i in range(n):
        hs[i] = util.cln_sighash(cln, txs[i], blob)
        assert ref.ref_ecdsa_sign(util.P(sk), util.P(hs[i]), util.P(sig[i]))
    sig[::9, 12] ^= 1
    want = util.ref_verify(ref, 0, hs, np.tile(pub33, (n, 1)), sig)
    a, b = both(lambda: engine.check_tx_sigs(0, txs, blob, np.tile(pub33, (n, 1)), sig).copy())
    assert np.array_equal(a, want) and np.array_equal(b, want)
    a, b = both(lambda: (engine.verify_samekey(0, pub33, hs, sig).copy(), engine.verify_samekey(1, pubxy, hs, sig).copy()))
    assert all(np.array_equal(x, want) for x in a + b)
    w = util.corrupt(util.make_signed(90, seed=5), every=4)

    def queue():
        for i in range(90):
            kind = i % 3
            engine.enqueue(kind, w["msg"][i], w[KINDS[kind][0]][i], w[KINDS[kind][1]][i])
        return engine.flush().copy()
    a, b = both(queue)
    want = np.array([util.ref_verify(ref, i % 3, w["msg"][i:i + 1], w[KINDS[i % 3][0]][i:i + 1], w[KINDS[i % 3][1]][i:i + 1])[0] for i in range(90)], np.uint8)
    assert np.array_equal(a, want) and np.array_equal(b, want)


def test_ecdsa33_without_square_root_vs_plain_flow(engine, ref):
    """Throughput kernels, compressed and x-only keys: the flow that never takes the square root (k_main<3> + k_final_ecdsa33,
    k_main<4> + k_final_schnorr_ns; the default) and the plain flow give the reference's verdicts on random/corrupted triples
    at ragged sizes, off-curve keys, structured mutations, the crafted scalars that force the fall-back inside the final
    kernel, the tests.c edge cases and the BIP-340 vectors."""
    default = engine.small_max()
    engine.set_small_max(0)
    try:
        w = util.corrupt(util.make_signed(5000, seed=78), every=4)
        p = 2**256 - 2**32 - 977
        for i in range(60):  # x not on the curve
            x = int.from_bytes(bytes(w["pub33"][i, 1:]), "big")
            while pow((pow(x, 3, p) + 7) % p, (p - 1) // 2, p) == 1:
                x = (x + 1) % p
            w["pub33"][i, 1:] = np.frombuffer(x.to_bytes(32, "big"), np.uint8)
        w["pub33"][60, 0] = 4   # bad prefix
        w["pub33"][61, 1:] = 255  # x >= p
        want = util.ref_verify(ref, 0, w["msg"], w["pub33"], w["sig"], threads=4)
        assert not want[:62].any() and want.sum() > 3000
        m = util.make_signed(3000, seed=124)
        mutations.mutate(m, seed=10)
        mwant = util.ref_verify(ref, 0, m["msg"], m["pub33"], m["sig"], threads=4)
        amsg, apub33, _, asig = adversarial.load()
        cases = json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json")))
        h = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k)
        cm = np.concatenate([h(c["msg32"], 32) for c in cases])
        ck = np.concatenate([h(c["pub33"], 33) for c in cases])
        cs = np.concatenate([h(c["sig64"], 64) for c in cases])
        cwant = np.array([c["expected"] for c in cases], np.uint8)
        ws = util.corrupt(util.make_signed(5000, seed=79), every=3)
        ws["xonly"][:60] = w["pub33"][:60, 1:]   # x-only keys off the curve
        ws["ssig"][60:80, 32:] = 0               # s = 0: the comb sum is the point at infinity
        swant = util.ref_verify(ref, 2, ws["msg"], ws["xonly"], ws["ssig"], threads=4)
        assert not swant[:80].any() and swant.sum() > 2000
        vecs = json.load(open(os.path.join(GOLD, "bip340.json")))
        bm = np.concatenate([h(v["msg32"], 32) for v in vecs])
        bk = np.concatenate([h(v["xonly"], 32) for v in vecs])
        bs = np.concatenate([h(v["sig64"], 64) for v in vecs])
        bwant = np.array([v["expected"] for v in vecs], np.uint8)
        for on in (True, False):
            engine.set_nosqrt(on)
            for n in (1, 15, 16, 17, 255, 256, 257, 4097, 5000):
                assert np.array_equal(engine.verify(0, w["msg"][:n], w["pub33"][:n], w["sig"][:n]), want[:n]), (on, n)
            assert np.array_equal(engine.verify(0, m["msg"], m["pub33"], m["sig"]), mwant), on
            assert engine.verify(0, amsg, apub33, asig).all(), on
            assert np.array_equal(engine.verify(0, cm, ck, cs), cwant), on
            for n in (1, 16, 17, 4097, 5000):  # BIP-340 takes the same switch
                assert np.array_equal(engine.verify(2, ws["msg"][:n], ws["xonly"][:n], ws["ssig"][:n]), swant[:n]), (on, n)
            assert np.array_equal(engine.verify(2, bm, bk, bs), bwant), on
    finally:
        engine.set_nosqrt(True)
        engine.set_small_max(default)
