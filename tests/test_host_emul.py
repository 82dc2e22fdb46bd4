"""CPU-only: the engine's device headers compiled for the host (tests/host_emul) vs Python integers,
the oracle and the golden vectors.  Everything above the inline-PTX primitives is covered here; the
PTX forms of those primitives are covered by the -m gpu tests."""
import ctypes
import json
import os
import random

import numpy as np
import pytest

from tests import adversarial, util

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
P = util.P
p, n = util.P_FIELD, util.N_ORDER
LAM = adversarial.LAMBDA


def L(x):
    return (ctypes.c_uint32 * 8)(*[(x >> (32 * i)) & 0xFFFFFFFF for i in range(8)])


def V(a, k=8):
    return sum(int(a[i]) << (32 * i) for i in range(k))


def feop(E, op, a, b=0):
    o = (ctypes.c_uint32 * 8)()
    E.emul_fe_op(op, L(a), L(b), o)
    return V(o)


def scop(E, op, a, b=0):
    o = (ctypes.c_uint32 * 8)()
    E.emul_sc_op(op, L(a), L(b), o)
    return V(o)


EDGE = [0, 1, 2, p - 1, p, p + 1, 2**256 - 1, 2**256 - 2, 2**32 + 977, 2**32 + 976, 2**255, p - 2, (p + 1) // 2,
        2**224, 977, 2**256 - 2**32 - 978, 2**64 - 1, (2**256 - 1) ^ (2**128 - 1)]


def test_field_ops_vs_python(emul):
    rnd = random.Random(1)
    vals = EDGE + [rnd.getrandbits(256) for _ in range(120)]
    for a in vals:
        for b in rnd.sample(vals, 10) + EDGE[:9]:
            assert feop(emul, 0, a, b) == a * b % p
            assert feop(emul, 2, a, b) == (a + b) % p
            assert feop(emul, 3, a, b) == (a - b) % p
            raw = (ctypes.c_uint32 * 8)()
            for op in (0, 2, 3):  # weak form: any value < 2^256 congruent to the result
                emul.emul_fe_op_raw(op, L(a), L(b), raw)
                exp = [a * b, 0, a + b, a - b][op]
                assert V(raw) % p == exp % p
        assert feop(emul, 1, a) == a * a % p
        assert feop(emul, 6, a) == (-a) % p
        for k in (2, 3, 8, 65535):
            assert feop(emul, 7, a, k) == k * a % p
        assert feop(emul, 8, a) == 3 * a % p and feop(emul, 9, a) == 8 * a % p
    for a in vals[:50]:
        assert feop(emul, 4, a) == pow(a, p - 2, p)
        s = feop(emul, 5, a)
        if pow(a % p, (p - 1) // 2, p) in (0, 1):
            assert s * s % p == a % p
        else:
            assert s == 0


def test_scalar_ops_vs_python(emul):
    rnd = random.Random(2)
    vals = [0, 1, 2, n - 1, n - 2, (n - 1) // 2, (n + 1) // 2, 2**128, 2**255] + [rnd.randrange(n) for _ in range(80)]
    for a in vals:
        for b in rnd.sample(vals, 8):
            assert scop(emul, 0, a, b) == a * b % n
            assert scop(emul, 2, a, b) == (a + b) % n
        assert scop(emul, 3, a) == (-a) % n
    for a in vals[:16]:
        assert scop(emul, 1, a) == pow(a, n - 2, n)
    for i in range(150):
        t = [2**512 - 1, 0, 2**256, n * n, (n - 1) ** 2, 2**512 - 2**256][i] if i < 6 else rnd.getrandbits(512)
        arr = (ctypes.c_uint32 * 16)(*[(t >> (32 * k)) & 0xFFFFFFFF for k in range(16)])
        o = (ctypes.c_uint32 * 8)()
        emul.emul_sc_reduce512(arr, o)
        assert V(o) == t % n


def test_glv_split_and_recoding_invariants(emul):
    rnd = random.Random(3)
    specials = [v % n for v in adversarial.special_scalars()]
    for u2 in specials + [rnd.randrange(n) for _ in range(300)]:
        u1 = rnd.choice(specials) if u2 & 1 else rnd.randrange(n)
        k1 = (ctypes.c_uint32 * 5)()
        k2 = (ctypes.c_uint32 * 5)()
        gd = (ctypes.c_int * 16)()
        emul.emul_prepare(L(u1), L(u2), k1, k2, gd)
        a, b = V(k1, 5), V(k2, 5)
        sa, sb = a >> 159, b >> 159
        a &= (1 << 159) - 1
        b &= (1 << 159) - 1
        assert a & 1 and b & 1 and a < 2**131 and b < 2**131  # odd halves, top window value <= 7
        A, B = (-a if sa else a), (-b if sb else b)
        assert (A + B * LAM - u2) % n == 0
        assert sum(gd[i] << (16 * i) for i in range(16)) == u1
        assert all(-32768 <= gd[i] <= 32768 for i in range(15)) and 0 <= gd[15] <= 65536


def test_device_sha256_paths(emul):
    import hashlib
    rnd = np.random.default_rng(4)
    for ln in [0, 1, 55, 56, 63, 64, 65, 119, 120, 127, 128, 174, 1000]:
        d = rnd.integers(0, 256, size=max(ln, 1), dtype=np.uint8)
        o = np.zeros(32, np.uint8)
        emul.emul_sha256d(P(d), ctypes.c_size_t(ln), P(o))
        assert bytes(o) == hashlib.sha256(hashlib.sha256(bytes(d[:ln])).digest()).digest(), ln
    tag = hashlib.sha256(b"BIP0340/challenge").digest()
    for _ in range(5):
        r, px, m = (rnd.integers(0, 256, size=32, dtype=np.uint8) for _ in range(3))
        o = np.zeros(32, np.uint8)
        emul.emul_bip340_challenge(P(r), P(px), P(m), P(o))
        assert bytes(o) == hashlib.sha256(tag + tag + bytes(r) + bytes(px) + bytes(m)).digest()


def test_gtable_entries(emul, ref):
    emul.emul_gtable_build()
    for row, d in [(0, 1), (0, 2), (0, 32768), (1, 1), (7, 12345), (15, 65536), (15, 1), (14, 32768), (3, 77)]:
        e = row * 32768 + d - 1
        xy = (ctypes.c_uint32 * 16)()
        emul.emul_gtable_get(e, xy)
        k = (d << (16 * row)) % n
        kb = np.frombuffer(k.to_bytes(32, "big"), dtype=np.uint8).copy()
        out = np.zeros(64, np.uint8)
        assert ref.ref_scalar_base_mult(P(kb), P(out))
        assert V(xy[:8]).to_bytes(32, "big") + V(xy[8:]).to_bytes(32, "big") == bytes(out)
        xy2 = (ctypes.c_uint32 * 16)()
        emul.emul_gtable_entry_device_algo(e, xy2)  # the double-and-add + Fermat path the K4 kernel uses
        assert list(xy) == list(xy2)


def emul_verify(emul, kind, msg, key, sig):
    out = np.zeros(msg.shape[0], np.uint8)
    msg, key, sig = (np.ascontiguousarray(a) for a in (msg, key, sig))
    emul.emul_verify_batch(kind, P(msg), P(key), P(sig), ctypes.c_size_t(msg.shape[0]), P(out))
    return out


def test_full_verify_random_and_corrupted(emul, ref):
    w = util.corrupt(util.make_signed(700, seed=5), every=3)
    for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s])
        assert np.array_equal(emul_verify(emul, kind, w["msg"], w[k], w[s]), want), kind


def test_full_verify_golden_vectors(emul):
    h = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()
    for v in json.load(open(os.path.join(GOLD, "wycheproof_ecdsa.json"))):
        if v["sig64"] is None:
            continue
        assert emul_verify(emul, 0, h(v["msg32"], 32), h(v["pub33"], 33), h(v["sig64"], 64))[0] == v["expected"], v["tcId"]
        assert emul_verify(emul, 1, h(v["msg32"], 32), h(v["pubxy"], 64), h(v["sig64"], 64))[0] == v["expected"], v["tcId"]
    for v in json.load(open(os.path.join(GOLD, "bip340.json"))):
        assert emul_verify(emul, 2, h(v["msg32"], 32), h(v["xonly"], 32), h(v["sig64"], 64))[0] == v["expected"], v["index"]


def test_full_verify_adversarial_scalars(emul, ref):
    msg, pub33, pubxy, sig = adversarial.load()
    assert msg.shape[0] > 1000
    want = util.ref_verify(ref, 0, msg, pub33, sig)
    assert want.all(), "crafted signatures must be valid under the reference"
    assert np.array_equal(emul_verify(emul, 0, msg, pub33, sig), want)
    assert np.array_equal(emul_verify(emul, 1, msg, pubxy, sig), want)
    # and the same signatures against a wrong message must fail identically
    msg2 = msg.copy()
    msg2[:, 31] ^= 1
    want2 = util.ref_verify(ref, 0, msg2, pub33, sig)
    assert np.array_equal(emul_verify(emul, 0, msg2, pub33, sig), want2)


def test_device_bip143_preimage_vs_libwally(emul, cln):
    """Row N2: the device-side BIP143 sighash (host build of the kernel source) vs libwally's bip143_signature_hash."""
    import lightning_b200 as L
    assert emul.emul_sizeof_tx_item() == ctypes.sizeof(L.SvTx)
    rng = np.random.default_rng(31)
    txs, blob = util.make_htlc_txs(rng, 200)
    buf = np.frombuffer(blob, dtype=np.uint8)
    for i in range(200):
        out = np.zeros(32, np.uint8)
        assert emul.emul_bip143(ctypes.byref(txs[i]), P(buf), P(out)) == 1
        assert np.array_equal(out, util.cln_sighash(cln, txs[i], blob)), (i, txs[i].sighash_type)


def test_samekey_path(emul, ref):
    """Row N3: one key, many signatures — table built once, ladder-only verification (host build of the kernel code)."""
    rng = np.random.default_rng(6)
    n = 90
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    sig = np.zeros((n, 64), np.uint8)
    for i in range(n):
        assert ref.ref_ecdsa_sign(P(sk), P(msg[i]), P(sig[i]))
    msg[5, 0] ^= 1; sig[17, 40] ^= 1; sig[33, 32:] = 255; sig[60, :32] = 0
    want = util.ref_verify(ref, 0, msg, np.tile(pub33, (n, 1)), sig)
    for kind, key in ((0, pub33), (1, pubxy)):
        out = np.zeros(n, np.uint8)
        emul.emul_verify_samekey(kind, P(key), P(msg), P(sig), ctypes.c_size_t(n), P(out))
        assert np.array_equal(out, want), kind
    bad = pub33.copy(); bad[0] = 5
    out = np.ones(n, np.uint8)
    emul.emul_verify_samekey(0, P(bad), P(msg), P(sig), ctypes.c_size_t(n), P(out))
    assert not out.any()


def test_mutation_differential(emul, ref):
    """~3,000 structured mutations (boundary values of r, s, x, m; swapped/negated fields; random flips) of valid
    triples: the host build of the kernel code and the reference must agree on every verdict, for all three kinds."""
    from tests import mutations
    w = util.make_signed(3000, seed=123)
    cls = mutations.mutate(w, seed=9)
    for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s], threads=4)
        got = emul_verify(emul, kind, w["msg"], w[k], w[s])
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, (kind, bad[:5], cls[bad[:5]], want[bad[:5]])
        assert 100 < want.sum() < 2900


def test_ecdsa_edge_cases_tests_c_7069(emul, ref):
    """test_ecdsa_edge_cases (tests.c:7069-7297) as (msg, key, sig) triples: infinity, r = 0, s = 0, messages 0 / 1 / -1
    with crafted keys, r = p - n, nonce n-1, unparsable compact signature — host build of the kernel code vs the fixture
    (whose expectations were taken from the reference's public API at generation time and are re-checked here)."""
    cases = json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json")))
    h = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()
    for c in cases:
        m, k, s = h(c["msg32"], 32), h(c["pub33"], 33), h(c["sig64"], 64)
        assert util.ref_verify(ref, 0, m, k, s)[0] == c["expected"], c["name"]
        assert emul_verify(emul, 0, m, k, s)[0] == c["expected"], c["name"]


def test_bip143_bolt3_and_general_shapes_vs_libwally(emul):
    """BOLT #3 Appendix C HTLC transactions (channeld/test/run-full_channel.c:635-673): the device-side BIP143 code (host
    build) reproduces libwally's sighash; and for multi-input / multi-output transactions the serialised-span forms of
    sv_tx (what the check_tx_sig drop-in passes) match bitcoin_tx_hash_for_sig for every sighash type
    (tests/golden/bip143_libwally.json: libwally's sighash of each seeded transaction, made by make_golden.py)."""
    import lightning_b200 as L
    recs = json.load(open(os.path.join(GOLD, "bolt3_htlc_txs.json")))
    for r in recs:
        t = L.SvTx()
        t.version, t.locktime, t.sequence, t.sighash_type = r["version"], r["locktime"], r["sequence"], 1
        t.prev_txid[:] = list(bytes.fromhex(r["prev_txid"]))
        t.prev_index = r["prev_index"]
        ws, os_ = bytes.fromhex(r["wscript"]), bytes.fromhex(r["out_script"])
        t.script_off, t.script_len, t.out_script_off, t.out_script_len = 0, len(ws), len(ws), len(os_)
        t.input_amount, t.output_amount = r["input_amount"], r["output_amount"]
        buf = np.frombuffer(ws + os_, dtype=np.uint8)
        out = np.zeros(32, np.uint8)
        assert emul.emul_bip143(ctypes.byref(t), P(buf), P(out)) == 1
        assert bytes(out).hex() == r["sighash"], r["name"]
    wally = json.load(open(os.path.join(GOLD, "bip143_libwally.json")))
    assert len(wally) == 120
    rng = np.random.default_rng(8)
    le = lambda v, n: int(v).to_bytes(n, "little")

    def varint(v):
        return bytes([v]) if v < 0xfd else b"\xfd" + le(v, 2)
    for it in range(120):
        nin, nout = int(rng.integers(1, 4)), int(rng.integers(1, 7))
        ins = [(bytes(rng.integers(0, 256, size=32, dtype=np.uint8)), int(rng.integers(0, 9)), int(rng.integers(0, 2**32))) for _ in range(nin)]
        outs = [(int(rng.integers(0, 2**40)), bytes(rng.integers(0, 256, size=int(rng.choice([0, 22, 34, 300])), dtype=np.uint8))) for _ in range(nout)]
        lock = int(rng.integers(0, 2**32))
        inp = int(rng.integers(0, nin))
        ws = bytes(rng.integers(0, 256, size=int(rng.choice([1, 2, 133, 252, 253, 700])), dtype=np.uint8))
        amount = int(rng.integers(0, 2**45))
        sht = int(rng.choice([1, 0x83, 2, 3, 0x81, 0x82]))
        want = np.frombuffer(bytes.fromhex(wally[it]), dtype=np.uint8)
        # the adapter's layout: script, serialised outputs, outpoints, sequences
        t = L.SvTx()
        t.version, t.locktime, t.sequence, t.sighash_type = 2, lock, ins[inp][2], sht
        t.prev_txid[:] = list(ins[inp][0])
        t.prev_index = ins[inp][1]
        t.input_amount = amount
        blob = bytearray(ws)
        t.script_off, t.script_len = 0, len(ws)
        t.out_script_off = len(blob)
        ser = lambda o: le(o[0], 8) + varint(len(o[1])) + o[1]
        if (sht & 0x1f) == 3:
            if inp < nout:
                blob += ser(outs[inp])
                t.flags |= 1
            else:
                t.flags |= 4
        else:
            for o in outs:
                blob += ser(o)
            t.flags |= 1
        t.out_script_len = len(blob) - t.out_script_off
        if nin > 1:
            t.flags |= 2
            t.prevouts_off = len(blob)
            for a in ins:
                blob += a[0] + le(a[1], 4)
            t.prevouts_len = 36 * nin
            t.sequences_off = len(blob)
            for a in ins:
                blob += le(a[2], 4)
            t.sequences_len = 4 * nin
        buf = np.frombuffer(bytes(blob) + b"\0", dtype=np.uint8)
        out = np.zeros(32, np.uint8)
        assert emul.emul_bip143(ctypes.byref(t), P(buf), P(out)) == 1
        assert np.array_equal(out, want), (it, nin, nout, inp, hex(sht), len(ws))


def test_small_batch_path_all_vector_sets(emul, ref):
    """The small-batch schedule (two GLV half-ladders + comb sum joined by full Jacobian additions, unbatched scalar side;
    k_small on the device) gives the reference's verdicts on every vector set the throughput path is held to: random +
    corrupted, structured mutations, adversarial scalars (where the partial sums collide, cancel or vanish), Wycheproof,
    BIP-340, the tests.c edge cases."""
    from tests import mutations
    PAIR_CAP = [150]  # the thread-pair emulation is slow: the first 150 items of every set, ALL adversarial signatures

    def small(kind, msg, key, sig):
        out = np.zeros(msg.shape[0], np.uint8)
        msg, key, sig = (np.ascontiguousarray(a) for a in (msg, key, sig))
        emul.emul_verify_small_batch(kind, P(msg), P(key), P(sig), ctypes.c_size_t(msg.shape[0]), P(out))
        # and with the half ladders on lane PAIRS (what k_small runs): two host threads per half ladder, results crossing
        # at a mailbox where the device uses warp shuffles
        m = min(msg.shape[0], PAIR_CAP[0])
        out2 = np.zeros(m, np.uint8)
        emul.emul_verify_small_pair_batch(kind, P(msg), P(key), P(sig), ctypes.c_size_t(m), P(out2))
        assert np.array_equal(out2, out[:m]), "pair-lane half ladders disagree with the single-lane schedule"
        return out
    w = util.corrupt(util.make_signed(400, seed=15), every=3)
    w2 = util.make_signed(900, seed=16)
    mutations.mutate(w2, seed=3)
    for ww in (w, w2):
        for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
            want = util.ref_verify(ref, kind, ww["msg"], ww[k], ww[s], threads=4)
            assert np.array_equal(small(kind, ww["msg"], ww[k], ww[s]), want), kind
    msg, pub33, pubxy, sig = adversarial.load()
    PAIR_CAP[0] = 10**9
    assert small(0, msg, pub33, sig).all()
    PAIR_CAP[0] = 150
    assert small(1, msg, pubxy, sig).all()
    msg2 = msg.copy()
    msg2[:, 31] ^= 1
    assert np.array_equal(small(0, msg2, pub33, sig), util.ref_verify(ref, 0, msg2, pub33, sig))
    h = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()
    for v in json.load(open(os.path.join(GOLD, "wycheproof_ecdsa.json"))):
        if v["sig64"] is not None:
            assert small(0, h(v["msg32"], 32), h(v["pub33"], 33), h(v["sig64"], 64))[0] == v["expected"], v["tcId"]
    for v in json.load(open(os.path.join(GOLD, "bip340.json"))):
        assert small(2, h(v["msg32"], 32), h(v["xonly"], 32), h(v["sig64"], 64))[0] == v["expected"], v["index"]
    for c in json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json"))):
        assert small(0, h(c["msg32"], 32), h(c["pub33"], 33), h(c["sig64"], 64))[0] == c["expected"], c["name"]


def test_bip340_batch_verification_group_equations(emul, ref):
    """Row N3: random-linear-combination batch verification, host build of every stage (preparation, signed 6-bit recoding,
    bucket window sums, Horner combination, G term): a group of valid signatures satisfies its equation whatever the seed;
    one bad signature (wrong message, flipped s, someone else's key) fails ITS group only; encoding failures (r >= p, s >= n,
    x not on the curve) are excluded and do not poison the group."""
    n = 1024 + 90  # one full group and a ragged one
    w = util.make_signed(n, seed=77)
    msg, key, sig = w["msg"].copy(), w["xonly"].copy(), w["ssig"].copy()
    want = util.ref_verify(ref, 2, msg, key, sig, threads=4)
    assert want.all()

    def run(m, k, s, seed):
        ok = np.zeros(n, np.uint8)
        gok = np.zeros(2, np.uint8)
        sd = np.frombuffer(seed, dtype=np.uint8).copy()
        emul.emul_schnorr_batch(P(np.ascontiguousarray(m)), P(np.ascontiguousarray(k)), P(np.ascontiguousarray(s)), ctypes.c_size_t(n), P(sd), P(ok), P(gok))
        return ok, gok
    for seed in (bytes(32), bytes(range(32))):
        ok, gok = run(msg, key, sig, seed)
        assert ok.all() and list(gok) == [1, 1]
    # encoding failures drop out without poisoning
    s2, k2 = sig.copy(), key.copy()
    s2[5, :32] = 255        # r >= p
    s2[6, 32:] = 255        # s >= n
    k2[7, :] = 0
    k2[7, 31] = 5           # x = 5 is not on the curve
    ok, gok = run(msg, k2, s2, bytes(range(32)))
    assert list(np.nonzero(ok == 0)[0]) == [5, 6, 7] and list(gok) == [1, 1]
    assert not util.ref_verify(ref, 2, msg[5:8], k2[5:8], s2[5:8]).any()
    # a well-formed but wrong signature fails its own group only
    for mutate, grp in ((lambda m, k, s: m.__setitem__((1050, 3), m[1050, 3] ^ 1), 1), (lambda m, k, s: s.__setitem__((17, 40), s[17, 40] ^ 2), 0),
                        (lambda m, k, s: k.__setitem__(300, k[301].copy()), 0)):
        m3, k3, s3 = msg.copy(), key.copy(), sig.copy()
        mutate(m3, k3, s3)
        ok, gok = run(m3, k3, s3, bytes(range(32)))
        if ok.all():  # (a flipped s may land >= n: then it is an encoding failure instead)
            expect = [1, 1]
            expect[grp] = 0
            assert list(gok) == expect


def test_ecdsa33_without_square_root_vs_plain_path(emul, ref):
    """Compressed-key ECDSA has two flows in the engine (verify.cuh "without the square root"): the linear-in-y form with a
    batched division, and the plain path with the real square root.  Both must give the reference's verdicts; random
    workloads must stay on the fast flow, while the crafted scalars (u1*G = +-u2*Q, u1 = 0, r + n candidates) and keys whose
    x is not on the curve are the cases the fast flow hands back."""
    emul.emul_last_exact_count.restype = ctypes.c_size_t
    w = util.corrupt(util.make_signed(600, seed=77), every=4)
    # keys not on the curve (x^3 + 7 a non-residue), valid-looking otherwise
    bad = w["pub33"][:50].copy()
    for i in range(50):
        x = int.from_bytes(bytes(bad[i, 1:]), "big")
        while pow((pow(x, 3, p) + 7) % p, (p - 1) // 2, p) == 1:
            x = (x + 1) % p
        bad[i, 1:] = np.frombuffer(x.to_bytes(32, "big"), np.uint8)
    w["pub33"][:50] = bad
    want = util.ref_verify(ref, 0, w["msg"], w["pub33"], w["sig"])
    assert not want[:50].any()
    amsg, apub33, _, asig = adversarial.load()
    awant = util.ref_verify(ref, 0, amsg, apub33, asig)
    cases = json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json")))
    h = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()
    try:
        for exact in (0, 1):
            emul.emul_set_ecdsa33_exact(exact)
            assert np.array_equal(emul_verify(emul, 0, w["msg"], w["pub33"], w["sig"]), want), exact
            if not exact:
                assert emul.emul_last_exact_count() == 0  # nothing on a random workload needs the plain path
            assert np.array_equal(emul_verify(emul, 0, amsg, apub33, asig), awant), exact
            if not exact:
                assert emul.emul_last_exact_count() > 0   # the crafted ones do
            for c in cases:
                assert emul_verify(emul, 0, h(c["msg32"], 32), h(c["pub33"], 33), h(c["sig64"], 64))[0] == c["expected"], (exact, c["name"])
            # the per-item byte of the gossip path: bit 0 = the key parses (secp256k1_ec_pubkey_parse), bit 1 = r, s < n
            n_items = w["msg"].shape[0]
            out, aux = np.zeros(n_items, np.uint8), np.zeros(n_items, np.uint8)
            emul.emul_verify_batch_aux(0, P(w["msg"]), P(w["pub33"]), P(w["sig"]), ctypes.c_size_t(n_items), P(out), P(aux))
            assert np.array_equal(out, want)
            tmp33, tmp64 = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
            for i in range(n_items):
                kd = ref.ref_pubkey_convert(P(np.ascontiguousarray(w["pub33"][i])), ctypes.c_size_t(33), P(tmp33), P(tmp64))
                ps = ref.ref_make_opaque_sig(P(np.ascontiguousarray(w["sig"][i])), P(tmp64))
                assert aux[i] == (1 if kd else 0) | (2 if ps else 0), (exact, i, aux[i], kd, ps)
            # BIP-340 through the same switch: random / corrupted triples, x-only keys off the curve, s = 0 (the comb sum is
            # the point at infinity: handed to the plain flow), and the official vectors
            ws = util.corrupt(util.make_signed(400, seed=79), every=3)
            ws["xonly"][:40] = w["pub33"][:40, 1:]   # off the curve
            ws["ssig"][40:50, 32:] = 0               # s = 0
            swant = util.ref_verify(ref, 2, ws["msg"], ws["xonly"], ws["ssig"])
            assert not swant[:50].any() and swant.sum() > 150
            assert np.array_equal(emul_verify(emul, 2, ws["msg"], ws["xonly"], ws["ssig"]), swant), exact
            if not exact:
                assert emul.emul_last_exact_count() == 10
            for v in json.load(open(os.path.join(GOLD, "bip340.json"))):
                assert emul_verify(emul, 2, h(v["msg32"], 32), h(v["xonly"], 32), h(v["sig64"], 64))[0] == v["expected"], (exact, v["index"])
            # the small-batch schedule follows the same switch (k_small<kind, nosqrt>): single-lane and lane-pair half ladders,
            # verdicts and the per-item byte
            sm = np.zeros(n_items, np.uint8)
            emul.emul_verify_small_batch(0, P(w["msg"]), P(w["pub33"]), P(w["sig"]), ctypes.c_size_t(n_items), P(sm))
            assert np.array_equal(sm, want), exact
            m = 120
            out2, aux2 = np.zeros(m, np.uint8), np.zeros(m, np.uint8)
            emul.emul_verify_small_pair_batch_aux(0, P(w["msg"]), P(w["pub33"]), P(w["sig"]), ctypes.c_size_t(m), P(out2), P(aux2))
            assert np.array_equal(out2, want[:m]) and np.array_equal(aux2, aux[:m]), exact
            sm = np.zeros(ws["msg"].shape[0], np.uint8)
            emul.emul_verify_small_batch(2, P(ws["msg"]), P(ws["xonly"]), P(ws["ssig"]), ctypes.c_size_t(sm.shape[0]), P(sm))
            assert np.array_equal(sm, swant), exact
            sm = np.zeros(amsg.shape[0], np.uint8)
            emul.emul_verify_small_batch(0, P(amsg), P(apub33), P(asig), ctypes.c_size_t(sm.shape[0]), P(sm))
            assert np.array_equal(sm, awant), exact
    finally:
        emul.emul_set_ecdsa33_exact(0)


def test_linear_form_algebra_against_plain_jacobian_addition(emul, ref):
    """The identity the no-sqrt flows rest on, checked directly on the host build: for S = (X, Y, y*Zs), T Jacobian and
    c = y^2, ns_linear_form's D, B, N, CG satisfy D == y*B exactly when r = x(S + T), N == Y3*B and CG*y == Z3^3, with
    S + T computed by the plain addition formulas.  200 random configurations (points from the reference's k*G)."""
    rng = random.Random(2718)

    def point():
        k = rng.randrange(1, n)
        out = np.zeros(64, np.uint8)
        assert ref.ref_scalar_base_mult(P(np.frombuffer(k.to_bytes(32, "big"), np.uint8).copy()), P(out))
        return limbs(int.from_bytes(bytes(out[:32]), "big")) + limbs(int.from_bytes(bytes(out[32:]), "big"))

    def limbs(v):
        return [(v >> (32 * i)) & 0xFFFFFFFF for i in range(8)]
    arr = lambda xs: (ctypes.c_uint32 * len(xs))(*xs)
    emul.emul_ns_linear_check.restype = ctypes.c_int
    for _ in range(200):
        vals = [limbs(rng.randrange(1, p)) for _ in range(3)]
        assert emul.emul_ns_linear_check(arr(point()), arr(point()), arr(vals[0]), arr(vals[1]), arr(vals[2])) == 15


def test_no_sqrt_flows_larger_random_sample(emul, ref):
    """10,000 reference-signed triples per kind (every third one corrupted) through the flows without the square root —
    throughput schedule (park + batched division) and, for BIP-340, the small-batch schedule — against the reference."""
    w = util.corrupt(util.make_signed(10000, seed=4242), every=3)
    for kind, k, s in ((0, "pub33", "sig"), (2, "xonly", "ssig")):
        want = util.ref_verify(ref, kind, w["msg"], w[k], w[s], threads=4)
        got = emul_verify(emul, kind, w["msg"], w[k], w[s])
        assert np.array_equal(got, want), kind
        assert 6000 < want.sum() < 7000
    sm = np.zeros(3000, np.uint8)
    emul.emul_verify_small_batch(2, P(np.ascontiguousarray(w["msg"][:3000])), P(np.ascontiguousarray(w["xonly"][:3000])),
                                 P(np.ascontiguousarray(w["ssig"][:3000])), ctypes.c_size_t(3000), P(sm))
    assert np.array_equal(sm, util.ref_verify(ref, 2, w["msg"][:3000], w["xonly"][:3000], w["ssig"][:3000], threads=4))
