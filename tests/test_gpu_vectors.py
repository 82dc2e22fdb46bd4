"""GPU: reference vector sets ported in round 2 and the C-ABI entry points that round 1 exported but never executed.

  * test_ecdsa_edge_cases (tests.c:7069-7297)                                 -> engine, all ECDSA key forms
  * BOLT #3 Appendix C HTLC transactions (channeld/test/run-full_channel.c)   -> sv_verify_tx_host, check_tx_sig,
                                                                                 check_tx_sigs_bip143_batch
  * check_tx_sig with the reference signature vs CLN's OWN unmodified check_tx_sig on arbitrary transactions
  * sigcheck_channel_update_batch / sigcheck_node_announcement_batch, cln_sigverify_init / shutdown
"""
import ctypes
import json
import os

import numpy as np
import pytest

import lightning_b200 as L
from tests import gossip, util

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
P = util.P
H = lambda s, k: np.frombuffer(bytes.fromhex(s), dtype=np.uint8).reshape(1, k).copy()


def test_ecdsa_edge_cases_tests_c_7069(engine, ref):
    cases = json.load(open(os.path.join(GOLD, "ecdsa_edge_cases.json")))
    msg = np.concatenate([H(c["msg32"], 32) for c in cases])
    pub = np.concatenate([H(c["pub33"], 33) for c in cases])
    sig = np.concatenate([H(c["sig64"], 64) for c in cases])
    want = np.array([c["expected"] for c in cases], np.uint8)
    assert np.array_equal(util.ref_verify(ref, 0, msg, pub, sig), want)  # the fixture still matches the reference
    got = engine.verify(0, msg, pub, sig)
    assert np.array_equal(got, want), [c["name"] for c, g, w in zip(cases, got, want) if g != w]
    # the same through pre-decompressed keys (check_signed_hash's form) and one call at a time
    xy = np.zeros((len(cases), 64), np.uint8)
    for i in range(len(cases)):
        p33 = np.zeros(33, np.uint8)
        assert ref.ref_pubkey_convert(P(np.ascontiguousarray(pub[i])), ctypes.c_size_t(33), P(p33), P(xy[i]))
    assert np.array_equal(engine.verify(1, msg, xy, sig), want)
    for i in range(len(cases)):
        assert engine.verify(0, msg[i:i + 1], pub[i:i + 1], sig[i:i + 1])[0] == want[i], cases[i]["name"]
    assert want.sum() >= 6 and (want == 0).sum() >= 10


def _bolt3():
    return json.load(open(os.path.join(GOLD, "bolt3_htlc_txs.json")))


def _svtx_from_bolt3(recs):
    txs = (L.SvTx * len(recs))()
    blob = bytearray()
    for t, r in zip(txs, recs):
        t.version, t.locktime, t.sequence, t.sighash_type = r["version"], r["locktime"], r["sequence"], 1
        t.prev_txid[:] = list(bytes.fromhex(r["prev_txid"]))
        t.prev_index = r["prev_index"]
        ws, os_ = bytes.fromhex(r["wscript"]), bytes.fromhex(r["out_script"])
        t.script_off, t.script_len = len(blob), len(ws)
        blob += ws
        t.out_script_off, t.out_script_len = len(blob), len(os_)
        blob += os_
        t.input_amount, t.output_amount = r["input_amount"], r["output_amount"]
    return txs, bytes(blob)


def test_bolt3_appendix_c_htlc_signatures_device_bip143(engine):
    """The spec's own signatures (remote and local HTLC signature of each of the five HTLC transactions) verify through
    sv_verify_tx_host, i.e. with the BIP143 sighash assembled and hashed on the device; the sighash equals libwally's."""
    recs = _bolt3()
    for who in (0, 1):
        txs, blob = _svtx_from_bolt3(recs)
        key = np.concatenate([H(r["sigs"][who]["pub33"], 33) for r in recs])
        sig = np.concatenate([H(r["sigs"][who]["sig64"], 64) for r in recs])
        v, sh = engine.check_tx_sigs(0, txs, blob, key, sig, want_sighash=True)
        assert [bytes(x).hex() for x in sh] == [r["sighash"] for r in recs]
        assert v.all()
        sig[2, 40] ^= 1  # and a corrupted one does not
        txs[4].input_amount += 1  # nor one whose amount differs (BIP143 commits to it)
        v = engine.check_tx_sigs(0, txs, blob, key, sig)
        assert list(v) == [1, 1, 0, 1, 0]


class _Cln:
    """typed view of the harness entry points used below (oracle/cln_harness.c)"""

    def __init__(self, cln):
        self.c = cln
        vp, sz, u32, u64 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint32, ctypes.c_uint64
        cln.cln_tx_new.restype = vp
        cln.cln_tx_new.argtypes = [u32, u32]
        cln.cln_tx_add_input.argtypes = [vp, ctypes.c_char_p, u32, u32]
        cln.cln_tx_add_output.argtypes = [vp, u64, ctypes.c_char_p, sz]
        cln.cln_tx_free.argtypes = [vp]
        cln.cln_tx_set_input_amount.argtypes = [u64]
        cln.cln_tal_bytes.restype = vp
        cln.cln_tal_bytes.argtypes = [ctypes.c_char_p, sz]
        cln.cln_tal_free.argtypes = [vp]
        cln.cln_sizeof_bitcoin_signature.restype = sz
        cln.cln_make_tx_sig_args.argtypes = [vp, u32, vp, vp, vp]
        cln.cln_tx_sighash.argtypes = [vp, ctypes.c_uint, vp, u32, vp]
        cln.cln_check_tx_sig.argtypes = [vp, sz, vp, vp, vp, vp]


def _dropin_tx(engine, cln):
    lib = engine.lib
    lib.check_tx_sig.restype = ctypes.c_bool
    lib.check_tx_sig.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    lib.cln_sigverify_set_tx_hooks.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.cln_sigverify_set_tx_hooks(ctypes.cast(cln.cln_tal_bytelen_hook, ctypes.c_void_p), ctypes.cast(cln.cln_tx_input_amount_hook, ctypes.c_void_p))
    return lib


def test_check_tx_sig_reference_signature_bolt3(engine, cln_live):
    """bitcoin/signature.h:120 check_tx_sig(tx, input_num, redeemscript, witness_script, key, sig) exported by the engine,
    fed the reference's own struct bitcoin_tx (libwally wally_tx inside) — BOLT #3's HTLC transactions."""
    cln = cln_live
    C = _Cln(cln)
    lib = _dropin_tx(engine, cln)
    assert cln.cln_sizeof_bitcoin_signature() == 68
    for r in _bolt3():
        tx = cln.cln_tx_new(r["version"], r["locktime"])
        assert cln.cln_tx_add_input(tx, bytes.fromhex(r["prev_txid"]), r["prev_index"], r["sequence"]) == 0
        os_ = bytes.fromhex(r["out_script"])
        assert cln.cln_tx_add_output(tx, r["output_amount"], os_, len(os_)) == 0
        ws = bytes.fromhex(r["wscript"])
        tal_ws = cln.cln_tal_bytes(ws, len(ws))
        cln.cln_tx_set_input_amount(r["input_amount"])
        for s in r["sigs"]:
            bs, pk = np.zeros(68, np.uint8), np.zeros(64, np.uint8)
            assert cln.cln_make_tx_sig_args(P(H(s["sig64"], 64)[0]), 1, P(H(s["pub33"], 33)[0]), P(bs), P(pk))
            assert cln.cln_check_tx_sig(tx, 0, None, tal_ws, P(pk), P(bs)) == 1
            assert lib.check_tx_sig(tx, 0, None, tal_ws, P(pk), P(bs)) is True
            bs[10] ^= 1
            assert cln.cln_check_tx_sig(tx, 0, None, tal_ws, P(pk), P(bs)) == 0
            assert lib.check_tx_sig(tx, 0, None, tal_ws, P(pk), P(bs)) is False
        cln.cln_tal_free(tal_ws)
        cln.cln_tx_free(tx)


def test_check_tx_sig_vs_cln_own_on_arbitrary_transactions(engine, ref_live, cln_live):
    """Differential: the engine's check_tx_sig against CLN's OWN unmodified check_tx_sig (bitcoin/signature.c:194-221 over
    libwally's BIP143) on transactions of 1-3 inputs and 1-6 outputs (commitment-like shapes included), scripts from 1 to
    700 bytes (CLN itself asserts on an empty one: libwally refuses a non-NULL zero-length script), every sighash type incl. the ones the gate refuses, witness and non-witness script argument, SIGHASH_SINGLE
    with and without a matching output; signatures made over libwally's sighash with the signature's own type."""
    ref, cln = ref_live, cln_live
    C = _Cln(cln)
    lib = _dropin_tx(engine, cln)
    rng = np.random.default_rng(2026)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))
    seen = {"accept": 0, "reject": 0, "gate": 0}
    for it in range(160):
        nin, nout = int(rng.integers(1, 4)), int(rng.integers(1, 7))
        tx = cln.cln_tx_new(2, int(rng.integers(0, 2)) * int(rng.integers(1, 2**31)))
        for _ in range(nin):
            assert cln.cln_tx_add_input(tx, bytes(rng.integers(0, 256, size=32, dtype=np.uint8)), int(rng.integers(0, 5)),
                                        int(rng.integers(0, 2**32))) == 0
        for _ in range(nout):
            sc = bytes(rng.integers(0, 256, size=int(rng.choice([0, 22, 34, 34, 34, 300])), dtype=np.uint8))
            assert cln.cln_tx_add_output(tx, int(rng.integers(0, 2**40)), sc or None, len(sc)) == 0
        inp = int(rng.integers(0, nin))
        ws = bytes(rng.integers(0, 256, size=int(rng.choice([1, 2, 71, 133, 142, 252, 253, 700])), dtype=np.uint8))
        tal_ws = cln.cln_tal_bytes(ws, len(ws))
        cln.cln_tx_set_input_amount(int(rng.integers(0, 2**45)))
        sht = int(rng.choice([1, 1, 1, 0x83, 0x83, 2, 3, 0x81, 0x82]))
        as_witness = bool(rng.random() < 0.85)
        h = np.zeros(32, np.uint8)
        cln.cln_tx_sighash(tx, inp, tal_ws, sht, P(h))
        sig = np.zeros(64, np.uint8)
        assert ref.ref_ecdsa_sign(P(sk), P(h), P(sig))
        mode = it % 4
        if mode == 1:
            sig[int(rng.integers(0, 64))] ^= 1 << int(rng.integers(0, 8))
        bs, pk = np.zeros(68, np.uint8), np.zeros(64, np.uint8)
        if not cln.cln_make_tx_sig_args(P(sig), sht, P(pub33), P(bs), P(pk)):
            continue  # flipped into r/s >= n: CLN's wire parser would not have produced a struct
        if mode == 2:
            cln.cln_tx_set_input_amount(int(rng.integers(0, 2**45)))  # signed for another amount
        a = (None, tal_ws) if as_witness else (tal_ws, None)
        want = cln.cln_check_tx_sig(tx, inp, a[0], a[1], P(pk), P(bs))
        got = lib.check_tx_sig(tx, inp, a[0], a[1], P(pk), P(bs))
        assert int(got) == want, (it, nin, nout, inp, len(ws), hex(sht), as_witness, mode)
        gate_refuses = sht != 1 and (not as_witness or sht != 0x83)
        if gate_refuses:
            assert want == 0
            seen["gate"] += 1
        else:
            seen["accept" if want else "reject"] += 1
        cln.cln_tal_free(tal_ws)
        cln.cln_tx_free(tx)
    assert seen["accept"] > 30 and seen["reject"] > 30 and seen["gate"] > 10, seen


def test_check_tx_sigs_bip143_batch_through_c_abi(engine, ref, cln):
    """check_tx_sigs_bip143_batch (include/cln_dropin.h) called through the C ABI: BOLT #3's five HTLC transactions with the
    remote HTLC key, then a second batch with per-signature sighash types — the gate of signature.c:206-211 refuses
    everything but ALL and SINGLE|ANYONECANPAY even when the signature itself is good."""
    lib = engine.lib
    recs = _bolt3()
    txs, blob = _svtx_from_bolt3(recs)
    n = len(recs)
    bsigs = np.zeros((n, 68), np.uint8)
    pk = np.zeros(64, np.uint8)
    for i, r in enumerate(recs):
        s = r["sigs"][0]
        assert cln.cln_make_tx_sig_args(P(H(s["sig64"], 64)[0]), 1, P(H(s["pub33"], 33)[0]), P(bsigs[i]), P(pk))
    ok = (ctypes.c_bool * n)()
    lib.check_tx_sigs_bip143_batch(ctypes.byref(txs), blob, ctypes.c_size_t(len(blob)), P(pk), P(bsigs), ctypes.c_size_t(n), ok)
    assert list(ok) == [True] * n
    # per-signature sighash types on synthetic HTLC transactions signed by one key
    rng = np.random.default_rng(5)
    n = 64
    txs, blob = util.make_htlc_txs(rng, n)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))
    bsigs = np.zeros((n, 68), np.uint8)
    want = []
    for i in range(n):
        h = util.cln_sighash(cln, txs[i], blob)
        sig = np.zeros(64, np.uint8)
        assert ref.ref_ecdsa_sign(P(sk), P(h), P(sig))
        if i % 5 == 4:
            sig[33] ^= 2
        assert cln.cln_make_tx_sig_args(P(sig), int(txs[i].sighash_type), P(pub33), P(bsigs[i]), P(pk))
        good = util.ref_verify(ref, 0, h.reshape(1, 32), pub33.reshape(1, 33), sig.reshape(1, 64))[0] == 1
        want.append(bool(good and txs[i].sighash_type in (1, 0x83)))
    ok = (ctypes.c_bool * n)()
    lib.check_tx_sigs_bip143_batch(ctypes.byref(txs), blob, ctypes.c_size_t(len(blob)), P(pk), P(bsigs), ctypes.c_size_t(n), ok)
    assert list(ok) == want
    assert sum(want) > 10 and want.count(False) > 20


def test_sigcheck_update_and_node_batches_and_init_shutdown(engine, cln):
    """sigcheck_channel_update_batch / sigcheck_node_announcement_batch through the C ABI vs gossipd/sigcheck.c compiled
    unmodified; cln_sigverify_shutdown + cln_sigverify_init re-create the drop-ins' context."""
    import struct
    lib = engine.lib
    msgs = gossip.load_subset()
    chans = {}
    for m in msgs:
        if m[:2] == b"\x01\x00":
            flen = struct.unpack(">H", m[258:260])[0]
            p = 260 + flen + 32
            chans[m[p:p + 8]] = (m[p + 8:p + 41], m[p + 41:p + 74])
    cus = [m for m in msgs if m[:2] == b"\x01\x02" and m[98:106] in chans][:300]
    batch = []
    for j, m in enumerate(cus):
        b = bytearray(m)
        if j % 6 == 5:
            b[2 + (j % 64)] ^= 1  # a signature bit
        if j % 50 == 49:
            b = b[:130]  # cut short of the fixed layout
        batch.append(bytes(b))
    batch.append(msgs[0])  # a channel_announcement handed to the channel_update entry point: malformed there
    signers = np.zeros((len(batch), 33), np.uint8)
    want = []
    for i, m in enumerate(batch):
        if m[:2] != b"\x01\x02":
            want.append(-1)
            continue
        nid = chans[bytes(cus[i][98:106])][cus[i][111] & 1]
        signers[i] = np.frombuffer(nid, dtype=np.uint8)
        want.append(cln.cln_sigcheck_channel_update(m, ctypes.c_size_t(len(m)), P(np.ascontiguousarray(signers[i]))))
    arr = (ctypes.c_char_p * len(batch))(*batch)
    lens = (ctypes.c_size_t * len(batch))(*[len(x) for x in batch])
    st = (ctypes.c_int * len(batch))()
    lib.sigcheck_channel_update_batch(arr, lens, P(signers), ctypes.c_size_t(len(batch)), st)
    assert list(st) == want
    assert want.count(0) > 200 and want.count(1) > 30 and want.count(-1) >= 5
    # shutdown drops the process-wide context; init builds a fresh one; results are unchanged
    lib.cln_sigverify_shutdown()
    lib.cln_sigverify_init(0)
    nas = [m for m in msgs if m[:2] == b"\x01\x01"][:120]
    nb = [bytes(bytearray(m[:40]) + bytes([m[40] ^ (1 if j % 7 == 0 else 0)]) + m[41:]) for j, m in enumerate(nas)]
    want = [cln.cln_sigcheck_node_announcement(m, ctypes.c_size_t(len(m))) for m in nb]
    arr = (ctypes.c_char_p * len(nb))(*nb)
    lens = (ctypes.c_size_t * len(nb))(*[len(x) for x in nb])
    st = (ctypes.c_int * len(nb))()
    lib.sigcheck_node_announcement_batch(arr, lens, ctypes.c_size_t(len(nb)), st)
    assert list(st) == want and want.count(1) > 10 and want.count(0) > 90
    lib.cln_sigverify_shutdown()
    lib.cln_sigverify_shutdown()  # idempotent


def test_mixed_kinds_interleaved_config_c3(engine, ref):
    """BASELINE config C3 in miniature: ECDSA (33-byte and x||y keys) and BIP-340 items interleaved by a seeded shuffle
    with a kind tag per item, through sv_verify_mixed_host (device-side split per kind); every verdict vs the reference,
    at sizes on both sides of the small-path threshold; an unknown tag gives verdict 0."""
    w = util.corrupt(util.make_signed(9000, seed=31), every=6)
    rng = np.random.default_rng(6)
    for n in (1, 5, 64, 3000, 9000):
        kinds = rng.choice([0, 0, 1, 2, 2], size=n).astype(np.uint8)
        key = np.zeros((n, 64), np.uint8)
        sig = np.zeros((n, 64), np.uint8)
        want = np.zeros(n, np.uint8)
        for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
            sel = np.nonzero(kinds == kind)[0]
            key[sel, :w[k].shape[1]] = w[k][:n][sel]
            sig[sel] = w[s][:n][sel]
            if sel.size:
                want[sel] = util.ref_verify(ref, kind, np.ascontiguousarray(w["msg"][:n][sel]), np.ascontiguousarray(w[k][:n][sel]),
                                            np.ascontiguousarray(w[s][:n][sel]), threads=4)
        if n >= 64:
            kinds[7] = 9  # not a kind
            want[7] = 0
        got = engine.verify_mixed(kinds, w["msg"][:n], key, sig)
        assert np.array_equal(got, want), n
    assert 0 < want.sum() < want.size


def test_gossip_key_deduplication_same_status(engine, cln):
    """Row N3: a gossip batch repeats node keys heavily; with de-duplication every distinct key is decoded and tabulated once.
    Per-message status must be identical with the search on and off, and equal to gossipd's on a sample; corrupted keys
    (undecodable, flipped) and corrupted signatures included."""
    import struct
    msgs = gossip.load_subset()
    chans = {}
    for m in msgs:
        if m[:2] == b"\x01\x00":
            flen = struct.unpack(">H", m[258:260])[0]
            p = 260 + flen + 32
            chans[m[p:p + 8]] = (m[p + 8:p + 41], m[p + 41:p + 74])
    sel = [m for m in msgs if m[:2] in (b"\x01\x00", b"\x01\x01")] + [m for m in msgs if m[:2] == b"\x01\x02" and m[98:106] in chans]
    sel = sel * 3
    rng = np.random.default_rng(21)
    batch = []
    for m in sel:
        b = bytearray(m)
        if rng.random() < 0.05:
            while True:
                pos = int(rng.integers(2, len(b)))
                if pos not in (66, 67, 258, 259):
                    break
            b[pos] ^= 1 << int(rng.integers(0, 8))
        batch.append(bytes(b))
    signers = np.zeros((len(batch), 33), np.uint8)
    for i, m in enumerate(batch):
        if m[:2] == b"\x01\x02":
            ends = chans.get(bytes(m[98:106]))
            if ends:
                signers[i] = np.frombuffer(ends[m[111] & 1], dtype=np.uint8)
    engine.set_dedup(True)
    a = engine.verify_gossip(batch, signers).copy()
    distinct = engine.last_distinct_keys()
    engine.set_dedup(False)
    b = engine.verify_gossip(batch, signers).copy()
    engine.set_dedup(True)
    assert np.array_equal(a, b)
    items = sum(4 if m[:2] == b"\x01\x00" else 1 for m in batch)
    assert items > 15000 and 0 < distinct < 0.6 * items, (items, distinct)
    for i in rng.choice(len(batch), size=400, replace=False):
        m = batch[i]
        L_ = ctypes.c_size_t(len(m))
        if m[:2] == b"\x01\x00":
            want = cln.cln_sigcheck_channel_announcement(m, L_)
        elif m[:2] == b"\x01\x01":
            want = cln.cln_sigcheck_node_announcement(m, L_)
        else:
            want = cln.cln_sigcheck_channel_update(m, L_, P(np.ascontiguousarray(signers[i])))
        assert a[i] == want, (i, a[i], want)
    assert (a == 0).sum() > 0.8 * len(batch) and (a != 0).sum() > 100


def test_bip340_batch_verification_rlc(engine, ref):
    """Row N3: BIP-340 batch verification by random linear combination on the device.  Every verdict equals the reference's
    per-signature verdict: all-valid batches (every group passes), sparse bad signatures (only their groups fall back to
    one-by-one verification), the 10 %-corrupted mix (every group falls back), encoding failures (excluded, no fallback
    needed), ragged sizes, different seeds and the system's own randomness."""
    n = 5000
    w = util.make_signed(n, seed=88)
    msg, key, sig = w["msg"], w["xonly"], w["ssig"]
    v, gt, gf = engine.verify_schnorr_batch(msg, key, sig, seed32=bytes(range(32)))
    assert v.all() and gt == 5 and gf == 0
    v, gt, gf = engine.verify_schnorr_batch(msg, key, sig)  # seed from getrandom()
    assert v.all() and gf == 0
    for m in (1, 2, 31, 1023, 1024, 1025, 2049):
        v, gt, gf = engine.verify_schnorr_batch(msg[:m], key[:m], sig[:m], seed32=bytes(32))
        assert v.all() and gt == (m + 1023) // 1024 and gf == 0, m
    # sparse damage: three bad signatures in two groups, two encoding failures elsewhere
    m2, k2, s2 = msg.copy(), key.copy(), sig.copy()
    m2[100, 0] ^= 1
    s2[200, 45] ^= 4
    k2[3000] = k2[3001]
    s2[4500, :32] = 255
    k2[4600, :] = 0
    k2[4600, 31] = 5
    want = util.ref_verify(ref, 2, m2, k2, s2, threads=4)
    v, gt, gf = engine.verify_schnorr_batch(m2, k2, s2, seed32=bytes(range(32)))
    assert np.array_equal(v, want) and list(np.nonzero(want == 0)[0]) == [100, 200, 3000, 4500, 4600]
    assert gf == 2  # groups 0 and 2; the encoding failures in group 4 needed no fallback
    # heavy damage: every group falls back, verdicts still exact
    w3 = util.corrupt(util.make_signed(4000, seed=89), every=10)
    want = util.ref_verify(ref, 2, w3["msg"], w3["xonly"], w3["ssig"], threads=4)
    v, gt, gf = engine.verify_schnorr_batch(w3["msg"], w3["xonly"], w3["ssig"], seed32=bytes(32))
    assert np.array_equal(v, want) and gf == gt == 4 and 0 < want.sum() < want.size
    # BIP-340's own vectors (valid and invalid ones in one batch)
    vec = json.load(open(os.path.join(GOLD, "bip340.json")))
    m, k, s = (np.concatenate([H(x[f], z) for x in vec]) for f, z in (("msg32", 32), ("xonly", 32), ("sig64", 64)))
    v, _, _ = engine.verify_schnorr_batch(m, k, s, seed32=bytes(32))
    assert list(v) == [x["expected"] for x in vec]
