"""GPU: the engine against the committed golden vectors, the drop-in (CLN-signature) entry points,
and size-independent properties at the benchmark's full batch size."""
import ctypes
import json
import os

import numpy as np
import pytest

from tests import adversarial, gossip, util

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
P = util.P


def _rows(vec, field, n):
    return np.stack([np.frombuffer(bytes.fromhex(v[field]), dtype=np.uint8) for v in vec]).reshape(len(vec), n)


def test_wycheproof_ecdsa(engine):
    vec = [v for v in json.load(open(os.path.join(GOLD, "wycheproof_ecdsa.json"))) if v["sig64"] is not None]
    assert len(vec) == 273
    want = np.array([v["expected"] for v in vec], np.uint8)
    msg, sig = _rows(vec, "msg32", 32), _rows(vec, "sig64", 64)
    assert np.array_equal(engine.verify(0, msg, _rows(vec, "pub33", 33), sig), want)
    assert np.array_equal(engine.verify(1, msg, _rows(vec, "pubxy", 64), sig), want)


def test_bip340(engine):
    vec = json.load(open(os.path.join(GOLD, "bip340.json")))
    want = np.array([v["expected"] for v in vec], np.uint8)
    got = engine.verify(2, _rows(vec, "msg32", 32), _rows(vec, "xonly", 32), _rows(vec, "sig64", 64))
    assert np.array_equal(got, want)


def test_pubkey_parse_tables(engine):
    vec = [v for v in json.load(open(os.path.join(GOLD, "pubkey_parse.json"))) if "pub33" in v]
    xy, ok = engine.pubkey_parse(_rows(vec, "pub33", 33))
    for i, v in enumerate(vec):
        assert bool(ok[i]) == bool(v["expected"]), v
        if v["expected"]:
            assert bytes(xy[i]).hex() == v["xy"]


def test_adversarial_scalars(engine, ref):
    msg, pub33, pubxy, sig = adversarial.load()
    want = util.ref_verify(ref, 0, msg, pub33, sig)
    assert want.all()
    assert np.array_equal(engine.verify(0, msg, pub33, sig), want)
    assert np.array_equal(engine.verify(1, msg, pubxy, sig), want)
    msg2 = msg.copy()
    msg2[:, 31] ^= 1
    assert np.array_equal(engine.verify(0, msg2, pub33, sig), util.ref_verify(ref, 0, msg2, pub33, sig))


def test_gossip_replay_device_hashing(engine, ref):
    """config C4 in miniature: the mainnet gossip fixture tiled x7, device-side SHA-256d of msg[258:] / msg[66:],
    ~1 % of messages bit-flipped (signatures, keys or signed bytes; never the type/length fields, which CLN's
    wire parser would reject before any signature check); every verdict diffed against the reference."""
    msgs = [bytearray(m) for m in gossip.load_subset() * 7]
    rng = np.random.default_rng(1)
    for mi in rng.choice(len(msgs), size=len(msgs) // 100, replace=False):
        while True:
            pos = int(rng.integers(2, len(msgs[mi])))
            if pos not in (66, 67, 258, 259):
                break
        msgs[mi][pos] ^= 1 << int(rng.integers(0, 8))
    data, off, ln, key, sig, owner, which = gossip.items_of([bytes(m) for m in msgs])
    got = engine.verify_raw(0, data, off, ln, key, sig)
    h = np.zeros((off.size, 32), np.uint8)  # reference: CCAN sha256 twice (sha256_double), then parse + verify
    for i in range(off.size):
        seg = np.ascontiguousarray(data[int(off[i]):int(off[i]) + int(ln[i])])
        ref.ref_sha256d(P(seg), ctypes.c_size_t(seg.size), P(h[i]))
    want = util.ref_verify(ref, 0, h, key, sig, threads=8)
    assert np.array_equal(got, want)
    assert 0 < (want == 0).sum() < want.size // 10


def _dropin(engine):
    lib = engine.lib
    lib.check_signed_hash.restype = ctypes.c_bool
    lib.check_signed_hash_nodeid.restype = ctypes.c_bool
    lib.check_schnorr_sig.restype = ctypes.c_bool
    lib.pubkey_from_der.restype = ctypes.c_bool
    return lib


def test_dropin_cln_signatures(engine, ref):
    """check_signed_hash / check_signed_hash_nodeid / check_schnorr_sig / sha256_double / pubkey_from_der with
    CLN's own argument types (opaque libsecp256k1 structs produced by the reference's parsers)."""
    lib = _dropin(engine)
    w = util.corrupt(util.make_signed(120, seed=99), every=4)
    n_checked = 0
    for i in range(120):
        opk, osig = np.zeros(64, np.uint8), np.zeros(64, np.uint8)
        if not ref.ref_make_opaque_pubkey(P(np.ascontiguousarray(w["pub33"][i])), P(opk)):
            out = np.zeros(64, np.uint8)
            assert not lib.pubkey_from_der(P(np.ascontiguousarray(w["pub33"][i])), ctypes.c_size_t(33), P(out))
            continue
        out = np.zeros(64, np.uint8)
        assert lib.pubkey_from_der(P(np.ascontiguousarray(w["pub33"][i])), ctypes.c_size_t(33), P(out))
        assert np.array_equal(out, opk), "pubkey_from_der must produce the reference's opaque struct"
        if not ref.ref_make_opaque_sig(P(np.ascontiguousarray(w["sig"][i])), P(osig)):
            continue  # CLN refuses such a signature at wire-parse time (wire/fromwire.c:188-199)
        h = np.ascontiguousarray(w["msg"][i])
        want = ref.ref_check_signed_hash_opaque(P(h), P(osig), P(opk))
        assert bool(lib.check_signed_hash(P(h), P(osig), P(opk))) == bool(want), i
        nid = np.ascontiguousarray(w["pub33"][i])
        assert bool(lib.check_signed_hash_nodeid(P(h), P(osig), P(nid))) == bool(want), i
        s = np.ascontiguousarray(w["ssig"][i])
        want_s = ref.ref_check_schnorr_sig_opaque(P(h), P(opk), P(s))
        assert want_s >= 0
        assert bool(lib.check_schnorr_sig(P(h), P(opk), P(s))) == bool(want_s), i
        n_checked += 1
    assert n_checked > 80
    d = np.arange(200, dtype=np.uint8)
    out, want = np.zeros(32, np.uint8), np.zeros(32, np.uint8)
    for ln in (0, 1, 64, 174, 200):
        lib.sha256_double(P(out), P(d), ctypes.c_size_t(ln))
        ref.ref_sha256d(P(d), ctypes.c_size_t(ln), P(want))
        assert np.array_equal(out, want)


def test_dropin_gossip_batch_and_which_signature(engine, ref):
    lib = _dropin(engine)
    m = gossip.chan_ann_3703()
    good = [x for x in gossip.load_subset() if x[:2] == b"\x01\x00"][:50]
    msgs = [m, gossip.strip_features(m)] + good
    bad = bytearray(good[3]); bad[400] ^= 1  # inside bitcoin_key_2 / signed region -> all four fail, first wins
    msgs.append(bytes(bad))
    bad2 = bytearray(good[4]); bad2[2 + 64 * 2 + 5] ^= 1  # corrupt bitcoin_signature_1 only
    msgs.append(bytes(bad2))
    arr = (ctypes.c_char_p * len(msgs))(*msgs)
    lens = (ctypes.c_size_t * len(msgs))(*[len(x) for x in msgs])
    st = (ctypes.c_int * len(msgs))()
    lib.sigcheck_channel_announcement_batch(arr, lens, ctypes.c_size_t(len(msgs)), st)
    st = list(st)
    assert st[0] == 1, "as received: Bad node_signature_1 (run-check_channel_announcement.c:84)"
    assert st[1] == 2, "re-encoded without features: Bad node_signature_2 (:107)"
    assert st[2:52] == [0] * 50
    assert st[52] == 1 and st[53] == 3
    na = [x for x in gossip.load_subset() if x[:2] == b"\x01\x01"][:40]
    nb = bytearray(na[5]); nb[-1] ^= 1
    na.append(bytes(nb))
    arr = (ctypes.c_char_p * len(na))(*na)
    lens = (ctypes.c_size_t * len(na))(*[len(x) for x in na])
    st = (ctypes.c_int * len(na))()
    lib.sigcheck_node_announcement_batch(arr, lens, ctypes.c_size_t(len(na)), st)
    assert list(st) == [0] * 40 + [1]


def test_dropin_htlc_batch_shared_key(engine, ref):
    """channeld's HTLC loop shape: up to 483 signatures by ONE key over distinct sighashes."""
    lib = _dropin(engine)
    n = 483
    rng = np.random.default_rng(4)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, opk = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), None) and ref.ref_make_opaque_pubkey(P(pub33), P(opk))
    hashes = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    sigs = np.zeros((n, 68), np.uint8)  # struct bitcoin_signature: 64-byte opaque sig + enum (4 bytes)
    for i in range(n):
        s64, o = np.zeros(64, np.uint8), np.zeros(64, np.uint8)
        assert ref.ref_ecdsa_sign(P(sk), P(hashes[i]), P(s64)) and ref.ref_make_opaque_sig(P(s64), P(o))
        sigs[i, :64] = o
        sigs[i, 64] = 1
    hashes[17, 0] ^= 1
    sigs[300, 10] ^= 1
    ok = (ctypes.c_bool * n)()
    lib.check_tx_sigs_batch(P(hashes), P(sigs), P(opk), ctypes.c_size_t(n), ok)
    ok = np.array(list(ok))
    assert not ok[17] and not ok[300] and ok.sum() == n - 2


def test_full_size_properties(engine):
    """BASELINE config C2 size (1M): generator output is all-valid; corrupting known positions flips exactly
    those verdicts; verdicts are independent of batch position (shuffle -> same multiset, permuted)."""
    import torch
    n = 1_000_000
    msg = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    key = torch.empty((n, 33), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    ver = torch.empty(n, dtype=torch.uint8, device="cuda")
    engine.synth_device(0, 77, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr())
    engine.verify_device(0, msg.data_ptr(), key.data_ptr(), sig.data_ptr(), n, ver.data_ptr())
    engine.sync()
    assert int(ver.sum().item()) == n
    bad = torch.arange(3, n, 997, device="cuda")
    msg[bad, 7] ^= 0x20
    torch.cuda.synchronize()  # torch's stream produced the inputs; the engine runs on its own stream
    engine.verify_device(0, msg.data_ptr(), key.data_ptr(), sig.data_ptr(), n, ver.data_ptr())
    engine.sync()
    expect = torch.ones(n, dtype=torch.uint8, device="cuda")
    expect[bad] = 0
    assert torch.equal(ver, expect)
    perm = torch.randperm(n, device="cuda")
    m2, k2, s2 = msg[perm].contiguous(), key[perm].contiguous(), sig[perm].contiguous()
    v2 = torch.empty(n, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    engine.verify_device(0, m2.data_ptr(), k2.data_ptr(), s2.data_ptr(), n, v2.data_ptr())
    engine.sync()
    assert torch.equal(v2, expect[perm])


def test_config_c1_dropin_vs_cln_own_functions(engine, ref, cln):
    """Config C1 on the GPU: the same 1k triples through the engine's drop-in check_signed_hash /
    check_signed_hash_nodeid / check_schnorr_sig (CLN argument types, opaque structs built by CLN's own wire
    parsers) must agree call by call with CLN's unmodified functions."""
    lib = _dropin(engine)
    w = util.corrupt(util.make_signed(1000, seed=20260922), every=10)
    agree = 0
    for i in range(1000):
        m, k, s, ss = (np.ascontiguousarray(w[x][i]) for x in ("msg", "pub33", "sig", "ssig"))
        want = cln.cln_check_signed_hash(P(m), P(s), P(k))
        want_id = cln.cln_check_signed_hash_nodeid(P(m), P(s), P(k))
        osig, opk = np.zeros(64, np.uint8), np.zeros(64, np.uint8)
        if cln.cln_make_opaque(P(s), P(k), P(osig), P(opk)):
            assert int(lib.check_signed_hash(P(m), P(osig), P(opk))) == want, i
            assert int(lib.check_schnorr_sig(P(m), P(opk), P(ss))) == cln.cln_check_schnorr_sig(P(m), P(k), P(ss)), i
            agree += 1
        osig2 = np.zeros(64, np.uint8)
        if want_id >= 0 and ref.ref_make_opaque_sig(P(s), P(osig2)):
            assert int(lib.check_signed_hash_nodeid(P(m), P(osig2), P(k))) == want_id, i
    assert agree > 900
    # batch forms vs gossipd/sigcheck.c
    msgs = [x for x in gossip.load_subset() if x[:2] == b"\x01\x00"][:200]
    bad = [bytearray(x) for x in msgs[:40]]
    for j, b in enumerate(bad):
        b[2 + 64 * (j % 4) + 7] ^= 1
    allm = msgs + [bytes(b) for b in bad]
    arr = (ctypes.c_char_p * len(allm))(*allm)
    lens = (ctypes.c_size_t * len(allm))(*[len(x) for x in allm])
    st = (ctypes.c_int * len(allm))()
    lib.sigcheck_channel_announcement_batch(arr, lens, ctypes.c_size_t(len(allm)), st)
    want = [cln.cln_sigcheck_channel_announcement(x, ctypes.c_size_t(len(x))) for x in allm]
    assert list(st) == want


def test_gossip_truncated_but_validly_signed_is_malformed(engine, ref, cln):
    """ADVICE r1: a message cut short of its fixed layout but SIGNED CORRECTLY over the shortened tail must be status -1
    (CLN's generated fromwire_* refuse it), not 0.  channel_update needs all 138 bytes (htlc_maximum_msat is mandatory,
    wire/peer_wire.csv:366-377); node_announcement needs rgb_color, alias, addrlen and addrlen bytes of addresses (:353-362)."""
    import hashlib
    rng = np.random.default_rng(44)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))

    def sign_tail(body_after_sig):
        h = np.frombuffer(hashlib.sha256(hashlib.sha256(body_after_sig).digest()).digest(), dtype=np.uint8).copy()
        sig = np.zeros(64, np.uint8)
        assert ref.ref_ecdsa_sign(P(sk), P(h), P(sig))
        return bytes(sig)

    cu_body = bytes(rng.integers(0, 256, size=72, dtype=np.uint8))  # chain_hash .. htlc_maximum_msat
    na_fixed = b"\x00\x00" + b"\x00\x00\x00\x07" + bytes(pub33) + b"\x01\x02\x03" + bytes(32)  # flen=0, ts, id, rgb, alias
    addrs = bytes([1, 127, 0, 0, 1, 0x26, 0x07])
    na_body = na_fixed + len(addrs).to_bytes(2, "big") + addrs
    msgs, signers = [], []
    for cut in (72, 71, 64, 63, 40):  # full, then shorter and shorter channel_updates, each validly signed as cut
        body = cu_body[:cut]
        msgs.append(b"\x01\x02" + sign_tail(body) + body)
    for cut in (len(na_body), len(na_body) - 1, len(na_fixed) + 2, len(na_fixed) + 1, len(na_fixed), len(na_fixed) - 30, 2 + 4 + 33):
        body = na_body[:cut]
        msgs.append(b"\x01\x01" + sign_tail(body) + body)
    sg = np.tile(pub33, (len(msgs), 1))
    want = []
    for m in msgs:
        L = ctypes.c_size_t(len(m))
        want.append(cln.cln_sigcheck_channel_update(m, L, P(pub33)) if m[:2] == b"\x01\x02" else cln.cln_sigcheck_node_announcement(m, L))
    assert want == [0, -1, -1, -1, -1, 0, -1, -1, -1, -1, -1, -1], want
    assert list(engine.verify_gossip(msgs, sg)) == want


def test_gossip_device_side_slicing_vs_gossipd(engine, cln):
    """Row N1: raw wire messages in, the DEVICE finds signatures/keys/signed regions (k_gossip_slice), hashes and
    verifies; per-message status must equal what CLN's own gossipd/sigcheck.c returns for the same bytes."""
    import struct
    msgs = gossip.load_subset()
    chans = {}
    for m in msgs:
        if m[:2] == b"\x01\x00":
            flen = struct.unpack(">H", m[258:260])[0]
            p = 260 + flen + 32
            chans[m[p:p + 8]] = (m[p + 8:p + 41], m[p + 41:p + 74])
    sel = [m for m in msgs if m[:2] == b"\x01\x00"][:400] + [m for m in msgs if m[:2] == b"\x01\x01"][:200] + \
          [m for m in msgs if m[:2] == b"\x01\x02" and m[98:106] in chans][:300]
    rng = np.random.default_rng(12)
    batch = []
    for m in sel:
        b = bytearray(m)
        if rng.random() < 0.15:
            while True:
                pos = int(rng.integers(2, len(b)))
                if pos not in (66, 67, 258, 259):
                    break
            b[pos] ^= 1 << int(rng.integers(0, 8))
        batch.append(bytes(b))
    batch += [sel[0][:200], sel[401][:60], b"\x01\x03" + bytes(100), b"\x01", sel[5] + b"\x00" * 7,  # malformed / foreign / padded
              sel[601][:137], sel[601][:130], sel[402][:-1], sel[403][:120]]  # cut short of the fixed layout
    signers = np.zeros((len(batch), 33), np.uint8)
    want = []
    for i, m in enumerate(batch):
        L = ctypes.c_size_t(len(m))
        t = m[:2]
        if t == b"\x01\x00":
            want.append(cln.cln_sigcheck_channel_announcement(m, L))
        elif t == b"\x01\x01":
            want.append(cln.cln_sigcheck_node_announcement(m, L))
        elif t == b"\x01\x02" and len(m) >= 138:
            scid = bytes(m[98:106])
            if scid in chans:  # signer by direction bit, as gossmap_manage.c:920-922 selects it
                nid = chans[scid][m[111] & 1]
            else:  # a flip hit the scid: gossipd would not find the channel; feed some key -> must fail
                nid = chans[bytes(sel[600][98:106])][0] if len(sel) > 600 else bytes(33)
            signers[i] = np.frombuffer(nid, dtype=np.uint8)
            want.append(cln.cln_sigcheck_channel_update(m, L, P(np.ascontiguousarray(signers[i]))))
        else:
            want.append(-1)
    got = engine.verify_gossip(batch, signers)
    assert list(got) == want
    assert want.count(0) > 600 and sum(1 for w in want if w > 0) > 50 and want.count(-1) >= 3


def test_htlc_loop_device_side_bip143(engine, ref, cln):
    """Row N2: channeld's per-HTLC loop with the BIP143 sighash computed on the device: 483 HTLC transactions signed by
    one key (the reference signs libwally's sighash); sighashes must equal libwally's, verdicts the reference's."""
    n = 483
    rng = np.random.default_rng(77)
    txs, blob = util.make_htlc_txs(rng, n)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))
    sig = np.zeros((n, 64), np.uint8)
    want_hash = np.zeros((n, 32), np.uint8)
    for i in range(n):
        want_hash[i] = util.cln_sighash(cln, txs[i], blob)
        assert ref.ref_ecdsa_sign(P(sk), P(want_hash[i]), P(sig[i]))
    sig[100, 3] ^= 1
    txs[200].output_amount += 1      # a different transaction than the one that was signed
    txs[300].sighash_type = 0x183    # libwally refuses sighash bits above the low byte (tx_io.c:682) -> verdict 0
    keys = np.tile(pubxy, (n, 1))
    got, sh = engine.check_tx_sigs(1, txs, blob, keys, sig, want_sighash=True)
    ok = np.ones(n, bool); ok[[100, 200, 300]] = False
    assert np.array_equal(sh[[i for i in range(n) if i not in (200, 300)]], want_hash[[i for i in range(n) if i not in (200, 300)]])
    assert np.array_equal(got.astype(bool), ok)
    got33 = engine.check_tx_sigs(0, txs, blob, np.tile(pub33, (n, 1)), sig)
    assert np.array_equal(got33, got)


def test_host_api_chunking_and_pipelining(engine):
    """sv_verify_host above its internal chunk size (2^21) and with slice pipelining: 2.2 M synthesised signatures
    copied to (pageable) host memory, a few corrupted, verified through the host-buffer API."""
    import torch
    n = 2_200_000
    msg = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    key = torch.empty((n, 33), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    engine.synth_device(0, 4242, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr())
    engine.sync()
    m, k, s = msg.cpu().numpy(), key.cpu().numpy(), sig.cpu().numpy()
    bad = np.array([0, 1, 151551, 151552, 757759, 757760, 2097151, 2097152, 2097153, n - 1])
    m[bad, 9] ^= 0x40
    got = engine.verify(0, m, k, s)
    want = np.ones(n, np.uint8)
    want[bad] = 0
    assert np.array_equal(got, want)


def test_samekey_batch(engine, ref):
    """Row N3 on the GPU: 483 (and ragged counts of) signatures by one key through sv_verify_samekey_host."""
    rng = np.random.default_rng(8)
    sk = rng.integers(1, 256, size=32, dtype=np.uint8)
    pub33, pubxy = np.zeros(33, np.uint8), np.zeros(64, np.uint8)
    assert ref.ref_pubkey_create(P(sk), P(pub33), P(pubxy))
    for n in (1, 31, 33, 483, 5000):
        msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
        sig = np.zeros((n, 64), np.uint8)
        for i in range(n):
            assert ref.ref_ecdsa_sign(P(sk), P(msg[i]), P(sig[i]))
        for i in range(0, n, 7):
            msg[i, i % 32] ^= 2
        want = util.ref_verify(ref, 0, msg, np.tile(pub33, (n, 1)), sig)
        assert np.array_equal(engine.verify_samekey(0, pub33, msg, sig), want), n
        assert np.array_equal(engine.verify_samekey(1, pubxy, msg, sig), want), n
    bad = pub33.copy(); bad[5] ^= 1  # very likely not a curve point, certainly not the signer
    assert not engine.verify_samekey(0, bad, msg, sig).any()


def test_verifier_subdaemon(ref, cln, tmp_path):
    """Row N4: one GPU-owning process serving many clients over a unix socket with CLN-style framing (wire CSV codec),
    coalescing the requests of ALL clients into shared launches: 8 clients x 40 requests in flight, every verdict vs the
    reference; the daemon's own counters must show fewer launches than requests; gossip requests, malformed requests
    (answered with sigverifyd_error, connection kept), an absurd length prefix (connection closed, the others unaffected),
    socket mode 0600, and the inherited-fd mode lightningd would use."""
    import socket, stat, struct, subprocess, threading, time
    from lightning_b200 import build
    from lightning_b200 import sigverifyd_wire as W
    sock_path = str(tmp_path / "sv.sock")
    proc = subprocess.Popen([build.DAEMON, sock_path, "0"], stderr=subprocess.PIPE)
    try:
        for _ in range(600):
            if os.path.exists(sock_path):
                break
            time.sleep(0.1)
        assert os.path.exists(sock_path), "daemon did not come up"
        assert stat.S_IMODE(os.stat(sock_path).st_mode) == 0o600
        w = util.corrupt(util.make_signed(2400, seed=21), every=6)
        kinds = [(0, "pub33", "sig", 33), (1, "pubxy", "sig", 64), (2, "xonly", "ssig", 32)]
        want = [util.ref_verify(ref, k, w["msg"], w[kk], w[ss]) for k, kk, ss, _ in kinds]
        errors = []

        def client(ci):
            try:
                c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
                c.connect(sock_path)
                reqs = []
                for j in range(40):  # all requests of this client are sent before any reply is read
                    kind, kk, ss, ks = kinds[(ci + j) % 3]
                    lo = (ci * 40 + j) * 7 % 2300
                    n = 1 + (ci + j) % 60
                    sl = slice(lo, lo + n)
                    c.sendall(W.encode("sigverifyd_verify", req_id=ci * 1000 + j, kind=kind, n=n, hashes=w["msg"][sl].tobytes(),
                                       keylen=n * ks, keys=w[kk][sl].tobytes(), sigs=w[ss][sl].tobytes()))
                    reqs.append((ci * 1000 + j, kind, sl))
                got = {}
                for _ in reqs:
                    name, v = W.read_msg(c)
                    assert name == "sigverifyd_verify_reply", name
                    got[v["req_id"]] = v
                for rid, kind, sl in reqs:
                    assert np.array_equal(np.frombuffer(got[rid]["verdicts"], dtype=np.uint8), want[kind][sl]), (rid, kind)
                c.close()
            except Exception as ex:  # noqa: BLE001
                errors.append((ci, repr(ex)))
        th = [threading.Thread(target=client, args=(i,)) for i in range(8)]
        for t in th:
            t.start()
        for t in th:
            t.join(timeout=120)
        assert not errors, errors
        c = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        c.connect(sock_path)
        c.sendall(W.encode("sigverifyd_stats", req_id=5))
        name, st = W.read_msg(c)
        assert name == "sigverifyd_stats_reply" and st["requests"] == 320
        assert st["launches"] < st["requests"] and st["max_coalesced"] >= 2, st  # requests of different clients shared launches
        # malformed requests are answered, not fatal: bad kind, key bytes that do not match n
        c.sendall(W.encode("sigverifyd_verify", req_id=77, kind=9, n=0, hashes=b"", keylen=0, keys=b"", sigs=b""))
        assert W.read_msg(c) == ("sigverifyd_error", dict(req_id=77, code=1))
        c.sendall(W.encode("sigverifyd_verify", req_id=78, kind=0, n=1, hashes=bytes(32), keylen=32, keys=bytes(32), sigs=bytes(64)))
        assert W.read_msg(c) == ("sigverifyd_error", dict(req_id=78, code=1))
        # a gossip request: raw messages in, status per message out (255 = malformed), vs gossipd/sigcheck.c
        msgs = [m for m in gossip.load_subset() if m[:2] in (b"\x01\x00", b"\x01\x01")][:60]
        msgs[3] = msgs[3][:2] + bytes([msgs[3][2] ^ 1]) + msgs[3][3:]
        msgs[9] = msgs[9][:100]
        c.sendall(W.encode("sigverifyd_gossip", req_id=6, n=len(msgs), lens=[len(m) for m in msgs], signers=bytes(33 * len(msgs)),
                           bloblen=sum(len(m) for m in msgs), blob=b"".join(msgs)))
        name, g = W.read_msg(c)
        ref_status = []
        for m in msgs:
            L_ = ctypes.c_size_t(len(m))
            r = cln.cln_sigcheck_channel_announcement(m, L_) if m[:2] == b"\x01\x00" else cln.cln_sigcheck_node_announcement(m, L_)
            ref_status.append(255 if r < 0 else r)
        assert name == "sigverifyd_gossip_reply" and list(g["status"]) == ref_status
        # an absurd length prefix closes THAT connection; the daemon keeps serving the others
        bad = socket.socket(socket.AF_UNIX, socket.SOCK_STREAM)
        bad.connect(sock_path)
        bad.sendall(struct.pack(">I", 0xFFFFFFF0) + b"xx")
        assert bad.recv(4) == b""
        c.sendall(W.encode("sigverifyd_stats", req_id=8))
        assert W.read_msg(c)[0] == "sigverifyd_stats_reply"
        c.close()
    finally:
        proc.terminate()
        proc.wait(timeout=10)
    # inherited-fd mode: one end of a socketpair handed to the child, as lightningd does for its subdaemons
    a, b = socket.socketpair(socket.AF_UNIX, socket.SOCK_STREAM)
    proc = subprocess.Popen([build.DAEMON, "--fd", str(b.fileno()), "0"], pass_fds=[b.fileno()], stderr=subprocess.PIPE)
    b.close()
    try:
        a.settimeout(120)
        sl = slice(0, 5)
        a.sendall(W.encode("sigverifyd_verify", req_id=1, kind=0, n=5, hashes=w["msg"][sl].tobytes(), keylen=165,
                           keys=w["pub33"][sl].tobytes(), sigs=w["sig"][sl].tobytes()))
        name, v = W.read_msg(a)
        assert name == "sigverifyd_verify_reply" and np.array_equal(np.frombuffer(v["verdicts"], dtype=np.uint8), want[0][sl])
        a.close()
        assert proc.wait(timeout=30) == 0  # the parent went away: the daemon exits by itself
    finally:
        if proc.poll() is None:
            proc.terminate()
            proc.wait(timeout=10)
