#!/usr/bin/env python3
"""Generate the committed golden fixtures from the reference tree (run HERE, where /root/reference
exists; the GPU box only sees the generated files).  Vectors are data, not code:

  wycheproof_ecdsa.json   463 Wycheproof ECDSA secp256k1/SHA-256 "bitcoin" vectors
                          (src/wycheproof/ecdsa_secp256k1_sha256_bitcoin_test.json; driver tests.c:7415-7442),
                          DER signatures converted to the 64-byte compact form with the reference's own
                          strict DER parser (vectors it refuses to parse keep sig64 = null, verdict 0)
  bip340.json             BIP-340 vectors 0-14 as embedded in modules/schnorrsig/tests_impl.h:206-628
  pubkey_parse.json       valid / invalid 33-byte encodings from tests.c run_ec_pubkey_parse_test (:5893-)
  gossip_subset.bin/.json a slice of tests/data/routing_gossip_store (real mainnet channel_announcement,
                          node_announcement, channel_update messages; all signatures valid under the reference)
  routing_gossip_store    the reference's tests/data/routing_gossip_store itself (11,796 channel_announcements, 2,175
                          node_announcements, 9,703 channel_updates), copied byte for byte for the full-size C4 replay
  chan_ann_3703.json      the mainnet channel_announcement of gossipd/test/run-check_channel_announcement.c
  ecmult_kat.json         the two digests of tests.c:5657-5726 (SHA-256 over x*G for derived scalars)
  ecdsa_edge_cases.json   the verification cases of test_ecdsa_edge_cases (tests.c:7069-7297): R = infinity, r = 0, s = 0,
                          message 0 / 1 / -1 with crafted keys, the r + n wrap boundary (r = p - n), the nonce n-1 signature
                          of key 1, an all-0xff compact signature — as (msg32, pub33, sig64) triples.  The reference
                          calls its INTERNAL secp256k1_ecdsa_sig_verify there (no low-S rule); each triple records that
                          internal expectation as the source states it AND the public-API verdict (parse + low-S rule,
                          what CLN and the engine implement) obtained from oracle/_ref.  (:7300-7406 are nonce-function and
                          key-export cases of the SIGNING side: not on the verification path.)
  bolt3_htlc_txs.json     BOLT #3 Appendix C "commitment tx with all five HTLCs untrimmed (minimum feerate)": the five fully
                          signed HTLC transactions embedded in channeld/test/run-full_channel.c:635-673 (hex), parsed into
                          the fields BIP143 commits to, with both the remote and the local HTLC signature of each
  bip143_libwally.json    libwally's BIP143 sighash (CLN's bitcoin_tx_hash_for_sig, oracle/_ref) of 120 seeded random
                          transactions of 1-3 inputs and 1-6 outputs

Every expected verdict written here is re-checked against oracle/_ref (the unmodified reference) at
generation time.
"""
import ctypes
import hashlib
import json
import os
import re
import struct
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import util  # noqa: E402

REF = "/root/reference"
S = REF + "/external/libwally-core/src/secp256k1"
OUT = os.path.dirname(os.path.abspath(__file__))
ref = util.load_ref()
P = util.P


def arr(b):
    return np.frombuffer(bytes(b), dtype=np.uint8).copy()


def wycheproof():
    j = json.load(open(S + "/src/wycheproof/ecdsa_secp256k1_sha256_bitcoin_test.json"))
    out = []
    for g in j["testGroups"]:
        # "publicKey" (newer schema) or "key"
        keyobj = g.get("publicKey") or g.get("key")
        pk = bytes.fromhex(keyobj["uncompressed"])
        p33 = np.zeros(33, np.uint8)
        pxy = np.zeros(64, np.uint8)
        assert ref.ref_pubkey_convert(P(arr(pk)), ctypes.c_size_t(len(pk)), P(p33), P(pxy))
        for t in g["tests"]:
            msg = bytes.fromhex(t["msg"])
            h = hashlib.sha256(msg).digest()
            der = bytes.fromhex(t["sig"])
            s64 = np.zeros(64, np.uint8)
            ok = ref.ref_sig_der_to_compact(P(arr(der if der else b'\x00')), ctypes.c_size_t(len(der)), P(s64))
            exp = 1 if t["result"] == "valid" else 0
            assert t["result"] in ("valid", "invalid")
            if ok:
                got = util.ref_verify(ref, 0, arr(h).reshape(1, 32), p33.reshape(1, 33), s64.reshape(1, 64))[0]
            else:
                got = 0
            assert got == exp, (t["tcId"], got, exp)
            out.append(dict(tcId=t["tcId"], comment=t.get("comment", ""), msg32=h.hex(), pub33=bytes(p33).hex(),
                            pubxy=bytes(pxy).hex(), sig64=bytes(s64).hex() if ok else None, expected=exp))
    assert len(out) == 463, len(out)
    json.dump(out, open(OUT + "/wycheproof_ecdsa.json", "w"), indent=0)
    print("wycheproof:", len(out), "vectors,", sum(1 for o in out if o["sig64"]), "DER-parseable,",
          sum(o["expected"] for o in out), "valid")


def c_array(block, name):
    m = re.search(r"const unsigned char " + name + r"\[(?:32|64)?\]\s*=\s*\{([^}]*)\}", block)
    if not m:
        return None
    return bytes(int(x, 16) for x in re.findall(r"0x([0-9A-Fa-f]{2})", m.group(1)))


def bip340():
    src = open(S + "/src/modules/schnorrsig/tests_impl.h").read()
    start = src.index("static void test_schnorrsig_bip_vectors(void)")
    body = src[start:]
    blocks = re.split(r"/\* Test vector (\d+) \*/", body)
    out = []
    for i in range(1, len(blocks), 2):
        num, blk = int(blocks[i]), blocks[i + 1]
        if num > 14:
            break  # 15-18 use messages that are not 32 bytes; CLN always signs 32-byte hashes (signature.c:428)
        pk, msg, sig = c_array(blk, "pk"), c_array(blk, "msg"), c_array(blk, "sig")
        m = re.search(r"check_verify\(pk, msg, sizeof\(msg\), sig, (\d)\)", blk)
        if m:
            exp = int(m.group(1))
        else:
            assert "CHECK(!secp256k1_xonly_pubkey_parse" in blk, num
            exp, msg, sig = 0, bytes(32), bytes(64)
        got = util.ref_verify(ref, 2, arr(msg).reshape(1, 32), arr(pk).reshape(1, 32), arr(sig).reshape(1, 64))[0]
        assert got == exp, (num, got, exp)
        out.append(dict(index=num, xonly=pk.hex(), msg32=msg.hex(), sig64=sig.hex(), expected=exp))
    assert [o["index"] for o in out] == list(range(15))
    json.dump(out, open(OUT + "/bip340.json", "w"), indent=0)
    print("bip340:", len(out), "vectors,", sum(o["expected"] for o in out), "valid")


def pubkey_parse():
    src = open(S + "/src/tests.c").read()
    start = src.index("static void run_ec_pubkey_parse_test(void)")
    body = src[start:start + 40000]
    out = []
    for name, exp in (("valid", 1), ("invalid", 0)):
        m = re.search(r"const unsigned char " + name + r"\[\w+\]\[64\]\s*=\s*\{(.*?)\n    \};", body, re.S)
        rows = re.findall(r"\{([^{}]*)\}", m.group(1), re.S)
        for r in rows:
            xy = bytes(int(x, 16) for x in re.findall(r"0x([0-9A-Fa-f]{2})", r))
            assert len(xy) == 64
            # the reference test prepends 0x02/0x03 according to y parity for the compressed form
            for pfx in (2, 3):
                k = bytes([pfx]) + xy[:32]
                o33 = np.zeros(33, np.uint8)
                oxy = np.zeros(64, np.uint8)
                got = ref.ref_pubkey_convert(P(arr(k)), ctypes.c_size_t(33), P(o33), P(oxy))
                out.append(dict(pub33=k.hex(), expected=int(bool(got)), xy=bytes(oxy).hex() if got else None, table=name))
            k65 = arr(b"\x04" + xy)
            got65 = ref.ref_pubkey_convert(P(k65), ctypes.c_size_t(65), P(np.zeros(33, np.uint8)), P(np.zeros(64, np.uint8)))
            assert bool(got65) == bool(exp), (name, xy.hex())
            out.append(dict(pubxy=xy.hex(), expected=int(bool(got65)), table=name))
    json.dump(out, open(OUT + "/pubkey_parse.json", "w"), indent=0)
    print("pubkey_parse:", len(out), "encodings,", sum(o["expected"] for o in out), "valid")


WIRE_CHANNEL_ANNOUNCEMENT, WIRE_NODE_ANNOUNCEMENT, WIRE_CHANNEL_UPDATE = 256, 257, 258


def parse_gossip_store(path):
    """common/gossip_store.h:15-51 — 1 version byte, then records: be16 flags, be16 len, be32 crc, be32 ts, msg."""
    data = open(path, "rb").read()
    pos, msgs = 1, []
    while pos + 12 <= len(data):
        flags, ln, crc, ts = struct.unpack(">HHII", data[pos:pos + 12])
        msg = data[pos + 12:pos + 12 + ln]
        pos += 12 + ln
        if len(msg) >= 2:
            msgs.append((struct.unpack(">H", msg[:2])[0], msg))
    return msgs


def gossip_items(msgs):
    """Expand gossip messages into signature items exactly as gossipd/sigcheck.c does:
    channel_announcement: hash msg[258:], sigs at 2,66,130,194 by node_id_1, node_id_2, bitcoin_key_1, bitcoin_key_2
    node_announcement:    hash msg[66:],  sig at 2, key = node_id (after flen+features and timestamp)
    channel_update:       hash msg[66:],  sig at 2, key = node_id_{1|2} of the channel by channel_flags & 1"""
    chans = {}
    items = []  # (msg_index, hash_off, sig_off, key33)
    for mi, (typ, m) in enumerate(msgs):
        if typ == WIRE_CHANNEL_ANNOUNCEMENT:
            flen = struct.unpack(">H", m[258:260])[0]
            p = 260 + flen + 32
            scid = m[p:p + 8]
            p += 8
            keys = [m[p + 33 * k:p + 33 * k + 33] for k in range(4)]
            chans[scid] = (keys[0], keys[1])
            for k in range(4):
                items.append((mi, 258, 2 + 64 * k, keys[k]))
        elif typ == WIRE_NODE_ANNOUNCEMENT:
            flen = struct.unpack(">H", m[66:68])[0]
            p = 68 + flen + 4
            items.append((mi, 66, 2, m[p:p + 33]))
        elif typ == WIRE_CHANNEL_UPDATE:
            scid = m[2 + 64 + 32:2 + 64 + 32 + 8]
            chflags = m[2 + 64 + 32 + 8 + 4 + 1]
            if scid in chans:
                items.append((mi, 66, 2, chans[scid][chflags & 1]))
    return items


def gossip():
    msgs = parse_gossip_store(REF + "/tests/data/routing_gossip_store")
    counts = {}
    for t, _ in msgs:
        counts[t] = counts.get(t, 0) + 1
    print("gossip_store message types:", counts)
    # subset: first 1500 channel_announcements, the updates that reference them, first 400 node_announcements
    keep, nca, nna, ncu, scids = [], 0, 0, 0, set()
    for typ, m in msgs:
        if typ == WIRE_CHANNEL_ANNOUNCEMENT and nca < 1500:
            flen = struct.unpack(">H", m[258:260])[0]
            scids.add(m[260 + flen + 32:260 + flen + 40])
            keep.append((typ, m)); nca += 1
        elif typ == WIRE_NODE_ANNOUNCEMENT and nna < 400:
            keep.append((typ, m)); nna += 1
        elif typ == WIRE_CHANNEL_UPDATE and ncu < 1200 and m[98:106] in scids:
            keep.append((typ, m)); ncu += 1
    items = gossip_items(keep)
    # verify everything with the reference (sha256d + parse + verify)
    n = len(items)
    msg32 = np.zeros((n, 32), np.uint8); key = np.zeros((n, 33), np.uint8); sig = np.zeros((n, 64), np.uint8)
    for i, (mi, hoff, soff, k) in enumerate(items):
        m = keep[mi][1]
        tail = arr(m[hoff:])
        ref.ref_sha256d(P(tail), ctypes.c_size_t(tail.size), P(msg32[i]))
        key[i] = arr(k); sig[i] = arr(m[soff:soff + 64])
    v = util.ref_verify(ref, 0, msg32, key, sig)
    assert v.all(), f"{n - v.sum()} fixture signatures fail under the reference"
    blob = b"".join(struct.pack(">H", len(m)) + m for _, m in keep)
    open(OUT + "/gossip_subset.bin", "wb").write(blob)
    json.dump(dict(source="tests/data/routing_gossip_store (reference v26.04.1)", format="repeat: be16 len, wire message",
                   channel_announcements=nca, node_announcements=nna, channel_updates=ncu, signatures=n,
                   all_valid_under_reference=True, full_store_counts={str(k): v for k, v in counts.items()}),
              open(OUT + "/gossip_subset.json", "w"), indent=1)
    print("gossip subset:", nca, "CA,", nna, "NA,", ncu, "CU ->", n, "signatures, all valid;", len(blob), "bytes")


def gossip_store_full():
    """The whole fixture, byte for byte (7.6 MB): config C4 replays ALL of it (bench.py --config c4, tests/test_gpu_c4.py)."""
    import shutil
    shutil.copyfile(REF + "/tests/data/routing_gossip_store", OUT + "/routing_gossip_store")
    msgs = parse_gossip_store(OUT + "/routing_gossip_store")
    print("routing_gossip_store:", os.path.getsize(OUT + "/routing_gossip_store"), "bytes,", len(msgs), "records")


def chan_ann_3703():
    src = open(REF + "/gossipd/test/run-check_channel_announcement.c").read()
    m = re.search(r'tal_hexdata\(\w+,\s*"([0-9a-f]+)"', src)
    if not m:
        hexes = re.findall(r'"([0-9a-f]{64,})"', src)
        h = "".join(hexes)
    else:
        h = m.group(1)
    json.dump(dict(source="gossipd/test/run-check_channel_announcement.c (issue #3703, scid 628813x1594x1)", msg=h),
              open(OUT + "/chan_ann_3703.json", "w"), indent=1)
    print("chan_ann_3703:", len(h) // 2, "bytes")


def ecmult_kat():
    src = open(S + "/src/tests.c").read()
    def digest(name):
        m = re.search(r"static const unsigned char " + name + r"\[32\] = \{(.*?)\};", src, re.S)
        return bytes(int(x, 16) for x in re.findall(r"0x([0-9a-f]{2})", m.group(1))).hex()
    out = [dict(prefix=4808378, iters=1024, sha256=digest("expected32_6bit20")),
           dict(prefix=1607366309, iters=2048, sha256=digest("expected32_8bit8"))]
    json.dump(out, open(OUT + "/ecmult_kat.json", "w"), indent=1)
    print("ecmult_kat:", out)


def c_bytes(block, name):
    m = re.search(r"unsigned char " + name + r"\[\d*\]\s*=\s*\{([^}]*)\}", block)
    assert m, name
    return bytes(int(x, 16) for x in re.findall(r"0[xX]([0-9A-Fa-f]{2})", m.group(1)))


def ecdsa_edge_cases():
    from tests import adversarial as A
    N = util.N_ORDER
    src = open(S + "/src/tests.c").read()
    body = src[src.index("static void test_ecdsa_edge_cases(void)"):src.index("/* Nonce function corner cases. */")]
    blk = {}
    for title, key in (("Verify signature with r of zero fails", "r0"), ("Verify signature with s of zero fails", "s0"),
                       ("Verify signature with message 0 passes", "m0"), ("Verify signature with message 1 passes", "m1"),
                       ("Verify signature with message -1 passes", "mm1"), ("Signature where s would be zero", "sz")):
        i = body.index("/* " + title)
        blk[key] = body[i:body.index("\n    }\n", i)]
    b32 = lambda v: (v % 2**256).to_bytes(32, "big")
    inv = lambda v: pow(v, N - 2, N)
    G33 = bytes([2 + (A.GY & 1)]) + A.GX.to_bytes(32, "big")
    cases = []

    def add(name, pub33, r, s, m, internal, note=""):
        cases.append(dict(name=name, pub33=pub33.hex(), sig64=(b32(r) + b32(s)).hex(), msg32=b32(m).hex(), internal_sig_verify=internal, note=note))

    # tests.c:7073-7087: ss = (-1)^-1, sr = 1, key = 1*G, msg = ss -> the recomputed point is infinity
    add("infinity (s = -1: high)", G33, 1, inv(N - 1), inv(N - 1), 0)
    add("infinity, low-S form (r = 1, s = 1, m = -1, key G)", G33, 1, 1, N - 1, 0, "same point at infinity with a low s, so the public API reaches the branch too")
    add("r = 0", c_bytes(blk["r0"], "pubkey_mods_zero"), 0, 1, 0, 0)
    add("s = 0", c_bytes(blk["s0"], "pubkey"), 1, 0, 0, 0)
    for nm in ("pubkey", "pubkey2"):
        k = c_bytes(blk["m0"], nm)
        add(f"message 0, {nm}, s = 2", k, 2, 2, 0, 1)
        add(f"message 0, {nm}, s = -2", k, 2, N - 2, 0, 1, "valid for the internal function, high-S for the API")
        add(f"message 0, {nm}, s = 1", k, 2, 1, 0, 0)
    csr = int.from_bytes(c_bytes(blk["m1"], "csr"), "big")
    for nm in ("pubkey", "pubkey2"):
        k = c_bytes(blk["m1"], nm)
        add(f"message 1, {nm}, s = 1", k, csr, 1, 1, 1)
        add(f"message 1, {nm}, s = -1", k, csr, N - 1, 1, 1, "valid for the internal function, high-S for the API")
        add(f"message 1, {nm}, s = 1/2", k, csr, inv(2), 1, 0)
    csr = int.from_bytes(c_bytes(blk["mm1"], "csr"), "big")
    assert csr == util.P_FIELD - N  # r = p - n: the second x candidate r + n is NOT allowed (ecdsa_impl.h:253)
    k = c_bytes(blk["mm1"], "pubkey")
    add("message -1, r = p - n, s = 1", k, csr, 1, N - 1, 1)
    add("message -1, r = p - n, s = -1", k, csr, N - 1, N - 1, 1, "valid for the internal function, high-S for the API")
    add("message -1, r = p - n, s = 1/3", k, csr, inv(3), N - 1, 0)
    # tests.c:7232-7268: key = 1, nonce = n - 1 (nonce2), msg[31] = 0xaa: signing succeeds and the signature verifies
    msg = bytearray(c_bytes(blk["sz"], "msg"))
    msg[31] = 0xAA
    m = int.from_bytes(msg, "big")
    kk = int.from_bytes(c_bytes(blk["sz"], "nonce2"), "big")
    R = A.mul(kk, A.G)
    r = R[0] % N
    sv = inv(kk) * (m + r * 1) % N
    if sv > N // 2:
        sv = N - sv
    add("key 1, nonce n-1 (tests.c:7251-7258)", G33, r, sv, m, 1)
    cases.append(dict(name="compact signature of 64 x 0xff does not parse (tests.c:7296)", pub33=G33.hex(), sig64=(b"\xff" * 64).hex(),
                      msg32=bytes(msg).hex(), internal_sig_verify=None, note="secp256k1_ecdsa_signature_parse_compact == 0"))
    for c in cases:
        got = int(util.ref_verify(ref, 0, arr(bytes.fromhex(c["msg32"])).reshape(1, 32), arr(bytes.fromhex(c["pub33"])).reshape(1, 33),
                                  arr(bytes.fromhex(c["sig64"])).reshape(1, 64))[0])
        c["expected"] = got
        s_val = int(c["sig64"][64:], 16)
        if c["internal_sig_verify"] is not None and s_val <= N // 2:
            assert got == c["internal_sig_verify"], c  # with a low s the public API and the internal function agree
        if s_val > N // 2:
            assert got == 0, c
    assert sum(c["expected"] for c in cases) >= 6
    json.dump(cases, open(OUT + "/ecdsa_edge_cases.json", "w"), indent=0)
    print("ecdsa_edge_cases:", len(cases), "triples,", sum(c["expected"] for c in cases), "valid under the public API")


def parse_tx_hex(h):
    """segwit serialisation -> dict (version, ins[(txid, index, sequence)], outs[(amount, script)], witness[in][items], locktime)"""
    b = bytes.fromhex(h)
    pos = 0

    def rd(n):
        nonlocal pos
        v = b[pos:pos + n]
        pos += n
        return v

    def varint():
        v = rd(1)[0]
        if v < 0xfd:
            return v
        return int.from_bytes(rd({0xfd: 2, 0xfe: 4, 0xff: 8}[v]), "little")
    version = int.from_bytes(rd(4), "little")
    assert rd(2) == b"\x00\x01"
    ins = []
    for _ in range(varint()):
        txid = rd(32)
        idx = int.from_bytes(rd(4), "little")
        rd(varint())
        ins.append((txid, idx, int.from_bytes(rd(4), "little")))
    outs = []
    for _ in range(varint()):
        amt = int.from_bytes(rd(8), "little")
        outs.append((amt, rd(varint())))
    wit = [[rd(varint()) for _ in range(varint())] for _ in ins]
    locktime = int.from_bytes(rd(4), "little")
    assert pos == len(b)
    return dict(version=version, ins=ins, outs=outs, witness=wit, locktime=locktime)


def bolt3_htlc_txs():
    cln = util.load_cln()
    src = open(REF + "/channeld/test/run-full_channel.c").read()
    hexes = re.findall(r'raw_tx = tx_from_hex\(tmpctx, "([0-9a-f]+)"\);', src)
    names = re.findall(r"\*\s+(htlc_(?:success|timeout)_tx \(htlc #\d\)): [0-9a-f]+", src)
    assert len(hexes) == 5 and len(names) == 5
    # BOLT #3 Appendix C: htlc amounts 1000000 / 2000000 / 2000000 / 3000000 / 4000000 msat; at feerate 0 an HTLC transaction
    # spends its commitment output without a fee, so the input amount equals the single output's
    out = []
    for name, hx in zip(names, hexes):
        t = parse_tx_hex(hx)
        assert len(t["ins"]) == 1 and len(t["outs"]) == 1
        w = t["witness"][0]
        assert len(w) == 5 and w[0] == b""
        wscript = w[4]
        keys = re.findall(rb"\x21([\x02\x03].{32})", wscript, re.S)
        assert len(keys) == 2  # remote_htlcpubkey, local_htlcpubkey (bitcoin/script.c:732,849)
        rec = dict(name=name, hex=hx, version=t["version"], locktime=t["locktime"], prev_txid=t["ins"][0][0].hex(),
                   prev_index=t["ins"][0][1], sequence=t["ins"][0][2], input_amount=t["outs"][0][0], output_amount=t["outs"][0][0],
                   out_script=t["outs"][0][1].hex(), wscript=wscript.hex(), sigs=[])
        sh = np.zeros(32, np.uint8)
        rc = cln.cln_htlc_sighash(ctypes.c_uint32(t["version"]), ctypes.c_uint32(t["locktime"]), t["ins"][0][0], ctypes.c_uint32(t["ins"][0][1]),
                                  ctypes.c_uint32(t["ins"][0][2]), wscript, ctypes.c_size_t(len(wscript)), ctypes.c_uint64(t["outs"][0][0]),
                                  ctypes.c_uint64(t["outs"][0][0]), t["outs"][0][1], ctypes.c_size_t(len(t["outs"][0][1])), ctypes.c_uint32(1), P(sh))
        assert rc == 0
        rec["sighash"] = bytes(sh).hex()
        for who, der, key in (("remote_htlc_signature", w[1], keys[0]), ("local_htlc_signature", w[2], keys[1])):
            assert der[-1] == 1  # SIGHASH_ALL
            s64 = np.zeros(64, np.uint8)
            assert ref.ref_sig_der_to_compact(P(arr(der[:-1])), ctypes.c_size_t(len(der) - 1), P(s64))
            got = int(util.ref_verify(ref, 0, sh.reshape(1, 32), arr(key).reshape(1, 33), s64.reshape(1, 64))[0])
            assert got == 1, (name, who)  # the spec's vectors verify under the reference with libwally's sighash
            rec["sigs"].append(dict(who=who, pub33=key.hex(), sig64=bytes(s64).hex(), sighash_type=1, expected=1))
        out.append(rec)
    json.dump(out, open(OUT + "/bolt3_htlc_txs.json", "w"), indent=0)
    print("bolt3_htlc_txs:", len(out), "transactions,", sum(len(o["sigs"]) for o in out), "signatures, all valid under the reference")


def bip143_libwally():
    """libwally's sighash (bitcoin_tx_hash_for_sig via oracle/cln_harness.c) of the 120 seeded transactions that
    tests/test_host_emul.py::test_bip143_bolt3_and_general_shapes_vs_libwally draws; the draws here must stay in step."""
    cln = util.load_cln()
    vp = ctypes.c_void_p
    cln.cln_tx_new.restype = vp
    cln.cln_tx_new.argtypes = [ctypes.c_uint32, ctypes.c_uint32]
    cln.cln_tx_add_input.argtypes = [vp, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_uint32]
    cln.cln_tx_add_output.argtypes = [vp, ctypes.c_uint64, ctypes.c_char_p, ctypes.c_size_t]
    cln.cln_tx_free.argtypes = [vp]
    cln.cln_tx_set_input_amount.argtypes = [ctypes.c_uint64]
    cln.cln_tal_bytes.restype = vp
    cln.cln_tal_bytes.argtypes = [ctypes.c_char_p, ctypes.c_size_t]
    cln.cln_tal_free.argtypes = [vp]
    cln.cln_tx_sighash.argtypes = [vp, ctypes.c_uint, vp, ctypes.c_uint32, vp]
    rng = np.random.default_rng(8)
    out = []
    for it in range(120):
        nin, nout = int(rng.integers(1, 4)), int(rng.integers(1, 7))
        ins = [(bytes(rng.integers(0, 256, size=32, dtype=np.uint8)), int(rng.integers(0, 9)), int(rng.integers(0, 2**32))) for _ in range(nin)]
        outs = [(int(rng.integers(0, 2**40)), bytes(rng.integers(0, 256, size=int(rng.choice([0, 22, 34, 300])), dtype=np.uint8))) for _ in range(nout)]
        lock = int(rng.integers(0, 2**32))
        tx = cln.cln_tx_new(2, lock)
        for a in ins:
            assert cln.cln_tx_add_input(tx, *a) == 0
        for amt, sc in outs:
            assert cln.cln_tx_add_output(tx, amt, sc or None, len(sc)) == 0
        inp = int(rng.integers(0, nin))
        ws = bytes(rng.integers(0, 256, size=int(rng.choice([1, 2, 133, 252, 253, 700])), dtype=np.uint8))
        amount = int(rng.integers(0, 2**45))
        sht = int(rng.choice([1, 0x83, 2, 3, 0x81, 0x82]))
        tal_ws = cln.cln_tal_bytes(ws, len(ws))
        cln.cln_tx_set_input_amount(amount)
        want = np.zeros(32, np.uint8)
        cln.cln_tx_sighash(tx, inp, tal_ws, sht, P(want))
        out.append(bytes(want).hex())
        cln.cln_tal_free(tal_ws)
        cln.cln_tx_free(tx)
    json.dump(out, open(OUT + "/bip143_libwally.json", "w"), indent=0)
    print("bip143_libwally:", len(out), "sighashes")


if __name__ == "__main__":
    if len(sys.argv) > 1:  # regenerate only the named sets
        for name in sys.argv[1:]:
            globals()[name]()
        sys.exit(0)
    wycheproof()
    bip340()
    pubkey_parse()
    gossip()
    chan_ann_3703()
    ecmult_kat()
    ecdsa_edge_cases()
    bolt3_htlc_txs()
    bip143_libwally()
    gossip_store_full()
