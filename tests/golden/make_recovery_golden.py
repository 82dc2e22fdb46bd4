"""Writes the public-key recovery fixtures from the reference (run where /root/reference and oracle/_ref exist):

  tests/golden/recovery_vectors.json   (a) test_ecdsa_recovery_edge_cases of the recovery module (every recid);
                                       (b) the invoices of common/test/run-bolt11.c's test_b11 calls: signing hash, sig64,
                                       recid and the node id the file signs them with; each confirmed by
                                       secp256k1_ecdsa_recover, whose status and key are stored with every vector
  tests/golden/recovery_reference.npz  secp256k1_ecdsa_recover's answers for every workload of tests/recovery.py (input
                                       digest, statuses, 8-byte key digests)

The reference library is called through its public API (parse_compact, recover, serialize) in oracle/_ref/libsecp_ref.so.
The restated recoverable signer of tests/recovery.py is checked against secp256k1_ecdsa_sign_recoverable on the way.
"""
import ctypes
import hashlib
import json
import os
import re
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from tests import recovery, refcalls  # noqa: E402

REF = "/root/reference"
S = REF + "/external/libwally-core/src/secp256k1"
OUT = os.path.dirname(os.path.abspath(__file__))
live = recovery.LiveReference()


def c_bytes(block, name):
    m = re.search(r"unsigned char " + name + r"\[\d*\]\s*=\s*\{([^}]*)\}", block)
    assert m, name
    return bytes(int(x, 16) for x in re.findall(r"0[xX]([0-9A-Fa-f]{2})", m.group(1)))


_BECH32 = "qpzry9x8gf2tvdw0s3jn54khce6mua7l"


def _bolt11_signed(inv):
    """(signing hash, sig64, recid) of a BOLT #11 invoice: SHA-256 over the hrp bytes and the data words before the
    signature packed 5 bits at a time into bytes, zero-padded (common/bolt11.c, common/hash_u5.c)."""
    sep = inv.rfind("1")
    hrp, words = inv[:sep], [_BECH32.index(c) for c in inv[sep + 1:-6]]  # the last 6 characters are the checksum
    body, sigw = words[:-104], words[-104:]

    def pack(ws):
        acc, bits, out = 0, 0, bytearray()
        for w in ws:
            acc, bits = (acc << 5) | w, bits + 5
            while bits >= 8:
                bits -= 8
                out.append((acc >> bits) & 0xFF)
        if bits:
            out.append((acc << (8 - bits)) & 0xFF)
        return bytes(out)
    sig65 = pack(sigw)[:65]
    return hashlib.sha256(hrp.encode() + pack(body)).digest(), sig65[:64], sig65[64]


def recovery_vectors():
    """Public-key recovery: (a) test_ecdsa_recovery_edge_cases (modules/recovery/tests_impl.h:154-200), every recid;
    (b) the invoices of common/test/run-bolt11.c's test_b11 calls with the node id the file expects, each confirmed by the
    reference's secp256k1_ecdsa_recover."""
    src = open(S + "/src/modules/recovery/tests_impl.h").read()
    blk = src[src.index("static void test_ecdsa_recovery_edge_cases"):]
    msg = bytes(ord(c) for c in re.findall(r"'(.)'", blk[:blk.index("sig64[64]")]))
    assert len(msg) == 32
    out = []
    for name, sig in (("sig64", c_bytes(blk, "sig64")), ("sigb64", c_bytes(blk, "sigb64"))):
        for recid in range(4):
            out.append(dict(set="edge_cases", name=f"{name} recid {recid}", msg32=msg.hex(), sig64=sig.hex(), recid=recid))
    b11 = open(REF + "/common/test/run-bolt11.c").read()
    # every invoice is signed by test_sign's key (the file re-encodes each one with it and compares the strings)
    sk = re.search(r'hex_decode\("([0-9a-f]{64})",[^;]*&privkey', b11).group(1)
    pxy = refcalls.base_mult(int(sk, 16))
    node = bytes([2 + (pxy[63] & 1)]).hex() + bytes(pxy[:32]).hex()
    for inv in re.findall(r'test_b11\("(ln[0-9a-z]+|LN[0-9A-Z]+)"', b11):
        h, sig, recid = _bolt11_signed(inv.lower())
        out.append(dict(set="bolt11", name=inv[:24] + "...", msg32=h.hex(), sig64=sig.hex(), recid=recid, node_id=node))
    n = len(out)
    w = dict(msg=np.array([np.frombuffer(bytes.fromhex(o["msg32"]), np.uint8) for o in out]),
             sig=np.array([np.frombuffer(bytes.fromhex(o["sig64"]), np.uint8) for o in out]),
             recid=np.array([o["recid"] for o in out], np.uint8))
    xy, st = live.recover(w)
    for o, x, s in zip(out, xy, st):
        o["status"] = int(s)
        o["xy64"] = bytes(x).hex()
        if o["set"] == "bolt11":
            assert s == 1 and bytes([2 + (x[63] & 1)]).hex() + bytes(x[:32]).hex() == o["node_id"], o["name"]
    edge = [o["status"] for o in out if o["set"] == "edge_cases"]
    assert edge == [0, 1, 0, 0, 1, 1, 1, 1], edge  # tests_impl.h:185-192 and the (4, 4) loop
    json.dump(out, open(OUT + "/recovery_vectors.json", "w"), indent=1)
    print("recovery_vectors:", len(edge), "edge-case pairs,", n - len(edge), "BOLT #11 invoices")


def check_signer(count=200):
    """the restated recoverable signer against secp256k1_ecdsa_sign_recoverable"""
    lib = live.lib
    lib.secp256k1_ecdsa_sign_recoverable.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p,
                                                     ctypes.c_void_p, ctypes.c_void_p]
    lib.secp256k1_ecdsa_recoverable_signature_serialize_compact.argtypes = [ctypes.c_void_p, ctypes.c_char_p,
                                                                          ctypes.POINTER(ctypes.c_int), ctypes.c_char_p]
    for i in range(count):
        d = int.from_bytes(hashlib.sha256(b"d%d" % i).digest(), "big") % (recovery.N - 1) + 1
        m = hashlib.sha256(b"m%d" % i).digest()
        rs, sig, rid = ctypes.create_string_buffer(65), ctypes.create_string_buffer(64), ctypes.c_int()
        assert lib.secp256k1_ecdsa_sign_recoverable(live.ctx, rs, m, d.to_bytes(32, "big"), None, None) == 1
        lib.secp256k1_ecdsa_recoverable_signature_serialize_compact(live.ctx, sig, ctypes.byref(rid), rs)
        assert recovery.ecdsa_sign_recoverable(d, m) == (sig.raw, rid.value), i
    print("recoverable signer: restatement == reference on", count, "signatures")


def reference_answers():
    out = {}
    for name, w in recovery.sets().items():
        xy, st = live.recover(w, threads=os.cpu_count())
        out[name + "_inputs"] = np.array(recovery.input_digest(w))
        out[name + "_status"] = st
        out[name + "_keys"] = recovery.key_digests(xy)
        print(f"{name}: {st.size} items, status -1/0/1: {(st == -1).sum()}/{(st == 0).sum()}/{(st == 1).sum()}")
    np.savez_compressed(OUT + "/recovery_reference.npz", **out)


if __name__ == "__main__":
    check_signer()
    recovery_vectors()
    reference_answers()
