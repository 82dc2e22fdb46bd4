"""Public-key recovery workloads shared by the host-build and GPU tests (tests only).

Each builder returns a dict of arrays: msg (n, 32), sig (n, 64), recid (n,) uint8, and where the signer is known
signer (n, 64) with the signer's x || y (zeros where the item is not expected to give the signer's key back).

The reference's answers (secp256k1_ecdsa_recover of the unmodified library oracle/_ref builds) are kept in
tests/golden/recovery_reference.npz, which tests/golden/make_recovery_golden.py writes: per set a digest of the inputs,
the status of every item and the first 8 bytes of SHA-256(x || y) of every key, so that the tests compare bit for bit
without the reference being present.
"""
import ctypes
import hashlib
import hmac
import json
import os
import threading

import numpy as np

from tests import refcalls, util

N = util.N_ORDER
P_FIELD = util.P_FIELD
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "recovery_vectors.json")
REFERENCE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "recovery_reference.npz")


def _b32(v):
    return np.frombuffer(int(v).to_bytes(32, "big"), np.uint8)


def _int(a):
    return int.from_bytes(bytes(a), "big")


def _is_square(c):
    return pow(c % P_FIELD, (P_FIELD - 1) // 2, P_FIELD) in (0, 1)


def ecdsa_sign_recoverable(d, msg32):
    """secp256k1_ecdsa_sign_recoverable with the default nonce: (compact r || s, recid).  recid = (R.x >= n) << 1 | parity
    of R.y, bit 0 flipped when s is negated to low S (ecdsa_impl.h:280-296)."""
    m = int.from_bytes(msg32, "big") % N
    seed = d.to_bytes(32, "big") + m.to_bytes(32, "big")
    mac = lambda k, x: hmac.new(k, x, hashlib.sha256).digest()
    K, V = bytes(32), b"\x01" * 32
    K = mac(K, V + b"\x00" + seed)
    V = mac(K, V)
    K = mac(K, V + b"\x01" + seed)
    V = mac(K, V)
    while True:
        V = mac(K, V)
        k = int.from_bytes(V, "big")
        if 0 < k < N:
            rxy = refcalls.base_mult(k)
            rx = int.from_bytes(rxy[:32].tobytes(), "big")
            r = rx % N
            s = pow(k, -1, N) * (m + r * d) % N
            if r and s:
                break
        K = mac(K, V + b"\x00")
        V = mac(K, V)
    recid = (2 if rx >= N else 0) | int(rxy[63] & 1)
    if s > N // 2:
        s, recid = N - s, recid ^ 1
    return r.to_bytes(32, "big") + s.to_bytes(32, "big"), recid


def pack(items):
    """items: list of (msg32, sig64, recid[, signer xy64]) -> dict of arrays"""
    n = len(items)
    out = dict(msg=np.zeros((n, 32), np.uint8), sig=np.zeros((n, 64), np.uint8), recid=np.zeros(n, np.uint8),
               signer=np.zeros((n, 64), np.uint8))
    for i, it in enumerate(items):
        out["msg"][i] = np.frombuffer(bytes(it[0]), np.uint8)
        out["sig"][i] = np.frombuffer(bytes(it[1]), np.uint8)
        out["recid"][i] = it[2]
        if len(it) > 3 and it[3] is not None:
            out["signer"][i] = it[3]
    return out


def golden():
    """tests/golden/recovery_vectors.json: the reference's own edge cases and the BOLT #11 invoices, with the outcome the
    reference gave when the file was written"""
    vec = json.load(open(GOLDEN))
    items = [(bytes.fromhex(v["msg32"]), bytes.fromhex(v["sig64"]), v["recid"]) for v in vec]
    w = pack(items)
    w["status"] = np.array([v["status"] for v in vec], np.int8)
    w["xy"] = np.array([np.frombuffer(bytes.fromhex(v["xy64"]), np.uint8) for v in vec])
    return w, vec


def signed(n, seed):
    """n keys sign n messages with secp256k1_ecdsa_sign_recoverable (restated by ecdsa_sign_recoverable).  Every signature is
    tried with all four recids; its high-S twin (n - s) with recid ^ 1 (the same key) and with the same recid."""
    rng = np.random.default_rng(seed)
    items = []
    for _ in range(n):
        d = int.from_bytes(rng.integers(0, 256, 32, dtype=np.uint8).tobytes(), "big") % (N - 1) + 1
        m = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
        sig, recid = ecdsa_sign_recoverable(d, m)
        xy = refcalls.base_mult(d)
        for rid in range(4):
            items.append((m, sig, rid, xy if rid == recid else None))
        twin = sig[:32] + (N - _int(sig[32:])).to_bytes(32, "big")
        items.append((m, twin, recid ^ 1, xy))
        items.append((m, twin, recid, None))
    return pack(items)


def edge(seed):
    """Encoding refusals and degenerate scalars: r = 0, s = 0, r >= n, s >= n, recid 4 and 255, msg = 0 and msg = n
    (u1 = 0), and r whose x^3 + 7 is not a square."""
    rng = np.random.default_rng(seed)
    d = 0x1234567 + seed
    m = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
    sig, recid = ecdsa_sign_recoverable(d, m)
    r, s = _int(sig[:32]), _int(sig[32:])
    xy = refcalls.base_mult(d)
    items = []
    for rid in range(4):
        items += [(m, bytes(32) + sig[32:], rid), (m, sig[:32] + bytes(32), rid),
                  (m, N.to_bytes(32, "big") + sig[32:], rid), (m, (N + r % (2**256 - N)).to_bytes(32, "big") + sig[32:], rid),
                  (m, b"\xff" * 32 + sig[32:], rid), (m, sig[:32] + N.to_bytes(32, "big"), rid),
                  (m, sig[:32] + b"\xff" * 32, rid)]
    for rid in (4, 5, 7, 128, 255):
        items.append((m, sig, rid))
    for mv in (0, N, N + 1, 2**256 - 1):
        # u1 = -m/r is 0 for m = 0 and m = n: Q = (s/r) R alone
        items += [(mv.to_bytes(32, "big"), sig, rid) for rid in range(4)]
    x = 1 + int(rng.integers(1, 1 << 30))
    while _is_square(x ** 3 + 7):
        x += 1
    items += [(m, x.to_bytes(32, "big") + sig[32:], rid) for rid in range(4)]
    items.append((m, sig, recid, xy))
    return pack(items)


def constructed(seed, count=8):
    """Cases built from their algebra (as tests/adversarial.py does):
      * recid 2 / 3 with r < p - n where r + n is a curve x (the only signatures whose R.x >= n);
      * recid 2 / 3 with r >= p - n (r + n >= p: no such R);
      * s R = m G: Q = (s R - m G) / r = infinity, status 0;
      * s R = -m G: the final addition of -m/r G and s/r R is a doubling."""
    rng = np.random.default_rng(seed)
    rnd = lambda lim: int.from_bytes(rng.integers(0, 256, 40, dtype=np.uint8).tobytes(), "big") % lim
    items = []
    pmn = P_FIELD - N
    for _ in range(count):
        r = rnd(pmn - 1) + 1
        while not _is_square((r + N) ** 3 + 7):
            r = rnd(pmn - 1) + 1
        s = rnd(N - 1) + 1
        m = rng.integers(0, 256, 32, dtype=np.uint8).tobytes()
        for rid in range(4):
            items.append((m, _b32(r).tobytes() + _b32(s).tobytes(), rid))
        r2 = pmn + rnd(N - pmn)
        for rid in (2, 3):
            items.append((m, _b32(r2).tobytes() + _b32(s).tobytes(), rid))
    for _ in range(count):
        k = rnd(N - 1) + 1
        rxy = refcalls.base_mult(k)
        rx = _int(rxy[:32])
        if rx >= N:
            continue
        rid = int(rxy[63] & 1)
        s = rnd(N - 1) + 1
        for sign in (1, -1):
            m = (sign * s * k) % N  # s R = sign * m G
            items.append((_b32(m).tobytes(), _b32(rx).tobytes() + _b32(s).tobytes(), rid))
    return pack(items)


def sets():
    """the workloads the reference's answers are kept for, by name"""
    return {"golden": golden()[0], "signed": signed(2000, seed=31), "edge": edge(seed=5), "constructed": constructed(seed=77)}


def input_digest(w):
    h = hashlib.sha256()
    for k in ("msg", "sig", "recid"):
        h.update(np.ascontiguousarray(w[k]).tobytes())
    return h.hexdigest()


def key_digests(xy):
    """first 8 bytes of SHA-256 of every 64-byte key, (n, 8) uint8"""
    return np.array([np.frombuffer(hashlib.sha256(bytes(x)).digest()[:8], np.uint8) for x in xy], np.uint8).reshape(-1, 8)


def reference(name, w):
    """the reference's (status, key digests) for set `name`, checked to be about these very inputs"""
    z = np.load(REFERENCE)
    assert str(z[name + "_inputs"]) == input_digest(w), f"{name}: inputs differ from those the reference answered"
    return z[name + "_status"], z[name + "_keys"]


def mismatches(xy, st, want):
    """indices where (xy, st) differ from the reference's (status, key digests)"""
    want_st, want_keys = want
    return np.nonzero((st != want_st) | (key_digests(xy) != want_keys).any(axis=1))[0]


class LiveReference:
    """secp256k1_ecdsa_recoverable_signature_parse_compact + secp256k1_ecdsa_recover of oracle/_ref/libsecp_ref.so,
    called as common/bolt11.c:1018-1050 calls them (recid > 3 is refused before the library sees it)"""

    def __init__(self):
        self.lib = lib = util.load_ref()
        lib.secp256k1_context_create.restype = ctypes.c_void_p
        lib.secp256k1_context_create.argtypes = [ctypes.c_uint]
        for f in (lib.secp256k1_ecdsa_recoverable_signature_parse_compact, lib.secp256k1_ecdsa_recover,
                  lib.secp256k1_ec_pubkey_serialize):
            f.restype = ctypes.c_int
        lib.secp256k1_ecdsa_recoverable_signature_parse_compact.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_int]
        lib.secp256k1_ecdsa_recover.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p]
        lib.secp256k1_ec_pubkey_serialize.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.POINTER(ctypes.c_size_t),
                                                      ctypes.c_char_p, ctypes.c_uint]
        self.ctx = lib.secp256k1_context_create(1)  # SECP256K1_CONTEXT_NONE

    def one(self, msg32, sig64, recid):
        if recid > 3:
            return -1, bytes(64)
        rs, pk, out, ln = ctypes.create_string_buffer(65), ctypes.create_string_buffer(64), ctypes.create_string_buffer(65), ctypes.c_size_t(65)
        if not self.lib.secp256k1_ecdsa_recoverable_signature_parse_compact(self.ctx, rs, sig64, recid):
            return -1, bytes(64)
        if not self.lib.secp256k1_ecdsa_recover(self.ctx, pk, rs, msg32):
            return 0, bytes(64)
        self.lib.secp256k1_ec_pubkey_serialize(self.ctx, out, ctypes.byref(ln), pk, 2)  # SECP256K1_EC_UNCOMPRESSED
        return 1, out.raw[1:65]

    def recover(self, w, threads=1):
        """(xy (n, 64), status (n,) int8); the library calls release the GIL, so threads run in parallel"""
        n = w["msg"].shape[0]
        xy = np.zeros((n, 64), np.uint8)
        st = np.zeros(n, np.int8)

        def work(lo, hi):
            for i in range(lo, hi):
                s, k = self.one(w["msg"][i].tobytes(), w["sig"][i].tobytes(), int(w["recid"][i]))
                st[i], xy[i] = s, np.frombuffer(k, np.uint8)
        th = [threading.Thread(target=work, args=(n * t // threads, n * (t + 1) // threads)) for t in range(threads)]
        for t in th:
            t.start()
        for t in th:
            t.join()
        return xy, st


def load_emul():
    from lightning_b200 import build
    return ctypes.CDLL(build.build_host_emul_recover())


def emul_recover(emul, w, small=False):
    """the host build of the device code: throughput schedule, or the small-batch schedule with pair ladders"""
    n = w["msg"].shape[0]
    xy = np.zeros((n, 64), np.uint8)
    st = np.zeros(n, np.int8)
    fn = emul.emul_recover_small_pair_batch if small else emul.emul_recover_batch
    p = lambda a: np.ascontiguousarray(a).ctypes.data_as(ctypes.c_void_p)
    msg, sig, rid = (np.ascontiguousarray(w[k]) for k in ("msg", "sig", "recid"))
    fn(p(msg), p(sig), p(rid), ctypes.c_size_t(n), p(xy), p(st))
    return xy, st
