"""Shared test helpers: oracle loaders and seeded workload generation (tests only)."""
import ctypes
import os
import subprocess

import numpy as np

from tests import refcalls

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_ORDER = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
P_FIELD = 2**256 - 2**32 - 977
_p8 = ctypes.POINTER(ctypes.c_uint8)


def P(a):
    """A uint8 pointer to the contiguous array a; it keeps a, so that tests.refcalls can record what a call reads and writes."""
    p = a.ctypes.data_as(_p8)
    p._sv_arr = a
    return p


def _load_lib(name):
    path = os.path.join(ROOT, "oracle", "_ref", name)
    if not os.path.exists(path):
        raise RuntimeError(f"oracle/_ref/{name} is missing: it is built by oracle/Makefile where the reference's sources are")
    return ctypes.CDLL(path)


def load_ref():
    """The unmodified reference (libsecp256k1 + CCAN sha256), as built into oracle/_ref."""
    return _load_lib("libsecp_ref.so")


def load_cln():
    """CLN's own unmodified bitcoin/signature.c + gossipd/sigcheck.c over the libwally amalgamation (config C1)."""
    return _load_lib("libcln_ref.so")


def recorded_ref():
    """load_ref()'s answers as tests/golden/refcalls.bin recorded them (see tests/refcalls.py)."""
    return refcalls.Library("ref", load_ref)


def recorded_cln():
    return refcalls.Library("cln", load_cln)


def load_port():
    path = os.path.join(ROOT, "oracle", "libsecp_port.so")
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "oracle"), "port"], stdin=subprocess.DEVNULL)
    return ctypes.CDLL(path)


def load_emul():
    from lightning_b200 import build
    return ctypes.CDLL(build.build_host_emul())


def ref_verify(ref, kind, msg, key, sig, threads=1):
    n = msg.shape[0]
    out = np.zeros(n, np.uint8)
    fn = [ref.ref_ecdsa_verify_batch, ref.ref_ecdsa_verify_batch_xy, ref.ref_schnorr_verify_batch][kind]
    fn(P(msg), P(key), P(sig), ctypes.c_size_t(n), P(out), threads)
    return out


def make_signed(n, seed):
    """n seeded random keys/messages, signed as the reference's ref_pubkey_create / ref_ecdsa_sign / ref_schnorr_sign
    sign them (tests/refcalls.py restates those): returns dict of arrays."""
    rng = np.random.default_rng(seed)
    sk = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    msg = rng.integers(0, 256, size=(n, 32), dtype=np.uint8)
    pub33 = np.zeros((n, 33), np.uint8)
    pubxy = np.zeros((n, 64), np.uint8)
    sig = np.zeros((n, 64), np.uint8)
    xonly = np.zeros((n, 32), np.uint8)
    ssig = np.zeros((n, 64), np.uint8)
    for i in range(n):
        d = int.from_bytes(sk[i].tobytes(), "big")
        m = msg[i].tobytes()
        pubxy[i] = refcalls.base_mult(d)
        pub33[i, 0], pub33[i, 1:] = 2 + (pubxy[i, 63] & 1), pubxy[i, :32]
        sig[i] = np.frombuffer(refcalls.ecdsa_sign(d, m), np.uint8)
        s, x = refcalls.schnorr_sign(d, m)
        ssig[i], xonly[i] = np.frombuffer(s, np.uint8), np.frombuffer(x, np.uint8)
    return dict(msg=msg, pub33=pub33, pubxy=pubxy, sig=sig, xonly=xonly, ssig=ssig)


def corrupt(w, every=10):
    """SURVEY.md §8(d) corruption classes, round-robin on every `every`-th item (in place, returns w)."""
    n = w["msg"].shape[0]
    for cls, i in enumerate(range(0, n, every)):
        c = cls % 11
        j = (i + 1) % n
        if c == 0:
            w["msg"][i, 5] ^= 4
        elif c == 1:
            w["sig"][i, 7] ^= 1
            w["ssig"][i, 7] ^= 1
        elif c == 2:
            w["sig"][i, 40] ^= 1
            w["ssig"][i, 40] ^= 1
        elif c == 3:  # high S
            s = int.from_bytes(bytes(w["sig"][i, 32:]), "big")
            w["sig"][i, 32:] = np.frombuffer((N_ORDER - s).to_bytes(32, "big"), dtype=np.uint8)
            w["ssig"][i, 32:] = 255  # s >= n
        elif c == 4:  # someone else's key
            w["pub33"][i] = w["pub33"][j]
            w["pubxy"][i] = w["pubxy"][j]
            w["xonly"][i] = w["xonly"][j]
        elif c == 5:  # bad prefix / y off curve
            w["pub33"][i, 0] = 4
            w["pubxy"][i, 63] ^= 1
            w["xonly"][i, 31] ^= 1
        elif c == 6:  # x >= p
            w["pub33"][i, 1:] = 255
            w["pubxy"][i, :32] = 255
            w["xonly"][i, :] = 255
        elif c == 7:  # flip a key bit (usually lands on a non-residue or a different point)
            w["pub33"][i, 20] ^= 1
            w["pubxy"][i, 20] ^= 1
            w["xonly"][i, 20] ^= 1
        elif c == 8:  # wrong parity / negated R
            w["pub33"][i, 0] ^= 1
            w["ssig"][i, :32] = np.frombuffer(
                ((P_FIELD - int.from_bytes(bytes(w["ssig"][i, :32]), "big")) % P_FIELD).to_bytes(32, "big"), np.uint8)
        elif c == 9:  # r = 0 / r >= p
            w["sig"][i, :32] = 0
            w["ssig"][i, :32] = 255
        elif c == 10:  # s = 0 / r >= n
            w["sig"][i, 32:] = 0
            w["sig"][j % n, :32] = 255
    return w


def make_htlc_txs(rng, n):
    """n synthetic commitment-HTLC transaction inputs (shape: common/htlc_tx.c:10-69 — version 2, one input spending an
    HTLC output of the commitment tx, one P2WSH output, nSequence 0/1, locktime 0 or a cltv expiry; witness script
    sized like bitcoin/script.c:732/849 produce them; sighash ALL, or SINGLE|ANYONECANPAY with anchors
    (channeld/channeld.c:1105-1108)), plus a few other sighash types.  Returns (SvTx array, scripts blob)."""
    from lightning_b200 import SvTx
    txs = (SvTx * n)()
    blob = bytearray()
    for i in range(n):
        t = txs[i]
        t.version = 2
        t.locktime = int(rng.integers(0, 2)) * int(rng.integers(500000, 900000))
        t.sequence = int(rng.integers(0, 2))
        t.sighash_type = [1, 0x83, 1, 0x83, 2, 3, 0x81, 0x82][i % 8]
        t.prev_txid[:] = list(rng.integers(0, 256, size=32, dtype=np.uint8))
        t.prev_index = int(rng.integers(0, 600))
        ws = bytes(rng.integers(0, 256, size=int(rng.integers(130, 145)) if i % 11 else int(rng.integers(0, 400)), dtype=np.uint8))
        os_ = b"\x00\x20" + bytes(rng.integers(0, 256, size=32, dtype=np.uint8))
        t.script_off, t.script_len = len(blob), len(ws)
        blob += ws
        t.out_script_off, t.out_script_len = len(blob), len(os_)
        blob += os_
        t.input_amount = int(rng.integers(546, 10**9))
        t.output_amount = int(rng.integers(330, t.input_amount + 1))
    return txs, bytes(blob)


def cln_sighash(cln, t, blob):
    """The same sighash from libwally (what bitcoin_tx_hash_for_sig computes), via oracle/cln_harness.c."""
    out = np.zeros(32, np.uint8)
    ws = blob[t.script_off:t.script_off + t.script_len]
    os_ = blob[t.out_script_off:t.out_script_off + t.out_script_len]
    rc = cln.cln_htlc_sighash(ctypes.c_uint32(t.version), ctypes.c_uint32(t.locktime), bytes(t.prev_txid), ctypes.c_uint32(t.prev_index),
                              ctypes.c_uint32(t.sequence), ws, ctypes.c_size_t(len(ws)), ctypes.c_uint64(t.input_amount),
                              ctypes.c_uint64(t.output_amount), os_, ctypes.c_size_t(len(os_)), ctypes.c_uint32(t.sighash_type), P(out))
    assert rc == 0, rc
    return out
