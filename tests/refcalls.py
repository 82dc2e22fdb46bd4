"""The reference's answers, recorded.

Tests compare the engine with the unmodified reference: libsecp256k1 and CLN's own C, compiled by oracle/Makefile into
oracle/_ref from the reference's sources.  Those sources are not part of this repository, so every call a test makes
into them is kept in tests/golden/refcalls.bin: a digest of the function's name and of every input byte, with the
return value and the bytes the call wrote.  The tests replay that record, and a call whose inputs were never recorded
fails.

Conversions a test makes per item (hashing, key parsing, the libraries' opaque structs, key derivation, ECDSA and
BIP-340 signing) are not recorded: LOCAL restates them in Python over oracle/secp_port.c, and while recording every such call
runs both ways and must agree byte for byte.

To record, build oracle/_ref and run the tests with SV_REF_RECORD=<file>: the libraries are called for real and their
answers are merged with the committed record into <file>.  Arguments are ints, bytes, None, ctypes scalars, ctypes
arrays and pointers made by tests.util.P (which keeps the array it points into); handles into the reference's own
objects cannot be recorded, and a test that needs them takes the libraries themselves (the ref_live and cln_live
fixtures, which skip where oracle/_ref is not built).
"""
import atexit
import ctypes
import functools
import gzip
import hashlib
import hmac
import os
import struct

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refcalls.bin")
_record_path = os.environ.get("SV_REF_RECORD")
_store = None
_new = {}


# gzip of records in key order; a record is the 6-byte key, the return value (int64), a flags byte (0x80: returned None,
# 0x40: returned a bool, low 6 bits: number of buffers written) and per written buffer its argument index (u8), length
# (u32) and bytes
_HEAD, _BUF = struct.Struct("<6sqB"), struct.Struct("<BI")


def _load():
    global _store
    if _store is None:
        _store = {}
        if os.path.exists(GOLDEN):
            with gzip.open(GOLDEN, "rb") as f:
                data = f.read()
            o = 0
            while o < len(data):
                key, ret, flags = _HEAD.unpack_from(data, o)
                o += _HEAD.size
                wrote = {}
                for _ in range(flags & 0x3F):
                    i, n = _BUF.unpack_from(data, o)
                    o += _BUF.size
                    wrote[i] = data[o:o + n]
                    o += n
                _store[key] = (None if flags & 0x80 else bool(ret) if flags & 0x40 else ret, wrote)
    return _store


def _save():
    if not _new:
        return
    out = dict(_load())
    out.update(_new)
    parts = []
    for key in sorted(out):
        ret, wrote = out[key]
        flags = (0x80 if ret is None else 0x40 if isinstance(ret, bool) else 0) | len(wrote)
        parts.append(_HEAD.pack(key, int(ret or 0), flags))
        for i, b in sorted(wrote.items()):
            parts += [_BUF.pack(i, len(b)), b]
    with open(_record_path, "wb") as f:
        with gzip.GzipFile(fileobj=f, mode="wb", mtime=0) as g:
            g.write(b"".join(parts))


if _record_path:
    atexit.register(_save)


def _buffer(a):
    """The writable bytes behind an argument, or None for a value argument."""
    if isinstance(a, ctypes._Pointer):
        arr = getattr(a, "_sv_arr", None)
        if arr is None:
            raise TypeError("pointer argument not made by tests.util.P: its length is unknown, so it cannot be recorded")
        if not arr.flags.c_contiguous:
            raise TypeError("pointer into a non-contiguous array")
        return arr.reshape(-1).view(np.uint8)
    if isinstance(a, ctypes.Array):
        return np.frombuffer(a, dtype=np.uint8)
    return None


def _encode(a):
    if a is None or isinstance(a, (bool, int, float)):
        return repr(a).encode()
    if isinstance(a, bytes):
        return b"b" + a
    if isinstance(a, ctypes._SimpleCData):
        return repr(a.value).encode()
    buf = _buffer(a)
    if buf is None:
        raise TypeError(f"cannot record an argument of type {type(a).__name__}")
    return b"p" + buf.tobytes()


class _Fn:
    def __init__(self, lib, name):
        self.__dict__["_lib"], self.__dict__["_name"] = lib, name

    def __setattr__(self, k, v):  # argtypes / restype: only the real function has a use for them
        if self._lib.live is not None:
            setattr(getattr(self._lib.live, self._name), k, v)

    def __call__(self, *args):
        bufs = [_buffer(a) for a in args]
        local = LOCAL.get(f"{self._lib.name}.{self._name}")
        if local is not None:
            vals = [a.value if isinstance(a, ctypes._SimpleCData) else a for a in args]
            if self._lib.live is None:
                ret = local(vals, bufs)
                if ret is not NotImplemented:
                    return ret
            else:
                mine = [None if b is None else b.copy() for b in bufs]
                ret_local = local(vals, mine)
                if ret_local is not NotImplemented:
                    ret = getattr(self._lib.live, self._name)(*args)
                    same = all(b is None or np.array_equal(b, m) for b, m in zip(bufs, mine))
                    if (ret_local is not None and ret != ret_local) or not same:  # None: a void function
                        raise AssertionError(f"tests/refcalls.py LOCAL[{self._lib.name}.{self._name}] differs from the reference")
                    return ret
        h = hashlib.sha256(f"{self._lib.name}.{self._name}".encode())
        for a in args:
            e = _encode(a)
            h.update(len(e).to_bytes(8, "little"))
            h.update(e)
        key = h.digest()[:6]
        if self._lib.live is not None:
            before = [None if b is None else b.copy() for b in bufs]
            ret = getattr(self._lib.live, self._name)(*args)
            if not (ret is None or isinstance(ret, (bool, int))):
                raise TypeError(f"{self._name} returns {type(ret).__name__}, which cannot be recorded")
            wrote = {i: b.tobytes() for i, (b, b0) in enumerate(zip(bufs, before))
                     if b is not None and not np.array_equal(b, b0)}
            _new[key] = [ret, wrote]
            return ret
        rec = _load().get(key)
        if rec is None:
            raise LookupError(f"{self._lib.name}.{self._name}: no recorded answer for these inputs "
                              f"(record them with SV_REF_RECORD, see tests/refcalls.py)")
        ret, wrote = rec
        for i, b in wrote.items():
            bufs[i][:] = np.frombuffer(b, dtype=np.uint8)
        return ret


class Library:
    """A stand-in for one reference library: attribute access gives its functions, replayed or, when recording, live."""

    def __init__(self, name, load_live):
        self.name = name
        self.live = load_live() if _record_path else None
        self._fns = {}

    def __getattr__(self, fn):
        if fn.startswith("_"):
            raise AttributeError(fn)
        if fn not in self._fns:
            self._fns[fn] = _Fn(self, fn)
        return self._fns[fn]


# ---- LOCAL: per-item conversions restated; fn(values, buffers) writes what the C function writes and returns its value,
# or NotImplemented for inputs it does not cover (those are recorded) ----
N_ORDER = 0xFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFFEBAAEDCE6AF48A03BBFD25E8CD0364141
_p8 = ctypes.POINTER(ctypes.c_uint8)


@functools.lru_cache(maxsize=None)
def _port():
    from tests import util
    return util.load_port()


def _ptr(a):
    return a.ctypes.data_as(_p8)


def _parse33(pub):
    """x || y (big-endian) of a 33-byte SEC1 key, or None where secp256k1_ec_pubkey_parse refuses it."""
    xy = np.zeros(64, np.uint8)
    return xy if _port().port_pubkey_parse33(_ptr(np.ascontiguousarray(pub[:33])), _ptr(xy)) else None


def base_mult(k):
    """x || y of k*G for 0 < k < n (secp256k1_ec_pubkey_create), else None."""
    if not 0 < k < N_ORDER:
        return None
    xy = np.zeros(64, np.uint8)
    assert _port().port_scalar_base_mult(_ptr(np.frombuffer(k.to_bytes(32, "big"), np.uint8).copy()), _ptr(xy))
    return xy


def _compressed(xy):
    return np.concatenate([[2 + (xy[63] & 1)], xy[:32]]).astype(np.uint8)


def _le(xy):
    """libsecp256k1's opaque layout on a little-endian host: each 256-bit value as four 64-bit limbs, low limb first."""
    return np.concatenate([xy[31::-1], xy[:31:-1]])


def _sha256d(v, b):
    data = b[0][:v[1]].tobytes() if v[1] else b""
    b[2][:] = np.frombuffer(hashlib.sha256(hashlib.sha256(data).digest()).digest(), np.uint8)


def _pubkey_convert(v, b):
    if v[1] != 33:
        return NotImplemented
    xy = _parse33(b[0])
    if xy is None:
        return 0
    b[2][:], b[3][:] = _compressed(xy), xy
    return 1


def _opaque_pubkey(v, b):
    xy = _parse33(b[0])
    if xy is None:
        return 0
    b[1][:] = _le(xy)
    return 1


def _sig_ok(sig):
    return int.from_bytes(sig[:32].tobytes(), "big") < N_ORDER and int.from_bytes(sig[32:64].tobytes(), "big") < N_ORDER


def _opaque_sig(v, b):
    if not _sig_ok(b[0]):
        return 0
    b[1][:] = _le(b[0][:64])
    return 1


def _cln_opaque(v, b):
    xy = _parse33(b[1])
    if not _sig_ok(b[0]) or xy is None:
        return 0
    b[2][:], b[3][:] = _le(b[0][:64]), _le(xy)
    return 1


def _scalar_base_mult(v, b):
    xy = base_mult(int.from_bytes(b[0][:32].tobytes(), "big"))
    if xy is None:
        return 0
    b[1][:] = xy
    return 1


def _pubkey_create(v, b):
    xy = base_mult(int.from_bytes(b[0][:32].tobytes(), "big"))
    if xy is None:
        return 0
    b[1][:] = _compressed(xy)
    if b[2] is not None:
        b[2][:] = xy
    return 1


def ecdsa_sign(d, msg32):
    """secp256k1_ecdsa_sign with its default nonce (RFC 6979 HMAC-SHA256 over key || msg mod n): compact r || s, low s."""
    m = int.from_bytes(msg32, "big") % N_ORDER
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
        if 0 < k < N_ORDER:
            r = int.from_bytes(base_mult(k)[:32].tobytes(), "big") % N_ORDER
            s = pow(k, -1, N_ORDER) * (m + r * d) % N_ORDER
            if r and s:
                break
        K = mac(K, V + b"\x00")
        V = mac(K, V)
    return r.to_bytes(32, "big") + min(s, N_ORDER - s).to_bytes(32, "big")


def _tagged_hash(tag, data):
    t = hashlib.sha256(tag).digest()
    return hashlib.sha256(t + t + data).digest()


def schnorr_sign(d, msg32):
    """secp256k1_schnorrsig_sign32 without auxiliary randomness (BIP-340's nonce over 32 zero bytes): (sig64, xonly32)."""
    pxy = base_mult(d)
    px = pxy[:32].tobytes()
    if pxy[63] & 1:
        d = N_ORDER - d
    masked = bytes(a ^ b for a, b in zip(d.to_bytes(32, "big"), _tagged_hash(b"BIP0340/aux", bytes(32))))
    k = int.from_bytes(_tagged_hash(b"BIP0340/nonce", masked + px + msg32), "big") % N_ORDER
    rxy = base_mult(k)
    if rxy[63] & 1:
        k = N_ORDER - k
    rx = rxy[:32].tobytes()
    e = int.from_bytes(_tagged_hash(b"BIP0340/challenge", rx + px + msg32), "big") % N_ORDER
    return rx + ((k + e * d) % N_ORDER).to_bytes(32, "big"), px


def _seckey(b):
    d = int.from_bytes(b[:32].tobytes(), "big")
    return d if 0 < d < N_ORDER else None


def _ecdsa_sign(v, b):
    d = _seckey(b[0])
    if d is None:
        return 0
    b[2][:] = np.frombuffer(ecdsa_sign(d, b[1][:32].tobytes()), np.uint8)
    return 1


def _schnorr_sign(v, b):
    d = _seckey(b[0])
    if d is None:
        return 0
    sig, xonly = schnorr_sign(d, b[1][:32].tobytes())
    b[2][:], b[3][:] = np.frombuffer(sig, np.uint8), np.frombuffer(xonly, np.uint8)
    return 1


LOCAL = {
    "ref.ref_sha256d": _sha256d,
    "ref.ref_pubkey_convert": _pubkey_convert,
    "ref.ref_make_opaque_pubkey": _opaque_pubkey,
    "ref.ref_make_opaque_sig": _opaque_sig,
    "ref.ref_scalar_base_mult": _scalar_base_mult,
    "ref.ref_pubkey_create": _pubkey_create,
    "ref.ref_ecdsa_sign": _ecdsa_sign,
    "ref.ref_schnorr_sign": _schnorr_sign,
    "cln.cln_make_opaque": _cln_opaque,
}
