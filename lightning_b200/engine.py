"""ctypes binding of libcln_sigverify.so — the Python mirror of include/cln_sigverify.h.

The method names follow the reference surface they stand in for (bitcoin/signature.h:
check_signed_hash :85, check_schnorr_sig :129; common/node_id.h: check_signed_hash_nodeid :80;
bitcoin/shadouble.h: sha256_double), batched.  There is no Python or CPU implementation behind
this class: if the CUDA library or a GPU is missing, construction raises.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SV_LIB") or os.path.join(_HERE, "libcln_sigverify.so")  # SV_LIB: build variants (dev)

KIND_ECDSA33 = 0
KIND_ECDSA_XY = 1
KIND_SCHNORR = 2
KEY_SIZE = {KIND_ECDSA33: 33, KIND_ECDSA_XY: 64, KIND_SCHNORR: 32}

_c8 = ctypes.POINTER(ctypes.c_uint8)


class EngineError(RuntimeError):
    pass


class SvTx(ctypes.Structure):
    """sv_tx (include/cln_sigverify.h): the BIP143-relevant fields of a one-input one-output segwit transaction."""
    _fields_ = [("version", ctypes.c_uint32), ("locktime", ctypes.c_uint32), ("sequence", ctypes.c_uint32),
                ("sighash_type", ctypes.c_uint32), ("prev_txid", ctypes.c_uint8 * 32), ("prev_index", ctypes.c_uint32),
                ("script_off", ctypes.c_uint32), ("script_len", ctypes.c_uint32), ("out_script_off", ctypes.c_uint32),
                ("out_script_len", ctypes.c_uint32), ("flags", ctypes.c_uint32), ("input_amount", ctypes.c_uint64),
                ("output_amount", ctypes.c_uint64), ("prevouts_off", ctypes.c_uint32), ("prevouts_len", ctypes.c_uint32),
                ("sequences_off", ctypes.c_uint32), ("sequences_len", ctypes.c_uint32)]


class SvInfo(ctypes.Structure):
    _fields_ = [("device", ctypes.c_int), ("sm_count", ctypes.c_int), ("main_block", ctypes.c_int),
                ("main_grid", ctypes.c_int), ("main_regs", ctypes.c_int), ("gtable_bytes", ctypes.c_size_t),
                ("scratch_bytes", ctypes.c_size_t), ("launches", ctypes.c_ulonglong), ("l2_persist_bytes", ctypes.c_size_t), ("l2_max_persist_bytes", ctypes.c_size_t)]


def load_library():
    if not os.path.exists(LIB_PATH):
        raise EngineError(
            f"{LIB_PATH} is missing: build it with `python -m lightning_b200.build` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, sz, i = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    lib.sv_create.argtypes = [ctypes.POINTER(vp), i]
    lib.sv_destroy.argtypes = [vp]
    lib.sv_destroy.restype = None
    lib.sv_last_error.argtypes = [vp]
    lib.sv_last_error.restype = ctypes.c_char_p
    lib.sv_key_size.argtypes = [i]
    lib.sv_key_size.restype = sz
    lib.sv_verify_host.argtypes = [vp, i, vp, vp, vp, sz, vp]
    lib.sv_verify_host_raw.argtypes = [vp, i, vp, sz, vp, vp, vp, vp, sz, vp]
    lib.sv_verify_device.argtypes = [vp, i, vp, vp, vp, sz, vp, vp, vp]
    lib.sv_verify_gossip_host.argtypes = [vp, vp, sz, vp, vp, sz, vp, vp]
    lib.sv_verify_tx_host.argtypes = [vp, i, vp, vp, sz, vp, vp, sz, vp, vp]
    lib.sv_verify_samekey_host.argtypes = [vp, i, vp, vp, vp, sz, vp]
    lib.sv_sync.argtypes = [vp, vp]
    lib.sv_get_stream.argtypes = [vp]
    lib.sv_set_profiling.argtypes = [vp, i]
    lib.sv_get_last_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float)]
    lib.sv_get_stream.restype = vp
    lib.sv_enqueue.argtypes = [vp, i, vp, vp, vp]
    lib.sv_enqueue.restype = ctypes.c_long
    lib.sv_pending.argtypes = [vp]
    lib.sv_pending.restype = sz
    lib.sv_flush.argtypes = [vp, vp, sz]
    lib.sv_sha256d_host.argtypes = [vp, vp, sz, vp, vp, sz, vp]
    lib.sv_pubkey_parse_host.argtypes = [vp, vp, sz, vp, vp]
    lib.sv_recover_host.argtypes = [vp, vp, vp, vp, sz, vp, vp]
    lib.sv_synth_device.argtypes = [vp, i, ctypes.c_uint64, sz, vp, vp, vp, vp]
    lib.sv_selftest_host.argtypes = [vp, i, vp, vp, sz, vp]
    lib.sv_verify_mixed_host.argtypes = [vp, vp, vp, vp, vp, sz, vp]
    lib.sv_verify_mixed_device.argtypes = [vp, vp, vp, vp, vp, sz, vp, vp]
    lib.sv_verify_schnorr_batch_host.argtypes = [vp, vp, vp, vp, sz, vp, vp, vp, vp]
    lib.sv_set_dedup.argtypes = [vp, i]
    lib.sv_set_nosqrt.argtypes = [vp, i]
    lib.sv_last_distinct_keys.argtypes = [vp]
    lib.sv_last_distinct_keys.restype = ctypes.c_uint
    lib.sv_set_small_max.argtypes = [vp, sz]
    lib.sv_get_small_max.argtypes = [vp]
    lib.sv_get_small_max.restype = sz
    lib.sv_get_info.argtypes = [vp, ctypes.POINTER(SvInfo)]
    lib.sv_probe.argtypes = [vp, i, ctypes.POINTER(ctypes.c_double)]
    lib.sv_probe_imad_peak.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
    lib.sv_host_alloc.argtypes = [sz]
    lib.sv_host_alloc.restype = vp
    lib.sv_host_free.argtypes = [vp]
    lib.sv_host_free.restype = None
    return lib


def _u8(a, shape_tail):
    a = np.ascontiguousarray(a, dtype=np.uint8)
    if a.ndim == 1:
        a = a.reshape(-1, shape_tail)
    if a.shape[1] != shape_tail:
        raise ValueError(f"expected (*, {shape_tail}) uint8, got {a.shape}")
    return a


class SigVerifier:
    """One engine context on one GPU (sv_ctx)."""

    def __init__(self, device=0):
        self.lib = load_library()
        self._ctx = ctypes.c_void_p()
        rc = self.lib.sv_create(ctypes.byref(self._ctx), int(device))
        if rc != 0:
            msg = self.lib.sv_last_error(None).decode()
            self._ctx = ctypes.c_void_p()
            raise EngineError(f"sv_create(device={device}) failed ({rc}): {msg}")
        self.device = int(device)

    def close(self):
        if getattr(self, "_ctx", None) and self._ctx.value:
            self.lib.sv_destroy(self._ctx)
            self._ctx = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            raise EngineError(f"{what} failed ({rc}): {self.lib.sv_last_error(self._ctx).decode()}")

    # ---- host-buffer API -------------------------------------------------------------------
    def verify(self, kind, msg32, key, sig64):
        """Batch verify; returns a uint8 verdict vector.  Host numpy arrays in, host array out."""
        msg32 = _u8(msg32, 32)
        key = _u8(key, KEY_SIZE[kind])
        sig64 = _u8(sig64, 64)
        n = msg32.shape[0]
        if key.shape[0] != n or sig64.shape[0] != n:
            raise ValueError("length mismatch")
        out = np.zeros(n, dtype=np.uint8)
        self._check(self.lib.sv_verify_host(self._ctx, kind, msg32.ctypes.data, key.ctypes.data, sig64.ctypes.data,
                                            n, out.ctypes.data), "sv_verify_host")
        return out

    def check_signed_hash(self, hash32, sig64, pubxy64):
        """bitcoin/signature.c:174 check_signed_hash, batched (pre-decompressed keys)."""
        return self.verify(KIND_ECDSA_XY, hash32, pubxy64, sig64)

    def check_signed_hash_nodeid(self, hash32, sig64, node_id33):
        """common/node_id.c:72 check_signed_hash_nodeid, batched (33-byte keys)."""
        return self.verify(KIND_ECDSA33, hash32, node_id33, sig64)

    def check_schnorr_sig(self, hash32, xonly32, sig64):
        """bitcoin/signature.c:408 check_schnorr_sig, batched (x-only keys)."""
        return self.verify(KIND_SCHNORR, hash32, xonly32, sig64)

    def verify_raw(self, kind, data, off, length, key, sig64):
        """Verify over SHA256d(data[off:off+len]) computed on the device (gossipd/sigcheck.c path)."""
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        key = _u8(key, KEY_SIZE[kind])
        sig64 = _u8(sig64, 64)
        n = off.shape[0]
        out = np.zeros(n, dtype=np.uint8)
        self._check(self.lib.sv_verify_host_raw(self._ctx, kind, data.ctypes.data, data.size, off.ctypes.data,
                                                length.ctypes.data, key.ctypes.data, sig64.ctypes.data, n,
                                                out.ctypes.data), "sv_verify_host_raw")
        return out

    def verify_gossip(self, msgs, cu_signers=None):
        """Raw gossip wire messages in, one status per message out (0 ok, 1..4 first bad signature, -1 malformed);
        the device slices, hashes and verifies (gossipd/sigcheck.c, batched).  cu_signers: (n,33) or None."""
        lens = np.array([len(m) for m in msgs], dtype=np.uint32)
        offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64) if len(msgs) else np.zeros(0, np.uint64)
        blob = np.frombuffer(b"".join(bytes(m) for m in msgs), dtype=np.uint8)
        n = len(msgs)
        status = np.zeros(max(n, 1), dtype=np.int32)
        sg = None
        if cu_signers is not None:
            sg = _u8(cu_signers, 33)
        self._check(self.lib.sv_verify_gossip_host(self._ctx, blob.ctypes.data, blob.size, offs.ctypes.data, lens.ctypes.data, n,
                                                   sg.ctypes.data if sg is not None else None, status.ctypes.data),
                    "sv_verify_gossip_host")
        return status[:n]

    def verify_samekey(self, kind, key, msg32, sig64):
        """n ECDSA signatures by ONE key (channeld's HTLC loop): the key's table is built once on the device."""
        msg32 = _u8(msg32, 32)
        sig64 = _u8(sig64, 64)
        k = np.ascontiguousarray(key, dtype=np.uint8).reshape(-1)
        assert k.size == KEY_SIZE[kind]
        n = msg32.shape[0]
        out = np.zeros(max(n, 1), dtype=np.uint8)
        self._check(self.lib.sv_verify_samekey_host(self._ctx, kind, k.ctypes.data, msg32.ctypes.data, sig64.ctypes.data, n,
                                                    out.ctypes.data), "sv_verify_samekey_host")
        return out[:n]

    def check_tx_sigs(self, kind, txs, scripts, key, sig64, want_sighash=False):
        """check_tx_sig (bitcoin/signature.c:194) for n one-input one-output transactions with the BIP143 sighash
        computed on the device.  txs: ctypes array of SvTx; scripts: bytes blob; key (n, keysize); sig64 (n, 64)."""
        n = len(txs)
        key = _u8(key, KEY_SIZE[kind])
        sig64 = _u8(sig64, 64)
        blob = np.frombuffer(bytes(scripts) if len(scripts) else b"\0", dtype=np.uint8)
        out = np.zeros(max(n, 1), dtype=np.uint8)
        sh = np.zeros((max(n, 1), 32), dtype=np.uint8)
        self._check(self.lib.sv_verify_tx_host(self._ctx, kind, ctypes.addressof(txs), blob.ctypes.data, len(scripts),
                                               key.ctypes.data, sig64.ctypes.data, n, out.ctypes.data,
                                               sh.ctypes.data if want_sighash else None), "sv_verify_tx_host")
        return (out[:n], sh[:n]) if want_sighash else out[:n]

    def sha256_double(self, data, off, length):
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        length = np.ascontiguousarray(length, dtype=np.uint32)
        n = off.shape[0]
        out = np.zeros((n, 32), dtype=np.uint8)
        self._check(self.lib.sv_sha256d_host(self._ctx, data.ctypes.data, data.size, off.ctypes.data,
                                             length.ctypes.data, n, out.ctypes.data), "sv_sha256d_host")
        return out

    def pubkey_parse(self, key33):
        key33 = _u8(key33, 33)
        n = key33.shape[0]
        xy = np.zeros((n, 64), dtype=np.uint8)
        ok = np.zeros(n, dtype=np.uint8)
        self._check(self.lib.sv_pubkey_parse_host(self._ctx, key33.ctypes.data, n, xy.ctypes.data, ok.ctypes.data),
                    "sv_pubkey_parse_host")
        return xy, ok

    def recover(self, msg32, sig64, recid):
        """secp256k1_ecdsa_recover, batched (common/bolt11.c:1018-1050, lightningd/signmessage.c:178-193).  msg32 (n, 32),
        sig64 (n, 64) compact r || s, recid (n,) bytes.  Returns (xy64 (n, 64) uint8, status (n,) int8): 1 = key x || y,
        0 = no key (all zero), -1 = encoding refused (r >= n, s >= n or recid > 3)."""
        msg32, sig64 = _u8(msg32, 32), _u8(sig64, 64)
        recid = np.ascontiguousarray(recid, dtype=np.uint8).reshape(-1)
        n = msg32.shape[0]
        if sig64.shape[0] != n or recid.shape[0] != n:
            raise ValueError("length mismatch")
        xy = np.zeros((n, 64), dtype=np.uint8)
        status = np.zeros(n, dtype=np.int8)
        self._check(self.lib.sv_recover_host(self._ctx, msg32.ctypes.data, sig64.ctypes.data, recid.ctypes.data, n,
                                             xy.ctypes.data, status.ctypes.data), "sv_recover_host")
        return xy, status

    def verify_mixed(self, kinds, msg32, key64, sig64):
        """Interleaved batch: kinds (n,) uint8 SV_KIND_* tags, keys in 64-byte slots; verdicts in item order."""
        kinds = np.ascontiguousarray(kinds, dtype=np.uint8).reshape(-1)
        msg32, key64, sig64 = _u8(msg32, 32), _u8(key64, 64), _u8(sig64, 64)
        n = kinds.shape[0]
        out = np.zeros(max(n, 1), dtype=np.uint8)
        self._check(self.lib.sv_verify_mixed_host(self._ctx, kinds.ctypes.data, msg32.ctypes.data, key64.ctypes.data,
                                                  sig64.ctypes.data, n, out.ctypes.data), "sv_verify_mixed_host")
        return out[:n]

    def verify_schnorr_batch(self, msg32, xonly32, sig64, seed32=None):
        """BIP-340 batch verification (random linear combination per group of 1024, one-by-one for failed groups).
        Returns (verdicts, groups_total, groups_failed)."""
        msg32, xonly32, sig64 = _u8(msg32, 32), _u8(xonly32, 32), _u8(sig64, 64)
        n = msg32.shape[0]
        out = np.zeros(max(n, 1), dtype=np.uint8)
        gt, gf = ctypes.c_uint32(), ctypes.c_uint32()
        seed = np.ascontiguousarray(np.frombuffer(bytes(seed32), dtype=np.uint8)) if seed32 is not None else None
        self._check(self.lib.sv_verify_schnorr_batch_host(self._ctx, msg32.ctypes.data, xonly32.ctypes.data, sig64.ctypes.data, n,
                                                          seed.ctypes.data if seed is not None else None, out.ctypes.data,
                                                          ctypes.byref(gt), ctypes.byref(gf)), "sv_verify_schnorr_batch_host")
        return out[:n], gt.value, gf.value

    def set_dedup(self, on=True):
        self._check(self.lib.sv_set_dedup(self._ctx, 1 if on else 0), "sv_set_dedup")

    def set_nosqrt(self, on=True):
        """compressed-key ECDSA batches: the flow without the square root (default) or the plain one"""
        self._check(self.lib.sv_set_nosqrt(self._ctx, 1 if on else 0), "sv_set_nosqrt")

    def last_distinct_keys(self):
        return self.lib.sv_last_distinct_keys(self._ctx)

    def set_small_max(self, n):
        """largest batch that takes the small-batch (latency) path; 0 = always the throughput kernels"""
        self._check(self.lib.sv_set_small_max(self._ctx, int(n)), "sv_set_small_max")

    def small_max(self):
        return self.lib.sv_get_small_max(self._ctx)

    def selftest(self, op, a, b=None):
        """Run primitive `op` (SV_ST_* of cln_sigverify.h) of the device arithmetic on operands a, b: (n, 8) uint32
        little-endian limbs each; returns (n, 16) uint32.  Test support."""
        a = np.ascontiguousarray(a, dtype=np.uint32).reshape(-1, 8)
        b = np.zeros_like(a) if b is None else np.ascontiguousarray(b, dtype=np.uint32).reshape(-1, 8)
        if a.shape != b.shape:
            raise ValueError("operand shape mismatch")
        out = np.zeros((a.shape[0], 16), dtype=np.uint32)
        self._check(self.lib.sv_selftest_host(self._ctx, int(op), a.ctypes.data, b.ctypes.data, a.shape[0], out.ctypes.data),
                    "sv_selftest_host")
        return out

    # ---- deferral queue --------------------------------------------------------------------
    def enqueue(self, kind, msg32, key, sig64):
        m = np.ascontiguousarray(msg32, dtype=np.uint8)
        k = np.ascontiguousarray(key, dtype=np.uint8)
        s = np.ascontiguousarray(sig64, dtype=np.uint8)
        assert m.size == 32 and k.size == KEY_SIZE[kind] and s.size == 64
        idx = self.lib.sv_enqueue(self._ctx, kind, m.ctypes.data, k.ctypes.data, s.ctypes.data)
        if idx < 0:
            raise EngineError(f"sv_enqueue failed ({idx})")
        return idx

    def pending(self):
        return self.lib.sv_pending(self._ctx)

    def flush(self):
        n = self.pending()
        out = np.zeros(max(n, 1), dtype=np.uint8)
        self._check(self.lib.sv_flush(self._ctx, out.ctypes.data, n), "sv_flush")
        return out[:n]

    # ---- device-buffer API (pointers: ints, e.g. torch tensor .data_ptr()) -----------------
    def verify_device(self, kind, d_msg, d_key, d_sig, n, d_verdict, d_bitmap=0, stream=0):
        self._check(self.lib.sv_verify_device(self._ctx, kind, d_msg, d_key, d_sig, n, d_verdict, d_bitmap or None,
                                              stream or None), "sv_verify_device")

    def synth_device(self, kind, seed, n, d_msg, d_key, d_sig, stream=0):
        self._check(self.lib.sv_synth_device(self._ctx, kind, seed, n, d_msg, d_key, d_sig, stream or None),
                    "sv_synth_device")

    def stream_handle(self):
        """cudaStream_t of the context's own stream (wrap with torch.cuda.ExternalStream to time on it)."""
        return self.lib.sv_get_stream(self._ctx)

    def sync(self, stream=0):
        self._check(self.lib.sv_sync(self._ctx, stream or None), "sv_sync")

    def set_profiling(self, on=True):
        self._check(self.lib.sv_set_profiling(self._ctx, 1 if on else 0), "sv_set_profiling")

    def last_timing(self):
        """(prep_ms, main_ms) device time of the last verify launch pair; call after sync()."""
        a, b = ctypes.c_float(), ctypes.c_float()
        self._check(self.lib.sv_get_last_timing(self._ctx, ctypes.byref(a), ctypes.byref(b)), "sv_get_last_timing")
        return a.value, b.value

    def host_alloc(self, nbytes):
        """Pinned host buffer as a numpy uint8 array (cudaHostAlloc); free with host_free(arr)."""
        p = self.lib.sv_host_alloc(nbytes)
        if not p:
            raise EngineError("sv_host_alloc failed")
        buf = (ctypes.c_uint8 * nbytes).from_address(p)
        arr = np.frombuffer(buf, dtype=np.uint8)
        self._pinned = getattr(self, "_pinned", {})
        self._pinned[arr.ctypes.data] = p
        return arr

    def host_free(self, arr):
        p = getattr(self, "_pinned", {}).pop(arr.ctypes.data, None)
        if p:
            self.lib.sv_host_free(p)

    def info(self):
        inf = SvInfo()
        self._check(self.lib.sv_get_info(self._ctx, ctypes.byref(inf)), "sv_get_info")
        return {f[0]: getattr(inf, f[0]) for f in SvInfo._fields_}

    def probe(self, mode):
        v = ctypes.c_double()
        self._check(self.lib.sv_probe(self._ctx, mode, ctypes.byref(v)), "sv_probe")
        return v.value
