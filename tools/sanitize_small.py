"""Small end-to-end run of every kernel, meant to be executed under compute-sanitizer."""
import os, sys, ctypes
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import lightning_b200 as L
from tests import util
ref = util.load_ref()
eng = L.SigVerifier(0)
w = util.corrupt(util.make_signed(300, seed=3), every=5)
for n in (1, 5, 300):
    for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
        got = eng.verify(kind, w["msg"][:n], w[k][:n], w[s][:n])
        want = util.ref_verify(ref, kind, w["msg"][:n], w[k][:n], w[s][:n])
        assert np.array_equal(got, want), (n, kind)
print("batch ok")
lib = eng.lib
lib.check_schnorr_sig.restype = ctypes.c_bool
opk = np.zeros(64, np.uint8)
assert ref.ref_make_opaque_pubkey(util.P(np.ascontiguousarray(w["pub33"][1])), util.P(opk))
r = lib.check_schnorr_sig(util.P(np.ascontiguousarray(w["msg"][1])), util.P(opk), util.P(np.ascontiguousarray(w["ssig"][1])))
print("dropin schnorr", r)
# newer entry points: gossip slicing, BIP143, same-key
from tests import gossip
msgs = gossip.load_subset()
sel = [m for m in msgs if m[:2] == b"\x01\x00"][:20] + [m for m in msgs if m[:2] == b"\x01\x01"][:20] + [b"\x01\x00" + bytes(50)]
print("gossip", list(eng.verify_gossip(sel))[-3:])
rng = np.random.default_rng(1)
txs, blob = util.make_htlc_txs(rng, 40)
keys = np.tile(w["pubxy"][0], (40, 1))
print("tx", eng.check_tx_sigs(1, txs, blob, keys, w["sig"][:40]).sum())
print("samekey", eng.verify_samekey(0, w["pub33"][0], w["msg"][:70], w["sig"][:70]).sum())
# round 2: both dispatch paths, mixed kinds, key de-duplication, BIP-340 batch verification, the self-test kernel
eng.set_small_max(0)
for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
    got = eng.verify(kind, w["msg"], w[k], w[s])
    assert np.array_equal(got, util.ref_verify(ref, kind, w["msg"], w[k], w[s])), kind
eng.set_small_max(8192)
print("throughput kernels on a small batch ok")
kinds = (np.arange(300) % 3).astype(np.uint8)
key = np.zeros((300, 64), np.uint8)
sig = np.zeros((300, 64), np.uint8)
for kind, (k, s) in enumerate([("pub33", "sig"), ("pubxy", "sig"), ("xonly", "ssig")]):
    sel = np.nonzero(kinds == kind)[0]
    key[sel, :w[k].shape[1]] = w[k][sel]
    sig[sel] = w[s][sel]
print("mixed", eng.verify_mixed(kinds, w["msg"], key, sig).sum())
big = [m for m in msgs if m[:2] in (b"\x01\x00", b"\x01\x01")][:1500]
eng.set_small_max(0)  # the key search only runs above the small-batch limit
st = eng.verify_gossip(big)
eng.set_small_max(8192)
print("gossip with de-duplication", int((st == 0).sum()), "of", len(big), "distinct keys", eng.last_distinct_keys())
w2 = util.make_signed(1100, seed=4)
v, gt, gf = eng.verify_schnorr_batch(w2["msg"], w2["xonly"], w2["ssig"], seed32=bytes(32))
print("schnorr batch", int(v.sum()), gt, gf)
w2["ssig"][5, 40] ^= 1
v, gt, gf = eng.verify_schnorr_batch(w2["msg"], w2["xonly"], w2["ssig"], seed32=bytes(32))
print("schnorr batch with one bad signature", int(v.sum()), gt, gf)
a = np.random.default_rng(2).integers(0, 2**32, size=(64, 8), dtype=np.uint32)
for op in (0, 1, 2, 3, 20, 24, 28, 31, 32):
    eng.selftest(op, a, a[::-1].copy())
print("selftest ops ok")
