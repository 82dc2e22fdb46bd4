"""Public-key recovery on the B200 (sv_recover_host, SigVerifier.recover, ecdsa_recover_batch) against the reference's
secp256k1_ecdsa_recover, on the small-batch kernel and on the throughput kernels."""
import ctypes

import numpy as np
import pytest

from tests import recovery as R
from tests.util import P

pytestmark = pytest.mark.gpu

SMALL_CAP = 8192


@pytest.fixture(scope="module")
def cases():
    """every set the reference's answers are kept for, concatenated: inputs, statuses, key digests"""
    sets = R.sets()
    want = [R.reference(name, w) for name, w in sets.items()]
    keys = ("msg", "sig", "recid", "signer")
    w = {k: np.concatenate([s[k] for s in sets.values()]) for k in keys}
    return w, np.concatenate([s for s, _ in want]), np.concatenate([d for _, d in want])


def _recover(engine, w, lo=0, hi=None, chunk=None):
    hi = w["msg"].shape[0] if hi is None else hi
    chunk = chunk or (hi - lo)
    xs, ss = [], []
    for a in range(lo, hi, chunk):
        b = min(hi, a + chunk)
        x, s = engine.recover(w["msg"][a:b], w["sig"][a:b], w["recid"][a:b])
        xs.append(x)
        ss.append(s)
    return np.concatenate(xs), np.concatenate(ss)


def _same(got, want, what):
    bad = R.mismatches(got[0], got[1], want)
    assert bad.size == 0, f"{what}: {bad.size} items differ from the reference, first {bad[:8].tolist()}"


@pytest.mark.parametrize("small_max", [SMALL_CAP, 0])
def test_all_sets_both_paths(engine, cases, small_max):
    w, ws, wd = cases
    old = engine.small_max()
    engine.set_small_max(small_max)
    try:
        got = _recover(engine, w, chunk=4096 if small_max else None)
    finally:
        engine.set_small_max(old)
    _same(got, (ws, wd), f"small_max={small_max}")
    signer = w["signer"].any(axis=1)
    assert (got[1][signer] == 1).all() and np.array_equal(got[0][signer], w["signer"][signer])
    assert set(np.unique(ws).tolist()) == {-1, 0, 1}


def test_ragged_sizes(engine, cases):
    w, ws, wd = cases
    assert engine.small_max() == SMALL_CAP
    for n in (1, 2, 31, 32, 33, 63, 64, 65, 483, 4095, 4096, 4097, 8191, 8192, 8193, 8200):
        got = _recover(engine, w, 0, n)
        _same(got, (ws[:n], wd[:n]), f"n={n}")
    # the same items at an offset: a batch boundary never lines up with a prep or final batch of the first call
    got = _recover(engine, w, 37, 37 + 8200)
    _same(got, (ws[37:37 + 8200], wd[37:37 + 8200]), "offset 37")


def test_recovered_keys_verify(engine, cases):
    """every key recovered from a low-s signature verifies that signature (secp256k1_ecdsa_verify's low-S rule)"""
    w, ws, wd = cases
    xy, st = _recover(engine, w)
    _same((xy, st), (ws, wd), "all sets")
    s = w["sig"][:, 32:]
    half = np.frombuffer((R.N // 2).to_bytes(32, "big"), np.uint8)
    low = np.array([bytes(x) <= bytes(half) for x in s])
    sel = np.nonzero((st == 1) & low)[0]
    assert sel.size > 4000
    from lightning_b200 import KIND_ECDSA_XY
    v = engine.verify(KIND_ECDSA_XY, w["msg"][sel], xy[sel], w["sig"][sel])
    assert v.all()


def test_batch_above_host_chunk(engine):
    """2.2 M synthetic signatures (more than one SV_HOST_CHUNK slice of 2^21): recid 0 first, recid 1 for the items whose
    key did not come back; together they must give every signer's key"""
    import torch
    from lightning_b200 import KIND_ECDSA33
    n = (1 << 21) + 100_000
    msg = torch.empty((n, 32), dtype=torch.uint8, device="cuda")
    key = torch.empty((n, 33), dtype=torch.uint8, device="cuda")
    sig = torch.empty((n, 64), dtype=torch.uint8, device="cuda")
    engine.synth_device(KIND_ECDSA33, 91, n, msg.data_ptr(), key.data_ptr(), sig.data_ptr())
    engine.sync()
    m, k, s = (t.cpu().numpy() for t in (msg, key, sig))
    del msg, key, sig

    def matches(xy, st):
        return (st == 1) & ((xy[:, 63] & 1) == k[:, 0] - 2) & (xy[:, :32] == k[:, 1:]).all(axis=1)

    xy, st = engine.recover(m, s, np.zeros(n, np.uint8))
    hit = matches(xy, st)
    assert 0.4 * n < hit.sum() < 0.6 * n
    miss = np.nonzero(~hit)[0]
    xy1, st1 = engine.recover(m[miss], s[miss], np.ones(miss.size, np.uint8))
    assert (st1 == 1).all()
    assert (((xy1[:, 63] & 1) == k[miss, 0] - 2) & (xy1[:, :32] == k[miss, 1:]).all(axis=1)).all()


def test_dropin_bolt11_vectors(engine):
    """ecdsa_recover_batch on the struct CLN holds after secp256k1_ecdsa_recoverable_signature_parse_compact: the BOLT #11
    invoices of common/test/run-bolt11.c give the node id the file signs with"""
    w, vec = R.golden()
    sel = [i for i, v in enumerate(vec) if v["set"] == "bolt11"]
    n = len(sel)
    sigs = np.zeros((n, 65), np.uint8)
    for j, i in enumerate(sel):
        sigs[j, :32] = w["sig"][i, 31::-1]
        sigs[j, 32:64] = w["sig"][i, 63:31:-1]
        sigs[j, 64] = w["recid"][i]
    hashes = np.ascontiguousarray(w["msg"][sel])
    keys = np.zeros((n, 64), np.uint8)
    ok = (ctypes.c_bool * n)()
    engine.lib.ecdsa_recover_batch(P(sigs), P(hashes), ctypes.c_size_t(n), P(keys), ok)
    assert all(ok)
    for j, i in enumerate(sel):
        x, y = keys[j, 31::-1], keys[j, 63:31:-1]
        assert bytes([2 + (y[31] & 1)]).hex() + bytes(x).hex() == vec[i]["node_id"]
    # a corrupted signature still recovers some key, just not the node's; s = 0 recovers none and leaves the key zero
    sigs[0, 40] ^= 1
    sigs[1, 32:64] = 0
    keys[:] = 7
    engine.lib.ecdsa_recover_batch(P(sigs), P(hashes), ctypes.c_size_t(n), P(keys), ok)
    assert ok[0] and not ok[1] and all(ok[2:])
    assert bytes(keys[0, 31::-1]).hex() != vec[sel[0]]["node_id"][2:] and not keys[1].any()
