"""Public-key recovery, host build of the device code (tests/host_emul/emul_recover.cpp) against the reference's
secp256k1_ecdsa_recover (its answers as tests/golden/recovery_reference.npz keeps them).

Both schedules the engine runs are compared: the throughput one (r inverted in batches of 32, Q parked, keys in batches of
16) and the small-batch one (one lone inversion of r, half ladders on lane pairs, one field inversion per item)."""
import numpy as np
import pytest

from tests import recovery as R

SCHEDULES = [False, True]


@pytest.fixture(scope="module")
def emul_rec():
    return R.load_emul()


def _check(emul, name, w, small):
    got_xy, got_st = R.emul_recover(emul, w, small=small)
    bad = R.mismatches(got_xy, got_st, R.reference(name, w))
    assert bad.size == 0, f"{bad.size} items differ from the reference, first {bad[:8].tolist()}"
    return got_xy, got_st


@pytest.mark.parametrize("small", SCHEDULES)
def test_golden_vectors(emul_rec, small):
    w, vec = R.golden()
    xy, st = _check(emul_rec, "golden", w, small)
    assert np.array_equal(st, w["status"]) and np.array_equal(xy, w["xy"])
    # tests_impl.h:185-192: the first signature recovers with recid 1 only, (4, 4) with every recid
    assert st[:8].tolist() == [0, 1, 0, 0, 1, 1, 1, 1]
    for v, x in zip(vec, xy):
        if v["set"] == "bolt11":
            assert bytes([2 + (x[63] & 1)]).hex() + bytes(x[:32]).hex() == v["node_id"]


@pytest.mark.parametrize("small", SCHEDULES)
def test_signed_all_recids_and_high_s_twins(emul_rec, small):
    w = R.signed(2000, seed=31)
    xy, st = _check(emul_rec, "signed", w, small)
    signer = w["signer"].any(axis=1)
    assert signer.sum() == 4000
    # the signature's own recid and its high-S twin with recid ^ 1 both give the signer's key: no low-S rule
    assert (st[signer] == 1).all() and np.array_equal(xy[signer], w["signer"][signer])


@pytest.mark.parametrize("small", SCHEDULES)
def test_edge_encodings(emul_rec, small):
    w = R.edge(seed=5)
    xy, st = _check(emul_rec, "edge", w, small)
    assert (st == -1).sum() >= 5 * 4 + 5 and (st == 0).any() and (st == 1).any()
    assert not xy[st != 1].any()
    assert st[-1] == 1 and np.array_equal(xy[-1], w["signer"][-1])


@pytest.mark.parametrize("small", SCHEDULES)
def test_constructed_cases(emul_rec, small):
    w = R.constructed(seed=77)
    xy, st = _check(emul_rec, "constructed", w, small)
    # r + n lifts for recid 2 / 3 where r < p - n, never where r >= p - n
    per_seed = 6
    lifted = np.concatenate([st[i * per_seed:i * per_seed + 4] for i in range(8)])
    assert (lifted[[k for k in range(lifted.size) if k % 4 >= 2]] == 1).all()
    too_big = np.concatenate([st[i * per_seed + 4:i * per_seed + 6] for i in range(8)])
    assert (too_big == 0).all()
    # s R = m G gives infinity (status 0), s R = -m G a doubling (status 1)
    tail = st[8 * per_seed:]
    assert tail.size >= 2 and (tail[0::2] == 0).all() and (tail[1::2] == 1).all()
