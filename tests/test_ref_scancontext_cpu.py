"""The oracle's ScanContext against the REFERENCE's own code: src/Scancontext.cpp + include/Scancontext.h compiled UNMODIFIED
(with the vendored nanoflann) into oracle/_ref/libref_scancontext.so on a small Eigen::MatrixXd stand-in -- descriptor, ring /
sector keys, distanceBtnScanContext and detectLoopClosureID end to end.  Live when the library exists, and against its
committed outputs everywhere."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
from make_golden_scancontext import database, frames  # noqa: E402

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "scancontext_reference.npz"))
NUM_EXCLUDE_RECENT = 50  # Scancontext.h:86


def oracle_detect(oracle_mod, db, q):
    """detectLoopClosureID as the node runs it: the query is saved first, the tree holds all but the 50 most recent.
    The 10 ring-key candidates are the float 10-NN by brute force (the reference's nanoflann tree returns the same set on
    the database of test_golden_cpu.py::test_oracle_ringkey_candidates_match_reference_golden; on this database the
    stored detect_id / detect_yaw are what catches a different set), then the best candidate by distanceBtnScanContext."""
    n_search = len(db) + 1 - NUM_EXCLUDE_RECENT
    qd = q.astype(np.float64)
    rk_db = np.stack([oracle_mod.sc_keys(d.astype(np.float64))[0] for d in db[:n_search]]).astype(np.float32)
    rk_q = oracle_mod.sc_keys(qd)[0].astype(np.float32)
    d2 = ((rk_db.astype(np.float64) - rk_q.astype(np.float64)) ** 2).sum(axis=1)
    best, arg, align = 10000000.0, 0, 0
    for c in np.argsort(d2, kind="stable")[:10]:
        d, s = oracle_mod.sc_distance(qd, db[c].astype(np.float64))
        if d < best:
            best, arg, align = d, int(c), s
    return (arg, align) if best < 0.13 else (-1, align)


def test_oracle_scancontext_equals_reference_golden(oracle_mod):
    for k, cloud in enumerate(frames()):
        d = oracle_mod.sc_make(cloud)
        assert np.array_equal(d, GOLD[f"desc{k}"]) and (d != 0).sum() > 100
        rk, sk = oracle_mod.sc_keys(d)
        assert np.array_equal(np.ravel(rk), GOLD[f"ring_key{k}"]) and np.array_equal(np.ravel(sk), GOLD[f"sector_key{k}"])
    db, queries, ids, shifts, pairs = database()
    for n, (j, c) in enumerate(pairs):
        dist, shift = oracle_mod.sc_distance(queries[j].astype(np.float64), db[c].astype(np.float64))
        assert dist == GOLD["pair_dist"][n] and shift == GOLD["pair_shift"][n], (j, c)
    for j in range(len(queries)):
        lid, align = oracle_detect(oracle_mod, db, queries[j])
        assert lid == GOLD["detect_id"][j], j
        assert abs(np.float32(np.deg2rad(align * 6.0)) - GOLD["detect_yaw"][j]) < 1e-6, j
    assert (GOLD["detect_id"][:6] == ids[:6]).all() and (GOLD["detect_id"][8:] == -1).all()


def test_oracle_scancontext_equals_reference_live(oracle_mod, ilsm):
    if oracle_mod.ref_scancontext() is None:
        pytest.skip("oracle/_ref/libref_scancontext.so not built (needs the reference tree)")
    S = ilsm.synth
    rng = np.random.default_rng(13)
    # descriptors of raw point sets, including points beyond 80 m, on bin boundaries and at the origin
    for k in range(3):
        pts = np.concatenate([rng.normal(0, 30, (4000, 3)) * [1, 1, 0.1], [[0, 0, 0], [80.0, 0, 1], [0, -80.0, 1], [4.0, 0.0, 2], [-4.0, 0.0, 2],
                                                                             [0.0, 4.0, 2], [120.0, 5.0, 1]]]).astype(np.float32)
        assert np.array_equal(oracle_mod.sc_make(pts), oracle_mod.ref_sc_make(pts)), k
    db = S.sc_database_range(100, 180, 400)
    q, ids, _ = S.sc_queries(db, 6, seed=21)
    for j in range(6):
        for c in (int(ids[j]), 0, 33, 79):
            assert oracle_mod.sc_distance(q[j].astype(np.float64), db[c].astype(np.float64)) == oracle_mod.ref_sc_distance(q[j], db[c]), (j, c)
        assert oracle_detect(oracle_mod, db, q[j])[0] == oracle_mod.ref_sc_detect(db, q[j])[0], j
    # an empty descriptor against a populated one: the reference divides 0 / 0, NaN never beats its initial 10000000 and
    # that is what distanceBtnScanContext returns; the oracle reports "no match" as a distance far above any threshold too
    d, _ = oracle_mod.ref_sc_distance(np.zeros((20, 60)), db[3])
    assert d == 10000000.0 and oracle_mod.sc_distance(np.zeros((20, 60)), db[3].astype(np.float64))[0] > 1e6
