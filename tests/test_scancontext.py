"""ScanContext (K5): oracle sanity on CPU, GPU parity (-m gpu), and the sharded top-k exchange with gloo on CPU."""
import os
import sys

import numpy as np
import pytest


def test_oracle_sc_recovers_known_shift(oracle_mod, ilsm):
    db = ilsm.synth.sc_database(300)
    q, ids, shifts = ilsm.synth.sc_queries(db, 12)
    for j in range(len(q)):
        dist, idx, sh = oracle_mod.sc_topk(db.astype(np.float64), q[j].astype(np.float64), 3)
        assert idx[0] == ids[j] and sh[0] == shifts[j] and dist[0] < 0.13  # SC_DIST_THRES, Scancontext.h:91
        assert dist[1] > 0.3


def test_oracle_sc_superset_of_reference_candidates(oracle_mod, ilsm):
    """detectLoopClosureID scores 10 ring-key candidates (reference nanoflann, the committed candidate sets of
    tests/golden/ringkey_nanoflann.npz); brute-force scoring of every entry is a superset: same distance/shift for those
    ids, and a top-1 at least as good."""
    import hashlib
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ringkey_nanoflann.npz"))
    n, s0, nq, s1 = [int(v) for v in g["seeds"]]
    db32 = ilsm.synth.sc_database(n, seed=s0)
    q, _, _ = ilsm.synth.sc_queries(db32, nq, seed=s1)
    assert np.array_equal(np.frombuffer(hashlib.sha256(db32.tobytes() + q.tobytes()).digest(), np.uint8), g["sha256"])
    db = db32.astype(np.float64)
    for j in range(len(q)):
        dist, idx, sh = oracle_mod.sc_topk(db, q[j].astype(np.float64), len(db))
        lut = {int(i): (d, s) for d, i, s in zip(dist, idx, sh)}
        best = 10000000.0
        for c in g["candidates"][j]:
            d, s = oracle_mod.sc_distance(q[j].astype(np.float64), db[int(c)])
            assert lut[int(c)] == (d, s)
            best = min(best, d)
        assert dist[0] <= best


def test_oracle_sc_make(oracle_mod):
    pts = np.array([[10.0, 0.1, 1.0], [10.0, 0.2, 3.0], [-5.0, -5.0, -1.0], [100.0, 0.0, 9.0], [0.0, 30.0, 0.5]], np.float32)
    d = oracle_mod.sc_make(pts)
    assert d.shape == (20, 60) and d.max() == 5.0 and (d != 0).sum() == 3  # two points share a bin, one is beyond 80 m
    rk, sk = oracle_mod.sc_keys(d)
    assert np.isclose(rk.sum() * 60, d.sum()) and np.isclose(sk.sum() * 20, d.sum())


def test_merge_topk_is_deterministic(ilsm):
    dist = np.array([0.5, 0.1, 0.1, np.inf, 0.3, 0.7])
    ids = np.array([7, 9, 3, -1, 11, 2], np.int32)
    sh = np.array([1, 2, 3, 0, 5, 6], np.int32)
    od, oi, os_ = ilsm.merge_topk(dist, ids, sh, 4)
    assert oi.tolist() == [3, 9, 11, 7] and os_.tolist() == [3, 2, 5, 1] and od.tolist() == [0.1, 0.1, 0.3, 0.5]


def _shard_worker(rank, world, port, n_db, k, out):
    """One rank of the sharded query path with the CPU oracle standing in for the GPU scorer: local top-k on the
    rank's contiguous shard, one all_gather of k x (dist, id, shift), identical merge on every rank."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import ilsm_b200 as ilsm
    import oracle
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    db = ilsm.synth.sc_database(n_db)
    q, ids, shifts = ilsm.synth.sc_queries(db, 3)
    lo, hi = ilsm.shard_range(n_db, rank, world)
    results = []
    for j in range(len(q)):
        d, i, s = oracle.sc_topk(db[lo:hi].astype(np.float64), q[j].astype(np.float64), k)
        i = np.where(i >= 0, i + lo, -1).astype(np.int32)
        gd, gi, gs = ilsm.allgather_topk(d, i, s)
        results.append(ilsm.merge_topk(gd, gi, gs, k))
    if rank == 0:
        np.savez(out, dist=np.stack([r[0] for r in results]), ids=np.stack([r[1] for r in results]),
                 shifts=np.stack([r[2] for r in results]), true_ids=ids, true_shifts=shifts)
    dist.destroy_process_group()


def test_sharded_topk_gloo_world2(tmp_path, oracle_mod, ilsm):
    import torch.multiprocessing as mp
    n_db, k = 240, 5
    out = str(tmp_path / "merged.npz")
    port = 29500 + (os.getpid() % 2000)
    mp.spawn(_shard_worker, args=(2, port, n_db, k, out), nprocs=2, join=True)
    r = np.load(out)
    db = ilsm.synth.sc_database(n_db)
    q, ids, shifts = ilsm.synth.sc_queries(db, 3)
    for j in range(3):
        d, i, s = oracle_mod.sc_topk(db.astype(np.float64), q[j].astype(np.float64), k)
        assert np.array_equal(r["ids"][j], i) and np.array_equal(r["shifts"][j], s) and np.array_equal(r["dist"][j], d)
        assert r["ids"][j][0] == ids[j] and r["shifts"][j][0] == shifts[j]


# ------------------------------------------------------------------------------------------------- GPU parity
@pytest.mark.gpu
def test_gpu_sc_make_matches_oracle(ctx, oracle_mod, ilsm, cfg_full):
    sc = ilsm.ScanContextDb(ctx)
    for pts in (cfg_full["cloud"], cfg_full["map_surf"][:30000], np.zeros((0, 3), np.float32)):
        got = sc.make_scancontext(pts)
        want = oracle_mod.sc_make(pts) if len(pts) else np.zeros((20, 60))
        assert np.array_equal(got.astype(np.float64), want)
    sc.close()


@pytest.mark.gpu
def test_gpu_sc_topk_matches_oracle(ctx, oracle_mod, ilsm):
    db = ilsm.synth.sc_database(2000)
    db[17] = 0.0                      # an all-empty descriptor: no effective column -> "no match" distance
    db[18, :, 10:20] = 0.0            # partially empty columns
    q, ids, shifts = ilsm.synth.sc_queries(db, 8)
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db[:700])
    sc.add(db[700:])                  # growth keeps the contents
    assert len(sc) == 2000
    for j in range(len(q)):
        d, i, s = sc.query_topk(q[j], k=10)
        wd, wi, ws = oracle_mod.sc_topk(db.astype(np.float64), q[j].astype(np.float64), 10)
        assert np.array_equal(i, wi) and np.array_equal(s, ws)
        assert np.allclose(d, wd, rtol=1e-12, atol=1e-14)
        assert i[0] == ids[j] and s[0] == shifts[j]
    # excluding the most recent entries (NUM_EXCLUDE_RECENT) and a shard offset
    d, i, s = sc.query_topk(q[0], k=5, n_search=1950, id_offset=1000)
    wd, wi, ws = oracle_mod.sc_topk(db[:1950].astype(np.float64), q[0].astype(np.float64), 5)
    assert np.array_equal(i, wi + 1000) and np.array_equal(s, ws)
    # fewer entries than k
    d, i, s = sc.query_topk(q[0], k=8, n_search=3)
    assert (i[3:] == -1).all() and np.isinf(d[3:]).all()
    sc.close()


@pytest.mark.gpu
def test_gpu_sc_sharded_equals_unsharded(ctx, oracle_mod, ilsm):
    """R shards simulated in one process: per-shard local top-k + merge == top-k over the whole database."""
    db = ilsm.synth.sc_database(3000, seed=99)
    q, ids, shifts = ilsm.synth.sc_queries(db, 4, seed=100)
    whole = ilsm.ScanContextDb(ctx)
    whole.add(db)
    for R in (2, 4, 8):
        shards = []
        for r in range(R):
            lo, hi = ilsm.shard_range(len(db), r, R)
            s = ilsm.ScanContextDb(ctx)
            s.add(db[lo:hi])
            shards.append((s, lo))
        for j in range(len(q)):
            parts = [s.query_topk(q[j], k=10, id_offset=lo) for s, lo in shards]
            md, mi, ms = ilsm.merge_topk(np.concatenate([p[0] for p in parts]), np.concatenate([p[1] for p in parts]),
                                         np.concatenate([p[2] for p in parts]), 10)
            wd, wi, ws = whole.query_topk(q[j], k=10)
            assert np.array_equal(mi, wi) and np.array_equal(ms, ws) and np.array_equal(md, wd)
        for s, _ in shards:
            s.close()
    whole.close()


@pytest.mark.gpu
def test_gpu_sc_candidates_match_reference_nanoflann(ctx, oracle_mod, ilsm):
    """detectLoopClosureID the reference's way (Scancontext.cpp:283-312): the 10 ring-key candidates must be the result
    set of the REFERENCE'S OWN nanoflann tree (KDTreeVectorOfVectorsAdaptor, oracle/_ref -- prebuilt, it travels with
    the snapshot), in its order, and the loop id / distance / shift those of the candidate loop over them."""
    if oracle_mod.ref() is None:
        pytest.skip("oracle/_ref/libref_nanoflann.so not available")
    db = ilsm.synth.sc_database(600, seed=7)
    q, ids, shifts = ilsm.synth.sc_queries(db, 12, seed=8)
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db[:250])
    sc.add(db[250:])  # ring keys follow the database through growth
    dbd = db.astype(np.float64)
    for n_search in (600, 550, 37, 12):
        for j in range(len(q)):
            cid, ckd, cd, cs = sc.query_candidates(q[j], 10, n_search)
            arg, best, align, ref_ids = oracle_mod.sc_detect_loop_reference(dbd[:n_search], q[j].astype(np.float64))
            m = min(10, n_search)
            assert np.array_equal(cid[:m], ref_ids[:m]), (n_search, j)
            assert (cid[m:] == -1).all() and np.isinf(cd[m:]).all()
            assert (np.diff(ckd[:m]) >= 0).all()
            for t in range(m):  # every candidate's distance / shift = distanceBtnScanContext
                wd, ws = oracle_mod.sc_distance(q[j].astype(np.float64), dbd[cid[t]])
                assert abs(cd[t] - wd) <= 1e-12 and cs[t] == ws
            loop, dmin, sh, nn = sc.detect_loop_closure_id(q[j], n_search)
            assert nn == arg and sh == align and abs(dmin - best) <= 1e-12
            assert loop == (arg if best < 0.13 else -1)
    # a tree with fewer entries than candidates (51..59 keyframes in all): every entry is a candidate, the rest is padding
    cid, ckd, cd, cs = sc.query_candidates(q[0], 10, 7)
    assert sorted(cid[:7].tolist()) == list(range(7)) and (cid[7:] == -1).all() and (np.diff(ckd[:7]) >= 0).all()
    # the query re-renders of database entries are found when their entry is inside the window (ring keys are
    # rotation-invariant), and the exhaustive search agrees there
    for j in range(len(q)):
        loop, dmin, sh, nn = sc.detect_loop_closure_id(q[j], 600)
        assert nn == ids[j] and sh == shifts[j]
        assert sc.detect_loop_closure_id(q[j], 600, exhaustive=True)[3] == ids[j]
    sc.close()


@pytest.mark.gpu
def test_gpu_sc_candidates_golden_reference_sets(ctx, ilsm):
    """The committed reference candidate sets (tests/golden/ringkey_nanoflann.npz, made by the reference's tree)."""
    import hashlib
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ringkey_nanoflann.npz"))
    n, s0, nq, s1 = [int(v) for v in g["seeds"]]
    db = ilsm.synth.sc_database(n, seed=s0)
    qs, _, _ = ilsm.synth.sc_queries(db, nq, seed=s1)
    assert np.array_equal(np.frombuffer(hashlib.sha256(db.tobytes() + qs.tobytes()).digest(), np.uint8), g["sha256"])
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db)
    for j in range(nq):
        cid, _, _, _ = sc.query_candidates(qs[j], 10)
        assert np.array_equal(cid, g["candidates"][j].astype(np.int32)), j
    sc.close()


@pytest.mark.gpu
def test_gpu_sc_batch_equals_single_queries(ctx, ilsm):
    db = ilsm.synth.sc_database(1500, seed=21)
    q, _, _ = ilsm.synth.sc_queries(db, 9, seed=22)
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db)
    bd, bi, bs = sc.query_topk_batch(q, k=10, n_search=1400, id_offset=5)
    for j in range(len(q)):
        d, i, s = sc.query_topk(q[j], k=10, n_search=1400, id_offset=5)
        assert np.array_equal(bd[j], d) and np.array_equal(bi[j], i) and np.array_equal(bs[j], s)
    # without a communicator the sharded entry point is the batch query
    sd, si, ss = sc.query_topk_sharded(q, k=10, n_search=1400, id_offset=5)
    assert np.array_equal(sd, bd) and np.array_equal(si, bi) and np.array_equal(ss, bs)
    sc.close()


def _edge_case_db(ilsm, n, seed):
    db = ilsm.synth.sc_database(n, seed=seed)
    db[17] = 0.0                      # an all-empty descriptor: no effective column
    db[18, :, 10:20] = 0.0            # partially empty columns
    db[19] = db[3]                    # exact duplicates of other entries
    db[20] = np.roll(db[3], 7, axis=1)
    db[21, :, :] = db[21, :, :1]      # every column identical: the sector-key alignment is a 60-way tie
    return db


@pytest.mark.gpu
def test_gpu_sc_prefilter_approximates_exact(ctx, oracle_mod, ilsm):
    """The tensor-core prefilter (scancontext_tc.cu) against the exact scorer, pair by pair: an unflagged pair must carry
    the exact aligned shift (fastAlignUsingVkey) and a distance within the stated bound of distanceBtnScanContext's."""
    db = _edge_case_db(ilsm, 1500, 31)
    q, ids, shifts = ilsm.synth.sc_queries(db, 8, seed=32)
    q[7] = db[21]                     # a query whose own alignment is ambiguous against everything
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db)
    D, S = sc.prefilter_debug(q)
    dbd, qd = db.astype(np.float64), q.astype(np.float64)
    keys = dbd.mean(axis=1)           # sector keys: column means (Scancontext.cpp:222-235)
    flagged = D < 0               # -1: flagged outright; <= -2: one of two alignments, -2 - (lower bound of the distance)
    dual = D <= -2
    assert flagged[:7].mean() < 0.05, flagged.mean()
    assert (D[:7] == -1).mean() < 0.01, (D[:7] == -1).mean()
    worst = 0.0
    for j in range(8):
        qk = qd[j].mean(axis=0)
        for c in range(0, len(db), 3):
            if dual[j, c]:
                wd, _ = oracle_mod.sc_distance(qd[j], dbd[c])
                lo = -2.0 - float(D[j, c])
                assert lo <= min(wd, 1e30) + 1.5e-3, (j, c, lo, wd)
                continue
            if flagged[j, c]:
                continue
            norms = [np.linalg.norm(qk - np.roll(keys[c], s)) for s in range(60)]
            assert int(np.argmin(norms)) == int(S[j, c]), (j, c)
            wd, _ = oracle_mod.sc_distance(qd[j], dbd[c])
            if wd < 1e6:
                worst = max(worst, abs(float(D[j, c]) - wd))
            else:
                assert D[j, c] > 1e6
    assert worst <= 1.5e-3, worst
    # degenerate pairs are flagged, not guessed: the all-equal-columns entry and query
    assert flagged[:, 21].all() and flagged[7].all()
    sc.close()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [10, 1, 16])
def test_gpu_sc_tc_batch_equals_exact_scan(ctx, oracle_mod, ilsm, k):
    """A shard large enough for the two-step path (prefilter + exact rescoring): the reported top-k must be the one the
    exact scan of every entry gives -- ids, shifts and distances -- including empty descriptors, duplicates (distance
    ties resolved by id) and alignment ties."""
    db = _edge_case_db(ilsm, 6000, 41)
    q, ids, shifts = ilsm.synth.sc_queries(db, 11, seed=42)
    q[9] = db[21]
    q[10] = 0.0                       # an empty query: nothing is effective
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db)
    bd, bi, bs = sc.query_topk_batch(q, k=k, n_search=5950, id_offset=100)
    dbd = db[:5950].astype(np.float64)
    for j in range(len(q) - 1):  # (the all-zero query is checked against the single-query exact path below: its sector-key
        # alignment is a 60-way tie that summation order decides, in the reference as much as here)
        wd, wi, ws = oracle_mod.sc_topk(dbd, q[j].astype(np.float64), k)
        assert np.array_equal(bi[j], np.where(wi >= 0, wi + 100, -1)), (j, bi[j], wi)
        if j == 9:  # constant sector key: every shift ties exactly, rounding noise decides -- ids and distances only
            continue
        assert np.array_equal(bs[j], ws), j
        fin = np.isfinite(wd)
        assert np.allclose(bd[j][fin], wd[fin], rtol=1e-12, atol=1e-14), j
    for j in range(9):
        assert bi[j, 0] == ids[j] + 100 and bs[j, 0] == shifts[j]
    # the single-query entry point keeps the plain exact scan: same answers
    for j in (0, 9, 10):  # 9: the query IS an entry -- its distance to itself is a tiny NEGATIVE number and must still sort first
        d1, i1, s1 = sc.query_topk(q[j], k=k, n_search=5950, id_offset=100)
        assert np.array_equal(i1, bi[j]) and np.array_equal(s1, bs[j]) and np.array_equal(d1, bd[j])
    assert bi[9, 0] == 121 and abs(bd[9, 0]) < 1e-12
    sc.close()


@pytest.mark.gpu
def test_gpu_scancontext_matches_reference_code_golden(ctx, ilsm):
    """The CUDA ScanContext against outputs of the REFERENCE's own code (Scancontext.cpp compiled unmodified,
    tests/golden/make_golden_scancontext.py): descriptors bit for bit, column-shift distances / shifts of 48 pairs, and
    detectLoopClosureID (the reference's nanoflann tree + candidate loop + 0.13 threshold) for 12 queries."""
    import os, sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    from make_golden_scancontext import database, frames
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "scancontext_reference.npz"))
    sc = ilsm.ScanContextDb(ctx)
    for k, cloud in enumerate(frames()):
        assert np.array_equal(np.asarray(sc.make_scancontext(cloud), np.float64), gold[f"desc{k}"]), k
    db, queries, ids, shifts, pairs = database()
    sc.add(db[:251])  # what the reference's tree holds when the 301st keyframe asks: all but the 50 most recent
    for j in range(len(queries)):
        lid, best, align, _ = sc.detect_loop_closure_id(queries[j])
        assert lid == gold["detect_id"][j], j
        if lid >= 0:
            assert abs(np.float32(np.deg2rad(align * 6.0)) - gold["detect_yaw"][j]) < 1e-6, j
    sc.close()
    # pair distances through the exhaustive scorer over the whole database
    sc = ilsm.ScanContextDb(ctx)
    sc.add(db)
    for j in range(len(queries)):
        d, i, s = sc.query_topk(queries[j], k=16)
        full = {int(ii): (float(dd), int(ss)) for dd, ii, ss in zip(d, i, s)}
        for n, (jj, c) in enumerate(pairs):
            if jj == j and c in full:
                assert abs(full[c][0] - gold["pair_dist"][n]) <= 1e-12 and full[c][1] == gold["pair_shift"][n], (j, c)
    sc.close()
