"""IVFRABITQ on the device against the CPU restatement (tests/rabitq_oracle.py): codes byte-equal, the scan's
refine_all result bit-equal on shared index state, filters, recall of a device-trained index, re-rank, index files."""
import os

import numpy as np
import pytest

import rabitq_oracle as rq
from vearch_b200 import index as gidx, synth

pytestmark = pytest.mark.gpu

MNAME = {rq.METRIC_L2: "L2", rq.METRIC_IP: "InnerProduct"}


def _index(d, nlist, nb, metric, qb=4, nprobe=8, **extra):
    p = {"ncentroids": nlist, "nprobe": nprobe, "metric_type": MNAME[metric], "nb_bits": nb, "qb": qb}
    p.update(extra)
    return gidx.GammaIndex("IVFRABITQ", d, p)


def _shared_state(d, n, nlist, nb, metric, seed=1, integer=False):
    db = synth.sift_like(n, d, seed=seed)
    if integer:
        db = np.round(db).astype(np.float32)
    rng = np.random.default_rng(seed)
    cent = db[rng.choice(n, nlist, replace=False)].copy()
    idx = _index(d, nlist, nb, metric)
    idx.add_vectors(db)
    idx.set_centroids(cent)
    idx.add_pending()
    return idx, db, cent


def _assert_same(dg, ig, do, io):
    assert np.array_equal(dg, do)
    # equal scores may list their ids in either order only inside a tie group
    for r in range(dg.shape[0]):
        if not np.array_equal(ig[r], io[r]):
            for s in np.unique(dg[r]):
                m = dg[r] == s
                assert sorted(ig[r][m]) == sorted(io[r][m])


@pytest.mark.parametrize("integer", [False, True])
def test_encode_bytes_equal(integer):
    for d in (8, 100, 128):
        for nb in (1, 2, 4, 9):
            metric = rq.METRIC_IP if integer else rq.METRIC_L2
            db = synth.sift_like(3000, d, seed=d + nb)
            if integer:
                db = np.round(db).astype(np.float32)
            cent = db[:8].copy()
            assign = np.arange(3000) % 8
            idx = _index(d, 8, nb, metric)
            idx.set_centroids(cent)
            got = idx.rabitq_encode(db, assign)
            want = rq.encode(db, cent, assign, nb, metric)
            assert got.shape == (3000, rq.code_size(d, nb))
            assert np.array_equal(got, want), (d, nb, np.argwhere(got != want)[:5])
            idx.close()


@pytest.mark.parametrize("metric", [rq.METRIC_L2, rq.METRIC_IP])
@pytest.mark.parametrize("nb", [1, 4, 9])
def test_search_preassigned_matches_refine_all(metric, nb):
    d, n, nlist, nq, k, nprobe = 128, 12000, 24, 24, 20, 6
    idx, db, cent = _shared_state(d, n, nlist, nb, metric)
    xq = synth.sift_like(nq, d, seed=7)
    off, codes, ids = idx.export_lists()
    assert np.array_equal(codes, rq.encode(db[ids], cent, np.repeat(np.arange(nlist), np.diff(off)), nb, metric))
    cd, keys = idx.coarse_search(xq, nprobe)
    for qb in (1, 4, 8, 0):
        for centered in (False, True):
            params = {"qb": qb, "centered": centered}
            consts = idx.rabitq_query_consts(xq, keys, qb, centered)
            pre = rq.query_prep(np.repeat(xq, nprobe, 0), cent[keys.reshape(-1)], qb, centered, nb, metric)
            assert np.array_equal(consts[..., 4].reshape(-1), pre["base"])
            if qb:
                assert np.array_equal(consts[..., 0].reshape(-1), pre["vl"])
                assert np.array_equal(consts[..., 1].reshape(-1), pre["delta"])
                assert np.array_equal(consts[..., 6].reshape(-1).view(np.int32), pre["sq"].astype(np.int32))
            dg, ig = idx.search_preassigned(xq, k, keys, cd, params=params)
            do, io = rq.search_preassigned(off, codes, ids, cent, xq, k, keys, nb, metric, qb=qb, centered=centered)
            if qb == 0:
                np.testing.assert_allclose(dg, do, rtol=1e-5)
                assert (ig == io).mean() > 0.98
            else:
                _assert_same(dg, ig, do, io)
    idx.close()


@pytest.mark.parametrize("metric", [rq.METRIC_L2, rq.METRIC_IP])
def test_filters_tombstones_and_compaction(metric):
    d, n, nlist, nq, k, nprobe, nb = 100, 8000, 16, 16, 30, 5, 4
    idx, db, cent = _shared_state(d, n, nlist, nb, metric, seed=3)
    xq = synth.sift_like(nq, d, seed=8)
    cd, keys = idx.coarse_search(xq, nprobe)
    rng = np.random.default_rng(0)
    delb = np.packbits(rng.random(n) < 0.3, bitorder="little")
    filb = np.packbits(rng.random(n) < 0.6, bitorder="little")
    off, codes, ids = idx.export_lists()
    dg, _ = idx.search_preassigned(xq, k, keys, cd)
    lo, hi = float(np.median(dg[:, 0])), float(np.median(dg[:, -1]))
    lo, hi = min(lo, hi), max(lo, hi)
    for kw in ({"del_bitmap": delb}, {"filter_bitmap": filb}, {"del_bitmap": delb, "filter_bitmap": filb},
               {"min_score": lo, "max_score": hi}):
        dg, ig = idx.search_preassigned(xq, k, keys, cd, **kw)
        do, io = rq.search_preassigned(off, codes, ids, cent, xq, k, keys, nb, metric, **kw)
        _assert_same(dg, ig, do, io)
    # update_vector tombstones the old entry and re-encodes into the new list; compaction keeps the answer
    for vid in range(0, 400, 7):
        idx.update_vector(vid, db[(vid * 31) % n] + 0.5)
    for stage in ("updated", "compacted"):
        if stage == "compacted":
            idx.compact()
        off, codes, ids = idx.export_lists()
        assert (ids < 0).sum() == len(range(0, 400, 7))  # compaction re-packs the slabs, tombstones stay
        dg, ig = idx.search_preassigned(xq, k, keys, cd)
        do, io = rq.search_preassigned(off, codes, ids, cent, xq, k, keys, nb, metric)
        _assert_same(dg, ig, do, io)
    idx.close()


def _recall(ig, gt, r):
    return float(np.mean([gt[i] in ig[i, :r] for i in range(len(gt))]))


@pytest.mark.parametrize("metric", [rq.METRIC_L2, rq.METRIC_IP])
def test_recall_device_trained(metric):
    d, n, nq, k = 128, 40000, 200, 100
    nlist = int(min(4 * np.sqrt(n), n // 39))
    db = synth.sift_like(n, d, seed=11)
    xq = synth.sift_like(nq, d, seed=12)
    if metric == rq.METRIC_L2:
        gt = np.argmin(((xq[:, None, :].astype(np.float64) - db[None]) ** 2).sum(-1), 1)
    else:
        gt = np.argmax(xq.astype(np.float64) @ db.T.astype(np.float64), 1)
    report = {}
    for nb in (1, 2, 4, 9):
        idx = _index(d, nlist, nb, metric, nprobe=80, training_threshold=min(200 * nlist, n))
        idx.add_vectors(db)
        idx.train()
        idx.add_pending()
        _, ig = idx.search(xq, k)
        assert idx.last_scan_kernel == "rabitq_scan_kernel"
        rec = [_recall(ig, gt, r) for r in (1, 10, 100)]
        report[nb] = rec
        if nb >= 2:
            assert rec[0] >= 0.5 and rec[1] >= 0.8 and rec[2] >= 0.9, (nb, rec)
        idx.close()
    print("IVFRABITQ recall@1/10/100 by nb_bits:", report)


def test_rerank_scores_are_exact_and_qb_falls_back():
    d, n, nlist, nq, k = 128, 10000, 32, 16, 10
    db = synth.sift_like(n, d, seed=21)
    xq = synth.sift_like(nq, d, seed=22)
    idx = _index(d, nlist, 4, rq.METRIC_L2, nprobe=8, training_threshold=n)
    idx.add_vectors(db)
    idx.train()
    idx.add_pending()
    dg, ig = idx.search(xq, k, params={"recall_num": 100})
    flat = gidx.GammaIndex("FLAT", d, {"metric_type": "L2"})
    flat.add_vectors(db)
    for q in range(nq):
        fb = np.zeros((n + 7) // 8, np.uint8)
        for v in ig[q]:
            fb[v >> 3] |= 1 << (v & 7)
        df, if_ = flat.search(xq[q:q + 1], k, filter_bitmap=fb)
        assert np.array_equal(dg[q], df[0]) and sorted(ig[q]) == sorted(if_[0])
    # an out-of-range qb in a search is not an error: the model's qb serves it
    d4, i4 = idx.search(xq, k)
    for bad in (9, -1):
        db_, ib_ = idx.search(xq, k, params={"qb": bad})
        assert np.array_equal(db_, d4) and np.array_equal(ib_, i4)
    flat.close()
    idx.close()


@pytest.mark.parametrize("params, msg", [
    ({"nb_bits": 0}, "invalid nb_bits =0 should be integer in [1, 9]"),
    ({"nb_bits": 10}, "invalid nb_bits =10 should be integer in [1, 9]"),
    ({"qb": -1}, "invalid qb =-1 should be integer in [0, 8]"),
    ({"qb": 9}, "invalid qb =9 should be integer in [0, 8]"),
    ({"nprobe": 64}, "nprobe should less than ncentroids"),
])
def test_model_param_errors(params, msg):
    p = {"ncentroids": 32, "nprobe": 8}
    p.update(params)
    with pytest.raises(gidx.GammaError, match=msg.replace("[", r"\[").replace("]", r"\]")):
        gidx.GammaIndex("IVFRABITQ", 16, p)


@pytest.mark.parametrize("nb", [1, 4])
def test_index_file_round_trip(tmp_path, nb):
    d, n, nlist, nq, k = 100, 6000, 16, 16, 10
    idx, db, cent = _shared_state(d, n, nlist, nb, rq.METRIC_IP, seed=31)
    idx.update_vector(5, db[6])  # one tombstone in the file
    idx.dump(tmp_path, "f")
    raw = open(os.path.join(tmp_path, "f", "ivfrabitq.index"), "rb").read()
    lists = [idx.get_list(l) for l in range(nlist)]
    assert raw == rq.index_file_bytes(d, rq.METRIC_IP, nb, 4, 8, cent, lists, n)
    xq = synth.sift_like(nq, d, seed=32)
    d0, i0 = idx.search(xq, k)
    fresh = _index(d, nlist, nb, rq.METRIC_IP)
    fresh.add_vectors(db)
    fresh.update_vector(5, db[6])
    assert fresh.load(tmp_path, "f") == n
    d1, i1 = fresh.search(xq, k)
    assert np.array_equal(d0, d1) and np.array_equal(i0, i1)
    # a file whose nb_bits does not match the table is refused with a message
    other = _index(d, nlist, 2 if nb == 4 else 4, rq.METRIC_IP)
    other.add_vectors(db)
    with pytest.raises(gidx.GammaError, match="bad magic|nb_bits|code_size"):
        other.load(tmp_path, "f")
    for x in (idx, fresh, other):
        x.close()


def _engine(tmp_path, params, d):
    from vearch_b200 import engine, wire
    e = engine.GammaEngine(str(tmp_path), space_name="rq")
    e.create_table("rq", d, "IVFRABITQ", params, fields=(("_id", wire.DT_STRING, False),))
    return e


def test_engine_end_to_end(tmp_path):
    from vearch_b200 import engine
    d, n, nq = 32, 4000, 16
    db = synth.sift_like(n, d, seed=41)
    xq = synth.sift_like(nq, d, seed=42)
    E = engine.GammaEngine(str(tmp_path / "bad"))
    for bad, msg in (({"nb_bits": 0}, "invalid nb_bits =0"), ({"nb_bits": 10}, "invalid nb_bits =10"),
                     ({"qb": -1}, "invalid qb =-1"), ({"qb": 9}, "invalid qb =9"),
                     ({"nprobe": 64}, "nprobe should less than ncentroids")):
        p = {"ncentroids": 16, "nprobe": 8}
        p.update(bad)
        with pytest.raises(engine.GammaStatusError) as ei:
            E.create_table("t", d, "IVFRABITQ", p)
        assert msg in ei.value.msg
    E.close()
    params = {"ncentroids": 16, "nprobe": 8, "metric_type": "L2", "nb_bits": 4, "qb": 4, "training_threshold": 2000,
              "hnsw": {"nlinks": 32, "efConstruction": 100}}
    e = _engine(tmp_path, params, d)
    for i, v in enumerate(db):
        assert e.add_doc(f"doc{i}", v) == 0
    assert e.build_index() == 0
    e.wait_indexed(n)
    ip = {"nprobe": 16, "qb": 4, "recall_num": 100}
    res = e.search(xq, 10, index_params=ip)
    got = [[it["fields"]["_id"].decode() for it in r["items"]] for r in res]
    gt = np.argmin(((xq[:, None, :] - db[None]) ** 2).sum(-1), 1)
    assert np.mean([f"doc{gt[q]}" in got[q] for q in range(nq)]) >= 0.9
    for q in range(nq):  # re-ranked: exact distances
        assert res[q]["items"][0]["score"] == float(((xq[q] - db[int(got[q][0][3:])]) ** 2).sum())
    # an out-of-range qb in a search falls back to the model's qb
    assert e.search(xq, 10, index_params=dict(ip, qb=9)) == res
    assert e.memory_info()["index_mem"] > 0
    assert e.dump() == 0
    e.close()
    e2 = _engine(tmp_path, params, d)
    assert e2.load() == 0
    e2.wait_indexed(n)
    assert e2.search(xq, 10, index_params=ip) == res
    e2.close()


def test_concurrent_adds_and_searches_agree_with_final_state():
    import threading
    d, n, nlist, nq, k = 64, 20000, 32, 8, 10
    db = synth.sift_like(n, d, seed=51)
    xq = synth.sift_like(nq, d, seed=52)
    idx = _index(d, nlist, 4, rq.METRIC_L2, nprobe=nlist, training_threshold=5000)
    idx.add_vectors(db[:5000])
    idx.train()
    idx.add_pending()
    errors = []

    def adder():
        try:
            for s in range(5000, n, 1000):
                idx.add_vectors(db[s:s + 1000])
                idx.add_pending()
        except Exception as ex:  # noqa: BLE001
            errors.append(ex)

    def searcher():
        try:
            for _ in range(20):
                dg, ig = idx.search(xq, k)
                assert ((ig >= -1) & (ig < n)).all()
        except Exception as ex:  # noqa: BLE001
            errors.append(ex)

    th = [threading.Thread(target=adder)] + [threading.Thread(target=searcher) for _ in range(3)]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    dg, ig = idx.search(xq, k)
    off, codes, ids = idx.export_lists()
    cent = idx.get_centroids()
    keys = np.tile(np.arange(nlist), (nq, 1))
    do, io = rq.search_preassigned(off, codes, ids, cent, xq, k, keys, 4, rq.METRIC_L2)
    _assert_same(dg, ig, do, io)
    idx.close()


def test_large_codes_scan_or_are_refused():
    # d = 4096 at 9 bits: 4624-byte codes still fit two 16-code stages of the scan's ring
    d, n, nlist, k = 4096, 300, 8, 10
    idx, db, cent = _shared_state(d, n, nlist, 9, rq.METRIC_L2, seed=61)
    xq = synth.sift_like(4, d, seed=62)
    cd, keys = idx.coarse_search(xq, 2)
    off, codes, ids = idx.export_lists()
    dg, ig = idx.search_preassigned(xq, k, keys, cd)
    do, io = rq.search_preassigned(off, codes, ids, cent, xq, k, keys, 9, rq.METRIC_L2)
    _assert_same(dg, ig, do, io)
    idx.close()
    # d = 8192 at 9 bits does not: refused when the index is created, not at its first search
    with pytest.raises(gidx.GammaError, match="too large for the scan"):
        gidx.GammaIndex("IVFRABITQ", 8192, {"ncentroids": 4, "nprobe": 2, "nb_bits": 9})
