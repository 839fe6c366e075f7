"""IVFRABITQ codec and scans on the CPU restatement (tests/rabitq_oracle.py): layout, estimator accuracy,
the reference's two-stage scan against refine_all, and the index-file framing."""
import numpy as np
import pytest

import rabitq_oracle as rq
from vearch_b200 import synth


def _pairs(n, d, seed):
    rng = np.random.default_rng(seed)
    c = rng.normal(size=(1, d)).astype(np.float32)
    x = (c + rng.normal(size=(n, d))).astype(np.float32)
    q = (c + rng.normal(size=(n, d))).astype(np.float32)
    return x, q, c


@pytest.mark.parametrize("d", [1, 7, 8, 100, 128, 768])
def test_code_size_and_layout(d):
    rng = np.random.default_rng(d)
    x = rng.normal(size=(16, d)).astype(np.float32)
    c = np.zeros((1, d), np.float32)
    P = (d + 7) // 8
    for nb in range(1, 10):
        cs = rq.code_size(d, nb)
        assert cs == (P + 8 if nb == 1 else nb * P + 16)
        codes = rq.encode(x, c, np.zeros(16, np.int64), nb, rq.METRIC_L2)
        assert codes.shape == (16, cs)
        f = rq.decode_fields(codes, d, nb)
        # the sign plane is the top bit of the total code; padding bits of the last byte are zero
        assert np.array_equal(f["b"], (x > 0).astype(np.int64))
        assert np.array_equal(f["t"] >> (nb - 1), f["b"])
        if d % 8:
            assert not (codes[:, P - 1] >> (d % 8)).any()
        np.testing.assert_array_equal(f["or_c"], rq._seqdot(x, x))


def _estimates(nb, qb, metric, n=2000, d=128, centered=False):
    x, q, c = _pairs(n, d, seed=nb * 10 + qb)
    codes = rq.encode(x, c, np.zeros(n, np.int64), nb, metric)
    f = rq.decode_fields(codes, d, nb)
    pre = rq.query_prep(q[:1], c, qb, centered, nb, metric)
    est = rq.estimate(f, pre, 0, qb, nb, metric)
    xd, qd = x.astype(np.float64), q[0].astype(np.float64)
    true = ((xd - qd) ** 2).sum(1) if metric == rq.METRIC_L2 else xd @ qd
    return est.astype(np.float64), true


@pytest.mark.parametrize("metric", [rq.METRIC_L2, rq.METRIC_IP])
def test_nine_bit_estimate_is_close(metric):
    # nb_bits 9 and qb 8: the estimate of the distance is within 1 % of the exact value on every pair
    est, true = _estimates(9, 8, metric)
    scale = np.abs(true).mean()
    assert np.abs(est - true).max() <= 0.01 * scale


def test_one_bit_estimate_is_unbiased():
    # RaBitQ's 1-bit estimate of <q - c, x - c> is unbiased: the mean error over random pairs is near zero
    est, true = _estimates(1, 8, rq.METRIC_IP)
    err = est - true
    assert abs(err.mean()) < 0.05 * err.std() + 1e-3 * np.abs(true).mean()
    assert np.abs(err).mean() < 0.25 * np.abs(true).mean()


@pytest.mark.parametrize("centered", [False, True])
def test_more_bits_are_more_accurate(centered):
    errs = []
    for nb in (1, 2, 4, 9):
        est, true = _estimates(nb, 8, rq.METRIC_L2, centered=centered)
        errs.append(np.abs(est - true).mean())
    assert errs == sorted(errs, reverse=True), errs


@pytest.mark.parametrize("metric", [rq.METRIC_L2, rq.METRIC_IP])
def test_two_stage_agrees_with_refine_all(metric):
    d, n, nlist, nq, k, nprobe = 64, 6000, 16, 24, 10, 6
    db = synth.sift_like(n, d, seed=5)
    xq = synth.sift_like(nq, d, seed=6)
    rng = np.random.default_rng(0)
    cent = db[rng.choice(n, nlist, replace=False)]
    assign = np.argmin(((db[:, None, :] - cent[None]) ** 2).sum(-1), 1)
    order = np.argsort(assign, kind="stable")
    off = np.zeros(nlist + 1, np.int64)
    np.cumsum(np.bincount(assign, minlength=nlist), out=off[1:])
    codes = rq.encode(db[order], cent, assign[order], 4, metric)
    keys = np.argsort(((xq[:, None, :] - cent[None]) ** 2).sum(-1), 1)[:, :nprobe]
    d_all, i_all = rq.search_preassigned(off, codes, order, cent, xq, k, keys, 4, metric, qb=4, mode="refine_all")
    d_two, i_two = rq.search_preassigned(off, codes, order, cent, xq, k, keys, 4, metric, qb=4, mode="two_stage")
    agree = np.mean([len(set(a) & set(b)) / k for a, b in zip(i_all, i_two)])
    assert agree >= 0.99, agree


def test_index_file_framing():
    # an independent restatement of the Iwrq / Iwrr layout, field by field, against the oracle's writer
    d, nlist = 12, 3
    rng = np.random.default_rng(1)
    cent = rng.normal(size=(nlist, d)).astype(np.float32)
    for nb in (1, 5):
        cs = rq.code_size(d, nb)
        lists = [(rng.integers(0, 256, size=(n, cs), dtype=np.uint8), np.arange(n, dtype=np.int64) + 10 * l)
                 for l, n in enumerate((2, 0, 3))]
        got = rq.index_file_bytes(d, rq.METRIC_IP, nb, 4, 2, cent, lists, 5)
        u8, i32, i64 = (lambda v: np.uint8(v).tobytes()), (lambda v: np.int32(v).tobytes()), (lambda v: np.int64(v).tobytes())
        hdr = lambda nt: i32(d) + i64(nt) + i64(1 << 20) + i64(1 << 20) + u8(1) + i32(0)
        want = (b"Iwrr" if nb > 1 else b"Iwrq") + hdr(5) + i64(nlist) + i64(2) + b"IxFI" + hdr(nlist)
        want += i64(cent.size) + cent.tobytes() + u8(0) + i64(0)
        want += i64(d) + i64(cs) + i32(0) + (i64(nb) if nb > 1 else b"") + i64(cs) + u8(1) + u8(4)
        want += b"ilar" + i64(nlist) + i64(cs) + b"full" + i64(nlist) + i64(2) + i64(0) + i64(3)
        for c, ids in lists:
            want += c.tobytes() + ids.tobytes()
        want += i64(5)  # the reference writes int64_t indexed_count here (IvFl writes an int)
        assert got == want
