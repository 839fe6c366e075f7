"""CPU restatement of the IVFRABITQ codec and scans (DESIGN.md section 5b).

TEST INFRASTRUCTURE ONLY: imported by the RaBitQ tests and __graft_entry__.smoke(); the product
package never imports it.  Every float value is computed in numpy float32, one rounded operation
at a time, and every float reduction runs sequentially over the dimensions in index order
(acc = acc + a_j * b_j, j = 0 .. d-1, starting from 0).  The CUDA kernels (kernels_rabitq.cu)
evaluate the same expressions with unfused __fmul_rn / __fadd_rn in the same order, so codes
are byte-equal and scores bit-equal.

Code of one vector (residual r = x - c against its list's centroid c), little endian:
    nb_bits == 1:  sign plane [P] | or_c f32 | f1 f32                              -> P + 8 bytes
    nb_bits  > 1:  sign plane [P] | or_c f32 | f1 f32 | f_error f32
                   | extra planes [(nb_bits-1) * P] | f_ex f32                     -> nb_bits * P + 16 bytes
with P = ceil(d / 8).  A plane holds one bit per dimension, dimension j at bit (j & 7) of byte j >> 3.
The total code of dimension j is t_j = b_j << ex | e'_j (ex = nb_bits - 1), where b_j = (r_j > 0) is
the sign bit and e'_j (plane k = bit k) the extra code.
"""
import numpy as np

METRIC_IP = 0
METRIC_L2 = 1
FLT_MAX = np.float32(3.4028234663852886e38)
NSCALE = 64       # candidate rescale factors of the extra-bit search
EPS0 = np.float32(1.9)  # confidence factor of the 1-bit error bound (two-stage scan only)

f32 = np.float32


def code_size(d, nb_bits):
    P = (d + 7) // 8
    return P + 8 if nb_bits == 1 else nb_bits * P + 16


def _seqdot(a, b):
    """sum_j a[:, j] * b[:, j] in float32, j ascending, unfused."""
    acc = np.zeros(a.shape[0], np.float32)
    for j in range(a.shape[1]):
        acc = acc + a[:, j] * b[:, j]
    return acc


def _pack_plane(bits):
    """bits: (n, d) bool -> (n, P) uint8, dimension j at bit j & 7 of byte j >> 3."""
    return np.packbits(bits.astype(np.uint8), axis=1, bitorder="little")


def _unpack_plane(plane, d):
    return np.unpackbits(plane, axis=1, count=d, bitorder="little").astype(np.int64)


def _as_bytes(v):
    return np.ascontiguousarray(v, np.float32).view(np.uint8).reshape(-1, 4)


def encode(x, centroids, assign, nb_bits, metric):
    """Codes (n, code_size) uint8 of rows x, each against centroids[assign[i]]."""
    x = np.ascontiguousarray(x, np.float32)
    n, d = x.shape
    c = np.ascontiguousarray(centroids, np.float32)[np.asarray(assign, np.int64)]
    r = x - c
    b = r > 0
    ra = np.abs(r)
    rn = _seqdot(r, r)
    cr = _seqdot(c, r)
    sabs = np.zeros(n, np.float32)
    for j in range(d):
        sabs = sabs + ra[:, j]
    or_c = rn if metric == METRIC_L2 else cr
    half = sabs * f32(0.5)
    with np.errstate(divide="ignore", invalid="ignore"):
        f1 = np.where(sabs > 0, rn / np.where(half > 0, half, f32(1)), f32(0)).astype(np.float32)
    P = (d + 7) // 8
    out = np.zeros((n, code_size(d, nb_bits)), np.uint8)
    out[:, :P] = _pack_plane(b)
    out[:, P:P + 4] = _as_bytes(or_c)
    out[:, P + 4:P + 8] = _as_bytes(f1)
    if nb_bits == 1:
        return out
    # 1-bit error factor: |r| sqrt((1 - <o,xb>^2) / <o,xb>^2) / sqrt(d - 1), <o,xb> = sum|r_j| / (|r| sqrt d)
    nr = np.sqrt(rn)
    with np.errstate(divide="ignore", invalid="ignore"):
        dp = sabs / (nr * np.sqrt(f32(d)))
        t = dp * dp
        u = np.maximum((f32(1) - t) / t, f32(0))
        fe = (nr * np.sqrt(u)) / np.sqrt(f32(max(d - 1, 1)))
    fe = np.where((dp > 0) & (d > 1), fe, f32(0)).astype(np.float32)
    out[:, P + 8:P + 12] = _as_bytes(fe)
    ex = nb_bits - 1
    emax = (1 << ex) - 1
    e = extra_codes(ra, ex)
    w = (2 * e + 1).astype(np.float32)
    ipb = _seqdot(ra, w)
    with np.errstate(divide="ignore", invalid="ignore"):
        fx = np.where(ipb > 0, rn / np.where(ipb > 0, ipb * f32(0.5), f32(1)), f32(0)).astype(np.float32)
    ep = np.where(b, e, emax - e)
    o = P + 12
    for k in range(ex):
        out[:, o + k * P:o + (k + 1) * P] = _pack_plane(((ep >> k) & 1).astype(bool))
    out[:, o + ex * P:o + ex * P + 4] = _as_bytes(fx)
    return out


def extra_codes(ra, ex):
    """Magnitude codes e_j in [0, 2^ex - 1] of |r| (n, d): the rescale s_i = (2^ex * (i+1)/64) / max_j|r_j|,
    i = 0..63, whose codes e_j = min(floor(|r_j| * s_i), 2^ex - 1) maximise
    sum_j |r_j| (2 e_j + 1) / sqrt(sum_j (2 e_j + 1)^2)   (first i wins ties)."""
    n, d = ra.shape
    emax = (1 << ex) - 1
    m = np.zeros(n, np.float32)
    for j in range(d):
        m = np.maximum(m, ra[:, j])
    best = np.full(n, -np.inf, np.float32)
    best_e = np.zeros((n, d), np.int64)
    msafe = np.where(m > 0, m, f32(1))
    for i in range(NSCALE):
        kf = f32(i + 1) / f32(NSCALE)
        s = (f32(1 << ex) * kf) / msafe
        e = np.minimum(np.floor(ra * s[:, None]).astype(np.int64), emax)
        w = (2 * e + 1)
        ip = _seqdot(ra, w.astype(np.float32))
        ny = (w * w).sum(axis=1)
        cos = ip / np.sqrt(ny.astype(np.float32))
        better = cos > best
        best = np.where(better, cos, best)
        best_e[better] = e[better]
    best_e[m == 0] = 0
    return best_e


def decode_fields(codes, d, nb_bits):
    """-> dict of t (n, d) int64 total codes, b (n, d) sign bits, or_c, f1, f_error, f_ex."""
    codes = np.ascontiguousarray(codes, np.uint8)
    P = (d + 7) // 8
    b = _unpack_plane(codes[:, :P], d)
    fl = lambda o: np.ascontiguousarray(codes[:, o:o + 4]).view(np.float32).reshape(-1)
    res = {"b": b, "or_c": fl(P), "f1": fl(P + 4)}
    if nb_bits == 1:
        res["t"] = b
        return res
    ex = nb_bits - 1
    o = P + 12
    ep = np.zeros_like(b)
    for k in range(ex):
        ep |= _unpack_plane(codes[:, o + k * P:o + (k + 1) * P], d) << k
    res["t"] = (b << ex) | ep
    res["f_error"] = fl(P + 8)
    res["f_ex"] = fl(o + ex * P)
    return res


def query_prep(q, c, qb, centered, nb_bits, metric):
    """Per-pair constants of query rows q (n, d) against centroid rows c (n, d).
    Returns dict: qr (residual), qq (n, d) int64 quantised query, vl, delta, sq, p0, p1, base, g_error."""
    q = np.ascontiguousarray(q, np.float32)
    c = np.ascontiguousarray(c, np.float32)
    n, d = q.shape
    qr = q - c
    qn = _seqdot(qr, qr)
    qc = _seqdot(q, c)
    base = qn if metric == METRIC_L2 else qc
    cB = f32((1 << nb_bits) - 1) * f32(0.5)
    res = {"qr": qr, "base": base, "g_error": EPS0 * np.sqrt(qn), "cB": cB}
    if qb == 0:
        return res
    levels = f32((1 << qb) - 1)
    if centered:
        a = np.abs(qr).max(axis=1)
        vl = -a
        delta = (a * f32(2)) / levels
    else:
        vl = qr.min(axis=1)
        delta = (qr.max(axis=1) - vl) / levels
    with np.errstate(divide="ignore"):
        inv = np.where(delta > 0, f32(1) / np.where(delta > 0, delta, f32(1)), f32(0)).astype(np.float32)
    qq = np.floor((qr - vl[:, None]) * inv[:, None] + f32(0.5)).astype(np.int64)
    qq = np.clip(qq, 0, (1 << qb) - 1)
    sq = qq.sum(axis=1)
    res.update(qq=qq, vl=vl.astype(np.float32), delta=delta.astype(np.float32), sq=sq,
               p0=cB * sq.astype(np.float32), p1=np.full(n, cB * f32(d), np.float32))
    return res


def estimate(fields, pre, i, qb, nb_bits, metric, one_bit=False):
    """Scores of every code in `fields` against pair i of `pre` (one_bit: the sign-bit-only estimate)."""
    t = fields["b"] if one_bit else fields["t"]
    f = fields["f1"] if (one_bit or nb_bits == 1) else fields["f_ex"]
    if qb == 0:
        cB = f32(0.5) if one_bit else pre["cB"]
        qr = pre["qr"][i]
        g = np.zeros(t.shape[0], np.float32)
        for j in range(t.shape[1]):
            g = g + qr[j] * (t[:, j].astype(np.float32) - cB)
    else:
        sqt = t @ pre["qq"][i]
        st = t.sum(axis=1)
        if one_bit:
            p0 = f32(0.5) * f32(pre["sq"][i])
            p1 = f32(0.5) * f32(t.shape[1])
        else:
            p0, p1 = pre["p0"][i], pre["p1"][i]
        e1 = sqt.astype(np.float32) - p0
        e2 = st.astype(np.float32) - p1
        g = pre["delta"][i] * e1 + pre["vl"][i] * e2
    ip = f * g
    s = pre["base"][i] + fields["or_c"]
    return (s - f32(2) * ip) if metric == METRIC_L2 else (s + ip)


def score2ord(s, metric):
    b = np.ascontiguousarray(s, np.float32).view(np.uint32)
    o = np.where(b & np.uint32(0x80000000), ~b, b | np.uint32(0x80000000)).astype(np.uint32)
    return o if metric == METRIC_L2 else (~o).astype(np.uint32)


def _bit(bm, vid):
    return (bm[vid >> 3] >> (vid & 7)) & 1


def _valid(ids, del_bitmap, filter_bitmap):
    ok = ids >= 0
    v = np.where(ok, ids, 0)
    if filter_bitmap is not None:
        ok &= _bit(np.asarray(filter_bitmap, np.uint8), v).astype(bool)
    if del_bitmap is not None:
        ok &= ~_bit(np.asarray(del_bitmap, np.uint8), v).astype(bool)
    return ok


def _finish(keys, k, metric):
    """Sorted best keys -> (scores, ids) in the engine's output order (DESIGN.md section 4)."""
    dis = np.full(k, FLT_MAX if metric == METRIC_L2 else -FLT_MAX, np.float32)
    ids = np.full(k, -1, np.int64)
    keys = np.sort(np.asarray(keys, np.uint64))[:k]
    o = (keys >> np.uint64(32)).astype(np.uint32)
    if metric == METRIC_L2:
        b = np.where(o & np.uint32(0x80000000), o & np.uint32(0x7FFFFFFF), ~o).astype(np.uint32)
    else:
        x = (~o).astype(np.uint32)
        b = np.where(x & np.uint32(0x80000000), x & np.uint32(0x7FFFFFFF), ~x).astype(np.uint32)
    sc = b.view(np.float32)
    vid = (keys & np.uint64(0xFFFFFFFF)).astype(np.int64)
    if metric == METRIC_IP:  # equal scores: larger id first (heap_reorder of a CMin heap)
        order = np.lexsort((-vid, o))
        sc, vid = sc[order], vid[order]
    dis[:len(keys)] = sc
    ids[:len(keys)] = vid
    return dis, ids


def search_preassigned(list_off, list_codes, list_ids, centroids, xq, k, keys, nb_bits, metric, qb=4,
                       centered=False, mode="refine_all", del_bitmap=None, filter_bitmap=None,
                       min_score=-FLT_MAX, max_score=FLT_MAX):
    """IVFRABITQ scan of the lists keys[q] for every query.  mode 'refine_all': top-k by the full
    nb_bits estimate over every valid entry (what the GPU returns).  mode 'two_stage': the reference's
    scan, which computes the full estimate only where the 1-bit estimate, widened by f_error * g_error,
    can still beat the current k-th best (scan-order dependent)."""
    xq = np.ascontiguousarray(xq, np.float32)
    nq, d = xq.shape
    keys = np.asarray(keys, np.int64)
    list_off = np.asarray(list_off, np.int64)
    list_ids = np.asarray(list_ids, np.int64)
    centroids = np.ascontiguousarray(centroids, np.float32)
    out_d = np.empty((nq, k), np.float32)
    out_i = np.empty((nq, k), np.int64)
    cache = {}
    for q in range(nq):
        ls = [int(l) for l in keys[q] if 0 <= l < len(list_off) - 1]
        pre = query_prep(np.repeat(xq[q:q + 1], len(ls), 0), centroids[ls] if ls else np.zeros((0, d), np.float32),
                         qb, centered, nb_bits, metric)
        cand = []
        heap = []  # two-stage: sorted keys of the current best k
        for i, l in enumerate(ls):
            a, b = list_off[l], list_off[l + 1]
            if a == b:
                continue
            if l not in cache:
                cache[l] = decode_fields(list_codes[a:b], d, nb_bits)
            fields = cache[l]
            ids = list_ids[a:b]
            ok = _valid(ids, del_bitmap, filter_bitmap)
            s = estimate(fields, pre, i, qb, nb_bits, metric)
            if mode == "refine_all":
                ok &= (s >= min_score) & (s <= max_score)
                kk = (score2ord(s, metric).astype(np.uint64) << np.uint64(32)) | (ids.astype(np.uint64) & np.uint64(0xFFFFFFFF))
                cand.append(kk[ok])
                continue
            s1 = estimate(fields, pre, i, qb, nb_bits, metric, one_bit=True) if nb_bits > 1 else s
            err = fields["f_error"] * pre["g_error"][i] if nb_bits > 1 else np.zeros_like(s)
            bound = (s1 - f32(2) * err) if metric == METRIC_L2 else (s1 + err)
            kk = (score2ord(s, metric).astype(np.uint64) << np.uint64(32)) | (ids.astype(np.uint64) & np.uint64(0xFFFFFFFF))
            for e in np.nonzero(ok)[0]:
                if len(heap) >= k and nb_bits > 1:
                    worst = heap[-1] >> np.uint64(32)
                    if score2ord(np.float32([bound[e]]), metric)[0] > worst:
                        continue
                if not (min_score <= s[e] <= max_score):
                    continue
                if len(heap) < k or kk[e] < heap[-1]:
                    heap.append(kk[e])
                    heap.sort()
                    del heap[k:]
        allk = np.concatenate(cand) if mode == "refine_all" and cand else np.asarray(heap, np.uint64)
        out_d[q], out_i[q] = _finish(allk, k, metric)
    return out_d, out_i


# ---- index file (DESIGN.md section 5b): the reference's Iwrq / Iwrr framing -------------------------
def ivf_header_bytes(d, ntotal, metric, nlist, nprobe, centroids):
    import struct
    mt = 1 if metric == METRIC_L2 else 0
    hdr = lambda nt: struct.pack("<iqqqBi", d, nt, 1 << 20, 1 << 20, 1, mt)
    out = hdr(ntotal) + struct.pack("<QQ", nlist, nprobe)
    out += (b"IxF2" if metric == METRIC_L2 else b"IxFI") + hdr(nlist)
    c = np.ascontiguousarray(centroids, np.float32)
    out += struct.pack("<Q", c.size) + c.tobytes()
    out += struct.pack("<BQ", 0, 0)
    return out


def index_file_bytes(d, metric, nb_bits, qb, nprobe, centroids, lists, indexed_count):
    """<dir>/<name>/ivfrabitq.index as the engine writes it: lists = [(codes (n, code_size) uint8, ids (n,) int64)]."""
    import struct
    nlist = len(lists)
    cs = code_size(d, nb_bits)
    out = (b"Iwrq" if nb_bits == 1 else b"Iwrr") + ivf_header_bytes(d, indexed_count, metric, nlist, nprobe, centroids)
    out += struct.pack("<QQi", d, cs, 1 if metric == METRIC_L2 else 0)
    if nb_bits > 1:
        out += struct.pack("<Q", nb_bits)
    out += struct.pack("<QBB", cs, 1, qb)
    out += b"ilar" + struct.pack("<QQ", nlist, cs) + b"full" + struct.pack("<Q", nlist)
    out += b"".join(struct.pack("<Q", len(ids)) for _, ids in lists)
    for codes, ids in lists:
        if len(ids):
            out += np.ascontiguousarray(codes, np.uint8).tobytes() + np.ascontiguousarray(ids, "<i8").tobytes()
    return out + struct.pack("<q", indexed_count)  # int64_t indexed_count (gamma_index_ivfrabitq.cc:870-877)
