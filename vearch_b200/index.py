"""Host-side mirror of the reference's index interface for the hot path.

Names follow the reference: `index_factory`, `train / add / search` of the faiss-like wrappers
(internal/engine/index/index.h:  vearch::IndexIVFFlat, vearch::IndexIVFPQ, index_factory) and
the IndexModel plug-in verbs `Indexing / Add / Search` (internal/engine/index/index_model.h:229-335).
Everything below is a thin ctypes shim over include/gamma_b200_index.h; all compute happens in
vearch_b200/libgamma.so (sm_100a CUDA).  There is no CPU fallback.
"""
import ctypes as C
import json

import numpy as np

from . import _lib

METRIC_IP = 0  # DistanceComputeType::INNER_PRODUCT (gamma's default)
METRIC_L2 = 1
FLT_MAX = 3.4028234663852886e38


class GammaError(RuntimeError):
    pass


def _check(rc, what):
    if rc != 0:
        raise GammaError(f"{what} failed (rc={rc}): {_lib.last_error()}")


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _bitmap(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.uint8)


class GammaIndex:
    """One vector field's raw store + index model on one GPU."""

    def __init__(self, index_type, d, params=None, device=0):
        self.index_type = index_type.upper()
        self.d = int(d)
        self.device = device
        pj = json.dumps(params or {}).encode()
        self._h = _lib.lib().gb_index_create(self.index_type.encode(), self.d, pj, device)
        if not self._h:
            raise GammaError(f"create {index_type}: {_lib.last_error()}")

    def close(self):
        if getattr(self, "_h", None):
            _lib.lib().gb_index_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- properties -------------------------------------------------------------------
    @property
    def ntotal(self):
        return int(_lib.lib().gb_index_ntotal(self._h))

    @property
    def indexed_count(self):
        return int(_lib.lib().gb_index_indexed_count(self._h))

    @property
    def is_trained(self):
        return bool(_lib.lib().gb_index_is_trained(self._h))

    @property
    def training_threshold(self):
        return int(_lib.lib().gb_index_training_threshold(self._h))

    @property
    def nlist(self):
        return int(_lib.lib().gb_index_nlist(self._h))

    @property
    def code_size(self):
        return int(_lib.lib().gb_index_code_size(self._h))

    def mem_bytes(self, which=0):
        return int(_lib.lib().gb_index_mem_bytes(self._h, which))

    # ---- build --------------------------------------------------------------------------
    def add_vectors(self, x):
        """VectorManager::AddToStore: append raw vectors (host ndarray or torch CUDA tensor)."""
        if hasattr(x, "is_cuda") and x.is_cuda:
            assert x.dtype.is_floating_point and x.dim() == 2 and x.shape[1] == self.d and x.stride(1) == 1
            _check(_lib.lib().gb_index_add_vectors_device(self._h, x.shape[0], C.c_void_p(x.data_ptr()), x.stride(0)),
                   "add_vectors_device")
            return
        x = _f32(x)
        assert x.ndim == 2 and x.shape[1] == self.d
        _check(_lib.lib().gb_index_add_vectors(self._h, x.shape[0], _ptr(x)), "add_vectors")

    def train(self):
        """IndexModel::Indexing(): train on the first training_threshold stored vectors."""
        _check(_lib.lib().gb_index_train(self._h), "train")

    def add_pending(self, del_bitmap=None):
        """VectorManager::AddRTVecsToIndex: index everything stored but not yet indexed."""
        b = _bitmap(del_bitmap)
        _check(_lib.lib().gb_index_add_pending(self._h, _ptr(b)), "add_pending")

    def add(self, x):
        """faiss-like add (index/index.h): store + index."""
        self.add_vectors(x)
        self.add_pending()

    def update_vector(self, vid, x):
        x = _f32(x).reshape(-1)
        _check(_lib.lib().gb_index_update_vector(self._h, vid, _ptr(x)), "update_vector")

    def get_vector(self, vid):
        out = np.empty(self.d, np.float32)
        _check(_lib.lib().gb_index_get_vector(self._h, vid, _ptr(out)), "get_vector")
        return out

    def get_vectors(self, start, n):
        out = np.empty((n, self.d), np.float32)
        _check(_lib.lib().gb_index_get_vectors(self._h, start, n, _ptr(out)), "get_vectors")
        return out

    # ---- search -------------------------------------------------------------------------
    def search(self, x, k, params=None, brute_force=False, del_bitmap=None, filter_bitmap=None, min_score=-FLT_MAX,
               max_score=FLT_MAX):
        """IndexModel::Search. Returns (scores[nq,k] float32, ids[nq,k] int64)."""
        x = _f32(x)
        assert x.ndim == 2 and x.shape[1] == self.d
        nq = x.shape[0]
        dis = np.empty((nq, k), np.float32)
        ids = np.empty((nq, k), np.int64)
        pj = json.dumps(params).encode() if params else b""
        db, fb = _bitmap(del_bitmap), _bitmap(filter_bitmap)
        bits = 0
        for b in (db, fb):
            if b is not None:
                bits = max(bits, b.size * 8)
        rc = _lib.lib().gb_index_search(self._h, nq, _ptr(x), k, pj, int(brute_force), _ptr(db), _ptr(fb), bits,
                                        C.c_float(min_score), C.c_float(max_score), _ptr(dis), _ptr(ids))
        _check(rc, "search")
        return dis, ids

    def search_device(self, x, k, params=None, brute_force=False, out=None):
        """Queries and results stay in HBM (torch CUDA tensors); asynchronous on torch's current stream."""
        import torch
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        nq = x.shape[0]
        if out is None:
            out = (torch.empty((nq, k), dtype=torch.float32, device=x.device),
                   torch.empty((nq, k), dtype=torch.int64, device=x.device))
        pj = json.dumps(params).encode() if params else b""
        st = torch.cuda.current_stream(x.device).cuda_stream
        rc = _lib.lib().gb_index_search_device(self._h, nq, C.c_void_p(x.data_ptr()), x.stride(0), k, pj,
                                               int(brute_force), C.c_void_p(out[0].data_ptr()),
                                               C.c_void_p(out[1].data_ptr()), C.c_void_p(st))
        _check(rc, "search_device")
        return out

    def search_device_keys(self, x, k, params=None, brute_force=False, out_keys=None):
        """Like search_device, returning only the nq x k int64 result keys (score bits << 32 | doc id, best first):
        what a partition contributes to merge_partition_keys_device."""
        import torch
        assert x.is_cuda and x.dtype == torch.float32 and x.dim() == 2 and x.stride(1) == 1
        nq = x.shape[0]
        if out_keys is None:
            out_keys = torch.empty((nq, k), dtype=torch.int64, device=x.device)
        pj = json.dumps(params).encode() if params else b""
        st = torch.cuda.current_stream(x.device).cuda_stream
        rc = _lib.lib().gb_index_search_device_keys(self._h, nq, C.c_void_p(x.data_ptr()), x.stride(0), k, pj, int(brute_force),
                                                    C.c_void_p(out_keys.data_ptr()), None, None, C.c_void_p(st))
        _check(rc, "search_device_keys")
        return out_keys

    def stage_times(self):
        """{stage: ms} summed over the searches since the last call (set_scan_timing(True) first)."""
        p, n = C.c_void_p(), C.c_int()
        _check(_lib.lib().gb_index_stage_times(self._h, C.byref(p), C.byref(n)), "stage_times")
        js = C.string_at(p.value, n.value).decode()
        C.CDLL(None).free(C.c_void_p(p.value))
        return json.loads(js)

    def set_scan_timing(self, on):
        _lib.lib().gb_index_set_scan_timing(self._h, int(on))

    @property
    def last_scan_ms(self):
        return float(_lib.lib().gb_index_last_scan_ms(self._h))

    @property
    def last_scan_kernel(self):
        return _lib.lib().gb_index_last_scan_kernel(self._h).decode()

    @property
    def last_scan_info(self):
        return json.loads(_lib.lib().gb_index_last_scan_info(self._h).decode() or "{}")

    # ---- index-state exchange (parity tests) -------------------------------------------
    def set_centroids(self, c):
        c = _f32(c)
        _check(_lib.lib().gb_index_set_centroids(self._h, _ptr(c), c.shape[0]), "set_centroids")

    def get_centroids(self):
        out = np.empty((self.nlist, self.d), np.float32)
        _check(_lib.lib().gb_index_get_centroids(self._h, _ptr(out)), "get_centroids")
        return out

    @property
    def pq_m(self):
        return int(_lib.lib().gb_index_pq_m(self._h))

    def set_pq_centroids(self, pq):
        pq = _f32(pq)
        assert pq.shape == (self.pq_m, 256, self.d // self.pq_m)
        _check(_lib.lib().gb_index_set_pq_centroids(self._h, _ptr(pq)), "set_pq_centroids")

    def get_pq_centroids(self):
        m = self.pq_m
        out = np.empty((m, 256, self.d // m), np.float32)
        _check(_lib.lib().gb_index_get_pq_centroids(self._h, _ptr(out)), "get_pq_centroids")
        return out

    def get_precomputed_table(self):
        out = np.empty((self.nlist, self.pq_m, 256), np.float32)
        _check(_lib.lib().gb_index_get_precomputed_table(self._h, _ptr(out)), "get_precomputed_table")
        return out

    @property
    def has_opq(self):
        return bool(_lib.lib().gb_index_has_opq(self._h))

    def set_opq(self, A):
        A = _f32(A)
        assert A.shape == (self.d, self.d)
        _check(_lib.lib().gb_index_set_opq(self._h, _ptr(A)), "set_opq")

    def get_opq(self):
        A = np.empty((self.d, self.d), np.float32)
        _check(_lib.lib().gb_index_get_opq(self._h, _ptr(A)), "get_opq")
        return A

    def apply_opq(self, x):
        x = _f32(x)
        out = np.empty_like(x)
        _check(_lib.lib().gb_index_apply_opq(self._h, x.shape[0], _ptr(x), _ptr(out)), "apply_opq")
        return out

    def list_len(self, l):
        return int(_lib.lib().gb_index_list_len(self._h, l))

    def get_list(self, l):
        n = self.list_len(l)
        codes = np.empty((n, self.code_size), np.uint8)
        ids = np.empty(n, np.int64)
        if n:
            _check(_lib.lib().gb_index_get_list(self._h, l, _ptr(codes), _ptr(ids)), "get_list")
        return codes, ids

    def export_lists(self):
        """CSR view (list_off, codes, ids) of every inverted list, for the oracle."""
        lens = np.array([self.list_len(l) for l in range(self.nlist)], np.int64)
        off = np.zeros(self.nlist + 1, np.int64)
        np.cumsum(lens, out=off[1:])
        codes = np.empty((int(off[-1]), self.code_size), np.uint8)
        ids = np.empty(int(off[-1]), np.int64)
        for l in range(self.nlist):
            if lens[l]:
                c, i = self.get_list(l)
                codes[off[l]:off[l + 1]] = c
                ids[off[l]:off[l + 1]] = i
        return off, codes, ids

    @property
    def mirror_builds(self):
        return int(_lib.lib().gb_index_mirror_builds(self._h))

    def compact(self):
        _check(_lib.lib().gb_index_compact(self._h), "compact")

    def dump(self, directory, abs_name):
        """IndexModel::Dump in gamma's own format: <directory>/<abs_name>/{ivfflat,ivfpq}.index."""
        _check(_lib.lib().gb_index_dump(self._h, str(directory).encode(), abs_name.encode()), "dump")

    def load(self, directory, abs_name):
        """IndexModel::Load; returns load_num (0: no file).  The vectors must already be in the store."""
        n = np.zeros(1, np.int64)
        _check(_lib.lib().gb_index_load(self._h, str(directory).encode(), abs_name.encode(), _ptr(n)), "load")
        return int(n[0])

    def tombstone(self, l, pos):
        _check(_lib.lib().gb_index_tombstone(self._h, l, pos), "tombstone")

    def coarse_search(self, x, nprobe):
        x = _f32(x)
        nq = x.shape[0]
        dis = np.empty((nq, nprobe), np.float32)
        ids = np.empty((nq, nprobe), np.int64)
        _check(_lib.lib().gb_index_coarse_search(self._h, nq, _ptr(x), nprobe, _ptr(dis), _ptr(ids)), "coarse_search")
        return dis, ids

    def search_preassigned(self, x, k, keys, coarse_dis, params=None, del_bitmap=None, filter_bitmap=None,
                           min_score=-FLT_MAX, max_score=FLT_MAX):
        x = _f32(x)
        keys = np.ascontiguousarray(keys, np.int64)
        coarse_dis = _f32(coarse_dis)
        nq, nprobe = keys.shape
        dis = np.empty((nq, k), np.float32)
        ids = np.empty((nq, k), np.int64)
        pj = json.dumps(params).encode() if params else b""
        db, fb = _bitmap(del_bitmap), _bitmap(filter_bitmap)
        bits = 0
        for b in (db, fb):
            if b is not None:
                bits = max(bits, b.size * 8)
        rc = _lib.lib().gb_index_search_preassigned(self._h, nq, _ptr(x), k, _ptr(keys), _ptr(coarse_dis), nprobe, pj,
                                                    _ptr(db), _ptr(fb), bits, C.c_float(min_score),
                                                    C.c_float(max_score), _ptr(dis), _ptr(ids))
        _check(rc, "search_preassigned")
        return dis, ids

    def pq_encode(self, x, assign):
        x = _f32(x)
        assign = np.ascontiguousarray(assign, np.int64)
        codes = np.empty((x.shape[0], self.pq_m), np.uint8)
        _check(_lib.lib().gb_index_pq_encode(self._h, x.shape[0], _ptr(x), _ptr(assign), _ptr(codes)), "pq_encode")
        return codes

    def rabitq_encode(self, x, assign):
        """IVFRABITQ: RaBitQ codes (n x code_size uint8) of x against centroids[assign], on the device."""
        x = _f32(x)
        assign = np.ascontiguousarray(assign, np.int64)
        codes = np.empty((x.shape[0], self.code_size), np.uint8)
        _check(_lib.lib().gb_index_rabitq_encode(self._h, x.shape[0], _ptr(x), _ptr(assign), _ptr(codes)), "rabitq_encode")
        return codes

    def rabitq_query_consts(self, x, keys, qb, centered=False):
        """IVFRABITQ: the scan's per-(query, probe) constants, [nq, nprobe, 8] float32 (DESIGN.md section 5b)."""
        x = _f32(x)
        keys = np.ascontiguousarray(keys, np.int64)
        nq, nprobe = keys.shape
        out = np.empty((nq, nprobe, 8), np.float32)
        _check(_lib.lib().gb_index_rabitq_query_consts(self._h, nq, _ptr(x), _ptr(keys), nprobe, qb, int(centered), _ptr(out)),
               "rabitq_query_consts")
        return out


def index_factory(d, description, metric=METRIC_L2, device=0, **extra):
    """index/index.h index_factory: "IVF1024,Flat" | "IVF4096,PQ16x8" | "Flat"."""
    parts = [p.strip() for p in description.split(",")]
    params = dict(extra)
    params["metric_type"] = "L2" if metric == METRIC_L2 else "InnerProduct"
    if len(parts) == 1 and parts[0].lower() == "flat":
        return GammaIndex("FLAT", d, params, device)
    if len(parts) == 2 and parts[0].upper().startswith("IVF"):
        params["ncentroids"] = int(parts[0][3:])
        params.setdefault("nprobe", min(params.get("nprobe", 80), params["ncentroids"]))
        if parts[1].lower() == "flat":
            return GammaIndex("IVFFLAT", d, params, device)
        if parts[1].upper().startswith("PQ"):
            m, _, nbits = parts[1][2:].partition("x")
            params["nsubvector"] = int(m)
            params["nbits_per_idx"] = int(nbits or 8)
            return GammaIndex("IVFPQ", d, params, device)
    raise GammaError(f"unsupported index description {description!r}")


def kmeans(x, k, niter=25, seed=1234, spherical=False, max_points_per_centroid=256, device=0):
    x = _f32(x)
    n, d = x.shape
    cent = np.empty((k, d), np.float32)
    obj = np.zeros(niter, np.float32)
    _check(_lib.lib().gb_kmeans(device, _ptr(x), n, d, k, niter, seed, int(spherical), max_points_per_centroid,
                                _ptr(cent), _ptr(obj)), "kmeans")
    return cent, obj


def kmeans_update(x, k, assign, device=0):
    x = _f32(x)
    assign = np.ascontiguousarray(assign, np.int64)
    cent = np.empty((k, x.shape[1]), np.float32)
    _check(_lib.lib().gb_kmeans_update(device, _ptr(x), x.shape[0], x.shape[1], k, _ptr(assign), _ptr(cent)),
           "kmeans_update")
    return cent


def merge_partitions_device(dis, ids, metric):
    """dis/ids: torch CUDA tensors [nparts, nq, k] -> merged ([nq,k], [nq,k]) on the same device."""
    import torch
    nparts, nq, k = dis.shape
    od = torch.empty((nq, k), dtype=torch.float32, device=dis.device)
    oi = torch.empty((nq, k), dtype=torch.int64, device=dis.device)
    st = torch.cuda.current_stream(dis.device).cuda_stream
    _check(_lib.lib().gb_merge_partitions_device(dis.device.index or 0, C.c_void_p(dis.data_ptr()),
                                                 C.c_void_p(ids.data_ptr()), nparts, nq, k, metric,
                                                 C.c_void_p(od.data_ptr()), C.c_void_p(oi.data_ptr()), C.c_void_p(st)),
           "merge_partitions_device")
    return od, oi


def merge_partition_keys_device(keys, metric):
    """keys: torch CUDA int64 tensor [nparts, nq, k] of partition result keys -> merged ([nq,k] scores, [nq,k] ids with
    ids = partition << 32 | local id) in the router's order (internal/client/client.go:1530-1609)."""
    import torch
    nparts, nq, k = keys.shape
    od = torch.empty((nq, k), dtype=torch.float32, device=keys.device)
    oi = torch.empty((nq, k), dtype=torch.int64, device=keys.device)
    st = torch.cuda.current_stream(keys.device).cuda_stream
    _check(_lib.lib().gb_merge_partition_keys_device(keys.device.index or 0, C.c_void_p(keys.data_ptr()), nparts, nq, k, metric,
                                                     C.c_void_p(od.data_ptr()), C.c_void_p(oi.data_ptr()), C.c_void_p(st)),
           "merge_partition_keys_device")
    return od, oi


def debug_dist_matrix(x, c, metric, use_tc, device=0):
    """score matrix through the exact CUDA-core kernel (use_tc=0) or the tcgen05 3xTF32 kernel (use_tc=1)."""
    x, c = _f32(x), _f32(c)
    out = np.empty((x.shape[0], c.shape[0]), np.float32)
    fn = _lib.lib().gb_debug_dist_matrix
    fn.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    _check(fn(device, _ptr(x), x.shape[0], _ptr(c), c.shape[0], x.shape[1], metric, int(use_tc), _ptr(out)),
           "debug_dist_matrix")
    return out
