"""ctypes loader for vearch_b200/libgamma.so.  Fails loudly when the CUDA library is missing:
there is no CPU fallback in this package."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libgamma.so")

_lib = None


class GammaLibraryMissing(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise GammaLibraryMissing(
                f"{SO_PATH} not built; run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback)")
        _lib = C.CDLL(SO_PATH, mode=C.RTLD_LOCAL)
        _declare(_lib)
    return _lib


def _declare(l):
    vp, i32, i64, f32 = C.c_void_p, C.c_int, C.c_int64, C.c_float
    cstr = C.c_char_p
    l.gb_last_error.restype = cstr
    l.gb_device_count.restype = i32
    l.gb_launch_count.restype = C.c_longlong
    l.gb_index_create.restype = vp
    l.gb_index_create.argtypes = [cstr, i32, cstr, i32]
    l.gb_index_destroy.restype = None
    l.gb_index_destroy.argtypes = [vp]
    l.gb_index_add_vectors.argtypes = [vp, i64, vp]
    l.gb_index_add_vectors_device.argtypes = [vp, i64, vp, i64]
    l.gb_index_update_vector.argtypes = [vp, i64, vp]
    l.gb_index_get_vector.argtypes = [vp, i64, vp]
    l.gb_index_get_vectors.argtypes = [vp, i64, i64, vp]
    l.gb_index_train.argtypes = [vp]
    l.gb_index_add_pending.argtypes = [vp, vp]
    for n in ("gb_index_ntotal", "gb_index_indexed_count"):
        getattr(l, n).restype = i64
        getattr(l, n).argtypes = [vp]
    l.gb_index_is_trained.argtypes = [vp]
    l.gb_index_training_threshold.argtypes = [vp]
    l.gb_index_mem_bytes.restype = i64
    l.gb_index_mem_bytes.argtypes = [vp, i32]
    l.gb_index_search.argtypes = [vp, i32, vp, i32, cstr, i32, vp, vp, i64, f32, f32, vp, vp]
    l.gb_index_search_device.argtypes = [vp, i32, vp, i64, i32, cstr, i32, vp, vp, vp]
    l.gb_index_search_device_keys.argtypes = [vp, i32, vp, i64, i32, cstr, i32, vp, vp, vp, vp]
    l.gb_index_stage_times.argtypes = [vp, C.POINTER(C.c_void_p), C.POINTER(C.c_int)]
    l.gb_merge_partition_keys_device.argtypes = [i32, vp, i32, i32, i32, i32, vp, vp, vp]
    l.gb_index_set_scan_timing.restype = None
    l.gb_index_set_scan_timing.argtypes = [vp, i32]
    l.gb_index_last_scan_ms.restype = f32
    l.gb_index_last_scan_ms.argtypes = [vp]
    l.gb_index_last_scan_kernel.restype = cstr
    l.gb_index_last_scan_kernel.argtypes = [vp]
    l.gb_index_last_scan_info.restype = cstr
    l.gb_index_last_scan_info.argtypes = [vp]
    l.gb_index_nlist.argtypes = [vp]
    l.gb_index_set_centroids.argtypes = [vp, vp, i32]
    l.gb_index_get_centroids.argtypes = [vp, vp]
    l.gb_index_pq_m.argtypes = [vp]
    l.gb_index_set_pq_centroids.argtypes = [vp, vp]
    l.gb_index_get_pq_centroids.argtypes = [vp, vp]
    l.gb_index_get_precomputed_table.argtypes = [vp, vp]
    l.gb_index_has_opq.argtypes = [vp]
    l.gb_index_set_opq.argtypes = [vp, vp]
    l.gb_index_get_opq.argtypes = [vp, vp]
    l.gb_index_apply_opq.argtypes = [vp, i64, vp, vp]
    l.gb_index_list_len.argtypes = [vp, i32]
    l.gb_index_code_size.argtypes = [vp]
    l.gb_index_get_list.argtypes = [vp, i32, vp, vp]
    l.gb_index_tombstone.argtypes = [vp, i32, i32]
    l.gb_index_dump.argtypes = [vp, cstr, cstr]
    l.gb_index_compact.argtypes = [vp]
    l.gb_index_mirror_builds.argtypes = [vp]
    l.gb_index_load.argtypes = [vp, cstr, cstr, vp]
    l.gb_index_coarse_search.argtypes = [vp, i32, vp, i32, vp, vp]
    l.gb_index_search_preassigned.argtypes = [vp, i32, vp, i32, vp, vp, i32, cstr, vp, vp, i64, f32, f32, vp, vp]
    l.gb_index_pq_encode.argtypes = [vp, i64, vp, vp, vp]
    l.gb_index_rabitq_encode.argtypes = [vp, i64, vp, vp, vp]
    l.gb_index_rabitq_query_consts.argtypes = [vp, i32, vp, vp, i32, i32, i32, vp]
    l.gb_kmeans.argtypes = [i32, vp, i64, i32, i32, i32, i64, i32, i32, vp, vp]
    l.gb_kmeans_update.argtypes = [i32, vp, i64, i32, i32, vp, vp]
    l.gb_merge_partitions_device.argtypes = [i32, vp, vp, i32, i32, i32, i32, vp, vp, vp]


def last_error():
    return lib().gb_last_error().decode("utf-8", "replace")
