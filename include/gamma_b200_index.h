/*
 * gamma_b200_index.h -- C-ABI of the index-model seam of the gamma hot path on B200.
 *
 * This is the secondary drop-in seam of SURVEY.md 8(b): the shape of the reference's IndexModel
 * plug-in interface (internal/engine/index/index_model.h:229-335) and of its faiss-like wrappers
 * vearch::IndexIVFFlat / IndexIVFPQ / index_factory (internal/engine/index/index.h), flattened to
 * extern "C" with plain pointers and sizes.  The primary seam (the 23 gamma symbols the Go
 * partition server binds through cgo) is include/gamma_api.h and is implemented on top of this
 * one.  Every entry point runs CUDA kernels on the chosen device; there is no CPU path, and
 * creation fails if no CUDA device is present.
 *
 * Conventions: int-returning calls give 0 on success, -1 on error (gb_last_error() has the
 * message, thread-local), -2 when the request was killed.  Metric ids: 0 = InnerProduct,
 * 1 = L2 (squared).  Results are nq x k row-major, best first; unfilled slots have id -1 and
 * score +FLT_MAX (L2) / -FLT_MAX (IP), exactly what faiss heap_reorder leaves behind.
 */
#ifndef GAMMA_B200_INDEX_H_
#define GAMMA_B200_INDEX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gb_index gb_index;

const char *gb_last_error(void);
int gb_device_count(void);
/* kernels launched by this library since load (bench.py's gpu_launches evidence) */
long long gb_launch_count(void);

/* reflector().GetNewIndex(type) + IndexModel::Init(model_parameters, training_threshold)
 * (index/reflector.h:68-80, vector/vector_manager.cc:171; gamma_index_ivfflat.cc:215-291,
 * gamma_index_ivfpq.cc:112-231).  index_type: "FLAT" | "IVFFLAT" | "IVFPQ".
 * model_params_json keys: ncentroids, nprobe, metric_type ("L2"|"InnerProduct"), nsubvector,
 * nbits_per_idx, training_threshold, bucket_init_size, bucket_max_size (may be NULL/""). */
gb_index *gb_index_create(const char *index_type, int dimension, const char *model_params_json, int device);
void gb_index_destroy(gb_index *index);

/* VectorManager::AddToStore (vector_manager.cc:455): append n raw vectors (n x d fp32). */
int gb_index_add_vectors(gb_index *index, int64_t n, const float *x);
int gb_index_add_vectors_device(gb_index *index, int64_t n, const float *x_dev, int64_t ld);
/* Engine::Update (search/engine.cc:774-850): RawVector update in place + IndexModel::Update (old list
 * entry tombstoned, vector re-appended to its new list; realtime_mem_data.cc:298-320) */
int gb_index_update_vector(gb_index *index, int64_t vid, const float *x);
int gb_index_get_vector(gb_index *index, int64_t vid, float *out);
int gb_index_get_vectors(gb_index *index, int64_t start, int64_t n, float *out); /* n x d */

/* IndexModel::Indexing(): train on the first training_threshold stored vectors
 * (gamma_index_ivfflat.cc:342-411, gamma_index_ivfpq.cc:296-376). */
int gb_index_train(gb_index *index);
/* VectorManager::AddRTVecsToIndex (vector_manager.cc:572-702) -> IndexModel::Add: index every
 * stored vector that is not indexed yet.  del_bitmap (host, may be NULL): docids deleted before
 * they were indexed are skipped (gamma_index_ivfflat.cc:436). */
int gb_index_add_pending(gb_index *index, const uint8_t *del_bitmap);

int64_t gb_index_ntotal(gb_index *index);        /* stored vectors */
int64_t gb_index_indexed_count(gb_index *index); /* vectors present in the index */
int gb_index_is_trained(gb_index *index);
int gb_index_training_threshold(gb_index *index);
int64_t gb_index_mem_bytes(gb_index *index, int which /* 0 = index, 1 = raw vectors */);

/* IndexModel::Search (index_model.h:296-298) with the RetrievalContext flattened:
 * retrieval_params_json = the request's index_params (nprobe, metric_type, recall_num,
 * parallel_on_queries; gamma_index_ivfpq.cc:233-294), brute_force => FLAT scan,
 * del_bitmap / filter_bitmap = docids_bitmap / scalar filter as dense LSB-first bitmaps of
 * bitmap_bits bits (NULL = none), [min_score, max_score] = IsSimilarScoreValid window. */
int gb_index_search(gb_index *index, int nq, const float *x, int k, const char *retrieval_params_json,
                    int brute_force, const uint8_t *del_bitmap, const uint8_t *filter_bitmap, int64_t bitmap_bits,
                    float min_score, float max_score, float *out_scores, int64_t *out_ids);
/* Same with queries and results resident in HBM (x_dev: nq rows, stride ld floats) on `stream`
 * (a cudaStream_t, may be NULL).  Asynchronous: results are ready when the stream is. */
int gb_index_search_device(gb_index *index, int nq, const float *x_dev, int64_t ld, int k,
                           const char *retrieval_params_json, int brute_force, float *out_scores_dev,
                           int64_t *out_ids_dev, void *stream);
/* Same, additionally (or only: out_scores_dev / out_ids_dev may be NULL) writing the nq x k result KEYS,
 * (order-preserving score bits << 32) | local doc id, best first, 0xFF..FF padded: what one partition
 * contributes to the cross-partition merge (one all-gather instead of scores + ids). */
int gb_index_search_device_keys(gb_index *index, int nq, const float *x_dev, int64_t ld, int k,
                                const char *retrieval_params_json, int brute_force, unsigned long long *out_keys_dev,
                                float *out_scores_dev, int64_t *out_ids_dev, void *stream);
/* {"stage": ms, ...}: device time per stage of the searches run since the last call with timing enabled
 * (CUDA events on the launching stream); *json_out is malloc'd, the caller frees it */
int gb_index_stage_times(gb_index *index, char **json_out, int *out_len);
/* device time of the dominant scan kernel(s) of the last search, ms (0 unless timing enabled) */
void gb_index_set_scan_timing(gb_index *index, int on);
float gb_index_last_scan_ms(gb_index *index);
/* name of the scan kernel(s) that served the last search (bench roofline label) */
const char *gb_index_last_scan_kernel(gb_index *index);
/* JSON details of the path that served the last search (e.g. probes scanned exactly before the tensor-core filter) */
const char *gb_index_last_scan_info(gb_index *index);

/* ---- index-state exchange (parity tests share centroids / codebooks / lists with the oracle,
 * SURVEY.md 8c; also the substrate for Dump/Load) ---- */
int gb_index_nlist(gb_index *index);
int gb_index_set_centroids(gb_index *index, const float *centroids, int nlist); /* marks trained */
int gb_index_get_centroids(gb_index *index, float *centroids);
int gb_index_pq_m(gb_index *index);
int gb_index_set_pq_centroids(gb_index *index, const float *pq); /* [M][256][dsub] */
int gb_index_get_pq_centroids(gb_index *index, float *pq);
int gb_index_get_precomputed_table(gb_index *index, float *table); /* [nlist][M][256] */
/* OPQ rotation of an IVFPQ index created with "opq": {"nsubvector": M} (gamma_index_ivfpq.cc:168-178):
 * A is d x d row-major, y = A x; apply runs the device path the index itself uses */
int gb_index_has_opq(gb_index *index);
int gb_index_set_opq(gb_index *index, const float *A);
int gb_index_get_opq(gb_index *index, float *A);
int gb_index_apply_opq(gb_index *index, int64_t n, const float *x, float *out);
int gb_index_list_len(gb_index *index, int list);
int gb_index_code_size(gb_index *index);
/* copy one inverted list to the host: codes = len x code_size bytes, ids = len int64 */
int gb_index_get_list(gb_index *index, int list, uint8_t *codes, int64_t *ids);
int gb_index_tombstone(gb_index *index, int list, int pos);
/* IndexModel::Dump / Load (index/index_model.h) in gamma's own file formats -- "IvFl" / "IwPQ" header,
 * IndexFlat quantizer, "ilar" inverted lists (index/impl/gamma_index_ivfflat.cc:807-892,
 * gamma_index_ivfpq.cc:1019-1116, index/index_io.cc:108-194): <dir>/<abs_name>/{ivfflat,ivfpq}.index.
 * dump: 0 on success (also when untrained: nothing written, like the reference).  load: the vectors
 * the file indexes must already be in the store (gb_index_add); *load_num = vectors covered, 0 if
 * there is no file.  FLAT indexes: both are no-ops. */
int gb_index_dump(gb_index *index, const char *dir, const char *abs_name);
/* re-pack the inverted lists into one tight allocation (the growable lists of
 * realtime_mem_data.cc never give memory back; neither do ours until this runs).  Also done
 * automatically after a bulk add when more than half of the list memory is dead. */
int gb_index_compact(gb_index *index);
/* test hook: how often the tensor-core mirror of the lists (DESIGN.md section 2) was built in full; appends
 * that fit the reserved tiles update it in place and do not count */
int gb_index_mirror_builds(gb_index *index);
int gb_index_load(gb_index *index, const char *dir, const char *abs_name, int64_t *load_num);
/* quantizer->search (gamma_index_ivfflat.cc:568) */
int gb_index_coarse_search(gb_index *index, int nq, const float *x, int nprobe, float *out_dis, int64_t *out_ids);
/* search_preassigned (gamma_index_ivfflat.cc:579, gamma_index_ivfpq.cc:730) with caller-given
 * probe lists and coarse distances */
int gb_index_search_preassigned(gb_index *index, int nq, const float *x, int k, const int64_t *keys,
                                const float *coarse_dis, int nprobe, const char *retrieval_params_json,
                                const uint8_t *del_bitmap, const uint8_t *filter_bitmap, int64_t bitmap_bits,
                                float min_score, float max_score, float *out_scores, int64_t *out_ids);
/* pq.compute_codes on residuals (gamma_index_ivfpq.cc:489-494) */
int gb_index_pq_encode(gb_index *index, int64_t n, const float *x, const int64_t *assign, uint8_t *codes);
/* IVFRABITQ: rabitq.compute_codes_core on residuals (gamma_index_ivfrabitq.cc:304-418), codes n x code_size */
int gb_index_rabitq_encode(gb_index *index, int64_t n, const float *x, const int64_t *assign, uint8_t *codes);
/* IVFRABITQ test hook: the scan's per-(query, probe) constants, out = nq x nprobe x 8 floats
 * {vl, delta, cB*sum qq, cB*d, |q-c|^2 (L2) or <q,c> (IP), 1.9 |q-c|, sum qq (int32 bits), cB} (DESIGN.md section 5b) */
int gb_index_rabitq_query_consts(gb_index *index, int nq, const float *x, const int64_t *keys, int nprobe, int qb,
                                 int centered, float *out);

/* ---- standalone kernels exposed for tests / bench ---- */
/* faiss Clustering restated (k-means), host in/out; obj (niter floats) may be NULL */
int gb_kmeans(int device, const float *x, int64_t n, int d, int k, int niter, int64_t seed, int spherical,
              int max_points_per_centroid, float *centroids, float *obj);
/* centroid update only: centroids[c] = mean of x[assign == c] in point order */
int gb_kmeans_update(int device, const float *x, int64_t n, int d, int k, const int64_t *assign, float *centroids);
/* router merge (internal/client/client.go:1530-1609) on device memory: dis/ids are
 * nparts x nq x k, outputs nq x k with ids = (partition << 32) | local id */
int gb_merge_partitions_device(int device, const float *dis_dev, const int64_t *ids_dev, int nparts, int nq, int k,
                               int metric, float *out_dis_dev, int64_t *out_ids_dev, void *stream);
/* the same merge from the partitions' result keys [nparts][nq][k] (gb_index_search_device_keys) */
int gb_merge_partition_keys_device(int device, const unsigned long long *keys_dev, int nparts, int nq, int k, int metric,
                                   float *out_dis_dev, int64_t *out_ids_dev, void *stream);

/* exact (CUDA-core fp32) or tensor-core (tcgen05 3xTF32) score matrix, host in/out: out[n][m] */
int gb_debug_dist_matrix(int device, const float *x, int n, const float *c, int m, int d, int metric, int use_tc,
                         float *out);

/* ---- host-logic test hooks: run the C++ wire codecs of the gamma boundary without a GPU ---- */
/* RequestConcurrentController (search/engine.cc:47-119): op 0 threshold, 1 in-flight, 2 set threshold (<= 0: system value),
 * 3 Acquire(value) -> 1/0, 4 Release(value) */
int gb_debug_concurrency(int op, int value);
int gb_debug_parse_search_request(const char *buf, int len, char **json_out, int *out_len);
int gb_debug_roundtrip_doc(const char *buf, int len, char **out, int *out_len);
int gb_debug_parse_table(const char *buf, int len, char **json_out, int *out_len);
int gb_debug_encode_response(int nq, int k, const double *scores, const char *const *keys, int total, char **out,
                             int *out_len);

#ifdef __cplusplus
}
#endif
#endif /* GAMMA_B200_INDEX_H_ */
