// Host-callable launchers of the sm_100a kernels (one per row of SURVEY.md 8a).
// Plain pointers + stream, no torch types.  All device matrices are row-major fp32 with a row
// stride ("ld") that is a multiple of 4 floats so rows are 16-byte aligned.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace gb {

constexpr int kMetricIP = 0;  // DistanceComputeType::INNER_PRODUCT (gamma default, gamma_index_ivfflat.cc:55)
constexpr int kMetricL2 = 1;

// number of kernels launched by this library so far (bench.py's gpu_launches evidence)
void note_launch(int n = 1);
long long launch_count();

struct FilterArgs {            // RetrievalContext (index/index_model.h:86-110)
  const uint32_t* del_bits;    // bit set => docid deleted            (nullable)
  const uint32_t* filter_bits; // bit set => docid passes the filter  (nullable = no filter)
  float min_score, max_score;  // IsSimilarScoreValid window
};

// ---- K1/K2/K6/K8: tiled exact distance kernel ------------------------------------------
// out[i][j] = |X_i - C_j|^2 (L2) or <X_i, C_j> (IP), i<n, j<m.  d multiple of 4.
cudaError_t launch_dist_matrix(const float* X, int64_t ldx, int n, const float* C, int64_t ldc, int m, int d,
                               int metric, float* out, int64_t ldo, cudaStream_t st);
// best[i] = min over j of key(score(X_i,C_j), j + col_base) via atomicMin; caller pre-fills
// best with 0xFF.. .  Lowest j wins ties (faiss IndexFlat::assign, "first minimum wins").
cudaError_t launch_dist_argmin(const float* X, int64_t ldx, int n, const float* C, int64_t ldc, int m, int d,
                               int metric, unsigned long long* best, int col_base, cudaStream_t st);

// tensor-core (tcgen05, 3xTF32) variants of the two calls above (norms accumulated in-kernel).
// Scores agree with the exact kernel to ~1e-6 relative and are bit-equal on integer-valued
// operands below 2^11.
cudaError_t launch_dist_matrix_tc(const float* X, int64_t ldx, int n, const float* C, int64_t ldc, int m, int d,
                                  int metric, float* out, int64_t ldo, cudaStream_t st);
cudaError_t launch_dist_argmin_tc(const float* X, int64_t ldx, int n, const float* C, int64_t ldc, int m, int d,
                                  int metric, unsigned long long* best, cudaStream_t st);

// ---- K7: top-k selection / merge ----------------------------------------------------------
// Per row r: select the k best of m candidates.  Input is either scores (fp32, vid = id_base+col)
// or ready-made keys.  Output keys sorted ascending (sentinel padded) in out_keys[r*k..].
cudaError_t launch_select_scores(const float* scores, int64_t ld, int nrows, int m, int64_t id_base, int k, int metric,
                                 FilterArgs f, unsigned long long* out_keys, int64_t out_stride, cudaStream_t st);
cudaError_t launch_select_keys(const unsigned long long* keys, int64_t ld, int nrows, int m, int k,
                               unsigned long long* out_keys, int64_t out_stride, cudaStream_t st);
// keys -> (score, id) in the reference's output order (heap_reorder): L2 (score, id) ascending;
// IP score descending, larger id first among equal scores.  Sentinels -> id -1, score +-FLT_MAX.
cudaError_t launch_decode_keys(const unsigned long long* keys, int64_t ld, int nrows, int k, int metric, float* out_dis,
                               int64_t* out_ids, int64_t id_or /* OR-ed into valid ids */, cudaStream_t st);
// keys -> int32 ids / float scores only (coarse quantiser output)
cudaError_t launch_split_keys(const unsigned long long* keys, int64_t n, int metric, float* out_scores, int32_t* out_ids,
                              cudaStream_t st);

// ---- K3: IVF-Flat list scan ---------------------------------------------------------------
struct ListDirectory {            // device-resident mirror of RTInvertIndex (T1)
  const float* const* vecs;       // [nlist] -> len x dpad fp32 rows (codes_array_)
  const uint8_t* const* codes;    // [nlist] -> len x M bytes (IVFPQ)
  const int64_t* const* ids;      // [nlist] -> len int64, top bit = tombstone (idx_array_)
  const int* len;                 // [nlist] published length
  int nlist;
};
// partial[q][part][k]; *nparts_out (<= ivfflat_scan_nparts) = parts actually written per query.
// One CTA per (query, group of (probe, split) work items).
cudaError_t launch_ivfflat_scan(const float* xq, int64_t ldq, int nq, int d, const int32_t* probe_ids, int nprobe,
                                ListDirectory dir, int max_list_len, int avg_list_len, int k, int metric, FilterArgs f,
                                unsigned long long* partial, int* nparts_out, cudaStream_t st);
int ivfflat_scan_nparts(int nprobe, int max_list_len);

// K3 list-major (tensor cores): (query, probe) pairs grouped by list; tile = 128 pairs x 128 rows.
struct LmTile {
  int list, pair0, npairs, row0, nrows, seg;
  int grp;  // ordinal of this (list, pair group): its slot in the staged-query scratch
};
// scores[pair_off[j] + r] = score(query pair_q[j], row r of its list)
cudaError_t launch_ivf_listmajor_tc(const float* xq, int64_t ldq, int d, const LmTile* tiles, int ntiles,
                                    const int32_t* pair_q, const int64_t* pair_off, ListDirectory dir, int metric,
                                    float* scores, cudaStream_t st);
// device-side grouping of the (query, probe) pairs by list: histogram + scans (totals[0..2] = score
// floats, tiles, valid pairs), then slot assignment and the tile table
cudaError_t launch_lm_count_scan(const int32_t* probe_ids, int64_t npairs, ListDirectory dir, int32_t* cnt,
                                 int32_t* start, int64_t* base_off, int32_t* tile_start, int64_t* totals,
                                 cudaStream_t st);
cudaError_t launch_lm_assign_tiles(const int32_t* probe_ids, int64_t npairs, int nprobe, ListDirectory dir,
                                   const int32_t* cnt, const int32_t* start, int32_t* cursor, const int64_t* base_off,
                                   const int32_t* tile_start, int32_t* pair_q, int64_t* pair_off, int64_t* seg_off,
                                   LmTile* tiles, cudaStream_t st);
// per query: stream its nprobe score segments (seg_off[q*nprobe+p], -1 = none), filter, top-k -> out_keys[q][k]
cudaError_t launch_seg_select(const float* scores, const int64_t* seg_off, const int32_t* probe_ids, int nq, int nprobe,
                              ListDirectory dir, int k, int metric, FilterArgs f, unsigned long long* out_keys,
                              cudaStream_t st);

// K3 list-major with a fused top-k epilogue (k <= kLmkMaxK): work item = (list, 128 pairs, row segment);
// the CTA walks the segment's 128-row tiles, every thread keeps the k best keys of its (query, list)
// pair in shared memory and admits candidates against a per-query bound shared through tau_g.
// out[(j * nseg_max + seg) * k + i], j = q * nprobe + p; unused slots must be pre-set to the sentinel.
constexpr int kLmkMaxK = 64;
constexpr int kLmkSegRows = 2048;
// grouping: cnt/start/cursor/item_start/grp_start: [nlist] ints; totals = {groups, items, pairs} (device side)
cudaError_t launch_lmk_group(const int32_t* probe_ids, int64_t npairs, ListDirectory dir, int nseg_max, int32_t* cnt,
                             int32_t* start, int32_t* cursor, int32_t* item_start, int32_t* grp_start, int64_t* totals,
                             int64_t* pair_j, LmTile* items, cudaStream_t st);
// TMA-fed variant (kernels_tc.cu, "mirror"): the lists are kept a second time pre-split (TF32 head +
// fp32 remainder) and pre-tiled in the exact shared-memory operand layout, so a K chunk of a 128-row
// tile is one contiguous 16 KiB block a single cp.async.bulk brings in; row norms are precomputed.
struct TcMirrorView {
  const float* base;     // tile t of the index at base + t * tile_floats(k16)
  const int64_t* tile0;  // [nlist + 1] first tile of every list
  const float* norms;    // [total_tiles * 128] |y|^2, 0 for padding rows
  int k16;               // row length rounded up to the K chunk (16)
};
inline int64_t tc_mirror_tile_floats(int k16) { return (int64_t)128 * k16 * 2; }
// rows just appended to the lists (row i of x -> position pos[i] of list list[i], list < 0: skipped)
cudaError_t launch_tc_mirror_append(const float* x, int64_t ldx, int64_t n, int d, int k16, const int32_t* list,
                                    const int32_t* pos, const int64_t* tile0, float* mirror, float* norms, cudaStream_t st);
cudaError_t launch_tc_mirror_build(ListDirectory dir, int d, int k16, const int64_t* tile0, int64_t total_tiles,
                                   float* mirror, float* norms, cudaStream_t st);
// a_scratch: per pair group nk chunks of 16 KiB (hi, lo) of the group's 128 queries; a_norms: [group][128]
cudaError_t launch_lm_stage_queries(const float* xq, int64_t ldq, int d, int k16, const LmTile* items, int max_items,
                                    const int64_t* totals, const int64_t* pair_j, int nprobe, float* a_scratch,
                                    float* a_norms, cudaStream_t st);
cudaError_t launch_ivf_listmajor_tma(const float* a_scratch, const float* a_norms, TcMirrorView mv, const LmTile* items,
                                     int max_items, const int64_t* totals, const int64_t* pair_j, int nprobe,
                                     ListDirectory dir, int k, int nseg_max, int metric, FilterArgs f,
                                     unsigned long long* tau_g, unsigned long long* out, cudaStream_t st);
cudaError_t launch_ivf_listmajor_topk(const float* xq, int64_t ldq, int d, const LmTile* items, int max_items,
                                      const int64_t* totals, const int64_t* pair_j, int nprobe, ListDirectory dir, int k,
                                      int nseg_max, int metric, FilterArgs f, unsigned long long* tau_g,
                                      unsigned long long* out, cudaStream_t st);

// ---- OPQ training helpers (kernels_build.cu) ---------------------------------------------------
// out[i][j] = x[i][j] - mean_j (columns >= d zeroed up to ldo); mean computed on device
cudaError_t launch_center_rows(const float* x, int64_t ldx, int64_t n, int d, float* out, int64_t ldo, cudaStream_t st);
// out[j][i] = x[i][j]  (n x d -> d x n, row stride ldo >= n)
cudaError_t launch_transpose(const float* x, int64_t ldx, int64_t n, int d, float* out, int64_t ldo, cudaStream_t st);
// recon[i][m * dsub + j] = pq[m][codes[i][m]][j]
cudaError_t launch_pq_decode(const uint8_t* codes, int64_t n, const float* pq_centroids, int M, int dsub, float* recon,
                             int64_t ldr, cudaStream_t st);

// ---- K4/K5: IVF-PQ look-up tables + ADC scan --------------------------------------------
// ip[q][m][c] = <x_q|m, pq_m[c]>   (pq.compute_inner_prod_table)
cudaError_t launch_pq_ip_table(const float* xq, int64_t ldq, int nq, const float* pq_centroids, int M, int dsub,
                               float* ip, cudaStream_t st);
// T[l][m][c] = |pq_m[c]|^2 + 2 <centroid_l|m, pq_m[c]>  (IndexIVFPQ::precompute_table)
cudaError_t launch_pq_precompute_table(const float* coarse, int64_t ldc, int nlist, const float* pq_centroids, int M,
                                       int dsub, float* T, cudaStream_t st);
// partial[q][group][k], group = ceil(nprobe/pg) CTAs per query, each scanning pg (<= 32) probed lists.
// coarse_dis = dis0 per (q, probe).  T nullable for IP.
// ld_probe: row stride of probe_ids / coarse_dis (0 = nprobe; > nprobe scans the first nprobe probes of
// every row).  gate_cnt: when non-null only queries with gate_cnt[q] > gate_cap are scanned.
cudaError_t launch_ivfpq_scan(const float* ip_table, int nq, const int32_t* probe_ids, const float* coarse_dis,
                              int nprobe, int pg, ListDirectory dir, int M, const float* T, int k, int metric,
                              FilterArgs f, unsigned long long* partial, cudaStream_t st, int ld_probe = 0,
                              const int* gate_cnt = nullptr, int gate_cap = 0, const int* row_limit = nullptr,
                              bool sorted_out = true);  // false: partial[..][k - 1] = the largest key, the others in any order

// ---- K5 list-major: tensor-core filter + exact re-score (kernels_pqtc.cu) ---------------------------
bool pqtc_supported(int M, int dsub);
void pqtc_debug_counters(unsigned long long out[4], bool reset);  // GB_PQTC_DBG diagnostics
size_t pqtc_pair_meta_bytes();
// cb[m][c][.] = fp16(-2 sb pq) (L2) / fp16(-sb pq) (IP), sb = rmax2[1] a power of two; nrm[m][c] = |pq[m][c]|^2; rmax2[0] = sum_m max_c nrm
cudaError_t launch_pqtc_tables(const float* pq, int M, int dsub, int metric, uint16_t* cb, float* nrm, float* rmax2,
                               cudaStream_t st);
// phase A's plan: per query its first P_q probes in full (fewest with >= target entries together, at most pa_max);
// probes_a / probes_b = probe_ids with the other phase's probes set to -1, row_limit[q][p] = rows phase A scores exactly
cudaError_t launch_pqtc_plan_phase_a(const int32_t* probe_ids, int64_t npairs, int nprobe, int pa_max, long long target,
                                     const int* list_len, int32_t* probes_a, int32_t* probes_b, int* row_limit,
                                     cudaStream_t st);
// per pair group: fp16 operand tile (rows scaled by their own power of two) of (x - centroid) (L2) / x (IP) rows + the pairs' filter thresholds from
// bound_keys[q][kprime - 1] (phase A's k'-th key); queries without a bound get cand_cnt = cap + 1
cudaError_t launch_pq_stage_pairs(const float* xq, int64_t ldq, int d, const float* coarse, int64_t ldc, const LmTile* items,
                                  int max_items, const int64_t* totals, const int64_t* pair_j, int nprobe,
                                  const float* coarse_dis, const unsigned long long* bound_keys, int64_t bound_stride,
                                  int kprime, const float* rmax2, FilterArgs f, int metric, float eps_scale,
                                  unsigned char* a_scratch, void* meta, int* cand_cnt, int cap, const int* row_limit, cudaStream_t st);
// persistent kernel, one CTA per SM: candidates (probe << 32 | position) appended to cand[q][cap]
cudaError_t launch_pqtc_scan(const unsigned char* a_scratch, const void* meta, const uint16_t* cb, const float* pqnorm, const int64_t* pqnorm_off,
                             const LmTile* items, int max_items, const int64_t* totals, ListDirectory dir, int M, int dsub,
                             FilterArgs f, int metric, int* cand_cnt, unsigned long long* cand, int cap, int num_sms,
                             cudaStream_t st);
// |r_e|^2 of every list entry: out[off[l] + pos] (L2; cached beside the lists, streamed to the filter kernel with the codes)
cudaError_t launch_pq_entry_norms(ListDirectory dir, int nlist, int max_len, int M, const float* nrm, const int64_t* off,
                                  float* out, cudaStream_t st);
// out[q][kprime] = best kprime of keys_a[q] + the re-scored candidates (queries with cand_cnt > cap untouched)
cudaError_t launch_pq_rescore(const float* ip_table, int nq, const int32_t* probe_ids, const float* coarse_dis, int nprobe,
                              ListDirectory dir, int M, const float* T, const int* cand_cnt, const unsigned long long* cand,
                              int cap, const unsigned long long* keys_a, int64_t keys_a_stride, int kprime, int metric,
                              const int* row_limit, FilterArgs f, bool sorted_out, unsigned long long* out, cudaStream_t st);
// queries with cand_cnt > cap: out[q] = best kprime of partial[q][ngroups][kprime]
cudaError_t launch_pq_fallback_merge(const int* cand_cnt, int cap, int nq, const unsigned long long* partial, int ngroups,
                                     int kprime, unsigned long long* out, cudaStream_t st);
// K5r exact re-rank of ADC candidates (gamma_index_ivfpq.cc:675-726)
cudaError_t launch_rerank(const unsigned long long* cand_keys, int ncand, int nq, const float* xq, int64_t ldq, int d,
                          const float* const* raw_segments, int seg_shift, int64_t ld_raw, int k, int metric,
                          FilterArgs f, unsigned long long* out_keys, cudaStream_t st);

// ---- IVFRABITQ: RaBitQ codes, query quantisation, scan (kernels_rabitq.cu; DESIGN.md section 5b) ---------
// bytes per entry: sign plane (P = ceil(d/8)) + {or_c, f1} (1 bit) or
// sign plane + {or_c, f1, f_error} + (nb_bits - 1) extra planes + {f_ex} (multi-bit)
__host__ __device__ inline int rabitq_code_size(int d, int nb_bits) {
  const int P = (d + 7) / 8;
  return nb_bits == 1 ? P + 8 : nb_bits * P + 16;
}
// per-(query, probe) constants: {vl, delta, cB * sum qq, cB * d, |q-c|^2 (L2) / <q,c> (IP), 1.9 |q-c|, sum qq (int bits), cB}
constexpr int kRabitqConsts = 8;
// codes[i] = code of x_i - coarse[assign_i] (assign < 0: centroid 0, the row is not appended)
cudaError_t launch_rabitq_encode(const float* x, int64_t ldx, int64_t n, int d, const float* coarse, int64_t ldc,
                                 const int32_t* assign, int nb_bits, int metric, uint8_t* codes, cudaStream_t st);
// pair j = q * nprobe + p: consts[j][8], planes[j][qb][ceil(d/32)] (qb > 0)
cudaError_t launch_rabitq_query_prep(const float* xq, int64_t ldq, int nq, int d, const int32_t* probe_ids, int nprobe,
                                     const float* coarse, int64_t ldc, int nlist, int qb, bool centered, int nb_bits,
                                     int metric, float* consts, uint32_t* planes, cudaStream_t st);
// partial[q][group][k] sorted keys, group = ceil(nprobe / pg) CTAs per query (pg <= 32)
// false if the scan's shared-memory ring (two stages of at least 16 codes) cannot hold codes of this shape
bool rabitq_scan_supported(int d, int nb_bits);
// (qb = 0: the float query residual x_q - c is formed in the scan from xq and coarse)
cudaError_t launch_rabitq_scan(const float* consts, const uint32_t* planes, const float* xq, int64_t ldq,
                               const float* coarse, int64_t ldc, int nq,
                               const int32_t* probe_ids, int nprobe, int pg, ListDirectory dir, int d, int nb_bits, int qb,
                               int k, int metric, FilterArgs f, unsigned long long* partial, cudaStream_t st);

// ---- K6/K8: build-side kernels ------------------------------------------------------------
// centroids[c] = (sum of x[perm[off[c]..off[c+1])] in that order) * (1/count); empty => zeros
cudaError_t launch_segment_mean(const float* x, int64_t ldx, int d, const int32_t* perm, const int32_t* off, int k,
                                float* centroids, int64_t ldc, cudaStream_t st);
// out = x - centroids[assign]
cudaError_t launch_residual(const float* x, int64_t ldx, int64_t n, int d, const float* centroids, int64_t ldc,
                            const int32_t* assign, float* out, int64_t ldo, cudaStream_t st);
// codes[i][m] = argmin_c |(x_i - coarse[assign_i])|m - pq_m[c]|^2 (coarse nullable => no residual)
cudaError_t launch_pq_encode(const float* x, int64_t ldx, int64_t n, const float* coarse, int64_t ldc,
                             const int32_t* assign, const float* pq_centroids, int M, int dsub, uint8_t* codes,
                             cudaStream_t st);
// copy a column slice [col0, col0+w) of x into a dense n x ldo buffer (zero padded to ldo)
cudaError_t launch_slice_cols(const float* x, int64_t ldx, int64_t n, int col0, int w, float* out, int64_t ldo,
                              cudaStream_t st);
// gather rows: out[i] = x[idx[i]]
cudaError_t launch_gather_rows(const float* x, int64_t ldx, const int32_t* idx, int64_t n, int d, float* out,
                               int64_t ldo, cudaStream_t st);
// scale rows to unit L2 norm in place (spherical k-means)
cudaError_t launch_normalize_rows(float* x, int64_t ldx, int64_t n, int d, cudaStream_t st);
// IVF append (RTInvertIndex::AddKeys): row i -> list[i] at pos[i]
cudaError_t launch_ivf_append_vecs(const float* x, int64_t ldx, int64_t n, int d, const int32_t* list, const int32_t* pos,
                                   float* const* list_vecs, int64_t* const* list_ids, int64_t vid0, cudaStream_t st);
cudaError_t launch_ivf_append_codes(const uint8_t* codes, int64_t n, int M, const int32_t* list, const int32_t* pos,
                                    uint8_t* const* list_codes, int64_t* const* list_ids, int64_t vid0,
                                    cudaStream_t st);
cudaError_t launch_fill_u64(unsigned long long* p, int64_t n, unsigned long long v, cudaStream_t st);
cudaError_t launch_pad_rows(const float* src, int64_t n, int d, float* dst, int64_t ldd, cudaStream_t st);

}  // namespace gb
