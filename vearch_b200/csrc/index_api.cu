// extern "C" surface of include/gamma_b200_index.h.
#include <strings.h>

#include <algorithm>
#include <vector>

#include "../../include/gamma_b200_index.h"
#include "common.cuh"
#include "index.h"
#include "json.h"
#include "params.h"

using namespace gb;

struct gb_index {
  Index* impl;
};

namespace gb {

// IVFFlatModelParams::Parse / IVFPQModelParams::Parse (gamma_index_ivfflat.cc:64-196,
// gamma_index_ivfpq.h:1031-1257)
bool parse_model_params(const std::string& text, ModelParams* mp, std::string* err) {
  if (text.empty()) return true;
  JsonValue jv;
  if (!JsonParser::parse(text, &jv) || jv.type != JsonValue::Object) {
    *err = "parse model parameters error: " + text;
    return false;
  }
  int v;
  if (jv.get("ncentroids")) {
    if (!jv.get_int("ncentroids", &v)) {
      *err = "parse ncentroids error";
      return false;
    }
    if (v > 0) mp->ncentroids = v;
  }
  if (jv.get_int("nprobe", &v)) {
    if (v < -1) {
      *err = "invalid nprobe =" + std::to_string(v);
      return false;
    }
    if (v > 0) mp->nprobe = v;
    if (mp->nprobe > mp->ncentroids) {
      *err = "nprobe should less than ncentroids";
      return false;
    }
  }
  if (jv.get_int("nsubvector", &v)) {
    if (v < -1) {
      *err = "invalid nsubvector =" + std::to_string(v);
      return false;
    }
    if (v > 0) mp->nsubvector = v;
  }
  if (const JsonValue* opq = jv.get("opq")) {  // gamma_index_ivfpq.h:1202-1216
    if (opq->type == JsonValue::Object && opq->get_int("nsubvector", &v)) {
      if (v < -1) {
        *err = "invalid opq_nsubvector = " + std::to_string(v);
        return false;
      }
      if (v > 0) mp->opq_nsubvector = v;
    }
  }
  if (jv.get_int("nbits_per_idx", &v)) {
    if (v < -1) {
      *err = "invalid nbits_per_idx =" + std::to_string(v);
      return false;
    }
    if (v > 0) mp->nbits = v;
  }
  if (jv.get_int("bucket_init_size", &v)) {
    if (v < -1) {
      *err = "invalid bucket_init_size =" + std::to_string(v);
      return false;
    }
    if (v > 0) mp->bucket_init_size = v;
  }
  if (jv.get_int("bucket_max_size", &v)) {
    if (v < -1) {
      *err = "invalid bucket_max_size =" + std::to_string(v);
      return false;
    }
    if (v > 0) mp->bucket_max_size = v;
  }
  if (jv.get_int("training_threshold", &v) && v > 0) mp->training_threshold = v;
  // IVFRABITQ (gamma_index_ivfrabitq.h:335-537): kept as given, range-checked by create_index("IVFRABITQ")
  if (jv.get("nb_bits")) {
    if (!jv.get_int("nb_bits", &v)) {
      *err = "invalid nb_bits should be integer in [1, 9]";
      return false;
    }
    mp->nb_bits = v;
  }
  if (jv.get("qb")) {
    if (!jv.get_int("qb", &v)) {
      *err = "invalid qb should be integer in [0, 8]";
      return false;
    }
    mp->qb = v;
  }
  std::string mt;
  if (jv.get_string("metric_type", &mt)) {
    if (strcasecmp("L2", mt.c_str()) && strcasecmp("InnerProduct", mt.c_str())) {
      *err = "invalid metric_type = " + mt;
      return false;
    }
    mp->metric = !strcasecmp("L2", mt.c_str()) ? kMetricL2 : kMetricIP;
  }
  return true;
}

// GammaIVFPQIndex::Parse / GammaIVFFlatIndex::Parse (gamma_index_ivfpq.cc:233-294,
// gamma_index_ivfflat.cc:293-340): invalid values fall back to the index defaults.
bool parse_retrieval_params(const std::string& text, RetrievalParams* rp, std::string* err) {
  if (text.empty()) return true;
  JsonValue jv;
  if (!JsonParser::parse(text, &jv) || jv.type != JsonValue::Object) {
    *err = "parse retrieval parameters error: " + text;
    return false;
  }
  std::string mt;
  if (jv.get_string("metric_type", &mt)) rp->metric = !strcasecmp("L2", mt.c_str()) ? kMetricL2 : kMetricIP;
  int v;
  if (jv.get_int("recall_num", &v) && v > 0) rp->recall_num = v;
  if (jv.get_int("nprobe", &v) && v > 0) rp->nprobe = v;
  if (jv.get_int("parallel_on_queries", &v)) rp->parallel_on_queries = v != 0;
  if (jv.get_int("qb", &v)) rp->qb = v < 0 ? -2 : v;  // IVFRABITQ; out of range => the model's qb
  bool b;
  if (jv.get_bool("centered", &b)) rp->centered = b;
  return true;
}

}  // namespace gb

static int fill_ctx(SearchContext* ctx, const char* rp_json, int brute_force, const uint8_t* del_bitmap,
                    const uint8_t* filter_bitmap, int64_t bitmap_bits, float min_score, float max_score) {
  std::string err;
  if (!parse_retrieval_params(rp_json ? rp_json : "", &ctx->params, &err)) {
    set_last_error(err);
    return -1;
  }
  ctx->params.brute_force = brute_force != 0;
  ctx->del_bitmap = del_bitmap;
  ctx->filter_bitmap = filter_bitmap;
  ctx->bitmap_bits = bitmap_bits;
  ctx->min_score = min_score;
  ctx->max_score = max_score;
  return 0;
}

#define IDX_OR_FAIL(idx)                 \
  if (!(idx) || !(idx)->impl) {          \
    set_last_error("null index handle"); \
    return -1;                           \
  }

extern "C" {

const char* gb_last_error(void) { return last_error(); }

long long gb_launch_count(void) { return launch_count(); }

int gb_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

gb_index* gb_index_create(const char* index_type, int dimension, const char* model_params_json, int device) {
  ModelParams mp;
  std::string err;
  if (!parse_model_params(model_params_json ? model_params_json : "", &mp, &err)) {
    set_last_error(err);
    return nullptr;
  }
  Index* impl = create_index(index_type ? index_type : "", dimension, mp, device, 20);
  if (!impl) return nullptr;
  gb_index* h = new gb_index;
  h->impl = impl;
  return h;
}

void gb_index_destroy(gb_index* index) {
  if (!index) return;
  if (index->impl) {
    cudaSetDevice(index->impl->device());
    delete index->impl;
  }
  delete index;
}

int gb_index_add_vectors(gb_index* index, int64_t n, const float* x) {
  IDX_OR_FAIL(index);
  return index->impl->add_vectors(x, n);
}
int gb_index_add_vectors_device(gb_index* index, int64_t n, const float* x_dev, int64_t ld) {
  IDX_OR_FAIL(index);
  return index->impl->add_vectors_device(x_dev, ld, n);
}
int gb_index_update_vector(gb_index* index, int64_t vid, const float* x) {
  IDX_OR_FAIL(index);
  cudaSetDevice(index->impl->device());
  return index->impl->update_vector(vid, x);  // RawVector update + IndexModel::Update
}
int gb_index_get_vector(gb_index* index, int64_t vid, float* out) {
  IDX_OR_FAIL(index);
  cudaSetDevice(index->impl->device());
  return index->impl->store().get_host(vid, out);
}
int gb_index_get_vectors(gb_index* index, int64_t start, int64_t n, float* out) {
  IDX_OR_FAIL(index);
  cudaSetDevice(index->impl->device());
  return index->impl->store().get_rows_host(start, n, out);
}
int gb_index_train(gb_index* index) {
  IDX_OR_FAIL(index);
  return index->impl->train();
}
int gb_index_add_pending(gb_index* index, const uint8_t* del_bitmap) {
  IDX_OR_FAIL(index);
  return index->impl->add_pending(del_bitmap);
}
int64_t gb_index_ntotal(gb_index* index) { return index && index->impl ? index->impl->store().size() : -1; }
int64_t gb_index_indexed_count(gb_index* index) { return index && index->impl ? index->impl->indexed_count() : -1; }
int gb_index_is_trained(gb_index* index) { return index && index->impl ? (int)index->impl->trained() : 0; }
int gb_index_training_threshold(gb_index* index) {
  return index && index->impl ? index->impl->training_threshold() : -1;
}
int64_t gb_index_mem_bytes(gb_index* index, int which) {
  if (!index || !index->impl) return -1;
  return which == 0 ? index->impl->index_mem_bytes() : index->impl->store().mem_bytes();
}

int gb_index_search(gb_index* index, int nq, const float* x, int k, const char* retrieval_params_json, int brute_force,
                    const uint8_t* del_bitmap, const uint8_t* filter_bitmap, int64_t bitmap_bits, float min_score,
                    float max_score, float* out_scores, int64_t* out_ids) {
  IDX_OR_FAIL(index);
  SearchContext ctx;
  if (fill_ctx(&ctx, retrieval_params_json, brute_force, del_bitmap, filter_bitmap, bitmap_bits, min_score, max_score))
    return -1;
  return index->impl->search(ctx, nq, x, k, out_scores, out_ids);
}

int gb_index_search_device(gb_index* index, int nq, const float* x_dev, int64_t ld, int k,
                           const char* retrieval_params_json, int brute_force, float* out_scores_dev,
                           int64_t* out_ids_dev, void* stream) {
  IDX_OR_FAIL(index);
  SearchContext ctx;
  if (fill_ctx(&ctx, retrieval_params_json, brute_force, nullptr, nullptr, 0, -3.4028235e38f, 3.4028235e38f)) return -1;
  return index->impl->search_device(ctx, nq, x_dev, ld, k, out_scores_dev, out_ids_dev,
                                    static_cast<cudaStream_t>(stream));
}

int gb_index_search_device_keys(gb_index* index, int nq, const float* x_dev, int64_t ld, int k,
                                const char* retrieval_params_json, int brute_force, unsigned long long* out_keys_dev,
                                float* out_scores_dev, int64_t* out_ids_dev, void* stream) {
  IDX_OR_FAIL(index);
  SearchContext ctx;
  if (fill_ctx(&ctx, retrieval_params_json, brute_force, nullptr, nullptr, 0, -3.4028235e38f, 3.4028235e38f)) return -1;
  return index->impl->search_device(ctx, nq, x_dev, ld, k, out_scores_dev, out_ids_dev, static_cast<cudaStream_t>(stream),
                                    out_keys_dev);
}

// {"stage": ms, ...} of the searches run since the last call while scan timing was on (malloc'd, caller frees)
int gb_index_stage_times(gb_index* index, char** json_out, int* out_len) {
  IDX_OR_FAIL(index);
  std::string js = "{";
  bool first = true;
  for (auto& kv : index->impl->stage_times()) {
    char buf[64];
    snprintf(buf, sizeof(buf), "%.6f", kv.second);
    js += std::string(first ? "" : ", ") + "\"" + kv.first + "\": " + buf;
    first = false;
  }
  js += "}";
  char* p = static_cast<char*>(malloc(js.size() + 1));
  if (!p) return -1;
  memcpy(p, js.c_str(), js.size() + 1);
  *json_out = p;
  *out_len = (int)js.size();
  return 0;
}

void gb_index_set_scan_timing(gb_index* index, int on) {
  if (index && index->impl) index->impl->set_time_scan(on != 0);
}
const char* gb_index_last_scan_kernel(gb_index* index) {
  return index && index->impl ? index->impl->last_scan_kernel() : "";
}
const char* gb_index_last_scan_info(gb_index* index) { return index && index->impl ? index->impl->last_scan_info() : "{}"; }
float gb_index_last_scan_ms(gb_index* index) { return index && index->impl ? index->impl->last_scan_ms() : 0.f; }

static IVFFlatIndex* as_ivf(gb_index* index) {
  if (!index || !index->impl) return nullptr;
  return dynamic_cast<IVFFlatIndex*>(index->impl);
}
static IVFPQIndex* as_pq(gb_index* index) {
  if (!index || !index->impl) return nullptr;
  return dynamic_cast<IVFPQIndex*>(index->impl);
}
static IVFRaBitQIndex* as_rq(gb_index* index) {
  if (!index || !index->impl) return nullptr;
  return dynamic_cast<IVFRaBitQIndex*>(index->impl);
}
#define IVF_OR_FAIL(v, index)                \
  IVFFlatIndex* v = as_ivf(index);           \
  if (!v) {                                  \
    set_last_error("not an IVF index");      \
    return -1;                               \
  }
#define PQ_OR_FAIL(v, index)                 \
  IVFPQIndex* v = as_pq(index);              \
  if (!v) {                                  \
    set_last_error("not an IVFPQ index");    \
    return -1;                               \
  }

int gb_index_nlist(gb_index* index) {
  IVF_OR_FAIL(ivf, index);
  return ivf->nlist();
}
int gb_index_set_centroids(gb_index* index, const float* centroids, int nlist) {
  IVF_OR_FAIL(ivf, index);
  return ivf->set_centroids(centroids, nlist);
}
int gb_index_get_centroids(gb_index* index, float* centroids) {
  IVF_OR_FAIL(ivf, index);
  return ivf->get_centroids(centroids);
}
int gb_index_pq_m(gb_index* index) {
  PQ_OR_FAIL(pq, index);
  return pq->M();
}
int gb_index_set_pq_centroids(gb_index* index, const float* pqc) {
  PQ_OR_FAIL(pq, index);
  return pq->set_pq_centroids(pqc);
}
int gb_index_get_pq_centroids(gb_index* index, float* pqc) {
  PQ_OR_FAIL(pq, index);
  return pq->get_pq_centroids(pqc);
}
int gb_index_get_precomputed_table(gb_index* index, float* table) {
  PQ_OR_FAIL(pq, index);
  return pq->get_precomputed_table(table);
}
int gb_index_has_opq(gb_index* index) {
  IVFPQIndex* pq = index && index->impl ? dynamic_cast<IVFPQIndex*>(index->impl) : nullptr;
  return pq && pq->has_opq() ? 1 : 0;
}
int gb_index_set_opq(gb_index* index, const float* A) {
  IDX_OR_FAIL(index);
  IVFPQIndex* pq = dynamic_cast<IVFPQIndex*>(index->impl);
  return pq ? pq->set_opq(A) : -1;
}
int gb_index_get_opq(gb_index* index, float* A) {
  IDX_OR_FAIL(index);
  IVFPQIndex* pq = dynamic_cast<IVFPQIndex*>(index->impl);
  return pq ? pq->get_opq(A) : -1;
}
int gb_index_apply_opq(gb_index* index, int64_t n, const float* x, float* out) {
  IDX_OR_FAIL(index);
  IVFPQIndex* pq = dynamic_cast<IVFPQIndex*>(index->impl);
  return pq ? pq->apply_opq_host(x, n, out) : -1;
}
int gb_index_mirror_builds(gb_index* index) {
  if (!index || !index->impl) return -1;
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index->impl);
  return ivf ? ivf->mirror_builds() : 0;
}
int gb_index_compact(gb_index* index) {
  IDX_OR_FAIL(index);
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index->impl);
  return ivf ? ivf->compact_lists() : 0;
}
int gb_index_dump(gb_index* index, const char* dir, const char* abs_name) {
  IDX_OR_FAIL(index);
  if (!dir || !abs_name) return -1;
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index->impl);
  return ivf ? ivf->dump_gamma(dir, abs_name) : 0;
}
int gb_index_load(gb_index* index, const char* dir, const char* abs_name, int64_t* load_num) {
  IDX_OR_FAIL(index);
  if (!dir || !abs_name || !load_num) return -1;
  *load_num = 0;
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index->impl);
  return ivf ? ivf->load_gamma(dir, abs_name, load_num) : 0;
}
int gb_index_list_len(gb_index* index, int list) {
  IVF_OR_FAIL(ivf, index);
  if (!ivf->lists() || list < 0 || list >= ivf->nlist()) return 0;
  return ivf->lists()->lens()[list];
}
int gb_index_code_size(gb_index* index) {
  IVF_OR_FAIL(ivf, index);
  IVFPQIndex* pq = as_pq(index);
  if (IVFRaBitQIndex* rq = as_rq(index)) return rabitq_code_size(rq->d(), rq->nb_bits());
  return pq ? pq->M() : ((ivf->d() + 3) / 4 * 4) * 4;
}
int gb_index_get_list(gb_index* index, int list, uint8_t* codes, int64_t* ids) {
  IVF_OR_FAIL(ivf, index);
  if (!ivf->lists()) return -1;
  cudaSetDevice(ivf->device());
  std::vector<uint8_t> c;
  std::vector<int64_t> i;
  if (ivf->lists()->download_list(list, &c, &i)) return -1;
  if (codes && !c.empty()) memcpy(codes, c.data(), c.size());
  if (ids && !i.empty()) memcpy(ids, i.data(), i.size() * 8);
  return 0;
}
int gb_index_tombstone(gb_index* index, int list, int pos) {
  IVF_OR_FAIL(ivf, index);
  if (!ivf->lists()) return -1;
  cudaSetDevice(ivf->device());
  return ivf->lists()->tombstone(list, pos, nullptr);
}
int gb_index_coarse_search(gb_index* index, int nq, const float* x, int nprobe, float* out_dis, int64_t* out_ids) {
  IVF_OR_FAIL(ivf, index);
  return ivf->coarse_search_host(nq, x, nprobe, out_dis, out_ids);
}
int gb_index_search_preassigned(gb_index* index, int nq, const float* x, int k, const int64_t* keys,
                                const float* coarse_dis, int nprobe, const char* retrieval_params_json,
                                const uint8_t* del_bitmap, const uint8_t* filter_bitmap, int64_t bitmap_bits,
                                float min_score, float max_score, float* out_scores, int64_t* out_ids) {
  IVF_OR_FAIL(ivf, index);
  SearchContext ctx;
  if (fill_ctx(&ctx, retrieval_params_json, 0, del_bitmap, filter_bitmap, bitmap_bits, min_score, max_score)) return -1;
  return ivf->search_preassigned_host(ctx, nq, x, k, keys, coarse_dis, nprobe, out_scores, out_ids);
}
int gb_index_rabitq_encode(gb_index* index, int64_t n, const float* x, const int64_t* assign, uint8_t* codes) {
  IVFRaBitQIndex* rq = as_rq(index);
  if (!rq) {
    set_last_error("not an IVFRABITQ index");
    return -1;
  }
  return rq->encode_host(x, n, assign, codes);
}
int gb_index_rabitq_query_consts(gb_index* index, int nq, const float* x, const int64_t* keys, int nprobe, int qb,
                                 int centered, float* out) {
  IVFRaBitQIndex* rq = as_rq(index);
  if (!rq) {
    set_last_error("not an IVFRABITQ index");
    return -1;
  }
  return rq->query_consts_host(nq, x, keys, nprobe, qb, centered != 0, out);
}
int gb_index_pq_encode(gb_index* index, int64_t n, const float* x, const int64_t* assign, uint8_t* codes) {
  PQ_OR_FAIL(pq, index);
  return pq->encode_host(x, n, assign, codes);
}

int gb_kmeans(int device, const float* x, int64_t n, int d, int k, int niter, int64_t seed, int spherical,
              int max_points_per_centroid, float* centroids, float* obj) {
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("no CUDA device");
    return -1;
  }
  cudaStream_t st;
  GB_CUDA(cudaStreamCreate(&st));
  int rc = -1;
  {
    Scratch s(st);
    const int dpad = (d + 3) / 4 * 4;
    float* dx = s.alloc_n<float>((size_t)n * dpad);
    float* dc = s.alloc_n<float>((size_t)k * dpad);
    if (dx && dc && cudaMemsetAsync(dx, 0, (size_t)n * dpad * 4, st) == cudaSuccess &&
        cudaMemsetAsync(dc, 0, (size_t)k * dpad * 4, st) == cudaSuccess &&
        cudaMemcpy2DAsync(dx, (size_t)dpad * 4, x, (size_t)d * 4, (size_t)d * 4, n, cudaMemcpyHostToDevice, st) ==
            cudaSuccess) {
      KMeansParams kp;
      kp.niter = niter;
      kp.seed = seed;
      kp.spherical = spherical != 0;
      kp.max_points_per_centroid = max_points_per_centroid;
      std::vector<float> o;
      rc = kmeans_device(dx, dpad, n, d, k, kp, dc, dpad, st, obj ? &o : nullptr);
      if (rc == 0) {
        if (cudaMemcpy2DAsync(centroids, (size_t)d * 4, dc, (size_t)dpad * 4, (size_t)d * 4, k, cudaMemcpyDeviceToHost,
                              st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
          rc = -1;
        if (obj)
          for (size_t i = 0; i < o.size(); i++) obj[i] = o[i];
      }
    }
  }
  cudaStreamSynchronize(st);
  cudaStreamDestroy(st);
  return rc;
}

int gb_kmeans_update(int device, const float* x, int64_t n, int d, int k, const int64_t* assign, float* centroids) {
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("no CUDA device");
    return -1;
  }
  cudaStream_t st = nullptr;
  Scratch s(st);
  const int dpad = (d + 3) / 4 * 4;
  float* dx = s.alloc_n<float>((size_t)n * dpad);
  float* dc = s.alloc_n<float>((size_t)k * dpad);
  int32_t* dperm = s.alloc_n<int32_t>(n);
  int32_t* doff = s.alloc_n<int32_t>(k + 1);
  if (!dx || !dc || !dperm || !doff) return -1;
  std::vector<int32_t> off(k + 1, 0), perm(n), cur(k);
  for (int64_t i = 0; i < n; i++) off[assign[i] + 1]++;
  for (int c = 0; c < k; c++) {
    off[c + 1] += off[c];
    cur[c] = off[c];
  }
  for (int64_t i = 0; i < n; i++) perm[cur[assign[i]]++] = (int32_t)i;
  GB_CUDA(cudaMemsetAsync(dx, 0, (size_t)n * dpad * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dx, (size_t)dpad * 4, x, (size_t)d * 4, (size_t)d * 4, n, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(dperm, perm.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(doff, off.data(), (size_t)(k + 1) * 4, cudaMemcpyHostToDevice, st));
  GB_CUDA(launch_segment_mean(dx, dpad, d, dperm, doff, k, dc, dpad, st));
  GB_CUDA(cudaMemcpy2DAsync(centroids, (size_t)d * 4, dc, (size_t)dpad * 4, (size_t)d * 4, k, cudaMemcpyDeviceToHost,
                            st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int gb_debug_dist_matrix(int device, const float* x, int n, const float* c, int m, int d, int metric, int use_tc,
                         float* out) {
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("no CUDA device");
    return -1;
  }
  cudaStream_t st = nullptr;
  Scratch s(st);
  const int dpad = (d + 3) / 4 * 4;
  const int64_t ldo = (m + 3) / 4 * 4;
  float* dx = s.alloc_n<float>((size_t)n * dpad);
  float* dc = s.alloc_n<float>((size_t)m * dpad);
  float* dout = s.alloc_n<float>((size_t)n * ldo);
  if (!dx || !dc || !dout) return -1;
  GB_CUDA(cudaMemsetAsync(dx, 0, (size_t)n * dpad * 4, st));
  GB_CUDA(cudaMemsetAsync(dc, 0, (size_t)m * dpad * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dx, (size_t)dpad * 4, x, (size_t)d * 4, (size_t)d * 4, n, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpy2DAsync(dc, (size_t)dpad * 4, c, (size_t)d * 4, (size_t)d * 4, m, cudaMemcpyHostToDevice, st));
  if (use_tc) {
    GB_CUDA(launch_dist_matrix_tc(dx, dpad, n, dc, dpad, m, dpad, metric, dout, ldo, st));
  } else {
    GB_CUDA(launch_dist_matrix(dx, dpad, n, dc, dpad, m, dpad, metric, dout, ldo, st));
  }
  GB_CUDA(cudaMemcpy2DAsync(out, (size_t)m * 4, dout, (size_t)ldo * 4, (size_t)m * 4, n, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int gb_merge_partitions_device(int device, const float* dis_dev, const int64_t* ids_dev, int nparts, int nq, int k,
                               int metric, float* out_dis_dev, int64_t* out_ids_dev, void* stream) {
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("no CUDA device");
    return -1;
  }
  return merge_partitions_device(dis_dev, ids_dev, nparts, nq, k, metric, out_dis_dev, out_ids_dev,
                                 static_cast<cudaStream_t>(stream));
}

int gb_merge_partition_keys_device(int device, const unsigned long long* keys_dev, int nparts, int nq, int k, int metric,
                                   float* out_dis_dev, int64_t* out_ids_dev, void* stream) {
  if (cudaSetDevice(device) != cudaSuccess) {
    set_last_error("no CUDA device");
    return -1;
  }
  return merge_partition_keys_device(keys_dev, nparts, nq, k, metric, out_dis_dev, out_ids_dev,
                                     static_cast<cudaStream_t>(stream));
}

}  // extern "C"
