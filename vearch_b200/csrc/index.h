// Host side of the hot path: device-resident raw vectors, inverted lists, and the three index
// models, mirroring the reference's IndexModel plug-in interface
// (index/index_model.h:229-335: Init / Indexing / Add / Search, RetrievalContext,
// RetrievalParameters) so that the engine above it (engine.cc) reads like search/engine.cc +
// vector/vector_manager.cc.  No CPU compute path exists here: every Search/Train/Add call runs
// CUDA kernels and fails if the device is unavailable.
#pragma once
#include <stdio.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <condition_variable>
#include <memory>
#include <atomic>
#include <mutex>
#include <thread>
#include <shared_mutex>
#include <string>
#include <vector>

#include "kernels.h"

namespace gb {

void set_last_error(const std::string& msg);
const char* last_error();
#define GB_CUDA(expr)                                                                              \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      ::gb::set_last_error(std::string(#expr) + ": " + cudaGetErrorString(e__) + " @" __FILE__ ":" + \
                           std::to_string(__LINE__));                                              \
      return -1;                                                                                   \
    }                                                                                              \
  } while (0)

// Stream-ordered scratch allocations released when the object dies.
class Scratch {
 public:
  explicit Scratch(cudaStream_t st) : st_(st) {}
  ~Scratch();
  void* alloc(size_t bytes);  // nullptr on failure (last_error set)
  template <typename T>
  T* alloc_n(size_t n) {
    return static_cast<T*>(alloc(n * sizeof(T)));
  }
  cudaStream_t stream() const { return st_; }

 private:
  cudaStream_t st_;
  std::vector<void*> ptrs_;
};

// MemoryRawVector on device (vector/memory_raw_vector.cc:152-240): append-only fp32 rows kept in
// fixed-size HBM segments, row stride dpad (d rounded up to 4 floats, zero padded).
class RawStore {
 public:
  RawStore(int d, int seg_shift);
  ~RawStore();
  int d() const { return d_; }
  int dpad() const { return dpad_; }
  int64_t size() const { return n_; }
  int seg_shift() const { return seg_shift_; }
  int64_t seg_rows() const { return (int64_t)1 << seg_shift_; }
  int nsegs() const { return (int)segs_.size(); }
  const float* seg(int i) const { return segs_[i].base; }
  const float* const* d_segs() const { return d_segs_; }
  // rows: n x d floats (stride d) on host, or n x dpad (stride ld) on device
  int append_host(const float* x, int64_t n, cudaStream_t st);
  int append_device(const float* x, int64_t ld, int64_t n, cudaStream_t st);
  int update_host(int64_t vid, const float* x, cudaStream_t st);
  int get_host(int64_t vid, float* out) const;
  int get_rows_host(int64_t start, int64_t n, float* out) const;  // n x d, stride d
  // contiguous copy of rows [0, n) (training slab, GetVectorHeader): returns device ptr, owned by `s`
  const float* contiguous(int64_t n, Scratch& s);
  int64_t mem_bytes() const { return phys_bytes_; }  // physical HBM behind the store

 private:
  int ensure(int64_t n_total);
  int new_segment();
  int map_rows(int si, int64_t rows);
  struct Seg {
    float* base = nullptr;
    bool vmm = false;
    size_t va_bytes = 0, mapped = 0, gran = 0;
    std::vector<std::pair<unsigned long long, size_t>> chunks;  // (CUmemGenericAllocationHandle, bytes), in address order
  };
  int d_, dpad_, seg_shift_, device_ = 0;
  int64_t n_ = 0, phys_bytes_ = 0;
  std::vector<Seg> segs_;
  float** d_segs_ = nullptr;  // device array [kMaxSegs]
  static constexpr int kMaxSegs = 65536;
};

// RTInvertIndex / RealTimeMemData on device (index/realtime/realtime_mem_data.{h,cc}): per-list
// growable arrays of fixed-size codes + int64 ids (top bit = tombstone), entries in insertion
// order, length published after the data.
class IvfLists {
 public:
  IvfLists(int nlist, int code_bytes);
  ~IvfLists();
  int nlist() const { return nlist_; }
  int max_len() const { return max_len_; }
  int64_t total() const { return total_; }
  const std::vector<int>& lens() const { return h_len_; }
  uint64_t uid() const { return uid_; }  // distinguishes list sets (reset_index builds a new one)
  ListDirectory directory() const;
  // make room for add[l] more entries in every list; grows by copy (x1.5) when needed
  int reserve(const std::vector<int>& add, cudaStream_t st);
  // device arrays of per-list base pointers (valid after reserve)
  void* const* d_data() const { return d_data_; }
  int64_t* const* d_ids() const { return d_ids_; }
  // account for appended entries and publish the new lengths (after the scatter kernel, same stream)
  int commit(const std::vector<int>& add, cudaStream_t st);
  // tombstone one entry (Update path, realtime_mem_data.cc:298-320)
  int tombstone(int list, int pos, cudaStream_t st);
  // host copies for dump / parity tests
  int download_list(int l, std::vector<uint8_t>* codes, std::vector<int64_t>* ids) const;
  // append position of list l (valid after reserve): where the next entry's code / id goes
  void* list_data(int l) const { return static_cast<char*>(h_data_[l]) + (size_t)h_len_[l] * code_bytes_; }
  int64_t* list_ids(int l) const { return h_ids_[l] + h_len_[l]; }
  int64_t mem_bytes() const { return bytes_; }
  // bytes the lists would occupy packed tightly; compact() re-packs them into one fresh slab and
  // frees every old one (copy-on-grow never reuses the regions it leaves behind).  The caller must
  // exclude concurrent searches; in-flight kernels are drained before the old slabs go.
  int64_t packed_bytes() const;
  int compact(cudaStream_t st);

 private:
  void* slab_alloc(size_t bytes);
  int nlist_, code_bytes_;
  uint64_t uid_;
  std::vector<void*> h_data_;
  std::vector<int64_t*> h_ids_;
  std::vector<int> h_len_, h_cap_;
  void** d_data_ = nullptr;
  int64_t** d_ids_ = nullptr;
  int* d_len_ = nullptr;
  int max_len_ = 0;
  int64_t total_ = 0, bytes_ = 0;
  std::vector<void*> slabs_;
  char* slab_cur_ = nullptr;
  size_t slab_left_ = 0;
};

struct ModelParams {  // index/impl/gamma_index_ivfpq.h:1031-1257, gamma_index_ivfflat.cc:40-196
  int ncentroids = 2048;
  int nprobe = 80;
  int metric = kMetricIP;       // gamma default: InnerProduct
  int nsubvector = 0;           // 0 => d/2 ... see IVFPQIndex::init (gamma_index_ivfpq.cc:122-124)
  int nbits = 8;
  int training_threshold = 0;   // 0 => engine default
  int bucket_init_size = 1000;
  int bucket_max_size = 1280000;
  int opq_nsubvector = 0;       // > 0: OPQ rotation in front of the IVFPQ index (gamma_index_ivfpq.h:1202-1216)
  int nb_bits = 4;              // IVFRABITQ bits per dimension, [1, 9] (gamma_index_ivfrabitq.h:335-537)
  int qb = 4;                   // IVFRABITQ query bits, [0, 8]; 0 = float query
};

struct RetrievalParams {  // gamma_index_ivfpq.cc:233-294, gamma_index_ivfflat.cc:293-340
  int nprobe = -1;
  int metric = -1;  // -1 => index metric
  int recall_num = -1;
  int parallel_on_queries = 1;
  bool brute_force = false;
  int qb = -1;            // IVFRABITQ: query bits for this search; outside [0, 8] => the model's qb
  bool centered = false;  // IVFRABITQ: quantise the query on a grid symmetric around zero
};

struct SearchContext {  // RetrievalContext / SearchCondition (common/gamma_common_data.h:33-121)
  const uint8_t* del_bitmap = nullptr;     // host, bit set => deleted
  const uint8_t* filter_bitmap = nullptr;  // host, bit set => allowed (nullptr => no filter)
  int64_t bitmap_bits = 0;
  float min_score = -3.4028235e38f, max_score = 3.4028235e38f;
  bool search_unindexed_tail = false;  // table.enable_realtime: brute-force the not-yet-indexed vectors too
  RetrievalParams params;
};

class Index {
 public:
  Index(const std::string& type, int d, const ModelParams& mp, int device, int seg_shift);
  virtual ~Index();
  const std::string& type() const { return type_; }
  int d() const { return d_; }
  int device() const { return device_; }
  int metric() const { return mp_.metric; }
  const ModelParams& model_params() const { return mp_; }
  RawStore& store() { return *store_; }
  int64_t indexed_count() const { return indexed_count_; }
  bool trained() const { return trained_; }
  virtual int training_threshold() const { return 0; }

  // AddToStore (vector_manager.cc:455): append raw vectors, host rows n x d
  int add_vectors(const float* x, int64_t n);
  int add_vectors_device(const float* x, int64_t ld, int64_t n);
  // IndexModel::Indexing(): train on the first `num` stored vectors
  virtual int train() { trained_ = true; return 0; }
  // VectorManager::AddRTVecsToIndex (vector_manager.cc:572-702): index all not-yet-indexed rows
  virtual int add_pending(const uint8_t* del_bitmap) { indexed_count_ = store_->size(); return 0; }
  // Engine::Update -> RawVector update + IndexModel::Update (search/engine.cc:774-850;
  // realtime_mem_data.cc:298-320: old entry tombstoned, vector re-appended to its new list)
  virtual int update_vector(int64_t vid, const float* x);
  // IndexModel::Search (index_model.h:296): x = nq x d floats; out = nq x k, unfilled id -1.
  // Returns 0, -1 on error (last_error), -2 if killed.  x/out pointers are host unless *_dev.
  int search(const SearchContext& ctx, int nq, const float* x, int k, float* out_dis, int64_t* out_ids);
  // one H2D -> kernels -> D2H round trip on the calling thread's stream
  int search_direct(const SearchContext& ctx, int nq, const float* x, int k, float* out_dis, int64_t* out_ids);
  // out_keys_dev (optional): the nq x k result keys, (order-preserving score bits << 32) | vid, best first,
  // sentinel padded -- what the multi-GPU merge exchanges (one all-gather instead of scores + ids)
  int search_device(const SearchContext& ctx, int nq, const float* x_dev, int64_t ldx, int k, float* out_dis_dev,
                    int64_t* out_ids_dev, cudaStream_t st, unsigned long long* out_keys_dev = nullptr);
  // forget the trained state and the index structures, keep the raw vectors (Engine::RebuildIndex ->
  // VectorManager::ReCreateVectorIndexes, search/engine.cc:991-1089): the next train() starts over
  virtual int reset_index() { return 0; }
  virtual int64_t index_mem_bytes() const { return 0; }
  // stop the background worker (request coalescer); also run from an atexit hook for objects the host
  // never closed, so no thread of ours is inside the CUDA runtime while it is being torn down
  void quiesce();
  // device time spent in the dominant scan kernel(s) since the last call (ms), for the bench
  // roofline: CUDA events recorded on the launching stream around the scan launches, read here.
  float last_scan_ms();
  std::vector<std::pair<std::string, float>> stage_times();
  void set_time_scan(bool on) { time_scan_ = on; }
  const char* last_scan_kernel() const { return last_scan_kernel_; }
  const char* last_scan_info() const { return last_scan_info_; }  // JSON details of the last scan path (bench)

 protected:
  // GammaFLATIndex::Search (gamma_index_flat.cc:130-370) over rows [0, nrows)
  int flat_search_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                      int64_t nrows, unsigned long long* out_keys, Scratch& s, int64_t row_begin = 0);
  virtual int search_keys_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                              unsigned long long* out_keys, Scratch& s) = 0;
  int upload_bitmaps(const SearchContext& ctx, FilterArgs* f, Scratch& s);

  std::string type_;
  int d_, dpad_, device_;
  ModelParams mp_;
  std::unique_ptr<RawStore> store_;
  int64_t indexed_count_ = 0;
  bool trained_ = false;
  mutable std::shared_mutex mu_;  // searches shared, index mutation exclusive
  // Kernels of a search keep reading the list directory (lengths, base pointers), the centroids and the raw-store
  // segments AFTER the search call released mu_ (device-resident searches are asynchronous).  Every search leaves an
  // event on its stream; whoever mutates those structures takes mu_ exclusively (no new search can enqueue) and then
  // drains the events, so no kernel of an earlier search observes a directory that changes under it.
  void note_search_enqueued(cudaStream_t st);
  void drain_searches();
  std::mutex inflight_mu_;
  std::vector<cudaEvent_t> inflight_;
  std::mutex build_mu_;           // serialises train / add_pending / update_vector (one writer at a time)

  // Request coalescing (SURVEY 8f N-3; reference: the batching thread of its GPU index,
  // index/impl/gpu/gamma_index_ivfflat_gpu.cc:302-396): concurrent small Search calls with the
  // same (k, retrieval params, score window, no bitmaps) are merged into one device batch by a
  // worker thread; callers block until their slice of the result is ready.
  struct CoReq {
    const SearchContext* ctx;
    int nq, k;
    const float* x;
    float* out_dis;
    int64_t* out_ids;
    int rc = 0;
    bool done = false;
    std::string err;
  };
  void coalesce_loop();
  bool coalescable(const SearchContext& ctx, int nq) const;
  std::mutex co_mu_;
  std::condition_variable co_cv_, co_done_cv_;
  std::vector<CoReq*> co_queue_;
  std::thread co_thread_;
  bool co_stop_ = false, co_started_ = false;
  cudaStream_t build_stream_ = nullptr;
  // grow-only cache of multi-GB scratch (list-major score segments): stream-ordered pools re-map
  // such blocks on every search when the caller's stream is the legacy default stream
  void* big_acquire(size_t bytes, cudaStream_t st);
  void big_release(void* p, cudaStream_t st);
  struct BigBuf {
    void* p;
    size_t cap;
    bool busy;
    cudaEvent_t done;
  };
  std::mutex big_mu_;
  std::vector<BigBuf> big_;
  void scan_timer_begin(cudaStream_t st);
  void scan_timer_end(cudaStream_t st);
  // per-stage device times (bench breakdown): CUDA events on the launching stream around each stage of a
  // search while set_time_scan(true); stage_times() sums them per name since the last call
  void stage_begin(const char* name, cudaStream_t st);
  void stage_end(cudaStream_t st);
  struct StageEv {
    const char* name;
    cudaEvent_t e0, e1;
  };
  std::vector<StageEv> stage_events_;
  struct StageScope {
    Index* ix;
    cudaStream_t st;
    StageScope(Index* i, const char* name, cudaStream_t s) : ix(i), st(s) { ix->stage_begin(name, st); }
    ~StageScope() { ix->stage_end(st); }
  };
  std::mutex ev_mu_;
  std::vector<std::pair<cudaEvent_t, cudaEvent_t>> scan_events_;
  bool time_scan_ = false;
  const char* last_scan_kernel_ = "";  // which scan path served the last search (bench roofline label)
  char last_scan_info_[160] = "{}";
};

class FlatIndex : public Index {
 public:
  FlatIndex(int d, const ModelParams& mp, int device, int seg_shift) : Index("FLAT", d, mp, device, seg_shift) {
    trained_ = true;
  }

 protected:
  int search_keys_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                      unsigned long long* out_keys, Scratch& s) override;
};

// k-means on device (faiss Clustering restated; DESIGN.md K6)
struct KMeansParams {
  int niter = 25;
  int64_t seed = 1234;
  bool spherical = false;
  int max_points_per_centroid = 256;
  bool hot_start = false;  // keep the centroids passed in as the initial state (ProductQuantizer::Train_hot_start)
};
int kmeans_device(const float* x, int64_t ldx, int64_t n, int d, int k, const KMeansParams& kp, float* centroids,
                  int64_t ldc, cudaStream_t st, std::vector<float>* obj);

class IVFFlatIndex : public Index {
 public:
  IVFFlatIndex(int d, const ModelParams& mp, int device, int seg_shift, const std::string& type = "IVFFLAT");
  ~IVFFlatIndex() override;
  int training_threshold() const override;
  int train() override;
  int add_pending(const uint8_t* del_bitmap) override;
  int update_vector(int64_t vid, const float* x) override;
  int reset_index() override;
  int64_t index_mem_bytes() const override;
  int nlist() const { return nlist_; }
  // parity hooks: exchange index state with the oracle
  int set_centroids(const float* host, int nlist);  // marks trained
  int get_centroids(float* host) const;
  IvfLists* lists() { return lists_.get(); }
  // quantizer->search (ivfflat.cc:568): top-nprobe lists per query
  int coarse_search_host(int nq, const float* x, int nprobe, float* out_dis, int64_t* out_ids);
  // search_preassigned with caller-provided (keys, coarse_dis): host in/out
  virtual int search_preassigned_host(const SearchContext& ctx, int nq, const float* x, int k, const int64_t* keys,
                                      const float* coarse_dis, int nprobe, float* out_dis, int64_t* out_ids);
  // gamma's own index files (index_io.cu): <dir>/<abs_name>/{ivfflat,ivfpq}.index.  load: the vector
  // store must already hold the vectors the file indexes; *load_num = IndexModel::Load's load_num
  // re-pack the inverted lists into one tight slab (IvfLists::compact); also done automatically after
  // a bulk add_pending when more than half of the slab space is dead
  int compact_lists();
  int mirror_builds() const { return mirror_.builds; }  // test hook
  int dump_gamma(const std::string& dir, const std::string& abs_name);
  int load_gamma(const std::string& dir, const std::string& abs_name, int64_t* load_num);

 protected:
  virtual const char* gamma_file_name() const;
  virtual int dump_gamma_extra(FILE* f) { (void)f; return 0; }
  virtual int load_gamma_extra(FILE* f) { (void)f; return 0; }
  int search_keys_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                      unsigned long long* out_keys, Scratch& s) override;
  int coarse_dev(int nq, const float* xq, int nprobe, int metric, int32_t* probe_ids, float* coarse_dis, Scratch& s);
  virtual int scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                       const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
                       Scratch& s);
  // list-major IVF-Flat scan on the tensor cores (kernels_tc.cu); returns 1 if not applicable
  int scan_listmajor_dev(const FilterArgs& f, int metric, int nq, const float* xq, int k, const int32_t* probe_ids,
                         int nprobe, unsigned long long* out_keys, Scratch& s);
  int assign_dev(const float* x, int64_t ldx, int64_t n, int32_t* assign_dev_out, Scratch& s);
  int resolve_nprobe(const SearchContext& ctx) const;
  virtual int code_bytes() const { return dpad_ * 4; }
  virtual int append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                           const int32_t* d_assign, Scratch& s);
  virtual int train_extra(const float* xtrain, int64_t n, Scratch& s) { (void)xtrain; (void)n; (void)s; return 0; }
  // vector transform in front of the index (OPQ, gamma_index_ivfpq.cc:362-364, 422, 470, 585-590): applied to the
  // training slab (which also trains it), to vectors on their way into the lists and to queries; the raw store
  // and the exact re-rank keep the original vectors.  Default: identity (returns x).
  virtual const float* train_transform(const float* xt, int64_t n, Scratch& s) { (void)n; (void)s; return xt; }
  virtual const float* transform_dev(const float* x, int64_t n, Scratch& s) { (void)n; (void)s; return x; }

  // index rows [vid0, vid0+n) (device pointer x, stride dpad) into the lists
  int index_batch(const float* x, int64_t n, int64_t vid0, const uint8_t* del_bitmap);

  int nlist_;
  float* d_centroids_ = nullptr;  // [nlist][dpad]
  std::unique_ptr<IvfLists> lists_;
  std::vector<uint64_t> vid2pos_;  // vid -> (list << 32 | pos), ~0 = not in a list (vid_bucket_no_pos_)

  // Tensor-core mirror of the lists (IVFFLAT only; kernels_tc.cu): every list once more, pre-split and
  // pre-tiled in the shared-memory operand layout so the list-major kernel is fed by cp.async.bulk.
  // Built by the first list-major search, kept current in place by appends that fit its reserve,
  // rebuilt when a list outgrows it; users hold mirror_rw_ shared from the freshness check until their
  // kernels are enqueued, the rebuilder takes it exclusively and drains the device first.  Skipped
  // (register-staged kernel instead) when HBM is too full for it.
  struct TcMirror {
    float* base = nullptr;
    float* norms = nullptr;
    int64_t* d_tile0 = nullptr;
    int64_t tiles = 0, cap_tiles = 0;
    std::vector<int> lens;        // rows mirrored per list
    std::vector<int> list_tiles;  // tiles reserved per list (a little slack, so appends go in place)
    bool disabled = false;
    int builds = 0;  // full (re)builds so far
  } mirror_;
  // appends keep the mirror current in place while the reserved tiles last; otherwise it goes stale and the
  // next list-major search rebuilds it
  int mirror_append(const float* x, int64_t n, const int32_t* d_list, const int32_t* d_pos, const std::vector<int>& add,
                    cudaStream_t st);
  std::shared_mutex mirror_rw_;
  int ensure_mirror(std::shared_lock<std::shared_mutex>& lk, cudaStream_t st);  // 0 = usable and current
};

class IVFPQIndex : public IVFFlatIndex {
 public:
  IVFPQIndex(int d, const ModelParams& mp, int device, int seg_shift);
  ~IVFPQIndex() override;
  int training_threshold() const override;
  int64_t index_mem_bytes() const override;
  int M() const { return M_; }
  int dsub() const { return dsub_; }
  int set_pq_centroids(const float* host);  // [M][256][dsub]; rebuilds the precomputed table
  int get_pq_centroids(float* host) const;
  int get_precomputed_table(float* host) const;
  int encode_host(const float* x, int64_t n, const int64_t* assign, uint8_t* codes_out);
  int search_preassigned_host(const SearchContext& ctx, int nq, const float* x, int k, const int64_t* keys,
                              const float* coarse_dis, int nprobe, float* out_dis, int64_t* out_ids) override;

 protected:
  int scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
               const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
               Scratch& s) override;
  int code_bytes() const override { return M_; }
  const char* gamma_file_name() const override;

 public:
  int reset_index() override {
    opq_trained_ = false;
    return IVFFlatIndex::reset_index();
  }

 protected:
  int dump_gamma_extra(FILE* f) override;
  int load_gamma_extra(FILE* f) override;
  int append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                   const int32_t* d_assign, Scratch& s) override;
  int train_extra(const float* xtrain, int64_t n, Scratch& s) override;
  int rebuild_table(cudaStream_t st);
  // list-major scan through the tensor-core filter (kernels_pqtc.cu); 1 = not applicable
  int scan_listmajor_pq(const FilterArgs& f, int metric, int nq, const float* xq, int kk, const float* ip,
                        const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* adc_out,
                        bool need_sorted, Scratch& s);

  const float* train_transform(const float* xt, int64_t n, Scratch& s) override;
  const float* transform_dev(const float* x, int64_t n, Scratch& s) override;

  int M_, dsub_;
  float* d_pq_ = nullptr;     // [M][256][dsub]
  float* d_table_ = nullptr;  // [nlist][M][256] (L2 only)
  uint16_t* d_cb16_ = nullptr;  // [M][256][dsub] fp16, pre-scaled (tensor-core filter)
  float* d_cbnrm_ = nullptr;    // [M][256] |pq|^2, then rmax2, sb
  // |r_e|^2 of every list entry (L2), flat with 32-entry aligned list segments: built by the first list-major search
  // after the lists or the codebook changed (lists are append-only: same list set + same lengths = same content)
  struct PqNormCache {
    float* base = nullptr;
    int64_t* d_off = nullptr;
    size_t cap = 0;
    std::vector<int> lens;
    uint64_t lists_uid = 0, pq_gen = 0;
  } pqn_;
  std::mutex pqn_mu_;
  uint64_t pq_gen_ = 1;
  int ensure_pq_norms(cudaStream_t st);
  float* d_opq_ = nullptr;    // [d][dpad] rows of the OPQ rotation A (y = A x); nullptr: no OPQ
  bool opq_trained_ = false;

 public:
  bool has_opq() const { return d_opq_ != nullptr; }
  int set_opq(const float* host_A);        // d x d row-major; marks the rotation trained
  int get_opq(float* host_A) const;
  int apply_opq_host(const float* x, int64_t n, float* out);  // test hook: y = A x through the device path
};

// IVF with RaBitQ codes of the residuals (faiss IndexIVFRaBitQ behind gamma_index_ivfrabitq.{h,cc}); everything but
// the codec and the scan is the IVF-Flat machinery.  Scores: the full nb_bits estimate of every valid entry in the probed
// lists (DESIGN.md section 5b), optionally re-ranked exactly (recall_num).
class IVFRaBitQIndex : public IVFFlatIndex {
 public:
  IVFRaBitQIndex(int d, const ModelParams& mp, int device, int seg_shift);
  int training_threshold() const override;
  int nb_bits() const { return mp_.nb_bits; }
  int encode_host(const float* x, int64_t n, const int64_t* assign, uint8_t* codes_out);
  // test hook: the per-pair constants (nq x nprobe x kRabitqConsts) the scan uses
  int query_consts_host(int nq, const float* x, const int64_t* keys, int nprobe, int qb, bool centered, float* out);
  int resolve_qb(const SearchContext& ctx) const;

 protected:
  int code_bytes() const override { return rabitq_code_size(d_, mp_.nb_bits); }
  const char* gamma_file_name() const override;
  int dump_gamma_extra(FILE* f) override;
  int load_gamma_extra(FILE* f) override;
  int append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                   const int32_t* d_assign, Scratch& s) override;
  int scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
               const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
               Scratch& s) override;
};

// reflector (index/reflector.h:68-80): type name -> index object
Index* create_index(const std::string& type, int d, const ModelParams& mp, int device, int seg_shift);

// cross-partition merge (router semantics, internal/client/client.go:1530-1609) on device:
// in: nparts x nq x k (dis, ids) sorted per partition; out: nq x k, ids = (part << 32) | local id
int merge_partitions_device(const float* dis, const int64_t* ids, int nparts, int nq, int k, int metric, float* out_dis,
                            int64_t* out_ids, cudaStream_t st);
// the same merge straight from the partitions' result keys [nparts][nq][k] (Index::search_device out_keys_dev)
int merge_partition_keys_device(const unsigned long long* keys, int nparts, int nq, int k, int metric, float* out_dis,
                                int64_t* out_ids, cudaStream_t st);

}  // namespace gb
