// SURVEY 8f N-1: gamma's on-disk index files, byte for byte, so a partition dumped by the CPU engine
// loads into this one without retraining (and the other way round).
//
// Layout (little endian; faiss "fourcc" = the four characters in file order), restated from
//   GammaIVFFlatIndex::Dump / Load   index/impl/gamma_index_ivfflat.cc:807-892   <dir>/<name>/ivfflat.index
//   GammaIVFPQIndex::Dump / Load     index/impl/gamma_index_ivfpq.cc:1019-1116   <dir>/<name>/ivfpq.index
//   write_ivf_header, write_index_header, write_direct_map, write_product_quantizer,
//   WriteInvertedLists / ReadInvertedLists                                      index/index_io.cc:15-194
//   faiss::write_index(IndexFlat) (faiss v1.14.1 impl/index_write.cpp; not vendored: restated)
//
//   u32  "IvFl" | "IwPQ"
//   ivf header : index header { i32 d, i64 ntotal, i64 1<<20, i64 1<<20, u8 is_trained, i32 metric (0 = IP, 1 = L2) }
//                u64 nlist, u64 nprobe,
//                quantizer = u32 "IxF2" | "IxFI", index header (ntotal = nlist), u64 nlist*d, nlist*d fp32
//                direct map = u8 type (0 = none), u64 0
//   IwPQ only  : u8 by_residual, u64 code_size, u64 d, u64 M, u64 nbits, u64 M*ksub*dsub, fp32 centroids [M][ksub][dsub]
//   lists      : u32 "ilar", u64 nlist, u64 code_bytes, u32 "full", u64 nlist, u64 sizes[nlist],
//                per non-empty list: codes[size * code_bytes], i64 ids[size] (top bit = tombstone)
//   Iwrq/Iwrr  : RaBitQuantizer { u64 d, u64 code_size, i32 metric, (Iwrr only) u64 nb_bits }, u64 code_size,
//                u8 by_residual, u8 qb   (gamma_index_ivfrabitq.cc:836-951; widths of the faiss members unpinned)
//   IvFl only  : i32 indexed_count (int, gamma_index_ivfflat.cc:828)
//   Iwrq/Iwrr  : i64 indexed_count (int64_t, gamma_index_ivfrabitq.cc:870-877)
// An IndexHNSWFlat coarse quantiser ("IHNf") is read for its centroids (the graph is skipped: the coarse
// search here is exact); Dump always writes the IndexFlat form.  An OPQ block ("LTra") follows the product quantizer when the table has opq.
#include <errno.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <memory>

#include "index.h"

namespace gb {

namespace {

struct FileCloser {
  void operator()(FILE* f) const {
    if (f) fclose(f);
  }
};
using FilePtr = std::unique_ptr<FILE, FileCloser>;

constexpr uint32_t fourcc(const char (&s)[5]) {
  return (uint32_t)(uint8_t)s[0] | (uint32_t)(uint8_t)s[1] << 8 | (uint32_t)(uint8_t)s[2] << 16 |
         (uint32_t)(uint8_t)s[3] << 24;
}

template <class T>
bool wr(FILE* f, const T& v) {
  return fwrite(&v, sizeof(T), 1, f) == 1;
}
template <class T>
bool rd(FILE* f, T* v) {
  return fread(v, sizeof(T), 1, f) == 1;
}
bool wr_bytes(FILE* f, const void* p, size_t n) { return n == 0 || fwrite(p, 1, n, f) == n; }
bool rd_bytes(FILE* f, void* p, size_t n) { return n == 0 || fread(p, 1, n, f) == n; }

// write_index_header (index_io.cc:15-23)
bool wr_index_header(FILE* f, int d, int64_t ntotal, int metric) {
  const int64_t dummy = 1 << 20;
  const uint8_t trained = 1;
  const int32_t mt = metric == kMetricL2 ? 1 : 0;  // faiss::METRIC_INNER_PRODUCT = 0, METRIC_L2 = 1
  return wr<int32_t>(f, d) && wr<int64_t>(f, ntotal) && wr(f, dummy) && wr(f, dummy) && wr(f, trained) && wr(f, mt);
}
struct IndexHeader {
  int32_t d = 0, metric = 0;
  int64_t ntotal = 0;
  uint8_t trained = 0;
};
bool rd_index_header(FILE* f, IndexHeader* h) {
  int64_t dummy;
  if (!(rd(f, &h->d) && rd(f, &h->ntotal) && rd(f, &dummy) && rd(f, &dummy) && rd(f, &h->trained) && rd(f, &h->metric)))
    return false;
  if (h->metric > 1) {  // faiss writes metric_arg for the exotic metrics
    float arg;
    if (!rd(f, &arg)) return false;
  }
  return true;
}

int fail(const std::string& msg) {
  set_last_error(msg);
  return -1;
}

}  // namespace

const char* IVFFlatIndex::gamma_file_name() const { return "ivfflat.index"; }
const char* IVFPQIndex::gamma_file_name() const { return "ivfpq.index"; }
const char* IVFRaBitQIndex::gamma_file_name() const { return "ivfrabitq.index"; }

static uint32_t gamma_fourcc(const std::string& type, int nb_bits) {
  if (type == "IVFFLAT") return fourcc("IvFl");
  if (type == "IVFPQ") return fourcc("IwPQ");
  return nb_bits == 1 ? fourcc("Iwrq") : fourcc("Iwrr");
}

// ---- Dump -----------------------------------------------------------------------------------
int IVFFlatIndex::dump_gamma(const std::string& dir, const std::string& abs_name) {
  if (!trained_) return 0;  // "gamma index is not trained, skip dumping" (ivfflat.cc:808-811)
  std::lock_guard<std::mutex> bg(build_mu_);  // no list mutation while the lists are copied out
  cudaSetDevice(device_);
  const std::string index_dir = dir + "/" + abs_name;
  mkdir(dir.c_str(), 0755);
  if (mkdir(index_dir.c_str(), 0755) && errno != EEXIST) return fail("mkdir error, index dir=" + index_dir);
  const std::string path = index_dir + "/" + gamma_file_name();
  FilePtr fp(fopen(path.c_str(), "wb"));
  FILE* f = fp.get();
  if (!f) return fail("cannot open " + path);
  const bool is_pq = type_ != "IVFFLAT";
  bool ok = wr<uint32_t>(f, gamma_fourcc(type_, mp_.nb_bits));
  // write_ivf_header (index_io.cc:41-47)
  ok = ok && wr_index_header(f, d_, indexed_count_, mp_.metric);
  ok = ok && wr<uint64_t>(f, (uint64_t)nlist_) && wr<uint64_t>(f, (uint64_t)mp_.nprobe);
  std::vector<float> cent((size_t)nlist_ * d_);
  if (get_centroids(cent.data())) return -1;
  ok = ok && wr<uint32_t>(f, mp_.metric == kMetricL2 ? fourcc("IxF2") : fourcc("IxFI"));
  ok = ok && wr_index_header(f, d_, nlist_, mp_.metric);
  ok = ok && wr<uint64_t>(f, (uint64_t)cent.size()) && wr_bytes(f, cent.data(), cent.size() * 4);  // WRITEXBVECTOR
  ok = ok && wr<uint8_t>(f, 0) && wr<uint64_t>(f, 0);                                              // direct map: none
  if (!ok) return fail("write error in " + path);
  if (dump_gamma_extra(f)) return fail("write error in " + path);
  // WriteInvertedLists (index_io.cc:108-141)
  const uint64_t cb = is_pq ? (uint64_t)code_bytes() : (uint64_t)d_ * 4;
  ok = wr<uint32_t>(f, fourcc("ilar")) && wr<uint64_t>(f, (uint64_t)nlist_) && wr<uint64_t>(f, cb) &&
       wr<uint32_t>(f, fourcc("full")) && wr<uint64_t>(f, (uint64_t)nlist_);
  const std::vector<int> lens = lists_->lens();
  for (int l = 0; ok && l < nlist_; l++) ok = wr<uint64_t>(f, (uint64_t)lens[l]);
  std::vector<uint8_t> codes, packed;
  std::vector<int64_t> ids;
  for (int l = 0; ok && l < nlist_; l++) {
    if (lens[l] == 0) continue;
    if (lists_->download_list(l, &codes, &ids)) return -1;
    const size_t n = (size_t)lens[l];
    if (ids.size() < n) return fail("list shrank during dump");
    const uint8_t* src = codes.data();
    if (!is_pq && dpad_ != d_) {  // our rows are padded to a multiple of 4 floats; gamma's are not
      packed.resize(n * cb);
      for (size_t r = 0; r < n; r++) memcpy(packed.data() + r * cb, codes.data() + r * (size_t)dpad_ * 4, cb);
      src = packed.data();
    }
    ok = wr_bytes(f, src, n * cb) && wr_bytes(f, ids.data(), n * 8);
  }
  if (ok && type_ == "IVFFLAT") ok = wr<int32_t>(f, (int32_t)indexed_count_);  // ivfflat.cc:835
  if (ok && type_ == "IVFRABITQ") ok = wr<int64_t>(f, indexed_count_);         // ivfrabitq.cc:870-877
  if (!ok || fflush(f)) return fail("write error in " + path);
  return 0;
}

int IVFPQIndex::dump_gamma_extra(FILE* f) {
  std::vector<float> pq((size_t)M_ * 256 * dsub_);
  if (get_pq_centroids(pq.data())) return -1;
  // by_residual, code_size, write_product_quantizer (ivfpq.cc:1037-1039, index_io.cc:92-98)
  bool ok = wr<uint8_t>(f, 1) && wr<uint64_t>(f, (uint64_t)M_) && wr<uint64_t>(f, (uint64_t)d_) &&
            wr<uint64_t>(f, (uint64_t)M_) && wr<uint64_t>(f, 8) && wr<uint64_t>(f, (uint64_t)pq.size()) &&
            wr_bytes(f, pq.data(), pq.size() * 4);
  if (ok && has_opq()) {  // write_opq (index_io.cc:230-246): "LTra", have_bias, A, b, d_in, d_out, is_trained
    std::vector<float> A((size_t)d_ * d_);
    if (get_opq(A.data())) return -1;
    ok = wr<uint32_t>(f, fourcc("LTra")) && wr<uint8_t>(f, 0) && wr<uint64_t>(f, (uint64_t)A.size()) &&
         wr_bytes(f, A.data(), A.size() * 4) && wr<uint64_t>(f, 0) && wr<int32_t>(f, d_) && wr<int32_t>(f, d_) &&
         wr<uint8_t>(f, 1);
  }
  return ok ? 0 : -1;
}

// ---- Load -----------------------------------------------------------------------------------
int IVFFlatIndex::load_gamma(const std::string& dir, const std::string& abs_name, int64_t* load_num) {
  *load_num = 0;
  const std::string path = dir + "/" + abs_name + "/" + gamma_file_name();
  FilePtr fp(fopen(path.c_str(), "rb"));
  FILE* f = fp.get();
  if (!f) return 0;  // "isn't existed, skip loading": it should train again after load (ivfflat.cc:846-850)
  std::lock_guard<std::mutex> bg(build_mu_);
  cudaSetDevice(device_);
  if (lists_ && lists_->total() > 0) return fail("load into a non-empty index");
  const bool is_pq = type_ != "IVFFLAT";
  uint32_t h = 0;
  if (!rd(f, &h) || h != gamma_fourcc(type_, mp_.nb_bits)) return fail("bad magic in " + path);
  IndexHeader ih, qh;
  uint64_t nlist = 0, nprobe = 0, n = 0;
  if (!rd_index_header(f, &ih) || !rd(f, &nlist) || !rd(f, &nprobe)) return fail("truncated ivf header in " + path);
  if (ih.d != d_ || (int64_t)nlist != nlist_)
    return fail("index file does not match the table: d=" + std::to_string(ih.d) + " nlist=" + std::to_string(nlist));
  if ((ih.metric == 1 ? kMetricL2 : kMetricIP) != mp_.metric) return fail("index file metric differs from the table's");
  if (!rd(f, &h)) return fail("truncated quantizer in " + path);
  if (h == fourcc("IHNf")) {
    // IndexHNSWFlat coarse quantizer (quantizer_type 1, gamma_index_ivfflat.cc:252-263): index header,
    // the HNSW graph (write_hnsw, index_io.cc:196-212: five vectors, five ints), then the IndexFlat that
    // stores the centroids.  The graph only approximates "nearest centroids"; this engine finds them
    // exactly with one dense tensor-core contraction, so the graph is skipped and the centroids are kept.
    IndexHeader hh;
    if (!rd_index_header(f, &hh)) return fail("truncated HNSW quantizer in " + path);
    const size_t elem[5] = {8, 4, 4, 8, 4};  // assign_probas, cum_nneighbor_per_level, levels, offsets, neighbors
    for (size_t e : elem) {
      uint64_t cnt = 0;
      if (!rd(f, &cnt) || cnt > ((uint64_t)1 << 40) || fseek(f, (long)(cnt * e), SEEK_CUR)) return fail("bad HNSW graph in " + path);
    }
    int32_t scalars[5];  // entry_point, max_level, efConstruction, efSearch, (deprecated) upper_beam
    if (!rd_bytes(f, scalars, sizeof scalars) || !rd(f, &h)) return fail("truncated HNSW quantizer in " + path);
  }
  if (h != fourcc("IxF2") && h != fourcc("IxFI") && h != fourcc("IxFl"))
    return fail("unsupported coarse quantizer in " + path + " (IndexFlat, or IndexHNSWFlat over IndexFlat)");
  if (!rd_index_header(f, &qh) || !rd(f, &n) || qh.d != d_ || qh.ntotal != nlist_ || n != (uint64_t)nlist_ * d_)
    return fail("bad quantizer in " + path);
  std::vector<float> cent((size_t)nlist_ * d_);
  if (!rd_bytes(f, cent.data(), cent.size() * 4)) return fail("truncated quantizer in " + path);
  uint8_t dm_type = 0;
  if (!rd(f, &dm_type) || !rd(f, &n)) return fail("truncated direct map in " + path);
  if (dm_type != 0 || n != 0) return fail("direct maps are not supported");  // gamma never maintains one
  if (set_centroids(cent.data(), nlist_)) return -1;
  if (load_gamma_extra(f)) return -1;
  // ReadInvertedLists (index_io.cc:143-194)
  uint32_t lt = 0;
  uint64_t nb = 0, cb = 0, ns = 0;
  if (!rd(f, &h) || !rd(f, &nb) || !rd(f, &cb) || !rd(f, &lt) || h != fourcc("ilar") || lt != fourcc("full"))
    return fail("bad inverted-list header in " + path);
  const uint64_t want_cb = is_pq ? (uint64_t)code_bytes() : (uint64_t)d_ * 4;
  if (nb != (uint64_t)nlist_ || cb != want_cb) {
    // kIndexError: "unsupported inverted list format, it need rebuilding!" (ivfflat.cc:866-869)
    indexed_count_ = 0;
    return 0;
  }
  if (!rd(f, &ns) || ns != nb) return fail("bad inverted-list sizes in " + path);
  std::vector<uint64_t> sizes(nlist_);
  if (!rd_bytes(f, sizes.data(), sizes.size() * 8)) return fail("truncated inverted-list sizes in " + path);
  std::vector<int> add(nlist_);
  for (int l = 0; l < nlist_; l++) {
    if (sizes[l] > (uint64_t)INT32_MAX) return fail("inverted list too long");
    add[l] = (int)sizes[l];
  }
  cudaStream_t st = build_stream_;
  {
    std::unique_lock<std::shared_mutex> lk(mu_);
    if (lists_->reserve(add, st)) return -1;
  }
  std::vector<uint8_t> codes, padded;
  std::vector<int64_t> ids;
  int64_t live = 0, max_vid = -1;
  std::vector<uint64_t> v2p;  // vid_bucket_no_pos_, installed only if the whole file loads
  const size_t my_cb = (size_t)code_bytes();
  for (int l = 0; l < nlist_; l++) {
    const size_t len = sizes[l];
    if (!len) continue;
    codes.resize(len * cb);
    ids.resize(len);
    if (!rd_bytes(f, codes.data(), codes.size()) || !rd_bytes(f, ids.data(), len * 8)) return fail("truncated list in " + path);
    const uint8_t* src = codes.data();
    if (my_cb != cb) {  // IVF-Flat with d % 4 != 0: pad rows to our stride
      padded.assign(len * my_cb, 0);
      for (size_t r = 0; r < len; r++) memcpy(padded.data() + r * my_cb, codes.data() + r * cb, cb);
      src = padded.data();
    }
    GB_CUDA(cudaMemcpyAsync(lists_->list_data(l), src, len * my_cb, cudaMemcpyHostToDevice, st));
    GB_CUDA(cudaMemcpyAsync(lists_->list_ids(l), ids.data(), len * 8, cudaMemcpyHostToDevice, st));
    GB_CUDA(cudaStreamSynchronize(st));  // the staging vectors are reused by the next list
    for (size_t pos = 0; pos < len; pos++) {
      const int64_t id = ids[pos];
      if (id < 0) continue;             // deleted_nums_[bno]++ (index_io.cc:178-181)
      live++;
      max_vid = std::max(max_vid, id);
      if ((size_t)id >= v2p.size()) v2p.resize(std::max<size_t>((size_t)id + 1, v2p.size() * 2), ~(uint64_t)0);
      v2p[id] = (uint64_t)l << 32 | (uint64_t)pos;
    }
  }
  int64_t indexed = live;  // IwPQ: ReadInvertedLists' running count (total - tombstones)
  if (type_ == "IVFFLAT") {
    int32_t cnt = 0;
    if (!rd(f, &cnt) || cnt < 0) return fail("invalid indexed count in " + path);  // ivfflat.cc:871-878
    indexed = cnt;
  } else if (type_ == "IVFRABITQ") {
    int64_t cnt = 0;
    if (!rd(f, &cnt) || cnt < 0) return fail("invalid indexed count in " + path);  // ivfrabitq.cc:928-936
    indexed = cnt;
  }
  if (indexed > store_->size() || max_vid >= store_->size())
    return fail("index file covers " + std::to_string(std::max(indexed, max_vid + 1)) + " vectors, the vector store holds " +
                std::to_string(store_->size()));
  {  // publish: nothing above this point changed what a search can see
    std::unique_lock<std::shared_mutex> lk(mu_);
    if (lists_->commit(add, st)) return -1;
  }
  GB_CUDA(cudaStreamSynchronize(st));
  vid2pos_.swap(v2p);
  indexed_count_ = indexed;
  *load_num = indexed;
  return 0;
}

int IVFPQIndex::load_gamma_extra(FILE* f) {
  uint8_t by_residual = 0;
  uint64_t code_size = 0, d = 0, M = 0, nbits = 0, n = 0;
  if (!rd(f, &by_residual) || !rd(f, &code_size) || !rd(f, &d) || !rd(f, &M) || !rd(f, &nbits) || !rd(f, &n))
    return fail("truncated product quantizer");
  if (!by_residual) return fail("by_residual = false is not supported");
  if (d != (uint64_t)d_ || M != (uint64_t)M_ || nbits != 8 || code_size != (uint64_t)M_ || n != (uint64_t)M_ * 256 * dsub_)
    return fail("product quantizer does not match the table: d=" + std::to_string(d) + " M=" + std::to_string(M) +
                " nbits=" + std::to_string(nbits));
  std::vector<float> pq((size_t)n);
  if (!rd_bytes(f, pq.data(), pq.size() * 4)) return fail("truncated product quantizer");
  if (has_opq()) {  // read_opq (index_io.cc:248-270); whether the block is there is decided by the table's params
    uint32_t h = 0;
    uint8_t have_bias = 0, trained = 0;
    uint64_t na = 0, nb = 0;
    int32_t din = 0, dout = 0;
    if (!rd(f, &h) || h != fourcc("LTra") || !rd(f, &have_bias) || !rd(f, &na) || na != (uint64_t)d_ * d_)
      return fail("bad OPQ block (table has opq, file does not match)");
    std::vector<float> A((size_t)na);
    if (!rd_bytes(f, A.data(), A.size() * 4) || !rd(f, &nb) || fseek(f, (long)(nb * 4), SEEK_CUR) || !rd(f, &din) ||
        !rd(f, &dout) || !rd(f, &trained) || din != d_ || dout != d_ || have_bias)
      return fail("bad OPQ block");
    if (set_opq(A.data())) return -1;
  }
  return set_pq_centroids(pq.data());  // also recomputes the precomputed table (ivfpq.cc:1093-1095)
}

// RaBitQuantizer block, code_size, by_residual, qb (gamma_index_ivfrabitq.cc:836-951, index_io.cc:269-295)
int IVFRaBitQIndex::dump_gamma_extra(FILE* f) {
  const uint64_t cs = (uint64_t)code_bytes();
  bool ok = wr<uint64_t>(f, (uint64_t)d_) && wr<uint64_t>(f, cs) && wr<int32_t>(f, mp_.metric == kMetricL2 ? 1 : 0);
  if (mp_.nb_bits > 1) ok = ok && wr<uint64_t>(f, (uint64_t)mp_.nb_bits);
  ok = ok && wr<uint64_t>(f, cs) && wr<uint8_t>(f, 1) && wr<uint8_t>(f, (uint8_t)mp_.qb);
  return ok ? 0 : -1;
}

int IVFRaBitQIndex::load_gamma_extra(FILE* f) {
  uint64_t d = 0, cs = 0, nb = 1, cs2 = 0;
  int32_t mt = 0;
  uint8_t by_residual = 0, qb = 0;
  if (!rd(f, &d) || !rd(f, &cs) || !rd(f, &mt) || (mp_.nb_bits > 1 && !rd(f, &nb)) || !rd(f, &cs2) ||
      !rd(f, &by_residual) || !rd(f, &qb))
    return fail("truncated RaBitQ quantizer");
  if (!by_residual) return fail("by_residual = false is not supported");
  if (d != (uint64_t)d_ || nb != (uint64_t)mp_.nb_bits || (mt == 1 ? kMetricL2 : kMetricIP) != mp_.metric)
    return fail("RaBitQ quantizer does not match the table: d=" + std::to_string(d) + " nb_bits=" + std::to_string(nb));
  if (cs != (uint64_t)code_bytes() || cs2 != cs)
    return fail("RaBitQ code_size " + std::to_string(cs) + " is inconsistent with d=" + std::to_string(d) +
                " nb_bits=" + std::to_string(nb) + " (expected " + std::to_string(code_bytes()) + ")");
  if (qb > 8) return fail("invalid qb =" + std::to_string(qb) + " should be integer in [0, 8]");
  mp_.qb = qb;
  return 0;
}

}  // namespace gb
