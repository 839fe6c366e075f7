// Engine (see engine.h).  Reference call sites cited inline.
#include "engine.h"

#include <float.h>
#include <stdio.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <fstream>
#include <map>

#include "json.h"
#include "params.h"
#include "wire.h"

namespace gb {

std::string Status::ToString() const {  // util/status.cc:43-100
  const char* type = "";
  switch (code) {
    case kOk: return "OK";
    case kNotFound: type = "NotFound: "; break;
    case kIndexError: type = "IndexError: "; break;
    case kNotSupported: type = "Not implemented: "; break;
    case kInvalidArgument: type = "Invalid argument: "; break;
    case kIOError: type = "IO error: "; break;
    case kBusy: type = "Resource busy: "; break;
    case kTimedOut: type = "Operation timed out: "; break;
    case kCanceled: type = "Operation canceled: "; break;
    case kMemoryExceeded: type = "Memory exceed limit: "; break;
    default: type = "Unknown code: "; break;
  }
  return std::string(type) + msg;
}

// ---- vearchpb.SearchRequest (router_grpc.proto:168-191; request.cc:17-91) --------------------
static bool parse_filter(const PbField& f, bool is_term, SearchRequestPB::Filter* fl) {
  fl->is_term = is_term;
  PbReader v(f.data, f.len);
  PbField vf;
  while (v.next(&vf)) {
    if (vf.num == 1 && vf.wire == 2) fl->field.assign(reinterpret_cast<const char*>(vf.data), vf.len);
    if (vf.num == 2 && vf.wire == 2) fl->lower.assign(reinterpret_cast<const char*>(vf.data), vf.len);
    if (is_term) {
      if (vf.num == 3 && vf.wire == 0) fl->is_union = (int)vf.val;
    } else {
      if (vf.num == 3 && vf.wire == 2) fl->upper.assign(reinterpret_cast<const char*>(vf.data), vf.len);
      if (vf.num == 4 && vf.wire == 0) fl->include_lower = vf.val != 0;
      if (vf.num == 5 && vf.wire == 0) fl->include_upper = vf.val != 0;
      if (vf.num == 6 && vf.wire == 0) fl->is_union = (int)vf.val;
    }
  }
  return !v.error();
}

bool QueryRequestPB::parse(const uint8_t* data, size_t len) {
  PbReader r(data, len);
  PbField f;
  while (r.next(&f)) {
    switch (f.num) {
      case 2:
        if (f.wire == 2) document_ids.emplace_back(reinterpret_cast<const char*>(f.data), f.len);
        break;
      case 3: partition_id = (int)f.val; break;
      case 5:
      case 6: {
        if (f.wire != 2) break;
        SearchRequestPB::Filter fl;
        if (!parse_filter(f, f.num == 6, &fl)) return false;
        filters.push_back(std::move(fl));
        break;
      }
      case 7:
        if (f.wire == 2) fields.emplace_back(reinterpret_cast<const char*>(f.data), f.len);
        break;
      case 9: limit = (int)f.val; break;
      case 15: filter_operator = (int)f.val; break;
      case 17: offset = (int)f.val; break;
      default: break;
    }
  }
  return !r.error();
}

bool SearchRequestPB::parse(const uint8_t* data, size_t len) {
  PbReader r(data, len);
  PbField f;
  while (r.next(&f)) {
    switch (f.num) {
      case 1: {  // RequestHead: only params (field 7, map<string,string>) matter
        if (f.wire != 2) break;
        PbReader h(f.data, f.len);
        PbField hf;
        while (h.next(&hf)) {
          if (hf.num != 7 || hf.wire != 2) continue;
          PbReader e(hf.data, hf.len);
          PbField ef;
          std::string k, v;
          while (e.next(&ef)) {
            if (ef.wire != 2) continue;
            if (ef.num == 1) k.assign(reinterpret_cast<const char*>(ef.data), ef.len);
            if (ef.num == 2) v.assign(reinterpret_cast<const char*>(ef.data), ef.len);
          }
          if (k == "request_id") request_id = v;
          if (k == "partition_id") partition_id = atoi(v.c_str());
        }
        if (h.error()) return false;
        break;
      }
      case 2: req_num = (int)f.val; break;
      case 3: topn = (int)f.val; break;
      case 4: brute_force_search = (int)f.val; break;
      case 5: {  // VectorQuery
        if (f.wire != 2) break;
        VecQuery q;
        PbReader v(f.data, f.len);
        PbField vf;
        while (v.next(&vf)) {
          if (vf.num == 1 && vf.wire == 2) q.name.assign(reinterpret_cast<const char*>(vf.data), vf.len);
          if (vf.num == 2 && vf.wire == 2) q.value.assign(reinterpret_cast<const char*>(vf.data), vf.len);
          if (vf.num == 3 && vf.wire == 1) q.min_score = pb_double(vf.val), q.has_min = true;
          if (vf.num == 4 && vf.wire == 1) q.max_score = pb_double(vf.val), q.has_max = true;
          if (vf.num == 6 && vf.wire == 2) q.index_type.assign(reinterpret_cast<const char*>(vf.data), vf.len);
        }
        if (v.error()) return false;
        vec_fields.push_back(std::move(q));
        break;
      }
      case 6:
        if (f.wire == 2) fields.emplace_back(reinterpret_cast<const char*>(f.data), f.len);
        break;
      case 7:
      case 8: {
        if (f.wire != 2) break;
        Filter fl;
        if (!parse_filter(f, f.num == 8, &fl)) return false;
        (fl.is_term ? n_term_filters : n_range_filters)++;
        filters.push_back(std::move(fl));
        break;
      }
      case 9:
        if (f.wire == 2) index_params.assign(reinterpret_cast<const char*>(f.data), f.len);
        break;
      case 10: multi_vector_rank = (int)f.val; break;
      case 15:
        if (f.wire == 2) ranker.assign(reinterpret_cast<const char*>(f.data), f.len);
        break;
      case 11: l2_sqrt = f.val != 0; break;
      case 16: trace = f.val != 0; break;
      case 17: filter_operator = (int)f.val; break;
      case 20: offset = (int)f.val; break;
      default: break;  // unknown / unused fields are skipped
    }
  }
  return !r.error();
}

// ---- kill switch ---------------------------------------------------------------------------
static std::mutex g_kill_mu;
static std::map<std::pair<std::string, int>, int> g_killed;
void Engine::SetKill(const std::string& request_id, int partition_id, int reason) {
  std::lock_guard<std::mutex> g(g_kill_mu);
  g_killed[{request_id, partition_id}] = reason;
}
void Engine::ClearKill(const std::string& request_id, int partition_id) {
  std::lock_guard<std::mutex> g(g_kill_mu);
  g_killed.erase({request_id, partition_id});
}
bool Engine::IsKilled(const std::string& request_id, int partition_id) {
  if (request_id.empty()) return false;
  std::lock_guard<std::mutex> g(g_kill_mu);
  return g_killed.count({request_id, partition_id}) != 0;
}

// ---- admission control (search/engine.cc:47-119) ----------------------------------------------
static int read_proc_int(const char* path) {  // the reference popen()s `cat <path>`; same number, no shell
  int v = -1;
  if (FILE* fp = fopen(path, "r")) {
    if (fscanf(fp, "%d", &v) != 1) v = -1;
    fclose(fp);
  }
  return v;
}
RequestConcurrentController& RequestConcurrentController::GetInstance() {
  static RequestConcurrentController instance;
  return instance;
}
RequestConcurrentController::RequestConcurrentController() {
  const int threads_max = read_proc_int("/proc/sys/kernel/threads-max");
  const int max_map_count = read_proc_int("/proc/sys/vm/max_map_count");
  const int pid_max = read_proc_int("/proc/sys/kernel/pid_max");
  max_threads_ = std::min(std::min(threads_max, pid_max), max_map_count / 2);
  const int host_threads = std::max(1u, std::thread::hardware_concurrency());
  system_threshold_ = (int)((max_threads_ * 0.5) / (host_threads + 1));
  if (system_threshold_ <= 0) system_threshold_ = 1;  // the reference aborts (LOG(FATAL)); a library must not
  concurrent_threshold_ = system_threshold_;
  if (const char* e = getenv("GAMMA_CONCURRENT_THRESHOLD")) set_threshold(atoi(e));
}
void RequestConcurrentController::set_threshold(int t) { concurrent_threshold_ = t > 0 ? t : system_threshold_; }
bool RequestConcurrentController::Acquire(int req_num) {
  const int num = cur_concurrent_num_.fetch_add(req_num);
  return num < concurrent_threshold_;
}
void RequestConcurrentController::Release(int req_num) { cur_concurrent_num_.fetch_sub(req_num); }
namespace {
struct AdmissionGuard {  // every return path of Engine::Search releases what it acquired
  int n;
  bool permit;
  explicit AdmissionGuard(int req_num) : n(req_num), permit(RequestConcurrentController::GetInstance().Acquire(req_num)) {}
  ~AdmissionGuard() { RequestConcurrentController::GetInstance().Release(n); }
};
}  // namespace

// ---------------------------------------------------------------------------------------------
Engine::Engine(const std::string& path, const std::string& space_name, int device)
    : path_(path), space_name_(space_name), device_(device) {}

namespace {
struct LiveEngines {
  std::mutex mu;
  std::vector<Engine*> all;
};
LiveEngines& live_engines() {
  static LiveEngines* s = new LiveEngines;  // leaked on purpose
  return *s;
}
void quiesce_all_engines() {
  std::vector<Engine*> v;
  {
    std::lock_guard<std::mutex> g(live_engines().mu);
    v = live_engines().all;
  }
  for (Engine* e : v) e->quiesce();
}
}  // namespace

void Engine::quiesce() {
  int st = indexing_state_.load();
  if (st != 0) indexing_state_.store(3);
  idx_cv_.notify_all();
  if (indexing_thread_.joinable()) indexing_thread_.join();
}

Engine::~Engine() {
  // Close: stop the indexing thread (search/engine.cc Engine::~Engine / Close)
  {
    std::lock_guard<std::mutex> g(live_engines().mu);
    auto& a = live_engines().all;
    a.erase(std::remove(a.begin(), a.end(), this), a.end());
  }
  quiesce();
  cudaSetDevice(device_);
  index_.reset();
}

// Engine::CreateTable (search/engine.cc:582-690) + TableInfo::Deserialize (table.cc:30-157) +
// VectorManager::CreateVectorTable (vector_manager.cc:343-453)
Status Engine::CreateTable(const uint8_t* fb, size_t len) {
  std::unique_lock<std::shared_mutex> lk(mu_);
  if (created_table_) return Status::Make(kInvalidArgument, "table is created");
  FbTable t = FbTable::root(fb, len);
  if (!t.ok()) return Status::Make(kInvalidArgument, "table deserialize error");
  table_name_ = t.str(0);
  fields_.clear();
  field_idx_.clear();
  bool has_id = false;
  for (size_t i = 0; i < t.vec_len(1); i++) {
    FbTable f = t.vec_table(1, i);
    FieldDef fd{f.str(0), (int)f.scalar<int8_t>(1, 0), f.scalar<uint8_t>(2, 0) != 0};
    if (fd.name == "_id") has_id = true;
    field_idx_[fd.name] = (int)fields_.size();
    fields_.push_back(fd);
  }
  if (!has_id) {  // the key field always exists (table/table.cc)
    field_idx_["_id"] = (int)fields_.size();
    fields_.push_back({"_id", DT_STRING, false});
  }
  values_.assign(fields_.size(), {});
  sidx_.assign(fields_.size(), ScalarIndex());
  for (size_t fi = 0; fi < fields_.size(); fi++) sidx_[fi].built = fields_[fi].indexed;
  size_t nvec = t.vec_len(2);
  if (nvec == 0) return Status::Make(kInvalidArgument, space_name_ + " table has no vector field");
  FbTable v = t.vec_table(2, 0);
  vec_name_ = v.str(0);
  dim_ = v.scalar<int32_t>(3, 0);
  if (dim_ <= 0) return Status::Make(kInvalidArgument, "invalid vector dimension");
  std::string table_index_params = t.str(4);
  refresh_interval_ = t.scalar<int32_t>(5, 1000);
  enable_id_cache_ = t.scalar<uint8_t>(6, 0) != 0;
  enable_realtime_ = t.scalar<uint8_t>(7, 0) != 0;
  training_threshold_ = 0;
  {
    JsonValue jv;
    int tt = 0;
    if (!table_index_params.empty() && JsonParser::parse(table_index_params, &jv) && jv.get_int("training_threshold", &tt) &&
        tt > 0)
      training_threshold_ = tt;
  }
  // index type of the vector field: first entry of `indexes` with a matching field_name
  // (vector_manager.cc:365-373)
  index_type_.clear();
  for (size_t i = 0; i < t.vec_len(8); i++) {
    FbTable ix = t.vec_table(8, i);
    if (ix.str(2) == vec_name_ && !ix.str(1).empty()) {
      index_type_ = ix.str(1);
      index_params_ = ix.str(4);
      break;
    }
  }
  if (index_type_.empty()) return Status::Make(kInvalidArgument, vec_name_ + " index type is empty");
  ModelParams mp;
  std::string err;
  if (!parse_model_params(index_params_, &mp, &err)) return Status::Make(kInvalidArgument, err);
  if (table_index_params.empty() && mp.training_threshold > training_threshold_)
    training_threshold_ = mp.training_threshold;  // table.cc:143-150
  if (training_threshold_ > 0) mp.training_threshold = training_threshold_;
  Index* idx = create_index(index_type_, dim_, mp, device_, 20);
  if (!idx) return Status::Make(index_type_ == "FLAT" || index_type_ == "IVFFLAT" || index_type_ == "IVFPQ" ||
                                        index_type_ == "IVFRABITQ"
                                    ? kInvalidArgument
                                    : kNotSupported,
                                last_error());
  index_.reset(idx);
  extra_.clear();
  for (size_t vi = 1; vi < nvec; vi++) {  // the other vector fields: same rules, their own index each
    FbTable ev = t.vec_table(2, vi);
    VecField vf;
    vf.name = ev.str(0);
    vf.dim = ev.scalar<int32_t>(3, 0);
    if (vf.dim <= 0 || vf.name.empty() || vf.name == vec_name_) return Status::Make(kInvalidArgument, "invalid vector field");
    for (size_t i = 0; i < t.vec_len(8); i++) {
      FbTable ix = t.vec_table(8, i);
      if (ix.str(2) == vf.name && !ix.str(1).empty()) {
        vf.index_type = ix.str(1);
        vf.index_params = ix.str(4);
        break;
      }
    }
    if (vf.index_type.empty()) return Status::Make(kInvalidArgument, vf.name + " index type is empty");
    ModelParams emp;
    if (!parse_model_params(vf.index_params, &emp, &err)) return Status::Make(kInvalidArgument, err);
    if (training_threshold_ > 0) emp.training_threshold = training_threshold_;
    Index* eidx = create_index(vf.index_type, vf.dim, emp, device_, 20);
    if (!eidx) return Status::Make(kInvalidArgument, last_error());
    vf.index.reset(eidx);
    extra_.push_back(std::move(vf));
  }
  {  // registered after the index (and so after CUDA start-up): at exit the engine's thread stops first
    std::lock_guard<std::mutex> g(live_engines().mu);
    static bool hooked = (atexit(quiesce_all_engines), true);
    (void)hooked;
    live_engines().all.push_back(this);
  }
  if (training_threshold_ <= 0) training_threshold_ = index_->training_threshold();
  created_table_ = true;
  // <path>/<table>.schema, as the reference writes it (engine.cc:676-684)
  if (!path_.empty()) {
    mkdir(path_.c_str(), 0755);
    std::ofstream f(path_ + "/" + table_name_ + ".schema", std::ios::binary);
    if (f) f.write(reinterpret_cast<const char*>(fb), (std::streamsize)len);
  }
  return Status::OK();
}

Index* Engine::index_of(const std::string& vec_name, int* dim) {
  if (vec_name == vec_name_) {
    *dim = dim_;
    return index_.get();
  }
  for (auto& e : extra_)
    if (e.name == vec_name) {
      *dim = e.dim;
      return e.index.get();
    }
  return nullptr;
}

int Engine::flush_pending_locked() {
  if (pending_n_ == 0) return 0;
  // Row i of every vector field must stay document i: a field is appended only while its store is as long as the
  // primary one was when this flush began, so a retry after a partial failure appends exactly the missing fields,
  // and the pending buffers are dropped only when every field has taken its rows.
  const int64_t base = index_->store().size();
  for (auto& e : extra_) {
    if (e.index->store().size() == base + pending_n_) continue;  // taken by an earlier, partially failed flush
    if (e.index->store().size() != base || (int64_t)e.pending.size() != (int64_t)pending_n_ * e.dim) {
      set_last_error("vector fields out of step (field " + e.name + ")");
      return -1;
    }
    if (e.index->add_vectors(e.pending.data(), pending_n_)) return -1;
  }
  int rc = index_->add_vectors(pending_.data(), pending_n_);
  if (rc) return rc;
  for (auto& e : extra_) e.pending.clear();
  pending_.clear();
  pending_n_ = 0;
  return 0;
}

// Engine::AddOrUpdate (search/engine.cc:691-772) + Doc::Deserialize (doc.cc:43-76)
int Engine::AddOrUpdate(const uint8_t* fb, size_t len) {
  if (!created_table_) return -1;
  FbTable d = FbTable::root(fb, len);
  if (!d.ok()) return -3;
  std::string key;
  std::vector<DocField> table_fields;
  const uint8_t* vec = nullptr;
  size_t vec_len = 0;
  bool has_vec = false;
  std::vector<std::pair<const uint8_t*, size_t>> evec(extra_.size(), {nullptr, 0});
  for (size_t i = 0; i < d.vec_len(0); i++) {
    FbTable f = d.vec_table(0, i);
    DocField df;
    df.name = f.str(0);
    const uint8_t* p = nullptr;
    size_t n = 0;
    f.bytes(1, &p, &n);
    df.data_type = f.scalar<int8_t>(2, 0);
    if (df.name == "_id") key.assign(reinterpret_cast<const char*>(p), n);
    if (df.data_type == DT_VECTOR) {
      if (df.name == vec_name_) {
        vec = p;
        vec_len = n;
        has_vec = true;
      }
      for (size_t ei = 0; ei < extra_.size(); ei++)
        if (df.name == extra_[ei].name) evec[ei] = {p, n};
    } else {
      if (!field_idx_.count(df.name)) continue;  // "Unknown field" (doc.cc:66-69)
      df.value.assign(reinterpret_cast<const char*>(p), n);
      table_fields.push_back(std::move(df));
    }
  }
  std::unique_lock<std::shared_mutex> lk(mu_);
  auto it = key2docid_.find(key);
  int docid = it == key2docid_.end() ? -1 : it->second;
  if (docid != -1 && docid < max_docid_) {  // Update (engine.cc:703-710, 774-850)
    for (auto& f : table_fields) {
      const int fi = field_idx_[f.name];
      values_[fi][docid] = f.value;
      scalar_index_put(fi, docid, f.value);
    }
    if (has_vec) {
      if (vec_len != (size_t)dim_ * 4) return -1;
      std::vector<float> x(dim_);
      memcpy(x.data(), vec, vec_len);
      if (flush_pending_locked()) return -1;
      if (index_->update_vector(docid, x.data())) return -1;
    }
    for (size_t ei = 0; ei < extra_.size(); ei++) {
      if (!evec[ei].first) continue;
      if (evec[ei].second != (size_t)extra_[ei].dim * 4) return -1;
      std::vector<float> x(extra_[ei].dim);
      memcpy(x.data(), evec[ei].first, evec[ei].second);
      if (flush_pending_locked()) return -1;
      if (extra_[ei].index->update_vector(docid, x.data())) return -1;
    }
    return 0;
  } else if (docid >= max_docid_) {
    return -2;
  }
  // CheckDoc (engine.cc:802-813): every vector field present with d*4 bytes
  if (!has_vec || vec_len != (size_t)dim_ * 4) return -3;
  for (size_t ei = 0; ei < extra_.size(); ei++)
    if (!evec[ei].first || evec[ei].second != (size_t)extra_[ei].dim * 4) return -3;
  if (key.empty()) return -3;
  for (size_t fi = 0; fi < fields_.size(); fi++) values_[fi].emplace_back();
  for (auto& f : table_fields) values_[field_idx_[f.name]][max_docid_] = f.value;
  values_[field_idx_["_id"]][max_docid_] = key;
  for (size_t fi = 0; fi < fields_.size(); fi++)
    if (fields_[fi].indexed) scalar_index_put((int)fi, max_docid_, values_[fi][max_docid_]);
  keys_.push_back(key);
  key2docid_[key] = max_docid_;
  pending_.resize((size_t)(pending_n_ + 1) * dim_);
  memcpy(pending_.data() + (size_t)pending_n_ * dim_, vec, vec_len);
  for (size_t ei = 0; ei < extra_.size(); ei++) {
    auto& e = extra_[ei];
    e.pending.resize((size_t)(pending_n_ + 1) * e.dim);
    memcpy(e.pending.data() + (size_t)pending_n_ * e.dim, evec[ei].first, evec[ei].second);
  }
  pending_n_++;
  ++max_docid_;
  if ((size_t)(max_docid_ >> 3) + 1 > del_bitmap_.size()) del_bitmap_.resize((size_t)(max_docid_ >> 3) + 4096, 0);
  if (pending_n_ >= 8192 && flush_pending_locked()) return -5;
  // auto-start indexing (engine.cc:753-761)
  if (refresh_interval_ >= 0 && indexing_state_.load() == 0 && index_status_.load() == 0 &&
      max_docid_ - delete_num_ >= training_threshold_ &&
      now_ms() - last_train_failure_ms_.load() >= kTrainRetryMs) {  // a failed training is retried after a back-off
    lk.unlock();
    BuildIndex();
  }
  return 0;
}

// Engine::Delete (search/engine.cc:852-879)
int Engine::Delete(const std::string& key) {
  std::unique_lock<std::shared_mutex> lk(mu_);
  auto it = key2docid_.find(key);
  if (it == key2docid_.end() || it->second < 0) return -1;
  int docid = it->second;
  if ((del_bitmap_[docid >> 3] >> (docid & 7)) & 1) return 0;
  del_bitmap_[docid >> 3] |= (uint8_t)(1u << (docid & 7));
  ++delete_num_;
  key2docid_.erase(it);  // table_->Delete(key)
  return 0;
}

void Engine::serialize_doc(int docid, bool with_docid, std::string* out) {
  FbBuilder b;
  std::vector<FbBuilder::Off> offs;
  auto add_field = [&](const std::string& name, const std::string& value, int dt) {
    FbBuilder::Off v = b.create_bytes(value.data(), value.size(), false);
    FbBuilder::Off n = b.create_string(name);
    b.start_table(3);
    b.add_offset(0, n);
    b.add_offset(1, v);
    if (dt) b.add_scalar<int8_t>(2, (int8_t)dt);
    offs.push_back(b.end_table());
  };
  if (docid >= 0) {
    for (size_t fi = 0; fi < fields_.size(); fi++) add_field(fields_[fi].name, values_[fi][docid], fields_[fi].data_type);
    if (with_docid) add_field("_docid", std::string(reinterpret_cast<const char*>(&docid), 4), DT_INT);
    std::vector<float> x(dim_);
    bool got = false;
    int64_t stored = index_->store().size();
    if (docid < stored) {
      got = index_->store().get_host(docid, x.data()) == 0;
    } else if (docid - stored < pending_n_) {
      memcpy(x.data(), pending_.data() + (size_t)(docid - stored) * dim_, (size_t)dim_ * 4);
      got = true;
    }
    if (got) add_field(vec_name_, std::string(reinterpret_cast<const char*>(x.data()), (size_t)dim_ * 4), DT_VECTOR);
    for (auto& e : extra_) {
      std::vector<float> ex(e.dim);
      bool egot = false;
      if (docid < stored) {
        egot = e.index->store().get_host(docid, ex.data()) == 0;
      } else if (docid - stored < pending_n_) {
        memcpy(ex.data(), e.pending.data() + (size_t)(docid - stored) * e.dim, (size_t)e.dim * 4);
        egot = true;
      }
      if (egot) add_field(e.name, std::string(reinterpret_cast<const char*>(ex.data()), (size_t)e.dim * 4), DT_VECTOR);
    }
  }
  FbBuilder::Off fv = b.create_offset_vector(offs);
  b.start_table(1);
  b.add_offset(0, fv);
  b.finish(b.end_table());
  out->assign(reinterpret_cast<const char*>(b.data()), b.size());
}

// Engine::GetDoc (search/engine.cc:881-948)
int Engine::GetDocByKey(const std::string& key, std::string* fb_out) {
  std::shared_lock<std::shared_mutex> lk(mu_);
  cudaSetDevice(device_);
  auto it = key2docid_.find(key);
  if (it == key2docid_.end() || it->second < 0) {
    serialize_doc(-1, false, fb_out);
    return -1;
  }
  int docid = it->second;
  if ((del_bitmap_[docid >> 3] >> (docid & 7)) & 1) {
    serialize_doc(-1, false, fb_out);
    return -1;
  }
  serialize_doc(docid, false, fb_out);
  return 0;
}
int Engine::GetDocByDocid(int docid, bool next, std::string* fb_out) {
  std::shared_lock<std::shared_mutex> lk(mu_);
  cudaSetDevice(device_);
  auto deleted = [&](int id) { return ((del_bitmap_[id >> 3] >> (id & 7)) & 1) != 0; };
  if ((next ? docid < -1 : docid < 0) || docid >= max_docid_) {
    serialize_doc(-1, false, fb_out);
    return -1;
  }
  if (next) {
    while (++docid < max_docid_)
      if (!deleted(docid)) break;
    if (docid >= max_docid_) {
      serialize_doc(-1, false, fb_out);
      return -1;
    }
  } else if (deleted(docid)) {
    serialize_doc(-1, false, fb_out);
    return -1;
  }
  serialize_doc(docid, next, fb_out);
  return 0;
}

// ---- scalar filters ------------------------------------------------------------------------------
// Filter() semantics per field type (table/scalar_index_manager.cc:294-345):
//   numeric: lower == upper -> Equal (NotEqual when is_union == Not); only one bound -> <, <=, >, >=;
//            both -> Range with the include flags.  Values are the field type's raw little-endian bytes.
//   string / string array: lower_value split at \001 -> In (NotIn when is_union == Not); a string-array
//            document matches when any of its \001-separated elements does.
// Search(): the per-filter sets are intersected (operator And) or united (Or).  A filter on a field
// without a scalar index, or an empty result, means "no result" (scalar_index_manager.cc:598-610).
namespace {
template <typename T>
int cmp_num(const std::string& a, const std::string& b) {
  T x, y;
  memcpy(&x, a.data(), sizeof(T));
  memcpy(&y, b.data(), sizeof(T));
  return x < y ? -1 : (x > y ? 1 : 0);
}
// -2: not comparable (wrong width)
int cmp_typed(int dt, const std::string& a, const std::string& b) {
  size_t w = (dt == DT_INT || dt == DT_FLOAT) ? 4 : (dt == DT_BOOL ? 1 : 8);
  if (a.size() != w || b.size() != w) return -2;
  switch (dt) {
    case DT_INT: return cmp_num<int32_t>(a, b);
    case DT_FLOAT: return cmp_num<float>(a, b);
    case DT_DOUBLE: return cmp_num<double>(a, b);
    case DT_BOOL: return cmp_num<uint8_t>(a, b);
    default: return cmp_num<int64_t>(a, b);  // DT_LONG, DT_DATE
  }
}
std::vector<std::string> split001(const std::string& s) {
  std::vector<std::string> out;
  size_t a = 0;
  while (true) {
    size_t b = s.find('\001', a);
    out.push_back(s.substr(a, b == std::string::npos ? std::string::npos : b - a));
    if (b == std::string::npos) break;
    a = b + 1;
  }
  return out;
}
}  // namespace

static bool is_float_type(int dt) { return dt == DT_FLOAT || dt == DT_DOUBLE; }
static bool is_string_type(int dt) { return dt == DT_STRING || dt == DT_STRINGARRAY; }
// raw little-endian field bytes -> (int64 | double); false: wrong width for the type
static bool decode_num(int dt, const std::string& v, int64_t* iv, double* fv) {
  const size_t w = (dt == DT_INT || dt == DT_FLOAT) ? 4 : (dt == DT_BOOL ? 1 : 8);
  if (v.size() != w) return false;
  switch (dt) {
    case DT_INT: {
      int32_t x;
      memcpy(&x, v.data(), 4);
      *iv = x;
      return true;
    }
    case DT_FLOAT: {
      float x;
      memcpy(&x, v.data(), 4);
      *fv = x;
      return true;
    }
    case DT_DOUBLE: memcpy(fv, v.data(), 8); return true;
    case DT_BOOL: *iv = (uint8_t)v[0]; return true;
    default: memcpy(iv, v.data(), 8); return true;  // DT_LONG, DT_DATE
  }
}

void Engine::scalar_index_put(int fi, int docid, const std::string& value) {
  if (fi >= (int)sidx_.size() || !sidx_[fi].built) return;
  ScalarIndex& si = sidx_[fi];
  const int dt = fields_[fi].data_type;
  if (is_string_type(dt)) {
    if (dt == DT_STRINGARRAY) {
      for (const auto& e : split001(value)) {
        auto& pl = si.postings[e];
        if (pl.empty() || pl.back() != docid) pl.push_back(docid);
      }
    } else {
      auto& pl = si.postings[value];
      if (pl.empty() || pl.back() != docid) pl.push_back(docid);
    }
    return;
  }
  if ((int)si.ok.size() <= docid) {
    si.ok.resize((size_t)docid + 1, 0);
    if (is_float_type(dt)) si.f64.resize((size_t)docid + 1, 0.0);
    else si.i64.resize((size_t)docid + 1, 0);
  }
  int64_t iv = 0;
  double fv = 0;
  si.ok[docid] = decode_num(dt, value, &iv, &fv) ? 1 : 0;
  if (is_float_type(dt)) si.f64[docid] = fv;
  else si.i64[docid] = iv;
}

void Engine::scalar_index_rebuild(int fi) {
  if (fi >= (int)sidx_.size()) sidx_.resize(fields_.size());
  ScalarIndex& si = sidx_[fi];
  si = ScalarIndex();
  si.built = true;
  for (int d = 0; d < (int)values_[fi].size(); d++) scalar_index_put(fi, d, values_[fi][d]);
}

int64_t Engine::eval_filters(const std::vector<SearchRequestPB::Filter>& filters, int op, std::vector<uint8_t>* bitmap) const {
  const int n = max_docid_;
  const size_t nbytes = (size_t)(n >> 3) + 1;
  bitmap->assign(nbytes, 0);
  std::vector<uint8_t> cur(nbytes);
  bool first = true;
  auto set_bit = [&](int d) { cur[d >> 3] |= (uint8_t)(1u << (d & 7)); };
  for (const auto& fl : filters) {
    auto it = field_idx_.find(fl.field);
    if (it == field_idx_.end() || !fields_[it->second].indexed) return 0;
    const int fi = it->second, dt = fields_[fi].data_type;
    const bool is_str = is_string_type(dt);
    if (fl.lower.empty() && (is_str || fl.upper.empty())) continue;  // Filter() returns an untouched result
    if (fi >= (int)sidx_.size() || !sidx_[fi].built) return 0;
    const ScalarIndex& si = sidx_[fi];
    std::fill(cur.begin(), cur.end(), 0);
    const bool neg = fl.is_union == 2;
    if (is_str) {
      // In / NotIn over the inverted map; postings may hold documents whose value has changed since: re-check
      const std::vector<std::string> items = split001(fl.lower);
      for (const auto& item : items) {
        auto pit = si.postings.find(item);
        if (pit == si.postings.end()) continue;
        for (int d : pit->second) {
          if (d >= n) continue;
          const std::string& v = values_[fi][d];
          bool in;
          if (dt == DT_STRINGARRAY) {
            in = false;
            for (const auto& e : split001(v))
              if (e == item) in = true;
          } else {
            in = v == item;
          }
          if (in) set_bit(d);
        }
      }
      if (neg) {
        for (size_t i = 0; i < nbytes; i++) cur[i] = (uint8_t)~cur[i];
      }
    } else {
      int64_t lo_i = 0, hi_i = 0;
      double lo_f = 0, hi_f = 0;
      const bool has_lo = !fl.lower.empty(), has_hi = !fl.upper.empty();
      const bool lo_ok = has_lo && decode_num(dt, fl.lower, &lo_i, &lo_f);
      const bool hi_ok = has_hi && decode_num(dt, fl.upper, &hi_i, &hi_f);
      const bool equal = fl.lower == fl.upper;
      const int m = std::min<int>(n, (int)si.ok.size());
      auto scan = [&](auto* col, auto lo, auto hi) {
        for (int d = 0; d < m; d++) {
          if (!si.ok[d]) continue;
          const auto v = col[d];
          bool hit;
          if (equal) {
            hit = lo_ok && (neg ? v != lo : v == lo);
          } else {
            hit = true;
            if (has_lo) hit = lo_ok && (v > lo || (v == lo && fl.include_lower));
            if (hit && has_hi) hit = hi_ok && (v < hi || (v == hi && fl.include_upper));
          }
          if (hit) set_bit(d);
        }
      };
      if (is_float_type(dt)) scan(si.f64.data(), lo_f, hi_f);
      else scan(si.i64.data(), lo_i, hi_i);
    }
    if (n & 7) cur[nbytes - 1] &= (uint8_t)((1u << (n & 7)) - 1u);  // no bits at or above max_docid
    else cur[nbytes - 1] = 0;
    if (first) {
      bitmap->swap(cur);
      cur.resize(bitmap->size());
      first = false;
    } else if (op == 0) {
      for (size_t i = 0; i < cur.size(); i++) (*bitmap)[i] &= cur[i];
    } else if (op == 1) {
      for (size_t i = 0; i < cur.size(); i++) (*bitmap)[i] |= cur[i];
    }
  }
  if (first) return 0;
  int64_t card = 0;
  for (uint8_t b : *bitmap) card += __builtin_popcount(b);
  return card;
}

// Engine::Search (search/engine.cc:242-402) + VectorManager::Search (vector_manager.cc:739-1079)
// + Response::Serialize (response.cc:46-185)
Status Engine::Search(const SearchRequestPB& req, std::string* pb_out) {
  if (!created_table_) return Status::Make(kInvalidArgument, space_name_ + " table not created");
  if (req.req_num <= 0) return Status::Make(kInvalidArgument, space_name_ + " req_num should not less than 0");
  // engine.cc:252-260: Status::ResourceExhausted() = kBusy + "Resource temporarily unavailable"
  AdmissionGuard admission(req.req_num);
  if (!admission.permit) return Status::Make(kBusy, "Resource temporarily unavailable");
  if (req.topn <= 0) return Status::Make(kInvalidArgument, "limit[topN] is zero");
  if (req.vec_fields.empty()) return Status::Make(kInvalidArgument, "no vector query");
  if (req.vec_fields.size() > 1) return SearchMulti(req, pb_out);
  const auto& vq = req.vec_fields[0];
  int qdim = 0;
  Index* qindex = index_of(vq.name, &qdim);
  if (!qindex) return Status::Make(kInvalidArgument, "Query name " + vq.name + " not exist in created vector table");
  int brute = req.brute_force_search;
  if (brute == 2 && index_status_.load() != 2) brute = 1;
  if (brute == 0 && index_status_.load() != 2 && max_docid_ > 100 && !enable_realtime_)
    return Status::Make(kIndexError, space_name_ + " index not trained, brute_force_search is 0, max_docid_ = " +
                                         std::to_string(max_docid_) + ", threshold = 100");
  int n = (int)(vq.value.size() / ((size_t)qdim * 4));
  if (n <= 0) return Status::Make(kInvalidArgument, "Search n shouldn't less than 0!");
  if (IsKilled(req.request_id, req.partition_id)) return Status::Make(kMemoryExceeded, "");
  SearchContext ctx;
  std::string err;
  if (!parse_retrieval_params(req.index_params, &ctx.params, &err)) return Status::Make(kInvalidArgument, err);
  ctx.params.brute_force = brute != 0;
  ctx.search_unindexed_tail = enable_realtime_;
  // proto3 drops zero-valued doubles; the router always sends a window (doc_query.go:1220-1226)
  ctx.min_score = vq.has_min ? (float)std::max(vq.min_score, -(double)FLT_MAX) : (vq.has_max ? 0.f : -FLT_MAX);
  ctx.max_score = vq.has_max ? (float)std::min(vq.max_score, (double)FLT_MAX) : (vq.has_min ? 0.f : FLT_MAX);
  if (!vq.has_min && !vq.has_max) {
    ctx.min_score = -FLT_MAX;
    ctx.max_score = FLT_MAX;
  }
  const int topN = req.topn + req.offset;
  std::vector<float> x((size_t)n * qdim);
  memcpy(x.data(), vq.value.data(), x.size() * 4);
  std::vector<float> dis((size_t)n * topN);
  std::vector<int64_t> ids((size_t)n * topN);
  std::vector<uint8_t> bm, fbm;
  int total_docs;
  {
    std::unique_lock<std::shared_mutex> wl(mu_, std::defer_lock);
    std::shared_lock<std::shared_mutex> rl(mu_);
    bool need_flush = pending_n_ > 0;
    rl.unlock();
    if (need_flush) {
      wl.lock();
      if (flush_pending_locked()) return Status::Make(kIndexError, last_error());
      wl.unlock();
    }
    rl.lock();
    if (delete_num_ > 0) {
      bm.assign(del_bitmap_.begin(), del_bitmap_.begin() + (max_docid_ >> 3) + 1);
      ctx.del_bitmap = bm.data();
      ctx.bitmap_bits = max_docid_;
    }
    total_docs = doc_num();
    if (!req.filters.empty()) {  // ScalarIndexQuery (search/engine.cc:349-366, 525-580)
      if (eval_filters(req.filters, req.filter_operator, &fbm) == 0) {
        PbWriter resp;
        for (int i = 0; i < req.req_num; i++) {
          PbWriter sr, st;
          st.put_int32(1, 0);
          st.put_int32(3, 0);
          sr.put_message(5, st.out);
          sr.put_string(6, space_name_ + " no result: numeric filter return 0 result");
          resp.put_message(2, sr.out);
        }
        *pb_out = resp.out;
        return Status::OK();
      }
      ctx.filter_bitmap = fbm.data();
      ctx.bitmap_bits = max_docid_;
    }
  }
  int rc = qindex->search(ctx, n, x.data(), topN, dis.data(), ids.data());
  if (rc == -2 || IsKilled(req.request_id, req.partition_id)) return Status::Make(kMemoryExceeded, "");
  if (rc != 0) return Status::Make(kInvalidArgument, "faild search of query " + vq.name + ": " + last_error());

  serialize_results(req, n, topN, dis.data(), ids.data(), total_docs, pb_out);
  return Status::OK();
}

Engine::FieldSel Engine::select_fields(const std::vector<std::string>& names) {
  FieldSel sel;
  if (!names.empty()) {
    int dim;
    for (auto& nme : names) {
      if (index_of(nme, &dim))
        sel.vecs.push_back(nme);
      else if (field_idx_.count(nme))
        sel.attr.push_back(field_idx_[nme]);
    }
  } else {
    for (size_t fi = 0; fi < fields_.size(); fi++) sel.attr.push_back((int)fi);
  }
  std::sort(sel.attr.begin(), sel.attr.end(), [&](int a, int b) { return fields_[a].name < fields_[b].name; });
  return sel;
}

void Engine::serialize_results(const SearchRequestPB& req, int n, int topN, const float* dis, const int64_t* ids,
                               int total_docs, std::string* pb_out) {
  std::shared_lock<std::shared_mutex> rl(mu_);
  const FieldSel sel = select_fields(req.fields);
  PbWriter resp;
  Status okst;
  for (int i = 0; i < req.req_num && i < n; i++) {
    PbWriter sr;
    // field order on the wire follows the field numbers, like the C++ serializer
    double max_score = -DBL_MAX;
    PbWriter items;
    for (int j = req.offset; j < topN; j++) {
      int64_t docid = ids[(size_t)i * topN + j];
      if (docid < 0) continue;  // vector_manager.cc:1059
      double score = dis[(size_t)i * topN + j];
      max_score = std::max(max_score, score);
      PbWriter item;
      item.put_double(1, score);
      put_doc_fields((int)docid, sel, &item);
      items.put_message(7, item.out);
    }
    sr.put_double(2, max_score);
    PbWriter st;
    st.put_int32(1, total_docs);
    st.put_int32(3, total_docs);
    sr.put_message(5, st.out);
    sr.put_string(6, okst.ToString());
    sr.out += items.out;
    resp.put_message(2, sr.out);
  }
  *pb_out = resp.out;
}

// WeightedRanker::Parse (common/common_query_data.h:257-300)
static bool parse_ranker(const std::string& raw, size_t nvec, std::vector<double>* w, std::string* err) {
  w->assign(nvec, 1.0 / (double)nvec);
  if (raw.empty()) return true;
  *err = "weighted ranker params err: " + raw;
  JsonValue jv;
  if (!JsonParser::parse(raw, &jv) || !jv.get("type") || !jv.get("params")) return false;
  const JsonValue* arr = jv.get("params");
  if (arr->type != JsonValue::Array) return false;
  if (arr->arr.size() != nvec) {
    *err = "weighted ranker params: " + raw + ", length don't equal to " + std::to_string(nvec);
    return false;
  }
  for (size_t i = 0; i < nvec; i++) {
    if (arr->arr[i].type != JsonValue::Number) return false;
    (*w)[i] = arr->arr[i].num;
  }
  return true;
}

Status Engine::SearchMulti(const SearchRequestPB& req, std::string* pb_out) {
  const size_t nvec = req.vec_fields.size();
  std::vector<Index*> idx(nvec);
  std::vector<int> dims(nvec);
  int n = -1;
  for (size_t j = 0; j < nvec; j++) {
    const auto& vq = req.vec_fields[j];
    idx[j] = index_of(vq.name, &dims[j]);
    if (!idx[j]) return Status::Make(kInvalidArgument, "Query name " + vq.name + " not exist in created vector table");
    const int nj = (int)(vq.value.size() / ((size_t)dims[j] * 4));
    if (nj <= 0 || (n >= 0 && nj != n)) return Status::Make(kInvalidArgument, "Search n shouldn't less than 0!");
    n = nj;
  }
  std::vector<double> weights;
  std::string err;
  if (!parse_ranker(req.ranker, nvec, &weights, &err)) return Status::Make(kInvalidArgument, err);
  int brute = req.brute_force_search;
  if (brute == 2 && index_status_.load() != 2) brute = 1;
  if (brute == 0 && index_status_.load() != 2 && max_docid_ > 100 && !enable_realtime_)
    return Status::Make(kIndexError, space_name_ + " index not trained, brute_force_search is 0, max_docid_ = " +
                                         std::to_string(max_docid_) + ", threshold = 100");
  if (IsKilled(req.request_id, req.partition_id)) return Status::Make(kMemoryExceeded, "");
  SearchContext base;
  if (!parse_retrieval_params(req.index_params, &base.params, &err)) return Status::Make(kInvalidArgument, err);
  base.params.brute_force = brute != 0;
  base.search_unindexed_tail = enable_realtime_;
  const int topN = req.topn + req.offset;
  std::vector<uint8_t> bm, fbm;
  int total_docs;
  {
    std::unique_lock<std::shared_mutex> wl(mu_);
    if (pending_n_ > 0 && flush_pending_locked()) return Status::Make(kIndexError, last_error());
    if (delete_num_ > 0) {
      bm.assign(del_bitmap_.begin(), del_bitmap_.begin() + (max_docid_ >> 3) + 1);
      base.del_bitmap = bm.data();
      base.bitmap_bits = max_docid_;
    }
    total_docs = doc_num();
    if (!req.filters.empty()) {
      if (eval_filters(req.filters, req.filter_operator, &fbm) == 0) {
        PbWriter resp;
        for (int i = 0; i < req.req_num; i++) {
          PbWriter sr, st;
          st.put_int32(1, 0);
          st.put_int32(3, 0);
          sr.put_message(5, st.out);
          sr.put_string(6, space_name_ + " no result: numeric filter return 0 result");
          resp.put_message(2, sr.out);
        }
        *pb_out = resp.out;
        return Status::OK();
      }
      base.filter_bitmap = fbm.data();
      base.bitmap_bits = max_docid_;
    }
  }
  // every field on its own, topN each (vector_manager.cc:790-852)
  std::vector<std::vector<float>> dis(nvec, std::vector<float>((size_t)n * topN));
  std::vector<std::vector<int64_t>> ids(nvec, std::vector<int64_t>((size_t)n * topN));
  for (size_t j = 0; j < nvec; j++) {
    const auto& vq = req.vec_fields[j];
    SearchContext ctx = base;
    ctx.min_score = vq.has_min ? (float)std::max(vq.min_score, -(double)FLT_MAX) : (vq.has_max ? 0.f : -FLT_MAX);
    ctx.max_score = vq.has_max ? (float)std::min(vq.max_score, (double)FLT_MAX) : (vq.has_min ? 0.f : FLT_MAX);
    if (!vq.has_min && !vq.has_max) ctx.min_score = -FLT_MAX, ctx.max_score = FLT_MAX;
    std::vector<float> x((size_t)n * dims[j]);
    memcpy(x.data(), vq.value.data(), x.size() * 4);
    int rc = idx[j]->search(ctx, n, x.data(), topN, dis[j].data(), ids[j].data());
    if (rc == -2 || IsKilled(req.request_id, req.partition_id)) return Status::Make(kMemoryExceeded, "");
    if (rc != 0) return Status::Make(kInvalidArgument, "faild search of query " + vq.name + ": " + last_error());
  }
  // docid join (vector_manager.cc:900-964): a document survives when EVERY field returned it; its score is
  // the weighted sum of the per-field scores; docid order unless multi_vector_rank asks for score order
  std::vector<float> out_dis((size_t)n * topN, 0.f);
  std::vector<int64_t> out_ids((size_t)n * topN, -1);
  const bool l2 = index_->metric() == kMetricL2;
  for (int i = 0; i < n; i++) {
    std::map<int64_t, std::pair<int, double>> acc;  // docid -> (fields seen, score)
    for (size_t j = 0; j < nvec; j++)
      for (int r = 0; r < topN; r++) {
        const int64_t d = ids[j][(size_t)i * topN + r];
        if (d < 0) continue;
        auto& e = acc[d];
        e.first++;
        e.second += (double)((float)dis[j][(size_t)i * topN + r] * (float)weights[j]);  // float product, as the reference
      }
    std::vector<std::pair<int64_t, double>> common;
    for (auto& kv : acc)
      if (kv.second.first == (int)nvec) common.push_back({kv.first, kv.second.second});
    if (req.multi_vector_rank == 1)
      std::sort(common.begin(), common.end(), [l2](const std::pair<int64_t, double>& a, const std::pair<int64_t, double>& b) {
        return l2 ? a.second < b.second : a.second > b.second;
      });
    for (size_t r = 0; r < common.size() && r < (size_t)topN; r++) {
      out_ids[(size_t)i * topN + r] = common[r].first;
      out_dis[(size_t)i * topN + r] = (float)common[r].second;
    }
  }
  serialize_results(req, n, topN, out_dis.data(), out_ids.data(), total_docs, pb_out);
  return Status::OK();
}

void Engine::put_doc_fields(int docid, const FieldSel& sel, PbWriter* item) {
  for (int fi : sel.attr) {
    PbWriter fld;
    fld.put_string(1, fields_[fi].name);
    const std::string& val = values_[fi][docid];
    fld.put_bytes(3, val.data(), val.size());
    item->put_message(2, fld.out);
  }
  for (const auto& vn : sel.vecs) {
    int dim = 0;
    Index* ix = index_of(vn, &dim);
    std::vector<float> vbuf(dim);
    if (ix && ix->store().get_host(docid, vbuf.data()) == 0) {
      PbWriter fld;
      fld.put_string(1, vn);
      fld.put_bytes(3, vbuf.data(), (size_t)dim * 4);
      item->put_message(2, fld.out);
    }
  }
}

// Engine::Query (search/engine.cc:404-523): documents by key (by docid when partition_id > 0), or the
// first `limit` live documents that pass the scalar filters, as one SearchResult with score-less items
Status Engine::Query(const QueryRequestPB& req, std::string* pb_out) {
  if (!created_table_) return Status::Make(kInvalidArgument, space_name_ + " table not created");
  {
    // documents accepted but not yet uploaded must be visible to GetDoc-style reads: flush under the exclusive
    // lock, then serve the query under the shared one (filters, field reads and the per-document device reads
    // of put_doc_fields do not block ingest or other searches)
    std::unique_lock<std::shared_mutex> wl(mu_);
    if (pending_n_ > 0 && flush_pending_locked()) return Status::Make(kIndexError, last_error());
  }
  std::shared_lock<std::shared_mutex> rl(mu_);
  std::vector<int> docids;
  auto deleted = [&](int d) { return ((del_bitmap_[d >> 3] >> (d & 7)) & 1) != 0; };
  if (!req.document_ids.empty()) {
    for (const auto& id : req.document_ids) {
      int docid = -1;
      if (req.partition_id > 0) {
        char* end = nullptr;
        long v = strtol(id.c_str(), &end, 10);
        if (id.empty() || *end != '\0' || v < 0 || v >= max_docid_) continue;
        docid = (int)v;
      } else {
        auto it = key2docid_.find(id);
        if (it == key2docid_.end()) continue;
        docid = it->second;
      }
      if (!deleted(docid)) docids.push_back(docid);
    }
  } else {
    const int topn = req.limit;
    std::vector<uint8_t> fbm;
    if (!req.filters.empty()) {
      if (eval_filters(req.filters, req.filter_operator, &fbm) == 0) {
        PbWriter resp, sr, st;
        st.put_int32(1, 0);
        st.put_int32(3, 0);
        sr.put_message(5, st.out);
        sr.put_string(6, space_name_ + " no result: numeric filter return 0 result");
        resp.put_message(2, sr.out);
        *pb_out = resp.out;
        return Status::OK();
      }
      int skipped = 0;
      for (int d = 0; d < max_docid_ && (int)docids.size() < topn; d++) {
        if (!((fbm[d >> 3] >> (d & 7)) & 1)) continue;
        if (skipped++ < req.offset) continue;  // ScalarIndexManager::Query drops `offset` hits first
        if (!deleted(d)) docids.push_back(d);
      }
    }
  }
  const FieldSel sel = select_fields(req.fields);
  PbWriter resp, sr, st, items;
  for (int d : docids) {
    PbWriter item;  // score 0.0: proto3 leaves it off the wire
    put_doc_fields(d, sel, &item);
    items.put_message(7, item.out);
  }
  sr.put_double(2, docids.empty() ? -DBL_MAX : 0.0);
  st.put_int32(1, (int)docids.size());
  st.put_int32(3, (int)docids.size());
  sr.put_message(5, st.out);
  sr.put_string(6, Status::OK().ToString());
  sr.out += items.out;
  resp.put_message(2, sr.out);
  *pb_out = resp.out;
  return Status::OK();
}

Status Engine::SetFieldIndexed(const std::string& field, bool indexed) {
  if (!created_table_) return Status::Make(kIOError, "table not initialized");
  std::unique_lock<std::shared_mutex> lk(mu_);
  int dim = 0;
  if (index_of(field, &dim))
    return Status::Make(kNotSupported, "the index of vector field " + field + " is fixed when the table is created");
  auto it = field_idx_.find(field);
  if (it == field_idx_.end()) return Status::Make(kInvalidArgument, "field " + field + " not found");
  fields_[it->second].indexed = indexed;
  if (indexed) {
    scalar_index_rebuild(it->second);  // AddFieldIndex builds the index over the documents already stored
  } else if (it->second < (int)sidx_.size()) {
    sidx_[it->second] = ScalarIndex();
  }
  return Status::OK();
}

int64_t Engine::now_ms() {
  return std::chrono::duration_cast<std::chrono::milliseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// Engine::BuildIndex / Engine::Indexing (search/engine.cc:951-988, 1091-1142)
int Engine::BuildIndex() {
  if (!created_table_) return -1;
  int expected = 0;
  if (!indexing_state_.compare_exchange_strong(expected, 1)) return 0;  // already in progress
  if (indexing_thread_.joinable()) indexing_thread_.join();
  indexing_thread_ = std::thread(&Engine::indexing_loop, this);
  return 0;
}

// Engine::RebuildIndex: only acts on a running, indexed engine; stops the indexing thread, drops the index
// structures of every vector field (the raw vectors stay) and starts over: train on the current first
// training_threshold vectors, re-add everything.  Both reference variants (build the new indexes aside, or
// drop first) end in the same state; here the old index is dropped first, so searches in between see the
// "index not trained" / brute-force rules of an un-indexed table.
int Engine::RebuildIndex(int drop_before_rebuild, int limit_cpu, int describe) {
  (void)drop_before_rebuild;
  (void)limit_cpu;
  if (!created_table_) return -1;
  if (indexing_state_.load() != 2 || index_status_.load() == 0) return 0;  // "index not running, no need to rebuild!"
  quiesce();
  indexing_state_.store(0);
  if (describe) return 0;
  cudaSetDevice(device_);
  {
    std::unique_lock<std::shared_mutex> lk(mu_);
    if (flush_pending_locked()) return -1;
  }
  if (index_->reset_index()) return -1;
  for (auto& e : extra_)
    if (e.index->reset_index()) return -1;
  index_status_.store(0);
  if (refresh_interval_ >= 0 && max_docid_ - delete_num_ >= training_threshold_) return BuildIndex();
  return 0;
}

void Engine::indexing_loop() {
  cudaSetDevice(device_);
  int expected = 1;
  if (!indexing_state_.compare_exchange_strong(expected, 2)) {
    indexing_state_.store(0);
    return;
  }
  {
    std::unique_lock<std::shared_mutex> lk(mu_);
    flush_pending_locked();
  }
  bool train_failed = index_->train() != 0;  // e.g. fewer vectors than training_threshold
  for (auto& e : extra_) train_failed = train_failed || e.index->train() != 0;
  if (train_failed) {
    // e.g. fewer vectors than training_threshold: remember when, so AddOrUpdate does not spawn and join a new
    // indexing thread for every document until the threshold is reached (BuildIndex retries after a back-off)
    last_train_failure_ms_.store(now_ms());
    indexing_state_.store(0);
    idx_cv_.notify_all();
    return;
  }
  bool has_error = false;
  while (indexing_state_.load() == 2) {
    if (has_error) {
      std::this_thread::sleep_for(std::chrono::milliseconds(200));
      continue;
    }
    std::vector<uint8_t> bm;
    {
      std::unique_lock<std::shared_mutex> lk(mu_);
      if (flush_pending_locked()) has_error = true;
      if (delete_num_ > 0) bm.assign(del_bitmap_.begin(), del_bitmap_.begin() + (max_docid_ >> 3) + 1);
    }
    if (!has_error && index_->add_pending(bm.empty() ? nullptr : bm.data()) != 0) has_error = true;
    for (auto& e : extra_)
      if (!has_error && e.index->add_pending(bm.empty() ? nullptr : bm.data()) != 0) has_error = true;
    if (!has_error) index_status_.store(2);
    // sleep refresh_interval ms, waking early on Close
    std::unique_lock<std::mutex> lk(idx_mu_);
    idx_cv_.wait_for(lk, std::chrono::milliseconds(refresh_interval_ > 0 ? refresh_interval_ : 1),
                     [this] { return indexing_state_.load() != 2; });
  }
  indexing_state_.store(0);
  idx_cv_.notify_all();
}

std::string Engine::EngineStatus() {  // search/engine.cc:1164-1176
  std::shared_lock<std::shared_mutex> lk(mu_);
  int64_t min_indexed = created_table_ && index_ ? index_->indexed_count() : 0;
  for (auto& e : extra_) min_indexed = std::min(min_indexed, e.index->indexed_count());  // min over the vector fields
  char buf[256];
  snprintf(buf, sizeof buf,
           "{\"backup_status\":0,\"doc_num\":%d,\"index_status\":%d,\"max_docid\":%d,\"min_indexed_num\":%lld}",
           doc_num(), index_status_.load(), max_docid_ - 1, (long long)min_indexed);
  return buf;
}

std::string Engine::MemoryInfo() {  // search/engine.cc:1178-1200
  std::shared_lock<std::shared_mutex> lk(mu_);
  long long table_mem = 0;
  for (auto& col : values_)
    for (auto& v : col) table_mem += (long long)v.size() + (long long)sizeof(std::string);
  long long index_mem = index_ ? index_->index_mem_bytes() : 0;
  long long vec_mem = index_ ? index_->store().mem_bytes() : 0;
  for (auto& e : extra_) index_mem += e.index->index_mem_bytes(), vec_mem += e.index->store().mem_bytes();
  char buf[256];
  snprintf(buf, sizeof buf,
           "{\"bitmap_mem\":%lld,\"field_range_mem\":0,\"index_mem\":%lld,\"table_mem\":%lld,\"vector_mem\":%lld}",
           (long long)del_bitmap_.size(), index_mem, table_mem, vec_mem);
  return buf;
}

int Engine::SetConfig(const std::string& json) {  // search/engine.cc:1764-1790
  JsonValue jv;
  if (!JsonParser::parse(json, &jv)) return -1;
  int v;
  if (jv.get_int("refresh_interval", &v)) refresh_interval_ = v;
  if (jv.get_int("slow_search_time", &v)) slow_search_time_ = v;
  bool b;
  if (jv.get_bool("enable_id_cache", &b)) enable_id_cache_ = b;
  return 0;
}
std::string Engine::GetConfig() {  // search/engine.cc:1792-1807
  char buf[256];
  snprintf(buf, sizeof buf,
           "{\"enable_id_cache\":%s,\"engine_cache_size\":0,\"refresh_interval\":%d,\"slow_search_time\":%d}",
           enable_id_cache_ ? "true" : "false", refresh_interval_, slow_search_time_);
  return buf;
}

// ---- Dump / Load (own snapshot format; byte-compatible gamma dumps are a "next" row) --------
namespace {
template <typename T>
void wr(std::ofstream& f, const T& v) {
  f.write(reinterpret_cast<const char*>(&v), sizeof(T));
}
void wr_str(std::ofstream& f, const std::string& s) {
  uint64_t n = s.size();
  wr(f, n);
  f.write(s.data(), (std::streamsize)n);
}
template <typename T>
bool rdv(std::ifstream& f, T* v) {
  return (bool)f.read(reinterpret_cast<char*>(v), sizeof(T));
}
bool rd_str(std::ifstream& f, std::string* s) {
  uint64_t n;
  if (!rdv(f, &n) || n > ((uint64_t)1 << 40)) return false;
  s->resize(n);
  return n == 0 || (bool)f.read(&(*s)[0], (std::streamsize)n);
}
}  // namespace

// Engine::Dump (search/engine.cc:1202-1247): <path>/retrieval_model_index/<name>.gbdump + dump.done
int Engine::Dump() {
  if (!created_table_) return -1;
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  if (flush_pending_locked()) return -1;
  std::string dir = path_ + "/retrieval_model_index";
  mkdir(path_.c_str(), 0755);
  mkdir(dir.c_str(), 0755);
  std::ofstream f(dir + "/" + table_name_ + ".gbdump", std::ios::binary | std::ios::trunc);
  if (!f) return -1;
  const char magic[8] = {'G', 'B', '2', '0', '0', 'D', 'M', 'P'};
  f.write(magic, 8);
  wr<int32_t>(f, 1);
  wr<int32_t>(f, max_docid_);
  wr<int32_t>(f, delete_num_);
  wr<int32_t>(f, dim_);
  wr<uint64_t>(f, fields_.size());
  for (size_t fi = 0; fi < fields_.size(); fi++)
    for (int d = 0; d < max_docid_; d++) wr_str(f, values_[fi][d]);
  wr_str(f, std::string(del_bitmap_.begin(), del_bitmap_.end()));
  std::vector<float> rows((size_t)max_docid_ * dim_);
  if (max_docid_ && index_->store().get_rows_host(0, max_docid_, rows.data())) return -1;
  f.write(reinterpret_cast<const char*>(rows.data()), (std::streamsize)(rows.size() * 4));
  int trained = index_->trained() ? 1 : 0;
  wr<int32_t>(f, trained);
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index_.get());
  IVFPQIndex* pq = dynamic_cast<IVFPQIndex*>(index_.get());
  if (trained && ivf) {
    std::vector<float> c((size_t)ivf->nlist() * dim_);
    if (ivf->get_centroids(c.data())) return -1;
    f.write(reinterpret_cast<const char*>(c.data()), (std::streamsize)(c.size() * 4));
    if (pq) {
      std::vector<float> p((size_t)pq->M() * 256 * pq->dsub());
      if (pq->get_pq_centroids(p.data())) return -1;
      f.write(reinterpret_cast<const char*>(p.data()), (std::streamsize)(p.size() * 4));
    }
  }
  f.close();
  // the index itself in gamma's own format (IndexModel::Dump via VectorManager::Dump,
  // vector_manager.cc:1155-1170): <dir>/<vector name>.000/{ivfflat,ivfpq}.index
  if (trained && ivf && ivf->dump_gamma(dir, vec_name_ + ".000")) return -1;
  for (auto& e : extra_) {  // the other vector fields: raw rows next to the table, index in gamma's format
    std::ofstream ef(dir + "/" + table_name_ + "." + e.name + ".gbvec", std::ios::binary | std::ios::trunc);
    std::vector<float> erows((size_t)max_docid_ * e.dim);
    if (!ef || (max_docid_ && e.index->store().get_rows_host(0, max_docid_, erows.data()))) return -1;
    wr<int32_t>(ef, max_docid_);
    wr<int32_t>(ef, e.dim);
    ef.write(reinterpret_cast<const char*>(erows.data()), (std::streamsize)(erows.size() * 4));
    if (ef.fail()) return -1;
    IVFFlatIndex* eivf = dynamic_cast<IVFFlatIndex*>(e.index.get());
    if (eivf && eivf->trained() && eivf->dump_gamma(dir, e.name + ".000")) return -1;
  }
  std::ofstream done(dir + "/dump.done");
  done << "ok";
  return f.fail() ? -1 : 0;
}

// Engine::Load (search/engine.cc:1278-1400): restore the newest complete dump, then let the
// indexing thread re-add the vectors (the lists are a deterministic function of the stored
// vectors and the trained state).
int Engine::Load() {
  if (!created_table_) return -1;
  cudaSetDevice(device_);
  std::string dir = path_ + "/retrieval_model_index";
  std::ifstream done(dir + "/dump.done");
  if (!done) return 0;  // nothing to load
  std::ifstream f(dir + "/" + table_name_ + ".gbdump", std::ios::binary);
  if (!f) return -1;
  char magic[8];
  int32_t ver, maxd, deln, dim;
  uint64_t nf;
  if (!f.read(magic, 8) || memcmp(magic, "GB200DMP", 8) || !rdv(f, &ver) || ver != 1 || !rdv(f, &maxd) || !rdv(f, &deln) ||
      !rdv(f, &dim) || dim != dim_ || !rdv(f, &nf) || nf != fields_.size())
    return -1;
  std::unique_lock<std::shared_mutex> lk(mu_);
  if (max_docid_ != 0) return -1;
  for (size_t fi = 0; fi < fields_.size(); fi++) {
    values_[fi].resize(maxd);
    for (int d = 0; d < maxd; d++)
      if (!rd_str(f, &values_[fi][d])) return -1;
  }
  std::string bm;
  if (!rd_str(f, &bm)) return -1;
  del_bitmap_.assign(bm.begin(), bm.end());
  del_bitmap_.resize(std::max<size_t>(del_bitmap_.size(), (size_t)(maxd >> 3) + 4096), 0);
  std::vector<float> rows((size_t)maxd * dim_);
  if (maxd && !f.read(reinterpret_cast<char*>(rows.data()), (std::streamsize)(rows.size() * 4))) return -1;
  int32_t trained;
  if (!rdv(f, &trained)) return -1;
  for (size_t fi = 0; fi < fields_.size(); fi++)
    if (fields_[fi].indexed) scalar_index_rebuild((int)fi);
  keys_.resize(maxd);
  int idf = field_idx_["_id"];
  for (int d = 0; d < maxd; d++) {
    keys_[d] = values_[idf][d];
    if (!((del_bitmap_[d >> 3] >> (d & 7)) & 1)) key2docid_[keys_[d]] = d;
  }
  max_docid_ = maxd;
  delete_num_ = deln;
  if (maxd && index_->add_vectors(rows.data(), maxd)) return -1;
  for (auto& e : extra_) {
    std::ifstream ef(dir + "/" + table_name_ + "." + e.name + ".gbvec", std::ios::binary);
    int32_t en = 0, ed = 0;
    if (!ef || !rdv(ef, &en) || !rdv(ef, &ed) || en != maxd || ed != e.dim) return -1;
    std::vector<float> erows((size_t)maxd * e.dim);
    if (maxd && !ef.read(reinterpret_cast<char*>(erows.data()), (std::streamsize)(erows.size() * 4))) return -1;
    if (maxd && e.index->add_vectors(erows.data(), maxd)) return -1;
    IVFFlatIndex* eivf = dynamic_cast<IVFFlatIndex*>(e.index.get());
    int64_t eload = 0;
    if (eivf) eivf->load_gamma(dir, e.name + ".000", &eload);  // trained state + lists; absent: trained again later
  }
  IVFFlatIndex* ivf = dynamic_cast<IVFFlatIndex*>(index_.get());
  IVFPQIndex* pq = dynamic_cast<IVFPQIndex*>(index_.get());
  if (trained && ivf) {
    std::vector<float> c((size_t)ivf->nlist() * dim_);
    if (!f.read(reinterpret_cast<char*>(c.data()), (std::streamsize)(c.size() * 4))) return -1;
    if (ivf->set_centroids(c.data(), ivf->nlist())) return -1;
    if (pq) {
      std::vector<float> p((size_t)pq->M() * 256 * pq->dsub());
      if (!f.read(reinterpret_cast<char*>(p.data()), (std::streamsize)(p.size() * 4))) return -1;
      if (pq->set_pq_centroids(p.data())) return -1;
    }
  }
  if (trained && ivf) {
    // IndexModel::Load: take the inverted lists from the index file when it matches this table; a
    // missing or refused file only means the indexing thread re-adds the vectors itself
    int64_t load_num = 0;
    if (ivf->load_gamma(dir, vec_name_ + ".000", &load_num) == 0 && load_num > 0) index_status_.store(2);
  }
  lk.unlock();
  if (trained) BuildIndex();  // train() is a no-op on a trained index; the loop adds what the file did not cover
  return 0;
}

}  // namespace gb
