// Host orchestration of the hot path (see index.h).  Reference call sites are cited inline.
#include <cuda.h>

#include "index.h"

#include <float.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <random>

#include "common.cuh"

namespace gb {

// ------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_last_error(const std::string& msg) { g_last_error = msg; }
const char* last_error() { return g_last_error.c_str(); }

static inline int64_t round_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// tensor-core (tcgen05 3xTF32) path for the dense query x centroid contraction: coarse search and
// the k-means assign step.  GB_TC=0 selects the exact CUDA-core kernel everywhere.  List assignment
// at add time always uses the exact kernel so list membership is deterministic against the oracle.
static bool tc_enabled() {
  static int v = [] {
    const char* e = getenv("GB_TC");
    return e ? atoi(e) : 1;
  }();
  return v != 0;
}

// SM count of a device, queried once (grids of the persistent kernels, work-splitting heuristics)
static int sm_count(int device) {
  static std::mutex mu;
  static std::vector<int> cache;
  std::lock_guard<std::mutex> lk(mu);
  if ((int)cache.size() <= device) cache.resize(device + 1, 0);
  if (!cache[device]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || n <= 0) n = 148;
    cache[device] = n;
  }
  return cache[device];
}

static cudaStream_t thread_stream(int device) {
  static thread_local cudaStream_t st[64] = {nullptr};
  if (device < 0 || device >= 64) return nullptr;
  if (!st[device]) {
    cudaSetDevice(device);
    cudaStreamCreateWithFlags(&st[device], cudaStreamNonBlocking);
  }
  return st[device];
}

// ------------------------------------------------------------------------------------------
Scratch::~Scratch() {
  for (void* p : ptrs_) cudaFreeAsync(p, st_);
}
void* Scratch::alloc(size_t bytes) {
  void* p = nullptr;
  if (bytes == 0) bytes = 16;
  cudaError_t e = cudaMallocAsync(&p, bytes, st_);
  if (e != cudaSuccess) {
    set_last_error(std::string("cudaMallocAsync(") + std::to_string(bytes) + "): " + cudaGetErrorString(e));
    return nullptr;
  }
  ptrs_.push_back(p);
  return p;
}
#define GB_ALLOC(var, T, n, s)                \
  T* var = (s).alloc_n<T>((size_t)(n));       \
  if (!var) return -1

// ------------------------------------------------------------------------------------------
// Segments are VIRTUAL address ranges of seg_rows rows; physical HBM is mapped into them in chunks as rows
// arrive (CUDA virtual memory management: cuMemAddressReserve / cuMemCreate / cuMemMap, reached through
// cudaGetDriverEntryPoint so the library still links only the static runtime).  A 100-document partition
// therefore costs one 2 MiB granule, not a 1M-row segment (3 GiB at d = 768), while row addresses stay
// stable and segment-contiguous for the kernels (MemoryRawVector grows incrementally as well,
// vector/memory_raw_vector.cc:152-240).  Without VMM support a segment is one cudaMalloc as before.
namespace {
struct VmmApi {
  CUresult (*reserve)(CUdeviceptr*, size_t, size_t, CUdeviceptr, unsigned long long) = nullptr;
  CUresult (*addr_free)(CUdeviceptr, size_t) = nullptr;
  CUresult (*create)(CUmemGenericAllocationHandle*, size_t, const CUmemAllocationProp*, unsigned long long) = nullptr;
  CUresult (*release)(CUmemGenericAllocationHandle) = nullptr;
  CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long) = nullptr;
  CUresult (*unmap)(CUdeviceptr, size_t) = nullptr;
  CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc*, size_t) = nullptr;
  CUresult (*granularity)(size_t*, const CUmemAllocationProp*, CUmemAllocationGranularity_flags) = nullptr;
  bool ok = false;
};
const VmmApi& vmm_api() {
  static const VmmApi api = [] {
    VmmApi a;
    const char* off = getenv("GB_VMM");
    if (off && atoi(off) == 0) return a;
    auto get = [](const char* name, void** fn) {
      cudaDriverEntryPointQueryResult q;
      return cudaGetDriverEntryPoint(name, fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess && *fn;
    };
    a.ok = get("cuMemAddressReserve", (void**)&a.reserve) && get("cuMemAddressFree", (void**)&a.addr_free) &&
           get("cuMemCreate", (void**)&a.create) && get("cuMemRelease", (void**)&a.release) && get("cuMemMap", (void**)&a.map) &&
           get("cuMemUnmap", (void**)&a.unmap) && get("cuMemSetAccess", (void**)&a.set_access) &&
           get("cuMemGetAllocationGranularity", (void**)&a.granularity);
    cudaGetLastError();
    return a;
  }();
  return api;
}
}  // namespace

RawStore::RawStore(int d, int seg_shift) : d_(d), dpad_((int)round_up(d, 4)), seg_shift_(seg_shift) {
  cudaMalloc(&d_segs_, sizeof(float*) * kMaxSegs);
  cudaGetDevice(&device_);
}
RawStore::~RawStore() {
  const VmmApi& api = vmm_api();
  for (Seg& sg : segs_) {
    if (!sg.vmm) {
      cudaFree(sg.base);
      continue;
    }
    size_t off = 0;
    for (auto& c : sg.chunks) {
      api.unmap((CUdeviceptr)sg.base + off, c.second);
      api.release(c.first);
      off += c.second;
    }
    api.addr_free((CUdeviceptr)sg.base, sg.va_bytes);
  }
  cudaFree(d_segs_);
}
int RawStore::new_segment() {
  if ((int)segs_.size() >= kMaxSegs) {
    set_last_error("raw store: too many segments");
    return -1;
  }
  Seg sg;
  const size_t bytes = (size_t)seg_rows() * dpad_ * 4;
  const VmmApi& api = vmm_api();
  if (api.ok) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device_;
    size_t gran = 0;
    if (api.granularity(&gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM) == CUDA_SUCCESS && gran > 0) {
      sg.gran = gran;
      sg.va_bytes = (size_t)round_up((int64_t)bytes, (int64_t)gran);
      CUdeviceptr p = 0;
      if (api.reserve(&p, sg.va_bytes, 0, 0, 0) == CUDA_SUCCESS) {
        sg.base = reinterpret_cast<float*>(p);
        sg.vmm = true;
      }
    }
  }
  if (!sg.vmm) {  // no VMM: the whole segment at once
    GB_CUDA(cudaMalloc(&sg.base, bytes));
    GB_CUDA(cudaMemset(sg.base, 0, bytes));
    sg.mapped = bytes;
    phys_bytes_ += (int64_t)bytes;
  }
  segs_.push_back(sg);
  GB_CUDA(cudaMemcpy(d_segs_ + segs_.size() - 1, &sg.base, sizeof(float*), cudaMemcpyHostToDevice));
  return 0;
}
// physical memory behind the first `rows` rows of segment si
int RawStore::map_rows(int si, int64_t rows) {
  Seg& sg = segs_[si];
  const size_t need = (size_t)rows * dpad_ * 4;
  if (need <= sg.mapped) return 0;
  const VmmApi& api = vmm_api();
  while (sg.mapped < need) {
    // geometric steps (a quarter of what is mapped, at least one granule, at most 256 MiB), never past the segment
    size_t step = std::max(sg.gran, std::min<size_t>(sg.mapped / 4, (size_t)256 << 20));
    step = (size_t)round_up((int64_t)std::max(step, std::min(need - sg.mapped, (size_t)256 << 20)), (int64_t)sg.gran);
    step = std::min(step, sg.va_bytes - sg.mapped);
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device_;
    CUmemGenericAllocationHandle hnd;
    if (api.create(&hnd, step, &prop, 0) != CUDA_SUCCESS) {
      set_last_error("raw store: out of device memory (cuMemCreate)");
      return -1;
    }
    const CUdeviceptr at = (CUdeviceptr)sg.base + sg.mapped;
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (api.map(at, step, 0, hnd, 0) != CUDA_SUCCESS || api.set_access(at, step, &acc, 1) != CUDA_SUCCESS) {
      api.release(hnd);
      set_last_error("raw store: cuMemMap failed");
      return -1;
    }
    GB_CUDA(cudaMemset(reinterpret_cast<void*>(at), 0, step));  // pad columns must read as zero
    sg.chunks.emplace_back(hnd, step);
    sg.mapped += step;
    phys_bytes_ += (int64_t)step;
  }
  return 0;
}
int RawStore::ensure(int64_t n_total) {
  while ((int64_t)segs_.size() * seg_rows() < n_total)
    if (new_segment()) return -1;
  for (int si = (int)(n_ >> seg_shift_); si < (int)segs_.size(); si++) {
    const int64_t rows = std::min<int64_t>(seg_rows(), n_total - (int64_t)si * seg_rows());
    if (rows > 0 && map_rows(si, rows)) return -1;
  }
  return 0;
}
int RawStore::append_host(const float* x, int64_t n, cudaStream_t st) {
  if (ensure(n_ + n)) return -1;
  int64_t done = 0;
  while (done < n) {
    int64_t vid = n_ + done;
    int64_t si = vid >> seg_shift_, off = vid & (seg_rows() - 1);
    int64_t cnt = std::min(n - done, seg_rows() - off);
    GB_CUDA(cudaMemcpy2DAsync(segs_[si].base + off * dpad_, (size_t)dpad_ * 4, x + done * d_, (size_t)d_ * 4, (size_t)d_ * 4,
                              (size_t)cnt, cudaMemcpyHostToDevice, st));
    done += cnt;
  }
  GB_CUDA(cudaStreamSynchronize(st));
  n_ += n;
  return 0;
}
int RawStore::append_device(const float* x, int64_t ld, int64_t n, cudaStream_t st) {
  if (ensure(n_ + n)) return -1;
  int64_t done = 0;
  while (done < n) {
    int64_t vid = n_ + done;
    int64_t si = vid >> seg_shift_, off = vid & (seg_rows() - 1);
    int64_t cnt = std::min(n - done, seg_rows() - off);
    GB_CUDA(cudaMemcpy2DAsync(segs_[si].base + off * dpad_, (size_t)dpad_ * 4, x + done * ld, (size_t)ld * 4,
                              (size_t)d_ * 4, (size_t)cnt, cudaMemcpyDeviceToDevice, st));
    done += cnt;
  }
  GB_CUDA(cudaStreamSynchronize(st));
  n_ += n;
  return 0;
}
int RawStore::update_host(int64_t vid, const float* x, cudaStream_t st) {
  if (vid < 0 || vid >= n_) return -1;
  int64_t si = vid >> seg_shift_, off = vid & (seg_rows() - 1);
  GB_CUDA(cudaMemcpyAsync(segs_[si].base + off * dpad_, x, (size_t)d_ * 4, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}
int RawStore::get_host(int64_t vid, float* out) const {
  if (vid < 0 || vid >= n_) return -1;
  int64_t si = vid >> seg_shift_, off = vid & (seg_rows() - 1);
  GB_CUDA(cudaMemcpy(out, segs_[si].base + off * dpad_, (size_t)d_ * 4, cudaMemcpyDeviceToHost));
  return 0;
}
int RawStore::get_rows_host(int64_t start, int64_t n, float* out) const {
  if (start < 0 || n < 0 || start + n > n_) return -1;
  int64_t done = 0;
  while (done < n) {
    int64_t vid = start + done;
    int64_t si = vid >> seg_shift_, off = vid & (seg_rows() - 1);
    int64_t cnt = std::min(n - done, seg_rows() - off);
    GB_CUDA(cudaMemcpy2D(out + done * d_, (size_t)d_ * 4, segs_[si].base + off * dpad_, (size_t)dpad_ * 4, (size_t)d_ * 4,
                         (size_t)cnt, cudaMemcpyDeviceToHost));
    done += cnt;
  }
  return 0;
}
const float* RawStore::contiguous(int64_t n, Scratch& s) {
  if (n <= seg_rows()) return segs_.empty() ? nullptr : segs_[0].base;
  float* buf = s.alloc_n<float>((size_t)n * dpad_);
  if (!buf) return nullptr;
  int64_t done = 0;
  while (done < n) {
    int64_t si = done >> seg_shift_;
    int64_t cnt = std::min(n - done, seg_rows());
    if (cudaMemcpyAsync(buf + done * dpad_, segs_[si].base, (size_t)cnt * dpad_ * 4, cudaMemcpyDeviceToDevice,
                        s.stream()) != cudaSuccess)
      return nullptr;
    done += cnt;
  }
  return buf;
}

// ------------------------------------------------------------------------------------------
static std::atomic<uint64_t> g_lists_uid{1};
IvfLists::IvfLists(int nlist, int code_bytes) : nlist_(nlist), code_bytes_(code_bytes), uid_(g_lists_uid.fetch_add(1)) {
  h_data_.assign(nlist, nullptr);
  h_ids_.assign(nlist, nullptr);
  h_len_.assign(nlist, 0);
  h_cap_.assign(nlist, 0);
  cudaMalloc(&d_data_, sizeof(void*) * nlist);
  cudaMalloc(&d_ids_, sizeof(int64_t*) * nlist);
  cudaMalloc(&d_len_, sizeof(int) * nlist);
  cudaMemset(d_data_, 0, sizeof(void*) * nlist);
  cudaMemset(d_ids_, 0, sizeof(int64_t*) * nlist);
  cudaMemset(d_len_, 0, sizeof(int) * nlist);
}
IvfLists::~IvfLists() {
  for (void* p : slabs_) cudaFree(p);
  cudaFree(d_data_);
  cudaFree(d_ids_);
  cudaFree(d_len_);
}
ListDirectory IvfLists::directory() const {
  ListDirectory dir;
  dir.vecs = reinterpret_cast<const float* const*>(d_data_);
  dir.codes = reinterpret_cast<const uint8_t* const*>(d_data_);
  dir.ids = reinterpret_cast<const int64_t* const*>(d_ids_);
  dir.len = d_len_;
  dir.nlist = nlist_;
  return dir;
}
void* IvfLists::slab_alloc(size_t bytes) {
  bytes = (size_t)round_up((int64_t)bytes, 256);
  if (bytes > slab_left_) return nullptr;
  void* p = slab_cur_;
  slab_cur_ += bytes;
  slab_left_ -= bytes;
  return p;
}
int IvfLists::reserve(const std::vector<int>& add, cudaStream_t st) {
  // pass 1: how many bytes do the growing lists need
  std::vector<int> newcap(nlist_, 0);
  size_t need_bytes = 0;
  for (int l = 0; l < nlist_; l++) {
    if (add[l] <= 0) continue;
    int64_t need = (int64_t)h_len_[l] + add[l];
    if (need <= h_cap_[l]) continue;
    // growth policy: at least x1.5 (reference grows by 1.1 + pi/2 - atan(n), realtime_mem_data.cc:110-113)
    int64_t nc = std::max<int64_t>(need, (int64_t)h_cap_[l] * 3 / 2);
    nc = round_up(nc, 32);
    if (nc > INT32_MAX) {
      set_last_error("inverted list too long");
      return -1;
    }
    newcap[l] = (int)nc;
    need_bytes += (size_t)round_up(nc * code_bytes_ + 16, 256) + (size_t)round_up(nc * 8, 256);
  }
  if (need_bytes == 0) return 0;
  if (need_bytes > slab_left_) {
    size_t slab = std::max<size_t>(need_bytes, (size_t)64 << 20);
    void* p = nullptr;
    GB_CUDA(cudaMalloc(&p, slab));
    slabs_.push_back(p);
    slab_cur_ = static_cast<char*>(p);
    slab_left_ = slab;
    bytes_ += (int64_t)slab;
  }
  for (int l = 0; l < nlist_; l++) {
    if (!newcap[l]) continue;
    void* nd = slab_alloc((size_t)newcap[l] * code_bytes_ + 16);
    int64_t* ni = static_cast<int64_t*>(slab_alloc((size_t)newcap[l] * 8));
    if (!nd || !ni) {
      set_last_error("slab exhausted");
      return -1;
    }
    if (h_len_[l] > 0) {  // copy-on-grow; the old region stays valid for in-flight searches
      GB_CUDA(cudaMemcpyAsync(nd, h_data_[l], (size_t)h_len_[l] * code_bytes_, cudaMemcpyDeviceToDevice, st));
      GB_CUDA(cudaMemcpyAsync(ni, h_ids_[l], (size_t)h_len_[l] * 8, cudaMemcpyDeviceToDevice, st));
    }
    h_data_[l] = nd;
    h_ids_[l] = ni;
    h_cap_[l] = newcap[l];
  }
  GB_CUDA(cudaMemcpyAsync(d_data_, h_data_.data(), sizeof(void*) * nlist_, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(d_ids_, h_ids_.data(), sizeof(int64_t*) * nlist_, cudaMemcpyHostToDevice, st));
  return 0;
}
int IvfLists::commit(const std::vector<int>& add, cudaStream_t st) {
  for (int l = 0; l < nlist_; l++) {
    h_len_[l] += add[l];
    total_ += add[l];
    if (h_len_[l] > max_len_) max_len_ = h_len_[l];
  }
  // length is published after the data (realtime_mem_data.cc:292-293): same stream, later op
  GB_CUDA(cudaMemcpyAsync(d_len_, h_len_.data(), sizeof(int) * nlist_, cudaMemcpyHostToDevice, st));
  return 0;
}
int64_t IvfLists::packed_bytes() const {
  int64_t b = 0;
  for (int l = 0; l < nlist_; l++) {
    if (h_len_[l] == 0) continue;
    const int64_t cap = round_up(h_len_[l], 32);
    b += round_up(cap * code_bytes_ + 16, 256) + round_up(cap * 8, 256);
  }
  return b;
}
int IvfLists::compact(cudaStream_t st) {
  const int64_t need = packed_bytes();
  if (need == 0 || slabs_.empty()) return 0;
  void* slab = nullptr;
  if (cudaMalloc(&slab, (size_t)need) != cudaSuccess) {
    cudaGetLastError();
    return 0;  // not enough room to re-pack: keep the current layout
  }
  char* cur = static_cast<char*>(slab);
  for (int l = 0; l < nlist_; l++) {
    if (h_len_[l] == 0) {
      h_data_[l] = nullptr, h_ids_[l] = nullptr, h_cap_[l] = 0;
      continue;
    }
    const int64_t cap = round_up(h_len_[l], 32);
    void* nd = cur;
    cur += round_up(cap * code_bytes_ + 16, 256);
    int64_t* ni = reinterpret_cast<int64_t*>(cur);
    cur += round_up(cap * 8, 256);
    GB_CUDA(cudaMemcpyAsync(nd, h_data_[l], (size_t)h_len_[l] * code_bytes_, cudaMemcpyDeviceToDevice, st));
    GB_CUDA(cudaMemcpyAsync(ni, h_ids_[l], (size_t)h_len_[l] * 8, cudaMemcpyDeviceToDevice, st));
    h_data_[l] = nd, h_ids_[l] = ni, h_cap_[l] = (int)cap;
  }
  GB_CUDA(cudaMemcpyAsync(d_data_, h_data_.data(), sizeof(void*) * nlist_, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(d_ids_, h_ids_.data(), sizeof(int64_t*) * nlist_, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaDeviceSynchronize());  // copies done, and no kernel of an earlier search still reads the old slabs
  for (void* p : slabs_) cudaFree(p);
  slabs_.assign(1, slab);
  slab_cur_ = nullptr;
  slab_left_ = 0;
  bytes_ = need;
  return 0;
}
int IvfLists::tombstone(int list, int pos, cudaStream_t st) {
  if (list < 0 || list >= nlist_ || pos < 0 || pos >= h_len_[list]) return -1;
  int64_t v;
  GB_CUDA(cudaMemcpyAsync(&v, h_ids_[list] + pos, 8, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  v |= kDelIdxMask;
  GB_CUDA(cudaMemcpyAsync(h_ids_[list] + pos, &v, 8, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}
int IvfLists::download_list(int l, std::vector<uint8_t>* codes, std::vector<int64_t>* ids) const {
  if (l < 0 || l >= nlist_) return -1;
  int len = h_len_[l];
  if (codes) {
    codes->resize((size_t)len * code_bytes_);
    if (len) GB_CUDA(cudaMemcpy(codes->data(), h_data_[l], codes->size(), cudaMemcpyDeviceToHost));
  }
  if (ids) {
    ids->resize(len);
    if (len) GB_CUDA(cudaMemcpy(ids->data(), h_ids_[l], (size_t)len * 8, cudaMemcpyDeviceToHost));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
namespace {
struct LiveIndexes {
  std::mutex mu;
  std::vector<Index*> all;
};
LiveIndexes& live_indexes() {
  static LiveIndexes* s = new LiveIndexes;  // leaked on purpose: must outlive every static destructor
  return *s;
}
void quiesce_all_indexes() {
  std::vector<Index*> v;
  {
    std::lock_guard<std::mutex> g(live_indexes().mu);
    v = live_indexes().all;
  }
  for (Index* i : v) i->quiesce();
}
}  // namespace

Index::Index(const std::string& type, int d, const ModelParams& mp, int device, int seg_shift)
    : type_(type), d_(d), dpad_((int)round_up(d, 4)), device_(device), mp_(mp) {
  cudaSetDevice(device_);
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device_) == cudaSuccess) {
    uint64_t thr = UINT64_MAX;  // keep scratch memory cached between searches
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  {  // the CUDA runtime is initialised by now, so this hook runs before its teardown
    std::lock_guard<std::mutex> g(live_indexes().mu);
    static bool hooked = (atexit(quiesce_all_indexes), true);
    (void)hooked;
    live_indexes().all.push_back(this);
  }
  store_.reset(new RawStore(d, seg_shift));
  cudaStreamCreateWithFlags(&build_stream_, cudaStreamNonBlocking);
}
void Index::quiesce() {
  {
    std::lock_guard<std::mutex> lk(co_mu_);
    co_stop_ = true;
  }
  co_cv_.notify_all();
  if (co_thread_.joinable()) co_thread_.join();
}

Index::~Index() {
  drain_searches();
  {
    std::lock_guard<std::mutex> g(live_indexes().mu);
    auto& a = live_indexes().all;
    a.erase(std::remove(a.begin(), a.end(), this), a.end());
  }
  quiesce();
  for (auto& b : big_) {
    cudaFree(b.p);
    cudaEventDestroy(b.done);
  }
  if (build_stream_) cudaStreamDestroy(build_stream_);
}
void* Index::big_acquire(size_t bytes, cudaStream_t st) {
  std::lock_guard<std::mutex> g(big_mu_);
  int best = -1;
  for (size_t i = 0; i < big_.size(); i++)
    if (!big_[i].busy && big_[i].cap >= bytes && (best < 0 || big_[i].cap < big_[best].cap)) best = (int)i;
  if (best < 0) {
    for (size_t i = 0; i < big_.size();) {  // drop idle buffers that are too small before growing
      if (!big_[i].busy) {
        cudaEventSynchronize(big_[i].done);
        cudaFree(big_[i].p);
        cudaEventDestroy(big_[i].done);
        big_.erase(big_.begin() + i);
      } else {
        i++;
      }
    }
    BigBuf b;
    b.cap = bytes + bytes / 4;
    b.busy = false;
    if (cudaMalloc(&b.p, b.cap) != cudaSuccess) {
      b.cap = bytes;
      if (cudaMalloc(&b.p, b.cap) != cudaSuccess) {
        set_last_error("cudaMalloc(" + std::to_string(bytes) + ") failed for scan scratch");
        return nullptr;
      }
    }
    cudaEventCreateWithFlags(&b.done, cudaEventDisableTiming);
    cudaEventRecord(b.done, st);
    big_.push_back(b);
    best = (int)big_.size() - 1;
  }
  big_[best].busy = true;
  cudaStreamWaitEvent(st, big_[best].done, 0);  // previous user's kernels (possibly on another stream)
  return big_[best].p;
}
void Index::big_release(void* p, cudaStream_t st) {
  std::lock_guard<std::mutex> g(big_mu_);
  for (auto& b : big_)
    if (b.p == p) {
      cudaEventRecord(b.done, st);
      b.busy = false;
    }
}
void Index::note_search_enqueued(cudaStream_t st) {
  cudaEvent_t e;
  if (cudaEventCreateWithFlags(&e, cudaEventDisableTiming) != cudaSuccess) return;
  cudaEventRecord(e, st);
  std::lock_guard<std::mutex> g(inflight_mu_);
  if (inflight_.size() >= 64) {  // forget the ones that have completed
    size_t w = 0;
    for (size_t i = 0; i < inflight_.size(); i++) {
      if (cudaEventQuery(inflight_[i]) == cudaSuccess)
        cudaEventDestroy(inflight_[i]);
      else
        inflight_[w++] = inflight_[i];
    }
    inflight_.resize(w);
    cudaGetLastError();  // cudaErrorNotReady from the queries is not an error
  }
  inflight_.push_back(e);
}
void Index::drain_searches() {
  std::lock_guard<std::mutex> g(inflight_mu_);
  for (cudaEvent_t e : inflight_) {
    cudaEventSynchronize(e);
    cudaEventDestroy(e);
  }
  inflight_.clear();
}
void Index::scan_timer_begin(cudaStream_t st) {
  if (!time_scan_) return;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  cudaEventRecord(e0, st);
  std::lock_guard<std::mutex> g(ev_mu_);
  scan_events_.emplace_back(e0, e1);
}
void Index::scan_timer_end(cudaStream_t st) {
  if (!time_scan_) return;
  std::lock_guard<std::mutex> g(ev_mu_);
  if (!scan_events_.empty()) cudaEventRecord(scan_events_.back().second, st);
}
void Index::stage_begin(const char* name, cudaStream_t st) {
  if (!time_scan_) return;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  cudaEventRecord(e0, st);
  std::lock_guard<std::mutex> g(ev_mu_);
  stage_events_.push_back({name, e0, e1});
}
void Index::stage_end(cudaStream_t st) {
  if (!time_scan_) return;
  std::lock_guard<std::mutex> g(ev_mu_);
  if (!stage_events_.empty()) cudaEventRecord(stage_events_.back().e1, st);
}
std::vector<std::pair<std::string, float>> Index::stage_times() {
  std::lock_guard<std::mutex> g(ev_mu_);
  std::vector<std::pair<std::string, float>> out;
  for (auto& ev : stage_events_) {
    float ms = 0.f;
    if (cudaEventSynchronize(ev.e1) != cudaSuccess || cudaEventElapsedTime(&ms, ev.e0, ev.e1) != cudaSuccess) ms = 0.f;
    cudaEventDestroy(ev.e0);
    cudaEventDestroy(ev.e1);
    bool found = false;
    for (auto& o : out)
      if (o.first == ev.name) o.second += ms, found = true;
    if (!found) out.emplace_back(ev.name, ms);
  }
  stage_events_.clear();
  return out;
}
float Index::last_scan_ms() {
  std::lock_guard<std::mutex> g(ev_mu_);
  float total = 0.f;
  for (auto& ev : scan_events_) {
    float ms = 0.f;
    if (cudaEventSynchronize(ev.second) == cudaSuccess && cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess)
      total += ms;
    cudaEventDestroy(ev.first);
    cudaEventDestroy(ev.second);
  }
  scan_events_.clear();
  return total;
}
int Index::add_vectors(const float* x, int64_t n) {
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  return store_->append_host(x, n, build_stream_);
}
int Index::add_vectors_device(const float* x, int64_t ld, int64_t n) {
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  return store_->append_device(x, ld, n, build_stream_);
}

int Index::upload_bitmaps(const SearchContext& ctx, FilterArgs* f, Scratch& s) {
  f->del_bits = nullptr;
  f->filter_bits = nullptr;
  f->min_score = ctx.min_score;
  f->max_score = ctx.max_score;
  // the kernels index bitmaps by vid; pad to cover every stored vector
  int64_t bits = std::max<int64_t>(ctx.bitmap_bits, store_->size());
  size_t words = (size_t)((bits + 31) / 32) + 1;
  size_t have = (size_t)((ctx.bitmap_bits + 7) / 8);
  for (int which = 0; which < 2; which++) {
    const uint8_t* src = which == 0 ? ctx.del_bitmap : ctx.filter_bitmap;
    if (!src) continue;
    uint32_t* dev = s.alloc_n<uint32_t>(words);
    if (!dev) return -1;
    // ids beyond the caller's bitmap: not deleted / not allowed
    GB_CUDA(cudaMemsetAsync(dev, 0, words * 4, s.stream()));
    GB_CUDA(cudaMemcpyAsync(dev, src, have, cudaMemcpyHostToDevice, s.stream()));
    if (which == 0)
      f->del_bits = dev;
    else
      f->filter_bits = dev;
  }
  return 0;
}

int Index::search_device(const SearchContext& ctx, int nq, const float* x_dev, int64_t ldx, int k, float* out_dis_dev,
                         int64_t* out_ids_dev, cudaStream_t st, unsigned long long* out_keys_dev) {
  if (nq <= 0) return 0;
  if (k <= 0 || k > 4096) {
    set_last_error("topK must be in [1, 4096]");
    return -1;
  }
  cudaSetDevice(device_);
  std::shared_lock<std::shared_mutex> lk(mu_);
  Scratch s(st);
  const float* xq = x_dev;
  int64_t ldq = ldx;
  if ((ldx & 3) || (reinterpret_cast<uintptr_t>(x_dev) & 15)) {  // re-pack into 16-byte aligned rows
    float* buf = s.alloc_n<float>((size_t)nq * dpad_);
    if (!buf) return -1;
    GB_CUDA(cudaMemsetAsync(buf, 0, (size_t)nq * dpad_ * 4, st));
    GB_CUDA(cudaMemcpy2DAsync(buf, (size_t)dpad_ * 4, x_dev, (size_t)ldx * 4, (size_t)d_ * 4, nq,
                              cudaMemcpyDeviceToDevice, st));
    xq = buf;
    ldq = dpad_;
  } else if (ldx < dpad_) {
    set_last_error("query row stride smaller than padded dimension");
    return -1;
  }
  FilterArgs f;
  if (upload_bitmaps(ctx, &f, s)) return -1;
  int metric = ctx.params.metric >= 0 ? ctx.params.metric : mp_.metric;
  GB_ALLOC(keys, unsigned long long, (size_t)nq * k, s);
  // the device kernels take a dense nq x dpad block
  if (ldq != dpad_) {
    float* buf = s.alloc_n<float>((size_t)nq * dpad_);
    if (!buf) return -1;
    GB_CUDA(cudaMemcpy2DAsync(buf, (size_t)dpad_ * 4, xq, (size_t)ldq * 4, (size_t)dpad_ * 4, nq,
                              cudaMemcpyDeviceToDevice, st));
    xq = buf;
  }
  int rc;
  if (ctx.params.brute_force || !trained_) {
    // brute-force fallback of the IVF models (gamma_index_ivfflat.cc:541-550, ivfpq.cc:561-570)
    rc = flat_search_dev(ctx, f, metric, nq, xq, k, store_->size(), keys, s);
  } else {
    rc = search_keys_dev(ctx, f, metric, nq, xq, k, keys, s);
    // enable_realtime (vector_manager.cc:854-889, 971-1053): vectors stored but not yet indexed are
    // searched brute-force (the reference's MemoryBuffer FLAT index) and merged by score
    const int64_t tail0 = indexed_count_, tail1 = store_->size();
    if (rc == 0 && ctx.search_unindexed_tail && tail1 > tail0) {
      GB_ALLOC(both, unsigned long long, (size_t)nq * 2 * k, s);
      GB_CUDA(cudaMemcpy2DAsync(both, (size_t)2 * k * 8, keys, (size_t)k * 8, (size_t)k * 8, nq,
                                cudaMemcpyDeviceToDevice, st));
      GB_ALLOC(tailk, unsigned long long, (size_t)nq * k, s);
      rc = flat_search_dev(ctx, f, metric, nq, xq, k, tail1, tailk, s, tail0);
      if (rc == 0) {
        GB_CUDA(cudaMemcpy2DAsync(both + k, (size_t)2 * k * 8, tailk, (size_t)k * 8, (size_t)k * 8, nq,
                                  cudaMemcpyDeviceToDevice, st));
        GB_CUDA(launch_select_keys(both, (int64_t)2 * k, nq, 2 * k, k, keys, k, st));
      }
    }
  }
  if (rc) {
    note_search_enqueued(st);
    return rc;
  }
  if (out_keys_dev) GB_CUDA(cudaMemcpyAsync(out_keys_dev, keys, (size_t)nq * k * 8, cudaMemcpyDeviceToDevice, st));
  if (out_dis_dev && out_ids_dev) GB_CUDA(launch_decode_keys(keys, k, nq, k, metric, out_dis_dev, out_ids_dev, 0, st));
  note_search_enqueued(st);
  return 0;
}

static bool coalesce_enabled() {
  static int v = [] {
    const char* e = getenv("GB_COALESCE");
    return e ? atoi(e) : 1;
  }();
  return v != 0;
}
static constexpr int kCoalesceMaxNq = 16;     // requests at most this large are merged
static constexpr int kCoalesceMaxBatch = 512;  // queries per merged device batch (reference kMaxBatch)

bool Index::coalescable(const SearchContext& ctx, int nq) const {
  return coalesce_enabled() && nq <= kCoalesceMaxNq && !ctx.del_bitmap && !ctx.filter_bitmap;
}

static bool same_signature(const SearchContext& a, int ka, const SearchContext& b, int kb) {
  return ka == kb && a.min_score == b.min_score && a.max_score == b.max_score && a.params.nprobe == b.params.nprobe &&
         a.params.metric == b.params.metric && a.params.recall_num == b.params.recall_num &&
         a.params.brute_force == b.params.brute_force && a.search_unindexed_tail == b.search_unindexed_tail &&
         a.params.qb == b.params.qb && a.params.centered == b.params.centered;
}

void Index::coalesce_loop() {
  cudaSetDevice(device_);
  std::vector<CoReq*> batch;
  std::vector<float> xs, dd;
  std::vector<int64_t> ii;
  for (;;) {
    batch.clear();
    {
      std::unique_lock<std::mutex> lk(co_mu_);
      co_cv_.wait(lk, [this] { return co_stop_ || !co_queue_.empty(); });
      if (co_stop_ && co_queue_.empty()) return;
      CoReq* first = co_queue_.front();
      int total = 0;
      for (size_t i = 0; i < co_queue_.size();) {  // whatever piled up while the previous batch ran
        CoReq* r = co_queue_[i];
        if (total + r->nq <= kCoalesceMaxBatch && same_signature(*first->ctx, first->k, *r->ctx, r->k)) {
          batch.push_back(r);
          total += r->nq;
          co_queue_.erase(co_queue_.begin() + i);
        } else {
          i++;
        }
      }
    }
    int total = 0;
    for (CoReq* r : batch) total += r->nq;
    const int k = batch[0]->k;
    int rc;
    if (batch.size() == 1) {
      rc = search_direct(*batch[0]->ctx, batch[0]->nq, batch[0]->x, k, batch[0]->out_dis, batch[0]->out_ids);
    } else {
      xs.resize((size_t)total * d_);
      dd.resize((size_t)total * k);
      ii.resize((size_t)total * k);
      size_t o = 0;
      for (CoReq* r : batch) {
        memcpy(xs.data() + o * d_, r->x, (size_t)r->nq * d_ * 4);
        o += r->nq;
      }
      rc = search_direct(*batch[0]->ctx, total, xs.data(), k, dd.data(), ii.data());
      o = 0;
      for (CoReq* r : batch) {
        if (rc == 0) {
          memcpy(r->out_dis, dd.data() + o * k, (size_t)r->nq * k * 4);
          memcpy(r->out_ids, ii.data() + o * k, (size_t)r->nq * k * 8);
        }
        o += r->nq;
      }
    }
    std::string err = rc ? last_error() : "";
    {
      std::lock_guard<std::mutex> lk(co_mu_);
      for (CoReq* r : batch) {
        r->rc = rc;
        r->err = err;
        r->done = true;
      }
    }
    co_done_cv_.notify_all();
  }
}

int Index::search(const SearchContext& ctx, int nq, const float* x, int k, float* out_dis, int64_t* out_ids) {
  if (nq <= 0) return 0;
  if (!coalescable(ctx, nq)) return search_direct(ctx, nq, x, k, out_dis, out_ids);
  CoReq req;
  req.ctx = &ctx, req.nq = nq, req.k = k, req.x = x, req.out_dis = out_dis, req.out_ids = out_ids;
  {
    std::unique_lock<std::mutex> lk(co_mu_);
    if (!co_started_) {
      co_started_ = true;
      co_thread_ = std::thread(&Index::coalesce_loop, this);
    }
    co_queue_.push_back(&req);
    co_cv_.notify_one();
    co_done_cv_.wait(lk, [&req] { return req.done; });
  }
  if (req.rc) set_last_error(req.err);
  return req.rc;
}

int Index::search_direct(const SearchContext& ctx, int nq, const float* x, int k, float* out_dis, int64_t* out_ids) {
  if (nq <= 0) return 0;
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  float* dq = nullptr;
  float* dd = nullptr;
  int64_t* di = nullptr;
  int rc = -1;
  do {
    if (cudaMallocAsync(&dq, (size_t)nq * dpad_ * 4, st) != cudaSuccess) break;
    if (cudaMallocAsync(&dd, (size_t)nq * k * 4, st) != cudaSuccess) break;
    if (cudaMallocAsync(&di, (size_t)nq * k * 8, st) != cudaSuccess) break;
    if (d_ != dpad_ && cudaMemsetAsync(dq, 0, (size_t)nq * dpad_ * 4, st) != cudaSuccess) break;
    if (cudaMemcpy2DAsync(dq, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, nq, cudaMemcpyHostToDevice, st) !=
        cudaSuccess)
      break;
    rc = search_device(ctx, nq, dq, dpad_, k, dd, di, st);
    if (rc) break;
    rc = -1;
    if (cudaMemcpyAsync(out_dis, dd, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
    if (cudaMemcpyAsync(out_ids, di, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, st) != cudaSuccess) break;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
      set_last_error(std::string("search: ") + cudaGetErrorString(e));
      break;
    }
    rc = 0;
  } while (0);
  if (rc == -1 && !*last_error()) set_last_error(std::string("search: ") + cudaGetErrorString(cudaGetLastError()));
  if (dq) cudaFreeAsync(dq, st);
  if (dd) cudaFreeAsync(dd, st);
  if (di) cudaFreeAsync(di, st);
  return rc;
}

// GammaFLATIndex::Search (gamma_index_flat.cc:130-370): every stored row, filters before top-k.
int Index::flat_search_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                           int64_t nrows, unsigned long long* out_keys, Scratch& s, int64_t row_begin) {
  (void)ctx;
  cudaStream_t st = s.stream();
  const int64_t flat_row_begin_ = row_begin;
  if (nrows <= row_begin) return launch_fill_u64(out_keys, (int64_t)nq * k, kKeySentinel, st) == cudaSuccess ? 0 : -1;
  const int64_t CC = std::min<int64_t>(131072, store_->seg_rows());  // DB rows per distance block
  struct Chunk {
    const float* base;
    int64_t id0;
    int cnt;
  };
  std::vector<Chunk> chunks;
  for (int64_t r = flat_row_begin_; r < nrows;) {
    int64_t si = r >> store_->seg_shift(), off = r & (store_->seg_rows() - 1);
    int64_t cnt = std::min<int64_t>(std::min(nrows - r, store_->seg_rows() - off), CC);
    chunks.push_back({store_->seg((int)si) + off * dpad_, r, (int)cnt});
    r += cnt;
  }
  const int nch = (int)chunks.size();
  int64_t ldo = round_up(std::min<int64_t>(CC, nrows - row_begin), 4);
  int QB = (int)std::max<int64_t>(1, std::min<int64_t>(nq, ((int64_t)1 << 28) / ldo));  // <= 1 GiB of scores
  GB_ALLOC(scores, float, (size_t)QB * ldo, s);
  unsigned long long* partial = out_keys;
  if (nch > 1) {
    partial = s.alloc_n<unsigned long long>((size_t)nq * nch * k);
    if (!partial) return -1;
  }
  last_scan_kernel_ = "dist_tile_kernel+select_rows_kernel";
  scan_timer_begin(st);
  for (int q0 = 0; q0 < nq; q0 += QB) {
    int qb = std::min(QB, nq - q0);
    for (int c = 0; c < nch; c++) {
      GB_CUDA(launch_dist_matrix(xq + (int64_t)q0 * dpad_, dpad_, qb, chunks[c].base, dpad_, chunks[c].cnt, dpad_,
                                 metric, scores, ldo, st));
      GB_CUDA(launch_select_scores(scores, ldo, qb, chunks[c].cnt, chunks[c].id0, k, metric, f,
                                   partial + ((int64_t)q0 * nch + c) * k, (int64_t)nch * k, st));
    }
  }
  if (nch > 1) GB_CUDA(launch_select_keys(partial, (int64_t)nch * k, nq, nch * k, k, out_keys, k, st));
  scan_timer_end(st);
  return 0;
}

int FlatIndex::search_keys_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                               unsigned long long* out_keys, Scratch& s) {
  return flat_search_dev(ctx, f, metric, nq, xq, k, store_->size(), out_keys, s);
}

// ------------------------------------------------------------------------------------------
// k-means (faiss::Clustering restated, SURVEY Appendix A).  Assign runs on device (K2 kernel with
// fused argmin), the centroid update is a deterministic segmented mean on device, the control
// logic (seeded permutations, empty-cluster split) runs on host.
static void rand_perm_mt(std::vector<int32_t>& perm, int64_t n, int64_t seed) {
  perm.resize(n);
  for (int64_t i = 0; i < n; i++) perm[i] = (int32_t)i;
  std::mt19937 mt((unsigned)seed);
  for (int64_t i = 0; i + 1 < n; i++) {
    int64_t i2 = i + (int64_t)(mt() % (uint32_t)(n - i));
    std::swap(perm[i], perm[i2]);
  }
}

int kmeans_device(const float* x_in, int64_t ldx_in, int64_t n_in, int d, int k, const KMeansParams& kp,
                  float* centroids, int64_t ldc, cudaStream_t st, std::vector<float>* obj) {
  if (n_in < k) {
    set_last_error("kmeans: fewer training points than centroids");
    return -1;
  }
  if (n_in > INT32_MAX) {
    set_last_error("kmeans: too many points");
    return -1;
  }
  Scratch s(st);
  const int dpad = (int)round_up(d, 4);
  const float* x = x_in;
  int64_t ldx = ldx_in, n = n_in;
  std::vector<int32_t> perm;
  if (kp.max_points_per_centroid > 0 && n_in > (int64_t)k * kp.max_points_per_centroid) {
    n = (int64_t)k * kp.max_points_per_centroid;
    rand_perm_mt(perm, n_in, kp.seed);
    GB_ALLOC(d_idx, int32_t, n, s);
    GB_CUDA(cudaMemcpyAsync(d_idx, perm.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    GB_ALLOC(xs, float, (size_t)n * dpad, s);
    GB_CUDA(launch_gather_rows(x_in, ldx_in, d_idx, n, d, xs, dpad, st));
    GB_CUDA(cudaStreamSynchronize(st));
    x = xs;
    ldx = dpad;
  }
  // initial centroids = first k entries of a seeded permutation (or the caller's, for a hot start)
  GB_ALLOC(d_perm, int32_t, n, s);
  GB_ALLOC(d_off, int32_t, k + 1, s);
  if (!kp.hot_start) {
    rand_perm_mt(perm, n, kp.seed + 1);
    GB_CUDA(cudaMemcpyAsync(d_perm, perm.data(), (size_t)k * 4, cudaMemcpyHostToDevice, st));
    GB_CUDA(launch_gather_rows(x, ldx, d_perm, k, d, centroids, ldc, st));
    if (kp.spherical) GB_CUDA(launch_normalize_rows(centroids, ldc, k, d, st));
  }
  GB_CUDA(cudaStreamSynchronize(st));

  GB_ALLOC(best, unsigned long long, n, s);
  std::vector<unsigned long long> h_best(n);
  std::vector<int32_t> h_off(k + 1), h_perm(n), cursor(k);
  std::vector<float> hassign(k), h_cent;
  const int metric = kp.spherical ? kMetricIP : kMetricL2;  // gamma's quantizer is IndexFlat(d, metric)
  const bool use_tc = tc_enabled() && k >= 64;
  for (int it = 0; it < kp.niter; it++) {
    GB_CUDA(launch_fill_u64(best, n, kKeySentinel, st));
    if (use_tc) {
      GB_CUDA(launch_dist_argmin_tc(x, ldx, (int)n, centroids, ldc, k, dpad, metric, best, st));
    } else {
      GB_CUDA(launch_dist_argmin(x, ldx, (int)n, centroids, ldc, k, dpad, metric, best, 0, st));
    }
    GB_CUDA(cudaMemcpyAsync(h_best.data(), best, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaStreamSynchronize(st));
    // stable counting sort of the points by label (point order inside a cluster = faiss's sum order)
    std::fill(h_off.begin(), h_off.end(), 0);
    double o = 0;
    for (int64_t i = 0; i < n; i++) {
      if ((uint32_t)h_best[i] >= (uint32_t)k) h_best[i] &= 0xFFFFFFFF00000000ull;  // NaN rows -> cluster 0
      h_off[(uint32_t)h_best[i] + 1]++;
      if (obj) o += ord2score((uint32_t)(h_best[i] >> 32), metric);
    }
    if (obj) obj->push_back((float)o);
    for (int c = 0; c < k; c++) {
      hassign[c] = (float)h_off[c + 1];
      h_off[c + 1] += h_off[c];
      cursor[c] = h_off[c];
    }
    for (int64_t i = 0; i < n; i++) h_perm[cursor[(uint32_t)h_best[i]]++] = (int32_t)i;
    GB_CUDA(cudaMemcpyAsync(d_perm, h_perm.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    GB_CUDA(cudaMemcpyAsync(d_off, h_off.data(), (size_t)(k + 1) * 4, cudaMemcpyHostToDevice, st));
    GB_CUDA(launch_segment_mean(x, ldx, d, d_perm, d_off, k, centroids, ldc, st));
    // split_clusters: re-seed empty clusters from big ones (EPS = 1/1024, rng(1234))
    bool any_empty = false;
    for (int c = 0; c < k; c++) any_empty |= (hassign[c] == 0);
    if (any_empty) {
      h_cent.resize((size_t)k * ldc);
      GB_CUDA(cudaMemcpyAsync(h_cent.data(), centroids, (size_t)k * ldc * 4, cudaMemcpyDeviceToHost, st));
      GB_CUDA(cudaStreamSynchronize(st));
      const float EPS = 1.0f / 1024.0f;
      std::mt19937 rng(1234u);
      for (int ci = 0; ci < k; ci++) {
        if (hassign[ci] != 0) continue;
        int cj;
        for (cj = 0;; cj = (cj + 1) % k) {
          float p = (hassign[cj] - 1.0f) / (float)(n - k);
          float r = (float)rng() / (float)4294967295u;
          if (r < p) break;
        }
        float* a = h_cent.data() + (size_t)ci * ldc;
        float* b = h_cent.data() + (size_t)cj * ldc;
        memcpy(a, b, sizeof(float) * d);
        for (int j = 0; j < d; j++) {
          if (j % 2 == 0) {
            a[j] *= 1 + EPS;
            b[j] *= 1 - EPS;
          } else {
            a[j] *= 1 - EPS;
            b[j] *= 1 + EPS;
          }
        }
        hassign[ci] = hassign[cj] / 2;
        hassign[cj] -= hassign[ci];
      }
      GB_CUDA(cudaMemcpyAsync(centroids, h_cent.data(), (size_t)k * ldc * 4, cudaMemcpyHostToDevice, st));
    }
    if (kp.spherical) GB_CUDA(launch_normalize_rows(centroids, ldc, k, d, st));
    GB_CUDA(cudaStreamSynchronize(st));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
IVFFlatIndex::IVFFlatIndex(int d, const ModelParams& mp, int device, int seg_shift, const std::string& type)
    : Index(type, d, mp, device, seg_shift), nlist_(mp.ncentroids) {
  cudaMalloc(&d_centroids_, (size_t)nlist_ * dpad_ * 4);
  cudaMemset(d_centroids_, 0, (size_t)nlist_ * dpad_ * 4);
}
IVFFlatIndex::~IVFFlatIndex() {
  if (mirror_.base) cudaFree(mirror_.base);
  if (mirror_.norms) cudaFree(mirror_.norms);
  if (mirror_.d_tile0) cudaFree(mirror_.d_tile0); cudaFree(d_centroids_); }

int IVFFlatIndex::training_threshold() const {
  // gamma_index_ivfflat.cc:239: default nlist * 200 ; Indexing() clamps to [39, 256] * nlist (:350-375)
  int64_t t = mp_.training_threshold ? mp_.training_threshold : (int64_t)nlist_ * 200;
  if (t < nlist_)
    t = (int64_t)nlist_ * 39;
  else if (t > (int64_t)nlist_ * 256)
    t = (int64_t)nlist_ * 256;
  return (int)t;
}
int64_t IVFFlatIndex::index_mem_bytes() const {
  const int64_t mirror = mirror_.cap_tiles * (tc_mirror_tile_floats((int)round_up(dpad_, 16)) * 4 + 512);
  return (int64_t)nlist_ * dpad_ * 4 + (lists_ ? lists_->mem_bytes() : 0) + mirror;
}
int IVFFlatIndex::set_centroids(const float* host, int nlist) {
  if (nlist != nlist_) {
    set_last_error("set_centroids: nlist mismatch");
    return -1;
  }
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  drain_searches();
  GB_CUDA(cudaMemset(d_centroids_, 0, (size_t)nlist_ * dpad_ * 4));
  GB_CUDA(cudaMemcpy2D(d_centroids_, (size_t)dpad_ * 4, host, (size_t)d_ * 4, (size_t)d_ * 4, nlist_,
                       cudaMemcpyHostToDevice));
  if (!lists_) lists_.reset(new IvfLists(nlist_, code_bytes()));
  trained_ = true;
  return 0;
}
int IVFFlatIndex::get_centroids(float* host) const {
  cudaSetDevice(device_);
  GB_CUDA(cudaMemcpy2D(host, (size_t)d_ * 4, d_centroids_, (size_t)dpad_ * 4, (size_t)d_ * 4, nlist_,
                       cudaMemcpyDeviceToHost));
  return 0;
}

// GammaIVFFlatIndex::Indexing (gamma_index_ivfflat.cc:342-411): train on the FIRST num vectors.
int IVFFlatIndex::train() {
  std::lock_guard<std::mutex> bg(build_mu_);
  if (trained_) return 0;
  cudaSetDevice(device_);
  int64_t num = training_threshold();
  if (num > store_->size()) {
    set_last_error("vector total count less than training_threshold");
    return -1;
  }
  std::unique_lock<std::shared_mutex> lk(mu_);
  drain_searches();
  cudaStream_t st = build_stream_;
  Scratch s(st);
  const float* xt = store_->contiguous(num, s);
  if (!xt) return -1;
  KMeansParams kp;
  const bool is_pq = (type_ == "IVFPQ" || type_ == "IVFRABITQ");
  kp.niter = is_pq ? 10 : 25;                              // gamma_index_ivfpq.cc:188, gamma_index_ivfrabitq.cc:55-300
  kp.spherical = is_pq && mp_.metric == kMetricIP;          // gamma_index_ivfpq.cc:189-191
  xt = train_transform(xt, num, s);  // OPQ: learn the rotation, continue on the rotated slab
  if (!xt) return -1;
  if (kmeans_device(xt, dpad_, num, d_, nlist_, kp, d_centroids_, dpad_, st, nullptr)) return -1;
  if (train_extra(xt, num, s)) return -1;
  GB_CUDA(cudaStreamSynchronize(st));
  if (!lists_) lists_.reset(new IvfLists(nlist_, code_bytes()));
  trained_ = true;
  return 0;
}

int IVFFlatIndex::assign_dev(const float* x, int64_t ldx, int64_t n, int32_t* out, Scratch& s) {
  cudaStream_t st = s.stream();
  GB_ALLOC(best, unsigned long long, n, s);
  GB_CUDA(launch_fill_u64(best, n, kKeySentinel, st));
  GB_CUDA(launch_dist_argmin(x, ldx, (int)n, d_centroids_, dpad_, nlist_, dpad_, mp_.metric, best, 0, st));
  GB_CUDA(launch_split_keys(best, n, mp_.metric, nullptr, out, st));
  return 0;
}

int IVFFlatIndex::append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                               const int32_t* d_assign, Scratch& s) {
  (void)d_assign;
  GB_CUDA(launch_ivf_append_vecs(x, dpad_, n, dpad_, d_list, d_pos, reinterpret_cast<float* const*>(lists_->d_data()),
                                 lists_->d_ids(), vid0, s.stream()));
  return 0;
}

// GammaIVFFlatIndex::Add (gamma_index_ivfflat.cc:413-474) driven like
// VectorManager::AddRTVecsToIndex (vector_manager.cc:572-702), in large device batches.
int IVFFlatIndex::index_batch(const float* x, int64_t n, int64_t vid0, const uint8_t* del_bitmap) {
  cudaStream_t st = build_stream_;
  Scratch s(st);
  x = transform_dev(x, n, s);  // OPQ rotation; the raw store keeps the original rows
  if (!x) return -1;
  GB_ALLOC(d_assign, int32_t, n, s);
  if (assign_dev(x, dpad_, n, d_assign, s)) return -1;
  std::vector<int32_t> h_list(n), h_pos(n);
  GB_CUDA(cudaMemcpyAsync(h_list.data(), d_assign, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  std::vector<int> add(nlist_, 0);
  const std::vector<int>& lens = lists_->lens();
  if ((int64_t)vid2pos_.size() < vid0 + n) vid2pos_.resize(vid0 + n, ~(uint64_t)0);
  for (int64_t i = 0; i < n; i++) {
    int64_t vid = vid0 + i;
    int l = h_list[i];
    if (del_bitmap && ((del_bitmap[vid >> 3] >> (vid & 7)) & 1)) {  // ivfflat.cc:436: deleted before indexing
      h_list[i] = -1;
      h_pos[i] = 0;
      continue;
    }
    if (l < 0 || l >= nlist_) l = (int)(vid % nlist_);  // ivfflat.cc:443-446
    h_list[i] = l;
    h_pos[i] = lens[l] + add[l]++;  // insertion (vid) order inside the list
    vid2pos_[vid] = ((uint64_t)l << 32) | (uint32_t)h_pos[i];
  }
  GB_ALLOC(d_list, int32_t, n, s);
  GB_ALLOC(d_pos, int32_t, n, s);
  GB_CUDA(cudaMemcpyAsync(d_list, h_list.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(d_pos, h_pos.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
  std::unique_lock<std::shared_mutex> lk(mu_);
  drain_searches();  // kernels of earlier searches read lengths and base pointers at run time
  if (lists_->reserve(add, st)) return -1;
  if (append_batch(x, n, vid0, d_list, d_pos, d_assign, s)) return -1;
  // data (lists AND their tensor-core mirror) first, the new lengths last (realtime_mem_data.cc:292-293)
  if (type_ == "IVFFLAT" && mirror_append(x, n, d_list, d_pos, add, st)) return -1;
  if (lists_->commit(add, st)) return -1;
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int IVFFlatIndex::add_pending(const uint8_t* del_bitmap) {
  std::lock_guard<std::mutex> bg(build_mu_);
  if (!trained_) return 0;
  cudaSetDevice(device_);
  const int64_t BATCH = 1 << 20;
  for (;;) {
    int64_t vid0 = indexed_count_, n = 0;
    const float* x = nullptr;
    {  // add_vectors (exclusive mu_) may append segments while we look: the segment table is read under the shared lock
      std::shared_lock<std::shared_mutex> lk(mu_);
      if (vid0 >= store_->size()) break;
      int64_t si = vid0 >> store_->seg_shift(), off = vid0 & (store_->seg_rows() - 1);
      n = std::min<int64_t>(std::min(store_->size() - vid0, store_->seg_rows() - off), BATCH);
      x = store_->seg((int)si) + off * dpad_;
    }
    if (index_batch(x, n, vid0, del_bitmap)) return -1;
    indexed_count_ += n;
  }
  // a bulk build leaves most of the slab space in regions the lists have outgrown: re-pack once the
  // waste is worth a copy (more than half of the live bytes and more than 1 GiB)
  if (lists_ && lists_->mem_bytes() - lists_->packed_bytes() > std::max<int64_t>((int64_t)1 << 30, lists_->packed_bytes() / 2)) {
    std::unique_lock<std::shared_mutex> lk(mu_);
    if (lists_->compact(build_stream_)) return -1;
  }
  return 0;
}

int IVFFlatIndex::reset_index() {
  std::lock_guard<std::mutex> bg(build_mu_);
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  std::unique_lock<std::shared_mutex> ml(mirror_rw_);
  cudaDeviceSynchronize();  // kernels of earlier device-resident searches may still read the lists
  lists_.reset();
  vid2pos_.clear();
  mirror_.lens.clear();
  indexed_count_ = 0;
  trained_ = false;
  return 0;
}

int IVFFlatIndex::compact_lists() {
  std::lock_guard<std::mutex> bg(build_mu_);
  if (!lists_) return 0;
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  return lists_->compact(build_stream_);
}

int Index::update_vector(int64_t vid, const float* x) {
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  return store_->update_host(vid, x, build_stream_);
}

// GammaIVFFlatIndex::Update / GammaIVFPQIndex::Update (gamma_index_ivfflat.cc:476-522,
// gamma_index_ivfpq.cc:402-453): tombstone the old entry, append the new vector to its list.
int IVFFlatIndex::update_vector(int64_t vid, const float* x) {
  std::lock_guard<std::mutex> bg(build_mu_);
  if (Index::update_vector(vid, x)) return -1;
  if (!trained_ || vid >= indexed_count_) return 0;  // not indexed yet: the add path will pick it up
  if (vid < (int64_t)vid2pos_.size() && vid2pos_[vid] != ~(uint64_t)0) {
    std::unique_lock<std::shared_mutex> lk(mu_);
    if (lists_->tombstone((int)(vid2pos_[vid] >> 32), (int)(uint32_t)vid2pos_[vid], build_stream_)) return -1;
  }
  int64_t si = vid >> store_->seg_shift(), off = vid & (store_->seg_rows() - 1);
  return index_batch(store_->seg((int)si) + off * dpad_, 1, vid, nullptr);
}

int IVFFlatIndex::resolve_nprobe(const SearchContext& ctx) const {
  int nprobe = mp_.nprobe;
  if (ctx.params.nprobe > 0 && ctx.params.nprobe <= nlist_) nprobe = ctx.params.nprobe;  // ivfflat.cc:551-559
  if (nprobe > nlist_) nprobe = nlist_;
  if (nprobe > 4096) nprobe = 4096;
  return nprobe;
}

// quantizer->search (gamma_index_ivfflat.cc:568 / gamma_index_ivfpq.cc:595)
int IVFFlatIndex::coarse_dev(int nq, const float* xq, int nprobe, int metric, int32_t* probe_ids, float* coarse_dis,
                             Scratch& s) {
  cudaStream_t st = s.stream();
  int64_t ldo = round_up(nlist_, 4);
  GB_ALLOC(scores, float, (size_t)nq * ldo, s);
  GB_ALLOC(keys, unsigned long long, (size_t)nq * nprobe, s);
  StageScope stage(this, "coarse_quantizer", st);
  if (tc_enabled() && nlist_ >= 64 && nq >= 32) {
    GB_CUDA(launch_dist_matrix_tc(xq, dpad_, nq, d_centroids_, dpad_, nlist_, dpad_, metric, scores, ldo, st));
  } else {
    GB_CUDA(launch_dist_matrix(xq, dpad_, nq, d_centroids_, dpad_, nlist_, dpad_, metric, scores, ldo, st));
  }
  FilterArgs nf{nullptr, nullptr, -FLT_MAX, FLT_MAX};
  GB_CUDA(launch_select_scores(scores, ldo, nq, nlist_, 0, nprobe, metric, nf, keys, nprobe, st));
  GB_CUDA(launch_split_keys(keys, (int64_t)nq * nprobe, metric, coarse_dis, probe_ids, st));
  return 0;
}

// List-major scan (DESIGN.md K3-LM): worthwhile when many queries of the batch probe each list.
// Host side: group the (query, probe) pairs by list (stable counting sort), give every pair a
// score segment of len(list) floats, cut (list, 128 pairs, 128 rows) tiles; device side: grouped
// GEMM on tcgen05 + segment select.
// GB_LISTMAJOR: 0 = off, 1 = on (fused top-k epilogue when k allows), 2 = on, always the dense-score variant
static int listmajor_mode() {  // read per call: tests flip it between searches of one process
  const char* e = getenv("GB_LISTMAJOR");
  return e ? atoi(e) : 1;
}
static bool listmajor_enabled() { return listmajor_mode() != 0; }
static bool tma_enabled() {  // GB_TC_MIRROR=0: never build the pre-tiled mirror (register-staged kernel)
  static int v = [] {
    const char* e = getenv("GB_TC_MIRROR");
    return e ? atoi(e) : 1;
  }();
  return v != 0;
}

// called from index_batch with mu_ held exclusively: no search is inside ensure_mirror.  Kernels of an
// earlier search_device may still be running, but they only look at rows below the lengths they were
// launched with, and the rows written here lie above those.
int IVFFlatIndex::mirror_append(const float* x, int64_t n, const int32_t* d_list, const int32_t* d_pos,
                                const std::vector<int>& add, cudaStream_t st) {
  if (!mirror_.base || mirror_.disabled || mirror_.lens.size() != (size_t)nlist_) return 0;
  std::vector<int> lens = lists_->lens();  // lengths BEFORE this batch is committed
  for (int l = 0; l < nlist_; l++) {
    if (mirror_.lens[l] != lens[l] || (int64_t)lens[l] + add[l] > (int64_t)mirror_.list_tiles[l] * 128) {
      mirror_.lens.clear();  // stale: outgrown (or out of step); rebuilt by the next list-major search
      return 0;
    }
    lens[l] += add[l];
  }
  GB_CUDA(launch_tc_mirror_append(x, dpad_, n, dpad_, (int)round_up(dpad_, 16), d_list, d_pos, mirror_.d_tile0, mirror_.base,
                                  mirror_.norms, st));
  mirror_.lens = lens;
  return 0;
}

int IVFFlatIndex::ensure_mirror(std::shared_lock<std::shared_mutex>& lk, cudaStream_t st) {
  if (type_ != "IVFFLAT" || !lists_) return 1;
  lk.lock();
  if (mirror_.disabled) return 1;
  if (mirror_.base && mirror_.lens == lists_->lens()) return 0;
  lk.unlock();
  {
    std::unique_lock<std::shared_mutex> x(mirror_rw_);
    if (!mirror_.disabled && !(mirror_.base && mirror_.lens == lists_->lens())) {
      const std::vector<int>& lens = lists_->lens();
      const int k16 = (int)round_up(dpad_, 16);
      const size_t tile_bytes = (size_t)tc_mirror_tile_floats(k16) * 4;
      cudaDeviceSynchronize();  // kernels of other searches may still be reading the mirror
      if (mirror_.base) cudaFree(mirror_.base);
      if (mirror_.norms) cudaFree(mirror_.norms);
      mirror_.base = mirror_.norms = nullptr;
      mirror_.cap_tiles = 0;
      size_t free_b = 0, total_b = 0;
      cudaMemGetInfo(&free_b, &total_b);
      std::vector<int64_t> tile0(nlist_ + 1, 0);
      std::vector<int> list_tiles(nlist_, 0);
      int64_t tiles = 0;
      for (int slack = 8; slack >= 0 && !mirror_.base; slack -= 8) {  // 1/8 more rows per list, else none
        for (int l = 0; l < nlist_; l++) {
          const int64_t rows = slack ? (int64_t)lens[l] + lens[l] / slack : lens[l];
          list_tiles[l] = (int)((rows + 127) / 128);
          tile0[l + 1] = tile0[l] + list_tiles[l];
        }
        tiles = tile0[nlist_];
        const size_t need = (size_t)std::max<int64_t>(tiles, 1) * (tile_bytes + 512);
        if (need + ((size_t)4 << 30) > free_b) continue;
        if (cudaMalloc(&mirror_.base, (size_t)std::max<int64_t>(tiles, 1) * tile_bytes) != cudaSuccess ||
            cudaMalloc(&mirror_.norms, (size_t)std::max<int64_t>(tiles, 1) * 512) != cudaSuccess) {
          if (mirror_.base) cudaFree(mirror_.base);
          mirror_.base = nullptr;
          cudaGetLastError();
        }
      }
      if (!mirror_.base) {
        mirror_.disabled = true;  // HBM too full for a second, doubled copy of the lists
      } else {
        mirror_.cap_tiles = tiles;
        mirror_.list_tiles = list_tiles;
      }
      if (!mirror_.disabled) {
        if (!mirror_.d_tile0 && cudaMalloc(&mirror_.d_tile0, sizeof(int64_t) * (nlist_ + 1)) != cudaSuccess) return -1;
        GB_CUDA(cudaMemcpyAsync(mirror_.d_tile0, tile0.data(), sizeof(int64_t) * (nlist_ + 1), cudaMemcpyHostToDevice, st));
        GB_CUDA(launch_tc_mirror_build(lists_->directory(), dpad_, k16, mirror_.d_tile0, tiles, mirror_.base, mirror_.norms,
                                       st));
        GB_CUDA(cudaStreamSynchronize(st));  // tile0 is a stack vector; other streams may use the mirror next
        mirror_.tiles = tiles;
        mirror_.lens = lens;
        mirror_.builds++;
      }
    }
  }
  lk.lock();
  if (mirror_.disabled) return 1;
  return (mirror_.base && mirror_.lens == lists_->lens()) ? 0 : 1;
}

int IVFFlatIndex::scan_listmajor_dev(const FilterArgs& f, int metric, int nq, const float* xq, int k,
                                     const int32_t* probe_ids, int nprobe, unsigned long long* out_keys, Scratch& s) {
  if (!tc_enabled() || !listmajor_enabled()) return 1;
  const int64_t npairs = (int64_t)nq * nprobe;
  if (npairs < (int64_t)nlist_ * 32 && !getenv("GB_LISTMAJOR_FORCE")) return 1;  // < 32 queries per list on average
  cudaStream_t st = s.stream();
  ListDirectory dir = lists_->directory();
  if (k <= kLmkMaxK && listmajor_mode() != 2) {
    // fused top-k epilogue: no score round trip through HBM, no host synchronisation
    const int nseg = (int)std::min<int64_t>(8, std::max<int64_t>(1, (lists_->max_len() + kLmkSegRows - 1) / kLmkSegRows));
    const int64_t max_items = (npairs / 128 + nlist_) * nseg;
    if (max_items > INT32_MAX) return 1;
    GB_ALLOC(d_cnt, int32_t, nlist_, s);
    GB_ALLOC(d_start, int32_t, nlist_, s);
    GB_ALLOC(d_cursor, int32_t, nlist_, s);
    GB_ALLOC(d_item_start, int32_t, nlist_, s);
    GB_ALLOC(d_grp_start, int32_t, nlist_, s);
    GB_ALLOC(d_totals, int64_t, 3, s);
    GB_ALLOC(d_pair_j, int64_t, npairs, s);
    GB_ALLOC(d_items, LmTile, max_items, s);
    GB_ALLOC(d_tau, unsigned long long, nq, s);
    const size_t nout = (size_t)npairs * nseg * k;
    GB_ALLOC(d_out, unsigned long long, nout, s);
    GB_CUDA(cudaMemsetAsync(d_tau, 0xFF, sizeof(unsigned long long) * nq, st));
    GB_CUDA(cudaMemsetAsync(d_out, 0xFF, sizeof(unsigned long long) * nout, st));
    GB_CUDA(launch_lmk_group(probe_ids, npairs, dir, nseg, d_cnt, d_start, d_cursor, d_item_start, d_grp_start, d_totals,
                             d_pair_j, d_items, st));
    const int k16 = (int)round_up(dpad_, 16);
    const int64_t max_groups = npairs / 128 + nlist_;
    const size_t slot_bytes = (size_t)128 * k16 * 8, a_bytes = (size_t)max_groups * (slot_bytes + 128 * 4);
    std::shared_lock<std::shared_mutex> mlk(mirror_rw_, std::defer_lock);
    bool tma = tma_enabled() && k <= 32 && k16 > 16 && a_bytes <= ((size_t)8 << 30) && ensure_mirror(mlk, st) == 0;
    if (tma) {
      float* a_scratch = static_cast<float*>(big_acquire(a_bytes, st));
      if (!a_scratch) return -1;
      auto rel_fn = [this, a_scratch, st](void*) { big_release(a_scratch, st); };
      std::unique_ptr<void, decltype(rel_fn)> rel(a_scratch, rel_fn);
      float* a_norms = reinterpret_cast<float*>(reinterpret_cast<char*>(a_scratch) + (size_t)max_groups * slot_bytes);
      TcMirrorView mv{mirror_.base, mirror_.d_tile0, mirror_.norms, k16};
      last_scan_kernel_ = "ivf_listmajor_tma_kernel";
      scan_timer_begin(st);
      GB_CUDA(launch_lm_stage_queries(xq, dpad_, dpad_, k16, d_items, (int)max_items, d_totals, d_pair_j, nprobe, a_scratch,
                                      a_norms, st));
      GB_CUDA(launch_ivf_listmajor_tma(a_scratch, a_norms, mv, d_items, (int)max_items, d_totals, d_pair_j, nprobe, dir, k,
                                       nseg, metric, f, d_tau, d_out, st));
      scan_timer_end(st);
    } else {
      last_scan_kernel_ = "ivf_listmajor_topk_kernel";
      scan_timer_begin(st);
      GB_CUDA(launch_ivf_listmajor_topk(xq, dpad_, dpad_, d_items, (int)max_items, d_totals, d_pair_j, nprobe, dir, k, nseg,
                                        metric, f, d_tau, d_out, st));
      scan_timer_end(st);
    }
    if (mlk.owns_lock()) mlk.unlock();
    GB_CUDA(launch_select_keys(d_out, (int64_t)nprobe * nseg * k, nq, nprobe * nseg * k, k, out_keys, k, st));
    return 0;
  }
  GB_ALLOC(d_cnt, int32_t, nlist_, s);
  GB_ALLOC(d_start, int32_t, nlist_, s);
  GB_ALLOC(d_cursor, int32_t, nlist_, s);
  GB_ALLOC(d_tile_start, int32_t, nlist_, s);
  GB_ALLOC(d_base_off, int64_t, nlist_, s);
  GB_ALLOC(d_totals, int64_t, 3, s);
  GB_CUDA(launch_lm_count_scan(probe_ids, npairs, dir, d_cnt, d_start, d_base_off, d_tile_start, d_totals, st));
  int64_t h_totals[3] = {0, 0, 0};
  GB_CUDA(cudaMemcpyAsync(h_totals, d_totals, sizeof(h_totals), cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  const int64_t total = h_totals[0], ntiles = h_totals[1];
  if (total > ((int64_t)3 << 30) || ntiles > INT32_MAX) return 1;  // > 12 GiB of scores: query-major scan instead
  GB_ALLOC(d_pair_q, int32_t, npairs, s);
  GB_ALLOC(d_pair_off, int64_t, npairs, s);
  GB_ALLOC(d_seg_off, int64_t, npairs, s);
  GB_ALLOC(d_tiles, LmTile, std::max<int64_t>(ntiles, 1), s);
  float* scores = static_cast<float*>(big_acquire((size_t)std::max<int64_t>(total, 1) * 4, st));
  if (!scores) return -1;
  auto rel_fn = [this, scores, st](void*) { big_release(scores, st); };
  std::unique_ptr<void, decltype(rel_fn)> rel(scores, rel_fn);  // released (event-stamped) on every exit path
  GB_CUDA(launch_lm_assign_tiles(probe_ids, npairs, nprobe, dir, d_cnt, d_start, d_cursor, d_base_off, d_tile_start,
                                 d_pair_q, d_pair_off, d_seg_off, d_tiles, st));
  last_scan_kernel_ = "ivf_listmajor_tc_kernel+seg_select_kernel";
  scan_timer_begin(st);
  GB_CUDA(launch_ivf_listmajor_tc(xq, dpad_, dpad_, d_tiles, (int)ntiles, d_pair_q, d_pair_off, dir, metric, scores, st));
  GB_CUDA(launch_seg_select(scores, d_seg_off, probe_ids, nq, nprobe, dir, k, metric, f, out_keys, st));
  scan_timer_end(st);
  return 0;
}

int IVFFlatIndex::scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                           const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
                           Scratch& s) {
  (void)ctx;
  (void)coarse_dis;
  cudaStream_t st = s.stream();
  if (type_ == "IVFFLAT") {
    // The list-major scan selects on 3xTF32 tensor-core scores (|x|^2 + |y|^2 - 2 x.y for L2: on SIFT-like float data,
    // |x|^2 ~ 40 d^2, the cancellation leaves ~1e-4 relative).  Its k winners are re-scored with the direct fp32 form
    // from the raw vectors and re-sorted (rerank_kernel, k rows per query), so every distance that leaves the index is
    // the exact-kernel value; on integer-valued data both forms are exact and nothing changes.
    GB_ALLOC(lm_keys, unsigned long long, (size_t)nq * k, s);
    int lm = scan_listmajor_dev(f, metric, nq, xq, k, probe_ids, nprobe, lm_keys, s);
    if (lm < 0) return lm;
    if (lm == 0) {
      if ((dpad_ & 3) == 0 && k <= 8192) {
        GB_CUDA(launch_rerank(lm_keys, k, nq, xq, dpad_, dpad_, store_->d_segs(), store_->seg_shift(), dpad_, k, metric, f,
                              out_keys, st));
      } else {
        GB_CUDA(cudaMemcpyAsync(out_keys, lm_keys, (size_t)nq * k * 8, cudaMemcpyDeviceToDevice, st));
      }
      return 0;
    }
  }
  int nparts = ivfflat_scan_nparts(nprobe, lists_->max_len());
  GB_ALLOC(partial, unsigned long long, (size_t)nq * nparts * k, s);
  last_scan_kernel_ = "ivfflat_scan_warp_kernel";
  scan_timer_begin(st);
  int avg_len = (int)(lists_->total() / std::max(1, nlist_));
  GB_CUDA(launch_ivfflat_scan(xq, dpad_, nq, dpad_, probe_ids, nprobe, lists_->directory(), lists_->max_len(), avg_len, k,
                              metric, f, partial, &nparts, st));
  scan_timer_end(st);
  GB_CUDA(launch_select_keys(partial, (int64_t)nparts * k, nq, nparts * k, k, out_keys, k, st));
  return 0;
}

// When a transform sits in front of the index the scan works on transformed queries while the exact re-rank
// needs the original ones: the search entry points leave both base pointers here for scan_dev (same thread).
static thread_local const float* tls_xq_transformed = nullptr;
static thread_local const float* tls_xq_raw = nullptr;
static const float* raw_queries_for(const float* xq) {
  return tls_xq_transformed && tls_xq_raw ? tls_xq_raw + (xq - tls_xq_transformed) : xq;
}

// GammaIVFFlatIndex::Search (gamma_index_ivfflat.cc:524-577)
int IVFFlatIndex::search_keys_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq_in,
                                  int k, unsigned long long* out_keys, Scratch& s) {
  const float* xq = transform_dev(xq_in, nq, s);
  if (!xq) return -1;
  struct TlsGuard {
    TlsGuard(const float* t, const float* r) { tls_xq_transformed = t == r ? nullptr : t, tls_xq_raw = r; }
    ~TlsGuard() { tls_xq_transformed = tls_xq_raw = nullptr; }
  } guard(xq, xq_in);
  const int nprobe = resolve_nprobe(ctx);
  const int QB = 16384;
  for (int q0 = 0; q0 < nq; q0 += QB) {
    int qb = std::min(QB, nq - q0);
    Scratch sb(s.stream());
    GB_ALLOC(probe_ids, int32_t, (size_t)qb * nprobe, sb);
    GB_ALLOC(coarse_dis, float, (size_t)qb * nprobe, sb);
    if (coarse_dev(qb, xq + (int64_t)q0 * dpad_, nprobe, metric, probe_ids, coarse_dis, sb)) return -1;
    if (scan_dev(ctx, f, metric, qb, xq + (int64_t)q0 * dpad_, k, probe_ids, coarse_dis, nprobe,
                 out_keys + (int64_t)q0 * k, sb))
      return -1;
  }
  return 0;
}

int IVFFlatIndex::coarse_search_host(int nq, const float* x, int nprobe, float* out_dis, int64_t* out_ids) {
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  std::shared_lock<std::shared_mutex> lk(mu_);
  Scratch s(st);
  GB_ALLOC(dq, float, (size_t)nq * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dq, 0, (size_t)nq * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dq, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, nq, cudaMemcpyHostToDevice, st));
  GB_ALLOC(ids, int32_t, (size_t)nq * nprobe, s);
  GB_ALLOC(dis, float, (size_t)nq * nprobe, s);
  const float* dqt = transform_dev(dq, nq, s);
  if (!dqt || coarse_dev(nq, dqt, nprobe, mp_.metric, ids, dis, s)) return -1;
  std::vector<int32_t> h((size_t)nq * nprobe);
  GB_CUDA(cudaMemcpyAsync(h.data(), ids, h.size() * 4, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaMemcpyAsync(out_dis, dis, h.size() * 4, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  for (size_t i = 0; i < h.size(); i++) out_ids[i] = h[i];
  return 0;
}

int IVFFlatIndex::search_preassigned_host(const SearchContext& ctx, int nq, const float* x, int k, const int64_t* keys,
                                          const float* coarse_dis, int nprobe, float* out_dis, int64_t* out_ids) {
  if (!trained_ || !lists_) {
    set_last_error("index not trained");
    return -1;
  }
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  std::shared_lock<std::shared_mutex> lk(mu_);
  Scratch s(st);
  GB_ALLOC(dq, float, (size_t)nq * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dq, 0, (size_t)nq * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dq, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, nq, cudaMemcpyHostToDevice, st));
  std::vector<int32_t> h((size_t)nq * nprobe);
  for (size_t i = 0; i < h.size(); i++) h[i] = (int32_t)keys[i];
  GB_ALLOC(ids, int32_t, h.size(), s);
  GB_ALLOC(dis, float, h.size(), s);
  GB_CUDA(cudaMemcpyAsync(ids, h.data(), h.size() * 4, cudaMemcpyHostToDevice, st));
  GB_CUDA(cudaMemcpyAsync(dis, coarse_dis, h.size() * 4, cudaMemcpyHostToDevice, st));
  FilterArgs f;
  if (upload_bitmaps(ctx, &f, s)) return -1;
  int metric = ctx.params.metric >= 0 ? ctx.params.metric : mp_.metric;
  GB_ALLOC(okeys, unsigned long long, (size_t)nq * k, s);
  const float* dqt = transform_dev(dq, nq, s);
  if (!dqt) return -1;
  tls_xq_transformed = dqt == dq ? nullptr : dqt, tls_xq_raw = dq;
  const int src = scan_dev(ctx, f, metric, nq, dqt, k, ids, dis, nprobe, okeys, s);
  tls_xq_transformed = tls_xq_raw = nullptr;
  if (src) return -1;
  GB_ALLOC(dd, float, (size_t)nq * k, s);
  GB_ALLOC(di, int64_t, (size_t)nq * k, s);
  GB_CUDA(launch_decode_keys(okeys, k, nq, k, metric, dd, di, 0, st));
  GB_CUDA(cudaMemcpyAsync(out_dis, dd, (size_t)nq * k * 4, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaMemcpyAsync(out_ids, di, (size_t)nq * k * 8, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------------------------------
IVFPQIndex::IVFPQIndex(int d, const ModelParams& mp, int device, int seg_shift)
    : IVFFlatIndex(d, mp, device, seg_shift, "IVFPQ") {
  M_ = mp.nsubvector > 0 ? mp.nsubvector : d / 2;  // gamma_index_ivfpq.cc:122-124
  if (M_ < 1) M_ = 1;
  dsub_ = d / M_;
  cudaMalloc(&d_pq_, (size_t)M_ * 256 * dsub_ * 4);
  cudaMemset(d_pq_, 0, (size_t)M_ * 256 * dsub_ * 4);
  if (mp.opq_nsubvector > 0) {  // faiss::OPQMatrix(d, opq_nsubvector, d) (gamma_index_ivfpq.cc:168-178)
    cudaMalloc(&d_opq_, (size_t)d * dpad_ * 4);
    cudaMemset(d_opq_, 0, (size_t)d * dpad_ * 4);
  }
}

// ---- OPQ (faiss::OPQMatrix restated; VectorTransform.cpp of faiss v1.14.1 is not vendored) -------------
// train: centre the (sub-sampled, <= 65536) training set, start from a random orthonormal matrix, then 50
// rounds of { project; train a PQ on the projection (40 k-means iterations in the first round, 4 hot-started
// ones afterwards, <= 1000 points per centroid); reconstruct; solve the orthogonal Procrustes problem
// min ||X R^T - Y|| by an SVD of X^T Y }.  The projection and X^T Y run on the device, the d x d SVD (one-sided
// Jacobi, double precision) on the host.  The random start cannot reproduce faiss's generator, so parity with
// the reference is statistical (recall), as for k-means.
namespace {
// A (d x d2, row-major) = U diag(s) V^T by one-sided Jacobi on the columns; returns U (d x d2) and V (d2 x d2)
void jacobi_svd(std::vector<double>& a, int d, int d2, std::vector<double>* u, std::vector<double>* v) {
  v->assign((size_t)d2 * d2, 0.0);
  for (int i = 0; i < d2; i++) (*v)[(size_t)i * d2 + i] = 1.0;
  for (int sweep = 0; sweep < 60; sweep++) {
    double off = 0;
    for (int p = 0; p < d2 - 1; p++)
      for (int q = p + 1; q < d2; q++) {
        double alpha = 0, beta = 0, gamma = 0;
        for (int i = 0; i < d; i++) {
          const double x = a[(size_t)i * d2 + p], y = a[(size_t)i * d2 + q];
          alpha += x * x, beta += y * y, gamma += x * y;
        }
        if (fabs(gamma) <= 1e-15 * sqrt(alpha * beta) || gamma == 0) continue;
        off = std::max(off, fabs(gamma) / sqrt(alpha * beta + 1e-300));
        const double zeta = (beta - alpha) / (2.0 * gamma);
        const double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
        const double c = 1.0 / sqrt(1.0 + t * t), sn = c * t;
        for (int i = 0; i < d; i++) {
          const double x = a[(size_t)i * d2 + p], y = a[(size_t)i * d2 + q];
          a[(size_t)i * d2 + p] = c * x - sn * y, a[(size_t)i * d2 + q] = sn * x + c * y;
        }
        for (int i = 0; i < d2; i++) {
          const double x = (*v)[(size_t)i * d2 + p], y = (*v)[(size_t)i * d2 + q];
          (*v)[(size_t)i * d2 + p] = c * x - sn * y, (*v)[(size_t)i * d2 + q] = sn * x + c * y;
        }
      }
    if (off < 1e-12) break;
  }
  u->assign((size_t)d * d2, 0.0);
  for (int j = 0; j < d2; j++) {
    double nrm = 0;
    for (int i = 0; i < d; i++) nrm += a[(size_t)i * d2 + j] * a[(size_t)i * d2 + j];
    nrm = sqrt(nrm);
    for (int i = 0; i < d; i++) (*u)[(size_t)i * d2 + j] = nrm > 1e-300 ? a[(size_t)i * d2 + j] / nrm : (i == j ? 1.0 : 0.0);
  }
}
}  // namespace

int IVFPQIndex::set_opq(const float* host_A) {
  if (!d_opq_) {
    set_last_error("index was created without opq");
    return -1;
  }
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  drain_searches();
  GB_CUDA(cudaMemset(d_opq_, 0, (size_t)d_ * dpad_ * 4));
  GB_CUDA(cudaMemcpy2D(d_opq_, (size_t)dpad_ * 4, host_A, (size_t)d_ * 4, (size_t)d_ * 4, d_, cudaMemcpyHostToDevice));
  opq_trained_ = true;
  return 0;
}
int IVFPQIndex::get_opq(float* host_A) const {
  if (!d_opq_) {
    set_last_error("index was created without opq");
    return -1;
  }
  cudaSetDevice(device_);
  GB_CUDA(cudaMemcpy2D(host_A, (size_t)d_ * 4, d_opq_, (size_t)dpad_ * 4, (size_t)d_ * 4, d_, cudaMemcpyDeviceToHost));
  return 0;
}

// y = A x for n rows (stride dpad, padding columns zero): one exact fp32 contraction against the rows of A
const float* IVFPQIndex::transform_dev(const float* x, int64_t n, Scratch& s) {
  if (!d_opq_ || !opq_trained_ || n <= 0) return x;
  cudaStream_t st = s.stream();
  float* y = s.alloc_n<float>((size_t)n * dpad_);
  if (!y) return nullptr;
  if (dpad_ != d_ && cudaMemsetAsync(y, 0, (size_t)n * dpad_ * 4, st) != cudaSuccess) return nullptr;
  for (int64_t r0 = 0; r0 < n; r0 += (1 << 20)) {
    const int nr = (int)std::min<int64_t>(n - r0, 1 << 20);
    if (launch_dist_matrix(x + r0 * dpad_, dpad_, nr, d_opq_, dpad_, d_, dpad_, kMetricIP, y + r0 * dpad_, dpad_, st) !=
        cudaSuccess) {
      set_last_error("opq apply failed");
      return nullptr;
    }
  }
  return y;
}

int IVFPQIndex::apply_opq_host(const float* x, int64_t n, float* out) {
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  std::shared_lock<std::shared_mutex> lk(mu_);
  Scratch s(st);
  GB_ALLOC(dx, float, (size_t)n * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dx, 0, (size_t)n * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dx, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, n, cudaMemcpyHostToDevice, st));
  const float* y = transform_dev(dx, n, s);
  if (!y) return -1;
  GB_CUDA(cudaMemcpy2DAsync(out, (size_t)d_ * 4, y, (size_t)dpad_ * 4, (size_t)d_ * 4, n, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

const float* IVFPQIndex::train_transform(const float* xt, int64_t n_in, Scratch& s) {
  if (!d_opq_) return xt;
  if (opq_trained_) return transform_dev(xt, n_in, s);
  cudaStream_t st = s.stream();
  const int d = d_, Mo = mp_.opq_nsubvector, dso = d / Mo, dsp = (int)round_up(dso, 4);
  int64_t n = std::min<int64_t>(n_in, 256 * 256);  // max_train_points
  const float* xs = xt;
  if (n < n_in) {
    std::vector<int32_t> perm;
    rand_perm_mt(perm, n_in, 1234);
    int32_t* d_idx = s.alloc_n<int32_t>(n);
    float* sub = s.alloc_n<float>((size_t)n * dpad_);
    if (!d_idx || !sub) return nullptr;
    if (cudaMemcpyAsync(d_idx, perm.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        launch_gather_rows(xt, dpad_, d_idx, n, dpad_, sub, dpad_, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
      return nullptr;
    xs = sub;
  }
  const int64_t ldn = round_up(n, 4);
  float* xc = s.alloc_n<float>((size_t)n * dpad_);      // centred training set
  float* xproj = s.alloc_n<float>((size_t)n * dpad_);
  float* recon = s.alloc_n<float>((size_t)n * dpad_);
  float* xT = s.alloc_n<float>((size_t)d * ldn);
  float* rT = s.alloc_n<float>((size_t)d * ldn);
  float* xxr = s.alloc_n<float>((size_t)d * dpad_);
  float* slice = s.alloc_n<float>((size_t)n * dsp);
  float* cent = s.alloc_n<float>((size_t)Mo * 256 * dsp);  // per-subspace centroids, kept across rounds
  float* pqc = s.alloc_n<float>((size_t)Mo * 256 * dso);
  uint8_t* codes = s.alloc_n<uint8_t>((size_t)n * Mo);
  if (!xc || !xproj || !recon || !xT || !rT || !xxr || !slice || !cent || !pqc || !codes) return nullptr;
  auto ck = [](cudaError_t e) { return e == cudaSuccess; };
  if (!ck(launch_center_rows(xs, dpad_, n, d, xc, dpad_, st)) || !ck(cudaMemsetAsync(xT, 0, (size_t)d * ldn * 4, st)) ||
      !ck(cudaMemsetAsync(rT, 0, (size_t)d * ldn * 4, st)) || !ck(cudaMemsetAsync(recon, 0, (size_t)n * dpad_ * 4, st)) ||
      !ck(launch_transpose(xc, dpad_, n, d, xT, ldn, st)))
    return nullptr;
  // random orthonormal start: Gaussian matrix (mt19937, seed 1234), Gram-Schmidt on the rows
  std::vector<double> R((size_t)d * d);
  {
    std::mt19937 rng(1234);
    std::normal_distribution<double> nd(0.0, 1.0);
    for (auto& v : R) v = nd(rng);
    for (int i = 0; i < d; i++) {
      for (int p = 0; p < i; p++) {
        double dot = 0;
        for (int j = 0; j < d; j++) dot += R[(size_t)i * d + j] * R[(size_t)p * d + j];
        for (int j = 0; j < d; j++) R[(size_t)i * d + j] -= dot * R[(size_t)p * d + j];
      }
      double nrm = 0;
      for (int j = 0; j < d; j++) nrm += R[(size_t)i * d + j] * R[(size_t)i * d + j];
      nrm = sqrt(nrm);
      for (int j = 0; j < d; j++) R[(size_t)i * d + j] /= nrm;
    }
  }
  std::vector<float> Rf((size_t)d * d), hx((size_t)d * dpad_);
  std::vector<double> a, U, V;
  const int niter = 50, niter_pq_0 = 40, niter_pq = 4;
  for (int it = 0; it < niter; it++) {
    for (size_t i = 0; i < R.size(); i++) Rf[i] = (float)R[i];
    if (!ck(cudaMemsetAsync(d_opq_, 0, (size_t)d * dpad_ * 4, st)) ||
        !ck(cudaMemcpy2DAsync(d_opq_, (size_t)dpad_ * 4, Rf.data(), (size_t)d * 4, (size_t)d * 4, d, cudaMemcpyHostToDevice, st)) ||
        !ck(cudaMemsetAsync(xproj, 0, (size_t)n * dpad_ * 4, st)) ||
        !ck(launch_dist_matrix(xc, dpad_, (int)n, d_opq_, dpad_, d, dpad_, kMetricIP, xproj, dpad_, st)))
      return nullptr;
    KMeansParams kp;
    kp.niter = it == 0 ? niter_pq_0 : niter_pq;
    kp.max_points_per_centroid = 1000;
    kp.hot_start = it > 0;
    for (int m = 0; m < Mo; m++) {
      if (!ck(launch_slice_cols(xproj, dpad_, n, m * dso, dso, slice, dsp, st))) return nullptr;
      if (kmeans_device(slice, dsp, n, dso, 256, kp, cent + (size_t)m * 256 * dsp, dsp, st, nullptr)) return nullptr;
      if (!ck(cudaMemcpy2DAsync(pqc + (size_t)m * 256 * dso, (size_t)dso * 4, cent + (size_t)m * 256 * dsp, (size_t)dsp * 4,
                                (size_t)dso * 4, 256, cudaMemcpyDeviceToDevice, st)))
        return nullptr;
    }
    if (!ck(launch_pq_encode(xproj, dpad_, n, nullptr, 0, nullptr, pqc, Mo, dso, codes, st)) ||
        !ck(launch_pq_decode(codes, n, pqc, Mo, dso, recon, dpad_, st)) || !ck(launch_transpose(recon, dpad_, n, d, rT, ldn, st)) ||
        !ck(launch_dist_matrix(xT, ldn, d, rT, ldn, d, (int)ldn, kMetricIP, xxr, dpad_, st)) ||
        !ck(cudaMemcpyAsync(hx.data(), xxr, (size_t)d * dpad_ * 4, cudaMemcpyDeviceToHost, st)) || !ck(cudaStreamSynchronize(st)))
      return nullptr;
    a.assign((size_t)d * d, 0.0);  // X^T Y, d x d
    for (int i = 0; i < d; i++)
      for (int j = 0; j < d; j++) a[(size_t)i * d + j] = hx[(size_t)i * dpad_ + j];
    jacobi_svd(a, d, d, &U, &V);
    // R^T = U V^T  =>  R[i][j] = sum_k V[i][k] U[j][k]
    for (int i = 0; i < d; i++)
      for (int j = 0; j < d; j++) {
        double acc = 0;
        for (int kk = 0; kk < d; kk++) acc += V[(size_t)i * d + kk] * U[(size_t)j * d + kk];
        R[(size_t)i * d + j] = acc;
      }
  }
  for (size_t i = 0; i < R.size(); i++) Rf[i] = (float)R[i];
  if (!ck(cudaMemsetAsync(d_opq_, 0, (size_t)d * dpad_ * 4, st)) ||
      !ck(cudaMemcpy2DAsync(d_opq_, (size_t)dpad_ * 4, Rf.data(), (size_t)d * 4, (size_t)d * 4, d, cudaMemcpyHostToDevice, st)) ||
      !ck(cudaStreamSynchronize(st)))
    return nullptr;
  opq_trained_ = true;
  return transform_dev(xt, n_in, s);
}

IVFPQIndex::~IVFPQIndex() {
  if (d_opq_) cudaFree(d_opq_);
  cudaFree(d_pq_);
  cudaFree(d_table_);
  cudaFree(d_cb16_);
  cudaFree(d_cbnrm_);
  if (pqn_.base) cudaFree(pqn_.base);
  if (pqn_.d_off) cudaFree(pqn_.d_off);
}
int IVFPQIndex::training_threshold() const {
  // gamma_index_ivfpq.cc:139-144: default max(nlist*200, 256); Indexing() clamps like IVFFLAT (:304-329)
  int64_t t = mp_.training_threshold ? mp_.training_threshold : std::max<int64_t>((int64_t)nlist_ * 200, 256);
  if (t < nlist_)
    t = (int64_t)nlist_ * 39;
  else if (t > (int64_t)nlist_ * 256)
    t = (int64_t)nlist_ * 256;
  return (int)t;
}
int64_t IVFPQIndex::index_mem_bytes() const {
  return IVFFlatIndex::index_mem_bytes() + (int64_t)M_ * 256 * dsub_ * 4 +
         (d_table_ ? (int64_t)nlist_ * M_ * 256 * 4 : 0);
}
int IVFPQIndex::rebuild_table(cudaStream_t st) {
  pq_gen_++;  // the per-entry norm cache belongs to the previous codebook
  // tables of the tensor-core filter (kernels_pqtc.cu): fp16 codebook pre-scaled by -2 sb (L2) / -sb (IP), sb a power of two,
  // centroid norms, and the bound on |r| its error margin uses
  if (pqtc_supported(M_, dsub_)) {
    if (!d_cb16_) GB_CUDA(cudaMalloc(&d_cb16_, (size_t)M_ * 256 * dsub_ * 2));
    if (!d_cbnrm_) GB_CUDA(cudaMalloc(&d_cbnrm_, ((size_t)M_ * 256 + 4) * 4));
    GB_CUDA(launch_pqtc_tables(d_pq_, M_, dsub_, mp_.metric, d_cb16_, d_cbnrm_, d_cbnrm_ + (size_t)M_ * 256, st));
  }
  if (mp_.metric != kMetricL2) return 0;  // IP: tab = ip table, dis0 = <x, centroid>
  if (!d_table_) GB_CUDA(cudaMalloc(&d_table_, (size_t)nlist_ * M_ * 256 * 4));
  GB_CUDA(launch_pq_precompute_table(d_centroids_, dpad_, nlist_, d_pq_, M_, dsub_, d_table_, st));
  return 0;
}
int IVFPQIndex::set_pq_centroids(const float* host) {
  cudaSetDevice(device_);
  std::unique_lock<std::shared_mutex> lk(mu_);
  drain_searches();
  GB_CUDA(cudaMemcpy(d_pq_, host, (size_t)M_ * 256 * dsub_ * 4, cudaMemcpyHostToDevice));
  if (rebuild_table(build_stream_)) return -1;
  GB_CUDA(cudaStreamSynchronize(build_stream_));
  return 0;
}
int IVFPQIndex::get_pq_centroids(float* host) const {
  cudaSetDevice(device_);
  GB_CUDA(cudaMemcpy(host, d_pq_, (size_t)M_ * 256 * dsub_ * 4, cudaMemcpyDeviceToHost));
  return 0;
}
int IVFPQIndex::get_precomputed_table(float* host) const {
  if (!d_table_) {
    set_last_error("no precomputed table (IP metric or untrained)");
    return -1;
  }
  cudaSetDevice(device_);
  GB_CUDA(cudaMemcpy(host, d_table_, (size_t)nlist_ * M_ * 256 * 4, cudaMemcpyDeviceToHost));
  return 0;
}

// faiss IndexIVFPQ::train_residual restated: residuals of (a subsample of <= 256*ksub) training
// vectors -> ProductQuantizer::train = M independent 256-means on the dsub-wide slices.
int IVFPQIndex::train_extra(const float* xtrain, int64_t n, Scratch& s) {
  cudaStream_t st = s.stream();
  if (d_ % M_ != 0) {
    set_last_error("dimension not divisible by nsubvector");
    return -1;
  }
  int64_t npq = std::min<int64_t>(n, 256 * 256);
  const float* xs = xtrain;
  if (npq < n) {
    std::vector<int32_t> perm;
    rand_perm_mt(perm, n, 1234);
    GB_ALLOC(d_idx, int32_t, npq, s);
    GB_CUDA(cudaMemcpyAsync(d_idx, perm.data(), (size_t)npq * 4, cudaMemcpyHostToDevice, st));
    GB_ALLOC(sub, float, (size_t)npq * dpad_, s);
    GB_CUDA(launch_gather_rows(xtrain, dpad_, d_idx, npq, dpad_, sub, dpad_, st));
    GB_CUDA(cudaStreamSynchronize(st));
    xs = sub;
  }
  GB_ALLOC(assign, int32_t, npq, s);
  if (assign_dev(xs, dpad_, npq, assign, s)) return -1;
  GB_ALLOC(resid, float, (size_t)npq * dpad_, s);
  GB_CUDA(launch_residual(xs, dpad_, npq, d_, d_centroids_, dpad_, assign, resid, dpad_, st));
  const int dsp = (int)round_up(dsub_, 4);
  GB_ALLOC(slice, float, (size_t)npq * dsp, s);
  GB_ALLOC(cent, float, (size_t)256 * dsp, s);
  KMeansParams kp;  // ClusteringParameters defaults: niter 25, seed 1234, max 256 points per centroid
  for (int m = 0; m < M_; m++) {
    GB_CUDA(launch_slice_cols(resid, dpad_, npq, m * dsub_, dsub_, slice, dsp, st));
    if (kmeans_device(slice, dsp, npq, dsub_, 256, kp, cent, dsp, st, nullptr)) return -1;
    GB_CUDA(cudaMemcpy2DAsync(d_pq_ + (size_t)m * 256 * dsub_, (size_t)dsub_ * 4, cent, (size_t)dsp * 4,
                              (size_t)dsub_ * 4, 256, cudaMemcpyDeviceToDevice, st));
  }
  return rebuild_table(st);
}

// GammaIVFPQIndex::Add (gamma_index_ivfpq.cc:455-540): residual -> pq.compute_codes -> AddKeys
int IVFPQIndex::append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                             const int32_t* d_assign, Scratch& s) {
  cudaStream_t st = s.stream();
  GB_ALLOC(codes, uint8_t, (size_t)n * M_, s);
  // residual is taken w.r.t. the assigned list (d_list == d_assign except for skipped rows)
  (void)d_assign;
  GB_CUDA(launch_pq_encode(x, dpad_, n, d_centroids_, dpad_, d_list, d_pq_, M_, dsub_, codes, st));
  GB_CUDA(launch_ivf_append_codes(codes, n, M_, d_list, d_pos, reinterpret_cast<uint8_t* const*>(lists_->d_data()),
                                  lists_->d_ids(), vid0, st));
  return 0;
}

int IVFPQIndex::encode_host(const float* x, int64_t n, const int64_t* assign, uint8_t* codes_out) {
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  Scratch s(st);
  GB_ALLOC(dx, float, (size_t)n * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dx, 0, (size_t)n * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dx, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, n, cudaMemcpyHostToDevice, st));
  std::vector<int32_t> h(n);
  for (int64_t i = 0; i < n; i++) h[i] = (int32_t)assign[i];
  GB_ALLOC(da, int32_t, n, s);
  GB_CUDA(cudaMemcpyAsync(da, h.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
  GB_ALLOC(codes, uint8_t, (size_t)n * M_, s);
  GB_CUDA(launch_pq_encode(dx, dpad_, n, d_centroids_, dpad_, da, d_pq_, M_, dsub_, codes, st));
  GB_CUDA(cudaMemcpyAsync(codes_out, codes, (size_t)n * M_, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// Cache of |r_e|^2 per list entry for the tensor-core filter.  Searches hold mu_ shared, appends hold it exclusively and
// drain in-flight searches before the lists change, so whenever the key (list set, lengths, codebook generation) differs
// from the cached one no kernel is reading the cache; the rebuild (one pass over the codes) is serialised by pqn_mu_ and
// synchronised before other streams may use it.
int IVFPQIndex::ensure_pq_norms(cudaStream_t st) {
  std::lock_guard<std::mutex> g(pqn_mu_);
  const std::vector<int>& lens = lists_->lens();
  if (pqn_.base && pqn_.lists_uid == lists_->uid() && pqn_.pq_gen == pq_gen_ && pqn_.lens == lens) return 0;
  std::vector<int64_t> off((size_t)nlist_ + 1, 0);
  for (int l = 0; l < nlist_; l++) off[l + 1] = off[l] + round_up(lens[l], 32);
  const size_t total = (size_t)off[nlist_] + 128;  // a tile's 16-byte rounded tail may run past the last entry
  if (total > pqn_.cap) {
    if (pqn_.base) {
      cudaDeviceSynchronize();
      cudaFree(pqn_.base);
      pqn_.base = nullptr;
    }
    const size_t cap = total + total / 4;
    if (cudaMalloc(&pqn_.base, cap * 4) != cudaSuccess) {
      cudaGetLastError();
      pqn_.cap = 0;
      return 1;  // no room: the caller scans with the exact kernel
    }
    pqn_.cap = cap;
  }
  if (!pqn_.d_off) GB_CUDA(cudaMalloc(&pqn_.d_off, sizeof(int64_t) * ((size_t)nlist_ + 1)));
  GB_CUDA(cudaMemcpyAsync(pqn_.d_off, off.data(), sizeof(int64_t) * ((size_t)nlist_ + 1), cudaMemcpyHostToDevice, st));
  GB_CUDA(launch_pq_entry_norms(lists_->directory(), nlist_, lists_->max_len(), M_, d_cbnrm_, pqn_.d_off, pqn_.base, st));
  GB_CUDA(cudaStreamSynchronize(st));
  pqn_.lens = lens;
  pqn_.lists_uid = lists_->uid();
  pqn_.pq_gen = pq_gen_;
  return 0;
}

// GB_PQTC=0: never use the tensor-core filter (exact LUT kernel for every probe); GB_PQTC=2: use it
// whenever the shape allows, whatever the batch size (tests)
static int pqtc_mode() {  // read per call: tests flip it between searches of one process
  const char* e = getenv("GB_PQTC");
  return e ? atoi(e) : 1;
}
// test hook: scales the filter's error margin (1 = the rigorous bound, 0 = no margin at all)
static float pqtc_eps_scale() {
  const char* e = getenv("GB_PQTC_EPS");
  return e ? (float)atof(e) : 1.0f;
}

// List-major IVF-PQ scan (kernels_pqtc.cu): exact scan of the first pa probes -> per-query bound ->
// tensor-core filter over the remaining probes -> exact re-score of the candidates.  Returns 1 when
// the batch / shape does not qualify (caller runs the exact kernel over all probes).
int IVFPQIndex::scan_listmajor_pq(const FilterArgs& f, int metric, int nq, const float* xq, int kk, const float* ip,
                                  const int32_t* probe_ids, const float* coarse_dis, int nprobe,
                                  unsigned long long* adc_out, bool need_sorted, Scratch& s) {
  const int mode = pqtc_mode();
  if (!mode || !tc_enabled() || !d_cb16_ || !pqtc_supported(M_, dsub_) || dpad_ != d_) return 1;
  if (kk > 2048 || nprobe < 2 || nprobe > 65535 || nq > 65535) return 1;  // (query, probe) travel as 16-bit fields of a candidate record
  const int64_t npairs = (int64_t)nq * nprobe;
  if (mode != 2 && npairs < (int64_t)nlist_ * 32) return 1;  // < 32 queries per list on average
  if (metric == kMetricL2) {
    const int nr = ensure_pq_norms(s.stream());
    if (nr) return nr;
  }
  cudaStream_t st = s.stream();
  ListDirectory dir = lists_->directory();
  // phase A, per query: its first probes in full -- the fewest whose lists hold >= 4 k' entries together (so that its
  // k'-th exact score is a tight bound B_q), at most pa_max; phase B filters the other probes.  GB_PQTC_PA=n: the
  // first n probes of every query; GB_PQTC_TARGET=t: t k' entries instead of 4 k'.
  int pa_max = std::min(nprobe - 1, 8);
  long long pa_target = 4 * (long long)kk;
  if (const char* e = getenv("GB_PQTC_PA")) {
    pa_max = std::max(1, std::min(nprobe - 1, atoi(e)));
    pa_target = LLONG_MAX;
  }
  if (const char* e = getenv("GB_PQTC_TARGET")) pa_target = std::max(1LL, atoll(e)) * kk;
  const int cap = std::max(2048, std::min(8192, next_pow2(8 * kk)));
  const int nsm = sm_count(device_);
  snprintf(last_scan_info_, sizeof(last_scan_info_),
           "{\"phase_a_max_probes\": %d, \"phase_a_target_entries\": %lld, \"candidate_cap\": %d, \"kprime\": %d}", pa_max,
           pa_target == LLONG_MAX ? -1LL : pa_target, cap, kk);
  GB_ALLOC(d_probes_a, int32_t, npairs, s);
  GB_ALLOC(d_probes_b, int32_t, npairs, s);
  GB_ALLOC(d_row_limit, int, npairs, s);
  GB_CUDA(launch_pqtc_plan_phase_a(probe_ids, npairs, nprobe, pa_max, pa_target, dir.len, d_probes_a, d_probes_b, d_row_limit,
                                   st));

  // ---- phase A: exact keys of each query's leading probes ----
  const int pgA = nq >= nsm * 4 ? std::min(pa_max, 32) : 1;  // one CTA per query when there are queries enough
  const int ngA = (pa_max + pgA - 1) / pgA;
  GB_ALLOC(partA, unsigned long long, (size_t)nq * ngA * kk, s);
  stage_begin("pq_phaseA_exact_scan", st);
  // one group per query: its k' best come back unordered with the largest (the bound) in slot k' - 1 -- nobody needs
  // them sorted (launch_select_keys below, used when the probes were split over groups, sorts anyway)
  GB_CUDA(launch_ivfpq_scan(ip, nq, d_probes_a, coarse_dis, pa_max, pgA, dir, M_, d_table_, kk, metric, f, partA, st, nprobe,
                            nullptr, 0, d_row_limit, /*sorted_out=*/ngA > 1));
  unsigned long long* keysA = partA;
  if (ngA > 1) {
    keysA = s.alloc_n<unsigned long long>((size_t)nq * kk);
    if (!keysA) return -1;
    GB_CUDA(launch_select_keys(partA, (int64_t)ngA * kk, nq, ngA * kk, kk, keysA, kk, st));
  }
  stage_end(st);

  // ---- phase B: group the remaining pairs by list, stage the operand tiles, filter ----
  const int nseg = (int)std::min<int64_t>(64, std::max<int64_t>(1, (lists_->max_len() + kLmkSegRows - 1) / kLmkSegRows));
  const int64_t max_groups = npairs / 128 + nlist_;
  const int64_t max_items = max_groups * nseg;
  if (max_items > INT32_MAX) return 1;
  GB_ALLOC(d_cnt, int32_t, nlist_, s);
  GB_ALLOC(d_start, int32_t, nlist_, s);
  GB_ALLOC(d_cursor, int32_t, nlist_, s);
  GB_ALLOC(d_item_start, int32_t, nlist_, s);
  GB_ALLOC(d_grp_start, int32_t, nlist_, s);
  GB_ALLOC(d_totals, int64_t, 3, s);
  GB_ALLOC(d_pair_j, int64_t, npairs, s);
  GB_ALLOC(d_items, LmTile, max_items, s);
  GB_ALLOC(d_cand_cnt, int, nq, s);
  const size_t tile_bytes = (size_t)(d_ / 8) * 2048;
  const size_t a_bytes = (size_t)max_groups * tile_bytes;
  const size_t meta_bytes = (size_t)max_groups * 128 * pqtc_pair_meta_bytes();
  const size_t cand_bytes = (size_t)nq * cap * 8;
  unsigned char* big = static_cast<unsigned char*>(big_acquire(a_bytes + meta_bytes + cand_bytes, st));
  if (!big) return -1;
  auto rel_fn = [this, big, st](void*) { big_release(big, st); };
  std::unique_ptr<void, decltype(rel_fn)> rel(big, rel_fn);
  unsigned char* a_scratch = big;
  void* meta = big + a_bytes;
  unsigned long long* cand = reinterpret_cast<unsigned long long*>(big + a_bytes + meta_bytes);
  stage_begin("pq_group_and_stage_pairs", st);
  GB_CUDA(cudaMemsetAsync(d_cand_cnt, 0, sizeof(int) * nq, st));
  GB_CUDA(launch_lmk_group(d_probes_b, npairs, dir, nseg, d_cnt, d_start, d_cursor, d_item_start, d_grp_start, d_totals,
                           d_pair_j, d_items, st));
  GB_CUDA(launch_pq_stage_pairs(xq, dpad_, d_, d_centroids_, dpad_, d_items, (int)max_items, d_totals, d_pair_j, nprobe,
                                coarse_dis, keysA, kk, kk, d_cbnrm_ + (size_t)M_ * 256, f, metric, pqtc_eps_scale(), a_scratch,
                                meta, d_cand_cnt, cap, d_row_limit, st));
  stage_end(st);
  scan_timer_begin(st);  // the dominant kernel: the roofline in bench.py is this launch alone
  stage_begin("pqtc_scan_kernel", st);
  GB_CUDA(launch_pqtc_scan(a_scratch, meta, d_cb16_, pqn_.base, pqn_.d_off, d_items, (int)max_items, d_totals, dir, M_, dsub_, f, metric,
                           d_cand_cnt, cand, cap, nsm, st));
  stage_end(st);
  scan_timer_end(st);
  stage_begin("pq_rescore_and_fallback", st);

  // ---- phase C: candidates -> reference arithmetic, merged with phase A's keys ----
  GB_CUDA(launch_pq_rescore(ip, nq, probe_ids, coarse_dis, nprobe, dir, M_, d_table_, d_cand_cnt, cand, cap, keysA, kk, kk,
                            metric, d_row_limit, f, need_sorted, adc_out, st));
  // queries whose candidate list overflowed (or that had no bound): exact kernel over all probes, flag-gated
  const int ngF = (nprobe + 31) / 32;
  GB_ALLOC(partF, unsigned long long, (size_t)nq * ngF * kk, s);
  GB_CUDA(launch_ivfpq_scan(ip, nq, probe_ids, coarse_dis, nprobe, 32, dir, M_, d_table_, kk, metric, f, partF, st, nprobe,
                            d_cand_cnt, cap));
  GB_CUDA(launch_pq_fallback_merge(d_cand_cnt, cap, nq, partF, ngF, kk, adc_out, st));
  stage_end(st);
  if (const char* dump = getenv("GB_PQTC_DUMP")) {  // debugging aid: candidate lists + phase A keys to a file
    std::vector<int> h(nq);
    std::vector<unsigned long long> hc((size_t)nq * cap), hk((size_t)nq * kk);
    GB_CUDA(cudaMemcpyAsync(h.data(), d_cand_cnt, sizeof(int) * nq, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaMemcpyAsync(hc.data(), cand, hc.size() * 8, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaMemcpyAsync(hk.data(), keysA, hk.size() * 8, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaStreamSynchronize(st));
    int64_t ht[3];
    GB_CUDA(cudaMemcpy(ht, d_totals, sizeof(ht), cudaMemcpyDeviceToHost));
    std::vector<int64_t> hpj((size_t)npairs);
    std::vector<LmTile> hit((size_t)ht[1]);
    GB_CUDA(cudaMemcpy(hpj.data(), d_pair_j, hpj.size() * 8, cudaMemcpyDeviceToHost));
    GB_CUDA(cudaMemcpy(hit.data(), d_items, hit.size() * sizeof(LmTile), cudaMemcpyDeviceToHost));
    if (FILE* fp = fopen(dump, "wb")) {
      const int hdr[8] = {nq, cap, kk, pa_max, (int)ht[1], (int)npairs, (int)sizeof(LmTile), (int)ht[2]};
      fwrite(hdr, 4, 8, fp);
      fwrite(h.data(), 4, h.size(), fp);
      fwrite(hc.data(), 8, hc.size(), fp);
      fwrite(hk.data(), 8, hk.size(), fp);
      fwrite(hpj.data(), 8, hpj.size(), fp);
      fwrite(hit.data(), sizeof(LmTile), hit.size(), fp);
      fclose(fp);
    }
  }
  if (getenv("GB_PQTC_STATS")) {  // diagnostics: candidates per query, overflowed queries
    std::vector<int> h(nq);
    GB_CUDA(cudaMemcpyAsync(h.data(), d_cand_cnt, sizeof(int) * nq, cudaMemcpyDeviceToHost, st));
    GB_CUDA(cudaStreamSynchronize(st));
    long long tot = 0, over = 0, mx = 0;
    for (int v : h) {
      if (v > cap) over++;
      else tot += v, mx = std::max<long long>(mx, v);
    }
    unsigned long long dc[4];
    pqtc_debug_counters(dc, true);
    int64_t ht[3];
    GB_CUDA(cudaMemcpy(ht, d_totals, sizeof(ht), cudaMemcpyDeviceToHost));
    std::vector<LmTile> hit((size_t)ht[1]);
    GB_CUDA(cudaMemcpy(hit.data(), d_items, hit.size() * sizeof(LmTile), cudaMemcpyDeviceToHost));
    long long tiles = 0, pair_rows = 0, rows = 0;
    for (const LmTile& t : hit) {
      tiles += (t.nrows + 127) / 128;
      pair_rows += (long long)t.npairs * t.nrows;
      rows += t.nrows;
    }
    fprintf(stderr, "[pqtc] nq=%d k'=%d pa_max=%d cap=%d: candidates mean %.1f max %lld, overflowed queries %lld, dbg counters %llu %llu; "
            "items %lld groups %lld tiles(128x128) %lld rows decoded %lld pair-rows %lld (tile fill %.3f)\n",
            nq, kk, pa_max, cap, nq > over ? (double)tot / (nq - over) : 0.0, mx, over, dc[0], dc[1], (long long)ht[1], (long long)ht[0],
            tiles, rows, pair_rows, tiles ? (double)pair_rows / ((double)tiles * 128 * 128) : 0.0);
  }
  return 0;
}

// GammaIVFPQIndex::search_preassigned (gamma_index_ivfpq.cc:730-947)
int IVFPQIndex::scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                         const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
                         Scratch& s) {
  cudaStream_t st = s.stream();
  if (metric != mp_.metric) {
    set_last_error("IVFPQ: per-request metric must equal the trained metric");
    return -1;
  }
  // recall_num / re-rank semantics: gamma_index_ivfpq.cc:764-770
  const bool rerank = ctx.params.recall_num > 0;
  int kk = k;
  if (ctx.params.recall_num > k) kk = ctx.params.recall_num;
  if (kk > 4096) {
    set_last_error("IVFPQ: recall_num / topn above 4096 is not supported");
    return -1;
  }
  GB_ALLOC(ip, float, (size_t)nq * M_ * 256, s);
  {
    StageScope stage(this, "pq_ip_table", st);
    GB_CUDA(launch_pq_ip_table(xq, dpad_, nq, d_pq_, M_, dsub_, ip, st));
  }
  unsigned long long* adc = out_keys;
  if (rerank) {
    adc = s.alloc_n<unsigned long long>((size_t)nq * kk);
    if (!adc) return -1;
  }
  // the exact re-rank takes its candidates in any order; without it the ADC keys are the result and must be sorted
  int lm = scan_listmajor_pq(f, metric, nq, xq, kk, ip, probe_ids, coarse_dis, nprobe, adc, !rerank, s);
  if (lm < 0) return -1;
  if (lm == 0) {
    last_scan_kernel_ = "pqtc_scan_kernel";
  } else {
    snprintf(last_scan_info_, sizeof(last_scan_info_), "{}");
    const int nsm = sm_count(device_);
    int pg = (int)std::min<int64_t>(32, std::max<int64_t>(1, (int64_t)nprobe * nq / ((int64_t)nsm * 32)));
    int ngroups = (nprobe + pg - 1) / pg;
    GB_ALLOC(partial, unsigned long long, (size_t)nq * ngroups * kk, s);
    last_scan_kernel_ = "ivfpq_scan_kernel";
    scan_timer_begin(st);
    stage_begin("ivfpq_scan_kernel", st);
    GB_CUDA(launch_ivfpq_scan(ip, nq, probe_ids, coarse_dis, nprobe, pg, lists_->directory(), M_, d_table_, kk, metric, f,
                              partial, st));
    stage_end(st);
    scan_timer_end(st);
    if (ngroups > 1) {
      GB_CUDA(launch_select_keys(partial, (int64_t)ngroups * kk, nq, ngroups * kk, kk, adc, kk, st));
    } else {
      GB_CUDA(cudaMemcpyAsync(adc, partial, (size_t)nq * kk * 8, cudaMemcpyDeviceToDevice, st));
    }
  }
  if (rerank) {
    // "for opq, rerank need raw vector" (gamma_index_ivfpq.cc:735): original queries against the raw store
    StageScope stage(this, "rerank_kernel", st);
    GB_CUDA(launch_rerank(adc, kk, nq, raw_queries_for(xq), dpad_, dpad_, store_->d_segs(), store_->seg_shift(), dpad_, k,
                          metric, f, out_keys, st));
  }
  return 0;
}

int IVFPQIndex::search_preassigned_host(const SearchContext& ctx, int nq, const float* x, int k, const int64_t* keys,
                                        const float* coarse_dis, int nprobe, float* out_dis, int64_t* out_ids) {
  return IVFFlatIndex::search_preassigned_host(ctx, nq, x, k, keys, coarse_dis, nprobe, out_dis, out_ids);
}

// ------------------------------------------------------------------------------------------
IVFRaBitQIndex::IVFRaBitQIndex(int d, const ModelParams& mp, int device, int seg_shift)
    : IVFFlatIndex(d, mp, device, seg_shift, "IVFRABITQ") {}

int IVFRaBitQIndex::training_threshold() const {
  // gamma_index_ivfrabitq.cc:243-290: the IVFPQ rule, default max(nlist*200, 256) clamped to [39, 256] * nlist
  int64_t t = mp_.training_threshold ? mp_.training_threshold : std::max<int64_t>((int64_t)nlist_ * 200, 256);
  if (t < nlist_)
    t = (int64_t)nlist_ * 39;
  else if (t > (int64_t)nlist_ * 256)
    t = (int64_t)nlist_ * 256;
  return (int)t;
}

// a search's qb outside [0, 8] is not an error: the model's qb is used (gamma_index_ivfrabitq.cc:180-232)
int IVFRaBitQIndex::resolve_qb(const SearchContext& ctx) const {
  const int qb = ctx.params.qb;
  if (qb >= 0 && qb <= 8) return qb;
  if (qb != -1) fprintf(stderr, "IVFRABITQ: invalid qb = %d in search, using the model's qb = %d\n", qb, mp_.qb);
  return mp_.qb;
}

// GammaIVFRaBitQIndex::Add (gamma_index_ivfrabitq.cc:304-418): code of the residual against the assigned list
int IVFRaBitQIndex::append_batch(const float* x, int64_t n, int64_t vid0, const int32_t* d_list, const int32_t* d_pos,
                                 const int32_t* d_assign, Scratch& s) {
  (void)d_assign;
  cudaStream_t st = s.stream();
  const int cs = code_bytes();
  GB_ALLOC(codes, uint8_t, (size_t)n * cs, s);
  GB_CUDA(launch_rabitq_encode(x, dpad_, n, d_, d_centroids_, dpad_, d_list, mp_.nb_bits, mp_.metric, codes, st));
  GB_CUDA(launch_ivf_append_codes(codes, n, cs, d_list, d_pos, reinterpret_cast<uint8_t* const*>(lists_->d_data()),
                                  lists_->d_ids(), vid0, st));
  return 0;
}

int IVFRaBitQIndex::encode_host(const float* x, int64_t n, const int64_t* assign, uint8_t* codes_out) {
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  Scratch s(st);
  const int cs = code_bytes();
  GB_ALLOC(dx, float, (size_t)n * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dx, 0, (size_t)n * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dx, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, n, cudaMemcpyHostToDevice, st));
  std::vector<int32_t> h(n);
  for (int64_t i = 0; i < n; i++) h[i] = (int32_t)assign[i];
  GB_ALLOC(da, int32_t, n, s);
  GB_CUDA(cudaMemcpyAsync(da, h.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
  GB_ALLOC(codes, uint8_t, (size_t)n * cs, s);
  GB_CUDA(launch_rabitq_encode(dx, dpad_, n, d_, d_centroids_, dpad_, da, mp_.nb_bits, mp_.metric, codes, st));
  GB_CUDA(cudaMemcpyAsync(codes_out, codes, (size_t)n * cs, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

int IVFRaBitQIndex::query_consts_host(int nq, const float* x, const int64_t* keys, int nprobe, int qb, bool centered,
                                      float* out) {
  if (qb < 0 || qb > 8) {
    set_last_error("qb should be in [0, 8]");
    return -1;
  }
  cudaSetDevice(device_);
  cudaStream_t st = thread_stream(device_);
  std::shared_lock<std::shared_mutex> lk(mu_);
  Scratch s(st);
  const size_t npairs = (size_t)nq * nprobe;
  GB_ALLOC(dq, float, (size_t)nq * dpad_, s);
  GB_CUDA(cudaMemsetAsync(dq, 0, (size_t)nq * dpad_ * 4, st));
  GB_CUDA(cudaMemcpy2DAsync(dq, (size_t)dpad_ * 4, x, (size_t)d_ * 4, (size_t)d_ * 4, nq, cudaMemcpyHostToDevice, st));
  std::vector<int32_t> h(npairs);
  for (size_t i = 0; i < npairs; i++) h[i] = (int32_t)keys[i];
  GB_ALLOC(ids, int32_t, npairs, s);
  GB_CUDA(cudaMemcpyAsync(ids, h.data(), npairs * 4, cudaMemcpyHostToDevice, st));
  GB_ALLOC(consts, float, npairs * kRabitqConsts, s);
  const int W = (d_ + 31) / 32;
  uint32_t* planes = qb > 0 ? s.alloc_n<uint32_t>(npairs * qb * W) : nullptr;
  if (qb > 0 && !planes) return -1;
  GB_CUDA(launch_rabitq_query_prep(dq, dpad_, nq, d_, ids, nprobe, d_centroids_, dpad_, nlist_, qb, centered, mp_.nb_bits,
                                   mp_.metric, consts, planes, st));
  GB_CUDA(cudaMemcpyAsync(out, consts, npairs * kRabitqConsts * 4, cudaMemcpyDeviceToHost, st));
  GB_CUDA(cudaStreamSynchronize(st));
  return 0;
}

// GammaIVFRaBitQIndex::search_preassigned (gamma_index_ivfrabitq.h:59-268, .cc:551-602) with every valid entry scored
// by the full nb_bits estimate; recall_num re-ranks that many candidates exactly from the raw vectors
int IVFRaBitQIndex::scan_dev(const SearchContext& ctx, const FilterArgs& f, int metric, int nq, const float* xq, int k,
                             const int32_t* probe_ids, const float* coarse_dis, int nprobe, unsigned long long* out_keys,
                             Scratch& s) {
  (void)coarse_dis;
  cudaStream_t st = s.stream();
  if (metric != mp_.metric) {
    set_last_error("IVFRABITQ: per-request metric must equal the trained metric");
    return -1;
  }
  const bool rerank = ctx.params.recall_num > 0;
  int kk = k;
  if (ctx.params.recall_num > k) kk = ctx.params.recall_num;
  if (kk > 4096) {
    set_last_error("IVFRABITQ: recall_num / topn above 4096 is not supported");
    return -1;
  }
  const int qb = resolve_qb(ctx);
  const size_t npairs = (size_t)nq * nprobe;
  const int W = (d_ + 31) / 32;
  GB_ALLOC(consts, float, npairs * kRabitqConsts, s);
  uint32_t* planes = nullptr;  // qb = 0: the scan forms the float residual itself
  if (qb > 0) {
    planes = s.alloc_n<uint32_t>(npairs * qb * W);
    if (!planes) return -1;
  }
  {
    StageScope stage(this, "rabitq_query_prep", st);
    GB_CUDA(launch_rabitq_query_prep(xq, dpad_, nq, d_, probe_ids, nprobe, d_centroids_, dpad_, nlist_, qb,
                                     ctx.params.centered, mp_.nb_bits, metric, consts, planes, st));
  }
  unsigned long long* cand = out_keys;
  if (rerank) {
    cand = s.alloc_n<unsigned long long>((size_t)nq * kk);
    if (!cand) return -1;
  }
  const int nsm = sm_count(device_);
  const int pg = (int)std::min<int64_t>(32, std::max<int64_t>(1, (int64_t)nprobe * nq / ((int64_t)nsm * 32)));
  const int ngroups = (nprobe + pg - 1) / pg;
  GB_ALLOC(partial, unsigned long long, (size_t)nq * ngroups * kk, s);
  last_scan_kernel_ = "rabitq_scan_kernel";
  snprintf(last_scan_info_, sizeof(last_scan_info_), "{\"nb_bits\": %d, \"qb\": %d, \"code_size\": %d, \"pg\": %d}",
           mp_.nb_bits, qb, code_bytes(), pg);
  scan_timer_begin(st);
  stage_begin("rabitq_scan_kernel", st);
  GB_CUDA(launch_rabitq_scan(consts, planes, xq, dpad_, d_centroids_, dpad_, nq, probe_ids, nprobe, pg, lists_->directory(), d_, mp_.nb_bits, qb,
                             kk, metric, f, partial, st));
  stage_end(st);
  scan_timer_end(st);
  if (ngroups > 1) {
    GB_CUDA(launch_select_keys(partial, (int64_t)ngroups * kk, nq, ngroups * kk, kk, cand, kk, st));
  } else {
    GB_CUDA(cudaMemcpyAsync(cand, partial, (size_t)nq * kk * 8, cudaMemcpyDeviceToDevice, st));
  }
  if (rerank) {
    StageScope stage(this, "rerank_kernel", st);
    GB_CUDA(launch_rerank(cand, kk, nq, xq, dpad_, dpad_, store_->d_segs(), store_->seg_shift(), dpad_, k, metric, f,
                          out_keys, st));
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
Index* create_index(const std::string& type, int d, const ModelParams& mp, int device, int seg_shift) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) {
    set_last_error("no CUDA device " + std::to_string(device) + " (this engine has no CPU path)");
    return nullptr;
  }
  if (d <= 0) {
    set_last_error("invalid dimension");
    return nullptr;
  }
  if (type == "FLAT") return new FlatIndex(d, mp, device, seg_shift);
  if (type == "IVFFLAT") {
    if (mp.ncentroids <= 0 || mp.nprobe > mp.ncentroids) {  // gamma_index_ivfflat.cc:277-286
      set_last_error("nprobe should be less than ncentroids");
      return nullptr;
    }
    return new IVFFlatIndex(d, mp, device, seg_shift);
  }
  if (type == "IVFPQ") {
    int M = mp.nsubvector > 0 ? mp.nsubvector : d / 2;
    if (M <= 0 || d % M != 0) {  // gamma_index_ivfpq.cc:125-133
      set_last_error("Dimension [" + std::to_string(d) + "] cannot divide by nsubvector [" + std::to_string(M) + "].");
      return nullptr;
    }
    if (mp.nbits != 8) {
      set_last_error("only nbits_per_idx = 8 is supported");
      return nullptr;
    }
    if (mp.opq_nsubvector > 0 && d % mp.opq_nsubvector != 0) {  // gamma_index_ivfpq.cc:169-176
      set_last_error(std::to_string(d) + " % " + std::to_string(mp.opq_nsubvector) +
                     " != 0, opq nsubvector should be divisible by dimension.");
      return nullptr;
    }
    if (mp.ncentroids <= 0 || mp.nprobe > mp.ncentroids) {
      set_last_error("nprobe should be less than ncentroids");
      return nullptr;
    }
    return new IVFPQIndex(d, mp, device, seg_shift);
  }
  if (type == "IVFRABITQ") {  // GammaIVFRaBitQIndex model-parameter checks (gamma_index_ivfrabitq.h:335-537)
    if (mp.nb_bits < 1 || mp.nb_bits > 9) {
      set_last_error("invalid nb_bits =" + std::to_string(mp.nb_bits) + " should be integer in [1, 9]");
      return nullptr;
    }
    if (mp.qb < 0 || mp.qb > 8) {
      set_last_error("invalid qb =" + std::to_string(mp.qb) + " should be integer in [0, 8]");
      return nullptr;
    }
    if (mp.ncentroids <= 0 || mp.nprobe > mp.ncentroids) {
      set_last_error("nprobe should less than ncentroids");
      return nullptr;
    }
    if (d > 8192) {  // the scan's integer core is exact in 32 bits up to here
      set_last_error("IVFRABITQ supports dimensions up to 8192");
      return nullptr;
    }
    if (!rabitq_scan_supported(d, mp.nb_bits)) {  // two stages of at least 16 codes must fit in shared memory
      set_last_error("IVFRABITQ: code_size " + std::to_string(rabitq_code_size(d, mp.nb_bits)) + " bytes (d=" +
                     std::to_string(d) + ", nb_bits=" + std::to_string(mp.nb_bits) +
                     ") is too large for the scan's shared-memory ring; use fewer nb_bits");
      return nullptr;
    }
    return new IVFRaBitQIndex(d, mp, device, seg_shift);
  }
  set_last_error("unsupported index type " + type);
  return nullptr;
}

// ------------------------------------------------------------------------------------------
namespace {
// Router merge (mergeSortedArrays, client.go:1530-1589) on device: per query, k-way merge keyed by
// (score, later partition first).  Input scores are already sorted per partition.
template <bool FROM_KEYS>  // FROM_KEYS: `ids` holds the partitions' result keys (score bits << 32 | local id)
__global__ void merge_partitions_kernel(const float* __restrict__ dis, const int64_t* __restrict__ ids, int nparts,
                                        int nq, int k, int metric, float* __restrict__ out_dis,
                                        int64_t* __restrict__ out_ids) {
  extern __shared__ unsigned long long mk[];  // [NP] keys, then [NP] payload
  const int q = blockIdx.x;
  const int total = nparts * k;
  int NP = 1;
  while (NP < total) NP <<= 1;
  unsigned long long* pay = mk + NP;
  for (int i = threadIdx.x; i < NP; i += blockDim.x) {
    unsigned long long key = kKeySentinel, pl = 0;
    if (i < total) {
      int p = i / k, j = i - p * k;
      // low word: later partition first, then rank inside the partition
      const uint32_t lo = ((uint32_t)(nparts - 1 - p) << 16) | (uint32_t)j;
      if (FROM_KEYS) {
        const unsigned long long pk = (unsigned long long)ids[((int64_t)p * nq + q) * k + j];
        if (pk != kKeySentinel) {
          key = make_key((uint32_t)(pk >> 32), lo);
          pl = ((unsigned long long)p << 32) | (uint32_t)pk;
        }
      } else {
        int64_t id = ids[((int64_t)p * nq + q) * k + j];
        if (id >= 0) {
          float s = dis[((int64_t)p * nq + q) * k + j];
          key = make_key(score2ord(s, metric), lo);
          pl = ((unsigned long long)p << 32) | (uint32_t)id;
        }
      }
    }
    mk[i] = key;
    pay[i] = pl;
  }
  __syncthreads();
  // bitonic sort on keys carrying the payload
  for (int kk = 2; kk <= NP; kk <<= 1)
    for (int j = kk >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < NP; i += blockDim.x) {
        int ixj = i ^ j;
        if (ixj > i) {
          unsigned long long a = mk[i], b = mk[ixj];
          bool up = ((i & kk) == 0);
          if ((a > b) == up) {
            mk[i] = b;
            mk[ixj] = a;
            unsigned long long t = pay[i];
            pay[i] = pay[ixj];
            pay[ixj] = t;
          }
        }
      }
      __syncthreads();
    }
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    if (i < NP && mk[i] != kKeySentinel) {
      out_dis[(int64_t)q * k + i] = ord2score((uint32_t)(mk[i] >> 32), metric);
      out_ids[(int64_t)q * k + i] = (int64_t)pay[i];
    } else {
      out_dis[(int64_t)q * k + i] = metric == kMetricL2 ? FLT_MAX : -FLT_MAX;
      out_ids[(int64_t)q * k + i] = -1;
    }
  }
}
}  // namespace

int merge_partition_keys_device(const unsigned long long* keys, int nparts, int nq, int k, int metric, float* out_dis,
                                int64_t* out_ids, cudaStream_t st) {
  if (nq <= 0) return 0;
  int NP = next_pow2(nparts * k);
  if (nparts > 65535 || k > 65535 || NP > 8192) {
    set_last_error("merge_partitions: nparts*k too large");
    return -1;
  }
  size_t smem = (size_t)NP * 16;
  if (smem > 48 * 1024)
    GB_CUDA(cudaFuncSetAttribute(merge_partitions_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  merge_partitions_kernel<true><<<nq, 256, smem, st>>>(nullptr, reinterpret_cast<const int64_t*>(keys), nparts, nq, k, metric,
                                                       out_dis, out_ids);
  note_launch();
  GB_CUDA(cudaGetLastError());
  return 0;
}

int merge_partitions_device(const float* dis, const int64_t* ids, int nparts, int nq, int k, int metric, float* out_dis,
                            int64_t* out_ids, cudaStream_t st) {
  if (nq <= 0) return 0;
  int NP = next_pow2(nparts * k);
  if (nparts > 65535 || k > 65535 || NP > 8192) {
    set_last_error("merge_partitions: nparts*k too large");
    return -1;
  }
  size_t smem = (size_t)NP * 16;
  if (smem > 48 * 1024)
    GB_CUDA(cudaFuncSetAttribute(merge_partitions_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  merge_partitions_kernel<false><<<nq, 256, smem, st>>>(dis, ids, nparts, nq, k, metric, out_dis, out_ids);
  note_launch();
  GB_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace gb
