// K8r / K4r / K5q: RaBitQ encoding, per-(query, probe) query quantisation and the IVFRABITQ scan.
//
// Replaces, in the reference (faiss IndexIVFRaBitQ behind gamma_index_ivfrabitq.{h,cc}):
//   rabitq.compute_codes_core(x, code, 1, centroid)  (gamma_index_ivfrabitq.cc:304-418)   -> rabitq_encode
//   the scanner's per-list query set-up (gamma_index_ivfrabitq.h:59-120)                   -> rabitq_query_prep
//   the list scan (gamma_index_ivfrabitq.h:120-268), with every valid entry scored by the
//   full nb_bits estimate ("refine_all", DESIGN.md section 5b)                             -> rabitq_scan
//
// Code layout and estimator: DESIGN.md section 5b and tests/rabitq_oracle.py.  Every float value is
// an unfused __f*_rn operation in the oracle's order; every float reduction runs over j = 0 .. d-1.
// The integer core of the scan is exact: the total code t_j (nb_bits planes, sign plane on top) and
// the qb-bit query qq_j (qb planes) give  sum_j qq_j t_j = sum_k sum_m 2^(k+m) popc(T_k & Q_m).
#include <float.h>

#include "common.cuh"
#include "kernels.h"

namespace gb {

namespace {

constexpr int RQ_NSCALE = 64;  // candidate rescale factors of the extra-bit search
constexpr int RQ_ENC_NT = 128;

__device__ __forceinline__ void st_f32(uint8_t* p, float v) {
  const uint32_t u = __float_as_uint(v);
  p[0] = (uint8_t)u, p[1] = (uint8_t)(u >> 8), p[2] = (uint8_t)(u >> 16), p[3] = (uint8_t)(u >> 24);
}

// One thread per vector running the oracle's sequential loops (encoding is not the hot path; byte
// equality with the oracle is what matters).
__global__ void __launch_bounds__(RQ_ENC_NT)
    rabitq_encode_kernel(const float* __restrict__ x, int64_t ldx, int64_t n, int d, const float* __restrict__ coarse,
                         int64_t ldc, const int32_t* __restrict__ assign, int nb_bits, int metric, uint8_t* __restrict__ codes,
                         int cs) {
  const int64_t i = (int64_t)blockIdx.x * RQ_ENC_NT + threadIdx.x;
  if (i >= n) return;
  const float* xi = x + i * ldx;
  const int a = assign[i];
  const float* ci = coarse + (int64_t)(a < 0 ? 0 : a) * ldc;  // rows with list -1 are not appended
  uint8_t* out = codes + i * cs;
  const int P = (d + 7) >> 3;
  float rn = 0.f, cr = 0.f, sabs = 0.f, m = 0.f;
  for (int j = 0; j < d; j++) {
    const float c = ci[j], r = __fsub_rn(xi[j], c), ra = fabsf(r);
    rn = __fadd_rn(rn, __fmul_rn(r, r));
    cr = __fadd_rn(cr, __fmul_rn(c, r));
    sabs = __fadd_rn(sabs, ra);
    m = fmaxf(m, ra);
  }
  for (int by = 0; by < P; by++) {
    uint32_t v = 0;
    for (int t = 0; t < 8; t++) {
      const int j = by * 8 + t;
      if (j < d && __fsub_rn(xi[j], ci[j]) > 0.f) v |= 1u << t;
    }
    out[by] = (uint8_t)v;
  }
  const float half = __fmul_rn(sabs, 0.5f);
  st_f32(out + P, metric == kMetricL2 ? rn : cr);
  st_f32(out + P + 4, sabs > 0.f ? __fdiv_rn(rn, half) : 0.f);
  if (nb_bits == 1) return;
  // 1-bit error factor |r| sqrt((1 - dp^2) / dp^2) / sqrt(d - 1), dp = sum|r_j| / (|r| sqrt d)
  const float nr = __fsqrt_rn(rn);
  const float dp = __fdiv_rn(sabs, __fmul_rn(nr, __fsqrt_rn((float)d)));
  const float t2 = __fmul_rn(dp, dp);
  const float u = fmaxf(__fdiv_rn(__fsub_rn(1.f, t2), t2), 0.f);
  float fe = __fdiv_rn(__fmul_rn(nr, __fsqrt_rn(u)), __fsqrt_rn((float)max(d - 1, 1)));
  if (!(dp > 0.f && d > 1)) fe = 0.f;
  st_f32(out + P + 8, fe);
  // extra bits: the rescale s_i = (2^ex (i+1)/64) / max|r_j| maximising the cosine with the code
  const int ex = nb_bits - 1, emax = (1 << ex) - 1;
  const float msafe = m > 0.f ? m : 1.f;
  float best = -INFINITY, bs = 0.f, bip = 0.f;
  for (int s_i = 0; s_i < RQ_NSCALE; s_i++) {
    const float kf = __fdiv_rn((float)(s_i + 1), (float)RQ_NSCALE);
    const float s = __fdiv_rn(__fmul_rn((float)(1 << ex), kf), msafe);
    float ip = 0.f;
    long long ny = 0;
    for (int j = 0; j < d; j++) {
      const float ra = fabsf(__fsub_rn(xi[j], ci[j]));
      const int e = min((int)floorf(__fmul_rn(ra, s)), emax);
      const int w = 2 * e + 1;
      ip = __fadd_rn(ip, __fmul_rn(ra, (float)w));
      ny += (long long)w * w;
    }
    const float cosv = __fdiv_rn(ip, __fsqrt_rn(__ll2float_rn(ny)));
    if (cosv > best) best = cosv, bs = s, bip = ip;
  }
  const int o = P + 12;
  for (int k = 0; k < ex; k++) {
    for (int by = 0; by < P; by++) {
      uint32_t v = 0;
      for (int t = 0; t < 8; t++) {
        const int j = by * 8 + t;
        if (j >= d) break;
        const float r = __fsub_rn(xi[j], ci[j]);
        const int e = m > 0.f ? min((int)floorf(__fmul_rn(fabsf(r), bs)), emax) : 0;
        const int ep = r > 0.f ? e : emax - e;
        v |= (uint32_t)((ep >> k) & 1) << t;
      }
      out[o + k * P + by] = (uint8_t)v;
    }
  }
  st_f32(out + o + ex * P, bip > 0.f ? __fdiv_rn(rn, __fmul_rn(bip, 0.5f)) : 0.f);
}

// One CTA per (query, probe): residual, its range, the qb-bit query as bit-planes (one ballot per
// plane and 32 dimensions) and the pair's constants.
constexpr int RQ_PREP_NT = 128;

__global__ void __launch_bounds__(RQ_PREP_NT)
    rabitq_query_prep_kernel(const float* __restrict__ xq, int64_t ldq, int nprobe, const int32_t* __restrict__ probe_ids,
                             const float* __restrict__ coarse, int64_t ldc, int nlist, int d, int qb, int centered,
                             int nb_bits, int metric, float* __restrict__ consts, uint32_t* __restrict__ planes) {
  extern __shared__ float qr[];  // [d]
  __shared__ float s_min[RQ_PREP_NT / 32], s_max[RQ_PREP_NT / 32];
  __shared__ int s_sq;
  const int64_t pair = blockIdx.x;
  const int q = (int)(pair / nprobe);
  const int l = probe_ids[pair];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int W = (d + 31) >> 5;
  float* cst = consts + pair * kRabitqConsts;
  if (l < 0 || l >= nlist) {  // not enough centroids: the scan skips the pair
    if (tid < kRabitqConsts) cst[tid] = 0.f;
    return;
  }
  const float* xr = xq + (int64_t)q * ldq;
  const float* cr = coarse + (int64_t)l * ldc;
  float mn = INFINITY, mx = -INFINITY;
  for (int j = tid; j < d; j += RQ_PREP_NT) {
    const float v = __fsub_rn(xr[j], cr[j]);
    qr[j] = v;
    if (centered) {
      mx = fmaxf(mx, fabsf(v));
    } else {
      mn = fminf(mn, v), mx = fmaxf(mx, v);
    }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, off));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, off));
  }
  if (lane == 0) s_min[warp] = mn, s_max[warp] = mx;
  if (tid == 0) s_sq = 0;
  __syncthreads();
  mn = s_min[0], mx = s_max[0];
  for (int w = 1; w < RQ_PREP_NT / 32; w++) mn = fminf(mn, s_min[w]), mx = fmaxf(mx, s_max[w]);
  float vl = 0.f, delta = 0.f;
  if (qb > 0) {
    const float levels = (float)((1 << qb) - 1);
    if (centered) {
      vl = -mx;
      delta = __fdiv_rn(__fmul_rn(mx, 2.f), levels);
    } else {
      vl = mn;
      delta = __fdiv_rn(__fsub_rn(mx, mn), levels);
    }
    const float inv = delta > 0.f ? __fdiv_rn(1.f, delta) : 0.f;
    const int qmax = (1 << qb) - 1;
    int sq = 0;
    for (int w = warp; w < W; w += RQ_PREP_NT / 32) {
      const int j = w * 32 + lane;
      int qq = 0;
      if (j < d) {
        qq = (int)floorf(__fadd_rn(__fmul_rn(__fsub_rn(qr[j], vl), inv), 0.5f));
        qq = min(max(qq, 0), qmax);
      }
      sq += qq;
      for (int m = 0; m < qb; m++) {
        const uint32_t word = __ballot_sync(0xffffffffu, (qq >> m) & 1);
        if (lane == 0) planes[(pair * qb + m) * W + w] = word;
      }
    }
    sq = __reduce_add_sync(0xffffffffu, sq);
    if (lane == 0) atomicAdd(&s_sq, sq);
  }
  __syncthreads();
  if (tid == 0) {
    float qn = 0.f, qc = 0.f;
    for (int j = 0; j < d; j++) {
      qn = __fadd_rn(qn, __fmul_rn(qr[j], qr[j]));
      qc = __fadd_rn(qc, __fmul_rn(xr[j], cr[j]));
    }
    const float cB = __fmul_rn((float)((1 << nb_bits) - 1), 0.5f);
    cst[0] = vl;
    cst[1] = delta;
    cst[2] = __fmul_rn(cB, (float)s_sq);
    cst[3] = __fmul_rn(cB, (float)d);
    cst[4] = metric == kMetricL2 ? qn : qc;
    cst[5] = __fmul_rn(1.9f, __fsqrt_rn(qn));
    cst[6] = __int_as_float(s_sq);
    cst[7] = cB;
  }
}

// ---------------- the scan ------------------------------------------------------------------------
constexpr int RQ_NT = 256;
constexpr int RQ_NST = 2;
constexpr int RQ_MAX_PG = 32;

// word w (dimensions 32w .. 32w+31) of a bit-plane of P bytes; bytes past the plane read as 0
__device__ __forceinline__ uint32_t plane_word(const uint8_t* p, int w, int P, bool aligned) {
  if (aligned) return reinterpret_cast<const uint32_t*>(p)[w];
  uint32_t v = 0;
#pragma unroll
  for (int b = 0; b < 4; b++) {
    const int by = 4 * w + b;
    if (by < P) v |= (uint32_t)p[by] << (8 * b);
  }
  return v;
}
__device__ __forceinline__ float ld_f32(const uint8_t* p, bool aligned) {
  if (aligned) return *reinterpret_cast<const float*>(p);
  return __uint_as_float((uint32_t)p[0] | (uint32_t)p[1] << 8 | (uint32_t)p[2] << 16 | (uint32_t)p[3] << 24);
}

__host__ __device__ inline int rq_tile_entries(int cs) {
  int e = (48 * 1024) / cs;
  e = e / 16 * 16;
  if (e > 512) e = 512;
  if (e < 16) e = 16;  // cp.async.bulk sources stay 16-byte aligned: tile_e * cs is a multiple of 16
  return e;
}

size_t rq_scan_smem(int d, int nb_bits, int qb, int k) {
  const int cs = rabitq_code_size(d, nb_bits);
  const int tile_e = rq_tile_entries(cs);
  const int KP = next_pow2(k < 16 ? 16 : k);
  const int SORTN = next_pow2(KP + tile_e + tile_e / 2);
  const int W = (d + 31) / 32;
  return (size_t)RQ_NST * tile_e * cs + (size_t)SORTN * 8 + (size_t)qb * W * 4 + (qb == 0 ? (size_t)d * 4 : 0);
}

// One CTA per (query, group of pg probed lists); thread = entry; TMA 1-D bulk copies of the lists'
// code bytes through an RQ_NST-stage ring with a flat (list, tile) iterator, so the next list's
// tiles are in flight while the pair constants switch.  NB = nb_bits (0: runtime nb_rt).
template <int METRIC, int NB>
__global__ void __launch_bounds__(RQ_NT, 1)
    rabitq_scan_kernel(const float* __restrict__ consts, const uint32_t* __restrict__ planes,
                       const float* __restrict__ xq, int64_t ldq, const float* __restrict__ coarse, int64_t ldc, const int32_t* __restrict__ probe_ids, int nprobe,
                       int pg, ListDirectory dir, int d, int nb_rt, int qb, int cs, int tile_e, int k, int KP, int SORTN,
                       FilterArgs f, unsigned long long* __restrict__ partial) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const int B = NB > 0 ? NB : nb_rt;
  const int tile_bytes = tile_e * cs;
  const int P = (d + 7) >> 3, W = (d + 31) >> 5;
  unsigned char* stages = smem_raw;
  unsigned long long* buf = reinterpret_cast<unsigned long long*>(stages + (size_t)RQ_NST * tile_bytes);
  uint32_t* qp = reinterpret_cast<uint32_t*>(buf + SORTN);  // [qb][W] query planes of the current pair
  float* qrs = reinterpret_cast<float*>(qp + qb * W);       // [d] query residual x_q - c (qb == 0 only)
  __shared__ __align__(8) uint64_t full_bar[RQ_NST];
  __shared__ int s_cnt;
  __shared__ unsigned long long s_tau;
  __shared__ int g_list[RQ_MAX_PG], g_len[RQ_MAX_PG], g_tile0[RQ_MAX_PG + 1];

  const int tid = threadIdx.x;
  const int q = blockIdx.y, grp = blockIdx.x;
  unsigned long long* out = partial + ((int64_t)q * gridDim.x + grp) * k;
  const int p0 = grp * pg;
  const int np = min(pg, nprobe - p0);
  const bool aligned = (P & 3) == 0 && (cs & 3) == 0;

  if (tid == 0) {
    int acc = 0;
    for (int i = 0; i < np; i++) {
      const int l = probe_ids[(int64_t)q * nprobe + p0 + i];
      const int len = (l >= 0 && l < dir.nlist) ? dir.len[l] : 0;
      g_list[i] = l;
      g_len[i] = len;
      g_tile0[i] = acc;
      acc += (len + tile_e - 1) / tile_e;
    }
    g_tile0[np > 0 ? np : 0] = acc;
    for (int s = 0; s < RQ_NST; s++) mbar_init(&full_bar[s], 1);
    mbar_fence_init();
  }
  CandQueue cq{buf, &s_cnt, &s_tau, k, KP, SORTN};
  cq.init();
  const int total_tiles = np > 0 ? g_tile0[np] : 0;
  if (total_tiles == 0) {
    for (int i = tid; i < k; i += RQ_NT) out[i] = kKeySentinel;
    return;
  }

  int pr_pi = 0;
  auto issue = [&](int gt) {
    while (gt >= g_tile0[pr_pi + 1]) pr_pi++;
    const int ti = gt - g_tile0[pr_pi];
    const int n_e = min(tile_e, g_len[pr_pi] - ti * tile_e);
    const uint32_t bytes = ((uint32_t)n_e * cs + 15u) & ~15u;
    const int s = gt % RQ_NST;
    mbar_arrive_expect_tx(&full_bar[s], bytes);
    bulk_g2s(stages + (size_t)s * tile_bytes, dir.codes[g_list[pr_pi]] + (int64_t)ti * tile_e * cs, bytes, &full_bar[s]);
  };
  if (tid == 0)
    for (int gt = 0; gt < RQ_NST && gt < total_tiles; gt++) issue(gt);

  int pi = -1;
  float vl = 0.f, delta = 0.f, pc0 = 0.f, pc1 = 0.f, base = 0.f, cB = 0.f;
  const int64_t* __restrict__ lids = nullptr;
  const int per_thread = (tile_e + RQ_NT - 1) / RQ_NT;
  const int ex = B - 1;
  const int o_ex = P + 12;                      // first extra plane
  const int o_f = B == 1 ? P + 4 : o_ex + ex * P;  // the estimator's factor
  int est = 0;

  for (int gt = 0; gt < total_tiles; gt++) {
    int npi = pi < 0 ? 0 : pi;
    while (gt >= g_tile0[npi + 1]) npi++;
    if (npi != pi) {  // first tile of a new list: the pair's constants and query planes
      pi = npi;
      const int64_t pair = (int64_t)q * nprobe + p0 + pi;
      const float* c = consts + pair * kRabitqConsts;
      vl = c[0], delta = c[1], pc0 = c[2], pc1 = c[3], base = c[4], cB = c[7];
      lids = dir.ids[g_list[pi]];
      for (int i = tid; i < qb * W; i += RQ_NT) qp[i] = planes[pair * qb * W + i];
      if (qb == 0)
        for (int i = tid; i < d; i += RQ_NT)  // formed here as in the prep kernel: no residual staged in HBM
          qrs[i] = __fsub_rn(xq[(int64_t)q * ldq + i], coarse[(int64_t)g_list[pi] * ldc + i]);
      __syncthreads();
    }
    const int ti = gt - g_tile0[pi];
    const int n_e = min(tile_e, g_len[pi] - ti * tile_e);
    const int s = gt % RQ_NST;
    mbar_wait(&full_bar[s], (gt / RQ_NST) & 1);
    const unsigned long long tau = s_tau;
    const float tb = key_bound<METRIC>(tau);
    const float lo_b = METRIC == kMetricL2 ? f.min_score : fmaxf(tb, f.min_score);
    const float hi_b = METRIC == kMetricL2 ? fminf(tb, f.max_score) : f.max_score;
    const unsigned char* st = stages + (size_t)s * tile_bytes;
    int pushed = 0;
    for (int u = 0; u < per_thread; u++) {
      const int e = u * RQ_NT + tid;
      float dis = 0.f;
      if (e < n_e) {
        const uint8_t* ce = st + (size_t)e * cs;
        float g;
        if (qb > 0) {
          uint32_t sqt = 0, stot = 0;
          for (int w = 0; w < W; w++) {
#pragma unroll
            for (int kk = 0; kk < (NB > 0 ? NB : 9); kk++) {
              if (NB == 0 && kk >= B) break;
              const uint32_t tw = plane_word(ce + (kk == B - 1 ? 0 : o_ex + kk * P), w, P, aligned);
              stot += (uint32_t)__popc(tw) << kk;
#pragma unroll 1
              for (int m = 0; m < qb; m++) sqt += (uint32_t)__popc(tw & qp[m * W + w]) << (kk + m);
            }
          }
          const float e1 = __fsub_rn(__uint2float_rn(sqt), pc0);
          const float e2 = __fsub_rn(__uint2float_rn(stot), pc1);
          g = __fadd_rn(__fmul_rn(delta, e1), __fmul_rn(vl, e2));
        } else {  // float query: sum_j qr_j (t_j - cB), j ascending
          g = 0.f;
          for (int j = 0; j < d; j++) {
            const int by = j >> 3, bit = j & 7;
            uint32_t t = 0;
            for (int kk = 0; kk < B; kk++) t |= (uint32_t)((ce[(kk == B - 1 ? 0 : o_ex + kk * P) + by] >> bit) & 1) << kk;
            g = __fadd_rn(g, __fmul_rn(qrs[j], __fsub_rn((float)t, cB)));
          }
        }
        const float ip = __fmul_rn(ld_f32(ce + o_f, aligned), g);
        const float s0 = __fadd_rn(base, ld_f32(ce + P, aligned));
        dis = METRIC == kMetricL2 ? __fsub_rn(s0, __fmul_rn(2.f, ip)) : __fadd_rn(s0, ip);
      }
      bool pred = e < n_e && dis <= hi_b && dis >= lo_b;
      unsigned long long key = kKeySentinel;
      if (pred) {
        const int64_t raw = lids[(int64_t)ti * tile_e + e];
        pred = raw >= 0;  // tombstone
        const uint32_t vid = (uint32_t)raw;
        if (pred) pred = ctx_is_valid(f.del_bits, f.filter_bits, vid);
        key = make_key(score2ord<METRIC>(dis), vid);
        pred = pred && key < tau;
      }
      cq.push_warp(pred, key);
      pushed |= pred ? 1 : 0;
    }
    est += __syncthreads_count(pushed) * per_thread;
    if (tid == 0 && gt + RQ_NST < total_tiles) issue(gt + RQ_NST);
    if (gt + 1 < total_tiles && est + tile_e > cq.cap()) {
      cq.flush();
      est = 0;
    }
  }
  __syncthreads();
  cq.flush(true);
  for (int i = tid; i < k; i += RQ_NT) out[i] = buf[i];
}

template <int METRIC, int NB>
cudaError_t launch_rq_scan_t(const float* consts, const uint32_t* planes, const float* xq, int64_t ldq, const float* coarse, int64_t ldc, int nq,
                             const int32_t* probe_ids, int nprobe, int pg, ListDirectory dir, int d, int nb_bits, int qb,
                             int k, FilterArgs f, unsigned long long* partial, cudaStream_t st) {
  const int cs = rabitq_code_size(d, nb_bits);
  const int tile_e = rq_tile_entries(cs);
  const int KP = next_pow2(k < 16 ? 16 : k);
  const int SORTN = next_pow2(KP + tile_e + tile_e / 2);
  const size_t smem = rq_scan_smem(d, nb_bits, qb, k);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  cudaError_t e = cudaFuncSetAttribute(rabitq_scan_kernel<METRIC, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  dim3 grid((nprobe + pg - 1) / pg, nq);
  rabitq_scan_kernel<METRIC, NB><<<grid, RQ_NT, smem, st>>>(consts, planes, xq, ldq, coarse, ldc, probe_ids, nprobe, pg, dir, d, nb_bits,
                                                           qb, cs, tile_e, k, KP, SORTN, f, partial);
  note_launch();
  return cudaGetLastError();
}

template <int METRIC>
cudaError_t launch_rq_scan_m(const float* consts, const uint32_t* planes, const float* xq, int64_t ldq, const float* coarse, int64_t ldc, int nq,
                             const int32_t* probe_ids, int nprobe, int pg, ListDirectory dir, int d, int nb_bits, int qb,
                             int k, FilterArgs f, unsigned long long* partial, cudaStream_t st) {
#define GB_RQ(NB) \
  return launch_rq_scan_t<METRIC, NB>(consts, planes, xq, ldq, coarse, ldc, nq, probe_ids, nprobe, pg, dir, d, nb_bits, qb, k, f, partial, st)
  switch (nb_bits) {
    case 1: GB_RQ(1);
    case 2: GB_RQ(2);
    case 4: GB_RQ(4);
    case 9: GB_RQ(9);
    default: GB_RQ(0);
  }
#undef GB_RQ
}

}  // namespace

bool rabitq_scan_supported(int d, int nb_bits) {
  return rq_scan_smem(d, nb_bits, 8, 16) <= 227 * 1024 && rq_scan_smem(d, nb_bits, 0, 16) <= 227 * 1024;
}

cudaError_t launch_rabitq_encode(const float* x, int64_t ldx, int64_t n, int d, const float* coarse, int64_t ldc,
                                 const int32_t* assign, int nb_bits, int metric, uint8_t* codes, cudaStream_t st) {
  if (n <= 0) return cudaSuccess;
  if (nb_bits < 1 || nb_bits > 9 || d <= 0) return cudaErrorInvalidValue;
  rabitq_encode_kernel<<<(unsigned)((n + RQ_ENC_NT - 1) / RQ_ENC_NT), RQ_ENC_NT, 0, st>>>(
      x, ldx, n, d, coarse, ldc, assign, nb_bits, metric, codes, rabitq_code_size(d, nb_bits));
  note_launch();
  return cudaGetLastError();
}

cudaError_t launch_rabitq_query_prep(const float* xq, int64_t ldq, int nq, int d, const int32_t* probe_ids, int nprobe,
                                     const float* coarse, int64_t ldc, int nlist, int qb, bool centered, int nb_bits,
                                     int metric, float* consts, uint32_t* planes, cudaStream_t st) {
  if (nq <= 0 || nprobe <= 0) return cudaSuccess;
  if (qb < 0 || qb > 8 || nb_bits < 1 || nb_bits > 9) return cudaErrorInvalidValue;
  const size_t smem = (size_t)d * 4;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(rabitq_query_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  rabitq_query_prep_kernel<<<(unsigned)((int64_t)nq * nprobe), RQ_PREP_NT, smem, st>>>(
      xq, ldq, nprobe, probe_ids, coarse, ldc, nlist, d, qb, centered ? 1 : 0, nb_bits, metric, consts, planes);
  note_launch();
  return cudaGetLastError();
}

cudaError_t launch_rabitq_scan(const float* consts, const uint32_t* planes, const float* xq, int64_t ldq, const float* coarse, int64_t ldc, int nq,
                               const int32_t* probe_ids, int nprobe, int pg, ListDirectory dir, int d, int nb_bits, int qb,
                               int k, int metric, FilterArgs f, unsigned long long* partial, cudaStream_t st) {
  if (nq <= 0 || nprobe <= 0) return cudaSuccess;
  if (k <= 0 || k > 4096 || nq > 65535 || pg < 1 || pg > RQ_MAX_PG || qb < 0 || qb > 8 || nb_bits < 1 || nb_bits > 9 ||
      d > 8192)
    return cudaErrorInvalidValue;
  if (metric == kMetricL2)
    return launch_rq_scan_m<kMetricL2>(consts, planes, xq, ldq, coarse, ldc, nq, probe_ids, nprobe, pg, dir, d, nb_bits, qb, k, f, partial, st);
  return launch_rq_scan_m<kMetricIP>(consts, planes, xq, ldq, coarse, ldc, nq, probe_ids, nprobe, pg, dir, d, nb_bits, qb, k, f, partial, st);
}

}  // namespace gb
