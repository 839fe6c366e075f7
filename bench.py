#!/usr/bin/env python
"""bench.py -- queries/s of the gamma vector-search hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload NAME] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of nq synthetic queries: coarse quantiser,
inverted-list scan (IVF-Flat) or LUT + ADC scan (+ exact re-rank) (IVF-PQ), top-k merge.
Default workload = the configuration the metric is quoted on: IVF-PQ d=128 M=16 nbits=8
nlist=4096 N=10M nq=10k (BASELINE.json configs[2]); other configs via --workload.

  value     GLOBAL queries/s on the database the metric string names (N = all partitions together),
            queries and results resident in HBM (CUDA events, max over ranks)
  e2e       the same through the public call with HOST buffers: pinned-host queries -> H2D ->
            search -> [NCCL all-gather of result keys + merge] -> D2H results, every step
  roofline  dominant scan kernel alone (CUDA events around that launch on the launching stream)
  stages    device time per stage of a step (coarse quantiser, tables, scan phases, re-rank, merge)
  cpu_baseline / --impl reference
            baseline/cpu_gamma.c (gamma's CPU path restated for speed: FMA / AVX-512, blocked sgemm)
            on this box's host cores, same index state, bounded query sample, median of 3

Multi-GPU (N > 1), one Vearch partition per rank/GPU; every query goes to every partition; the per-rank
result keys are all-gathered over NCCL (one collective) and merged on device in the router's order
(internal/client/client.go:1530-1609).
  --scaling weak   (default) a fixed partition per GPU (10M vectors each); the database grows with N, ideal = constant
                   global queries/s.  `partition_queries_per_s` (= value x N) and `scan_entries_per_s` are the
                   aggregate-work figures.
  --scaling strong a fixed database (--n-total, default the workload's N) split over the ranks.
The default run also carries, under `secondary`, BASELINE configs[4] measured the strong way at the same N: the 100M-vector
IVF-PQ database split over the N ranks (N=1 holds it all, N=8 holds 12.5M per GPU), plus C1/C2/C4 at N=1.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "flat_100k": dict(type="FLAT", d=128, n=100_000, nlist=0, nprobe=0, M=0, metric="L2", data="sift", nq=1000,
                      desc="FLAT brute-force L2 d=128 N=100k nq=1k (BASELINE configs[0])"),
    "ivfflat_1m": dict(type="IVFFLAT", d=128, n=1_000_000, nlist=1024, nprobe=32, M=0, metric="L2", data="sift",
                       nq=10_000, desc="IVF-Flat d=128 nlist=1024 nprobe=32 N=1M (BASELINE configs[1])"),
    "ivfpq_10m": dict(type="IVFPQ", d=128, n=10_000_000, nlist=4096, nprobe=32, M=16, metric="L2", data="sift",
                      nq=10_000, desc="IVF-PQ d=128 m=16 nbits=8 nlist=4096 N=10M (BASELINE configs[2])"),
    "ivfflat_768": dict(type="IVFFLAT", d=768, n=10_000_000, nlist=4096, nprobe=32, M=0, metric="InnerProduct",
                        data="embed", nq=10_000,
                        desc="IVF-Flat d=768 cosine nlist=4096 N=10M nq=10k (BASELINE configs[3])"),
    "ivfpq_100m": dict(type="IVFPQ", d=128, n=100_000_000, nlist=4096, nprobe=32, M=16, metric="L2", data="sift",
                       nq=10_000, scaling="strong",
                       desc="IVF-PQ d=128 N=100M split over the ranks' partitions (BASELINE configs[4])"),
}
CONFIGS4_TOTAL = 100_000_000  # BASELINE configs[4]: 100M vectors over the ranks' partitions (12.5M per GPU at N=8)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ivfpq_10m", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="", choices=["", "weak", "strong"])
    ap.add_argument("--n", type=int, default=0, help="override vectors per GPU (parity/dev runs)")
    ap.add_argument("--n-total", type=int, default=0, help="--scaling strong: vectors in the whole database")
    ap.add_argument("--nq", type=int, default=0)
    ap.add_argument("--nprobe", type=int, default=0)
    ap.add_argument("--recall-num", type=int, default=-1, help="IVF-PQ exact re-rank depth (0 = off)")
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--dataset", default="", choices=["", "sift", "hard", "embed"],
                    help="hard: overlapping clusters on a low-dimensional manifold, Zipf cluster weights")
    ap.add_argument("--auto-nprobe", action="store_true", help="smallest nprobe of the sweep with recall@10 >= 0.95")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the quick C1/C2/C4 lines of the default run")
    ap.add_argument("--profile", action="store_true",
                    help="cudaProfilerStart/Stop around the timed device steps (ncu --profile-from-start off)")
    ap.add_argument("--sweep", default="", help="nprobe:recall_num,... -> recall/QPS table on stderr, then exit")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the result of the last timed step as DIR/scores.npy (float32) and DIR/ids.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the result of this engine's timed step; --impl reference has none")
    return args


DUMP_LIMIT = 64_000_000  # bytes of .npy files --dump-outputs may write


def dump_outputs(out_dir, scores, ids):
    """Scores as float32, ids as float64 (exact: ids stay below 2^53).  A batch too large for DUMP_LIMIT is cut to a
    fixed, seeded sample of its queries; their row numbers in the batch go to query_rows.npy."""
    os.makedirs(out_dir, exist_ok=True)
    nq, k = scores.shape
    row_bytes = k * (4 + 8) + 8
    if nq * row_bytes > DUMP_LIMIT - 4096:  # 4 KiB: room for the .npy headers
        rows = np.sort(np.random.default_rng(0).choice(nq, (DUMP_LIMIT - 4096) // row_bytes, replace=False))
        scores, ids = scores[rows], ids[rows]
        np.save(os.path.join(out_dir, "query_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "scores.npy"), scores.astype(np.float32))
    np.save(os.path.join(out_dir, "ids.npy"), ids.astype(np.float64))


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, uuid):
        self.uuid = uuid
        self.proc = None
        self.lines = []
        self.first = 0

    def mark(self):
        self.first = len(self.lines)

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", self.uuid, f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)  # let the sample that covers the end of the window arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines[self.first:]:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0]))
                mx.append(float(p[1]))
            except ValueError:
                continue
            for nme, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(np.max(mx)) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def measured_peak(kind="hbm"):
    """HBM GB/s, or dense bf16 TFLOP/s (the sustained figure: the kernel is timed inside a step)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            if kind == "hbm":
                return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
            return float(j["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
        except Exception:
            pass
    if kind == "hbm":
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"
    return 1400.0, "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)"


def ncu_counters(workload, kernel):
    """Counters of `kernel` on `workload` from the committed ncu --set full capture (profiles/r2_ncu.json), or {}."""
    for name in ("r2_ncu.json", "r1_traffic.json"):
        try:
            j = json.load(open(os.path.join(ROOT, "profiles", name))).get(workload, {}).get(kernel)
        except Exception:
            j = None
        if j is not None:
            return j if isinstance(j, dict) else {"dram_bytes": j}
    return {}


def recall_stats(ids, gt):
    """(reference definition: true 1-NN in the first 10; standard 10-recall@10)"""
    k = min(10, ids.shape[1])
    r1 = float(np.mean([(gt[q, 0] in ids[q, :k]) for q in range(ids.shape[0])]))
    rk = float(np.mean([len(set(ids[q, :k]) & set(gt[q, :k])) / k for q in range(ids.shape[0])]))
    return r1, rk


# ------------------------------------------------------------------------------------------------
def generator(family):
    from vearch_b200 import synth
    return {"sift": synth.sift_like_torch, "hard": synth.sift_hard_torch, "embed": synth.embed_like_torch}[family]


def build_index(wl, n, rank, device, family):
    import torch
    from vearch_b200 import index as gidx
    d = wl["d"]
    params = {"metric_type": wl["metric"]}
    if wl["type"] != "FLAT":
        params.update(ncentroids=wl["nlist"], nprobe=min(wl["nprobe"], wl["nlist"]))
        if n < wl["nlist"] * 39:  # dev-size runs
            params["ncentroids"] = max(16, n // 100)
            params["nprobe"] = min(params["nprobe"], params["ncentroids"])
        params["training_threshold"] = min(n, params["ncentroids"] * 200)
    if wl["type"] == "IVFPQ":
        params.update(nsubvector=wl["M"], nbits_per_idx=8)
    idx = gidx.GammaIndex(wl["type"], d, params, device=device)
    t0 = time.time()
    gen = generator(family)
    chunk = 1 << 20
    for s in range(0, n, chunk):
        e = min(n, s + chunk)
        x = gen(e - s, d, seed=1234 + 1000 * rank + (s >> 20), device=f"cuda:{device}")
        idx.add_vectors(x)
        del x
    torch.cuda.synchronize()
    t1 = time.time()
    idx.train()
    t2 = time.time()
    idx.add_pending()
    t3 = time.time()
    build = {"gen_add_s": round(t1 - t0, 2), "train_s": round(t2 - t1, 2), "index_s": round(t3 - t2, 2)}
    return idx, params, build


def scan_work(idx, wl, xq_host, nprobe):
    """entries the probes of this batch scan, (query, list) pairs, list-length statistics"""
    if wl["type"] == "FLAT":
        return {"entries": float(xq_host.shape[0]) * idx.ntotal}
    lens = np.array([idx.list_len(l) for l in range(idx.nlist)], np.int64)
    _, keys = idx.coarse_search(xq_host, nprobe)
    valid = keys >= 0
    out = {"entries": float(lens[keys[valid]].sum()), "query_list_pairs": float(valid.sum()),
           "list_len_mean": float(lens.mean()), "list_len_cv": float(lens.std() / max(lens.mean(), 1e-9)),
           "probed_list_len_mean": float(lens[keys[valid]].mean()) if valid.any() else 0.0}
    out["_lens"], out["_keys"] = lens, keys
    return out


def algorithmic_bytes(wl, work, nq, k, recall_num, scan_only=True):
    """SURVEY.md 8(d) bytes of the SCAN kernel: per scanned entry (4d+8) B for IVF-Flat, (M+8) B for IVF-PQ plus the
    precomputed-table row M*256*4 B per (query, list); FLAT: N*4d per query.  (The re-rank gathers, recall_num*4d per
    query, belong to rerank_kernel and are reported separately.)"""
    d = wl["d"]
    if wl["type"] == "FLAT":
        return work["entries"] * 4 * d
    if wl["type"] == "IVFFLAT":
        return work["entries"] * (4 * d + 8)
    b = work["entries"] * (wl["M"] + 8)
    if wl["metric"] == "L2":
        b += work["query_list_pairs"] * wl["M"] * 256 * 4
    if not scan_only and recall_num > 0:
        b += nq * max(k, recall_num) * 4 * d
    return b


def make_roofline(idx, wl, wl_name, work, nq, k, recall_num, scan_ms, ms_per_step, default_shape):
    kname = idx.last_scan_kernel
    info = idx.last_scan_info
    abytes = algorithmic_bytes(wl, work, nq, k, recall_num)
    hbm_peak, hbm_src = measured_peak("hbm")
    tc_peak, tc_src = measured_peak("tensor")
    ncu = ncu_counters(wl_name if default_shape else "", kname)
    traffic = ncu.get("dram_bytes")
    sec = scan_ms / 1000 if scan_ms > 0 else None
    hbm_alg = abytes / sec / 1e9 if sec else None
    r = {"kernel": kname, "kernel_ms": scan_ms, "kernel_share_of_step": scan_ms / ms_per_step if ms_per_step else None,
         "traffic": traffic, "algorithmic_bytes_per_launch": abytes}
    r.update({kk: v for kk, v in work.items() if not kk.startswith("_")})
    secondary = {"hbm_algorithmic": {"achieved_gbs": hbm_alg, "peak_gbs": hbm_peak, "frac": hbm_alg / hbm_peak if hbm_alg else None,
                                     "note": "SURVEY 8(d) bytes (every query streams its own entries) / kernel time"}}
    if traffic and sec:
        secondary["dram"] = {"achieved_gbs": traffic / sec / 1e9, "frac": traffic / sec / 1e9 / hbm_peak,
                             "note": "ncu dram__bytes_read+write of the committed capture / live kernel time"}
    for key in ("issue_active_pct", "lsu_pipe_pct", "tensor_pipe_pct", "inst_per_entry", "lds_bank_conflict_pct",
                "l2_hit_pct", "warps_active_pct"):
        if key in ncu:
            secondary[key] = ncu[key]
    if kname == "pqtc_scan_kernel":
        # entries the tensor-core filter multiplies: the probes behind each query's phase A (index.cu scan_listmajor_pq:
        # phase A = the fewest leading probes, in full, whose lists hold >= target entries, at most pa_max)
        pa_max, target = int(info.get("phase_a_max_probes", 1)), int(info.get("phase_a_target_entries", -1))
        keys, lens = work["_keys"], work["_lens"]
        ll = np.where(keys >= 0, lens[np.maximum(keys, 0)], 0)
        if target > 0:
            reached = np.cumsum(ll[:, :pa_max], axis=1) >= target
            pa_q = np.where(reached.any(axis=1), reached.argmax(axis=1) + 1, pa_max)
        else:
            pa_q = np.full(keys.shape[0], pa_max)
        in_b = np.arange(keys.shape[1])[None, :] >= pa_q[:, None]
        ent_tc = float(ll[in_b].sum())
        info = dict(info, phase_a_probes_mean=float(pa_q.mean()), phase_a_entries_scanned=float(ll[~in_b].sum()))
        aflops = ent_tc * 2.0 * wl["d"]
        ach = aflops / sec / 1e12 if sec else None
        r.update({"bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach / tc_peak if ach else None,
                  "peak_source": tc_src, "algorithmic_flops_per_launch": aflops, "mma_kind": "kind::f16 (fp16 operands, power-of-two scaled; fp32 accumulate)",
                  "filter": info, "entries_filtered_on_tensor_cores": ent_tc,
                  "note": "list-major ADC: 2*d flop per (query, entry) pair of the probes behind each query's phase A; the codes are read once per "
                          "128 (query, list) pairs and decoded in shared memory, so neither HBM nor the 8(d) byte count binds it"})
    elif kname.startswith("ivf_listmajor"):
        aflops = work["entries"] * 2.0 * wl["d"]
        ach = aflops / sec / 1e12 if sec else None
        r.update({"bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach / tc_peak if ach else None,
                  "peak_source": tc_src, "algorithmic_flops_per_launch": aflops,
                  "mma_kind": "kind::tf32 x3 (error-compensated split: three MMAs per product, tf32 peak is half the bf16 figure)"})
    elif wl["type"] == "FLAT":
        import torch
        prop = torch.cuda.get_device_properties(torch.cuda.current_device())
        fma_peak = prop.multi_processor_count * 128 * 2 * 1.965e9 / 1e12  # fp32 lanes x 2 flop x max SM clock
        aflops = work["entries"] * (3.0 if wl["metric"] == "L2" else 2.0) * wl["d"]
        ach = aflops / sec / 1e12 if sec else None
        r.update({"bound": "fma", "achieved": ach, "peak": fma_peak, "unit": "TFLOP/s", "frac": ach / fma_peak if ach else None,
                  "peak_source": "SMs x 128 fp32 lanes x 2 x 1.965 GHz (CUDA-core FMA issue, not a tensor-pipe kernel)",
                  "algorithmic_flops_per_launch": aflops})
    else:
        r.update({"bound": "hbm", "achieved": hbm_alg, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_alg / hbm_peak if hbm_alg else None,
                  "peak_source": hbm_src})
        if hbm_alg and hbm_alg > hbm_peak:
            r["note"] = ("algorithmic bytes follow SURVEY 8(d) (every query streams its own entries); the kernel serves them from "
                         "L2, so HBM is not its bound: see secondary")
    r["secondary"] = secondary
    return r


def export_state(idx, wl):
    st = {}
    if wl["type"] == "FLAT":
        return st
    st["cent"] = idx.get_centroids()
    st["off"], st["codes"], st["ids"] = idx.export_lists()
    if wl["type"] == "IVFPQ":
        st["pq"] = idx.get_pq_centroids()
        st["T"] = idx.get_precomputed_table() if wl["metric"] == "L2" else None
    return st


def cpu_search(cg, wl, st, raw, xq, k, nprobe, recall_num):
    """gamma's CPU search path (baseline/cpu_gamma.c), one call = coarse + scan (+ re-rank)."""
    metric = cg.METRIC_L2 if wl["metric"] == "L2" else cg.METRIC_IP
    if wl["type"] == "FLAT":
        return cg.flat_search(raw, xq, k, metric)
    cd, keys = cg.coarse_search(st["cent"], xq, nprobe, metric)
    if wl["type"] == "IVFFLAT":
        vecs = st["codes"].view(np.float32).reshape(len(st["ids"]), -1)
        return cg.ivfflat_search_preassigned(st["off"], vecs, st["ids"], xq, k, keys, metric)
    return cg.ivfpq_search_preassigned(st["off"], st["codes"], st["ids"], st["cent"], st["pq"], st["T"], xq, k, keys, cd,
                                       metric, recall_num=max(recall_num, 0), raw=raw)


def time_cpu(idx, wl, xq_host, k, nprobe, recall_num, budget_s, reps=3):
    """median-of-reps CPU queries/s on a bounded sample of the batch; returns (qps, cores, sample text, ids)"""
    from baseline import cpu_gamma as cg
    cores = cg.set_threads()  # every core the cgroup grants, whatever OMP_NUM_THREADS says
    st = export_state(idx, wl)
    raw = idx.get_vectors(0, idx.ntotal) if (wl["type"] == "FLAT" or recall_num > 0) else None
    nq = xq_host.shape[0]
    t0 = time.time()
    cpu_search(cg, wl, st, raw, xq_host[:64], k, nprobe, recall_num)  # also warms the thread pool
    t0 = time.time()
    cpu_search(cg, wl, st, raw, xq_host[:64], k, nprobe, recall_num)
    per_q = (time.time() - t0) / 64
    nsamp = int(max(64, min(nq, budget_s / reps / max(per_q, 1e-7))))
    times, ids = [], None
    for _ in range(reps):
        t0 = time.time()
        _, ids = cpu_search(cg, wl, st, raw, xq_host[:nsamp], k, nprobe, recall_num)
        times.append(time.time() - t0)
    dt = float(np.median(times))
    text = (f"{nsamp} of {nq} queries per rep, median of {reps} reps ({', '.join('%.2f' % t for t in times)} s), "
            f"{cores} threads ({cg.isa()}), same index state (built on the GPU, exported)")
    return nsamp / dt, cores, text, ids, nsamp


# ------------------------------------------------------------------------------------------------
def measure(args, wl_name, wl, n_rank, rank, world, local, use_dist, family, steps, warmup, primary):
    """Build this rank's partition, time the device-resident and the end-to-end step; returns a dict (all ranks)."""
    import torch
    import torch.distributed as dist
    from vearch_b200 import _lib, index as gidx

    dev = f"cuda:{local}"
    nq = args.nq or wl["nq"]
    k = args.k
    nprobe = args.nprobe or wl["nprobe"]
    recall_num = args.recall_num if args.recall_num >= 0 else (400 if wl["type"] == "IVFPQ" else 0)
    sampler = None
    if primary:  # nvidia-smi needs a second or two before its first sample: started ahead of the index build
        uuid = str(torch.cuda.get_device_properties(local).uuid)
        uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        sampler = ClockSampler(uuid)
        sampler.start()
    idx, params, build = build_index(wl, n_rank, rank, local, family)
    if wl["type"] != "FLAT":
        nprobe = min(nprobe, params["ncentroids"])
    metric_id = gidx.METRIC_L2 if wl["metric"] == "L2" else gidx.METRIC_IP

    gen = generator(family)
    nbatches = warmup + steps
    # a distinct query batch per step (same on every rank), held in pinned host memory for e2e
    q_host = [torch.empty((nq, wl["d"]), dtype=torch.float32).pin_memory() for _ in range(nbatches)]
    q_dev = []
    for b in range(nbatches):
        x = gen(nq, wl["d"], seed=4321 + b, device=dev)
        q_dev.append(x)
        q_host[b].copy_(x)
    torch.cuda.synchronize()

    def sparams(npb, rn):
        p = {}
        if wl["type"] != "FLAT":
            p["nprobe"] = npb
        if wl["type"] == "IVFPQ" and rn > 0:
            p["recall_num"] = rn
        return p or None

    # ---- recall of this configuration against exact ground truth (untimed) --------------------
    ns = min(1000, nq)
    xs = q_host[0][:ns].numpy()
    _, gt_i = idx.search(xs, 10, brute_force=True)
    sweep = None
    if args.auto_nprobe and wl["type"] != "FLAT":
        sweep = []
        for npb in (1, 2, 4, 8, 16, 32, 64, 128):
            if npb > params["ncentroids"]:
                break
            _, ri_ = idx.search(xs, 10, params=sparams(npb, recall_num))
            a1, a10 = recall_stats(ri_, gt_i)
            sweep.append({"nprobe": npb, "recall@10_1nn": a1, "recall@10": a10})
            if a10 >= 0.95:
                break
        nprobe = sweep[-1]["nprobe"]
    if args.sweep:
        for item in args.sweep.split(","):
            npb, rn = (int(v) for v in item.split(":"))
            _, ri_ = idx.search(xs, 10, params=sparams(npb, rn))
            a1, a10 = recall_stats(ri_, gt_i)
            idx.search_device(q_dev[0], k, params=sparams(npb, rn))
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for b in range(1, min(4, nbatches)):
                idx.search_device(q_dev[b], k, params=sparams(npb, rn))
            torch.cuda.synchronize()
            qps = nq * (min(4, nbatches) - 1) / (time.perf_counter() - t0)
            print(json.dumps({"sweep": {"nprobe": npb, "recall_num": rn, "recall_1nn_top10": a1, "recall10": a10,
                                        "qps_device": qps}}), file=sys.stderr, flush=True)
        idx.close()
        return None
    sp = sparams(nprobe, recall_num)
    _, ri = idx.search(xs, 10, params=sp)
    r1, r10 = recall_stats(ri, gt_i)

    out_d = torch.empty((nq, k), dtype=torch.float32, device=dev)
    out_i = torch.empty((nq, k), dtype=torch.int64, device=dev)
    keys_buf = torch.empty((nq, k), dtype=torch.int64, device=dev)
    gather_keys = torch.empty((world, nq, k), dtype=torch.int64, device=dev) if use_dist else None
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    coll_events = []

    def search_and_merge(xq, timed):
        if not use_dist:
            idx.search_device(xq, k, params=sp, out=(out_d, out_i))
            return out_d, out_i
        idx.search_device_keys(xq, k, params=sp, out_keys=keys_buf)
        if timed:
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
        dist.all_gather_into_tensor(gather_keys, keys_buf)  # one collective: 8 B per (query, result)
        res = gidx.merge_partition_keys_device(gather_keys, metric_id)
        if timed:
            c1.record()
            coll_events.append((c0, c1))
        return res

    def step_device(b, timed=False):
        return search_and_merge(q_dev[b], timed)

    def step_e2e(b):
        xq = q_host[b].to(dev, non_blocking=True)  # H2D from pinned memory
        rd_, ri_ = search_and_merge(xq, False)
        return rd_.cpu(), ri_.cpu()  # D2H of the step's result

    def sync_all():
        torch.cuda.synchronize()
        if use_dist:
            dist.barrier()
            torch.cuda.synchronize()

    if sampler:
        sampler.mark()  # samples from here on: warm-up + both timed regions

    # ---- device-resident timing ----------------------------------------------------------------
    for b in range(warmup):
        step_device(b)
    sync_all()
    idx.set_scan_timing(True)
    _ = idx.last_scan_ms
    idx.stage_times()
    launches0 = _lib.lib().gb_launch_count()
    step_ms, scan_ms = [], []
    if args.profile and primary:
        torch.cuda.profiler.start()
    for s in range(steps):
        b = warmup + s
        flush.fill_(s)  # L2 flush between timed iterations (untimed)
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = step_device(b, timed=True)
        e1.record()
        sync_all()
        step_ms.append(e0.elapsed_time(e1))
        scan_ms.append(idx.last_scan_ms)
    if args.profile and primary:
        torch.cuda.profiler.stop()
    # copied before the end-to-end loop below reuses the result buffers
    outputs = (last[0].cpu().numpy(), last[1].cpu().numpy()) if args.dump_outputs and primary and rank == 0 else None
    launches = (_lib.lib().gb_launch_count() - launches0) / max(1, steps)
    stages = {kk: v / steps for kk, v in idx.stage_times().items()}
    idx.set_scan_timing(False)
    coll_ms = float(np.mean([a.elapsed_time(b_) for a, b_ in coll_events])) if coll_events else 0.0
    if use_dist:
        stages["allgather_keys_and_merge"] = coll_ms
    my = torch.tensor([float(np.sum(step_ms)), float(np.mean(scan_ms)), coll_ms, float(idx.ntotal)], device=dev, dtype=torch.float64)
    if use_dist:
        allr = torch.empty((world, 4), device=dev, dtype=torch.float64)
        dist.all_gather_into_tensor(allr, my)
        allr = allr.cpu().numpy()
    else:
        allr = my.cpu().numpy()[None, :]
    total_ms = float(allr[:, 0].max())  # max over ranks
    ms_per_step = total_ms / steps
    n_total = int(allr[:, 3].sum())

    # ---- end-to-end timing (host buffers, copies inside the timed region) ---------------------
    for b in range(warmup):
        step_e2e(b)
    sync_all()
    e2e_ms = []
    for s in range(steps):
        b = warmup + s
        flush.fill_(s)
        sync_all()
        t0 = time.perf_counter()
        step_e2e(b)
        torch.cuda.synchronize()
        e2e_ms.append((time.perf_counter() - t0) * 1000)
    e2e_total = float(np.sum(e2e_ms))
    if use_dist:
        t = torch.tensor([e2e_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_total = float(t.item())
    e2e_qps = nq / (e2e_total / steps / 1000)
    clocks = None
    if sampler:
        clocks = sampler.stop()
        clocks["window"] = "warm-up + timed device steps + timed end-to-end steps"

    # C-ABI host call (gb_index_search: host in, host out) for N=1: the reference-facing entry point
    cabi_qps = None
    if world == 1:
        for b in range(warmup):
            idx.search(q_host[b].numpy(), k, params=sp)
        cabi_s = 0.0
        for s in range(steps):
            flush.fill_(s)  # same L2 flush + full sync between timed calls as the device-resident loop
            torch.cuda.synchronize()
            xh = q_host[warmup + s].numpy()
            t0 = time.perf_counter()
            idx.search(xh, k, params=sp)  # returns after the D2H of the results
            cabi_s += time.perf_counter() - t0
        cabi_qps = nq * steps / cabi_s

    xq_host = q_host[warmup].numpy()
    work = scan_work(idx, wl, xq_host, nprobe)
    ent = torch.tensor([work["entries"]], device=dev, dtype=torch.float64)
    if use_dist:
        dist.all_reduce(ent)
    res = dict(idx=idx, wl=wl, wl_name=wl_name, params=params, build=build, nq=nq, k=k, nprobe=nprobe, recall_num=recall_num,
               sp=sp, r1=r1, r10=r10, sweep=sweep, ms_per_step=ms_per_step, scan_avg=float(np.mean(scan_ms)), launches=launches,
               stages=stages, per_rank=allr, n_total=n_total, e2e_qps=e2e_qps, cabi_qps=cabi_qps, clocks=clocks, work=work,
               entries_all_ranks=float(ent.item()), xq_host=xq_host, family=family, outputs=outputs)
    return res


def config_dict(wl, family, n_rank, n_total, world, nq, k, nprobe, recall_num, params, scaling):
    """identical in the `ours` and the `reference` arm (the driver compares the two config dicts)"""
    return {"workload": wl["desc"], "index": wl["type"], "d": wl["d"], "dataset": family, "n_per_gpu": n_rank, "n_total": n_total,
            "partitions": world, "nq_per_step": nq, "k": k, "nprobe": nprobe, "recall_num": recall_num, "index_params": params,
            "scaling_mode": scaling,
            "l2": "512 MiB write between timed steps + distinct query batch per step"}


def metric_string(wl, n_total, nq):
    return "queries/sec @ recall@10 (d=%d, N=%d, nq=%d)" % (wl["d"], n_total, nq)


def main():
    args = parse_args()
    wl_name = args.workload
    wl = WORKLOADS[wl_name]
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        args.gpus = world
    reference = args.impl == "reference"
    if reference and rank != 0:
        return 0  # the CPU arm runs on rank 0 alone

    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this engine has no CPU path")
    torch.cuda.set_device(local)
    dev = f"cuda:{local}"
    nparts = args.gpus  # partitions of the database = GPUs of the `ours` arm
    use_dist = world > 1 and not reference
    if use_dist:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(dev))

    family = args.dataset or wl["data"]
    scaling = args.scaling or wl.get("scaling", "weak")
    desc_wl = dict(wl)
    if scaling == "strong":
        n_total_cfg = args.n_total or wl["n"]
        n_rank = args.n or n_total_cfg // nparts
    else:
        n_rank = args.n or wl["n"]  # the same partition per GPU at every N: per-GPU work is fixed, ideal = constant queries/s
    wl = desc_wl

    # =============================================================================================
    if reference:
        # The reference arm: gamma's CPU engine cannot be built here (SURVEY.md 8c), so the CPU restatement built for speed
        # (baseline/cpu_gamma.c) is timed on this box's host cores.  Rank 0 builds ONE partition on its GPU (the same
        # builder as the `ours` arm), exports it, and searches it on the CPU.  With P partitions the same cores search them
        # one after another, and partitions are statistically identical: global queries/s = partition queries/s / P.
        res = measure_reference(args, wl_name, wl, n_rank, nparts, local, family, scaling)
        print(json.dumps(res))
        return 0

    res = measure(args, wl_name, wl, n_rank, rank, world, local, use_dist, family, args.steps, args.warmup, primary=True)
    if res is None:
        return 0
    default_shape = not (args.n or args.nq or args.nprobe or args.dataset or args.n_total)
    want_c5 = wl_name == "ivfpq_10m" and default_shape and not args.no_secondary and scaling == "weak"
    if rank != 0:
        res["idx"].close()
        del res
        if want_c5:  # every rank holds its share of the 100M database
            try:
                torch.cuda.empty_cache()
                w5 = WORKLOADS["ivfpq_100m"]
                r5 = measure(args, "ivfpq_100m", w5, CONFIGS4_TOTAL // world, rank, world, local, use_dist, w5["data"], 3, 3, primary=False)
                r5["idx"].close()
            except Exception as e:
                print(f"rank {rank}: configs[4] secondary failed: {e!r}", file=sys.stderr)
        if use_dist:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    idx, nq, k, nprobe, recall_num = res["idx"], res["nq"], res["k"], res["nprobe"], res["recall_num"]
    ms_per_step = res["ms_per_step"]
    value = nq / (ms_per_step / 1000)  # global queries/s on the world-partition database
    roofline = make_roofline(idx, wl, wl_name, res["work"], nq, k, recall_num, res["scan_avg"], ms_per_step, default_shape)

    # ---- CPU baseline on this box's host cores (bounded sample) ---------------------------------
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        qps, cores, text, ci_, nsamp = time_cpu(idx, wl, res["xq_host"], k, nprobe, recall_num, budget_s=20.0)
        _, gi_ = idx.search(res["xq_host"][:nsamp], k, params=res["sp"])
        agree = float((gi_ == ci_).mean())
        cpu = {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
               "sample": text + f"; id agreement with the GPU result {agree:.4f}"}

    per_rank = res["per_rank"]
    line = {"metric": metric_string(wl, res["n_total"], nq),
            "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": config_dict(wl, family, n_rank, res["n_total"], world, nq, k, nprobe, recall_num, res["params"], scaling),
            "quality": {"recall@10_1nn_in_top10": res["r1"], "recall@10_standard": res["r10"], "nprobe_sweep": res["sweep"]},
            "build_seconds": res["build"],
            "value_semantics": "global queries/s: every query is answered over ALL partitions of the N-vector database "
                               "(all-gather of result keys + merge included); weak scaling keeps the per-GPU partition fixed, so "
                               "the ideal is a constant value while N grows",
            "partition_queries_per_s": value * world,
            "scan_entries_per_s": res["entries_all_ranks"] / (ms_per_step / 1000),
            "per_rank": {"step_ms": [float(v) / args.steps for v in per_rank[:, 0]],
                         "scan_kernel_ms": [float(v) for v in per_rank[:, 1]],
                         "scan_kernel_ms_min_max": [float(per_rank[:, 1].min()), float(per_rank[:, 1].max())],
                         "allgather_merge_ms": [float(v) for v in per_rank[:, 2]],
                         "vectors": [int(v) for v in per_rank[:, 3]]},
            "stages_ms": res["stages"],
            "clocks": res["clocks"],
            # N=1: the reference-facing C-ABI call gb_index_search(host queries -> host results), H2D/D2H inside;
            # N>1: pinned-host H2D -> search -> NCCL all-gather of keys + merge -> D2H through the Python API
            "e2e": {"value": res["cabi_qps"] if res["cabi_qps"] else res["e2e_qps"], "unit": "queries/s",
                    "h2d_bytes_per_step": nq * wl["d"] * 4, "d2h_bytes_per_step": nq * k * 12,
                    "path": "gb_index_search C-ABI, host buffers" if res["cabi_qps"] else
                            "pinned H2D + search_device_keys + all_gather/merge + D2H",
                    "pinned_h2d_search_d2h_qps": res["e2e_qps"]},
            "gpu_launches": res["launches"],
            "roofline": roofline,
            "cpu_baseline": cpu}
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *res["outputs"])
    idx.close()
    del res

    sec = []
    # ---- BASELINE configs[4], strong scaling: the 100M database split over this run's ranks ----
    if want_c5:
        try:
            torch.cuda.empty_cache()
            w5 = WORKLOADS["ivfpq_100m"]
            r5 = measure(args, "ivfpq_100m", w5, CONFIGS4_TOTAL // world, rank, world, local, use_dist, w5["data"], 3, 3, primary=False)
            v5 = r5["nq"] / (r5["ms_per_step"] / 1000)
            pr = r5["per_rank"]
            sec.append({"workload": w5["desc"], "scaling": "strong", "metric": metric_string(w5, r5["n_total"], r5["nq"]),
                        "n_gpus": world, "n_per_gpu": CONFIGS4_TOTAL // world, "n_total": r5["n_total"], "value": v5,
                        "unit": "queries/s", "ms_per_step": r5["ms_per_step"], "steps": 3, "warmup": 3, "e2e_value": r5["cabi_qps"] or r5["e2e_qps"],
                        "recall@10_1nn": r5["r1"], "recall@10": r5["r10"], "nprobe": r5["nprobe"], "recall_num": r5["recall_num"],
                        "gpu_launches": r5["launches"], "stages_ms": r5["stages"],
                        "per_rank_scan_kernel_ms_min_max": [float(pr[:, 1].min()), float(pr[:, 1].max())],
                        "build_seconds": r5["build"]})
            r5["idx"].close()
            del r5
        except Exception as e:
            sec.append({"workload": "ivfpq_100m", "error": repr(e)[:300]})
    # ---- quick lines for the other single-GPU BASELINE configs (driver-run record of C1 / C2 / C4) ----
    if world == 1 and wl_name == "ivfpq_10m" and default_shape and not args.no_secondary:
        for name in ("flat_100k", "ivfflat_1m", "ivfflat_768"):
            try:
                w2 = WORKLOADS[name]
                torch.cuda.empty_cache()
                r2 = measure(args, name, w2, w2["n"], 0, 1, local, False, w2["data"], 3, 3, primary=False)
                v2 = r2["nq"] / (r2["ms_per_step"] / 1000)
                rf = make_roofline(r2["idx"], w2, name, r2["work"], r2["nq"], r2["k"], r2["recall_num"], r2["scan_avg"],
                                   r2["ms_per_step"], True)
                sec.append({"workload": w2["desc"], "value": v2, "unit": "queries/s", "ms_per_step": r2["ms_per_step"], "steps": 3,
                            "warmup": 3, "e2e_value": r2["cabi_qps"], "recall@10_1nn": r2["r1"], "recall@10": r2["r10"],
                            "nprobe": r2["nprobe"], "gpu_launches": r2["launches"], "stages_ms": r2["stages"],
                            "roofline": {kk: rf.get(kk) for kk in ("kernel", "kernel_ms", "bound", "achieved", "peak", "unit", "frac",
                                                                  "kernel_share_of_step", "secondary")}})
                r2["idx"].close()
                del r2
            except Exception as e:  # a secondary line must never take the primary one down
                sec.append({"workload": name, "error": repr(e)[:300]})
    if sec:
        line["secondary"] = sec

    print(json.dumps(line))
    if use_dist:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def measure_reference(args, wl_name, wl, n_rank, nparts, local, family, scaling):
    import torch
    from vearch_b200 import index as gidx
    nq = args.nq or wl["nq"]
    k = args.k
    nprobe = args.nprobe or wl["nprobe"]
    recall_num = args.recall_num if args.recall_num >= 0 else (400 if wl["type"] == "IVFPQ" else 0)
    idx, params, build = build_index(wl, n_rank, 0, local, family)
    if wl["type"] != "FLAT":
        nprobe = min(nprobe, params["ncentroids"])
    gen = generator(family)
    dev = f"cuda:{local}"
    nbatches = args.warmup + args.steps
    step_qps, texts, cores = [], [], 1
    budget = max(6.0, min(20.0, 120.0 / max(1, nbatches)))  # the whole run stays within a few minutes
    for b in range(nbatches):
        xq = gen(nq, wl["d"], seed=4321 + b, device=dev).cpu().numpy()
        qps, cores, text, _, _ = time_cpu(idx, wl, xq, k, nprobe, recall_num, budget_s=budget, reps=3)
        if b >= args.warmup:
            step_qps.append(qps)
            texts.append(text)
    n_total = idx.ntotal * nparts
    idx.close()
    qps_part = float(np.mean(step_qps))
    value = qps_part / nparts
    sample = (f"{texts[-1]}; {nparts} partition(s): the host cores search them one after another, partitions are statistically "
              f"identical, so global queries/s = queries/s on one partition / {nparts}")
    return {"impl": "reference", "metric": metric_string(wl, n_total, nq), "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * nq / value,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": config_dict(wl, family, n_rank, n_total, nparts, nq, k, nprobe, recall_num, params, scaling),
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}


if __name__ == "__main__":
    sys.exit(main())
