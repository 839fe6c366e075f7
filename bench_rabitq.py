"""IVFRABITQ benchmark on one GPU, measured the way bench.py measures: CUDA events around device-resident searches,
a 512 MiB L2 flush between timed steps, a distinct query batch per step and every shape warmed up first.

Workload (C3's shape): d=128, N=10 M SIFT-like vectors, nlist=4096, nq=10 k, nprobe 32, nb_bits in {1, 4, 9}, qb=4,
with and without an exact re-rank of recall_num=400; the IVFPQ M=16 index on the same data is timed in the same
call for comparison.  Prints one JSON line: per run the step time, queries/s, scan-kernel time, bytes and integer
operations per scanned entry (from shapes), the share of peak of the binding resource, index bytes per vector,
recall@1/10/100 of the true nearest neighbour on a query sample, and the card's name and power limit.

    python bench_rabitq.py [--n 10000000] [--nq 10000] [--out profiles/rabitq_c3.json]

Nothing is written into the tree unless --out is given.  Needs a CUDA device; there is no CPU path.
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

HBM_BPS = 7.7e12         # HGX B200 data sheet, per GPU
POPC_PER_SM_CLK = 16     # CUDA C++ Programming Guide throughput table (32-bit __popc per SM per clock)


def card():
    q = "name,power.limit,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(", ")
        return {"name": out[0], "power_limit_w": float(out[1]), "sm_max_mhz": float(out[2])}
    except Exception as ex:  # noqa: BLE001
        return {"name": None, "power_limit_w": None, "sm_max_mhz": None, "error": str(ex)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=10_000_000)
    ap.add_argument("--d", type=int, default=128)
    ap.add_argument("--nlist", type=int, default=4096)
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--nprobe", type=int, default=32)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--qb", type=int, default=4)
    ap.add_argument("--nb-bits", default="1,4,9")
    ap.add_argument("--recall-num", default="0,400")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--recall-sample", type=int, default=1000)
    ap.add_argument("--no-ivfpq", action="store_true")
    ap.add_argument("--out", default="", help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_rabitq.py needs a CUDA device (there is no CPU path)")
    torch.backends.cuda.matmul.allow_tf32 = False
    from vearch_b200 import index as gidx, synth

    dev = torch.device("cuda:0")
    info = card()
    d, n, nq, k, nprobe = args.d, args.n, args.nq, args.k, args.nprobe
    nbatch = args.warmup + args.steps
    chunk = 1 << 20

    def gen_db(s, e):
        return synth.sift_like_torch(e - s, d, seed=1234 + (s >> 20), device="cuda:0")

    q_dev = [synth.sift_like_torch(nq, d, seed=900 + b, device="cuda:0").contiguous() for b in range(nbatch)]
    xs = synth.sift_like_torch(args.recall_sample, d, seed=777, device="cuda:0")
    # true nearest neighbour of the recall sample (exact fp32 |x|^2 - 2<q,x> against every chunk)
    best_d = torch.full((xs.shape[0],), float("inf"), device=dev)
    best_i = torch.zeros((xs.shape[0],), dtype=torch.int64, device=dev)
    for s in range(0, n, chunk):
        x = gen_db(s, min(n, s + chunk))
        dd = (x * x).sum(1)[None, :] - 2.0 * xs @ x.T
        v, i = dd.min(1)
        upd = v < best_d
        best_d = torch.where(upd, v, best_d)
        best_i = torch.where(upd, i + s, best_i)
        del x, dd
    gt = best_i.cpu().numpy()
    xs_host = xs.cpu().numpy()
    q0_host = q_dev[0].cpu().numpy()
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def build(typ, extra):
        p = {"metric_type": "L2", "ncentroids": args.nlist, "nprobe": nprobe, "training_threshold": min(n, 200 * args.nlist)}
        p.update(extra)
        idx = gidx.GammaIndex(typ, d, p)
        t0 = time.time()
        for s in range(0, n, chunk):
            idx.add_vectors(gen_db(s, min(n, s + chunk)))
        torch.cuda.synchronize()
        idx.train()
        idx.add_pending()
        return idx, round(time.time() - t0, 2)

    def timed(idx, params):
        out = (torch.empty((nq, k), dtype=torch.float32, device=dev), torch.empty((nq, k), dtype=torch.int64, device=dev))
        for b in range(args.warmup):
            idx.search_device(q_dev[b], k, params=params, out=out)
        torch.cuda.synchronize()
        idx.set_scan_timing(True)
        _ = idx.last_scan_ms
        step_ms, scan_ms = [], []
        for s in range(args.steps):
            flush.fill_(s)  # L2 flush between timed steps (untimed)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            idx.search_device(q_dev[args.warmup + s], k, params=params, out=out)
            e1.record()
            torch.cuda.synchronize()
            step_ms.append(e0.elapsed_time(e1))
            scan_ms.append(idx.last_scan_ms)
        idx.set_scan_timing(False)
        _, ri = idx.search(xs_host, 100, params=params)
        rec = {f"recall@{r}": float(np.mean([gt[i] in ri[i, :r] for i in range(len(gt))])) for r in (1, 10, 100)}
        ms = float(np.median(step_ms))
        return {"ms_per_step": round(ms, 4), "qps": round(nq / ms * 1e3, 1), "scan_ms": round(float(np.median(scan_ms)), 4),
                "scan_kernel": idx.last_scan_kernel, **rec}

    def entries_scanned(idx):
        lens = np.array([idx.list_len(l) for l in range(idx.nlist)], np.int64)
        _, keys = idx.coarse_search(q0_host, nprobe)
        return float(lens[keys[keys >= 0]].sum())

    peak_popc = 148 * POPC_PER_SM_CLK * (info["sm_max_mhz"] or 0) * 1e6
    runs = []
    for nb in [int(v) for v in args.nb_bits.split(",")]:
        idx, build_s = build("IVFRABITQ", {"nb_bits": nb, "qb": args.qb})
        cs = idx.code_size
        ent = entries_scanned(idx)
        words = (d + 31) // 32
        popc = words * nb * (args.qb + 1)  # POPC per entry; each comes with an AND and a shift-add
        for rn in [int(v) for v in args.recall_num.split(",")]:
            params = {"nprobe": nprobe, "qb": args.qb}
            if rn > 0:
                params["recall_num"] = rn
            r = timed(idx, params)
            byts = ent * (cs + 8)
            t_hbm = byts / HBM_BPS
            t_int = ent * popc / peak_popc if peak_popc else float("nan")
            bound = "integer pipe (POPC)" if t_int > t_hbm else "HBM bytes"
            r.update(index="IVFRABITQ", nb_bits=nb, qb=args.qb, recall_num=rn, build_s=build_s, code_size=cs,
                     bytes_per_entry=cs + 8, popc_per_entry=popc, int_ops_per_entry=3 * popc,
                     entries_scanned_per_batch=ent, index_bytes_per_vector=round(idx.mem_bytes(0) / n, 2),
                     achieved_hbm_tbps=round(byts / (r["scan_ms"] * 1e-3) / 1e12, 3),
                     achieved_popc_per_s=round(ent * popc / (r["scan_ms"] * 1e-3), 1),
                     binding_resource=bound, share_of_peak=round(max(t_hbm, t_int) / (r["scan_ms"] * 1e-3), 4))
            runs.append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
        idx.close()
    if not args.no_ivfpq:
        idx, build_s = build("IVFPQ", {"nsubvector": 16, "nbits_per_idx": 8})
        for rn in [int(v) for v in args.recall_num.split(",")]:
            params = {"nprobe": nprobe}
            if rn > 0:
                params["recall_num"] = rn
            r = timed(idx, params)
            r.update(index="IVFPQ", M=16, recall_num=rn, build_s=build_s,
                     index_bytes_per_vector=round(idx.mem_bytes(0) / n, 2))
            runs.append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
        idx.close()
    line = json.dumps({"bench": "bench_rabitq", "card": info, "d": d, "n": n, "nlist": args.nlist, "nq": nq, "k": k,
                       "nprobe": nprobe, "steps": args.steps, "warmup": args.warmup, "l2_flush_mib": 512,
                       "peaks": {"hbm_bytes_per_s": HBM_BPS, "popc_per_s": peak_popc,
                                 "popc_source": "148 SMs x 16 POPC/clk (CUDA C++ Programming Guide) x clocks.max.sm"},
                       "runs": runs})
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
