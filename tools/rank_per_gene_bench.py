"""Time the ranks of held-out triplets per query gene (Model.rank_held_out_per_gene, tip_rank_per_gene) on one GPU and
write profiles/rank_per_gene_bench.json.

    python tools/rank_per_gene_bench.py [--out profiles/rank_per_gene_bench.json] [--quick]

Setup of tools/rank_held_out_bench.py and tools/rank_per_pair_bench.py: P = 6000 genes, the 1e6 Kuzmin-shaped links of
bench.py's cfg2 split into five folds after a seeded shuffle; fold 1 is the test set and the other four the train set.
Parameters are random, seeded; (K, S) = (3, 1), (10, 1), (10, 10).  Two view sets:
- all views: every ranked test triplet of fold 1, one view per gene (queries=None);
- query-gene views: the 77 query (hub) genes of the Kuzmin shape, listed; these hold the most test and train triplets.
Per workload: the queries and the views; the capture and count sweeps (the two tip_gene_rank_pass_kernel launches of a
call: device time from torch.profiler, median of 5 calls); pair scores per second of the count sweep (every pair of every
query once per round) and the share of the DMMA peak tip_measure_fma_peak(2) measured in the same run, at 2 S K flop per
score; the whole rank_held_out_per_gene call (host clock around the call, which ends in a device synchronise; median of 3
after one warm-up call); one tip_top_triplets_per_gene call at N = 20 on the same queries (CUDA events, median of 5) for
the ratio.
Baseline: the brute force, tip_score over every pair of a few queries and a sort of the scores, host clock around a
synchronised run; its extrapolation to all the workload's queries is labelled as such.  The GPU's name, power limit and
max SM clock are read with read-only nvidia-smi queries."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from predict_bench import gpu_info, params, time_calls  # noqa: E402
from rank_held_out_bench import fold1_model, host_time  # noqa: E402


def sweep_ms(torch, fn, reps=5):
    """Median device ms of the capture and the count launch of tip_gene_rank_pass_kernel over `reps` calls of fn."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if "tip_gene_rank_pass_kernel" in e.name and "CUDA" in str(e.device_type)),
                key=lambda e: e.time_range.start)
    dur = [e.time_range.elapsed_us() / 1e3 for e in ev]
    assert len(dur) == 2 * reps, len(dur)
    return float(np.median(dur[0::2])), float(np.median(dur[1::2]))


def brute_force(torch, lib, eng, th, pr, cand_np, qr, P):
    """Every pair of each query rank in qr through tip_score (first parameter set) and a full sort of its scores; host
    clock around a synchronised run, after one warm-up run."""
    eng.set_params(th[0], pr[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)

    def run():
        for r in qr:
            others = torch.cat([torch.arange(r, device=dev), torch.arange(r + 1, P, device=dev)])
            iu = torch.triu_indices(P - 1, P - 1, offset=1, device=dev)
            rr = torch.stack([others[iu[0]], others[iu[1]], torch.full((iu.shape[1],), r, device=dev)], 1).sort(dim=1).values
            g = cand[rr].to(torch.int32)
            g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
            s = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
            lib.tip_score(P, eng.K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()), ctypes.c_void_p(g3.data_ptr()),
                          g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                          ctypes.c_void_p(s.data_ptr()), eng._stream())
            torch.sort(s, descending=True)
    run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    run()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / len(qr)


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "rank_per_gene_bench needs a CUDA device"
    lib = _cabi.load()
    P, L = (1500, 100_000) if args.quick else (6000, 1_000_000)
    nq = max(4, int(round(P ** 0.5)))
    m = fold1_model(P, L)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    rank = np.empty(P, dtype=np.int64)
    rank[cand] = np.arange(P)
    train = m._train_packed(cand)
    peak = ctypes.c_double(0)
    _cabi.check(lib.tip_measure_fma_peak(2, ctypes.byref(peak)), "tip_measure_fma_peak")
    pairs = (P - 1) * (P - 2) // 2
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "links": L, "train_links": len(m.links),
           "test_links": len(m.test_links), "train_triplets": int(len(train)), "query_genes": nq, "pairs_per_query": pairs,
           "flop_rule": "2 S K per pair score", "workloads": [], "baseline": []}
    query_genes = ["g%d" % a for a in range(nq)]
    rng = np.random.default_rng(2027)
    for K, S in [(3, 1), (10, 1), (10, 10)]:
        th, pr = params(rng, P, K, S)
        sets = [(th[s], pr[s]) for s in range(S)]
        eng = EMEngine(P, K, device="cuda:0")
        m._engine, m._engine_key = eng, (P, K)           # rank_held_out_per_gene reuses this engine
        for name, queries in [("all views", None), ("query-gene views", query_genes)]:
            res = {}

            def call():
                res["r"] = m.rank_held_out_per_gene(queries, params=sets)
            sec, secs = host_time(call)
            r = res["r"]
            qr = np.array([rank[int(g[0][1:])] for g in r["genes"]], dtype=np.int32)
            cap_ms, cnt_ms = sweep_ms(torch, call)
            scores = len(qr) * pairs
            t20, _, _ = time_calls(torch, lambda: eng.top_triplets_per_gene(th, pr, cand, qr, train, 20))
            passes = int(lib.tip_top_triplets_per_gene_last_passes())
            w = {"K": K, "S": S, "views_set": name, "queries": len(qr), "views": r["views"], "positives": r["positives"],
                 "capture_ms": cap_ms, "count_ms": cnt_ms, "pair_scores_per_count_sweep": scores,
                 "count_pair_scores_per_s": scores / (cnt_ms * 1e-3),
                 "count_fp64_tflops": 2.0 * S * K * scores / (cnt_ms * 1e-3) / 1e12,
                 "count_share_of_dmma_peak": 2.0 * S * K * scores / (cnt_ms * 1e-3) / 1e12 / peak.value,
                 "call_s": sec, "call_s_calls": secs, "top20_per_gene_ms": t20, "top20_per_gene_passes": passes,
                 "sweeps_over_one_top20_call": (cap_ms + cnt_ms) / t20,
                 "hits_at": {str(k): v for k, v in r["hits_at"].items()}, "median_rank": r["median_rank"],
                 "mrr": r["mrr"], "auc_micro": r["auc_micro"], "auc_macro": r["auc_macro"]}
            if K == 10 and S == 1:
                timed = qr[:4].tolist()
                per_q = brute_force(torch, lib, eng, th, pr, cand, timed, P)
                b = {"K": K, "S": 1, "views_set": name, "queries": len(qr), "queries_timed": len(timed),
                     "seconds_per_query": per_q, "extrapolated_s": per_q * len(qr),
                     "speedup_over_extrapolated": per_q * len(qr) / sec,
                     "note": "tip_score over every pair of each timed query + a full sort of its scores, host clock around "
                             "a synchronised run; the whole-set time is extrapolated from the timed queries, not measured, "
                             "and leaves out finding the test triplets in the sorted lists"}
                print(json.dumps(b), flush=True)
                out["baseline"].append(b)
            print(json.dumps(w), flush=True)
            out["workloads"].append(w)
        m._engine = None
        del eng
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rank_per_gene_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
