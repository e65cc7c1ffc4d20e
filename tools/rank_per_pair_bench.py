"""Time the ranks of held-out triplets per query pair (Model.rank_held_out_per_pair, tip_rank_per_pair) on one GPU and
write profiles/rank_per_pair_bench.json.

    python tools/rank_per_pair_bench.py [--out profiles/rank_per_pair_bench.json] [--quick]

Setup of tools/rank_held_out_bench.py: P = 6000 genes, the 1e6 Kuzmin-shaped links of bench.py's cfg2 split into five
folds after a seeded shuffle; fold 1 is the test set and the other four the train set.  Parameters are random, seeded;
(K, S) = (3, 1), (10, 1), (10, 10).  Two view sets:
- all views: every ranked test triplet of fold 1, one view per pair of its genes (pairs=None);
- query-pair views: the pairs of two query (hub) genes, every one of the C(77, 2) pairs listed; these are the heavy rows
  (about 270 train and 65 test partners each).
Per workload: the distinct pairs and the views; the capture and count sweeps (the two tip_rank_pass_kernel launches of a
call: device time from torch.profiler, median of 5 calls); partner scores per second of the count sweep (every partner
of every pair once per round) and the share of the DMMA peak tip_measure_fma_peak(2) measured in the same run, at
2 S K flop per partner score; the whole rank_held_out_per_pair call (host clock around the call, which ends in a device
synchronise; median of 3 after one warm-up call); one tip_top_triplets_per_pair call at N = 20 on the same pairs (CUDA
events, median of 5) for the ratio.
Baseline: the exact composition, tip_top_triplets_per_pair with N = n - 2 and the train keys known, in chunks of
2^24 / (n - 2) pairs; one chunk is timed (CUDA events) and the time is extrapolated to all pairs by the chunk count, and
labelled as such.  The GPU's name, power limit and max SM clock are read with read-only nvidia-smi queries."""
from __future__ import annotations

import argparse
import ctypes
import itertools
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from predict_bench import gpu_info, params, time_calls  # noqa: E402
from rank_held_out_bench import fold1_model, host_time  # noqa: E402


def sweep_ms(torch, fn, reps=5):
    """Median device ms of the capture and the count launch of tip_rank_pass_kernel over `reps` calls of fn."""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if "tip_rank_pass_kernel" in e.name and "CUDA" in str(e.device_type)),
                key=lambda e: e.time_range.start)
    dur = [e.time_range.elapsed_us() / 1e3 for e in ev]
    assert len(dur) == 2 * reps, len(dur)
    return float(np.median(dur[0::2])), float(np.median(dur[1::2]))


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "rank_per_pair_bench needs a CUDA device"
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
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "links": L, "train_links": len(m.links),
           "test_links": len(m.test_links), "train_triplets": int(len(train)), "query_genes": nq,
           "flop_rule": "2 S K per partner score", "workloads": [], "baseline": []}
    query_pairs = [("g%d" % a, "g%d" % b) for a, b in itertools.combinations(range(nq), 2)]
    rng = np.random.default_rng(2026)
    for K, S in [(3, 1), (10, 1), (10, 10)]:
        th, pr = params(rng, P, K, S)
        sets = [(th[s], pr[s]) for s in range(S)]
        eng = EMEngine(P, K, device="cuda:0")
        m._engine, m._engine_key = eng, (P, K)           # rank_held_out_per_pair reuses this engine
        for name, pairs in [("all views", None), ("query-pair views", query_pairs)]:
            res = {}

            def call():
                res["r"] = m.rank_held_out_per_pair(pairs, params=sets)
            sec, secs = host_time(call)
            r = res["r"]
            pr_ranks = np.array([[rank[int(x[1:])] for x in p[0].split("+")] for p in r["pairs"]], dtype=np.int32)
            cap_ms, cnt_ms = sweep_ms(torch, call)
            scores = len(pr_ranks) * (P - 2)
            t20, _, _ = time_calls(torch, lambda: eng.top_triplets_per_pair(th, pr, cand, pr_ranks, train, 20))
            passes = int(lib.tip_top_triplets_per_pair_last_passes())
            w = {"K": K, "S": S, "views_set": name, "pairs": len(pr_ranks), "views": r["views"],
                 "positives": r["positives"], "capture_ms": cap_ms, "count_ms": cnt_ms,
                 "partner_scores_per_count_sweep": scores, "count_partner_scores_per_s": scores / (cnt_ms * 1e-3),
                 "count_fp64_tflops": 2.0 * S * K * scores / (cnt_ms * 1e-3) / 1e12,
                 "count_share_of_dmma_peak": 2.0 * S * K * scores / (cnt_ms * 1e-3) / 1e12 / peak.value,
                 "call_s": sec, "call_s_calls": secs, "top20_per_pair_ms": t20, "top20_per_pair_passes": passes,
                 "top20_per_pair_ms_per_pass": t20 / max(passes, 1),
                 "sweeps_over_one_top20_pass": (cap_ms + cnt_ms) / (t20 / max(passes, 1)),
                 "hits_at": {str(k): v for k, v in r["hits_at"].items()}, "median_rank": r["median_rank"],
                 "mrr": r["mrr"], "auc_micro": r["auc_micro"], "auc_macro": r["auc_macro"]}
            if K == 10 and S == 1:
                chunk = (1 << 24) // (P - 2)
                sub = pr_ranks[:chunk]
                tb, _, _ = time_calls(torch, lambda: eng.top_triplets_per_pair(th, pr, cand, sub, train, P - 2), reps=3)
                n_chunks = -(-len(pr_ranks) // chunk)
                b = {"K": K, "S": S, "views_set": name, "pairs": len(pr_ranks), "chunk_pairs": int(len(sub)),
                     "chunk_ms": tb, "chunks": n_chunks, "extrapolated_s": tb * n_chunks / 1e3,
                     "speedup_over_extrapolated": tb * n_chunks / 1e3 / sec,
                     "note": "tip_top_triplets_per_pair with N = n - 2 and the train keys known, one chunk of 2^24 / (n - 2) "
                             "pairs timed with CUDA events (median of 3); the whole-set time is that times the chunk count, "
                             "extrapolated, not measured, and leaves out finding the test partners in the lists"}
                print(json.dumps(b), flush=True)
                out["baseline"].append(b)
            print(json.dumps(w), flush=True)
            out["workloads"].append(w)
        m._engine = None
        del eng
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rank_per_pair_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
