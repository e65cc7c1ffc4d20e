"""Time the ranks of held-out triplets (Model.rank_held_out, tip_score_histogram) on one GPU and write
profiles/rank_held_out_bench.json.

    python tools/rank_held_out_bench.py [--out profiles/rank_held_out_bench.json] [--quick]

Setup of tools/predict_bench.py: P = 6000 genes, the 1e6 Kuzmin-shaped links of bench.py's cfg2, split into five folds
after a seeded shuffle; fold 1 is the test set and the other four the train set.  Parameters are random (Dirichlet theta
rows, p normalised over the rating), seeded; (K, S) = (3, 1), (3, 10), (10, 1), (10, 10).  Per workload:
- the counting sweep: ms per tip_score_histogram call (CUDA events, median of 5 calls, each window >= 20 ms), triplets/s,
  fp64 flop/s at 2 S K flop per triplet and its share of the DMMA peak tip_measure_fma_peak(2) measured in the same run;
  beside it one tip_top_triplets call at N = 1 000 with the train keys known, timed the same way, and its pass count;
- the whole Model.rank_held_out call at n_exact = 1e4, 1e5, 1e6 (host clock around the call, which ends in a device
  synchronise; median of 3 after one warm-up call).
Baseline at P = 1500, K = 4, S = 1 (the §4.5 baseline shape), 1e5 links: every triplet scored through tip_score in chunks,
and each test triplet's rank counted from them (a sort per chunk and a binary search per test triplet); host clock around a
synchronised run.  It is extrapolated to P = 6000 by the triplet count and labelled as such.  rank_held_out at the same
P, K, S and n_exact = 1e5 is timed beside it.  The GPU's name, power limit and max SM clock are read with read-only
nvidia-smi queries."""
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


def fold1_model(P, n_links):
    """A Model holding the Kuzmin-shaped links, fold 1 as test and the rest as train; genes named g<id>."""
    from trigenicinteractionpredictor_b200 import Model, synth
    g1, g2, g3, lab = synth.kuzmin_links_soa(P, n_links, seed=1)
    order = np.random.default_rng(7).permutation(n_links)
    per = n_links // 5
    test, train = order[per:2 * per], np.concatenate([order[:per], order[2 * per:]])
    soa = lambda ix: (g1[ix], g2[ix], g3[ix], (1 - lab[ix]).astype(np.int32), lab[ix].astype(np.int32))  # noqa: E731
    m = Model()
    m.set_links_soa(soa(train), soa(test), P=P)
    m.id_gene = {i: "g%d" % i for i in range(P)}
    m.gene_id = {v: k for k, v in m.id_gene.items()}
    return m


def host_time(fn, reps=3):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return float(np.median(times)), times


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "rank_held_out_bench needs a CUDA device"
    lib = _cabi.load()
    P, L = (1500, 100_000) if args.quick else (6000, 1_000_000)
    m = fold1_model(P, L)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    train = m._train_packed(cand)
    peak = ctypes.c_double(0)
    _cabi.check(lib.tip_measure_fma_peak(2, ctypes.byref(peak)), "tip_measure_fma_peak")
    trip = P * (P - 1) * (P - 2) // 6
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "links": L, "train_links": len(m.links),
           "test_links": len(m.test_links), "train_triplets": int(len(train)), "triplets": trip,
           "flop_rule": "2 S K per triplet", "sweep": [], "rank_held_out": [], "baseline": None}
    rng = np.random.default_rng(2026)
    for K, S in [(3, 1), (3, 10), (10, 1), (10, 10)]:
        th, pr = params(rng, P, K, S)
        eng = EMEngine(P, K, device="cuda:0")
        m._engine, m._engine_key = eng, (P, K)           # rank_held_out reuses this engine
        med, times, inner = time_calls(torch, lambda: eng.score_histogram(th, pr, cand))
        flop = 2.0 * S * K * trip
        tmed, _, _ = time_calls(torch, lambda: eng.top_triplets(th, pr, cand, train, 1000))
        passes = int(lib.tip_top_triplets_last_passes())
        w = {"K": K, "S": S, "hist_ms_per_call": med, "hist_ms_calls": times, "calls_per_window": inner,
             "triplets_per_s": trip / (med * 1e-3), "fp64_tflops": flop / (med * 1e-3) / 1e12,
             "share_of_dmma_peak": flop / (med * 1e-3) / 1e12 / peak.value,
             "top_triplets_ms_per_call": tmed, "top_triplets_passes": passes,
             "top_triplets_ms_per_pass": tmed / max(passes, 1), "hist_over_top_triplets_pass": med / (tmed / max(passes, 1))}
        print(json.dumps(w), flush=True)
        out["sweep"].append(w)
        sets = [(th[s], pr[s]) for s in range(S)]
        for n_exact in ([10_000, 100_000] if args.quick else [10_000, 100_000, 1_000_000]):
            res = {}

            def call():
                res["r"] = m.rank_held_out(n_exact=n_exact, params=sets)
            sec, secs = host_time(call)
            r = res["r"]
            exact = sum(1 for row in r["rows"] if row[4] == row[5])
            rr = {"K": K, "S": S, "n_exact": n_exact, "seconds": sec, "seconds_calls": secs, "universe": r["universe"],
                  "ranked": len(r["rows"]), "exact_ranks": exact, "positives": r["positives"],
                  "median_rank": r["median_rank"], "auc": r["auc"],
                  "recall_at": {str(k): v for k, v in r["recall_at"].items()}}
            print(json.dumps(rr), flush=True)
            out["rank_held_out"].append(rr)
        m._engine = None
        del eng
    out["baseline"] = baseline(torch, lib)
    return out


def baseline(torch, lib):
    """Brute force at P = 1500, K = 4, S = 1: every triplet through tip_score in chunks, each test triplet's rank counted
    against every chunk; and Model.rank_held_out on the same model beside it."""
    from trigenicinteractionpredictor_b200.engine import EMEngine
    P, K, L = 1500, 4, 100_000
    m = fold1_model(P, L)
    th, pr = params(np.random.default_rng(4), P, K, 1)
    eng = EMEngine(P, K, device="cuda:0")
    eng.set_params(th[0], pr[0])
    m._engine, m._engine_key = eng, (P, K)
    dev = eng.device
    cand_np = np.array(sorted(range(P), key=str), dtype=np.int32)
    cand = torch.from_numpy(cand_np).to(dev)
    t = m._soa(m.test_links)
    tg = torch.from_numpy(np.stack([np.asarray(x) for x in t[:3]], 1)).to(dev)
    t_sc = torch.empty(tg.shape[0], dtype=torch.float64, device=dev)

    def score(g, out):
        g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
        _cabi_check(lib.tip_score(P, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()),
                                  ctypes.c_void_p(g3.data_ptr()), g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()),
                                  ctypes.c_void_p(eng.p.data_ptr()), ctypes.c_void_p(out.data_ptr()), eng._stream()))

    def brute():
        score(tg, t_sc)
        before = torch.zeros(tg.shape[0], dtype=torch.int64, device=dev)
        j = 1
        while j < P - 1:
            parts, size = [], 0
            while j < P - 1 and size < 8_000_000:
                A, C = torch.meshgrid(torch.arange(j, device=dev), torch.arange(j + 1, P, device=dev), indexing="ij")
                parts.append(torch.stack([A.reshape(-1), torch.full((A.numel(),), j, device=dev), C.reshape(-1)], 1))
                size += j * (P - 1 - j)
                j += 1
            g = cand[torch.cat(parts)].to(torch.int32)
            s = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
            score(g, s)
            s = torch.sort(s).values
            before += s.numel() - torch.searchsorted(s, t_sc, right=True)
        return before
    brute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    brute()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    new, _ = host_time(lambda: m.rank_held_out(n_exact=100_000, params=[(th[0], pr[0])]))
    trip = P * (P - 1) * (P - 2) // 6
    trip6k = 6000 * 5999 * 5998 // 6
    return {"P": P, "K": K, "S": 1, "links": L, "brute_force_s": sec, "brute_force_triplets_per_s": trip / sec,
            "brute_force_extrapolated_P6000_s": sec * trip6k / trip, "rank_held_out_s": new, "speedup": sec / new,
            "note": "brute force: tip_score over every triplet in chunks of 8e6, a sort per chunk and a binary search per "
                    "test triplet, host clock around a synchronised run; the P = 6000 figure is extrapolated by the "
                    "triplet count, not measured"}


def _cabi_check(rc):
    assert rc == 0, rc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "rank_held_out_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
