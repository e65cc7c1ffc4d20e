"""Time tip_top_triplets_per_gene (per-gene top-N of unseen triplets) on one GPU and write
profiles/predict_per_gene_bench.json.

    python tools/predict_per_gene_bench.py [--out profiles/predict_per_gene_bench.json] [--quick]

Workloads: P = 6000 genes, N = 20 per query, the 1e6 Kuzmin-shaped links of bench.py's cfg2 as known triplets (as
tools/predict_bench.py); K = 10 with S = 1 and S = 10, and K = 3 with S = 1; queries: 100 random genes, and all 6 000.
Parameters are random (Dirichlet theta rows, p normalised over the rating), seeded.  Per workload: sweeps (passes), ms per
call (CUDA events, median of 5 calls, each call >= 20 ms), triplet evaluations per second (queries * C(P - 1, 2) * passes,
an upper bound of what the later sweeps score, as they skip resolved queries), fp64 flop/s at 2 S K flop per evaluation
and its share of the DMMA peak tip_measure_fma_peak(2) measured in the same run.  Baseline: every pair of a few queries
scored by tip_score with a torch.topk, timed, and extrapolated to every query of the workload (labelled as such).  The
GPU's name, power limit and max SM clock are read with read-only nvidia-smi queries."""
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

from predict_bench import gpu_info, known_from_cfg2, params, time_calls  # noqa: E402


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "predict_per_gene_bench needs a CUDA device"
    lib = _cabi.load()
    P, N, L = (1500, 20, 100_000) if args.quick else (6000, 20, 1_000_000)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = known_from_cfg2(P, L, cand)
    peak = ctypes.c_double(0)
    _cabi.check(lib.tip_measure_fma_peak(2, ctypes.byref(peak)), "tip_measure_fma_peak")
    pairs = (P - 1) * (P - 2) // 2
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "N": N, "known_links": L,
           "known_triplets": int(len(known)), "pairs_per_query": pairs,
           "flop_rule": "2 S K per triplet evaluation; evaluations = queries * C(P-1, 2) * passes", "workloads": [],
           "baseline": []}
    rng = np.random.default_rng(2025)
    few = np.sort(rng.choice(P, size=100, replace=False)).astype(np.int32)
    for K, S in [(10, 1), (10, 10), (3, 1)]:
        th, pr = params(rng, P, K, S)
        eng = EMEngine(P, K, device="cuda:0")
        for label, qr in [("100 random genes", few), ("all genes", np.arange(P, dtype=np.int32))]:
            res = {}

            def call():
                res["r"] = eng.top_triplets_per_gene(th, pr, cand, qr, known, N)
            med, times, inner = time_calls(torch, call)
            passes = int(lib.tip_top_triplets_per_gene_last_passes())
            evals = float(len(qr)) * pairs * passes
            flop = 2.0 * S * K * evals
            ids, sc, cnt = res["r"]
            w = {"K": K, "S": S, "queries": label, "n_query": int(len(qr)), "passes": passes, "ms_per_call": med,
                 "ms_calls": times, "calls_per_window": inner, "triplet_evals_per_s": evals / (med * 1e-3),
                 "fp64_tflops": flop / (med * 1e-3) / 1e12, "share_of_dmma_peak": flop / (med * 1e-3) / 1e12 / peak.value,
                 "rows": int(cnt.sum()), "min_rows": int(cnt.min()), "top_score": float(np.nanmax(sc[:, 0]))}
            print(json.dumps(w), flush=True)
            out["workloads"].append(w)
        out["baseline"].append(baseline(torch, lib, eng, th, pr, cand, few[:4], N, P))
        del eng
    return out


def baseline(torch, lib, eng, th, pr, cand_np, qr, N, P):
    """Every pair of each query through tip_score (first parameter set, S = 1) and a torch.topk; host clock around a
    synchronised run of all `qr` queries, extrapolated to 100 and to P queries."""
    eng.set_params(th[0], pr[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)

    def brute():
        for r in qr.tolist():
            others = torch.cat([torch.arange(r, device=dev), torch.arange(r + 1, P, device=dev)])
            iu = torch.triu_indices(P - 1, P - 1, offset=1, device=dev)
            rr = torch.stack([others[iu[0]], others[iu[1]], torch.full((iu.shape[1],), r, device=dev)], 1).sort(dim=1).values
            g = cand[rr].to(torch.int32)
            g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
            s = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
            lib.tip_score(P, eng.K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()), ctypes.c_void_p(g3.data_ptr()),
                          g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                          ctypes.c_void_p(s.data_ptr()), eng._stream())
            torch.topk(s, N)
    brute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    brute()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    per_q = sec / len(qr)
    return {"K": eng.K, "S": 1, "queries_timed": int(len(qr)), "seconds": sec, "seconds_per_query": per_q,
            "triplets_per_s": len(qr) * (P - 1) * (P - 2) / 2 / sec, "extrapolated_100_queries_s": 100 * per_q,
            "extrapolated_all_queries_s": P * per_q,
            "note": "tip_score over every pair of each query + torch.topk, host clock around a synchronised run; the 100- "
                    "and %d-query figures are extrapolated from the timed queries, not measured" % P}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predict_per_gene_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
