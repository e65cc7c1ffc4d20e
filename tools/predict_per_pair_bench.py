"""Time tip_top_triplets_per_pair (per-pair top-N of unseen triplets) on one GPU and write
profiles/predict_per_pair_bench.json.

    python tools/predict_per_pair_bench.py [--out profiles/predict_per_pair_bench.json] [--quick]

Workloads: P = 6000 genes, N = 20 per pair, the 1e6 Kuzmin-shaped links of bench.py's cfg2 as known triplets (as
tools/predict_bench.py); (K, S) = (10, 1), (10, 10), (3, 1); 1 000 and 100 000 pairs drawn from the Kuzmin query genes x
all genes, the shape of a double-mutant screen.  Parameters are random (Dirichlet theta rows, p normalised over the
rating), seeded.  Per workload: sweeps (passes), ms per call (CUDA events, median of 5 calls, each call >= 20 ms), triplet
evaluations per second (pairs * (P - 2) * passes, an upper bound of what the later sweeps score, as they skip resolved
pairs), fp64 flop/s at 2 S K flop per evaluation and its share of the DMMA peak tip_measure_fma_peak(2) measured in the
same run.  For the one-sweep rate, tip_top_triplets at N = 1 000 is timed at the same K and S.  Baseline: every partner of
a few pairs scored by tip_score and sorted, timed, and extrapolated to every pair of the workload (labelled as such).  The
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


def query_pairs(rng, P, n_pairs, cand):
    """Distinct pairs (rank, rank) of a Kuzmin query gene (ids 0 .. nq - 1, as synth.kuzmin_links_soa) and any other gene."""
    nq = max(4, int(round(P ** 0.5)))
    rank = np.empty(P, dtype=np.int64)
    rank[cand] = np.arange(P)
    q = rng.integers(0, nq, size=3 * n_pairs)
    g = rng.integers(0, P, size=3 * n_pairs)
    keep = q != g
    a, b = np.minimum(q[keep], g[keep]), np.maximum(q[keep], g[keep])
    _, first = np.unique(a * P + b, return_index=True)
    first = np.sort(first)[:n_pairs]
    assert len(first) == n_pairs
    return np.stack([rank[q[keep][first]], rank[g[keep][first]]], 1).astype(np.int32)


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "predict_per_pair_bench needs a CUDA device"
    lib = _cabi.load()
    P, N, L = (1500, 20, 100_000) if args.quick else (6000, 20, 1_000_000)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = known_from_cfg2(P, L, cand)
    peak = ctypes.c_double(0)
    _cabi.check(lib.tip_measure_fma_peak(2, ctypes.byref(peak)), "tip_measure_fma_peak")
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "N": N, "known_links": L,
           "known_triplets": int(len(known)), "partners_per_pair": P - 2,
           "flop_rule": "2 S K per triplet evaluation; evaluations = pairs * (P - 2) * passes", "workloads": [],
           "top_triplets": [], "baseline": []}
    rng = np.random.default_rng(2026)
    sizes = [1_000, 100_000] if not args.quick else [1_000, 10_000]
    pair_sets = {n: query_pairs(rng, P, n, cand) for n in sizes}
    for K, S in [(10, 1), (10, 10), (3, 1)]:
        th, pr = params(rng, P, K, S)
        eng = EMEngine(P, K, device="cuda:0")
        for n_pairs, prs in pair_sets.items():
            res = {}

            def call():
                res["r"] = eng.top_triplets_per_pair(th, pr, cand, prs, known, N)
            med, times, inner = time_calls(torch, call)
            passes = int(lib.tip_top_triplets_per_pair_last_passes())
            evals = float(n_pairs) * (P - 2) * passes
            flop = 2.0 * S * K * evals
            ids, sc, cnt = res["r"]
            w = {"K": K, "S": S, "n_pairs": n_pairs, "passes": passes, "ms_per_call": med, "ms_calls": times,
                 "calls_per_window": inner, "triplet_evals_per_s": evals / (med * 1e-3),
                 "fp64_tflops": flop / (med * 1e-3) / 1e12, "share_of_dmma_peak": flop / (med * 1e-3) / 1e12 / peak.value,
                 "rows": int(cnt.sum()), "min_rows": int(cnt.min()), "top_score": float(np.nanmax(sc[:, 0]))}
            print(json.dumps(w), flush=True)
            out["workloads"].append(w)

        def glob():
            eng.top_triplets(th, pr, cand, known, 1000)
        med, _, _ = time_calls(torch, glob)
        gp = int(lib.tip_top_triplets_last_passes())
        trip = P * (P - 1) * (P - 2) / 6
        t = {"K": K, "S": S, "N": 1000, "passes": gp, "ms_per_call": med, "triplet_evals_per_s": trip * gp / (med * 1e-3)}
        print(json.dumps(t), flush=True)
        out["top_triplets"].append(t)
        out["baseline"].append(baseline(torch, lib, eng, th, pr, cand, pair_sets[sizes[0]][:8], N, P, sizes))
        del eng
    return out


def baseline(torch, lib, eng, th, pr, cand_np, prs, N, P, sizes):
    """Every partner of each pair through tip_score (first parameter set, S = 1) and a sort of its scores; host clock
    around a synchronised run of all `prs` pairs, extrapolated to the workloads' pair counts."""
    eng.set_params(th[0], pr[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)

    def brute():
        for a, b in prs.tolist():
            c = torch.arange(P, device=dev)
            c = c[(c != a) & (c != b)]
            rr = torch.stack([torch.full_like(c, a), torch.full_like(c, b), c], 1).sort(dim=1).values
            g = cand[rr].to(torch.int32)
            g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
            s = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
            lib.tip_score(P, eng.K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()), ctypes.c_void_p(g3.data_ptr()),
                          g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                          ctypes.c_void_p(s.data_ptr()), eng._stream())
            torch.sort(s, descending=True, stable=True)
    brute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    brute()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    per = sec / len(prs)
    return {"K": eng.K, "S": 1, "pairs_timed": int(len(prs)), "seconds": sec, "seconds_per_pair": per,
            "triplets_per_s": len(prs) * (P - 2) / sec,
            **{"extrapolated_%d_pairs_s" % n: n * per for n in sizes},
            "note": "tip_score over every partner of each pair + a sort, host clock around a synchronised run; the "
                    "per-workload figures are extrapolated from the timed pairs, not measured"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predict_per_pair_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
