"""Time tip_top_pairs and tip_top_pairs_per_gene (the N best unseen gene pairs of the digenic model) on one GPU and write
profiles/predict_pairs_bench.json.

    python tools/predict_pairs_bench.py [--out profiles/predict_pairs_bench.json] [--quick]

Workloads: P = 6000 genes; known pairs: the first two genes of every triplet of the 1e6 Kuzmin-shaped links of bench.py's
cfg2 (as tools/predict_bench.py builds them); K in {3, 10} and S in {1, 10}; the global top-1000, and the per-gene top-20
for 100 random genes and for all 6 000.  Parameters are random (Dirichlet theta rows, qr normalised over the rating),
seeded.  Per workload: ms per call (CUDA events, median of 5 calls, each call >= 20 ms; the call includes the engine's
copies of the parameters), pair scores per second (C(P, 2) for the global call, queries * (P - 1) per gene) and the chunks
swept.  Baseline: tip_score_pairs over every pair for each of the S sets, summed, and a torch.sort of all C(P, 2) sums,
timed the same way.  The GPU's name, power limit and max SM clock are read with read-only nvidia-smi queries."""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from predict_bench import gpu_info, time_calls  # noqa: E402


def known_pairs_from_cfg2(P, n_links, cand):
    from trigenicinteractionpredictor_b200 import synth
    g1, g2, _, _ = synth.kuzmin_links_soa(P, n_links, seed=1)
    rank = np.empty(P, dtype=np.int64)
    rank[cand] = np.arange(P)
    r = np.sort(np.stack([rank[g1], rank[g2]], 1), axis=1)
    r = r[r[:, 0] < r[:, 1]]
    return np.unique((r[:, 0] << 21) | r[:, 1]).astype(np.uint64)


def pair_params(rng, P, K, S):
    th = np.stack([rng.dirichlet(np.ones(K), size=P) for _ in range(S)])
    q = rng.random((S, K, K, 2))
    return th, q / q.sum(axis=3, keepdims=True)


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "predict_pairs_bench needs a CUDA device"
    lib = _cabi.load()
    P, L = (1500, 100_000) if args.quick else (6000, 1_000_000)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = known_pairs_from_cfg2(P, L, cand)
    universe = P * (P - 1) // 2
    out = {"gpu": gpu_info(), "P": P, "known_links": L, "known_pairs": int(len(known)), "pairs": universe,
           "chunk_pairs": 1 << 21, "workloads": [], "baseline": []}
    rng = np.random.default_rng(2026)
    few = np.sort(rng.choice(P, size=100, replace=False)).astype(np.int32)
    ra, rb = np.triu_indices(P, 1)
    for K in (3, 10):
        eng = EMEngine(P, K, device="cuda:0")
        for S in (1, 10):
            th, q = pair_params(rng, P, K, S)
            res = {}

            def glob():
                res["g"] = eng.top_pairs(th, q, cand, known, 1000)
            med, times, inner = time_calls(torch, glob)
            w = {"K": K, "S": S, "mode": "global top-1000", "ms_per_call": med, "ms_calls": times,
                 "calls_per_window": inner, "pairs_per_s": universe / (med * 1e-3),
                 "chunks": int(lib.tip_top_pairs_last_chunks()), "rows": int(len(res["g"][1])),
                 "top_score": float(res["g"][1][0])}
            print(json.dumps(w), flush=True)
            out["workloads"].append(w)
            for label, qr in (("per-gene top-20, 100 random genes", few),
                              ("per-gene top-20, all genes", np.arange(P, dtype=np.int32))):
                def per():
                    res["q"] = eng.top_pairs_per_gene(th, q, cand, qr, known, 20)
                med, times, inner = time_calls(torch, per)
                w = {"K": K, "S": S, "mode": label, "n_query": int(len(qr)), "ms_per_call": med, "ms_calls": times,
                     "calls_per_window": inner, "pairs_per_s": len(qr) * (P - 1) / (med * 1e-3),
                     "chunks": int(lib.tip_top_pairs_per_gene_last_chunks()), "rows": int(res["q"][2].sum())}
                print(json.dumps(w), flush=True)
                out["workloads"].append(w)
            out["baseline"].append(baseline(torch, eng, th, q, cand, ra, rb))
        del eng
    return out


def baseline(torch, eng, th, q, cand, ra, rb):
    """tip_score_pairs over every pair for each set, summed in set order, then a descending torch.sort of the sums."""
    dev = eng.device
    a = torch.from_numpy(cand[ra]).to(dev)
    b = torch.from_numpy(cand[rb]).to(dev)
    d_th = [torch.from_numpy(np.ascontiguousarray(t).reshape(-1)).to(dev) for t in th]
    d_q = [np.ascontiguousarray(x) for x in q]

    def brute():
        acc = None
        for s in range(len(d_th)):
            eng.theta.copy_(d_th[s])
            eng.set_q(d_q[s])
            v = eng.score_pairs(a, b)
            acc = v if acc is None else acc + v
        torch.sort(acc, descending=True)
    med, times, inner = time_calls(torch, brute)
    return {"K": eng.K, "S": len(d_th), "ms_per_call": med, "ms_calls": times, "calls_per_window": inner,
            "pairs_per_s": len(ra) / (med * 1e-3),
            "note": "tip_score_pairs over all C(P, 2) pairs per set, summed, and a torch.sort (known pairs not removed)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predict_pairs_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
