"""Time tip_top_triplets (exhaustive top-N of unseen triplets) on one GPU and write profiles/predict_bench.json.

    python tools/predict_bench.py [--out profiles/predict_bench.json] [--quick]

Workloads: P = 6000 genes, N = 1000, the 1e6 Kuzmin-shaped links of bench.py's cfg2 (synth.kuzmin_links_soa) as known
triplets; K = 10 with S = 1 and S = 10 parameter sets, and K = 2..5 (the authors' range) with S = 1.  Parameters are
random (Dirichlet theta rows, p normalised over the rating), seeded.  Per workload: scoring passes, ms per call (CUDA
events, median of 5 calls, each call >= 20 ms), ms per pass (call / passes), triplets per second and achieved fp64 flop/s
(2 S K flop per triplet per pass) and their share of the DMMA peak tip_measure_fma_peak(2) measured in the same run.
Baseline: every triplet scored by tip_score (warp per triplet) in chunks with a running torch.topk, timed at P = 1500
and extrapolated to P = 6000 by the triplet count (labelled as such).  The GPU's name and power limit are read with
read-only nvidia-smi queries."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split("\n")[0]
        name, plim, clk = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": plim, "max_sm_clock": clk}
    except Exception as exc:  # noqa: BLE001
        return {"error": str(exc)}


def params(rng, P, K, S):
    th = np.stack([rng.dirichlet(np.ones(K), size=P) for _ in range(S)])
    pr = rng.random((S, K, K, K, 2))
    return th, pr / pr.sum(axis=4, keepdims=True)


def known_from_cfg2(P, n_links, cand):
    from trigenicinteractionpredictor_b200 import synth
    g1, g2, g3, _ = synth.kuzmin_links_soa(P, n_links, seed=1)
    rank = np.empty(P, dtype=np.int64)
    rank[cand] = np.arange(P)
    r = np.sort(np.stack([rank[g1], rank[g2], rank[g3]], 1), axis=1)
    return np.unique((r[:, 0] << 42) | (r[:, 1] << 21) | r[:, 2]).astype(np.uint64)


def time_calls(torch, fn, reps=5, min_ms=20.0):
    """Median over `reps` timed calls of CUDA-event milliseconds; a call that is shorter than min_ms is repeated inside the
    timed window until it is not, and the time is divided by the repeat count."""
    fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    inner = max(1, int(np.ceil(min_ms / max(e0.elapsed_time(e1), 1e-3))))
    times = []
    for _ in range(reps):
        e0.record()
        for _ in range(inner):
            fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1) / inner)
    return float(np.median(times)), times, inner


def run(args):
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    from trigenicinteractionpredictor_b200.engine import EMEngine
    assert torch.cuda.is_available(), "predict_bench needs a CUDA device"
    lib = _cabi.load()
    P, N, L = (1500, 100, 100_000) if args.quick else (6000, 1000, 1_000_000)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = known_from_cfg2(P, L, cand)
    peak = ctypes.c_double(0)
    _cabi.check(lib.tip_measure_fma_peak(2, ctypes.byref(peak)), "tip_measure_fma_peak")
    total = P * (P - 1) * (P - 2) // 6
    out = {"gpu": gpu_info(), "dmma_peak_tflops": peak.value, "P": P, "N": N, "known_links": L, "known_triplets": int(len(known)),
           "triplets": total, "flop_rule": "2 S K per triplet per pass", "workloads": []}
    rng = np.random.default_rng(2024)
    for K, S in [(10, 1), (10, 10), (2, 1), (3, 1), (4, 1), (5, 1)]:
        th, pr = params(rng, P, K, S)
        eng = EMEngine(P, K, device="cuda:0")
        res = {}

        def call():
            res["r"] = eng.top_triplets(th, pr, cand, known, N)
        med, times, inner = time_calls(torch, call)
        passes = int(lib.tip_top_triplets_last_passes())
        flop = 2.0 * S * K * total * passes
        ids, sc = res["r"]
        w = {"K": K, "S": S, "passes": passes, "ms_per_call": med, "ms_calls": times, "calls_per_window": inner,
             "ms_per_pass": med / passes, "triplets_per_s": total * passes / (med * 1e-3),
             "fp64_tflops": flop / (med * 1e-3) / 1e12, "share_of_dmma_peak": flop / (med * 1e-3) / 1e12 / peak.value,
             "rows": int(len(sc)), "top_score": float(sc[0]), "last_score": float(sc[-1])}
        print(json.dumps(w), flush=True)
        out["workloads"].append(w)
        del eng
    out["baseline"] = baseline(torch, lib, 1500 if not args.quick else 400, 4, N, P)
    return out


def baseline(torch, lib, Pb, K, N, P_target):
    """Every triplet through tip_score in chunks of ~8e6 with a running top-N (torch.topk)."""
    from trigenicinteractionpredictor_b200.engine import EMEngine
    rng = np.random.default_rng(7)
    th, pr = params(rng, Pb, K, 1)
    eng = EMEngine(Pb, K, device="cuda:0")
    eng.set_params(th[0], pr[0])
    dev = eng.device
    cand = torch.from_numpy(np.array(sorted(range(Pb), key=str), dtype=np.int32)).to(dev)

    def brute():
        best = torch.empty(0, dtype=torch.float64, device=dev)
        j = 1
        while j < Pb - 1:
            parts, size = [], 0
            while j < Pb - 1 and size < 8_000_000:
                A, C = torch.meshgrid(torch.arange(j, device=dev), torch.arange(j + 1, Pb, device=dev), indexing="ij")
                parts.append(torch.stack([cand[A.reshape(-1)], torch.full((A.numel(),), int(cand[j]), device=dev,
                                                                           dtype=torch.int32), cand[C.reshape(-1)]], 1))
                size += A.numel()
                j += 1
            g = torch.cat(parts).to(torch.int32)
            g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
            s = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
            lib.tip_score(Pb, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()), ctypes.c_void_p(g3.data_ptr()),
                          g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                          ctypes.c_void_p(s.data_ptr()), eng._stream())
            best = torch.topk(torch.cat([best, torch.topk(s, min(N, s.numel())).values]), N).values
        return best
    brute()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    brute()
    torch.cuda.synchronize()
    sec = time.perf_counter() - t0
    tb = Pb * (Pb - 1) * (Pb - 2) // 6
    tt = P_target * (P_target - 1) * (P_target - 2) // 6
    return {"P": Pb, "K": K, "S": 1, "triplets": tb, "seconds": sec, "triplets_per_s": tb / sec,
            "extrapolated_P": P_target, "extrapolated_seconds": sec * tt / tb,
            "note": "chunked tip_score + torch.topk, host clock around a synchronised run; the P = %d figure is extrapolated "
                    "by the triplet count, not measured" % P_target}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "predict_bench.json"))
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal, not a measurement)")
    args = ap.parse_args()
    res = run(args)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(res, fh, indent=1)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
