#!/usr/bin/env python3
"""bench.py - EM link-updates/s of the MMSBM hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape kuzmin|uniform]
                    [--skip cfg4,cfg3,fp32,k3,e2e,cpu,dist_check] [--dump-outputs DIR]

A "step" is one EM iteration (Model.make_iteration, TIP.py:984-1043) over one rank's link shard.
Headline workload at every N (weak scaling): BASELINE config 2 per GPU - Kuzmin-2018 trigenic shape, 6,000 genes,
K=10, the fold-1 training split of 1M triplets = 800,000 links per rank; with N>1 the links are sharded over the
ranks (N x 800,000 links in total) and every iteration sums the statistics across ranks (NVLink peer memory fused
into the M-step kernel, or NCCL).  On the same line, each with its own key: the uniform-triple shape of the same
size, BASELINE config 4 (1e8 links in total, STRONG scaling over the N ranks, `cfg4_strong`) and config 3 (50
random-restart samples spread over the N ranks, no communication, `cfg3_samples`).

Prints ONE JSON line on rank 0.  `value` = link-updates/s with inputs resident in HBM; `e2e` = the same through the
host-buffer C-ABI call (H2D of rows/theta/p and D2H of theta/p inside the timed region); `roofline` describes the
dominant kernel (the slot-segmented pass kernel) by SURVEY section 8d's accounting and names what binds it;
`cpu_baseline` is the reference's own Model.make_iteration (oracle/_ref, kind "reference") - or the oracle's
literal-loop port when the reference script did not travel (kind "port") - on this box's host cores.

`--dump-outputs DIR` writes what the last timed step of the headline computed - theta [P,K] and pr [K,K,K,2], the
parameters Model.make_iteration leaves its caller - as DIR/theta.npy and DIR/pr.npy (float64).  The inputs are
seeded, so two builds run with the same arguments can be compared output for output - to rounding, not bit for bit:
the E-step flushes its statistics with fp64 atomic adds, whose order varies from run to run.  Apart from DIR,
bench.py writes nothing into the source tree.
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes
import io
import json
import os
import statistics
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the tree may be read-only; leave no __pycache__ behind in it

P_GENES, K_GROUPS = 6000, 10
L_PER_GPU = 800_000
T_TEST = 200_000
CFG4_LINKS = 100_000_000
CFG3_SAMPLES = 50
METRIC = "EM link-updates/sec at K=10"
UNIT = "link-updates/s"


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """Samples SM clock / throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index: int, period_s: float = 0.002):
        self.index, self.period = index, period_s
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as exc:  # noqa: BLE001
            self.nv, self.err = None, str(exc)

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, nm in names.items():
                    if mask & bit:
                        self.reasons.add(nm)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(self.period)

    def start(self):
        if self.nv is not None:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()

    def stop(self) -> dict:
        if self._thr is not None:
            self._stop.set()
            self._thr.join()
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                    "note": "no NVML samples" if self.nv else "NVML unavailable"}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# --------------------------------------------------------------------------------------------- CPU legs
# One worker process per host core (the stand-in for the reference's `parallel --jobs N` over samples, run.sh:36-45;
# GNU parallel and pypy3 are not in the image).  Each worker holds ONE model on its own sample of links and a "step" is
# one EM iteration of every worker's model at the same time.
_W = {}


def _cpu_init(kind, seed0, n_links, P, K):
    """Pool initializer: build this worker's model.  kind "reference": the unmodified reference script from
    oracle/_ref (Model.get_traintest on files written here, initialize_parameters, then make_iteration per step);
    kind "port": the oracle's literal-loop restatement of the same loops."""
    import random
    import numpy as np
    seed = seed0 + os.getpid() % 9973
    rng = np.random.default_rng(seed)
    # a cfg2-shaped sample: ids drawn from P genes; every gene of the sample has a training link
    ids = rng.integers(0, P, size=(n_links, 3))
    ids[:, 1] = (ids[:, 0] + 1 + rng.integers(0, P - 1, n_links)) % P
    ids[:, 2] = (ids[:, 1] + 1 + rng.integers(0, P - 2, n_links)) % P
    ids[ids[:, 2] == ids[:, 0], 2] = (ids[ids[:, 2] == ids[:, 0], 2] + 1) % P
    lab = (rng.random(n_links) < 0.1).astype(int)
    _W["kind"], _W["n"] = kind, n_links
    if kind == "reference":
        from oracle import fetch_ref
        mod = fetch_ref.load_reference_module()
        tmp = tempfile.mkdtemp(prefix="tipref_")
        seen = {}
        with open(os.path.join(tmp, "train.dat"), "w") as fh:
            for (a, b, c), r in zip(ids.tolist(), lab.tolist()):
                key = tuple(sorted((a, b, c)))
                if len(set(key)) < 3 or key in seen:
                    continue
                seen[key] = 1
                fh.write("G%05d_G%05d_G%05d\t%d\n" % (key[0], key[1], key[2], r))
        with open(os.path.join(tmp, "test.dat"), "w") as fh:
            a, b, c = next(iter(seen))                 # a test link over genes that all have a training link (TIP.py:1018)
            fh.write("G%05d_G%05d_G%05d\t0\n" % (a, b, c))
        m = mod.Model()
        with contextlib.redirect_stdout(io.StringIO()):
            m.get_traintest(os.path.join(tmp, "train.dat"), os.path.join(tmp, "test.dat"))
        random.seed(seed)
        m.initialize_parameters(K)
        _W["model"], _W["n"] = m, len(m.links)
    else:
        from oracle import mmsbm_oracle as orc
        cnt = np.stack([1 - lab, lab], axis=1)
        used = np.unique(ids)
        remap = -np.ones(P, dtype=int)
        remap[used] = np.arange(len(used))
        theta = rng.dirichlet(np.ones(K), size=len(used)).tolist()
        pr = rng.random((K, K, K, 2))
        pr = (pr / pr.sum(axis=3, keepdims=True)).tolist()
        _W["orc"], _W["theta"], _W["pr"] = orc, theta, pr
        _W["ids"], _W["cnt"] = remap[ids].tolist(), cnt.tolist()


def _cpu_step(_):
    t0 = time.perf_counter()
    if _W["kind"] == "reference":
        _W["model"].make_iteration()
    else:
        _W["theta"], _W["pr"] = _W["orc"].em_step_loops(_W["theta"], _W["pr"], _W["ids"], _W["cnt"])[:2]
    return _W["n"], time.perf_counter() - t0


class CpuArm:
    """All host cores, one model per core.  step() = one EM iteration on every core; returns (links, seconds)."""

    def __init__(self, links_per_core, P, K, kind=None):
        import multiprocessing as mp
        from oracle import fetch_ref
        if kind is None:
            kind = "reference" if fetch_ref.load_reference_module() is not None else "port"
        self.kind, self.cores, self.links_per_core = kind, os.cpu_count() or 1, links_per_core
        self.pool = mp.get_context("spawn").Pool(self.cores, initializer=_cpu_init, initargs=(kind, 1000, links_per_core, P, K))

    def step(self):
        t0 = time.perf_counter()
        res = self.pool.map(_cpu_step, range(self.cores), chunksize=1)
        return sum(n for n, _ in res), time.perf_counter() - t0

    def close(self):
        self.pool.close()
        self.pool.join()

    def describe(self, secs):
        what = ("the unmodified reference TrigenicInteractionPredictor.py (oracle/_ref), Model.make_iteration" if self.kind == "reference"
                else "CPython literal-loop oracle port of Model.make_iteration (oracle/_ref absent)")
        return "%d cores x ~%d links per step, one model per core: %s, K=%d, P=%d (%.1f s); cost is linear in links" % (
            self.cores, self.links_per_core, what, K_GROUPS, P_GENES, secs)


def c_port_rate(n_links: int, P: int, K: int):
    """The literal-order C oracle with OpenMP on all cores (context only)."""
    import numpy as np
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(5)
    ids = rng.integers(0, P, size=(n_links, 3))
    lab = (rng.random(n_links) < 0.1).astype(np.int64)
    cnt = np.stack([1 - lab, lab], axis=1)
    theta = rng.dirichlet(np.ones(K), size=P)
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    cores = os.cpu_count() or 1
    orc.em_stats_c_mt(theta, pr, ids[:1000], cnt[:1000], cores)
    t0 = time.perf_counter()
    orc.em_stats_c_mt(theta, pr, ids, cnt, cores)
    return n_links / (time.perf_counter() - t0), cores


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on every host core - the unmodified
    TIP.py from oracle/_ref when it travelled with the tree (kind "reference"), else the oracle's port (kind "port").
    Same warm-up and step counts as asked; the links per core are sized so that the whole run stays within minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    warm, steps = max(args.warmup, 0), max(args.steps, 1)
    probe = CpuArm(100, P_GENES, K_GROUPS)
    probe.step()
    n, secs = probe.step()
    probe.close()
    per_core_rate = n / probe.cores / secs
    budget_s = 150.0
    links_per_core = int(max(60, min(1500, budget_s * per_core_rate / (warm + steps))))
    arm = CpuArm(links_per_core, P_GENES, K_GROUPS, kind=probe.kind)
    for _ in range(warm):
        arm.step()
    links, t_all = 0, 0.0
    for _ in range(steps):
        n, secs = arm.step()
        links += n
        t_all += secs
    arm.close()
    value = links / t_all
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warm, "ms_per_step": 1e3 * t_all / steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cfg2 shape (6000 genes, K=10): bounded sample of %d links per step" % (links // steps)},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(t_all),
                         "pypy3": "unavailable in image"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# --------------------------------------------------------------------------------------------- GPU arm
def _links(synth, shape, P, L, seed, dev):
    import torch
    if shape == "kuzmin":
        g1, g2, g3, lab = synth.kuzmin_links_soa(P, L, seed=seed, device=dev)
    else:
        g1, g2, g3, lab = synth.planted_links_soa(P, L, seed=seed, device=dev)
    g1[:P] = torch.arange(P, dtype=torch.int32, device=dev)            # every gene has a training link
    return g1, g2, g3, 1 - lab, lab


def _timed_replays(torch, eng, steps, warmup, flush_l2, dev):
    """ms of each of `steps` graph replays (CUDA events on the launching stream), L2 flushed before every one."""
    for _ in range(warmup):
        flush_l2()
        eng.graph_step()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    torch.cuda.synchronize(dev)
    for i in range(steps):
        flush_l2()
        ev0[i].record()
        eng.graph_step()
        ev1[i].record()
    torch.cuda.synchronize(dev)
    return [a.elapsed_time(b) for a, b in zip(ev0, ev1)]


def run_ours(args):
    import numpy as np
    import torch
    from trigenicinteractionpredictor_b200 import _cabi, synth
    from trigenicinteractionpredictor_b200 import dist as tdist
    from trigenicinteractionpredictor_b200.engine import EMEngine

    rank, world, local = tdist.init_from_env()
    if not torch.cuda.is_available():
        raise _cabi.TipLibraryError("bench.py needs a CUDA device (no CPU path exists)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    lib = _cabi.load()
    P, K = P_GENES, K_GROUPS
    skip = set(x for x in args.skip.split(",") if x)
    steps, warmup = args.steps, max(args.warmup, 3)
    L_local, L_total = L_PER_GPU, L_PER_GPU * world
    shape_txt = {"kuzmin": "Kuzmin-2018 trigenic shape ((query pair) x array gene, 77 hub genes of degree ~20,000)",
                 "uniform": "uniform random triples"}
    workload = ("cfg2: 6000 genes x 1M triplets, K=10, %s, fold-1 train split = 800,000 links per GPU" % shape_txt[args.shape]
                + ("" if world == 1 else "; %d link shards, statistics summed across ranks every iteration (%s)" % (
                    world, {"peer": "pushed into the peers' inboxes over NVLink peer memory, one handshake, local sum + M-step in one kernel",
                            "peer_rs": "reduce-scatter + M-step + all-gather in one kernel over NVLink peer memory",
                            "peer_gather": "every rank reads every peer buffer, fused into the M-step kernel",
                            "nccl": "NCCL allreduce"}[args.exchange])))

    group = torch.distributed.group.WORLD if world > 1 else None
    rng = np.random.default_rng(0)
    theta0 = rng.dirichlet(np.ones(K), size=P)
    pr0 = rng.random((K, K, K, 2))
    pr0 /= pr0.sum(axis=3, keepdims=True)
    flush = torch.empty(512 * 1024 * 1024, dtype=torch.uint8, device=dev)    # 4x the 126 MB L2

    def flush_l2():
        flush.zero_()

    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    # ------------------------------------------------------------------ headline: cfg2 per GPU, default E-step
    eng = EMEngine(P, K, device=dev, group=group, exchange=args.exchange)
    eng.set_train_links(*_links(synth, args.shape, P, L_local, 100 + rank, dev))
    eng.set_params(theta0, pr0)
    eng.capture_graphs()               # one iteration (E-step, statistics exchange, M-step) per CUDA graph
    launches_per_step = eng._graph_launches
    eng.set_params(theta0, pr0)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(warmup):
        flush_l2()
        eng.graph_step()
    tdist.barrier(group)
    torch.cuda.synchronize(dev)
    ms = _timed_replays(torch, eng, steps, 0, flush_l2, dev)
    tdist.barrier(group)
    total_ms = tdist.max_over_ranks(sum(ms), device=dev, group=group)
    ms_per_step = total_ms / steps
    value = L_total / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # taken here, before the informational replays below move the parameters on
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "theta.npy"), eng.theta.reshape(P, K).cpu().numpy())
        np.save(os.path.join(args.dump_outputs, "pr.npy"), eng.p.reshape(K, K, K, 2).cpu().numpy())

    # back-to-back replays, rows resident in L2 (how a real training run behaves) - informational
    torch.cuda.synchronize(dev)
    a.record()
    for _ in range(steps):
        eng.graph_step()
    b.record()
    torch.cuda.synchronize(dev)
    warm_ms = tdist.max_over_ranks(a.elapsed_time(b) / steps, device=dev, group=group)
    clocks = sampler.stop()

    # the kernels of one E-step, each timed with CUDA events on the launching stream (un-graphed, L2 flushed)
    seg3 = bool(eng.flags & _cabi.TIP_EM_SLOT_SEGMENTED)
    stage_ms = None
    if seg3:
        lib.tip_seg3_timing(1)
        acc = []
        buf = (ctypes.c_float * 5)()
        for _ in range(max(5, min(steps, 20))):
            flush_l2()
            eng.em_step()
            _cabi.check(lib.tip_seg3_last_timing(buf), "tip_seg3_last_timing")
            acc.append(list(buf))
        lib.tip_seg3_timing(0)
        stage_ms = [statistics.mean(x[i] for x in acc) for i in range(5)]
    n_rows = eng.train.n_rows

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps,
        "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload, "P": P, "K": K, "links_per_gpu": L_local, "links_total": L_total, "shape": args.shape,
                   "estep": "slot-segmented (TIP_EM_SLOT_SEGMENTED%s)" % (" | TIP_EM_GATHER_L1" if eng.flags & _cabi.TIP_EM_GATHER_L1 else "")
                   if seg3 else "flags %d" % eng.flags,
                   "l2": "flushed (512 MB memset) before every timed step", "cuda_graph": True},
        "value_l2_warm": L_total / (warm_ms * 1e-3),
        "gpu_launches": launches_per_step * steps,
        "clocks": clocks,
    }

    # replicas of theta / p must be bit-identical on every rank after the timed iterations
    if world > 1:
        chk = torch.stack([eng.theta.view(torch.int64).sum(), eng.p.view(torch.int64).sum()])
        allc = [torch.empty_like(chk) for _ in range(world)]
        torch.distributed.all_gather(allc, chk, group=group)
        line["replicas_bit_identical"] = bool(all(torch.equal(c, allc[0]) for c in allc))
        eng._check_peer()

    # ------------------------------------------------------------------ roofline of the dominant kernel
    if rank == 0:
        peak_dfma, peak_dmma, peak32 = _measure_peak(lib, 0), _measure_peak(lib, 2), _measure_peak(lib, 1)
        gath = ctypes.c_double(0.0)
        _cabi.check(lib.tip_measure_l2_gather(P, 8 * K, ctypes.byref(gath)), "tip_measure_l2_gather")
        peaks = _read_peaks()
        if seg3:
            k_ms = stage_ms[2] + stage_ms[3]
            flops = 6.0 * K ** 3 * L_local
            achieved = flops / (k_ms * 1e-3) / 1e12
            sect = (8 * K + 31) // 32 * 32
            l2_bytes = L_local * (6 * sect + 3 * 16 + 3 * 8)       # six theta rows, three row reads, s written once + read twice
            prof = _read_profile("r2_seg3_pass_metrics.json")
            line["roofline"] = {
                "bound": "fp64_fma", "achieved": achieved, "peak": peak_dmma, "unit": "TFLOP/s", "frac": achieved / peak_dmma,
                "traffic": prof.get("traffic_bytes"), "traffic_source": prof.get("source", "no ncu capture in the tree"),
                "kernel": "seg3_pass_kernel<10,...>: pass A + pass B/C launches (one E-step walks every link in three orders)",
                "kernel_ms": k_ms, "kernel_share_of_step": k_ms / ms_per_step if world == 1 else None,
                "kernel_share_of_serialised_estep": k_ms / sum(stage_ms),
                "share_note": "kernel_ms and estep_stage_ms are timed with the two pass launches SERIALISED (events between them); in "
                              "the graph-replayed step pass B + C starts while pass A drains, so kernel_ms / ms_per_step overstates "
                              "the share; the serialised share is the one to hold against the ncu launch list",
                "estep_stage_ms": dict(zip(["memset", "prep", "pass_a", "pass_bc", "finish"], stage_ms)),
                "flops_per_link_update": 6 * K ** 3,
                "accounting": "SURVEY 8d: achieved = 6 K^3 flop x links / duration of the kernel.  The kernel EXECUTES 8 K^2 flop "
                              "per link on the fp64 tensor path (DMMA) plus 4 K^3 per (gene, rating) in the prep / finish kernels: the "
                              "factorisation removes the K^3-per-link contraction, so the algorithmic rate is not a pipe utilisation",
                "peak_source": "tip_measure_fma_peak(kind 2: mma.sync m8n8k4 f64) measured in this run; DFMA chains read %.2f" % peak_dfma,
                "executed_tflops": 8.0 * K * K * L_local / (k_ms * 1e-3) / 1e12,
                "binding": {"resource": "L2 gather latency (six theta rows per link from L2; warps wait on the gathers)",
                            "l2_bytes_per_link": l2_bytes / L_local, "achieved_gbs": l2_bytes / (k_ms * 1e-3) / 1e9,
                            "peak_gbs": gath.value, "frac": l2_bytes / (k_ms * 1e-3) / 1e9 / gath.value,
                            "peak_source": "tip_measure_l2_gather: random %d-byte rows of a %d-row table, 16-byte L2-only loads, measured in this run" % (8 * K, P)},
                "ncu": {k: prof.get(k) for k in ("lts_t_bytes", "issue_active_pct", "fp64_pipe_pct", "stall_mix") if k in prof},
                "fp32_fma_peak": peak32,
                "hbm": {"algorithmic_bytes": 16 * n_rows, "achieved_gbs": 16 * n_rows * 3 / (k_ms * 1e-3) / 1e9,
                        "peak_gbs": peaks.get("hbm_gbs"), "peak_source": "MEASURED_PEAKS.json" if peaks else "absent",
                        "note": "three orders of the rows are streamed per E-step: 48 B per link"},
            }
        else:
            line["roofline"] = None
    else:
        line["roofline"] = None
        peak_dfma = peak32 = None

    # ------------------------------------------------------------------ the other shape at the same size
    other = "uniform" if args.shape == "kuzmin" else "kuzmin"
    if world == 1:
        eo = EMEngine(P, K, device=dev)
        eo.set_train_links(*_links(synth, other, P, L_local, 100 + rank, dev))
        eo.set_params(theta0, pr0)
        eo.capture_graphs()
        eo.set_params(theta0, pr0)
        mo = _timed_replays(torch, eo, steps, 3, flush_l2, dev)
        line["value_" + other] = L_total / (statistics.mean(mo) * 1e-3)
        line["value_" + args.shape] = value
        line["shape_ratio_kuzmin_over_uniform"] = (line["value_kuzmin"] / line["value_uniform"])
    else:
        eo = None

    # ------------------------------------------------------------------ the K^3-per-link kernel and the 1e-5 mode
    if world == 1 and "k3" not in skip:
        ek = EMEngine(P, K, device=dev, flags=_cabi.TIP_EM_DEFAULT)
        ek.set_train_links(*_links(synth, "uniform", P, L_local, 100 + rank, dev))
        ek.set_params(theta0, pr0)
        ek.capture_graphs()
        ek.set_params(theta0, pr0)
        mk = statistics.mean(_timed_replays(torch, ek, steps, 3, flush_l2, dev))
        line["k3_per_link_kernel"] = {
            "value": L_total / (mk * 1e-3), "ms_per_step": mk, "shape": "uniform",
            "roofline_frac_dfma": (6.0 * K ** 3 * L_local / (mk * 1e-3) / 1e12) / peak_dfma,
            "note": "em_fused_kernel<10>: 2 K^3 DFMA per link in registers (TIP_EM_DEFAULT); executes what it is charged for"}
        if "fp32" not in skip:
            e32 = EMEngine(P, K, device=dev, flags=_cabi.TIP_EM_FP32_COMPUTE)
            e32.train, e32.em_ws, e32.em_ws_bytes = ek.train, ek.em_ws, ek.em_ws_bytes
            e32.set_params(theta0, pr0)
            e32.capture_graphs()
            e32.set_params(theta0, pr0)
            m32 = statistics.mean(_timed_replays(torch, e32, steps, 3, flush_l2, dev))
            line["value_fp32_compute"] = L_total / (m32 * 1e-3)
            line["fp32_compute_roofline_frac"] = (6.0 * K ** 3 * L_local / (m32 * 1e-3) / 1e12) / peak32
            del e32
        del ek

    # ------------------------------------------------------------------ end to end through host buffers
    if "e2e" not in skip:
        line["e2e"] = _e2e(eng, lib, dev, group, world, theta0, pr0, L_total, args, tdist)
        if eo is not None:
            oth = _e2e(eo, lib, dev, group, world, theta0, pr0, L_total, args, tdist)
            line["e2e"]["other_shape"] = {"shape": other, "value": oth["value"], "ms_per_step": oth["ms_per_step"], "variants": oth["variants"]}
    del eng, eo
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ link-shard correctness gate (N > 1)
    if world > 1 and "dist_check" not in skip:
        line["dist_check"] = _dist_check(rank, world, dev, group, args.exchange, tdist)

    # ------------------------------------------------------------------ cfg4: 1e8 links, strong scaling
    if "cfg4" not in skip:
        line["cfg4_strong"] = _cfg4(rank, world, dev, group, args, theta0, pr0, flush_l2, synth, tdist)
    # ------------------------------------------------------------------ cfg3: 50 restarts, sample-parallel
    if "cfg3" not in skip:
        line["cfg3_samples"] = _cfg3(rank, world, dev, group, synth, tdist)

    if rank == 0:
        if world == 1 and "cpu" not in skip and not args.no_cpu:
            arm = CpuArm(1500, P, K)
            links, secs = 0, 0.0
            for _ in range(3):
                n, s = arm.step()
                links += n
                secs += s
            arm.close()
            crate, ccores = c_port_rate(40000, P, K)
            line["cpu_baseline"] = {
                "value": links / secs, "unit": UNIT, "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(secs),
                "c_port_openmp_value": crate, "c_port_cores": ccores, "pypy3": "unavailable in image"}
        else:
            line["cpu_baseline"] = None
        print(json.dumps(line))
    if world > 1:
        # ProcessGroupNCCL teardown (destroy_process_group / interpreter exit) was seen to hang on the
        # GPU boxes after all work had completed; leave without running it
        tdist.barrier(group)
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)
    return 0


def _dist_check(rank, world, dev, group, exchange, tdist):
    """A small problem, link-sharded over all ranks for 6 iterations (graph replays and eager iterations mixed), against
    the same iterations on rank 0 alone: theta / p within 1e-10, replicas bit-identical."""
    import numpy as np
    import torch
    from trigenicinteractionpredictor_b200.engine import EMEngine
    rng = np.random.default_rng(3)
    P, L, K = 500, 20000, 10
    g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
    g[:P, 0] = np.arange(P)
    lab = (rng.random(L) < 0.2).astype(np.int32)
    # every rank draws DIFFERENT initial parameters: set_params must make rank 0's win everywhere
    rr = np.random.default_rng(100 + rank)
    theta = rr.dirichlet(np.ones(K), size=P)
    pr = rr.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    lo, hi = tdist.shard_bounds(L, rank, world)
    eng = EMEngine(P, K, device=dev, group=group, exchange=exchange)
    eng.set_train_links(g[lo:hi, 0], g[lo:hi, 1], g[lo:hi, 2], 1 - lab[lo:hi], lab[lo:hi])
    eng.set_params(theta, pr)
    eng.em_iterations(4)
    eng.em_iteration()
    eng.em_iterations(1)
    th, p = eng.get_params()
    chk = torch.from_numpy(np.concatenate([th.ravel(), p.ravel()])).to(dev)
    allc = [torch.empty_like(chk) for _ in range(world)]
    torch.distributed.all_gather(allc, chk, group=group)
    same = all(torch.equal(c, allc[0]) for c in allc)
    err = None
    if rank == 0:
        r0 = np.random.default_rng(100)
        theta = r0.dirichlet(np.ones(K), size=P)
        pr = r0.random((K, K, K, 2))
        pr /= pr.sum(axis=3, keepdims=True)
        one = EMEngine(P, K, device=dev)
        one.set_train_links(g[:, 0], g[:, 1], g[:, 2], 1 - lab, lab)
        one.set_params(theta, pr)
        for _ in range(6):
            one.em_iteration()
        th1, p1 = one.get_params()
        err = max(float(np.max(np.abs(th - th1) / np.maximum(np.abs(th1), 1e-300))),
                  float(np.max(np.abs(p - p1) / np.maximum(np.abs(p1), 1e-300))))
    ok = same and (err is None or err < 1e-10)
    return {"status": "ok" if ok else "FAILED", "replicas_bit_identical": bool(same), "max_rel_err_vs_single_rank": err,
            "what": "P=500, 20,000 links over %d ranks, 6 iterations (4 graph replays, 1 eager, 1 replay), ranks seeded "
                    "differently; rank 0 recomputes alone" % world}


def _cfg4(rank, world, dev, group, args, theta0, pr0, flush_l2, synth, tdist):
    """BASELINE config 4: 6,000 genes x 1e8 triplets, K=10, link-sharded over the ranks (strong scaling)."""
    import torch
    from trigenicinteractionpredictor_b200.engine import EMEngine
    lo, hi = tdist.shard_bounds(CFG4_LINKS, rank, world)
    L = hi - lo
    eng = EMEngine(P_GENES, K_GROUPS, device=dev, group=group, exchange=args.exchange)
    eng.set_train_links(*_links(synth, "uniform", P_GENES, L, 4000 + rank, dev))
    torch.cuda.empty_cache()
    eng.set_params(theta0, pr0)
    eng.capture_graphs()
    eng.set_params(theta0, pr0)
    n = max(5, min(args.steps, 10))
    for _ in range(3):
        eng.graph_step()
    tdist.barrier(group)
    ms = _timed_replays(torch, eng, n, 0, flush_l2, dev)
    tdist.barrier(group)
    per = tdist.max_over_ranks(sum(ms), device=dev, group=group) / n
    eng._check_peer()
    out = {"value": CFG4_LINKS / (per * 1e-3), "unit": UNIT, "ms_per_step": per, "links_per_gpu": L, "links_total": CFG4_LINKS,
           "steps": n, "scaling": "strong", "shape": "uniform",
           "roofline_frac_6k3_over_dmma_peak": None}
    del eng
    torch.cuda.empty_cache()
    return out


def _cfg3(rank, world, dev, group, synth, tdist):
    """BASELINE config 3: 50 random restarts of cfg2 (800,000 training / 200,000 test triplets, K=10), restarts spread
    round-robin over the ranks with no communication (run.sh:36-45); each restart is the reference's sample loop
    (TIP.py:1253-1279: initialise from random.seed(1000 + s), iterate, likelihood check every 25 iterations after 100,
    stop at |dL/L| < 0.01, then held-out likelihood, scores and metrics) through the drop-in Model."""
    import random
    import torch
    from trigenicinteractionpredictor_b200 import TrigenicInteractionPredictor as tip
    g1, g2, g3, n0, n1 = _links(synth, "kuzmin", P_GENES, L_PER_GPU + T_TEST, 100, dev)
    tr = tuple(x[:L_PER_GPU].contiguous() for x in (g1, g2, g3, n0, n1))
    te = tuple(x[L_PER_GPU:].contiguous() for x in (g1, g2, g3, n0, n1))
    model = tip.Model(device=dev)
    model.set_links_soa(tr, te, P=P_GENES)
    mine = tdist.samples_for_rank(0, CFG3_SAMPLES, rank, world)
    random.seed(999)
    tip.train_sample(model, K_GROUPS, 130, 25, 100, verbose=False)        # warm-up restart: graphs, allocations
    tdist.barrier(group)
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    conv, iters, aucs = 0, 0, []
    for s in mine:
        random.seed(1000 + s)
        ok, it, _ = tip.train_sample(model, K_GROUPS, 10000, 25, 100, verbose=False)
        model.compute_likelihood('test')
        model.calculate_test_set_results()
        aucs.append(model.calculate_metrics()[3])
        conv += int(ok)
        iters += it
    torch.cuda.synchronize(dev)
    dt = tdist.max_over_ranks(time.perf_counter() - t0, device=dev, group=group)
    tot = torch.tensor([conv, iters, len(mine)], dtype=torch.int64, device=dev)
    if world > 1:
        torch.distributed.all_reduce(tot, group=group)
    conv, iters, n = (int(x) for x in tot.tolist())
    return {"samples_per_s": n / dt, "samples": n, "converged": conv, "seconds": dt, "em_iterations_total": iters,
            "link_updates_per_s": iters * L_PER_GPU / dt, "samples_on_rank0": len(mine), "auc_rank0_first": aucs[0] if aucs else None,
            "what": "50 restarts x (init on the host RNG, EM to convergence, held-out likelihood, scores, metrics); wall clock, max over ranks"}


def _measure_peak(lib, kind):
    out = ctypes.c_double(0.0)
    rc = lib.tip_measure_fma_peak(kind, ctypes.byref(out))
    if rc != 0:
        raise RuntimeError("tip_measure_fma_peak failed: %s" % lib.tip_last_error())
    return out.value


def _read_profile(name):
    """Per-launch figures of the dominant kernel from the committed ncu capture (profiles/<name>, written by
    tools/ncu_metrics_json.py); `traffic` in the roofline is FROM THIS FILE, not measured in the run."""
    try:
        with open(os.path.join(ROOT, "profiles", name)) as fh:
            m = json.load(fh)
        m["source"] = "profiles/" + name + " (ncu --set full capture, not measured in this run)"
        return m
    except Exception:  # noqa: BLE001
        return {}


def _read_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            return json.load(fh)
    except Exception:  # noqa: BLE001
        return {}


def _e2e(eng, lib, dev, group, world, theta0, pr0, L_total, args, tdist):
    """Same metric with HOST buffers: per step copy rows + deg + theta + p in, run one iteration, copy theta + p out.
    The rows travel in the 8-byte host format (tip_rows_compact_host) and are expanded on the device as they land;
    the 16-byte format is timed beside it (`rows16`)."""
    import numpy as np
    import torch
    from trigenicinteractionpredictor_b200 import _cabi
    P, K = eng.P, eng.K
    n_rows = eng.train.n_rows
    rows_h = eng.train.rows[:n_rows].cpu().pin_memory()
    rows8_h = torch.empty(max(n_rows, 1), dtype=torch.int64).pin_memory()
    rc = lib.tip_rows_compact_host(rows_h.data_ptr(), n_rows, rows8_h.data_ptr())
    if rc != 0:
        raise RuntimeError(lib.tip_last_error())
    deg_h = eng.train.deg.cpu().pin_memory()
    th_h = torch.from_numpy(np.ascontiguousarray(theta0)).pin_memory()
    p_h = torch.from_numpy(np.ascontiguousarray(pr0)).pin_memory()
    fixed = deg_h.numel() * 4 + th_h.numel() * 8 + p_h.numel() * 8
    d2h = th_h.numel() * 8 + p_h.numel() * 8
    steps = args.steps

    def make_step(compact, streamed=True, em_flags=0):
        if world == 1:
            src = rows8_h if compact else rows_h
            fl = (_cabi.TIP_ROWS_COMPACT8 if compact else 0) | em_flags

            def step():
                rc = lib.tip_em_iterations_host(P, K, src.data_ptr(), n_rows, eng.train.n_rows_r0,
                                                deg_h.data_ptr(), th_h.data_ptr(), p_h.data_ptr(), 1, fl)
                if rc != 0:
                    raise RuntimeError(lib.tip_last_error())
            return step
        src = rows8_h if compact else rows_h
        rows8_d = torch.empty(max(n_rows, 1), dtype=torch.int64, device=dev) if (compact and not streamed) else None

        def step():
            # small parameter copies first (the H2D engine is FIFO across streams), then the E-step follows the rows'
            # DMA front (tip_em_step_host_rows), statistics exchange, M-step
            eng.train.deg.copy_(deg_h, non_blocking=True)
            eng.theta.copy_(th_h.view(-1), non_blocking=True)
            eng.p.copy_(p_h.view(-1), non_blocking=True)
            if streamed:
                eng.em_iteration_host_rows(src, compact)
            else:
                # copy, (expand,) then the resident-row iteration
                if compact:
                    rows8_d.copy_(rows8_h, non_blocking=True)
                    rc = lib.tip_rows_expand(rows8_d.data_ptr(), eng.train.rows.data_ptr(), n_rows,
                                             torch.cuda.current_stream(dev).cuda_stream)
                    if rc != 0:
                        raise RuntimeError(lib.tip_last_error())
                else:
                    eng.train.rows.copy_(rows_h, non_blocking=True)
                if eng.flags & _cabi.TIP_EM_SLOT_SEGMENTED:
                    eng.reorder_rows()                # the rows are new every step: orders b, c and the schedules again
                eng.em_iteration()
            th_h.view(-1).copy_(eng.theta, non_blocking=True)
            p_h.view(-1).copy_(eng.p, non_blocking=True)
            torch.cuda.synchronize(dev)
        return step

    def timed(step):
        for _ in range(3):
            step()
        tdist.barrier(group)
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        torch.cuda.synchronize(dev)
        return tdist.max_over_ranks(time.perf_counter() - t0, device=dev, group=group)

    # The streamed E-step has the kernel poll rows that a concurrent copy delivers.  If this box cannot run the copy
    # beside the kernel (the kernel then gives up after 5 s and reports it), the copy-then-compute path of the same
    # library is timed instead - still the GPU path, just without the overlap - and the line says so.
    def run_both(streamed):
        d16, d8 = timed(make_step(False, streamed)), timed(make_step(True, streamed))
        ok = True
        if streamed and world > 1:
            flag = torch.tensor([0 if eng.host_rows_arrived() else 1], dtype=torch.int32, device=dev)
            torch.distributed.all_reduce(flag, group=group)
            ok = int(flag.item()) == 0
        return d16, d8, ok

    streamed = True
    try:
        ok = True
        if world > 1:                                 # one step first: a timed-out step costs 5 s on every rank
            make_step(True, True)()
            flag = torch.tensor([0 if eng.host_rows_arrived() else 1], dtype=torch.int32, device=dev)
            torch.distributed.all_reduce(flag, group=group)
            ok = int(flag.item()) == 0
        if ok:
            dt16, dt, ok = run_both(True)
    except RuntimeError as exc:                       # world == 1: tip_em_iterations_host returned -3
        print("bench: streamed host entry failed (%s)" % exc, file=sys.stderr)
        ok = False
    if not ok:
        streamed = False
        os.environ["TIP_HOST_NO_STREAM"] = "1"        # tip_em_iterations_host reads it on every call
        th_h.copy_(torch.from_numpy(np.ascontiguousarray(theta0)))
        p_h.copy_(torch.from_numpy(np.ascontiguousarray(pr0)))
        dt16, dt, _ = run_both(False)
    alt = None
    if world == 1:
        # the same call with the slot-segmented kernels: rows land, pass A runs while the copy stream sorts them into orders
        # b and c, then passes B + C.  The K^3-per-link kernel can follow the rows' DMA front but scatters with atomics (slow
        # on hub-shaped links); the faster of the two is the headline, the other is listed
        seg_flags = eng.flags & (_cabi.TIP_EM_SLOT_SEGMENTED | _cabi.TIP_EM_GATHER_L1)
        if seg_flags:
            th_h.copy_(torch.from_numpy(np.ascontiguousarray(theta0)))
            p_h.copy_(torch.from_numpy(np.ascontiguousarray(pr0)))
            dts = timed(make_step(True, True, seg_flags))
            alt = {"slot_segmented_after_landing": {"value": L_total * steps / dts, "ms_per_step": 1e3 * dts / steps},
                   "k3_following_the_dma_front": {"value": L_total * steps / dt, "ms_per_step": 1e3 * dt / steps, "streamed": streamed}}
            if dts < dt:
                dt = dts
        api = ("tip_em_iterations_host (C ABI, pinned host buffers, 8-byte rows: TIP_ROWS_COMPACT8), one iteration per call; "
               + ("slot-segmented kernels: the rows land, pass A runs while a second stream sorts them into the orders of slots b "
                  "and c, then passes B + C" if alt and dt == dts else
                  "the K^3-per-link kernel follows the rows' DMA front"))
    else:
        api = ("EMEngine.em_iteration_host_rows: pinned host buffers, 8-byte rows, tip_em_step_host_rows follows the DMA "
               "front (link-sharded, %s exchange)" % args.exchange)
        if streamed and (eng.flags & _cabi.TIP_EM_SLOT_SEGMENTED):
            # the other variant: rows land, are expanded and ordered on the device, then the slot-segmented iteration
            th_h.copy_(torch.from_numpy(np.ascontiguousarray(theta0)))
            p_h.copy_(torch.from_numpy(np.ascontiguousarray(pr0)))
            dts = timed(make_step(True, False))
            alt = {"slot_segmented_after_landing": {"value": L_total * steps / dts, "ms_per_step": 1e3 * dts / steps},
                   "k3_following_the_dma_front": {"value": L_total * steps / dt, "ms_per_step": 1e3 * dt / steps, "streamed": True}}
            if dts < dt:
                dt = dts
                api = ("pinned host buffers, 8-byte rows: copy, tip_rows_expand, tip_order_rows, then the slot-segmented iteration "
                       "(link-sharded, %s exchange)" % args.exchange)
    if not streamed:
        api += " - NOT streamed on this box (the streamed step gave up waiting for its rows): copy, then compute"
    # bytes are whole-job like `value`: every rank copies its own shard's rows plus the replicated parameters
    return {"value": L_total * steps / dt, "unit": UNIT, "streamed": streamed,
            "h2d_bytes_per_step": int(n_rows * 8 + fixed) * world, "d2h_bytes_per_step": int(d2h) * world,
            "bytes_are": "summed over the %d rank(s)" % world, "ms_per_step": 1e3 * dt / steps, "api": api, "variants": alt,
            "rows16": {"value": L_total * steps / dt16, "ms_per_step": 1e3 * dt16 / steps,
                       "h2d_bytes_per_step": int(n_rows * 16 + fixed) * world}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--shape", choices=["kuzmin", "uniform"], default="kuzmin",
                    help="link shape of the headline workload (BASELINE config 2 names the Kuzmin-2018 shape)")
    ap.add_argument("--skip", default="", help="comma list of legs to leave out: cfg4,cfg3,fp32,k3,e2e,cpu,dist_check")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--exchange", choices=["peer", "peer_rs", "peer_gather", "nccl"], default="peer",
                    help="N>1: how link-shard statistics are summed over NVLink peer memory: peer = statistics pushed into the "
                         "peers' inboxes, one handshake, local sum + M-step in one kernel; peer_rs = reduce-scatter + M-step + "
                         "all-gather in one kernel; peer_gather = every rank reads every buffer (round 1); nccl = NCCL allreduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write theta and pr after the last timed step of the headline as DIR/theta.npy, DIR/pr.npy (float64)")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes what the GPU path computed; it does not apply to --impl reference")
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
