"""Device-side state of one MMSBM model: packed link rows, theta, p, statistics - and the calls into
libtip.so that advance it.  PyTorch owns the memory and the streams; every number is produced by the
CUDA kernels behind the C ABI (include/tip.h).  There is no CPU path.

    eng = EMEngine(P, K, device)                       # optionally group=torch.distributed group
    eng.set_train_links(g1, g2, g3, n0, n1)            # this rank's link shard (ids in key slot order)
    eng.set_params(theta, p)                           # numpy fp64, reference layouts
    eng.em_iterations(n)                               # n x make_iteration (TIP.py:984-1043)
    eng.loglik("train")                                # compute_likelihood (TIP.py:952-974)
    eng.top_triplets(thetas, ps, cand, known, n)       # exhaustive top-n of unseen triplets (tip_top_triplets)
"""
from __future__ import annotations

import ctypes
import functools
import os

import numpy as np
import torch

from . import _cabi
from . import dist as _dist

# libtip.so keeps per-process caches that belong to ONE device (SM count, function attributes, the constant-bank
# staging buffer, events, the host-entry scratch): one CUDA device per process, the first engine decides which.
_PROCESS_DEVICE = None


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def _on_device(fn):
    """Run a method with the engine's device current: libtip launches on the CURRENT device (a default-stream handle
    of 0 carries no device), so every call into it must be made with `self.device` selected."""
    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


class PackedLinks:
    """Packed rows of one link set on the device (see include/tip.h)."""

    def __init__(self, rows, n_rows, n_rows_r0, n_real, deg):
        self.rows, self.n_rows, self.n_rows_r0, self.n_real, self.deg = rows, n_rows, n_rows_r0, n_real, deg
        self.rows3 = None     # slot-a | slot-b | slot-c orders back to back (tip_order_rows); rows is then its first third
        self.rows3_buf = None  # the buffer behind rows3: the three orders, then the tile schedules
        self.order_ws = None   # tip_order_rows workspace, kept for reorder_rows


def default_flags(K: int) -> int:
    """E-step formulation used when the caller does not choose one: the slot-segmented kernels (4K^2 FMA per
    link, no per-link atomics, indifferent to hub genes) wherever they are the fastest correct path."""
    # K sweep at 1e7 links (profiles/r2_k_sweep_10M.jsonl): K = 4: 0.67 vs 1.12 ms, K = 3: 0.96 vs 0.54 ms (K^3 per link wins)
    return _cabi.TIP_EM_SLOT_SEGMENTED if K >= 4 else _cabi.TIP_EM_DEFAULT


class EMEngine:
    def __init__(self, P: int, K: int, device=None, group=None, flags: int | None = None,
                 exchange: str = "peer"):
        if not torch.cuda.is_available():
            raise _cabi.TipLibraryError("no CUDA device: trigenicinteractionpredictor_b200 has no CPU path")
        self.lib = _cabi.load()
        self.P, self.K = int(P), int(K)
        self.device = torch.device(device if device is not None else "cuda:%d" % torch.cuda.current_device())
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        global _PROCESS_DEVICE
        if _PROCESS_DEVICE is None:
            _PROCESS_DEVICE = self.device.index
        elif _PROCESS_DEVICE != self.device.index:
            raise _cabi.TipLibraryError(
                "libtip.so holds per-process state of cuda:%d; a second device (cuda:%d) in the same process is not "
                "supported - run one process per GPU (torchrun / --dist)" % (_PROCESS_DEVICE, self.device.index))
        self.group = group
        self._auto_flags = flags is None
        self.flags = default_flags(int(K)) if flags is None else int(flags)
        # group=None means "this process alone" (NOT torch.distributed's default group): link shards are opt-in
        self.world = _dist.world_size(group) if group is not None else 1
        self.n_stats = int(self.lib.tip_stats_len(self.P, self.K))
        with torch.cuda.device(self.device):
            self.theta = torch.empty(self.P * self.K, dtype=torch.float64, device=self.device)
            self.p = torch.empty(2 * self.K ** 3, dtype=torch.float64, device=self.device)
            self.stats = torch.zeros(self.n_stats, dtype=torch.float64, device=self.device)
            self.ll_out = torch.zeros(1, dtype=torch.float64, device=self.device)
            self.ll_ws = torch.empty(int(self.lib.tip_loglik_workspace_bytes(self.P, self.K)), dtype=torch.uint8,
                                     device=self.device)
        # link shards: how the statistics are summed across ranks - "peer" (NVLink peer memory, fused into the
        # M-step kernel) or "nccl" (torch.distributed allreduce)
        self.peer = None
        self._iter = 0
        if self.world > 1 and exchange in ("peer", "peer_rs", "peer_gather"):
            with torch.cuda.device(self.device):
                self.peer = _dist.PeerExchange(self.n_stats, self.device, group, n_theta=self.P * self.K, n_p=2 * self.K ** 3,
                                               mode={"peer": "push", "peer_rs": "rs", "peer_gather": "gather"}[exchange])
                if self.peer.mode == "rs":
                    # the peers write this rank's slice of the new parameters: theta and p live in the shared buffer
                    self.theta, self.p = self.peer.theta(), self.peer.p()
        self.train: PackedLinks | None = None
        self.test: PackedLinks | None = None
        self.test_ids = None      # (g1, g2, g3, labels) int32 tensors in test order
        self.em_ws = None
        self.pairs = None         # digenic extension: int32 [n][4] rows {a, b, n0, n1}
        self.q = None             # its rating tensor q[K][K][2] and the statistic Sq[2][K*K]
        self.sq = None
        self._graphs = None
        self._graph_key = None
        self.launches = 0         # kernel launches issued by libtip on behalf of this engine

    # ------------------------------------------------------------------ link sets
    def _as_dev_i32(self, a):
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=torch.int32).contiguous()
        return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(self.device)

    @_on_device
    def pack(self, g1, g2, g3, n0, n1, want_deg=True) -> PackedLinks:
        """tip_pack_rows: SoA -> rows ordered (rating, slot-a gene) in 32-row single-rating tiles."""
        g1, g2, g3, n0, n1 = (self._as_dev_i32(x) for x in (g1, g2, g3, n0, n1))
        L = int(g1.numel())
        with torch.cuda.device(self.device):
            nb = ctypes.c_size_t(0)
            _cabi.check(self.lib.tip_pack_rows_workspace_bytes(L, ctypes.byref(nb)), "tip_pack_rows_workspace_bytes")
            ws = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
            rows = torch.empty((int(self.lib.tip_rows_capacity(L)), 4), dtype=torch.int32, device=self.device)
            deg = torch.zeros(self.P, dtype=torch.int32, device=self.device) if want_deg else None
            n_rows = ctypes.c_int64(0)
            part = (ctypes.c_int64 * 3)()
            st = torch.cuda.current_stream(self.device).cuda_stream
            _cabi.check(self.lib.tip_pack_rows(_ptr(g1), _ptr(g2), _ptr(g3), _ptr(n0), _ptr(n1), L, self.P, _ptr(ws),
                                               nb.value, _ptr(rows), ctypes.byref(n_rows), part, _ptr(deg),
                                               ctypes.c_void_p(st)), "tip_pack_rows")
            self.launches += 3
            rows = rows[: n_rows.value].clone() if n_rows.value < rows.shape[0] else rows
        return PackedLinks(rows, int(n_rows.value), int(part[0]), int(part[2]), deg)

    @_on_device
    def order_rows(self, links: PackedLinks):
        """tip_order_rows: append the slot-b and slot-c orders of the packed rows (TIP_EM_SLOT_SEGMENTED)."""
        n = links.n_rows
        with torch.cuda.device(self.device):
            nb = ctypes.c_size_t(0)
            _cabi.check(self.lib.tip_order_rows_workspace_bytes(n, ctypes.byref(nb)), "tip_order_rows_workspace_bytes")
            ws = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
            # one buffer: order a | order b | order c | schedules of the two launches
            n_i32 = 4 * n + (int(self.lib.tip_order_rows_out_bytes(n)) + 3) // 4
            flat = torch.empty(n_i32, dtype=torch.int32, device=self.device)
            rows3 = flat[: 12 * n].view(3 * n, 4)
            rows3[:n].copy_(links.rows[:n])
            _cabi.check(self.lib.tip_order_rows(_ptr(flat), n, links.n_rows_r0, _ptr(ws), nb.value,
                                                ctypes.c_void_p(flat.data_ptr() + n * 16), self._stream()), "tip_order_rows")
            self.launches += 10
            torch.cuda.current_stream(self.device).synchronize()
        links.rows3, links.rows, links.rows3_buf, links.order_ws = rows3, rows3[:n], flat, ws

    @_on_device
    def reorder_rows(self):
        """tip_order_rows again, in place and asynchronously, after new rows have been copied into `train.rows` (order a):
        the slot-b / slot-c orders and the schedules are derived from them on the device (bench.py's link-sharded
        end-to-end leg: the rows of every step arrive from the host)."""
        t = self.train
        n = t.n_rows
        _cabi.check(self.lib.tip_order_rows(_ptr(t.rows3_buf), n, t.n_rows_r0, _ptr(t.order_ws), int(t.order_ws.numel()),
                                            ctypes.c_void_p(t.rows3_buf.data_ptr() + n * 16), self._stream()), "tip_order_rows")
        self.launches += 10

    @_on_device
    def set_train_links(self, g1, g2, g3, n0, n1, global_deg=None):
        """This rank's shard of the training links.  `deg` (distinct links per gene, TIP.py:986-994) is
        summed over shards unless the caller supplies the global vector."""
        self.train = self.pack(g1, g2, g3, n0, n1, want_deg=True)
        if self.flags & _cabi.TIP_EM_SLOT_SEGMENTED:
            self.order_rows(self.train)
            if self._auto_flags:
                # hub-shaped links (the 64 busiest genes hold more than a fifth of all link ends, as in a
                # query-pair x array screen): gather theta through L1, see TIP_EM_GATHER_L1
                deg = self.train.deg.to(torch.int64)
                top = torch.topk(deg, min(64, deg.numel())).values.sum()
                hubs = bool((top * 5 > deg.sum()).item()) and deg.numel() > 640
                self.flags = (self.flags | _cabi.TIP_EM_GATHER_L1) if hubs else (self.flags & ~_cabi.TIP_EM_GATHER_L1)
        if global_deg is not None:
            self.train.deg = self._as_dev_i32(global_deg)
        elif self.world > 1:
            _dist.allreduce_sum_(self.train.deg, self.group)
        with torch.cuda.device(self.device):
            nb = ctypes.c_size_t(0)
            _cabi.check(self.lib.tip_em_workspace_bytes(self.P, self.K, self.train.n_rows, self.flags, ctypes.byref(nb)),
                        "tip_em_workspace_bytes")
            self.em_ws = torch.empty(max(nb.value, 8), dtype=torch.uint8, device=self.device)
            self.em_ws_bytes = nb.value
        self._graphs = None

    @_on_device
    def set_test_links(self, g1, g2, g3, n0, n1):
        self.test = self.pack(g1, g2, g3, n0, n1, want_deg=False)
        g1, g2, g3, n0 = (self._as_dev_i32(x) for x in (g1, g2, g3, n0))
        labels = (n0 == 0).to(torch.int32)            # TIP.py:560-563: 0 if n0 else 1
        self.test_ids = (g1, g2, g3, labels)

    @_on_device
    def set_pair_links(self, a, b, n0, n1):
        """Digenic extension (TrigenicInteractionPredictor_23.py): pair links that share theta.  Call after
        set_train_links: the degree of a gene then counts its distinct triplets AND pairs (_23.py:1584-1586, 1615-1616)."""
        if self.world > 1:
            raise NotImplementedError("pair links are not sharded: run the digenic model in one process")
        a, b, n0, n1 = (self._as_dev_i32(x) for x in (a, b, n0, n1))
        self.pairs = torch.stack([a, b, n0, n1], dim=1).contiguous()
        both = torch.cat([a, b]).to(torch.int64)
        self.train.deg = (self.train.deg.to(torch.int64) + torch.bincount(both, minlength=self.P)[: self.P]).to(torch.int32)
        self.q = torch.empty(2 * self.K * self.K, dtype=torch.float64, device=self.device)
        self.sq = torch.zeros(2 * self.K * self.K, dtype=torch.float64, device=self.device)
        self._graphs = None

    @_on_device
    def set_q(self, q):
        qq = torch.from_numpy(np.ascontiguousarray(q, dtype=np.float64).reshape(-1))
        assert qq.numel() == 2 * self.K * self.K
        self.q.copy_(qq, non_blocking=False)

    @_on_device
    def get_q(self) -> np.ndarray:
        return self.q.cpu().numpy().reshape(self.K, self.K, 2)

    def _pairs_estep(self, stats):
        _cabi.check(self.lib.tip_pairs_step(self.P, self.K, _ptr(self.pairs), int(self.pairs.shape[0]), _ptr(self.theta),
                                            _ptr(self.q), _ptr(stats), _ptr(self.sq), self._stream()), "tip_pairs_step")
        self.launches += 1

    def _pairs_mstep(self):
        _cabi.check(self.lib.tip_pairs_normalise(self.K, _ptr(self.sq), _ptr(self.q), self._stream()), "tip_pairs_normalise")
        self.launches += 1

    @_on_device
    def degrees(self) -> np.ndarray:
        return self.train.deg.cpu().numpy()

    # ------------------------------------------------------------------ parameters
    @_on_device
    def set_params(self, theta, p):
        th = torch.from_numpy(np.ascontiguousarray(theta, dtype=np.float64).reshape(-1))
        pp = torch.from_numpy(np.ascontiguousarray(p, dtype=np.float64).reshape(-1))
        assert th.numel() == self.P * self.K and pp.numel() == 2 * self.K ** 3
        self.theta.copy_(th, non_blocking=False)
        self.p.copy_(pp, non_blocking=False)
        if self.world > 1:
            # link shards: every rank must start from the SAME parameters (p is updated multiplicatively from the
            # local copy, so replicas that start apart never meet again): rank 0's copy wins
            _dist.broadcast_from_first_(self.theta, self.group)
            _dist.broadcast_from_first_(self.p, self.group)

    @_on_device
    def get_params(self):
        self._check_peer()
        return (self.theta.cpu().numpy().reshape(self.P, self.K),
                self.p.cpu().numpy().reshape(self.K, self.K, self.K, 2))

    # ------------------------------------------------------------------ EM
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check_peer(self):
        """Called wherever the host synchronises with the device: a peer barrier that timed out poisons the epoch
        (the statistics of that iteration were incomplete) - raise instead of carrying on with a wrong model."""
        if self.peer is not None:
            self.peer.check()

    def _peer_mstep(self, par, theta_pushed=False):
        if self.peer.mode == "push":
            pe = self.peer
            _cabi.check(self.lib.tip_peer_push_mstep(self.P, self.K, _ptr(pe.stats(par)), pe.inbox_ptrs[par], pe.flag_ptrs,
                                                     _ptr(pe.epoch), pe.rank, pe.world, pe.n_pad, 1 if theta_pushed else 0,
                                                     _ptr(self.train.deg), _ptr(self.theta), _ptr(self.p), self._stream()),
                        "tip_peer_push_mstep")
            self.launches += 1
            return
        if self.peer.mode == "rs":
            pe = self.peer
            _cabi.check(self.lib.tip_peer_mstep(self.P, self.K, pe.stats_ptrs[0], pe.theta_ptrs, pe.p_ptrs, pe.flag_ptrs,
                                                _ptr(pe.epoch), pe.rank, pe.world, _ptr(self.train.deg), self._stream()),
                        "tip_peer_mstep")
            self.launches += 1
            return
        _cabi.check(self.lib.tip_peer_barrier(self.peer.flag_ptrs, _ptr(self.peer.epoch), self.peer.rank,
                                              self.peer.world, self._stream()), "tip_peer_barrier")
        _cabi.check(self.lib.tip_normalise_peers(self.P, self.K, self.peer.stats_ptrs[par], self.peer.world,
                                                 _ptr(self.train.deg), _ptr(self.theta), _ptr(self.p),
                                                 self._stream()), "tip_normalise_peers")
        self.launches += 2

    @_on_device
    def em_step(self, stats=None):
        """E-step statistics of this rank's rows into `stats` (default self.stats); no normalisation."""
        t = self.train
        stats = self.stats if stats is None else stats
        seg3 = bool(self.flags & _cabi.TIP_EM_SLOT_SEGMENTED)
        _cabi.check(self.lib.tip_em_step(self.P, self.K, _ptr(t.rows3 if seg3 else t.rows), t.n_rows, t.n_rows_r0, _ptr(self.theta),
                                         _ptr(self.p), _ptr(stats), _ptr(self.em_ws), self.em_ws_bytes,
                                         self.flags, self._stream()), "tip_em_step")
        if self.flags & _cabi.TIP_EM_SLOT_SEGMENTED:
            self.launches += 4                      # prep, pass A, pass B+C, finish
        else:
            self.launches += 3 if (self.K > 4 and not (self.flags & _cabi.TIP_EM_FORCE_GENERIC)) else 2

    @_on_device
    def em_step_host_rows(self, h_rows: torch.Tensor, compact: bool, stats=None):
        """E-step of this rank's rows read from PINNED HOST memory (16-byte rows, or the 8-byte rows of
        tip_rows_compact_host): one copy on a side stream, the fused kernel follows the DMA front
        (tip_em_step_host_rows).  K <= 10, default flags."""
        t = self.train
        stats = self.stats if stats is None else stats
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self.device)
            self._stream_err = torch.zeros(64, dtype=torch.int32, device=self.device)
            self._rows_dev = None
        need = t.n_rows * (8 if compact else 16)
        if self._rows_dev is None or self._rows_dev.numel() < need:
            self._rows_dev = torch.empty(need, dtype=torch.uint8, device=self.device)
        _cabi.check(self.lib.tip_em_step_host_rows(
            self.P, self.K, ctypes.c_void_p(h_rows.data_ptr()), t.n_rows, t.n_rows_r0,
            _cabi.TIP_ROWS_COMPACT8 if compact else 0, _ptr(self._rows_dev), _ptr(self.theta), _ptr(self.p), _ptr(stats),
            _ptr(self.em_ws), self.em_ws_bytes, _ptr(self._stream_err), self._stream(),
            ctypes.c_void_p(self._copy_stream.cuda_stream)), "tip_em_step_host_rows")
        self.launches += 3 if self.K > 4 else 2

    @_on_device
    def host_rows_arrived(self) -> bool:
        """False when a streamed E-step gave up waiting for its rows (synchronises)."""
        bad = int(self._stream_err[0].item()) != 0
        if bad:
            self._stream_err.zero_()
        return not bad

    @_on_device
    def em_iteration_host_rows(self, h_rows: torch.Tensor, compact: bool):
        """em_iteration() with the E-step reading its rows from pinned host memory."""
        if self.peer is not None:
            par = (self._iter & 1) if self.peer.mode != "rs" else 0
            self._iter += 1
            self.em_step_host_rows(h_rows, compact, self.peer.stats(par))
            self._peer_mstep(par)
            return
        self.em_step_host_rows(h_rows, compact)
        if self.world > 1:
            _dist.allreduce_sum_(self.stats, self.group)
        self.normalise()

    @_on_device
    def normalise(self):
        _cabi.check(self.lib.tip_normalise(self.P, self.K, _ptr(self.stats), _ptr(self.train.deg), _ptr(self.theta),
                                           _ptr(self.p), self._stream()), "tip_normalise")
        self.launches += 1

    @_on_device
    def _iteration_body(self, par):
        """E-step, sum of statistics over link shards, M-step, on statistics buffer `par` of the peer exchange."""
        if self.peer is not None:
            if self.peer.mode == "rs":
                par = 0                                   # no double buffering: see tip_peer_mstep
            fused = (self.peer.mode == "push" and bool(self.flags & _cabi.TIP_EM_SLOT_SEGMENTED) and self.train.n_rows > 0
                     and os.environ.get("TIP_PEER_FUSED", "1") != "0")
            if fused:
                # the finish kernel of this E-step stores Ntheta into the peers' inboxes as it produces it
                pe = self.peer
                _cabi.check(self.lib.tip_em_set_push_targets(pe.inbox_ptrs[par], pe.rank, pe.world, pe.n_pad),
                            "tip_em_set_push_targets")
            self.em_step(self.peer.stats(par))
            self._peer_mstep(par, theta_pushed=fused)
            return
        self.em_step()
        if self.pairs is not None:
            self._pairs_estep(self.stats)         # pair terms of Ntheta on top of the triplets', Sq (old theta, old q)
        if self.world > 1:
            _dist.allreduce_sum_(self.stats, self.group)
        self.normalise()
        if self.pairs is not None:
            self._pairs_mstep()

    def em_iteration(self):
        """One make_iteration.  The peer exchange double-buffers the statistics: iteration i uses buffer i & 1, and
        `_iter` is the ONE counter eager iterations and graph replays both advance, so the two can be mixed."""
        self._iteration_body(self._iter & 1)
        self._iter += 1

    # ---- CUDA-graph replay of whole iterations (two graphs when the statistics are double-buffered) ----
    @_on_device
    def capture_graphs(self):
        with torch.cuda.device(self.device):
            self.em_iteration()                           # warm-up outside capture (function attributes, NCCL)
            torch.cuda.synchronize(self.device)
            self._graphs, self._graph_launches = [], 0
            for par in range(2 if (self.peer is not None and self.peer.mode != "rs") else 1):   # graph `par`: statistics buffer `par`
                g = torch.cuda.CUDAGraph()
                before = self.launches
                with torch.cuda.graph(g):
                    self._iteration_body(par)
                self._graph_launches = self.launches - before
                self.launches = before
                self._graphs.append(g)
            self._graph_key = (self.train.rows.data_ptr(), self.train.n_rows, self.flags)

    @_on_device
    def graph_step(self):
        self._graphs[self._iter % len(self._graphs)].replay()
        self._iter += 1
        self.launches += self._graph_launches

    def em_iterations(self, n: int, use_graph: bool = True):
        """n iterations; the (E-step, exchange, M-step) body is captured once in a CUDA graph and replayed
        (an iteration at K=10 on 1e6 links is a few hundred microseconds, so launch latency matters)."""
        if n <= 0:
            return
        if not use_graph or n < 4:
            for _ in range(n):
                self.em_iteration()
            return
        key = (self.train.rows.data_ptr(), self.train.n_rows, self.flags)
        if getattr(self, "_graphs", None) is None or self._graph_key != key:
            self.capture_graphs()
            n -= 1                                        # the warm-up iteration of capture_graphs counted
        for _ in range(n):
            self.graph_step()

    # ------------------------------------------------------------------ likelihood / scoring / metrics
    @_on_device
    def loglik(self, which: str = "train") -> float:
        links = self.train if which == "train" else self.test
        if links is None:
            raise ValueError("no %s links set" % which)
        _cabi.check(self.lib.tip_loglik(self.P, self.K, _ptr(links.rows), links.n_rows, links.n_rows_r0, _ptr(self.theta),
                                        _ptr(self.p), _ptr(self.ll_out), _ptr(self.ll_ws),
                                        self.flags & _cabi.TIP_EM_FORCE_GENERIC, self._stream()),
                    "tip_loglik")
        self.launches += 2 if (self.K <= 10 and not (self.flags & _cabi.TIP_EM_FORCE_GENERIC)) else 1
        if self.pairs is not None and which == "train":
            _cabi.check(self.lib.tip_pairs_loglik(self.P, self.K, _ptr(self.pairs), int(self.pairs.shape[0]), _ptr(self.theta),
                                                  _ptr(self.q), _ptr(self.ll_out), self._stream()), "tip_pairs_loglik")
            self.launches += 1
        if self.world > 1 and which == "train":
            _dist.allreduce_sum_(self.ll_out, self.group)
        value = float(self.ll_out.item())
        self._check_peer()
        return value

    @_on_device
    def step_loglik(self) -> float:
        """log-likelihood by-product of the last E-step of THIS rank's rows (of the parameters that step started
        from); needs TIP_EM_WITH_LOGLIK on the K-specialised path."""
        if self.peer is not None:
            return float(self.peer.stats(((self._iter - 1) & 1) if self.peer.mode != "rs" else 0)[-1].item())
        return float(self.stats[-1].item())

    @_on_device
    def scores(self) -> torch.Tensor:
        g1, g2, g3, _ = self.test_ids
        T = int(g1.numel())
        out = torch.empty(T, dtype=torch.float64, device=self.device)
        _cabi.check(self.lib.tip_score(self.P, self.K, _ptr(g1), _ptr(g2), _ptr(g3), T, _ptr(self.theta), _ptr(self.p),
                                       _ptr(out), self._stream()), "tip_score")
        self.launches += 1
        return out

    @_on_device
    def sort_scores(self, scores: torch.Tensor):
        """tip_sort_scores: (test-set index, score) in descending score order as numpy arrays."""
        T = int(scores.numel())
        nb = ctypes.c_size_t(0)
        _cabi.check(self.lib.tip_sort_scores_workspace_bytes(T, ctypes.byref(nb)), "tip_sort_scores_workspace_bytes")
        ws = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
        order = torch.empty(T, dtype=torch.int32, device=self.device)
        out = torch.empty(T, dtype=torch.float64, device=self.device)
        _cabi.check(self.lib.tip_sort_scores(_ptr(scores), T, _ptr(ws), nb.value, _ptr(order), _ptr(out), self._stream()),
                    "tip_sort_scores")
        self.launches += 2
        return order.cpu().numpy(), out.cpu().numpy()

    @_on_device
    def top_triplets(self, theta_stack, p_stack, cand, known, n: int):
        """tip_top_triplets: the `n` best triplets of the candidate genes under the mean of S models.
        theta_stack [S][P][K], p_stack [S][K][K][K][2] (numpy fp64); cand: gene ids in decimal-string order; known: sorted
        packed rank triples to leave out.  Returns (ids [m][3] int32 in slot order, scores [m] float64), best first."""
        th = np.ascontiguousarray(theta_stack, dtype=np.float64)
        pp = np.ascontiguousarray(p_stack, dtype=np.float64)
        S = int(th.shape[0])
        assert th.shape == (S, self.P, self.K) and pp.shape == (S, self.K, self.K, self.K, 2)
        cand = np.ascontiguousarray(cand, dtype=np.int32)
        known = np.ascontiguousarray(known, dtype=np.uint64)
        n_cand, n_known, n = int(cand.shape[0]), int(known.shape[0]), int(n)
        nb = ctypes.c_size_t(0)
        _cabi.check(self.lib.tip_top_triplets_workspace_bytes(n_cand, self.K, S, n_known, n, ctypes.byref(nb)),
                    "tip_top_triplets_workspace_bytes")
        d_th = torch.from_numpy(th.reshape(-1)).to(self.device)
        d_p = torch.from_numpy(pp.reshape(-1)).to(self.device)
        d_cand = torch.from_numpy(cand).to(self.device)
        d_known = torch.from_numpy(known.view(np.int64)).to(self.device) if n_known else None
        ws = torch.empty(max(nb.value, 1), dtype=torch.uint8, device=self.device)
        out_ids = torch.empty((max(n, 1), 3), dtype=torch.int32, device=self.device)
        out_sc = torch.empty(max(n, 1), dtype=torch.float64, device=self.device)
        m = ctypes.c_int64(0)
        _cabi.check(self.lib.tip_top_triplets(self.P, self.K, S, _ptr(d_th), _ptr(d_p), _ptr(d_cand), n_cand, _ptr(d_known),
                                              n_known, n, _ptr(ws), nb.value, _ptr(out_ids), _ptr(out_sc), ctypes.byref(m),
                                              self._stream()), "tip_top_triplets")
        m = int(m.value)
        return out_ids[:m].cpu().numpy(), out_sc[:m].cpu().numpy()

    @_on_device
    def metric_counts(self, scores: torch.Tensor, positives_number: int) -> dict:
        """Integer ingredients of calculate_metrics (TIP.py:583-637); ratios are formed by the caller."""
        labels = self.test_ids[3]
        T = int(scores.numel())
        nb = ctypes.c_size_t(0)
        _cabi.check(self.lib.tip_metrics_workspace_bytes(T, ctypes.byref(nb)), "tip_metrics_workspace_bytes")
        ws = torch.empty(nb.value, dtype=torch.uint8, device=self.device)
        out = torch.zeros(8, dtype=torch.int64, device=self.device)
        _cabi.check(self.lib.tip_metrics(_ptr(scores), _ptr(labels), T, int(positives_number), _ptr(ws), nb.value,
                                         _ptr(out), self._stream()), "tip_metrics")
        self.launches += 5
        o = out.cpu().numpy()
        cut = float(np.array([o[7]], dtype=np.int64).view(np.float64)[0])
        return {"wins": int(o[0]), "n_pos": int(o[1]), "n_neg": int(o[2]), "tp": int(o[3]), "fp": int(o[4]),
                "fn": int(o[5]), "tn": int(o[6]), "cut_value": cut}
