"""The kernels of the training and evaluation path outside the E-step, each against an exact reference at its edges.

Digestion (tip_pack_rows, tip_order_rows_by_gene, the 8-byte rows), the M-step (tip_normalise), scoring (tip_score),
ranking (tip_sort_scores), the metric counts (tip_metrics), the cross-sample reducer (tip_reduce_samples) and the digenic
pair kernels (tip_pairs_step / _normalise / _loglik) take K or the problem size at run time, and most of them run a
grid-stride loop over a grid capped at a few CTAs per SM.  A bug that shows only at K > 16, on the second pass of a
grid-stride loop or at a rating block of exactly 32 rows passes any test that runs one shape.  So every case here sits at
such an edge, and the sizes called "past the grid cap" are chosen from the device's SM count so that every thread's
grid-stride loop runs at least three times.

Nearly all of these kernels have an exact reference - integer counts, sorts, single IEEE operations - so most checks are
equalities.  Tolerances, where there are any: scores 1e-13 relative to scores_np (K^3-term sums in another order),
pair statistics and the pair log-likelihood 1e-12, the reducer's standard deviation 1e-13 (CPython squares with pow(),
the kernel with a product), the E-step over re-ordered rows 1e-11, whole digenic iterations 1e-10 (TIP_EM_FP32_COMPUTE
1e-5, the bound include/tip.h documents for that mode).

The kernels are called through the C ABI (_cabi.load()) on torch tensors, so each test pins a kernel, not the Python
layer above it; only the whole digenic iterations and the held-out chain go through Model.

test_every_kernel_has_a_row (no GPU) keeps COVERAGE honest: a kernel added to one of the files it scans without a row,
or a row whose kernel or test no longer exists, fails it.
"""
import contextlib
import ctypes
import functools
import io
import os
import random
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "trigenicinteractionpredictor_b200", "csrc")
EPS = 1e-10

# ---------------------------------------------------------------------------------------------------------------------
# 0. coverage table: every __global__ kernel of the scanned files -> the tests below that run it
# ---------------------------------------------------------------------------------------------------------------------
COVERAGE = {
    "tip_rows.cu": {
        "rows_make_keys_kernel": ["test_pack_rows_edges"],
        "rows_emit_kernel": ["test_pack_rows_edges"],
    },
    "tip_seg3.cu": {
        "order_keys_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
        "order_emit_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
        "order_hist_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
        "order_scan_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
        "order_scatter_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
        "sched_build_kernel": ["test_order_rows_by_gene_across_the_counting_switch"],
    },
    "tip_api.cu": {
        "rows_expand_kernel": ["test_compact_rows_round_trip"],
    },
    "tip_mstep.cu": {
        "normalise_kernel": ["test_normalise_vs_reference"],
    },
    "tip_generic.cu": {
        "gen_score_kernel": ["test_score_every_k", "test_score_past_the_grid_cap", "test_held_out_chain"],
    },
    "tip_metrics.cu": {
        "iota_kernel": ["test_sort_scores_order", "test_held_out_chain"],
        "neg_flag_kernel": ["test_metrics_vs_integer_counts", "test_held_out_chain"],
        "metrics_count_kernel": ["test_metrics_vs_integer_counts", "test_held_out_chain"],
    },
    "tip_reduce.cu": {
        "reduce_samples_kernel": ["test_reduce_samples_edges"],
    },
    "tip_pairs.cu": {
        "pairs_kernel": ["test_pairs_kernels_vs_oracle", "test_digenic_iterations_vs_oracle"],
        "pairs_normalise_kernel": ["test_pairs_kernels_vs_oracle", "test_digenic_iterations_vs_oracle"],
    },
}
# kernels of the scanned files that this file leaves out on purpose
LEFT_OUT = {
    "tip_seg3.cu": {
        "seg3_pass_kernel": "E-step: test_estep_coverage.py",
        "seg3_prep_kernel": "E-step: test_estep_coverage.py",
        "seg3_finish_kernel": "E-step: test_estep_coverage.py",
    },
    "tip_generic.cu": {
        "gen_estep_kernel": "E-step: test_estep_coverage.py",
        "gen_pstat_kernel": "E-step: test_estep_coverage.py",
        "gen_loglik_kernel": "log-likelihood: test_estep_coverage.py",
    },
    "tip_api.cu": {
        "fma_probe_kernel": "measurement probe (tip_measure_fma_peak), no result to check",
        "dmma_probe_kernel": "measurement probe (tip_measure_fma_peak), no result to check",
        "red_probe_kernel": "measurement probe (tip_measure_red_f64), no result to check",
        "gather_probe_kernel": "measurement probe (tip_measure_l2_gather), no result to check",
    },
}
# source files not scanned, and where their kernels are tested
FILES_ELSEWHERE = {
    "tip_em.cu": "E-step and log-likelihood kernels: test_estep_coverage.py",
    "tip_predict.cu": "prediction, ranking and gene-pair kernels: test_predict*.py, test_rank_*.py, "
                      "test_digenic_predict.py; at the sizes their limits accept: SCALE_COVERAGE in test_predict_scale.py",
    "tip_peer.cu": "peer_* and normalise_peers_kernel need two GPUs: test_gpu_dist.py",
}


def _strip_comments(src):
    return re.sub(r"//[^\n]*", "", re.sub(r"/\*.*?\*/", "", src, flags=re.S))


def _skip_parens(src, i):
    """index just past the parenthesised group that starts at the first '(' at or after i"""
    i = src.index("(", i)
    depth = 0
    while True:
        if src[i] == "(":
            depth += 1
        elif src[i] == ")":
            depth -= 1
            if depth == 0:
                return i + 1
        i += 1


def _kernels_in(path):
    """names of the __global__ functions defined in a source file"""
    src = _strip_comments(open(path, encoding="utf-8").read())
    names = set()
    for m in re.finditer(r"\b__global__\b", src):
        i = m.end()
        while True:
            w = re.compile(r"\s*(\w+)").match(src, i)
            i = w.end()
            if w.group(1) in ("__launch_bounds__", "__maxnreg__"):
                i = _skip_parens(src, i)
            elif w.group(1) != "void":
                names.add(w.group(1))
                break
    return names


def test_every_kernel_has_a_row():
    sources = {f for f in os.listdir(CSRC) if f.endswith(".cu")}
    scanned = set(COVERAGE) | set(LEFT_OUT)
    assert sources == scanned | set(FILES_ELSEWHERE), \
        "source files neither scanned nor listed in FILES_ELSEWHERE: %s" % sorted(sources - scanned - set(FILES_ELSEWHERE))
    problems = []
    for f in sorted(scanned):
        kernels = _kernels_in(os.path.join(CSRC, f))
        rows = set(COVERAGE.get(f, {})) | set(LEFT_OUT.get(f, {}))
        problems += ["%s: %s has no row" % (f, k) for k in sorted(kernels - rows)]
        problems += ["%s: the row %s names no kernel" % (f, k) for k in sorted(rows - kernels)]
        for k, tests in COVERAGE.get(f, {}).items():
            problems += ["%s: %s names a missing test %s" % (f, k, t) for t in tests if not callable(globals().get(t))]
    assert not problems, "; ".join(problems)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _lib():
    from trigenicinteractionpredictor_b200 import _cabi
    return _cabi.load()


def _err(lib):
    return (lib.tip_last_error() or b"").decode("utf-8", "replace")


def _sm(torch):
    return torch.cuda.get_device_properties(0).multi_processor_count


def _st(torch):
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _relerr(a, b):
    """max elementwise relative error; elements equal to each other (0 against 0 included) count as 0."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    err[a == b] = 0.0
    return float(err.max()) if err.size else 0.0


def _bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.int64)


def _params(P, K, seed):
    rng = np.random.default_rng(seed)
    theta = rng.dirichlet(np.ones(K), size=P)
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    return theta, pr


# ---------------------------------------------------------------------------------------------------------------------
# 1. digestion: tip_pack_rows, tip_order_rows_by_gene, the 8-byte rows
# ---------------------------------------------------------------------------------------------------------------------
def _pack_reference(P, g, n0, n1):
    """The rows of each rating block ordered (a, b, c) and padded with (0, 0, 0, r) to 32 rows, and the degrees."""
    exp = []
    for r, n in ((0, n0), (1, n1)):
        sel = np.nonzero(n > 0)[0]
        order = np.lexsort((g[sel, 2], g[sel, 1], g[sel, 0]))
        blk = np.stack([g[sel, 0], g[sel, 1], g[sel, 2], (n[sel] << 1) | r], axis=1)[order]
        pad = (-len(blk)) % 32
        blk = np.concatenate([blk.reshape(-1, 4), np.tile(np.array([[0, 0, 0, r]], dtype=np.int32), (pad, 1))])
        exp.append(blk.astype(np.int32))
    live = (n0 > 0) | (n1 > 0)
    deg = np.bincount(g[live].ravel(), minlength=P).astype(np.int32)
    return exp, deg


def _pack(torch, lib, P, g, n0, n1):
    """tip_pack_rows on the device: (rc, rows, h_part, degrees); the degree vector starts as garbage."""
    L = len(g)
    cols = [_dev(torch, np.ascontiguousarray(g[:, i], dtype=np.int32)) for i in range(3)]
    c0, c1 = _dev(torch, n0.astype(np.int32)), _dev(torch, n1.astype(np.int32))
    nb = ctypes.c_size_t(0)
    assert lib.tip_pack_rows_workspace_bytes(L, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    rows = torch.empty((int(lib.tip_rows_capacity(L)), 4), dtype=torch.int32, device="cuda")
    deg = torch.full((P,), -7, dtype=torch.int32, device="cuda")
    n_rows = ctypes.c_int64(-1)
    part = (ctypes.c_int64 * 3)(-1, -1, -1)
    rc = lib.tip_pack_rows(cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), c0.data_ptr(), c1.data_ptr(), L, P,
                           ws.data_ptr(), nb.value, rows.data_ptr(), ctypes.byref(n_rows), part, deg.data_ptr(), _st(torch))
    torch.cuda.synchronize()
    return rc, rows[: max(n_rows.value, 0)].cpu().numpy(), n_rows.value, list(part), deg.cpu().numpy()


PACK_CASES = ["no_links", "one_link", "rating0_only", "rating1_only", "blocks_of_31_and_33", "blocks_of_32",
              "links_without_counts", "links_with_both_counts", "counts_up_to_2^20", "ids_at_2^20-1", "past_the_grid_cap"]


def _pack_case(case, sm):
    rng = np.random.default_rng(PACK_CASES.index(case))
    P, L = 300, 1000
    g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
    n0 = rng.integers(0, 3, size=L).astype(np.int32)
    n1 = rng.integers(0, 3, size=L).astype(np.int32)
    if case == "no_links":
        g, n0, n1 = g[:0], n0[:0], n1[:0]
    elif case == "one_link":
        P, g, n0, n1 = 5, np.array([[4, 0, 2]], dtype=np.int32), np.array([0], np.int32), np.array([3], np.int32)
    elif case == "rating0_only":
        n0, n1 = np.maximum(n0, 1), np.zeros_like(n1)
    elif case == "rating1_only":
        n0, n1 = np.zeros_like(n0), np.maximum(n1, 1)
    elif case in ("blocks_of_31_and_33", "blocks_of_32"):
        # real rows per rating block: 31 and 33 (padding 1 and 31), or 32 and 32 (no padding)
        a, b = (31, 33) if case == "blocks_of_31_and_33" else (32, 32)
        g = g[: a + b]
        n0 = np.r_[np.ones(a, np.int32), np.zeros(b, np.int32)]
        n1 = np.r_[np.zeros(a, np.int32), rng.integers(1, 4, size=b).astype(np.int32)]
    elif case == "links_without_counts":
        # a third of the links have n0 = n1 = 0: no row and no degree; gene 299 appears in those links only
        n0[::3] = 0
        n1[::3] = 0
        g[g == P - 1] = 0
        g[::3, 1] = P - 1
    elif case == "links_with_both_counts":
        n0, n1 = np.maximum(n0, 1), np.maximum(n1, 1)
    elif case == "counts_up_to_2^20":
        n0 = rng.integers(0, 1 << 20, size=L, endpoint=True).astype(np.int32)
        n1 = rng.integers(0, 1 << 20, size=L, endpoint=True).astype(np.int32)
        n0[:3], n1[3:6] = 1 << 20, (1 << 20) - 1
    elif case == "ids_at_2^20-1":
        P = 1 << 20
        g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
        g[:8] = [[0, 0, 0], [P - 1, P - 1, P - 1], [0, P - 1, 0], [P - 1, 0, P - 1], [0, 0, P - 1], [P - 1, P - 1, 0],
                 [P - 1, 0, 0], [0, P - 1, P - 1]]
        n0[:8], n1[:8] = [1, 2, 0, 3, 1, 0, 2, 1], [1, 0, 2, 1, 0, 3, 1, 2]
    elif case == "past_the_grid_cap":
        P, L = 5000, 3 * sm * 8 * 256 + 1234
        g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
        n0 = rng.integers(0, 3, size=L).astype(np.int32)
        n1 = rng.integers(0, 3, size=L).astype(np.int32)
    return P, g, n0, n1


@pytest.mark.gpu
@pytest.mark.parametrize("case", PACK_CASES)
def test_pack_rows_edges(torch_cuda, case):
    """tip_pack_rows bit-exact against NumPy: the rows of each rating block, their padding, h_part and the degrees."""
    torch = torch_cuda
    lib = _lib()
    P, g, n0, n1 = _pack_case(case, _sm(torch))
    exp, deg = _pack_reference(P, g, n0, n1)
    rc, rows, n_rows, part, got_deg = _pack(torch, lib, P, g, n0, n1)
    assert rc == 0, _err(lib)
    n_real = int((n0 > 0).sum() + (n1 > 0).sum())
    assert part == [len(exp[0]), len(exp[1]), n_real] and n_rows == len(exp[0]) + len(exp[1]), (case, part, n_rows)
    for blk, lo in ((exp[0], 0), (exp[1], len(exp[0]))):
        got = rows[lo: lo + len(blk)]
        assert np.array_equal(got[:, :3], blk[:, :3]), case
        # rows of the same triplet (a repeated link) may come in either order: compare them sorted by count
        canon = lambda x: x[np.lexsort((x[:, 3], x[:, 2], x[:, 1], x[:, 0]))]  # noqa: E731
        assert np.array_equal(canon(got), canon(blk)), case
    assert np.array_equal(got_deg, deg), "degrees, %s" % case
    if case == "past_the_grid_cap":
        assert len(g) >= 3 * _sm(torch) * 8 * 256 and n_rows >= 3 * _sm(torch) * 8 * 256
    if case == "links_without_counts":
        assert deg[P - 1] == 0


@pytest.mark.gpu
def test_pack_rows_refuses_more_than_2_20_genes(torch_cuda):
    torch = torch_cuda
    lib = _lib()
    g = np.array([[0, 1, 2]], dtype=np.int32)
    rc, _, _, _, _ = _pack(torch, lib, (1 << 20) + 1, g, np.ones(1, np.int32), np.zeros(1, np.int32))
    assert rc != 0 and "2^20" in _err(lib)
    rc, _, _, _, _ = _pack(torch, lib, 1 << 20, g, np.ones(1, np.int32), np.zeros(1, np.int32))
    assert rc == 0, _err(lib)


COUNT_MAX_BINS = 12288             # tip_seg3.cu: kCountMaxBins, the shared-memory counters of the counting sort
ORDER_CASES = [(P, n) for P in (6142, 6143, 6144) for n in (12256, 12288, 12320)]


def _schedule_covers_every_tile(sched, nt, what):
    live = sched[sched != 0]
    assert np.all(sched[len(live):] == 0), what
    seen = np.zeros(nt, dtype=np.int64)
    for e in live.tolist():
        e &= 0x7FFFFFFF
        t0, cnt = e >> 3, e & 7
        assert 1 <= cnt <= 4 and t0 + cnt <= nt, what
        seen[t0: t0 + cnt] += 1
    assert np.all(seen == 1), "schedule %s does not hold every tile exactly once" % what


@pytest.mark.gpu
@pytest.mark.parametrize("P,n_rows", ORDER_CASES)
def test_order_rows_by_gene_across_the_counting_switch(torch_cuda, P, n_rows):
    """tip_order_rows_by_gene on both sides of its switch to the counting sort (2 (P + 1) <= 12288 and <= n_rows):
    the counting sort holds the (rating, gene) runs of tip_order_rows with the same rows in each, the radix fallback is
    bit-identical to it; both schedules hold every tile once; an E-step over the re-ordered rows matches the oracle."""
    torch = torch_cuda
    from oracle import mmsbm_oracle as orc
    from trigenicinteractionpredictor_b200.engine import EMEngine
    lib = _lib()
    K = 5
    counting = 2 * (P + 1) <= COUNT_MAX_BINS and 2 * (P + 1) <= n_rows
    rng = np.random.default_rng(P + n_rows)
    tiles = n_rows // 32
    real0, real1 = tiles // 2 * 32 - 3, (tiles - tiles // 2) * 32 - 17
    L = real0 + real1
    g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
    g[::5, 1] = 7                                   # a hub in slot b and slot c: runs across several tiles
    g[1::7, 2] = 11
    g[:4] = [[0, P - 1, 0], [P - 1, 0, P - 1], [3, P - 1, P - 1], [P - 1, 0, 0]]
    g[real0: real0 + 4] = g[:4]
    n0 = np.r_[rng.integers(1, 3, size=real0), np.zeros(real1, int)].astype(np.int32)
    n1 = np.r_[np.zeros(real0, int), rng.integers(1, 3, size=real1)].astype(np.int32)
    eng = EMEngine(P, K, flags=32)
    eng.set_train_links(g[:, 0], g[:, 1], g[:, 2], n0, n1)
    t = eng.train
    n = t.n_rows
    assert n == n_rows and t.n_rows_r0 == tiles // 2 * 32
    T = n // 32
    used = 12 * n + 3 * T                           # the three orders, then the schedules of the two launches
    want = t.rows3_buf.cpu().numpy()[:used]
    out = torch.zeros_like(t.rows3_buf)
    out[: 4 * n].copy_(t.rows3_buf[: 4 * n])
    ws = torch.empty_like(t.order_ws)
    rc = lib.tip_order_rows_by_gene(out.data_ptr(), n, t.n_rows_r0, P, ws.data_ptr(), int(ws.numel()),
                                    out.data_ptr() + n * 16, _st(torch))
    assert rc == 0, _err(lib)
    torch.cuda.synchronize()
    got = out.cpu().numpy()[:used]
    what = "P=%d n_rows=%d %s" % (P, n, "counting" if counting else "radix")
    if counting:
        blockid = (np.arange(n) >= t.n_rows_r0).astype(np.int64)
        for blk in (1, 2):
            w = want[4 * n * blk: 4 * n * (blk + 1)].reshape(n, 4)
            h = got[4 * n * blk: 4 * n * (blk + 1)].reshape(n, 4)
            assert np.array_equal(w[:, 0], h[:, 0]), "run layout, order %d, %s" % (blk, what)

            def canon(x):   # rows sorted by (rating block, gene with padding last, position in order a)
                gene = np.where(x[:, 3] < 0, 1 << 30, x[:, 0].astype(np.int64))
                return x[np.lexsort((x[:, 3], gene, blockid))]
            assert np.array_equal(canon(h), canon(w)) and np.array_equal(canon(w), w), "runs, order %d, %s" % (blk, what)
    else:
        assert np.array_equal(got, want), "the radix fallback differs from tip_order_rows, " + what
    sched = got[12 * n: used]
    _schedule_covers_every_tile(sched[:T], T, "a, " + what)
    _schedule_covers_every_tile(sched[T:], 2 * T, "bc, " + what)
    theta, pr = _params(P, K, P)
    t.rows3_buf.copy_(out)
    eng.set_params(theta, pr)
    eng.em_step()
    ent, enp, _ = orc.em_step_np(theta, pr, g.astype(np.int64), np.stack([n0, n1], axis=1).astype(np.int64),
                                 return_stats=True)
    st = eng.stats.cpu().numpy()
    S = st[P * K: P * K + 2 * K ** 3].reshape(2, K, K, K)
    assert _relerr(st[: P * K].reshape(P, K), ent) < 1e-11, "Ntheta, " + what
    assert _relerr(pr * np.moveaxis(S, 0, -1), enp) < 1e-11, "p * S, " + what


def test_order_rows_cases_cross_the_switch():
    counting = [2 * (P + 1) <= COUNT_MAX_BINS and 2 * (P + 1) <= n for P, n in ORDER_CASES]
    assert any(counting) and not all(counting)
    assert (6143, 12288) in ORDER_CASES and 2 * (6143 + 1) == 12288 == COUNT_MAX_BINS


GENE_MAX = (1 << 20) - 1


@pytest.mark.gpu
def test_compact_rows_round_trip(torch_cuda):
    """tip_rows_compact_host -> tip_rows_expand bit-exact at gene id 2^20 - 1 and count 7, over more rows than the
    expand kernel's grid covers in one pass; count 8, id 2^20 and the row that encodes to the arrival sentinel are
    refused (-1)."""
    torch = torch_cuda
    lib = _lib()
    n = 3 * _sm(torch) * 8 * 256 + 64
    rng = np.random.default_rng(20)
    rows = np.empty((n, 4), dtype=np.int32)
    rows[:, :3] = rng.integers(0, GENE_MAX + 1, size=(n, 3))
    cnt, r = rng.integers(0, 8, size=n), rng.integers(0, 2, size=n)
    rows[:, 3] = (cnt << 1) | r
    rows[:6, :3] = [[0, 0, 0], [GENE_MAX, GENE_MAX, GENE_MAX], [GENE_MAX, 0, 0], [0, GENE_MAX, 0], [0, 0, GENE_MAX],
                    [GENE_MAX, GENE_MAX, 0]]
    rows[:6, 3] = [0, (7 << 1) | 0, (7 << 1) | 1, 1, (7 << 1) | 1, (7 << 1) | 1]
    sentinel = (rows[:, :3] == GENE_MAX).all(axis=1) & (rows[:, 3] == 15)
    rows[sentinel, 3] = 14
    rows8 = np.zeros(n, dtype=np.uint64)
    assert lib.tip_rows_compact_host(rows.ctypes.data, n, rows8.ctypes.data) == 0, _err(lib)
    u = rows.astype(np.uint64)
    exp8 = u[:, 2] | (u[:, 1] << np.uint64(20)) | (u[:, 0] << np.uint64(40)) | ((u[:, 3] & np.uint64(1)) << np.uint64(60)) \
        | ((u[:, 3] >> np.uint64(1)) << np.uint64(61))
    assert np.array_equal(rows8, exp8)
    d8 = _dev(torch, rows8.view(np.int64))
    out = torch.full((n, 4), -5, dtype=torch.int32, device="cuda")
    assert lib.tip_rows_expand(d8.data_ptr(), out.data_ptr(), n, _st(torch)) == 0, _err(lib)
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy(), rows)
    bad_rows = [[1, 2, 3, (8 << 1) | 0], [1 << 20, 0, 0, 2], [0, 1 << 20, 0, 2], [0, 0, 1 << 20, 2],
                [GENE_MAX, GENE_MAX, GENE_MAX, 15]]
    for bad in bad_rows:
        one = np.array([rows[7], bad], dtype=np.int32)
        o8 = np.zeros(2, dtype=np.uint64)
        assert lib.tip_rows_compact_host(one.ctypes.data, 2, o8.ctypes.data) == -1, bad


# ---------------------------------------------------------------------------------------------------------------------
# 2. M-step: tip_normalise
# ---------------------------------------------------------------------------------------------------------------------
NORM_K = [1, 2, 3, 4, 9, 10, 11, 16, 17, 31, 32]


@pytest.mark.gpu
@pytest.mark.parametrize("K", NORM_K)
def test_normalise_vs_reference(torch_cuda, K):
    """theta = Ntheta / deg and p = n_r / ((eps + n_0) + n_1) with n_r = p_r * S_r are single IEEE operations; the kernel
    multiplies and adds separately (its SASS has DMUL then DADD, no contraction into DFMA), so both are asserted
    bit-identical.  P = 1037 (not a multiple of 256) and a P for which P K + K^3 runs every thread's grid-stride loop at
    least three times.  Genes of degree 0 give inf where their statistic is > 0 and nan where it is 0."""
    torch = torch_cuda
    lib = _lib()
    cap = _sm(torch) * 4 * 256
    for P in (1037, (3 * cap - K ** 3) // K + 5):
        rng = np.random.default_rng(P * 40 + K)
        K3 = K ** 3
        stats = np.zeros(int(lib.tip_stats_len(P, K)))
        nth = rng.random((P, K)) * rng.integers(1, 50, size=(P, 1))
        nth[rng.random((P, K)) < 0.1] = 0.0
        deg = rng.integers(1, 60, size=P).astype(np.int32)
        deg[5::97] = 0                                   # no link at all: inf where the statistic is > 0, nan where 0
        nth[5::194] = 0.0
        S = rng.random((2, K3)) * 100.0
        S[rng.random((2, K3)) < 0.1] = 0.0
        stats[: P * K] = nth.ravel()
        stats[P * K: P * K + 2 * K3] = S.ravel()
        p = rng.random((K3, 2))
        p /= p.sum(axis=1, keepdims=True)
        p[rng.random(K3) < 0.1] = (1.0, 0.0)
        d_stats, d_deg = _dev(torch, stats), _dev(torch, deg)
        d_theta = torch.full((P * K,), -1.0, dtype=torch.float64, device="cuda")
        d_p = _dev(torch, p.ravel())
        assert lib.tip_normalise(P, K, d_stats.data_ptr(), d_deg.data_ptr(), d_theta.data_ptr(), d_p.data_ptr(),
                                 _st(torch)) == 0, _err(lib)
        torch.cuda.synchronize()
        with np.errstate(divide="ignore", invalid="ignore"):
            th_exp = nth / deg[:, None].astype(np.float64)
        n0, n1 = p[:, 0] * S[0], p[:, 1] * S[1]
        d = (EPS + n0) + n1
        p_exp = np.stack([n0 / d, n1 / d], axis=1)
        th = d_theta.cpu().numpy().reshape(P, K)
        what = "K=%d P=%d" % (K, P)
        assert np.array_equal(th, th_exp, equal_nan=True), "theta, " + what
        assert np.array_equal(_bits(th[np.isfinite(th)]), _bits(th_exp[np.isfinite(th_exp)])), "theta bits, " + what
        zero = deg == 0
        assert np.all(np.isposinf(th[zero][nth[zero] > 0])) and np.all(np.isnan(th[zero][nth[zero] == 0])), what
        assert np.isnan(th).any() and np.isinf(th).any(), "the case must have genes of degree 0, " + what
        assert np.array_equal(_bits(d_p.cpu().numpy().reshape(K3, 2)), _bits(p_exp)), "p, " + what


# ---------------------------------------------------------------------------------------------------------------------
# 3. scoring: tip_score
# ---------------------------------------------------------------------------------------------------------------------
def _score(torch, lib, P, K, ids, theta, pr):
    T = len(ids)
    cols = [_dev(torch, np.ascontiguousarray(ids[:, i], dtype=np.int32)) for i in range(3)]
    out = torch.full((max(T, 1),), -3.0, dtype=torch.float64, device="cuda")
    d_th, d_p = _dev(torch, theta.ravel()), _dev(torch, pr.ravel())
    rc = lib.tip_score(P, K, cols[0].data_ptr(), cols[1].data_ptr(), cols[2].data_ptr(), T, d_th.data_ptr(), d_p.data_ptr(),
                       out.data_ptr(), _st(torch))
    assert rc == 0, _err(lib)
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _score_ids(P, T, rng):
    ids = rng.integers(0, P, size=(T, 3)).astype(np.int32)
    edge = np.array([[0, P - 1, 0], [P - 1, P - 1, P - 1], [0, 0, 0], [P - 1, 0, 3], [3, 0, P - 1]], dtype=np.int32)
    ids[: min(T, 5)] = edge[: min(T, 5)]
    if T >= 8:
        ids[7] = ids[1]                             # a repeated triplet
    return ids


@pytest.mark.gpu
@pytest.mark.parametrize("K", list(range(1, 33)))
def test_score_every_k(torch_cuda, K):
    """tip_score against scores_np at every K the library takes, T in {0, 1, 7, 8, 9} (8 warps per CTA), ids 0 and P - 1,
    a triplet of one gene three times and a repeated triplet (bit-identical scores)."""
    torch = torch_cuda
    from oracle import mmsbm_oracle as orc
    lib = _lib()
    P = 50
    theta, pr = _params(P, K, 300 + K)
    assert K == 1 or not np.allclose(pr, pr.transpose(1, 0, 2, 3))
    rng = np.random.default_rng(K)
    for T in (0, 1, 7, 8, 9):
        ids = _score_ids(P, T, rng)
        got = _score(torch, lib, P, K, ids, theta, pr)
        if T == 0:
            assert got[0] == -3.0, "T = 0 wrote a score"
            continue
        assert _relerr(got[:T], orc.scores_np(theta, pr, ids.astype(np.int64))) < 1e-13, "K=%d T=%d" % (K, T)
        if T >= 8:
            assert got[7] == got[1]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 4, 10])
def test_score_past_the_grid_cap(torch_cuda, K):
    torch = torch_cuda
    from oracle import mmsbm_oracle as orc
    lib = _lib()
    P = 2000
    T = 3 * _sm(torch) * 8 * 8 + 5                  # grid of sm * 8 CTAs of 8 warps: three passes and a partial one
    theta, pr = _params(P, K, 400 + K)
    ids = _score_ids(P, T, np.random.default_rng(400 + K))
    got = _score(torch, lib, P, K, ids, theta, pr)
    assert _relerr(got, orc.scores_np(theta, pr, ids.astype(np.int64))) < 1e-13


# ---------------------------------------------------------------------------------------------------------------------
# 4. ranking: tip_sort_scores
# ---------------------------------------------------------------------------------------------------------------------
SORT_T = [1, 2, 3, 255, 256, 257, 4095, 4096, 4097, 100_000, 5_000_000]
SORT_SETS = ["ties", "all_equal", "zeros", "subnormal", "spread", "one_ulp_apart"]


def _sort_scores_set(kind, T, rng):
    if kind == "ties":
        return np.round(rng.random(T), 2)
    if kind == "all_equal":
        return np.full(T, 0.3125)
    if kind == "zeros":
        s = rng.random(T)
        s[rng.random(T) < 0.3] = 0.0
        return s
    if kind == "subnormal":
        s = rng.integers(0, 1 << 12, size=T) * 5e-324 * 1024     # subnormals, with ties and exact zeros
        s[::7] = 2.2250738585072014e-308                         # the smallest normal number
        return s
    if kind == "one_ulp_apart":
        # a few values and their next 1..3 doubles: scores that differ in the last bit of the mantissa only
        base = rng.choice(np.array([0.1, 0.3, 2.0 / 3.0, 0.7]), size=T)
        return (base.view(np.int64) + rng.integers(0, 4, size=T)).view(np.float64)
    return 10.0 ** rng.uniform(-300, 0, size=T)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", SORT_SETS)
@pytest.mark.parametrize("T", SORT_T)
def test_sort_scores_order(torch_cuda, T, kind):
    """tip_sort_scores: the order identical to a stable descending argsort, the sorted values bit-identical."""
    torch = torch_cuda
    lib = _lib()
    s = _sort_scores_set(kind, T, np.random.default_rng(T + SORT_SETS.index(kind)))
    if kind == "subnormal" and T > 100:
        assert np.any((s > 0) & (s < 2.2250738585072014e-308))
    nb = ctypes.c_size_t(0)
    assert lib.tip_sort_scores_workspace_bytes(T, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    d_s = _dev(torch, s)
    order = torch.full((T,), -1, dtype=torch.int32, device="cuda")
    out = torch.empty(T, dtype=torch.float64, device="cuda")
    assert lib.tip_sort_scores(d_s.data_ptr(), T, ws.data_ptr(), nb.value, order.data_ptr(), out.data_ptr(), _st(torch)) == 0, \
        _err(lib)
    exp = np.argsort(-s, kind="stable")
    got = order.cpu().numpy()
    assert np.array_equal(got, exp), "order, T=%d %s: first difference at %d" % (T, kind, int(np.argmax(got != exp)))
    assert np.array_equal(_bits(out.cpu().numpy()), _bits(s[exp])), "sorted values, T=%d %s" % (T, kind)


@pytest.mark.gpu
def test_sort_scores_refuses_2_31(torch_cuda):
    torch = torch_cuda
    lib = _lib()
    one = torch.zeros(1, dtype=torch.float64, device="cuda")
    idx = torch.zeros(1, dtype=torch.int32, device="cuda")
    ws = torch.empty(256, dtype=torch.uint8, device="cuda")
    assert lib.tip_sort_scores(one.data_ptr(), 1 << 31, ws.data_ptr(), 256, idx.data_ptr(), one.data_ptr(), _st(torch)) != 0


# ---------------------------------------------------------------------------------------------------------------------
# 5. metrics: tip_metrics
# ---------------------------------------------------------------------------------------------------------------------
def _metrics_reference(s, lab, pn):
    """[wins, n_pos, n_neg, tp, fp, fn, tn, cut bits] in integers: wins counts (positive, negative) pairs with the
    positive strictly above; cut = the pn-th largest score (0.0 past the end); s >= cut counts as predicted positive."""
    T = len(s)
    cut = np.sort(s)[::-1][pn] if pn < T else 0.0
    pos, neg = s[lab != 0], np.sort(s[lab == 0])
    wins = int(np.searchsorted(neg, pos, side="left").sum())
    pred, y = s >= cut, lab != 0
    return [wins, int(y.sum()), int((~y).sum()), int((pred & y).sum()), int((pred & ~y).sum()), int((~pred & y).sum()),
            int((~pred & ~y).sum()), int(_bits(np.array([cut]))[0])]


def _metrics_device(torch, lib, d_s, d_lab, T, pn):
    nb = ctypes.c_size_t(0)
    assert lib.tip_metrics_workspace_bytes(T, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    out = torch.full((8,), -1, dtype=torch.int64, device="cuda")
    rc = lib.tip_metrics(d_s.data_ptr(), d_lab.data_ptr(), T, pn, ws.data_ptr(), nb.value, out.data_ptr(), _st(torch))
    assert rc == 0, _err(lib)
    return [int(x) for x in out.cpu().numpy()]


METRIC_CASES = ["one_positive", "one_negative", "no_positives", "no_negatives", "all_tied", "ties_at_the_cut",
                "past_the_grid_cap", "wins_past_2^32"]


def _metric_case(case, sm, rng):
    if case in ("one_positive", "one_negative"):
        return np.array([0.25]), np.array([case == "one_positive"], dtype=np.int32)
    T = 3001
    s = rng.random(T)
    lab = (rng.random(T) < 0.4).astype(np.int32)
    if case == "no_positives":
        lab[:] = 0
    elif case == "no_negatives":
        lab[:] = 1
    elif case == "all_tied":
        s[:] = 0.5
    elif case == "ties_at_the_cut":
        s = np.round(s, 1)
    elif case == "past_the_grid_cap":
        T = 3 * sm * 8 * 256 + 77                   # not a multiple of 256; three passes of sm * 8 CTAs of 256
        s, lab = np.round(rng.random(T), 4), (rng.random(T) < 0.3).astype(np.int32)
    elif case == "wins_past_2^32":
        T = 2_000_003
        s, lab = rng.random(T), (rng.random(T) < 0.5).astype(np.int32)
    return s, lab


@pytest.mark.gpu
@pytest.mark.parametrize("case", METRIC_CASES)
def test_metrics_vs_integer_counts(torch_cuda, case):
    """All 8 output words of tip_metrics equal to integer NumPy counts, at positives_number in {0, 1, T - 1, T, T + 5}
    (and inside a tie run at the cut)."""
    torch = torch_cuda
    lib = _lib()
    s, lab = _metric_case(case, _sm(torch), np.random.default_rng(METRIC_CASES.index(case)))
    T = len(s)
    pns = {0, 1, T - 1, T, T + 5}
    if case == "ties_at_the_cut":
        desc = np.sort(s)[::-1]
        mid = next(i for i in range(T // 2, T - 1) if desc[i - 1] == desc[i] == desc[i + 1])
        pns |= {mid, mid + 1}
    d_s, d_lab = _dev(torch, s), _dev(torch, lab)
    for pn in sorted(p for p in pns if p >= 0):
        exp = _metrics_reference(s, lab, pn)
        got = _metrics_device(torch, lib, d_s, d_lab, T, pn)
        assert got == exp, "%s, positives_number %d" % (case, pn)
    if case == "all_tied":
        assert exp[0] == 0
    if case == "wins_past_2^32":
        assert exp[0] > 1 << 32


@pytest.mark.gpu
def test_metrics_refusals(torch_cuda):
    """T = 0, a negative positives_number, a workspace one byte short, and T = 2^31: the exclusive scan of the negative
    flags accumulates in int32, so more than 2^31 - 1 negatives would wrap; all refused before any device work."""
    torch = torch_cuda
    lib = _lib()
    T = 1000
    d_s = _dev(torch, np.random.default_rng(0).random(T))
    d_lab = _dev(torch, np.zeros(T, dtype=np.int32))
    out = torch.zeros(8, dtype=torch.int64, device="cuda")
    nb = ctypes.c_size_t(0)
    assert lib.tip_metrics_workspace_bytes(T, ctypes.byref(nb)) == 0
    ws = torch.empty(nb.value, dtype=torch.uint8, device="cuda")
    call = lambda n, pn, wsb: lib.tip_metrics(d_s.data_ptr(), d_lab.data_ptr(), n, pn, ws.data_ptr(), wsb,  # noqa: E731
                                              out.data_ptr(), _st(torch))
    assert call(0, 0, nb.value) != 0
    assert call(T, -1, nb.value) != 0
    assert call(T, 0, nb.value - 1) != 0 and "workspace" in _err(lib)
    assert call(1 << 31, 0, nb.value) != 0 and "2^31" in _err(lib), _err(lib)
    torch.cuda.synchronize()
    assert not out.any(), "a refused call wrote its output"
    assert call(T, 0, nb.value) == 0, _err(lib)


# ---------------------------------------------------------------------------------------------------------------------
# 6. reducer: tip_reduce_samples
# ---------------------------------------------------------------------------------------------------------------------
def _reduce_reference(X, n_valid):
    """(mean, median, std, sorted) of every column of X[S][T] over its first n_valid[t] samples (clamped to S; 0 gives
    zeros), in the reference's operation order: the sums are sequential in sample order; columns are grouped by n so that
    the median index is one number per group."""
    S, T = X.shape
    n = np.minimum(n_valid, S)
    mean, median, std = np.zeros(T), np.zeros(T), np.zeros(T)
    srt = np.full((S, T), np.nan)
    for m in np.unique(n):
        if m <= 0:
            continue
        cols = np.nonzero(n == m)[0]
        x = X[:m, cols]
        acc = np.zeros(len(cols))
        for j in range(m):
            acc = acc + x[j]
        mu = acc / m
        v = np.sort(x, axis=0)
        if m % 2:
            med = v[round(m / 2)]
        else:
            med = (v[m // 2 - 1] + v[m // 2]) / 2
        acc2 = np.zeros(len(cols))
        for j in range(m):
            dv = v[j] - mu
            acc2 = acc2 + dv * dv
        mean[cols], median[cols], std[cols] = mu, med, np.sqrt(acc2 / m)
        srt[:m, cols] = v
    return mean, median, std, srt


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 2, 191, 192, 193])
def test_reduce_samples_edges(torch_cuda, S):
    """tip_reduce_samples at S = 191 / 192 (the last S on the shared-memory path, 32 threads per CTA) and 193 (the
    global-memory path), with d_n = NULL and with n_valid in {0, 1, S, S + 3} and values between, columns of equal values
    (std exactly 0), over enough triplets to run every thread's grid-stride loop at least three times.  Mean, median and
    the sorted copy bit-identical to the reference; std within 1e-13; the vectorised reference is itself held to
    reducer_oracle.reduce_values on a sample of columns."""
    torch = torch_cuda
    from oracle import reducer_oracle as ro
    lib = _lib()
    sm = _sm(torch)
    threads = min(256, (48 * 1024 // (8 * S)) // 32 * 32)
    T = 3 * (sm * 16 * threads if threads >= 32 else sm * 8 * 256) + 7
    rng = np.random.default_rng(S)
    X = rng.integers(0, 1000, size=(S, T), dtype=np.int16) * 0.001                     # ties inside columns
    eq = np.arange(5, T, 97)
    X[:, eq] = rng.integers(1, 1000, size=len(eq)) / 1024.0                            # sums exact: std exactly 0
    picks = [0, 1, S, S + 3] + sorted({max(S // 2, 1), max(S - 1, 1)})
    n_valid = np.array(picks, dtype=np.int32)[rng.integers(0, len(picks), size=T)]
    n_valid[:len(picks)] = picks
    d_x = _dev(torch, X)
    for label, nv in (("d_n = NULL", None), ("n_valid", n_valid)):
        d_sorted = torch.full((S, T), float("nan"), dtype=torch.float64, device="cuda")
        outs = [torch.full((T,), -1.0, dtype=torch.float64, device="cuda") for _ in range(3)]
        d_n = _dev(torch, nv) if nv is not None else None
        rc = lib.tip_reduce_samples(S, T, d_x.data_ptr(), d_n.data_ptr() if d_n is not None else None, d_sorted.data_ptr(),
                                    outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), _st(torch))
        assert rc == 0, _err(lib)
        torch.cuda.synchronize()
        n = np.full(T, S, dtype=np.int32) if nv is None else nv
        mean, median, std, srt = _reduce_reference(X, n)
        got_mean, got_median, got_std = (o.cpu().numpy() for o in outs)
        what = "S=%d T=%d %s" % (S, T, label)
        assert np.array_equal(_bits(got_mean), _bits(mean)), "mean, " + what
        assert np.array_equal(_bits(got_median), _bits(median)), "median, " + what
        assert _relerr(got_std, std) < 1e-13, "std, " + what
        live = ~np.isnan(srt)
        got_sorted = d_sorted.cpu().numpy()
        assert np.array_equal(_bits(got_sorted[live]), _bits(srt[live])), "sorted copy, " + what
        m = np.minimum(n, S)
        assert np.all(got_std[eq[m[eq] > 0]] == 0.0), "std of equal values, " + what
        zero = m == 0
        assert (not zero.any() or (np.all(got_mean[zero] == 0.0) and np.all(got_median[zero] == 0.0)
                                   and np.all(got_std[zero] == 0.0))), what
        for t in list(range(len(picks))) + rng.integers(0, T, size=40).tolist() + eq[:5].tolist():
            if m[t] > 0:
                vals = X[: m[t], t].tolist()
                r_mean, r_median, r_std = ro.reduce_values(vals)
                assert (r_mean, r_median) == (mean[t], median[t]) and vals == srt[: m[t], t].tolist(), (what, t)
                assert r_std == pytest.approx(std[t], rel=1e-13, abs=0.0), (what, t)


# ---------------------------------------------------------------------------------------------------------------------
# 7. digenic pair kernels
# ---------------------------------------------------------------------------------------------------------------------
def _pair_terms(theta, qr, ids2, cnt2):
    """The pair term of oracle/digenic_oracle.em_step_23_np: (Ntheta [P][K] of the pairs alone, Sq [2][K][K] with
    nqr = q * Sq)."""
    from oracle import digenic_oracle as dg
    P, K = theta.shape
    ntheta = np.zeros((P, K))
    d = dg.pair_denominators(theta, qr, ids2)
    s = cnt2 / d
    ta, tb = theta[ids2[:, 0]], theta[ids2[:, 1]]
    u = np.einsum("lj,ijr,lr->li", tb, qr, s, optimize=True)
    v = np.einsum("li,ijr,lr->lj", ta, qr, s, optimize=True)
    np.add.at(ntheta, ids2[:, 0], ta * u)
    np.add.at(ntheta, ids2[:, 1], tb * v)
    return ntheta, np.einsum("li,lj,lr->rij", ta, tb, s, optimize=True)


PAIR_K = [1, 2, 4, 5, 9, 16, 17, 31, 32]
PAIR_CASES = ["no_pairs", "mixed_counts", "hub"]


def _pair_case(case, P, rng):
    if case == "no_pairs":
        return np.zeros((0, 2), dtype=np.int32), np.zeros((0, 2), dtype=np.int32)
    if case == "mixed_counts":
        n = 600
        ids = rng.integers(0, P, size=(n, 2)).astype(np.int32)
        ids[:4] = [[0, P - 1], [P - 1, 0], [0, 0], [P - 1, P - 1]]
        ids[4:24, 1] = ids[4:24, 0]                  # pairs (a, a): a line naming one gene twice digests to one
        kind = np.arange(n) % 4                      # only n0, only n1, both, counts above 1
        c = rng.integers(1, 4, size=(n, 2))
        c[kind == 0, 1] = 0
        c[kind == 1, 0] = 0
        c[kind == 3] *= 3
        return ids, c.astype(np.int32)
    n = 100_000                                      # gene 0 in half of the pairs, in either slot
    ids = rng.integers(1, P, size=(n, 2)).astype(np.int32)
    hub = rng.random(n) < 0.5
    ids[hub, rng.integers(0, 2, size=int(hub.sum()))] = 0
    c = rng.integers(0, 2, size=(n, 2))
    c[c.sum(axis=1) == 0, rng.integers(0, 2, size=int((c.sum(axis=1) == 0).sum()))] = 1
    return ids, c.astype(np.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("case", PAIR_CASES)
@pytest.mark.parametrize("K", PAIR_K)
def test_pairs_kernels_vs_oracle(torch_cuda, K, case):
    """tip_pairs_step on zeroed statistics: its Ntheta rows and Sq against the pair term of em_step_23_np (1e-12); then
    tip_pairs_normalise bit-identical to q Sq / ((eps + n_0) + n_1) on the device's Sq and within 1e-12 of the oracle's,
    and tip_pairs_loglik against the pair part of loglik_23_np (1e-12).  No pairs: Sq = 0, q becomes 0."""
    torch = torch_cuda
    from oracle import digenic_oracle as dg
    lib = _lib()
    P = 200
    rng = np.random.default_rng(K * 10 + PAIR_CASES.index(case))
    theta = rng.dirichlet(np.ones(K), size=P)
    q = rng.random((K, K, 2))
    q /= q.sum(axis=2, keepdims=True)
    ids2, cnt2 = _pair_case(case, P, rng)
    n = len(ids2)
    if case == "hub":
        assert n >= 3 * _sm(torch) * 4 * 8 and (ids2 == 0).any(axis=1).sum() > n // 3
    pairs = _dev(torch, np.concatenate([ids2, cnt2], axis=1).astype(np.int32).reshape(-1, 4)) if n else None
    pairs_ptr = pairs.data_ptr() if n else None
    d_th, d_q = _dev(torch, theta.ravel()), _dev(torch, q.ravel())
    stats = torch.zeros(int(lib.tip_stats_len(P, K)), dtype=torch.float64, device="cuda")
    sq = torch.full((2 * K * K,), float("nan"), dtype=torch.float64, device="cuda")
    assert lib.tip_pairs_step(P, K, pairs_ptr, n, d_th.data_ptr(), d_q.data_ptr(), stats.data_ptr(), sq.data_ptr(),
                              _st(torch)) == 0, _err(lib)
    ll = torch.zeros(1, dtype=torch.float64, device="cuda")
    assert lib.tip_pairs_loglik(P, K, pairs_ptr, n, d_th.data_ptr(), d_q.data_ptr(), ll.data_ptr(), _st(torch)) == 0, _err(lib)
    torch.cuda.synchronize()
    st, got_sq = stats.cpu().numpy(), sq.cpu().numpy().reshape(2, K, K)
    nth_ref, sq_ref = _pair_terms(theta, q, ids2.astype(np.int64), cnt2.astype(np.float64))
    what = "K=%d %s" % (K, case)
    assert _relerr(st[: P * K].reshape(P, K), nth_ref) < 1e-12, "Ntheta, " + what
    assert not st[P * K:].any(), "tip_pairs_step wrote past Ntheta, " + what
    assert _relerr(got_sq, sq_ref) < 1e-12, "Sq, " + what
    ll_ref = float((cnt2 * np.log(dg.pair_denominators(theta, q, ids2.astype(np.int64)))).sum())
    assert ll.item() == pytest.approx(ll_ref, rel=1e-12, abs=0.0), "pair log-likelihood, " + what
    assert lib.tip_pairs_normalise(K, sq.data_ptr(), d_q.data_ptr(), _st(torch)) == 0, _err(lib)
    torch.cuda.synchronize()
    got_q = d_q.cpu().numpy().reshape(K, K, 2)
    n0, n1 = q[..., 0] * got_sq[0], q[..., 1] * got_sq[1]
    d = (EPS + n0) + n1
    assert np.array_equal(_bits(got_q), _bits(np.stack([n0 / d, n1 / d], axis=-1))), "q, " + what
    nq = q * np.moveaxis(sq_ref, 0, -1)
    assert _relerr(got_q, nq / ((EPS + nq[..., 0]) + nq[..., 1])[..., None]) < 1e-12, "q against the oracle, " + what
    if case == "no_pairs":
        assert not got_sq.any() and not got_q.any() and ll.item() == 0.0


ITER_K = [1, 4, 5, 9, 16, 17, 32]
ITER_FLAGS = [None, 0, 1, 32, 96, 8, 2]
ITER_ENTRIES = [(K, f) for K in ITER_K for f in ITER_FLAGS if (f != 8 or K >= 5) and (f != 2 or K <= 10)]


@functools.lru_cache(maxsize=None)
def _mixed_lines():
    """A mixed train file (triplet lines and pair lines; repeated lines give counts above 1; one pair line names one gene
    twice) in which genes G090..G119 appear only in pairs, and a test file over the same genes."""
    rng = np.random.default_rng(23)
    name = lambda i: "G%03d" % i  # noqa: E731
    train = []
    for t in range(400):
        a, b, c = rng.permutation(90)[:3] if t >= 30 else (3 * t, 3 * t + 1, 3 * t + 2)
        train.append("%s_%s_%s\t%d\n" % (name(a), name(b), name(c), int(rng.random() < 0.3)))
    for t in range(300):
        a, b = rng.permutation(120)[:2] if t >= 30 else (90 + t, int(rng.integers(0, 120)))
        if a == b:
            b = (b + 1) % 120
        train.append("%s_%s\t%d\n" % (name(a), name(b), int(rng.random() < 0.4)))
    train += train[5:25] + train[420:440]           # repeated sightings
    train.append("%s_%s\t1\n" % (name(7), name(7)))
    test = ["%s_%s_%s\t%d\n" % (name(3 * t), name(3 * t + 5), name(3 * t + 9), t % 2) for t in range(20)]
    test += ["%s_%s\t%d\n" % (name(90 + t), name(t), t % 2) for t in range(10)]
    return "".join(train), "".join(test)


@functools.lru_cache(maxsize=None)
def _digenic_oracle(K):
    """(theta, pr, qr, loglik) of the oracle for iterations 0..3 from the seeded initial parameters."""
    from oracle import digenic_oracle as dg
    train, _ = _mixed_lines()
    links3, links2, P = dg.digest_mixed(train.splitlines())
    ids3 = np.array([[int(x) for x in k.split("_")] for k in links3], dtype=np.int64)
    cnt3 = np.array(list(links3.values()), dtype=np.int64)
    ids2 = np.array([[int(x) for x in k.split("_")] for k in links2], dtype=np.int64)
    cnt2 = np.array(list(links2.values()), dtype=np.int64)
    th, pr, q = dg.init_params_23(P, K, random.Random(2300 + K))
    out = [(th, pr, q, dg.loglik_23_np(th, pr, q, ids3, cnt3, ids2, cnt2))]
    for _ in range(3):
        th, pr, q = dg.em_step_23_np(th, pr, q, ids3, cnt3, ids2, cnt2)
        out.append((th, pr, q, dg.loglik_23_np(th, pr, q, ids3, cnt3, ids2, cnt2)))
    return P, ids3, ids2, out


@pytest.mark.gpu
@pytest.mark.parametrize("K,flags", ITER_ENTRIES, ids=["K%d-flags%s" % e for e in ITER_ENTRIES])
def test_digenic_iterations_vs_oracle(torch_cuda, tmp_path, K, flags):
    """Three make_iterations of the digenic Model against em_step_23_np / loglik_23_np (1e-10; fp32 1e-5) with every
    E-step family the flags select, on a mixed file where some genes have pairs only: their degree comes from pairs
    alone, and the triplet E-step must leave their Ntheta rows for tip_pairs_step to fill."""
    from trigenicinteractionpredictor_b200.TrigenicInteractionPredictor_23 import Model
    train, test = _mixed_lines()
    (tmp_path / "train.dat").write_text(train, encoding="utf-8")
    (tmp_path / "test.dat").write_text(test, encoding="utf-8")
    m = Model(flags=flags)
    with contextlib.redirect_stdout(io.StringIO()):
        m.get_train_test(str(tmp_path / "train.dat"), str(tmp_path / "test.dat"))
    P, ids3, ids2, ref = _digenic_oracle(K)
    assert m.P == P
    pair_only = set(ids2.ravel().tolist()) - set(ids3.ravel().tolist())
    assert len(pair_only) >= 30 and (ids2[:, 0] == ids2[:, 1]).any()
    g3, _ = Model._arrays(m.links, 3)
    g2, _ = Model._arrays(m.dlinks, 2)
    assert np.array_equal(g3, ids3) and np.array_equal(g2, ids2)
    random.seed(2300 + K)
    m.initialize_parameters(K)
    assert np.array_equal(np.array(m.theta), ref[0][0]) and np.array_equal(np.array(m.qr), ref[0][2])
    tol = 1e-5 if flags == 2 else 1e-10
    assert m.compute_likelihood() == pytest.approx(ref[0][3], rel=tol)
    for it in range(1, 4):
        m.make_iteration()
        th, pr, q, ll = ref[it]
        what = "K=%d flags=%s iteration %d" % (K, flags, it)
        got_th = np.array(m.theta)
        assert _relerr(got_th, th) < tol, "theta, " + what
        assert _relerr(got_th[sorted(pair_only)], th[sorted(pair_only)]) < tol, "theta of pair-only genes, " + what
        assert _relerr(m.pr, pr) < tol, "pr, " + what
        assert _relerr(m.qr, q) < tol, "qr, " + what
        assert m.compute_likelihood() == pytest.approx(ll, rel=tol), "log-likelihood, " + what


# ---------------------------------------------------------------------------------------------------------------------
# 8. held-out chain at K outside the goldens: tip_score -> tip_sort_scores -> tip_metrics through Model
# ---------------------------------------------------------------------------------------------------------------------
def _triplets(P, n, rng):
    """n distinct triplets of distinct genes, each in decimal-string slot order"""
    out = set()
    while len(out) < n:
        out.add(tuple(sorted(rng.choice(P, size=3, replace=False).tolist(), key=str)))
    return np.array(sorted(out), dtype=np.int32)[rng.permutation(n)]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 4, 7, 17, 32])
def test_held_out_chain(torch_cuda, K):
    """Model.set_links_soa, calculate_test_set_results, calculate_metrics: scores within 1e-12 of scores_np, the results
    table equal to test_results of the device scores (exact ties forced by repeated theta rows), the metrics equal to
    oracle.metrics."""
    from oracle import mmsbm_oracle as orc
    from trigenicinteractionpredictor_b200 import Model
    rng = np.random.default_rng(800 + K)
    P = 60
    g = _triplets(P, 400, rng)
    g[:20] = np.array([sorted((3 * i, 3 * i + 1, 3 * i + 2), key=str) for i in range(20)], dtype=np.int32)
    g = np.unique(g, axis=0)[rng.permutation(len(np.unique(g, axis=0)))]
    lab = (rng.random(len(g)) < 0.3).astype(np.int32)
    n1 = lab.copy()
    n1[::17] *= 2                                   # n1 = 2 is not a single positive sighting (TIP.py:588)
    gt = _triplets(P, 500, rng)
    labt = (rng.random(len(gt)) < 0.3).astype(np.int32)
    m = Model()
    m.set_links_soa((g[:, 0], g[:, 1], g[:, 2], 1 - lab, n1), (gt[:, 0], gt[:, 1], gt[:, 2], 1 - labt, labt), P=P)
    random.seed(40 + K)
    m.initialize_parameters(K)
    th = np.array(m.theta)
    th[:] = th[rng.integers(0, 4, P)]               # four distinct theta rows: many exactly equal scores
    m.theta = th.tolist()
    pr = np.array(m.pr)
    m.calculate_test_set_results()
    sc = m._scores.cpu().numpy()
    assert _relerr(sc, orc.scores_np(th, pr, gt.astype(np.int64))) < 1e-12
    test_links = {"%d_%d_%d" % tuple(k): [int(1 - y), int(y)] for k, y in zip(gt.tolist(), labt.tolist())}
    train_links = {"%d_%d_%d" % tuple(k): [int(1 - y), int(c)] for k, y, c in zip(g.tolist(), lab.tolist(), n1.tolist())}
    assert len(test_links) == len(gt) and len(train_links) == len(g)
    exp = orc.test_results(sc, test_links)
    assert len({r[0] for r in exp}) < len(exp) // 2, "the case must contain exact ties"
    assert m.results == exp
    assert m.calculate_metrics() == orc.metrics(exp, train_links, len(test_links))
