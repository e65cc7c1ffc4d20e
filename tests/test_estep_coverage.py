"""Every E-step kernel instantiation against the fp64 NumPy oracle, and the link-set edges where the kernels split work.

The E-step kernels are templates on K, and each formulation flag of tip_em_step selects a different family of
instantiations.  They change shape with K exactly where kernels break: the 8 x 8 accumulator blocks (NB = (K + 7) / 8),
the gather mapping of the slot-segmented passes (UNIT, LPI, ITERS of S3<K>), where p lives (rotating constant slot for
K <= 10, the whole bank for K = 11..15, one rating at a time for K = 16), the per-lane scatter of odd K against the bulk
reductions of even K, and the register budget of each (K, MINB).  A correct K = 10 says little about K = 14 or K = 27,
so this file runs every (family, K) the library is built for:

  * MATRIX: one entry per (family, K, flags); each runs one step on a uniform and on a hub-shaped problem and checks the
    statistics, the log-likelihood, the normalised parameters and (slot-segmented) CUDA-graph replays.
  * test_every_instantiation_is_in_the_matrix (no GPU): the library's kernels, listed from its SASS, against MATRIX -
    a kernel variant added without an entry here fails on a machine without a GPU.
  * test_flags_select_the_family_the_matrix_names: the template arguments the flags actually launch (torch.profiler).
  * test_link_set_edges: one rating block empty, one or two tiles, genes without a link, few genes, exact zeros.

Tolerances: statistics and normalised parameters 1e-11 relative per element (TIP_EM_FP32_COMPUTE: 1e-5, the bound
include/tip.h documents for that mode), log-likelihood 1e-12, three graph replays 1e-10.  An element that is exactly 0 in
the oracle must be exactly 0 on the device.
"""
import functools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

RTOL = 1e-11
RTOL_FP32 = 1e-5
RTOL_LL = 1e-12
RTOL_ITER = 1e-10

TIP_EM_GATHER_L1 = 64

# ---------------------------------------------------------------------------------------------------------------------
# The instantiation matrix: (family, K, flags).  Families and the template arguments that name them:
#   plain     em_fused_kernel<K, MINB, LL=0, double, SEG=0, STREAM=0>   flags 0, K 1..16
#   anyK      gen_estep_kernel (run-time K, no template)                 flags 1 (TIP_EM_FORCE_GENERIC)
#   fp32      em_fused_kernel<K, MINB, 0, float, 0, 0>                   flags 2 (TIP_EM_FP32_COMPUTE), K 1..10
#   loglik    em_fused_kernel<K, MINB, 1, double, 0, 0>                  flags 4 (TIP_EM_WITH_LOGLIK), K 1..10
#   gene_seg  em_fused_kernel<K, MINB, 0, double, 1, 0>                  flags 8 (TIP_EM_GENE_SEGMENTED) for K 5..16,
#                                                                        flags 0 for K 17..32 (their only fused kernel)
#   stream    em_fused_kernel<K, MINB, 0, double, 0, 1>                  tip_em_step_host_rows / tip_em_iterations_host, K 1..10
#   slot_l2   seg3_pass_kernel<K, FIRST, CA=0> + seg3_finish_kernel<K>   flags 32 (TIP_EM_SLOT_SEGMENTED)
#   slot_l1   seg3_pass_kernel<K, FIRST, CA=1> + seg3_finish_kernel<K>   flags 32 | 64 (+ TIP_EM_GATHER_L1)
# ---------------------------------------------------------------------------------------------------------------------
ANY_K = [1, 2, 5, 10, 11, 16, 17, 26, 32]      # one run-time-K kernel: a spread of K is enough
MATRIX = ([("plain", K, 0) for K in range(1, 17)]
          + [("anyK", K, 1) for K in ANY_K]
          + [("fp32", K, 2) for K in range(1, 11)]
          + [("loglik", K, 4) for K in range(1, 11)]
          + [("gene_seg", K, 8 if K <= 16 else 0) for K in range(5, 33)]
          + [("stream", K, 0) for K in range(1, 11)]
          + [("slot_l2", K, 32) for K in range(1, 33)]
          + [("slot_l1", K, 32 | 64) for K in range(1, 33)])

FUSED_FAMILY = {           # em_fused_kernel<K, MINB, LL, T, SEG, STREAM>: (LL, T, SEG, STREAM) -> family (MINB follows K)
    ("0", "double", "0", "0"): "plain",
    ("0", "float", "0", "0"): "fp32",
    ("1", "double", "0", "0"): "loglik",
    ("0", "double", "1", "0"): "gene_seg",
    ("0", "double", "0", "1"): "stream",
}
SLOT_FAMILY = {"0": "slot_l2", "1": "slot_l1"}   # seg3_pass_kernel<K, FIRST, CA>: CA -> family (every step runs both FIRST)
BYPRODUCT = {"loglik", "anyK"}                    # families that leave sum n log d in the last statistics slot
SHAPES = ["uniform", "hubs"]


def _ids(entries):
    return ["%s-K%d" % (f, K) for f, K, _ in entries]


def _tol(family):
    return RTOL_FP32 if family == "fp32" else RTOL


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _relerr(a, b):
    """max elementwise relative error; elements equal to each other (0 against 0 included) count as 0."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    err = np.abs(a - b) / np.maximum(np.abs(b), 1e-300)
    err[a == b] = 0.0
    return float(err.max()) if err.size else 0.0


def _random_problem(P, L, K, seed):
    rng = np.random.default_rng(seed)
    g = rng.integers(0, P, size=(L, 3)).astype(np.int32)
    g[:P, 0] = np.arange(P)                       # every gene has a training link
    lab = (rng.random(L) < 0.15).astype(np.int32)
    theta = rng.dirichlet(np.ones(K), size=P)
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    return g, 1 - lab, lab, theta, pr


def _n_links(K):
    return 6000 if K <= 10 else (2000 if K <= 16 else 700)


@functools.lru_cache(maxsize=None)
def _problem(shape, K):
    """P = 300 genes; uniform links, or hub-shaped ones (a handful of query genes in all three key slots); counts of
    2 and 3 on some links, and some links seen with both ratings."""
    from trigenicinteractionpredictor_b200 import synth
    P, L = 300, _n_links(K)
    g, n0, n1, theta, pr = _random_problem(P, L, K, 700 + K)
    if shape == "hubs":
        a, b, c, lab = synth.kuzmin_links_soa(P, L, seed=K, n_query=6)
        g = np.stack([a, b, c], axis=1).astype(np.int32)
        g[:P, 0] = np.arange(P)
        n0, n1 = (1 - lab).astype(np.int32), lab.astype(np.int32)
    n0, n1 = n0.copy(), n1.copy()
    n0[5::37] += 2                                # repeated sightings: counts above one
    n1[9::41] += 1
    both = np.arange(L)[13::29]                   # links seen with both ratings: a row in each rating block
    n0[both] = np.maximum(n0[both], 1)
    n1[both] = np.maximum(n1[both], 1)
    return P, g, n0, n1, theta, pr


def _oracle(theta, pr, g, n0, n1):
    from oracle import mmsbm_oracle as orc
    ids = g.astype(np.int64)
    cnt = np.stack([n0, n1], axis=1).astype(np.int64)
    ent, enp, deg = orc.em_step_np(theta, pr, ids, cnt, return_stats=True)
    return ent, enp, deg, orc.loglik_np(theta, pr, ids, cnt)


@functools.lru_cache(maxsize=None)
def _problem_oracle(shape, K):
    P, g, n0, n1, theta, pr = _problem(shape, K)
    return _oracle(theta, pr, g, n0, n1)


@functools.lru_cache(maxsize=None)
def _oracle_iterations(shape, K, n):
    """(theta, p) after n oracle EM iterations from the problem's parameters."""
    from oracle import mmsbm_oracle as orc
    P, g, n0, n1, theta, pr = _problem(shape, K)
    if n == 0:
        return theta, pr
    if n == 1:
        ent, enp, deg, _ = _problem_oracle(shape, K)
        return orc.normalise_np(ent, enp, deg)
    th, p = _oracle_iterations(shape, K, n - 1)
    return orc.em_step_np(th, p, g.astype(np.int64), np.stack([n0, n1], axis=1).astype(np.int64))


def _engine(P, K, flags, g, n0, n1, theta, pr):
    from trigenicinteractionpredictor_b200.engine import EMEngine
    eng = EMEngine(P, K, flags=flags)
    eng.set_train_links(g[:, 0], g[:, 1], g[:, 2], n0, n1)
    eng.set_params(theta, pr)
    return eng


def _split_stats(st, P, K, pr):
    """(Ntheta [P][K], p * S [K][K][K][2]) of a statistics buffer."""
    nth = st[: P * K].reshape(P, K)
    S = st[P * K: P * K + 2 * K ** 3].reshape(2, K, K, K)
    return nth, pr * np.moveaxis(S, 0, -1)


def _check_stats(st, family, P, K, pr, ref, what):
    ent, enp, deg, ll = ref
    tol = _tol(family)
    nth, npr = _split_stats(st, P, K, pr)
    assert _relerr(nth, ent) < tol, "Ntheta, %s: %.3g" % (what, _relerr(nth, ent))
    assert _relerr(npr, enp) < tol, "p * S, %s: %.3g" % (what, _relerr(npr, enp))
    if family in BYPRODUCT:
        assert st[-1] == pytest.approx(ll, rel=RTOL_LL), "log-likelihood by-product, %s" % what
    else:
        assert st[-1] == 0.0, "log-likelihood slot written without TIP_EM_WITH_LOGLIK, %s" % what


def _check_step(family, flags, P, K, g, n0, n1, theta, pr, ref, what, params=True):
    """One tip_em_step of `flags` against the oracle's statistics, log-likelihood, degrees and (params) M-step."""
    from oracle import mmsbm_oracle as orc
    eng = _engine(P, K, flags, g, n0, n1, theta, pr)
    eng.em_step()
    _check_stats(eng.stats.cpu().numpy(), family, P, K, pr, ref, what)
    assert eng.loglik("train") == pytest.approx(ref[3], rel=RTOL_LL), "tip_loglik, %s" % what
    assert np.array_equal(eng.degrees(), ref[2].astype(np.int32)), "degrees, %s" % what
    if params:
        th1, pr1 = orc.normalise_np(ref[0], ref[1], ref[2])
        eng.normalise()
        th, p = eng.get_params()
        tol = _tol(family)
        assert _relerr(th, th1) < tol, "theta after the M-step, %s: %.3g" % (what, _relerr(th, th1))
        assert _relerr(p, pr1) < tol, "p after the M-step, %s: %.3g" % (what, _relerr(p, pr1))
    return eng


# ---------------------------------------------------------------------------------------------------------------------
# 1. the instantiation matrix
# ---------------------------------------------------------------------------------------------------------------------
STEP_ENTRIES = [e for e in MATRIX if e[0] != "stream"]
STREAM_ENTRIES = [e for e in MATRIX if e[0] == "stream"]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("family,K,flags", STEP_ENTRIES, ids=_ids(STEP_ENTRIES))
def test_estep_instantiation_vs_oracle(torch_cuda, family, K, flags, shape):
    P, g, n0, n1, theta, pr = _problem(shape, K)
    ref = _problem_oracle(shape, K)
    what = "%s K=%d flags=%d %s" % (family, K, flags, shape)
    eng = _check_step(family, flags, P, K, g, n0, n1, theta, pr, ref, what)
    if family.startswith("slot"):
        # em_iterations(n) captures the iteration into a CUDA graph from n = 4 on: one eager warm-up, then three replays
        eng.set_params(theta, pr)
        eng.em_iterations(4)
        assert eng._graphs is not None, "em_iterations(4) did not go through the CUDA graph"
        th, p = eng.get_params()
        tho, pro = _oracle_iterations(shape, K, 4)
        assert _relerr(th, tho) < RTOL_ITER and _relerr(p, pro) < RTOL_ITER, "graph replays, %s" % what


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("family,K,flags", STREAM_ENTRIES, ids=_ids(STREAM_ENTRIES))
def test_streamed_instantiation_vs_oracle(torch_cuda, family, K, flags, shape):
    """The streamed kernel (rows polled as the host-to-device copy lands): tip_em_step_host_rows with 16-byte and 8-byte
    host rows, then tip_em_iterations_host (streamed first iteration, resident ones behind it), against the oracle."""
    torch = torch_cuda
    from oracle import mmsbm_oracle as orc
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    P, g, n0, n1, theta, pr = _problem(shape, K)
    ref = _problem_oracle(shape, K)
    what = "streamed K=%d %s" % (K, shape)
    eng = _engine(P, K, flags, g, n0, n1, theta, pr)
    t = eng.train
    rows16 = t.rows.cpu().pin_memory()
    rows8 = torch.empty(t.n_rows, dtype=torch.int64).pin_memory()
    assert lib.tip_rows_compact_host(rows16.data_ptr(), t.n_rows, rows8.data_ptr()) == 0, lib.tip_last_error()
    for compact, src in ((False, rows16), (True, rows8)):
        eng.em_step_host_rows(src, compact)
        torch.cuda.synchronize()
        assert eng.host_rows_arrived(), "%s: the streamed step reported a stall or a checksum mismatch" % what
        _check_stats(eng.stats.cpu().numpy(), family, P, K, pr, ref, "%s, %d-byte rows" % (what, 8 if compact else 16))
    assert eng.loglik("train") == pytest.approx(ref[3], rel=RTOL_LL), "tip_loglik, %s" % what
    eng.normalise()
    th, p = eng.get_params()
    th1, pr1 = orc.normalise_np(ref[0], ref[1], ref[2])
    assert _relerr(th, th1) < RTOL and _relerr(p, pr1) < RTOL, "M-step after the streamed step, %s" % what
    rows = np.ascontiguousarray(t.rows.cpu().numpy())
    deg = np.ascontiguousarray(eng.degrees().astype(np.int32))
    tho, pro = _oracle_iterations(shape, K, 2)
    for row_flags, src in ((0, rows), (_cabi.TIP_ROWS_COMPACT8, rows8.numpy())):
        th_h, p_h = np.ascontiguousarray(theta.copy()), np.ascontiguousarray(pr.copy())
        rc = lib.tip_em_iterations_host(P, K, src.ctypes.data, t.n_rows, t.n_rows_r0, deg.ctypes.data, th_h.ctypes.data,
                                        p_h.ctypes.data, 2, row_flags)
        assert rc == 0, lib.tip_last_error()
        assert _relerr(th_h, tho) < RTOL_ITER and _relerr(p_h, pro) < RTOL_ITER, \
            "tip_em_iterations_host, %s, row flags %d" % (what, row_flags)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [4, 7, 13, 25])
def test_hub_shaped_links_switch_on_the_l1_gather(torch_cuda, K):
    """EMEngine without flags on hub-shaped links of more than 640 genes picks TIP_EM_GATHER_L1 by itself: the default
    training path on screen-shaped data; two iterations against the oracle."""
    from oracle import mmsbm_oracle as orc
    from trigenicinteractionpredictor_b200 import synth
    from trigenicinteractionpredictor_b200.engine import EMEngine
    P, L = 700, {4: 6000, 7: 6000, 13: 2000, 25: 1500}[K]
    _, _, _, theta, pr = _random_problem(P, P, K, 900 + K)
    a, b, c, lab = synth.kuzmin_links_soa(P, L, seed=100 + K, n_query=6)
    g = np.stack([a, b, c], axis=1).astype(np.int32)
    g[:P, 0] = np.arange(P)
    n0, n1 = (1 - lab).astype(np.int32), lab.astype(np.int32)
    n0[3::31] += 2
    eng = EMEngine(P, K)
    eng.set_train_links(g[:, 0], g[:, 1], g[:, 2], n0, n1)
    assert eng.flags & TIP_EM_GATHER_L1, "hub-shaped links, P = %d: the L1 gather was not chosen (flags %d)" % (P, eng.flags)
    eng.set_params(theta, pr)
    eng.em_iteration()
    eng.em_iteration()
    th, p = eng.get_params()
    ids, cnt = g.astype(np.int64), np.stack([n0, n1], axis=1).astype(np.int64)
    tho, pro = theta, pr
    for _ in range(2):
        tho, pro = orc.em_step_np(tho, pro, ids, cnt)
    assert _relerr(th, tho) < RTOL_ITER and _relerr(p, pro) < RTOL_ITER


# ---------------------------------------------------------------------------------------------------------------------
# 2. completeness: the library's E-step kernels against MATRIX (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
ESTEP_KERNELS = ("em_fused_kernel", "seg3_pass_kernel", "seg3_finish_kernel", "em_finalize_kernel", "loglik_fused_kernel")
_TEMPLATE = re.compile(r"\b(%s)<([^>]*)>" % "|".join(ESTEP_KERNELS))


def _template_args(text):
    """'(int)7, (bool)1' (cu++filt) or '7, true' (the profiler's demangler) -> ('7', '1')."""
    out = []
    for arg in text.split(","):
        arg = re.sub(r"^\((?:unsigned )?(?:int|bool)\)", "", arg.strip())
        out.append({"true": "1", "false": "0"}.get(arg, arg))
    return tuple(out)


def _estep_kernels_in(names):
    """(kernel, template args) of every templated E-step kernel among demangled names."""
    found = set()
    for name in names:
        m = _TEMPLATE.search(name)
        if m:
            found.add((m.group(1), _template_args(m.group(2))))
    return found


def _family_of(kernel, args):
    """The family an em_fused / seg3_pass instantiation belongs to (None: no family knows it)."""
    if kernel == "em_fused_kernel":
        return FUSED_FAMILY.get(args[2:6])
    if kernel == "seg3_pass_kernel":
        return SLOT_FAMILY.get(args[2])
    return None


def _reached_by(kernel, args):
    """(K, families): the instantiation runs whenever a matrix entry of one of `families` at K runs."""
    K = int(args[0])
    if kernel in ("em_fused_kernel", "seg3_pass_kernel"):
        fam = _family_of(kernel, args)
        return K, {fam} if fam else set()
    if kernel == "seg3_finish_kernel":
        return K, set(SLOT_FAMILY.values())
    if kernel == "em_finalize_kernel":               # the per-gene finish of every fused K^3 launch, K = 5..16
        return K, set(FUSED_FAMILY.values())
    return K, {f for f, _, _ in MATRIX}              # loglik_fused_kernel: every case calls eng.loglik


def _library_kernel_names():
    from trigenicinteractionpredictor_b200 import _cabi, build
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    cufilt = shutil.which("cu++filt") or "/usr/local/cuda/bin/cu++filt"
    if not (os.path.exists(cuobjdump) and os.path.exists(cufilt)):
        pytest.skip("cuobjdump or cu++filt not available")
    build.build()
    out = subprocess.run([cuobjdump, "-res-usage", _cabi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    mangled = sorted(set(re.findall(r"Function (\S+?):", out)))
    assert mangled, "no kernels listed in %s" % _cabi.LIB_PATH
    dem = subprocess.run([cufilt], input="\n".join(mangled) + "\n", capture_output=True, text=True, check=True).stdout
    return dem.splitlines()


def test_every_instantiation_is_in_the_matrix():
    names = _library_kernel_names()
    insts = _estep_kernels_in(names)
    assert insts, "no templated E-step kernel found among the library's kernels"
    entries = {(f, K) for f, K, _ in MATRIX}
    untested = []
    for kernel, args in sorted(insts):
        K, fams = _reached_by(kernel, args)
        if not any((f, K) in entries for f in fams):
            untested.append("%s<%s>" % (kernel, ", ".join(args)))
    assert not untested, "instantiations no MATRIX entry runs (add a family / K): %s" % "; ".join(untested)
    launched = {(_family_of(k, a), int(a[0])) for k, a in insts if k in ("em_fused_kernel", "seg3_pass_kernel")}
    generic = any(re.search(r"\bgen_estep_kernel\b", n) for n in names)
    stale = [(f, K, fl) for f, K, fl in MATRIX if not (generic if f == "anyK" else (f, K) in launched)]
    assert not stale, "MATRIX entries without an instantiation in the library: %s" % stale


# ---------------------------------------------------------------------------------------------------------------------
# 3. the flags launch the family the matrix names
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flags_select_the_family_the_matrix_names(torch_cuda):
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    checked = 0
    for K in (7, 21):
        g, n0, n1, theta, pr = _random_problem(200, 1500, K, 60 + K)
        for family, _, flags in [e for e in MATRIX if e[1] == K]:
            eng = _engine(200, K, flags, g, n0, n1, theta, pr)
            if family == "stream":
                rows8 = torch.empty(eng.train.n_rows, dtype=torch.int64).pin_memory()
                rows16 = eng.train.rows.cpu().pin_memory()
                assert lib.tip_rows_compact_host(rows16.data_ptr(), eng.train.n_rows, rows8.data_ptr()) == 0
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                if family == "stream":
                    eng.em_step_host_rows(rows8, True)
                else:
                    eng.em_step()
                torch.cuda.synchronize()
            names = {e.name for e in prof.events()}
            if not any("kernel" in n for n in names):
                pytest.skip("torch.profiler recorded no CUDA kernels")
            found = _estep_kernels_in(names)
            fams = {_family_of(k, a) for k, a in found if k in ("em_fused_kernel", "seg3_pass_kernel")}
            ks = {int(a[0]) for _, a in found}
            what = "K=%d flags=%d (%s): %s" % (K, flags, family, sorted(found))
            if family == "anyK":
                assert any("gen_estep_kernel" in n for n in names) and not fams, what
            else:
                assert fams == {family} and ks == {K}, what
            if family.startswith("slot"):
                assert {a[1] for k, a in found if k == "seg3_pass_kernel"} == {"0", "1"}, "pass A and pass B + C, " + what
                assert ("seg3_finish_kernel", (str(K),)) in found, what
            checked += 1
    assert checked == len([e for e in MATRIX if e[1] in (7, 21)])


# ---------------------------------------------------------------------------------------------------------------------
# 4. link-set edges
# ---------------------------------------------------------------------------------------------------------------------
EDGE_FAMILIES = [("plain", 0), ("anyK", 1), ("fp32", 2), ("loglik", 4), ("gene_seg", 8), ("slot_l2", 32), ("slot_l1", 96)]
EDGE_K = [3, 10, 13, 16, 21]
_FAMILY_K = {}
for _f, _K, _fl in MATRIX:
    _FAMILY_K.setdefault(_f, set()).add(_K)
EDGE_ENTRIES = [(f, K, 0 if (f == "gene_seg" and K > 16) else fl) for K in EDGE_K for f, fl in EDGE_FAMILIES
                if f == "anyK" or K in _FAMILY_K[f]]
EDGES = ["rating0_only", "rating1_only", "fewest_tiles", "genes_without_links", "few_genes", "sparse_parameters"]


def _params(P, K, seed):
    rng = np.random.default_rng(seed)
    theta = rng.dirichlet(np.ones(K), size=P)
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    return theta, pr


def _edge_cases(edge, K):
    """(label, P, g, n0, n1, theta, pr, compare_parameters) of one edge."""
    L = max(_n_links(K) // 3, 600)
    if edge in ("rating0_only", "rating1_only"):
        # one rating block is empty: n_rows_r0 == n_rows or n_rows_r0 == 0 (K = 16 uploads one rating of p at a time)
        P = 200
        g, _, _, theta, pr = _random_problem(P, L, K, 11 + K)
        cnt = np.ones(L, dtype=np.int32)
        cnt[4::19] = 3
        zero = np.zeros(L, dtype=np.int32)
        n0, n1 = (cnt, zero) if edge == "rating0_only" else (zero, cnt)
        yield edge, P, g, n0, n1, theta, pr, True
    elif edge == "fewest_tiles":
        # 1 real row (one tile), 31 and 32 (one tile), 33 (two tiles, 31 padding rows), and 33 split over the ratings
        rng = np.random.default_rng(K)
        for n, rating in ((1, 0), (31, 0), (32, 0), (33, 0), (33, 1), (33, None)):
            P = max(n, 3)
            g = rng.integers(0, P, size=(n, 3)).astype(np.int32)
            g[:, 0] = np.arange(n)
            if n < 3:
                g[0] = (2, 0, 1)
            r = np.arange(n) % 2 if rating is None else np.full(n, rating)
            theta, pr = _params(P, K, n)
            yield "%d rows, rating %s" % (n, "both" if rating is None else rating), P, g, \
                (1 - r).astype(np.int32), r.astype(np.int32), theta, pr, True
    elif edge == "genes_without_links":
        # ids from a subset of the genes: the others have no link, their Ntheta rows must be exactly 0 (no M-step: it
        # divides by their degree)
        P = 300
        rng = np.random.default_rng(K)
        used = np.sort(rng.choice(250, size=150, replace=False))
        g = used[rng.integers(0, used.size, size=(L, 3))].astype(np.int32)
        g[: used.size, 0] = used
        lab = (rng.random(L) < 0.2).astype(np.int32)
        theta, pr = _params(P, K, K)
        yield "150 of %d genes linked" % P, P, g, 1 - lab, lab, theta, pr, False
    elif edge == "few_genes":
        # below and just above the prep kernel's 16 genes per CTA, the finish kernel's 8-gene groups and 96-gene chunks
        for P in (3, 17, 97):
            g, n0, n1, theta, pr = _random_problem(P, L, K, P)
            n0 = n0.copy()
            n0[::7] += 1
            yield "P=%d" % P, P, g, n0, n1, theta, pr, True
        # every link the same triplet: one run of equal genes through every tile of every order
        g = np.tile(np.array([[2, 0, 1]], dtype=np.int32), (L, 1))
        rng = np.random.default_rng(K)
        n0 = rng.integers(0, 3, size=L).astype(np.int32)
        n1 = rng.integers(0, 2, size=L).astype(np.int32)
        n0[n0 + n1 == 0] = 1
        theta, pr = _params(3, K, 5)
        yield "one triplet", 3, g, n0, n1, theta, pr, True
    elif edge == "sparse_parameters":
        # one-hot theta rows, rows with exact zeros, p cells at exactly 0 or 1; two links whose three genes are one-hot on a
        # cell where p of their rating is 0: d = eps, s = n / d = 1e10
        P = 300
        g, n0, n1, theta, pr = _random_problem(P, L, K, 31 + K)
        rng = np.random.default_rng(K)
        hot = np.arange(0, P, 3)
        comp = rng.integers(0, K, size=P)
        theta[hot] = 0.0
        theta[hot, comp[hot]] = 1.0
        if K > 2:
            part = np.setdiff1d(np.arange(1, P, 5), hot)
            theta[part, : K // 2] = 0.0
            theta[part] /= theta[part].sum(axis=1, keepdims=True)
        cell = rng.random((K, K, K))
        pr[cell < 0.25] = (1.0, 0.0)
        pr[(cell >= 0.25) & (cell < 0.5)] = (0.0, 1.0)
        extra_g, extra_n0, extra_n1 = [], [], []
        for trip, r in (((0, 3, 6), 1), ((9, 12, 15), 0)):
            c = tuple(comp[list(trip)])
            if r == 0 and c == tuple(comp[[0, 3, 6]]):
                continue                                 # same cell as the first link: it cannot take both zeros
            pr[c] = (1.0, 0.0) if r == 1 else (0.0, 1.0)
            extra_g.append(trip)
            extra_n0.append(1 - r)
            extra_n1.append(r)
        g = np.concatenate([g, np.array(extra_g, dtype=np.int32)])
        n0 = np.concatenate([n0, np.array(extra_n0, dtype=np.int32)])
        n1 = np.concatenate([n1, np.array(extra_n1, dtype=np.int32)])
        yield "one-hot theta, p in {0, 1}", P, g, n0, n1, theta, pr, True


@pytest.mark.gpu
@pytest.mark.parametrize("edge", EDGES)
@pytest.mark.parametrize("family,K,flags", EDGE_ENTRIES, ids=_ids(EDGE_ENTRIES))
def test_link_set_edges(torch_cuda, family, K, flags, edge):
    for label, P, g, n0, n1, theta, pr, params in _edge_cases(edge, K):
        ref = _oracle(theta, pr, g, n0, n1)
        what = "%s K=%d flags=%d, %s: %s" % (family, K, flags, edge, label)
        eng = _check_step(family, flags, P, K, g, n0, n1, theta, pr, ref, what, params=params)
        t = eng.train
        if edge == "rating0_only":
            assert t.n_rows_r0 == t.n_rows > 0
        elif edge == "rating1_only":
            assert t.n_rows_r0 == 0 and t.n_rows > 0
        elif edge == "genes_without_links":
            nth = eng.stats.cpu().numpy()[: P * K].reshape(P, K)
            idle = ref[2] == 0
            assert idle.sum() == P - 150 and np.all(nth[idle] == 0.0), what
        elif edge == "sparse_parameters":
            from oracle import mmsbm_oracle as orc
            d = orc.EPS + orc.denominators_np(theta, pr, g.astype(np.int64))
            assert ((d == orc.EPS) & (np.stack([n0, n1], axis=1) > 0)).any(), "no link with d = eps: " + what
