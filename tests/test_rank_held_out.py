"""Ranks of held-out triplets among all unseen triplets (tip_score_histogram, EMEngine.score_histogram,
Model.rank_held_out, predict --held-out).

The oracle orders the universe U (every triplet of the candidates that is not a train key) with the exhaustive
`top_triplets_np` of tests/test_predict.py (pinned to oracle.mmsbm_oracle.predict_loops); a test triplet's rank is its
position + 1.  Device ranks may differ from the oracle's only inside runs of near-equal oracle scores (within 1e-12)."""
import ctypes
import itertools
import os
import random
import shutil
import subprocess
from math import comb

import numpy as np
import pytest

from tests.test_predict import BASE, TOL, _digested, _trained_base_model, check_against_oracle, pack_ranks, random_params, \
    top_triplets_np

MASK = np.uint64((1 << 21) - 1)


def universe_oracle(thetas, prs, cand, train):
    """(scores [|U|], packed ranks [|U|]) of U in the exact order: mean score descending, packed ranks ascending."""
    nc = len(cand)
    _, sc, k = top_triplets_np(thetas, prs, cand, train, max(comb(nc, 3), 1))
    return sc, k


def near_tie_runs(sc):
    """(first, last) 1-based rank of the run of near-equal scores that holds each position."""
    if len(sc) == 0:
        return np.empty(0, dtype=np.int64), np.empty(0, dtype=np.int64)
    brk = np.concatenate([[True], np.abs(sc[1:] - sc[:-1]) > TOL * np.abs(sc[:-1])])
    rid = np.cumsum(brk) - 1
    starts = np.flatnonzero(brk)
    ends = np.concatenate([starts[1:], [len(sc)]]) - 1
    return starts[rid] + 1, ends[rid] + 1


def key_of(ids):
    return "_".join(sorted(str(int(x)) for x in ids))


def synthetic_model(P, train, test):
    """A Model digested from dicts: genes G000.. with ids 0..P-1; train / test: {key: label}."""
    from trigenicinteractionpredictor_b200 import Model
    m = Model()
    m.P = P
    m.id_gene = {i: "G%04d" % i for i in range(P)}
    m.gene_id = {v: k for k, v in m.id_gene.items()}
    m.links = {k: [1 - lab, lab] for k, lab in train.items()}
    m.test_links = {k: [1 - lab, lab] for k, lab in test.items()}
    m._links_version += 1
    return m


def random_keys(rng, P, m):
    out = {}
    while len(out) < m:
        out[key_of(rng.choice(P, size=3, replace=False))] = int(rng.random() < 0.3)
    return out


def packed_of_key(key, rank):
    r = sorted(rank[int(x)] for x in key.split("_"))
    return (r[0] << 42) | (r[1] << 21) | r[2]


def oracle_case(rng, P, K, S, n_train, n_test, n_both=5):
    thetas, prs = random_params(rng, P, K, S)
    train = random_keys(rng, P, n_train)
    test = {k: lab for k, lab in random_keys(rng, P, n_test).items() if k not in train}
    for k in list(train)[:n_both]:
        test[k] = 1                                   # test keys that are also train keys: excluded
    m = synthetic_model(P, train, test)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    rank = {int(g): r for r, g in enumerate(cand.tolist())}
    train_packed = np.unique(np.array([packed_of_key(k, rank) for k in train], dtype=np.uint64))
    sc, k = universe_oracle(thetas, prs, cand, train_packed)
    first, last = near_tie_runs(sc)
    where = {int(x): i for i, x in enumerate(k.tolist())}
    return m, list(zip(thetas, prs)), train, test, rank, sc, k, first, last, where


def check_rows(res, rank, where, first, last, exact_upto):
    """Every interval meets the oracle's near-tie run of its triplet; ranks <= exact_upto are exact."""
    for key, names, label, score, lo, hi in res["rows"]:
        i = where[packed_of_key(key, rank)]
        assert lo <= hi and lo <= last[i] and hi >= first[i], (key, lo, hi, first[i], last[i])
        if last[i] <= exact_upto:
            assert lo == hi
        if lo == hi and lo <= exact_upto:
            assert first[i] <= lo <= last[i]


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_universe_oracle_equals_itertools_brute_force(S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(70 + S)
    P, K = 14, 3
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str))
    train = pack_ranks([0, 2, 5, 1], [1, 7, 6, 12], [13, 9, 11, 13])
    sc, k = universe_oracle(thetas, prs, cand, train)
    tl, pl = [t.tolist() for t in thetas], [p.tolist() for p in prs]
    rows = []
    for ra, rb, rc in itertools.combinations(range(P), 3):
        pk = (ra << 42) | (rb << 21) | rc
        if pk in set(int(x) for x in train.tolist()):
            continue
        x, y, z = (int(cand[i]) for i in (ra, rb, rc))
        rows.append((-sum(orc.predict_loops(t, p, x, y, z) for t, p in zip(tl, pl)) / S, pk))
    rows.sort()
    assert len(rows) == len(sc) == comb(P, 3) - 4
    bf_sc = -np.array([r[0] for r in rows])
    bf_k = np.array([r[1] for r in rows], dtype=np.uint64)
    ids = lambda kk: np.stack([(kk >> np.uint64(42)) & MASK, (kk >> np.uint64(21)) & MASK, kk & MASK], 1)  # noqa: E731
    check_against_oracle(ids(k), sc, ids(bf_k), bf_sc, len(rows))


def _restated_bins(values, L, NB, E):
    """The bin rule restated with frexp / ldexp instead of bit operations (non-negative values)."""
    out = []
    B = 1 << L
    key_top = ((E + 1) << L) - 1
    for v in np.asarray(values, dtype=np.float64).tolist():
        if v == 0.0:
            key = 0
        elif v < 2.0 ** -1022:                                   # subnormal: exponent field 0
            key = int(np.floor(np.ldexp(v, 1074 - 52 + L)))
        elif np.isinf(v):
            key = 2047 << L
        else:
            mant, ex = np.frexp(v)                              # v = mant 2^ex, mant in [0.5, 1)
            key = ((ex - 1 + 1023) << L) + int(np.floor((2.0 * mant - 1.0) * B))
        if key > key_top:
            out.append(0)
        elif key_top - key < NB * B:
            out.append(1 + key_top - key)
        else:
            out.append(NB * B + 1)
    return np.array(out)


@pytest.mark.parametrize("L,NB,E", [(7, 64, 1022), (7, 64, 40), (3, 4, 1023), (0, 1, 1000), (10, 16, 5), (7, 64, 2046)])
def test_host_bins_match_restatement(L, NB, E):
    from trigenicinteractionpredictor_b200.engine import BinLayout
    lay = BinLayout(L, NB, E)
    vals = [0.0, 5e-324, 2.0 ** -1074 * 3, 2.0 ** -1023, np.nextafter(2.0 ** -1022, 0), 2.0 ** -1022, 1.0, 0.75, np.inf]
    for e in range(E - 1023 - NB - 2, E - 1023 + 3):
        if -1074 <= e <= 1023:
            p = np.ldexp(1.0, e)
            vals += [p, np.nextafter(p, 0), np.nextafter(p, np.inf), p * (1 + 2.0 ** -L), np.nextafter(p * (1 + 2.0 ** -L), 0)]
    top = np.ldexp(1.0, E - 1023 + 1) if E < 2046 else np.finfo(np.float64).max   # the bound's binade ends below this
    vals += [np.nextafter(top, 0), top, np.finfo(np.float64).max]
    rng = np.random.default_rng(L * 100 + NB)
    vals += (rng.random(300) * 2.0 ** rng.integers(-60, 4, 300)).tolist()
    vals = np.array(vals, dtype=np.float64)
    got = lay.bins(vals)
    assert np.array_equal(got, _restated_bins(vals, L, NB, E))
    assert got.min() >= 0 and got.max() <= lay.n_bins - 1
    first, last = lay.bins_widened(vals)
    assert np.all(first <= got) and np.all(got <= last) and np.all(last - first <= 1)


def test_workspace_bytes_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_score_histogram_workspace_bytes(100, 10, 2, 7, 64, ctypes.byref(nb)) == 0 and nb.value > 0
    for args in [(100, 10, 39, 7, 64),        # S K = 390 > 384
                 (100, 2, 1, 11, 4),          # log2_bins > 10
                 (100, 2, 1, 7, 0),           # no binade
                 (100, 2, 1, 7, 129),         # 129 * 128 bins > 2^14
                 ((1 << 21) + 1, 2, 1, 7, 64), (100, 0, 1, 7, 64), (100, 2, 0, 7, 64), (100, 2, 1, -1, 64)]:
        assert lib.tip_score_histogram_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"S*K <= 384" in lib.tip_last_error() and b"n_binades * 2^log2_bins <= 16384" in lib.tip_last_error()
    assert lib.tip_score_histogram_workspace_bytes(1 << 21, 2, 1, 7, 128, ctypes.byref(nb)) == 0


def test_model_refusals():
    random.seed(2)
    m = _digested()
    m.initialize_parameters(2)
    with pytest.raises(ValueError, match="unknown gene names: NOPE1, NOPE2"):
        m.rank_held_out(10, genes=[m.id_gene[0], "NOPE1", "NOPE2"])
    with pytest.raises(ValueError, match="n_exact must be in"):
        m.rank_held_out(-1)
    with pytest.raises(ValueError, match="rank_held_out: params is empty"):
        m.rank_held_out(10, params=[])
    th = np.asarray(m.theta)
    with pytest.raises(ValueError, match="K = 1, the model has K = 2"):
        m.rank_held_out(10, params=[(th[:, :1], np.asarray(m.pr)[:1, :1, :1])])
    t2, p2 = random_params(np.random.default_rng(0), m.P, 2, 1)
    t3, p3 = random_params(np.random.default_rng(1), m.P, 3, 1)
    with pytest.raises(ValueError, match="rank_held_out: the parameter sets have different K"):
        _digested().rank_held_out(10, params=[(t2[0], p2[0]), (t3[0], p3[0])])
    m.test_links = {}
    with pytest.raises(ValueError, match="rank_held_out: the model has no test links"):
        m.rank_held_out(10)
    from trigenicinteractionpredictor_b200 import Model
    with pytest.raises(ValueError, match="rank_held_out needs a model digested"):
        Model().rank_held_out(10)


def test_cli_held_out_refusals(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    base = ["-t", tr, "-e", te, "-p", good, "--held-out"]
    qf = tmp_path / "q.txt"
    qf.write_text("%s\n" % m.id_gene[0])
    for extra in (["-q", str(qf)], ["-r", str(qf)], ["--include-known"]):
        assert main(base + extra) == 2
        assert "--held-out excludes" in capsys.readouterr().err
    assert main(base + ["-n", "-1"]) == 2
    assert ">= 0 with --held-out" in capsys.readouterr().err
    assert main(base + ["-n", "x"]) == 2
    assert "--top must be an integer" in capsys.readouterr().err


def test_sass_hist_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    body = [f for f in out.split("Function : ") if f.split("\n", 1)[0].find("tip_hist_pass_kernel") >= 0]
    assert len(body) == 1 and "DMMA.8x8x4" in body[0]


# ----------------------------------------------------------------------------------------------
# GPU tests
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _engine(P, K):
    from trigenicinteractionpredictor_b200.engine import EMEngine
    return EMEngine(P, K, device="cuda:0")


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("K", [1, 2, 3, 4, 10, 32])
@pytest.mark.parametrize("P", [40, 130])
def test_exact_ranks_match_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(P * 100 + K * 10 + S + 5)
    m, sets, train, test, rank, sc, k, first, last, where = oracle_case(rng, P, K, S, 3 * P, P + 60)
    res = m.rank_held_out(n_exact=comb(P, 3), params=sets, recall_at=(1, 10, len(sc)))
    assert res["universe"] == len(sc) == comb(P, 3) - len(train)
    assert res["excluded_train"] == 5 and res["excluded_genes"] == 0
    assert res["positives"] + res["negatives"] == len(test) - 5 == len(res["rows"])
    check_rows(res, rank, where, first, last, len(sc))
    assert all(lo == hi for *_, lo, hi in res["rows"])
    for key, names, label, score, lo, hi in res["rows"]:
        i = where[packed_of_key(key, rank)]
        assert abs(score - sc[i]) <= TOL * sc[i]
        assert label == test[key] and names == "_".join(sorted(m.id_gene[int(x)] for x in key.split("_")))
    los = [r[4] for r in res["rows"]]
    assert los == sorted(los)
    assert res["recall_at"][len(sc)]["positives"] in (None, (1.0, 1.0))


@pytest.mark.gpu
@pytest.mark.parametrize("K,S", [(4, 2), (10, 1), (32, 3)])
def test_intervals_contain_the_rank(torch_cuda, K, S):
    P = 130
    rng = np.random.default_rng(900 + K + S)
    m, sets, train, test, rank, sc, k, first, last, where = oracle_case(rng, P, K, S, 3000, 400)
    for n_exact in (0, 1, 10):
        res = m.rank_held_out(n_exact=n_exact, params=sets, recall_at=(1, 10, 1000, len(sc)))
        assert res["n_exact"] == n_exact and res["universe"] == len(sc)
        check_rows(res, rank, where, first, last, n_exact)
        lo = np.array([r[4] for r in res["rows"]])
        hi = np.array([r[5] for r in res["rows"]])
        assert np.all(lo[lo != hi] > n_exact) and np.all(hi <= len(sc))
        assert res["recall_at"][len(sc)]["positives"] == (1.0, 1.0)
        for N in (1, 10):
            r = res["recall_at"][N]["positives"]
            assert N > n_exact or r[0] == r[1]
        a_lo, a_hi = res["auc"]
        assert 0.0 <= a_lo <= a_hi <= 1.0
    # the histogram: all C(n, 3) scores, and bin by bin the oracle's sums except within 2^-40 of an edge
    thetas, prs = np.stack([s[0] for s in sets]), np.stack([s[1] for s in sets])
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    lay, hist = _engine(P, K).score_histogram(thetas, prs, cand)
    assert int(hist.sum()) == comb(P, 3)
    _, all_sc, _ = top_triplets_np(thetas, prs, cand, [], comb(P, 3))
    sums = all_sc * S
    f, l_ = lay.bins_widened(sums)
    edge = int((f != l_).sum())
    assert int(np.abs(hist - np.bincount(lay.bins(sums), minlength=lay.n_bins)).sum()) <= 2 * edge
    assert hist[0] == 0                                    # nothing above the bound


@pytest.mark.gpu
def test_histogram_at_the_sk_limit(torch_cuda):
    """S K = 384: the largest Q tile plus 8 194 bins still fit one block's shared memory."""
    P, K, S = 50, 32, 12
    rng = np.random.default_rng(384)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    lay, hist = _engine(P, K).score_histogram(np.stack(thetas), np.stack(prs), cand)
    assert int(hist.sum()) == comb(P, 3) and lay.n_bins == 64 * 128 + 2
    _, all_sc, _ = top_triplets_np(thetas, prs, cand, [], comb(P, 3))
    f, l_ = lay.bins_widened(all_sc * S)
    assert int(np.abs(hist - np.bincount(lay.bins(all_sc * S), minlength=lay.n_bins)).sum()) <= 2 * int((f != l_).sum())


@pytest.mark.gpu
def test_consistent_with_predict_top_triplets_including_known(torch_cuda):
    P, K, S = 60, 3, 2
    rng = np.random.default_rng(61)
    m, sets, train, test, rank, sc, k, first, last, where = oracle_case(rng, P, K, S, 400, 150)
    res = m.rank_held_out(n_exact=comb(P, 3), params=sets)
    got = {r[0]: r[4] for r in res["rows"]}
    rows = m.predict_top_triplets(comb(P, 3), exclude_known=False, params=sets)
    n_train_before = 0
    seen = 0
    for i, (s, key, names) in enumerate(rows):
        if key in got:
            assert got[key] == i + 1 - n_train_before
            seen += 1
        if key in train:
            n_train_before += 1
    assert seen == len(got)


@pytest.mark.gpu
def test_all_scores_tied(torch_cuda):
    """Identical theta rows and dyadic parameters: every score is the same number, ranks follow packed-rank order."""
    P, K = 70, 3
    theta = np.tile(np.array([0.5, 0.25, 0.25]), (P, 1))
    rng = np.random.default_rng(3)
    p1 = rng.integers(1, 4, size=(K, K, K)) / 4.0
    pr = np.stack([1.0 - p1, p1], axis=3)
    train = random_keys(rng, P, 300)
    test = {k: lab for k, lab in random_keys(rng, P, 120).items() if k not in train}
    m = synthetic_model(P, train, test)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    rank = {int(g): r for r, g in enumerate(cand.tolist())}
    tp = np.sort(np.array([packed_of_key(k, rank) for k in train], dtype=np.uint64))
    universe = comb(P, 3) - len(train)
    every = np.sort(pack_ranks(*np.array(list(itertools.combinations(range(P), 3))).T))
    lay, hist = _engine(P, K).score_histogram(theta[None], pr[None], cand)
    assert np.count_nonzero(hist) == 1 and int(hist.sum()) == comb(P, 3)
    for n_exact in (0, 50, universe):
        res = m.rank_held_out(n_exact=n_exact, params=[(theta, pr)])
        for key, names, label, score, lo, hi in res["rows"]:
            pk = packed_of_key(key, rank)
            want = 1 + int(np.searchsorted(every, np.uint64(pk))) - int(np.searchsorted(tp, np.uint64(pk)))
            if want <= n_exact:
                assert lo == hi == want
            else:
                assert lo == max(1, n_exact + 1) and hi == universe     # one bin: the interval is everything below the list


@pytest.mark.gpu
def test_excluded_test_keys(torch_cuda):
    P, K = 50, 3
    rng = np.random.default_rng(17)
    m, sets, train, test, rank, sc, k, first, last, where = oracle_case(rng, P, K, 1, 200, 80, n_both=7)
    genes = [m.id_gene[i] for i in range(0, P, 2)]          # half the genes
    res = m.rank_held_out(n_exact=1000, genes=genes, params=sets)
    ids = set(range(0, P, 2))
    outside = sum(1 for key in test if not {int(x) for x in key.split("_")} <= ids)
    both = sum(1 for key in test if key in train and {int(x) for x in key.split("_")} <= ids)
    assert res["excluded_genes"] == outside and res["excluded_train"] == both
    assert len(res["rows"]) == len(test) - outside - both
    n = len(genes)
    n_train_in = sum(1 for key in train if {int(x) for x in key.split("_")} <= ids)
    assert res["universe"] == comb(n, 3) - n_train_in
    cand = np.array(sorted(ids, key=str), dtype=np.int32)
    crank = {int(g): r for r, g in enumerate(cand.tolist())}
    tp = np.unique(np.array([packed_of_key(kk, crank) for kk in train if {int(x) for x in kk.split("_")} <= ids],
                            dtype=np.uint64))
    o_sc, o_k = universe_oracle([s[0] for s in sets], [s[1] for s in sets], cand, tp)
    f, l_ = near_tie_runs(o_sc)
    check_rows(res, crank, {int(x): i for i, x in enumerate(o_k.tolist())}, f, l_, 1000)


@pytest.mark.gpu
def test_p1500_histogram_against_tip_score(torch_cuda):
    """5.6e8 triplets: the histogram bin by bin against every score through tip_score in chunks, binned on the host;
    counts differ only by the scores within 2^-40 of a bin edge."""
    torch = torch_cuda
    P, K = 1500, 4
    rng = np.random.default_rng(1500)
    thetas, prs = random_params(rng, P, K, 1)
    cand_np = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    lay, hist = eng.score_histogram(np.stack(thetas), np.stack(prs), cand_np)
    assert int(hist.sum()) == comb(P, 3)
    eng.set_params(thetas[0], prs[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)
    direct = np.zeros(lay.n_bins, dtype=np.int64)
    edge = 0
    j = 1
    while j < P - 1:
        js, size = [], 0
        while j < P - 1 and size < 8_000_000:
            js.append(j)
            size += j * (P - 1 - j)
            j += 1
        parts = []
        for jj in js:
            A, C = torch.meshgrid(torch.arange(jj, device=dev), torch.arange(jj + 1, P, device=dev), indexing="ij")
            parts.append(torch.stack([A.reshape(-1), torch.full((A.numel(),), jj, device=dev), C.reshape(-1)], 1))
        g = cand[torch.cat(parts)].to(torch.int32)
        g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
        out = torch.empty(g.shape[0], dtype=torch.float64, device=dev)
        assert eng.lib.tip_score(P, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()),
                                 ctypes.c_void_p(g3.data_ptr()), g.shape[0], ctypes.c_void_p(eng.theta.data_ptr()),
                                 ctypes.c_void_p(eng.p.data_ptr()), ctypes.c_void_p(out.data_ptr()), eng._stream()) == 0
        s = out.cpu().numpy()
        direct += np.bincount(lay.bins(s), minlength=lay.n_bins)
        f, l_ = lay.bins_widened(s)
        edge += int((f != l_).sum())
    diff = int(np.abs(hist - direct).sum())
    print("p1500: %d of %d scores within 2^-40 of a bin edge; histogram differs by %d" % (edge, comb(P, 3), diff))
    assert diff <= 2 * edge and edge < 10_000


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3])
def test_golden_base(torch_cuda, K):
    m = _trained_base_model(K)
    cand = np.array(sorted(range(m.P), key=str), dtype=np.int32)
    U = comb(m.P, 3) - len(m._train_packed(cand))
    res = m.rank_held_out(n_exact=500, recall_at=(10, 500, U))
    assert res["universe"] == U
    assert res["positives"] + res["negatives"] + res["excluded_train"] + res["excluded_genes"] == len(m.test_links)
    assert res["recall_at"][U]["positives"] == (1.0, 1.0) and res["recall_at"][U]["negatives"] == (1.0, 1.0)
    r10 = res["recall_at"][10]["positives"]
    assert r10[0] == r10[1]
    for key, names, label, score, lo, hi in res["rows"][:50]:
        a, b, c = key.split("_")
        assert abs(score - m.do_prediction(a, b, c)) <= TOL * score
        assert label == (0 if m.test_links[key][0] else 1)
    th, pr = np.array(m.theta), np.array(m.pr)
    rank = {int(g): r for r, g in enumerate(cand.tolist())}
    sc, k = universe_oracle([th], [pr], cand, m._train_packed(cand))
    f, l_ = near_tie_runs(sc)
    check_rows(res, rank, {int(x): i for i, x in enumerate(k.tolist())}, f, l_, 500)


@pytest.mark.gpu
def test_train_with_save_params_then_predict_cli_held_out(torch_cuda, tmp_path):
    from trigenicinteractionpredictor_b200 import Model, main
    from trigenicinteractionpredictor_b200.predict import main as predict_main
    out = str(tmp_path) + os.sep
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["-t", tr, "-e", te, "-k", "2", "-i", "300", "-f", "5", "-b", "10", "-n", "2", "-o", out,
                 "--seed", "1000", "--save-params"]) == 0
    pred = str(tmp_path / "held.tsv")
    params = [out + "Sample_0_K2.npz", out + "Sample_1_K2.npz"]
    assert predict_main(["-t", tr, "-e", te, "-p", params[0], "-p", params[1], "--held-out", "-n", "2000", "-o", pred]) == 0
    text = open(pred, encoding="utf-8").read().split("\n")
    hdr = text.index("Rank\tPredicted Interaction\tReal Interaction\tID of genes\tGenes")
    summary = dict(line.split(":\t") for line in text[:hdr])
    mm = Model()
    mm.get_traintest(tr, te)
    U = comb(mm.P, 3) - len(mm._train_packed(np.array(sorted(range(mm.P), key=str), dtype=np.int32)))
    want = mm.rank_held_out(n_exact=2000, params=params, recall_at=(100, 1000, 10000, 100000, U))
    assert int(summary["Universe size"]) == U and int(summary["Exactly ranked"]) == 2000
    assert int(summary["Ranked positives"]) == want["positives"] and int(summary["Ranked negatives"]) == want["negatives"]
    for N in (100, 1000):                                      # below n_exact: exact values
        assert float(summary["Recall at %d" % N]) == want["recall_at"][N]["positives"][0]
    lo, hi = (float(x) for x in (summary["Universe AUC"].split("-") + [summary["Universe AUC"]])[:2])
    assert 0.0 <= lo <= hi <= 1.0
    assert want["recall_at"][U]["positives"] == (1.0, 1.0)
    body = [ln.split("\t") for ln in text[hdr + 1:] if ln]
    assert len(body) == want["positives"] + want["negatives"]
    assert [b[3] for b in body] == [r[0] for r in want["rows"]]
    for b, r in zip(body, want["rows"]):
        assert b[0] == (str(r[4]) if r[4] == r[5] else "%d-%d" % (r[4], r[5])) and float(b[1]) == r[3] and int(b[2]) == r[2]
