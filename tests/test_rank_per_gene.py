"""Ranks of held-out triplets among their query gene's unseen triplets (tip_rank_per_gene, EMEngine.rank_per_gene,
Model.rank_held_out_per_gene, predict --held-out-genes).

The oracle scores every pair of other candidates of a query with numpy: per region of the query's slot a K x K matrix of
the query, th_x^T M th_y (pinned to oracle.mmsbm_oracle.predict_loops by an itertools brute force), drops the train keys
and orders the rest by (score descending, packed ranks ascending); a test triplet's rank is its position + 1.  Device
ranks may differ from the oracle's only inside runs of near-equal oracle scores (within 1e-12), as in
tests/test_rank_per_pair.py.  Against tip_top_triplets_per_gene, which computes every score at the same place of the same
tile, ranks and score bits must agree exactly."""
import ctypes
import itertools
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from tests.test_predict import BASE, TOL, _digested, _trained_base_model, pack_ranks, random_params
from tests.test_rank_held_out import key_of, near_tie_runs, packed_of_key, random_keys, synthetic_model


def gene_oracle(thetas, prs, cand, train, r):
    """(packed ranks, mean scores) of the universe of the query of rank r, in rank order."""
    n = len(cand)
    others = np.array([x for x in range(n) if x != r], dtype=np.int64)
    if len(others) < 2:
        return np.empty(0, np.uint64), np.empty(0)
    iu, iv = np.triu_indices(len(others), 1)
    u, v = others[iu], others[iv]
    g = np.where(v < r, 0, np.where(u < r, 1, 2))
    s = np.zeros(len(u))
    cand = np.asarray(cand, dtype=np.int64)
    for th, pr in zip(thetas, prs):
        th = np.asarray(th, dtype=np.float64)[cand]
        p1, t = np.asarray(pr)[..., 1], th[r]
        M = [np.einsum("xyz,z->xy", p1, t), np.einsum("xyz,y->xz", p1, t), np.einsum("xyz,x->yz", p1, t)]
        for k in range(3):
            sel = g == k
            s[sel] += np.einsum("ix,xy,iy->i", th[u[sel]], M[k], th[v[sel]])
    s /= len(thetas)
    tri = np.sort(np.stack([u, v, np.full(len(u), r)], 1), 1)
    packed = pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2])
    keep = ~np.isin(packed, np.asarray(train, dtype=np.uint64))
    packed, s = packed[keep], s[keep]
    order = np.lexsort((packed, -s))
    return packed[order], s[order]


class Oracle:
    """Per-query oracles of a candidate list, cached: rank interval (near-tie run) and score of a triplet."""

    def __init__(self, thetas, prs, cand, train):
        self.args = (thetas, prs, np.asarray(cand), train)
        self.cache = {}

    def get(self, r):
        if r not in self.cache:
            packed, s = gene_oracle(*self.args, r)
            first, last = near_tie_runs(s)
            self.cache[r] = ({int(x): i for i, x in enumerate(packed.tolist())}, s, first, last)
        return self.cache[r]

    def check(self, r, packed, rank, score, universe):
        where, s, first, last = self.get(r)
        assert universe == len(s)
        i = where[packed]
        assert first[i] <= rank <= last[i], (r, packed, rank, first[i], last[i])
        assert abs(score - s[i]) <= TOL * s[i]


def check_model_result(m, res, sets, genes_ids=None):
    """Every view of a Model.rank_held_out_per_gene result against the oracle."""
    ids = sorted(range(m.P) if genes_ids is None else genes_ids, key=str)
    cand = np.array(ids, dtype=np.int32)
    rank = {int(g): r for r, g in enumerate(ids)}
    orc = Oracle([s[0] for s in sets], [s[1] for s in sets], cand, m._train_packed(cand))
    for gene, key, names, label, score, rk, universe in res["rows"]:
        q = rank[m.gene_id[gene]]
        assert q in [rank[int(x)] for x in key.split("_")]
        orc.check(q, packed_of_key(key, rank), rk, score, universe)
        assert names == "_".join(sorted(m.id_gene[int(x)] for x in key.split("_")))
        assert label == (0 if m.test_links[key][0] else 1)
    return orc


def _engine(P, K):
    from trigenicinteractionpredictor_b200.engine import EMEngine
    return EMEngine(P, K, device="cuda:0")


def check_against_per_gene(eng, thetas, prs, cand, qr, train, tq, tu, tv):
    """rank_per_gene against top_triplets_per_gene(known = train, n = C(n - 1, 2)) on the same queries: exact ranks and
    score bits."""
    n = len(cand)
    rank, score, universe = eng.rank_per_gene(thetas, prs, cand, qr, train, tq, tu, tv)
    ids, sc, counts = eng.top_triplets_per_gene(thetas, prs, cand, qr, train, (n - 1) * (n - 2) // 2)
    rk = {int(g): r for r, g in enumerate(np.asarray(cand).tolist())}
    pos = []
    for q in range(len(qr)):
        assert universe[q] == counts[q]
        pos.append({tuple(sorted(rk[int(x)] for x in row)): (k, s) for k, (row, s) in
                    enumerate(zip(ids[q, :counts[q]].tolist(), sc[q, :counts[q]].tolist()))})
    tset = set(int(x) for x in np.asarray(train, dtype=np.uint64).tolist())
    for j in range(len(tq)):
        q = int(tq[j])
        x, y, z = sorted((int(qr[q]), int(tu[j]), int(tv[j])))
        if (x << 42) | (y << 21) | z in tset:
            assert rank[j] == 0
            continue
        k, s = pos[q][(x, y, z)]
        assert rank[j] == k + 1, (j, q, (x, y, z), rank[j], k + 1)
        assert np.float64(score[j]).view(np.int64) == np.float64(s).view(np.int64)
    return rank, score, universe


def _train_of_query(rng, n, r, m, exclude=()):
    """m distinct packed train keys that contain rank r, and the pairs they use."""
    others = [x for x in range(n) if x != r]
    pairs = set()
    while len(pairs) < m:
        u, v = sorted(rng.choice(others, 2, replace=False).tolist())
        if (u, v) not in exclude:
            pairs.add((u, v))
    keys = [pack_ranks(*sorted((r, u, v))) for u, v in pairs]
    return np.array(keys, dtype=np.uint64), pairs


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_gene_oracle_equals_itertools_brute_force(S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(50 + S)
    P, K = 16, 3
    thetas, prs = random_params(rng, P, K, S)
    # ties on the packed ranks: genes 0 and 1 share theta, so pairs that differ only by them score the same
    for th in thetas:
        th[1] = th[0]
    cand = np.array(sorted(range(P), key=str))
    train = np.sort(pack_ranks([0, 2, 5, 1, 3, 0], [1, 7, 6, 3, 4, 5], [13, 9, 11, 13, 15, 6]))
    tset = set(int(x) for x in train.tolist())
    tl, pl = [t.tolist() for t in thetas], [p.tolist() for p in prs]
    for r in [0, 5, 7, P - 1]:
        packed, s = gene_oracle(thetas, prs, cand, train, r)
        rows = []
        for u, v in itertools.combinations([x for x in range(P) if x != r], 2):
            x, y, z = sorted((r, u, v))
            pk = (x << 42) | (y << 21) | z
            if pk in tset:
                continue
            gx, gy, gz = (int(cand[i]) for i in (x, y, z))
            rows.append((-sum(orc.predict_loops(t, p, gx, gy, gz) for t, p in zip(tl, pl)) / S, pk))
        rows.sort()
        assert len(rows) == len(packed) == (P - 1) * (P - 2) // 2 - sum(1 for k in tset if r in
                                                                         ((k >> 42), (k >> 21) & 0x1FFFFF, k & 0x1FFFFF))
        bf = -np.array([row[0] for row in rows])
        assert np.max(np.abs(bf - s) / np.maximum(bf, 1e-300)) < TOL
        first, last = near_tie_runs(bf)
        where = {int(x): i for i, x in enumerate(packed.tolist())}
        for i, (_, pk) in enumerate(rows):
            assert first[i] <= where[pk] + 1 <= last[i]
    # triplets {q, 0, y} and {q, 1, y} tie exactly: packed order
    packed, s = gene_oracle(thetas, prs, cand, train, 8)
    where = {int(x): i for i, x in enumerate(packed.tolist())}
    a, b = int(pack_ranks(0, 8, 12)), int(pack_ranks(1, 8, 12))
    if s[where[a]] == s[where[b]]:
        assert where[a] < where[b]


def test_workspace_and_abi_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_rank_per_gene_workspace_bytes(100, 10, 10, 2, 50, 30, ctypes.byref(nb)) == 0 and nb.value > 0
    for args in [(100, 10, 10, 39, 50, 30),          # S K = 390 > 384
                 ((1 << 21) + 1, 10, 2, 1, 0, 0), (100, -1, 2, 1, 0, 0), (100, 101, 2, 1, 0, 0),
                 (100, 10, 0, 1, 0, 0), (100, 10, 2, 0, 0, 0), (100, 10, 2, 1, -1, 0), (100, 10, 2, 1, (1 << 29) + 1, 0),
                 (100, 10, 2, 1, 0, -1), (100, 10, 2, 1, 0, 1 << 31)]:
        assert lib.tip_rank_per_gene_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"S*K <= 384" in lib.tip_last_error() and b"0 <= n_query <= n_cand" in lib.tip_last_error()
    assert lib.tip_rank_per_gene_workspace_bytes(100, 10, 2, 1, 0, 0, None) == -1
    # bad arguments are refused before any pointer is read
    assert lib.tip_rank_per_gene(10, 2, 200, None, None, None, 10, None, 1, None, 0, None, None, None, 0, None, 0, None, None,
                                 None, None) == -1
    assert b"S*K <= 384" in lib.tip_last_error()
    assert lib.tip_rank_per_gene(10, 2, 1, None, None, None, 10, None, 11, None, 0, None, None, None, 0, None, 0, None, None,
                                 None, None) == -1
    assert b"n_query <= n_cand" in lib.tip_last_error()
    assert lib.tip_rank_per_gene(10, 2, 1, None, None, None, 10, None, 1, None, 0, None, None, None, 0, None, 0, None, None,
                                 None, None) == -1
    assert b"null pointer" in lib.tip_last_error()


def test_model_refusals():
    random.seed(2)
    m = _digested()
    m.initialize_parameters(2)
    g0, g1 = m.id_gene[0], m.id_gene[1]
    with pytest.raises(ValueError, match="unknown gene names: NOPE1, NOPE2"):
        m.rank_held_out_per_gene([g0, "NOPE1"], genes=["NOPE2"])
    with pytest.raises(ValueError, match="unknown gene names: NOPE"):
        m.rank_held_out_per_gene(genes=[g0, "NOPE"])
    with pytest.raises(ValueError, match="rank_held_out_per_gene: duplicate query genes: %s" % g1):
        m.rank_held_out_per_gene([g0, g1, g1])
    with pytest.raises(ValueError, match="rank_held_out_per_gene: queries is empty"):
        m.rank_held_out_per_gene([])
    with pytest.raises(ValueError, match="rank_held_out_per_gene: params is empty"):
        m.rank_held_out_per_gene(params=[])
    t2, p2 = random_params(np.random.default_rng(0), m.P, 2, 1)
    t3, p3 = random_params(np.random.default_rng(1), m.P, 3, 1)
    with pytest.raises(ValueError, match="rank_held_out_per_gene: the parameter sets have different K"):
        _digested().rank_held_out_per_gene(params=[(t2[0], p2[0]), (t3[0], p3[0])])
    m.test_links = {}
    with pytest.raises(ValueError, match="rank_held_out_per_gene: the model has no test links"):
        m.rank_held_out_per_gene()
    from trigenicinteractionpredictor_b200 import Model
    with pytest.raises(ValueError, match="rank_held_out_per_gene needs a model digested"):
        Model().rank_held_out_per_gene()


def test_cli_held_out_genes_refusals(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    base = ["-t", tr, "-e", te, "-p", good, "--held-out-genes"]
    g0, g1 = m.id_gene[0], m.id_gene[1]
    pf = tmp_path / "p.txt"
    pf.write_text("%s+%s\n" % (g0, g1))
    for extra in (["-r", str(pf)], ["-n", "20"], ["--held-out"], ["--held-out-pairs"], ["--include-known"]):
        assert main(base + extra) == 2
        assert "--held-out-genes excludes" in capsys.readouterr().err
    # -q parsing and its errors are those of the per-gene predictor
    for text, msg in [("\n\n", "names no gene"), ("%s\nNOPE\n" % g0, "query genes not in the train / test files: NOPE"),
                      ("%s\n%s\n%s\n" % (g0, g1, g0), "query genes listed twice: %s" % g0)]:
        qf = tmp_path / "q.txt"
        qf.write_text(text)
        assert main(base + ["-q", str(qf)]) == 2
        assert msg in capsys.readouterr().err
    assert main(base + ["-q", str(tmp_path / "missing.txt")]) == 2
    assert "does not exist" in capsys.readouterr().err
    # the flags it excludes keep their own messages without it
    qf = tmp_path / "q.txt"
    qf.write_text("%s\n" % g0)
    assert main(["-t", tr, "-e", te, "-p", good, "--held-out-pairs", "-q", str(qf)]) == 2
    assert "--held-out-pairs excludes" in capsys.readouterr().err
    assert main(["-t", tr, "-e", te, "-p", good, "--held-out", "-q", str(qf)]) == 2
    assert "--held-out excludes" in capsys.readouterr().err


def test_sass_gene_rank_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    body = [f for f in out.split("Function : ") if f.split("\n", 1)[0].find("tip_gene_rank_pass_kernel") >= 0]
    assert len(body) == 1 and "DMMA.8x8x4" in body[0]


# ----------------------------------------------------------------------------------------------
# GPU tests
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def _case(rng, P, K, S, n_train, n_test, n_both=5):
    thetas, prs = random_params(rng, P, K, S)
    train = random_keys(rng, P, n_train)
    test = {k: lab for k, lab in random_keys(rng, P, n_test).items() if k not in train}
    for k in list(train)[:n_both]:
        test[k] = 1                                   # test keys that are also train keys: excluded
    return synthetic_model(P, train, test), list(zip(thetas, prs)), train, test


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("K", [1, 2, 3, 4, 10, 32])
@pytest.mark.parametrize("P", [40, 130])
def test_ranks_match_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(P * 100 + K * 10 + S + 11)
    m, sets, train, test = _case(rng, P, K, S, 3 * P, P + 60)
    # one gene in no ranked test triplet: a listed query without views (test keys that are train keys are not ranked)
    cand = sorted(range(P), key=str)
    free = cand[P // 2]
    test = {k: lab for k, lab in test.items() if k in train or str(free) not in k.split("_")}
    m = synthetic_model(P, train, test)
    res = m.rank_held_out_per_gene(params=sets, hits_at=(1, 10, P * P))
    ranked = len(test) - 5
    assert res["excluded_train"] == 5 and res["excluded_genes"] == 0
    assert res["views"] == 3 * ranked == len(res["rows"]) == res["positives"] + res["negatives"]
    check_model_result(m, res, sets)
    assert [g[0] for g in res["genes"]] == sorted(g[0] for g in res["genes"])
    assert sum(g[2] + g[3] for g in res["genes"]) == res["views"]
    for N in (1, 10):
        hp = res["hits_at"][N]["positives"]
        want = sum(1 for r in res["rows"] if r[3] == 1 and r[5] <= N) / max(res["positives"], 1)
        assert hp is None or hp == want
    assert res["hits_at"][P * P]["positives"] in (None, 1.0)
    # explicit queries in the caller's order: the genes of rank 0 and n - 1 (one or two regions empty), genes of test
    # triplets, and one without any
    queries = [m.id_gene[cand[0]], m.id_gene[cand[-1]]]
    for key in list(test)[:4]:
        queries.append(m.id_gene[int(key.split("_")[1])])
    queries = list(dict.fromkeys(queries)) + [m.id_gene[free]]
    res2 = m.rank_held_out_per_gene(queries, params=sets)
    check_model_result(m, res2, sets)
    assert [g[0] for g in res2["genes"]] == queries
    assert res2["genes"][-1][2:] == [0, 0, None, None]
    order = {g: i for i, g in enumerate(queries)}
    assert [order[r[0]] for r in res2["rows"]] == sorted(order[r[0]] for r in res2["rows"])
    same = {(r[0], r[1]): r for r in res["rows"]}
    for r2 in res2["rows"]:
        if (r2[0], r2[1]) in same:
            r = same[(r2[0], r2[1])]
            assert r2[5] == r[5] and r2[4] == r[4] and r2[6] == r[6]


@pytest.mark.gpu
@pytest.mark.parametrize("K,S", [(3, 1), (10, 2)])
def test_exactly_consistent_with_top_triplets_per_gene(torch_cuda, K, S):
    P = 200
    n = P
    rng = np.random.default_rng(29 + K)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    qr = np.concatenate([[0, n - 1, 1, n - 2], rng.choice(np.arange(2, n - 2), 36, replace=False)]).astype(np.int32)
    parts = [pack_ranks(*np.sort(rng.choice(P, (800, 3)), 1).T)]
    for r in qr[:12].tolist():
        parts.append(_train_of_query(rng, n, r, 60)[0])
    train = np.unique(np.concatenate(parts))
    tr = np.stack([(train >> np.uint64(s)) & np.uint64((1 << 21) - 1) for s in (42, 21, 0)], 1).astype(np.int64)
    train = train[(tr[:, 0] < tr[:, 1]) & (tr[:, 1] < tr[:, 2])]
    tq, tu, tv = [], [], []
    for q, r in enumerate(qr.tolist()):
        for _ in range(25):
            u, v = rng.choice([x for x in range(n) if x != r], 2, replace=False).tolist()
            tq.append(q)
            tu.append(u)
            tv.append(v)
    check_against_per_gene(_engine(P, K), np.stack(thetas), np.stack(prs), cand, qr, train, np.array(tq), np.array(tu),
                           np.array(tv))


@pytest.mark.gpu
def test_all_scores_tied(torch_cuda):
    """Identical theta rows and dyadic parameters: every score is the same number, so ranks follow packed order in U_q."""
    P, K = 60, 3
    theta = np.tile(np.array([0.5, 0.25, 0.25]), (P, 1))
    rng = np.random.default_rng(4)
    p1 = rng.integers(1, 4, size=(K, K, K)) / 4.0
    pr = np.stack([1.0 - p1, p1], axis=3)
    train = random_keys(rng, P, 300)
    test = {k: lab for k, lab in random_keys(rng, P, 100).items() if k not in train}
    m = synthetic_model(P, train, test)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    rank = {int(g): r for r, g in enumerate(cand.tolist())}
    tset = set(packed_of_key(k, rank) for k in train)
    res = m.rank_held_out_per_gene(params=[(theta, pr)])
    assert len(set(r[4] for r in res["rows"])) == 1
    for gene, key, names, label, score, rk, universe in res["rows"]:
        q = rank[m.gene_id[gene]]
        pk = packed_of_key(key, rank)
        before = [1 for u, v in itertools.combinations([x for x in range(P) if x != q], 2)
                  if int(pack_ranks(*sorted((q, u, v)))) < pk and int(pack_ranks(*sorted((q, u, v)))) not in tset]
        assert rk == 1 + len(before)


@pytest.mark.gpu
def test_triplets_that_score_zero(torch_cuda):
    """Half the genes sit in a group that interacts with nothing: their triplets score exactly 0 and tie on packed ranks."""
    P, K = 70, 3
    rng = np.random.default_rng(6)
    theta = rng.dirichlet(np.ones(2), size=P)
    theta = np.concatenate([theta, np.zeros((P, 1))], axis=1)
    theta[::2] = [0.0, 0.0, 1.0]
    p1 = rng.random((K, K, K))
    p1[2, :, :] = p1[:, 2, :] = p1[:, :, 2] = 0.0
    pr = np.stack([1.0 - p1, p1], axis=3)
    train = random_keys(rng, P, 200)
    test = {k: lab for k, lab in random_keys(rng, P, 120).items() if k not in train}
    m = synthetic_model(P, train, test)
    res = m.rank_held_out_per_gene(params=[(theta, pr)])
    assert sum(1 for r in res["rows"] if r[4] == 0.0) > 50
    orc = check_model_result(m, res, [(theta, pr)])
    cand = sorted(range(P), key=str)
    rank = {g: r for r, g in enumerate(cand)}
    for gene, key, names, label, score, rk, universe in res["rows"]:
        if score == 0.0:                   # exact zeros tie exactly: the order among them is packed order
            where, s, _, _ = orc.get(rank[m.gene_id[gene]])
            i = where[packed_of_key(key, rank)]
            assert s[i] == 0.0 and rk == i + 1


@pytest.mark.gpu
def test_universe_sizes_zero_one_two(torch_cuda):
    K = 2
    rng = np.random.default_rng(9)
    thetas, prs = random_params(rng, 4, K, 1)
    eng = _engine(4, K)
    th, pp = np.stack(thetas), np.stack(prs)
    cand = np.array([0, 1, 2, 3], dtype=np.int32)
    none = np.empty(0, np.uint64)
    # n = 4, query 1: C(3, 2) = 3 pairs; one, two and three train keys leave 2, 1 and 0
    qr = np.array([1], dtype=np.int32)
    tq, tu, tv = np.zeros(3, np.int32), np.array([0, 0, 2]), np.array([2, 3, 3])
    for train, want in [(pack_ranks([0], [1], [2]), 2), (pack_ranks([0, 0], [1, 1], [2, 3]), 1),
                        (pack_ranks([0, 0, 1], [1, 1, 2], [2, 3, 3]), 0)]:
        rank, score, universe = check_against_per_gene(eng, th, pp, cand, qr, np.sort(train), tq, tu, tv)
        assert universe.tolist() == [want]
        assert sorted(rank.tolist()) == sorted([0] * (3 - want) + list(range(1, want + 1)))
    # n = 3: |U| = 1, and 0 with its one train key; every query at once
    rank, score, universe = check_against_per_gene(eng, th, pp, cand[:3], np.array([2, 0, 1]), none, [0, 1, 2], [0, 1, 0],
                                                   [1, 2, 2])
    assert rank.tolist() == [1, 1, 1] and universe.tolist() == [1, 1, 1]
    rank, score, universe = eng.rank_per_gene(th, pp, cand[:3], np.array([0]), pack_ranks([0], [1], [2]), [0], [1], [2])
    assert rank.tolist() == [0] and universe.tolist() == [0]
    # n = 2: no pair at all
    rank, score, universe = eng.rank_per_gene(th, pp, cand[:2], np.array([1]), none, [], [], [])
    assert universe.tolist() == [0] and len(rank) == 0


@pytest.mark.gpu
def test_train_triplets_interleave_test_triplets(torch_cuda):
    """One query with 400 train and 400 test triplets drawn from the same pairs at random, so in score order they
    interleave: each rank subtracts the train triplets ahead of it."""
    P, K, S = 150, 4, 2
    rng = np.random.default_rng(31)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    r = 70
    pairs = list(itertools.combinations([x for x in range(P) if x != r], 2))
    pick = rng.choice(len(pairs), 800, replace=False)
    tr_pairs, te_pairs = [pairs[i] for i in pick[:400]], [pairs[i] for i in pick[400:]]
    train = np.sort(np.array([int(pack_ranks(*sorted((r, u, v)))) for u, v in tr_pairs], dtype=np.uint64))
    tu, tv = np.array([p[1] for p in te_pairs]), np.array([p[0] for p in te_pairs])   # the two other ranks in either order
    eng = _engine(P, K)
    rank, score, universe = check_against_per_gene(eng, np.stack(thetas), np.stack(prs), cand, np.array([r]), train,
                                                   np.zeros(400, np.int32), tu, tv)
    assert universe.tolist() == [len(pairs) - 400]
    # the train triplets do interleave: most test triplets have train triplets both ahead of them and behind them
    tri = np.sort(np.array([(r, u, v) for u, v in tr_pairs]), 1)
    tr_score = eng.score_sum(np.stack(thetas), np.stack(prs), cand[tri]) / S
    assert sum(1 for s in score.tolist() if (tr_score > s).any() and (tr_score < s).any()) > 300


@pytest.mark.gpu
def test_repeated_test_entries_and_known_keys(torch_cuda):
    P, K, S = 120, 4, 2
    rng = np.random.default_rng(23)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    qr = np.array([9, 50, 100], dtype=np.int32)
    train = pack_ranks([3, 3, 7, 0, 9], [9, 9, 50, 1, 50], [11, 40, 60, 2, 100])
    train = np.sort(np.concatenate([train, train[:2]]))                  # repeated keys count once
    tq = np.array([0, 0, 0, 1, 1, 0, 2, 2, 0], dtype=np.int32)
    tu = np.array([5, 5, 3, 60, 8, 3, 9, 50, 119], dtype=np.int32)
    tv = np.array([6, 6, 11, 7, 20, 40, 50, 9, 0], dtype=np.int32)      # (5, 6) twice; 3_9_11 / 7_50_60 / 3_9_40 / 9_50_100 are train
    rank, score, universe = check_against_per_gene(_engine(P, K), np.stack(thetas), np.stack(prs), cand, qr, train, tq, tu, tv)
    assert rank[0] == rank[1] and score[0] == score[1] and rank[0] > 0
    assert rank[2] == 0 and rank[3] == 0 and rank[5] == 0 and rank[6] == 0 and rank[7] == 0
    c = (P - 1) * (P - 2) // 2
    assert universe.tolist() == [c - 3, c - 2, c - 1]


@pytest.mark.gpu
@pytest.mark.parametrize("K,S", [(4, 1), (32, 12)])
def test_hub_query_takes_several_rounds(torch_cuda, K, S):
    """A hub query with 2 500 test triplets, more than one round holds in shared memory (2 048, fewer at S K = 384), and
    300 train triplets, beside two light queries: the hub's tiles are swept once per round."""
    P = 300
    rng = np.random.default_rng(77 + K)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    qr = np.array([5, 150, 298], dtype=np.int32)
    tq, tu, tv, parts = [], [], [], []
    for q, (r, nt) in enumerate(zip(qr.tolist(), [30, 2500, 40])):
        keys, tr_pairs = _train_of_query(rng, P, r, 300 if nt > 1000 else 20)
        parts.append(keys)
        te = set()
        while len(te) < nt:
            u, v = sorted(rng.choice([x for x in range(P) if x != r], 2, replace=False).tolist())
            if (u, v) not in tr_pairs:
                te.add((u, v))
        for u, v in sorted(te):
            tq.append(q)
            tu.append(u)
            tv.append(v)
        u, v = sorted(tr_pairs)[0]                   # a test entry that is a train key
        tq.append(q)
        tu.append(u)
        tv.append(v)
    train = np.unique(np.concatenate(parts))
    rank, score, universe = check_against_per_gene(_engine(P, K), np.stack(thetas), np.stack(prs), cand, qr, train,
                                                   np.array(tq), np.array(tu), np.array(tv))
    assert (rank == 0).sum() >= 3
    c = (P - 1) * (P - 2) // 2
    assert universe[1] == c - 300 - sum(1 for k in np.concatenate([parts[0], parts[2]]).tolist()
                                        if 150 in ((k >> 42), (k >> 21) & 0x1FFFFF, k & 0x1FFFFF))


@pytest.mark.gpu
def test_p1500_against_tip_score_and_sort(torch_cuda):
    P, K = 1500, 4
    rng = np.random.default_rng(1501)
    thetas, prs = random_params(rng, P, K, 1)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    qr = np.array([0, 777, P - 1], dtype=np.int32)
    train = np.unique(pack_ranks(*np.sort(rng.choice(P, (200000, 3)), 1).T))
    tr = np.stack([(train >> np.uint64(s)) & np.uint64((1 << 21) - 1) for s in (42, 21, 0)], 1).astype(np.int64)
    train = train[(tr[:, 0] < tr[:, 1]) & (tr[:, 1] < tr[:, 2])]
    tq = np.repeat(np.arange(len(qr)), 60)
    tu, tv = [], []
    for r in qr.tolist():
        for _ in range(60):
            u, v = rng.choice([x for x in range(P) if x != r], 2, replace=False).tolist()
            tu.append(u)
            tv.append(v)
    rank, score, universe = eng.rank_per_gene(np.stack(thetas), np.stack(prs), cand, qr, train, tq, tu, tv)
    tset = np.asarray(train, dtype=np.uint64)
    for q, r in enumerate(qr.tolist()):
        others = np.array([x for x in range(P) if x != r])
        iu, iv = np.triu_indices(len(others), 1)
        tri = np.sort(np.stack([others[iu], others[iv], np.full(len(iu), r)], 1), 1)
        packed = pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2])
        keep = ~np.isin(packed, tset)
        s = eng.score_sum(np.stack(thetas), np.stack(prs), cand[tri[keep]])
        packed = packed[keep]
        order = np.lexsort((packed, -s))
        packed, s = packed[order], s[order]
        first, last = near_tie_runs(s)
        where = {int(x): i for i, x in enumerate(packed.tolist())}
        assert universe[q] == len(packed)
        for j in np.flatnonzero(tq == q).tolist():
            pk = int(pack_ranks(*sorted((r, tu[j], tv[j]))))
            if pk not in where:
                assert rank[j] == 0
                continue
            i = where[pk]
            assert first[i] <= rank[j] <= last[i]
            assert abs(score[j] - s[i]) <= TOL * s[i]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3])
def test_golden_base(torch_cuda, K):
    m = _trained_base_model(K)
    res = m.rank_held_out_per_gene()
    assert res["positives"] + res["negatives"] == res["views"] == 3 * (len(m.test_links) - res["excluded_train"]
                                                                      - res["excluded_genes"])
    th, pr = np.array(m.theta), np.array(m.pr)
    sets = [(th, pr)]
    sub = dict(res)
    sub["rows"] = res["rows"][::7]
    check_model_result(m, sub, sets)
    for r in res["rows"][:30]:
        a, b, c = r[1].split("_")
        assert abs(r[4] - m.do_prediction(a, b, c)) <= TOL * r[4]
    if res["positives"]:
        assert res["mrr"] is not None and 0.0 < res["mrr"] <= 1.0
        assert res["auc_micro"] is None or 0.0 <= res["auc_micro"] <= 1.0


@pytest.mark.gpu
def test_train_with_save_params_then_predict_cli_held_out_genes(torch_cuda, tmp_path):
    from trigenicinteractionpredictor_b200 import Model, main
    from trigenicinteractionpredictor_b200.predict import main as predict_main
    out = str(tmp_path) + os.sep
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["-t", tr, "-e", te, "-k", "2", "-i", "300", "-f", "5", "-b", "10", "-n", "2", "-o", out,
                 "--seed", "1000", "--save-params"]) == 0
    params = [out + "Sample_0_K2.npz", out + "Sample_1_K2.npz"]
    mm = Model()
    mm.get_traintest(tr, te)
    for with_queries in (False, True):
        pred = str(tmp_path / "held_genes.tsv")
        argv = ["-t", tr, "-e", te, "-p", params[0], "-p", params[1], "--held-out-genes", "-o", pred]
        queries = None
        if with_queries:
            queries = list(dict.fromkeys(mm.id_gene[int(k.split("_")[1])] for k in list(mm.test_links)[:5]))
            (tmp_path / "queries.txt").write_text("".join("%s\n" % q for q in queries))
            argv += ["-q", str(tmp_path / "queries.txt")]
        assert predict_main(argv) == 0
        text = open(pred, encoding="utf-8").read().split("\n")
        hdr = text.index("Query gene\tRank\tGene universe\tPredicted Interaction\tReal Interaction\tID of genes\tGenes")
        summary = dict(line.split(":\t") for line in text[:hdr])
        want = mm.rank_held_out_per_gene(queries, params=params)
        assert int(summary["Views"]) == want["views"] and int(summary["Positive views"]) == want["positives"]
        assert int(summary["Query genes"]) == len(want["genes"])
        assert summary["Hits at 20"] == str(want["hits_at"][20]["positives"]) or want["hits_at"][20]["positives"] is None
        body = [ln.split("\t") for ln in text[hdr + 1:] if ln]
        assert len(body) == len(want["rows"])
        for b, r in zip(body, want["rows"]):
            assert b[0] == r[0] and int(b[1]) == r[5] and int(b[2]) == r[6] and float(b[3]) == r[4]
            assert int(b[4]) == r[3] and b[5] == r[1] and b[6] == r[2]
        if with_queries:
            assert [g[0] for g in want["genes"]] == queries


@pytest.mark.gpu
def test_bad_entries_are_refused(torch_cuda):
    from trigenicinteractionpredictor_b200 import _cabi
    K = 2
    thetas, prs = random_params(np.random.default_rng(1), 30, K, 1)
    eng = _engine(30, K)
    cand = np.arange(30, dtype=np.int32)
    args = (np.stack(thetas), np.stack(prs), cand)
    none = np.empty(0, np.uint64)
    for qr, tq, tu, tv, msg in [([30], [0], [1], [2], "query rank 30 of query 0 is not in"),
                                ([4, 4], [0], [1], [2], "query rank 4 appears twice"),
                                ([0], [1], [1], [2], "names query 1"), ([0], [0], [0], [2], "has ranks \\(0, 2\\)"),
                                ([0], [0], [2], [2], "has ranks \\(2, 2\\)"), ([0], [0], [1], [30], "has ranks \\(1, 30\\)"),
                                ([0], [0], [-1], [3], "has ranks \\(-1, 3\\)")]:
        with pytest.raises(_cabi.TipLibraryError, match=msg):
            eng.rank_per_gene(*args, np.array(qr), none, np.array(tq), np.array(tu), np.array(tv))
