"""Ranks of held-out triplets among their query pair's unseen partners (tip_rank_per_pair, EMEngine.rank_per_pair,
Model.rank_held_out_per_pair, predict --held-out-pairs).

The oracle scores every partner of a pair with numpy (the einsum of tests/test_predict.py, pinned to
oracle.mmsbm_oracle.predict_loops), drops the train keys and orders the rest by (score descending, rc ascending); a test
partner's rank is its position + 1.  Device ranks may differ from the oracle's only inside runs of near-equal oracle
scores (within 1e-12), as in tests/test_rank_held_out.py.  Against tip_top_triplets_per_pair, which computes every score
at the same place of the same tile, ranks and score bits must agree exactly."""
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


def pair_oracle(thetas, prs, cand, train, ra, rb):
    """(partner ranks, mean scores) of the universe of the pair (ra, rb), in rank order."""
    n = len(cand)
    c = np.array([x for x in range(n) if x != ra and x != rb], dtype=np.int64)
    tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
    keep = ~np.isin(pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2]), np.asarray(train, dtype=np.uint64))
    c, tri = c[keep], tri[keep]
    s = np.zeros(len(c))
    cand = np.asarray(cand, dtype=np.int64)
    for th, pr in zip(thetas, prs):
        g = np.asarray(th, dtype=np.float64)[cand[tri]]
        s += np.einsum("ix,iy,iz,xyz->i", g[:, 0], g[:, 1], g[:, 2], np.asarray(pr)[..., 1], optimize=True)
    s /= len(thetas)
    order = np.lexsort((c, -s))
    return c[order], s[order]


class Oracle:
    """Per-pair oracles of a candidate list, cached: rank interval (near-tie run) and score of a partner."""

    def __init__(self, thetas, prs, cand, train):
        self.args = (thetas, prs, np.asarray(cand), train)
        self.cache = {}

    def get(self, ra, rb):
        key = (min(ra, rb), max(ra, rb))
        if key not in self.cache:
            c, s = pair_oracle(*self.args, *key)
            first, last = near_tie_runs(s)
            self.cache[key] = ({int(x): i for i, x in enumerate(c.tolist())}, s, first, last)
        return self.cache[key]

    def check(self, ra, rb, rc, rank, score, universe):
        where, s, first, last = self.get(ra, rb)
        assert universe == len(s)
        i = where[rc]
        assert first[i] <= rank <= last[i], (ra, rb, rc, rank, first[i], last[i])
        assert abs(score - s[i]) <= TOL * s[i]


def check_model_result(m, res, sets, genes_ids=None):
    """Every view of a Model.rank_held_out_per_pair result against the oracle."""
    ids = sorted(range(m.P) if genes_ids is None else genes_ids, key=str)
    cand = np.array(ids, dtype=np.int32)
    rank = {int(g): r for r, g in enumerate(ids)}
    orc = Oracle([s[0] for s in sets], [s[1] for s in sets], cand, m._train_packed(cand))
    for pair, key, names, label, score, rk, universe in res["rows"]:
        a, b = (rank[m.gene_id[x]] for x in pair.split("+"))
        c = [rank[int(x)] for x in key.split("_") if rank[int(x)] not in (a, b)]
        assert len(c) == 1
        orc.check(a, b, c[0], rk, score, universe)
        assert names == "_".join(sorted(m.id_gene[int(x)] for x in key.split("_")))
        assert label == (0 if m.test_links[key][0] else 1)
    return orc


def _engine(P, K):
    from trigenicinteractionpredictor_b200.engine import EMEngine
    return EMEngine(P, K, device="cuda:0")


def _partner(ids, a, b):
    """The partner of a triplet of ranks that holds the pair (a, b)."""
    return [x for x in ids if x not in (a, b)][0]


def check_against_per_pair(eng, thetas, prs, cand, pr, train, tp, trc):
    """rank_per_pair against top_triplets_per_pair(known = train, n = n - 2) on the same pairs: exact ranks and bits."""
    n = len(cand)
    rank, score, universe = eng.rank_per_pair(thetas, prs, cand, pr, train, tp, trc)
    ids, sc, counts = eng.top_triplets_per_pair(thetas, prs, cand, pr, train, n - 2)
    rk = {int(g): r for r, g in enumerate(np.asarray(cand).tolist())}
    pos = []
    for q in range(len(pr)):
        a, b = int(pr[q][0]), int(pr[q][1])
        assert universe[q] == counts[q]
        pos.append({_partner([rk[int(x)] for x in row], a, b): (k, s) for k, (row, s) in
                    enumerate(zip(ids[q, :counts[q]].tolist(), sc[q, :counts[q]].tolist()))})
    tset = set(int(x) for x in np.asarray(train, dtype=np.uint64).tolist())
    for j in range(len(tp)):
        q, c = int(tp[j]), int(trc[j])
        a, b = sorted((int(pr[q][0]), int(pr[q][1])))
        x, y, z = sorted((a, b, c))
        if (x << 42) | (y << 21) | z in tset:
            assert rank[j] == 0
            continue
        k, s = pos[q][c]
        assert rank[j] == k + 1, (j, q, c, rank[j], k + 1)
        assert np.float64(score[j]).view(np.int64) == np.float64(s).view(np.int64)
    return rank, score, universe


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_pair_oracle_equals_itertools_brute_force(S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(40 + S)
    P, K = 20, 3
    thetas, prs = random_params(rng, P, K, S)
    # ties on rc: genes 0 and 1 share theta, so partners 0 and 1 of a pair score the same
    for th in thetas:
        th[1] = th[0]
    cand = np.array(sorted(range(P), key=str))
    train = pack_ranks([0, 2, 5, 1, 3], [1, 7, 6, 3, 4], [13, 9, 11, 13, 19])
    tset = set(int(x) for x in train.tolist())
    tl, pl = [t.tolist() for t in thetas], [p.tolist() for p in prs]
    for ra, rb in [(1, 13), (3, 4), (0, 19), (6, 11), (2, 3)]:
        c, s = pair_oracle(thetas, prs, cand, train, ra, rb)
        rows = []
        for rc in range(P):
            if rc in (ra, rb):
                continue
            x, y, z = sorted((ra, rb, rc))
            if (x << 42) | (y << 21) | z in tset:
                continue
            gx, gy, gz = (int(cand[i]) for i in (x, y, z))
            rows.append((-sum(orc.predict_loops(t, p, gx, gy, gz) for t, p in zip(tl, pl)) / S, rc))
        rows.sort()
        assert len(rows) == len(c)
        bf = -np.array([r[0] for r in rows])
        assert np.max(np.abs(bf - s) / np.maximum(bf, 1e-300)) < TOL
        first, last = near_tie_runs(bf)
        for i, (_, rc) in enumerate(rows):
            j = int(np.flatnonzero(c == rc)[0])
            assert first[i] <= j + 1 <= last[i]
    # partners 0 and 1 tie exactly in every pair that holds neither: rc order
    c, s = pair_oracle(thetas, prs, cand, train, 5, 8)
    i0, i1 = int(np.flatnonzero(c == 0)[0]), int(np.flatnonzero(c == 1)[0])
    if s[i0] == s[i1]:
        assert i0 < i1


def test_workspace_and_abi_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_rank_per_pair_workspace_bytes(100, 10, 10, 2, 50, 30, ctypes.byref(nb)) == 0 and nb.value > 0
    for args in [(100, 10, 10, 39, 50, 30),          # S K = 390 > 384
                 ((1 << 21) + 1, 10, 2, 1, 0, 0), (100, -1, 2, 1, 0, 0), (100, (1 << 24) + 1, 2, 1, 0, 0),
                 (100, 10, 0, 1, 0, 0), (100, 10, 2, 0, 0, 0), (100, 10, 2, 1, -1, 0), (100, 10, 2, 1, (1 << 29) + 1, 0),
                 (100, 10, 2, 1, 0, -1), (100, 10, 2, 1, 0, 1 << 31)]:
        assert lib.tip_rank_per_pair_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"S*K <= 384" in lib.tip_last_error() and b"0 <= n_test < 2^31" in lib.tip_last_error()
    assert lib.tip_rank_per_pair_workspace_bytes(100, 10, 2, 1, 0, 0, None) == -1
    # bad arguments are refused before any pointer is read
    assert lib.tip_rank_per_pair(10, 2, 200, None, None, None, 10, None, 1, None, 0, None, None, 0, None, 0, None, None,
                                 None, None) == -1
    assert b"S*K <= 384" in lib.tip_last_error()
    assert lib.tip_rank_per_pair(10, 2, 1, None, None, None, 10, None, 1, None, 0, None, None, 0, None, 0, None, None,
                                 None, None) == -1
    assert b"null pointer" in lib.tip_last_error()


def test_model_refusals():
    random.seed(2)
    m = _digested()
    m.initialize_parameters(2)
    g0, g1, g2 = m.id_gene[0], m.id_gene[1], m.id_gene[2]
    with pytest.raises(ValueError, match="unknown gene names: NOPE1, NOPE2"):
        m.rank_held_out_per_pair([(g0, "NOPE1")], genes=["NOPE2"])
    with pytest.raises(ValueError, match="unknown gene names: NOPE"):
        m.rank_held_out_per_pair(genes=[g0, "NOPE"])
    with pytest.raises(ValueError, match="rank_held_out_per_pair: a pair of one gene: %s\\+%s" % (g1, g1)):
        m.rank_held_out_per_pair([(g0, g2), (g1, g1)])
    with pytest.raises(ValueError, match="rank_held_out_per_pair: duplicate pairs"):
        m.rank_held_out_per_pair([(g0, g1), (g1, g0)])
    with pytest.raises(ValueError, match="rank_held_out_per_pair: pairs is empty"):
        m.rank_held_out_per_pair([])
    with pytest.raises(ValueError, match="rank_held_out_per_pair: a pair is not two gene names"):
        m.rank_held_out_per_pair([(g0, g1, g2)])
    with pytest.raises(ValueError, match="rank_held_out_per_pair: params is empty"):
        m.rank_held_out_per_pair(params=[])
    t2, p2 = random_params(np.random.default_rng(0), m.P, 2, 1)
    t3, p3 = random_params(np.random.default_rng(1), m.P, 3, 1)
    with pytest.raises(ValueError, match="rank_held_out_per_pair: the parameter sets have different K"):
        _digested().rank_held_out_per_pair(params=[(t2[0], p2[0]), (t3[0], p3[0])])
    m.test_links = {}
    with pytest.raises(ValueError, match="rank_held_out_per_pair: the model has no test links"):
        m.rank_held_out_per_pair()
    from trigenicinteractionpredictor_b200 import Model
    with pytest.raises(ValueError, match="rank_held_out_per_pair needs a model digested"):
        Model().rank_held_out_per_pair()


def test_cli_held_out_pairs_refusals(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    base = ["-t", tr, "-e", te, "-p", good, "--held-out-pairs"]
    qf = tmp_path / "q.txt"
    qf.write_text("%s\n" % m.id_gene[0])
    for extra in (["-q", str(qf)], ["--held-out"], ["--include-known"], ["-n", "20"]):
        assert main(base + extra) == 2
        assert "--held-out-pairs excludes" in capsys.readouterr().err
    # -r parsing and its errors are those of the pair predictor
    g0, g1 = m.id_gene[0], m.id_gene[1]
    cases = [("%s+%s+%s\n" % (g0, g1, g0), "is not a pair"), ("\n\n", "names no pair"), ("%s+NOPE\n" % g0, "NOPE"),
             ("%s+%s\n" % (g0, g0), "a pair of one gene"), ("%s+%s\n%s %s\n" % (g0, g1, g1, g0), "pairs listed twice")]
    for text, msg in cases:
        pf = tmp_path / "p.txt"
        pf.write_text(text)
        assert main(base + ["-r", str(pf)]) == 2
        assert msg in capsys.readouterr().err
    assert main(base + ["-r", str(tmp_path / "missing.txt")]) == 2
    assert "does not exist" in capsys.readouterr().err
    # --held-out still refuses -r
    pf = tmp_path / "p.txt"
    pf.write_text("%s+%s\n" % (g0, g1))
    assert main(["-t", tr, "-e", te, "-p", good, "--held-out", "-r", str(pf)]) == 2
    assert "--held-out excludes" in capsys.readouterr().err


def test_sass_rank_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    body = [f for f in out.split("Function : ") if f.split("\n", 1)[0].find("tip_rank_pass_kernel") >= 0]
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
    rng = np.random.default_rng(P * 100 + K * 10 + S + 7)
    m, sets, train, test = _case(rng, P, K, S, 3 * P, P + 60)
    res = m.rank_held_out_per_pair(params=sets, hits_at=(1, 10, P))
    ranked = len(test) - 5
    assert res["excluded_train"] == 5 and res["excluded_genes"] == 0
    assert res["views"] == 3 * ranked == len(res["rows"]) == res["positives"] + res["negatives"]
    check_model_result(m, res, sets)
    assert [p[0] for p in res["pairs"]] == sorted(p[0] for p in res["pairs"])
    assert sum(p[2] + p[3] for p in res["pairs"]) == res["views"]
    for N in (1, 10):
        hp = res["hits_at"][N]["positives"]
        want = sum(1 for r in res["rows"] if r[3] == 1 and r[5] <= N) / max(res["positives"], 1)
        assert hp is None or hp == want
    assert res["hits_at"][P]["positives"] in (None, 1.0)
    # explicit pairs, in the caller's order: some with test triplets, one without, names in either order
    pairs = []
    for key in list(test)[:6]:
        a, b, _ = key.split("_")
        pairs.append((m.id_gene[int(b)], m.id_gene[int(a)]))
    pairs = list(dict.fromkeys(pairs, None))
    free = next((x, y) for x, y in itertools.combinations(range(P), 2)
                if not any({str(x), str(y)} <= set(k.split("_")) for k in test))
    pairs.append((m.id_gene[free[0]], m.id_gene[free[1]]))
    res2 = m.rank_held_out_per_pair(pairs, params=sets)
    check_model_result(m, res2, sets)
    assert [p[0] for p in res2["pairs"]] == ["%s+%s" % p for p in pairs]
    assert res2["pairs"][-1][2:] == [0, 0, None, None]
    order = {"%s+%s" % p: i for i, p in enumerate(pairs)}
    assert [order[r[0]] for r in res2["rows"]] == sorted(order[r[0]] for r in res2["rows"])
    for r in res["rows"]:
        for r2 in res2["rows"]:
            if r2[1] == r[1] and set(r2[0].split("+")) == set(r[0].split("+")):
                assert r2[5] == r[5] and r2[4] == r[4] and r2[6] == r[6]


@pytest.mark.gpu
@pytest.mark.parametrize("K,S", [(3, 1), (10, 2)])
def test_exactly_consistent_with_top_triplets_per_pair(torch_cuda, K, S):
    P = 300
    rng = np.random.default_rng(17 + K)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    pr = np.array([rng.choice(P, 2, replace=False) for _ in range(150)], dtype=np.int32)
    pr = pr[np.unique(np.sort(pr, 1), axis=0, return_index=True)[1]]
    train = np.unique(np.concatenate([
        pack_ranks(*np.sort(np.stack([np.full(20, min(a, b)), np.full(20, max(a, b)),
                                      rng.choice([x for x in range(P) if x not in (a, b)], 20, replace=False)], 1), 1).T)
        for a, b in pr[:40].tolist()] + [pack_ranks(*np.sort(rng.choice(P, (500, 3)), 1).T)]))
    tr = np.stack([(train >> np.uint64(s)) & np.uint64((1 << 21) - 1) for s in (42, 21, 0)], 1).astype(np.int64)
    train = train[(tr[:, 0] < tr[:, 1]) & (tr[:, 1] < tr[:, 2])]
    tp, trc = [], []
    for q, (a, b) in enumerate(pr.tolist()):
        for c in rng.choice([x for x in range(P) if x not in (a, b)], 12, replace=False).tolist():
            tp.append(q)
            trc.append(c)
    check_against_per_pair(_engine(P, K), np.stack(thetas), np.stack(prs), cand, pr, train, np.array(tp), np.array(trc))


@pytest.mark.gpu
def test_all_scores_tied(torch_cuda):
    """Identical theta rows and dyadic parameters: every score is the same number, so ranks follow rc order in U_ab."""
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
    tset = set(packed_of_key(k, rank) for k in train)
    res = m.rank_held_out_per_pair(params=[(theta, pr)])
    assert len(set(r[4] for r in res["rows"])) == 1
    for pair, key, names, label, score, rk, universe in res["rows"]:
        a, b = sorted(rank[m.gene_id[x]] for x in pair.split("+"))
        c = [rank[int(x)] for x in key.split("_") if rank[int(x)] not in (a, b)][0]
        unseen = [x for x in range(c) if x not in (a, b) and packed_of_key(key_of(cand[[a, b, x]]), rank) not in tset]
        assert rk == 1 + len(unseen)


@pytest.mark.gpu
def test_partners_that_score_zero(torch_cuda):
    """Half the genes sit in a group that interacts with nothing: their partners score exactly 0 and tie on rc."""
    P, K = 90, 3
    rng = np.random.default_rng(5)
    theta = rng.dirichlet(np.ones(2), size=P)
    theta = np.concatenate([theta, np.zeros((P, 1))], axis=1)
    theta[::2] = [0.0, 0.0, 1.0]
    p1 = rng.random((K, K, K))
    p1[2, :, :] = p1[:, 2, :] = p1[:, :, 2] = 0.0
    pr = np.stack([1.0 - p1, p1], axis=3)
    train = random_keys(rng, P, 200)
    test = {k: lab for k, lab in random_keys(rng, P, 150).items() if k not in train}
    m = synthetic_model(P, train, test)
    res = m.rank_held_out_per_pair(params=[(theta, pr)])
    assert sum(1 for r in res["rows"] if r[4] == 0.0) > 50
    orc = check_model_result(m, res, [(theta, pr)])
    cand = sorted(range(P), key=str)
    rank = {g: r for r, g in enumerate(cand)}
    for pair, key, names, label, score, rk, universe in res["rows"]:
        if score == 0.0:                   # exact zeros tie exactly: the order among them is rc order
            a, b = (rank[m.gene_id[x]] for x in pair.split("+"))
            c = [rank[int(x)] for x in key.split("_") if rank[int(x)] not in (a, b)][0]
            where, s, _, _ = orc.get(a, b)
            assert s[where[c]] == 0.0 and rk == where[c] + 1


@pytest.mark.gpu
def test_repeated_test_entries_and_known_keys(torch_cuda):
    P, K, S = 120, 4, 2
    rng = np.random.default_rng(23)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    pr = np.array([[3, 9], [50, 7], [9, 3], [100, 101]], dtype=np.int32)     # pair 2 repeats pair 0
    train = pack_ranks([3, 3, 3, 7, 0], [9, 9, 20, 50, 1], [11, 40, 9 + 100, 60, 2])
    train = np.sort(np.concatenate([train, train[:2]]))                          # repeated keys count once
    tp = np.array([0, 0, 0, 1, 1, 2, 2, 3, 0], dtype=np.int32)
    trc = np.array([5, 5, 11, 60, 8, 5, 40, 0, 119], dtype=np.int32)            # (0, 5) twice; 11 / 60 / 40 are train
    eng = _engine(P, K)
    rank, score, universe = check_against_per_pair(eng, np.stack(thetas), np.stack(prs), cand, pr, train, tp, trc)
    assert rank[0] == rank[1] == rank[5] and score[0] == score[1] == score[5]
    assert rank[2] == 0 and rank[3] == 0 and rank[6] == 0
    assert universe.tolist() == [P - 2 - 2, P - 2 - 1, P - 2 - 2, P - 2]


@pytest.mark.gpu
def test_universe_sizes_zero_one_two(torch_cuda):
    K = 2
    rng = np.random.default_rng(8)
    thetas, prs = random_params(rng, 4, K, 1)
    eng = _engine(4, K)
    th, pp = np.stack(thetas), np.stack(prs)
    # n = 4: |U| = 2, then 1 and 0 with one and two train keys of the pair
    cand = np.array([0, 1, 2, 3], dtype=np.int32)
    pr = np.array([[0, 1]], dtype=np.int32)
    for train, want in [(np.empty(0, np.uint64), 2), (pack_ranks([0], [1], [3]), 1), (pack_ranks([0, 0], [1, 1], [2, 3]), 0)]:
        rank, score, universe = check_against_per_pair(eng, th, pp, cand, pr, train, np.array([0, 0]), np.array([2, 3]))
        assert universe.tolist() == [want]
        assert sorted(rank.tolist()) == ([1, 2] if want == 2 else [0, 1] if want == 1 else [0, 0])
    # n = 3: |U| = 1; n = 2: no partner at all
    rank, score, universe = eng.rank_per_pair(th, pp, cand[:3], np.array([[2, 0]]), np.empty(0, np.uint64), [0], [1])
    assert rank.tolist() == [1] and universe.tolist() == [1]
    rank, score, universe = eng.rank_per_pair(th, pp, cand[:2], np.array([[1, 0]]), np.empty(0, np.uint64), [], [])
    assert universe.tolist() == [0] and len(rank) == 0


@pytest.mark.gpu
def test_bad_entries_are_refused(torch_cuda):
    from trigenicinteractionpredictor_b200 import _cabi
    K = 2
    thetas, prs = random_params(np.random.default_rng(1), 30, K, 1)
    eng = _engine(30, K)
    cand = np.arange(30, dtype=np.int32)
    args = (np.stack(thetas), np.stack(prs), cand)
    none = np.empty(0, np.uint64)
    for pr, tp, trc, msg in [([[0, 30]], [0], [1], "rank 30 of pair 0 is not in"), ([[4, 4]], [0], [1], "same rank twice"),
                             ([[0, 1]], [1], [2], "names pair 1"), ([[0, 1]], [0], [1], "partner rank 1"),
                             ([[0, 1]], [0], [30], "partner rank 30"), ([[0, 1]], [0], [-1], "partner rank -1")]:
        with pytest.raises(_cabi.TipLibraryError, match=msg):
            eng.rank_per_pair(*args, np.array(pr), none, np.array(tp), np.array(trc))


def _heavy_case(rng, P, n_heavy_rows, n_test_row, n_train_row, big_test):
    """Pairs 0 .. n_heavy_rows - 1 share gene 0 and are consecutive in sorted order (one tile); each has n_test_row test
    partners and n_train_row train partners; one more pair (P - 2, P - 1) has big_test test partners and 300 train.
    Partners come from genes no listed pair names, so every pair's train keys are its own; each pair also gets one test
    entry that is a train key."""
    pr = [[0, 1 + i] for i in range(n_heavy_rows)] + [[P - 2, P - 1]]
    others = np.arange(n_heavy_rows + 1, P - 2)
    tp, trc, train = [], [], []
    for q, (a, b) in enumerate(pr):
        nt = big_test if q == len(pr) - 1 else n_test_row
        ntr = 300 if q == len(pr) - 1 else n_train_row
        pick = rng.choice(others, nt + ntr, replace=False)
        tp += [q] * nt
        trc += pick[:nt].tolist()
        t = np.sort(np.stack([np.full(ntr, a), np.full(ntr, b), pick[nt:]], 1), 1)
        train.append(pack_ranks(t[:, 0], t[:, 1], t[:, 2]))
        tp.append(q)
        trc.append(int(pick[nt]))
    return np.array(pr, dtype=np.int32), np.unique(np.concatenate(train)), np.array(tp), np.array(trc)


@pytest.mark.gpu
@pytest.mark.parametrize("K,S", [(4, 1), (32, 12)])
def test_heavy_pairs_take_several_rounds(torch_cuda, K, S):
    """A tile of 64 rows with 300 test and 300 train partners each, and a pair with 2 200 test partners: more entries
    than one round holds in shared memory (2 048, fewer at S K = 384), so the tiles are swept once per round."""
    P = 2600
    rng = np.random.default_rng(64 + K)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    pr, train, tp, trc = _heavy_case(rng, P, 64, 300, 300, 2200)
    rank, score, universe = check_against_per_pair(_engine(P, K), np.stack(thetas), np.stack(prs), cand, pr, train, tp, trc)
    assert (rank == 0).sum() == len(pr)
    assert universe.tolist() == [P - 2 - 300] * len(pr)


@pytest.mark.gpu
def test_p1500_against_tip_score_and_sort(torch_cuda):
    P, K = 1500, 4
    rng = np.random.default_rng(1500)
    thetas, prs = random_params(rng, P, K, 1)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    pr = np.array([rng.choice(P, 2, replace=False) for _ in range(24)], dtype=np.int32)
    train = np.unique(pack_ranks(*np.sort(rng.choice(P, (20000, 3)), 1).T))
    tr = np.stack([(train >> np.uint64(s)) & np.uint64((1 << 21) - 1) for s in (42, 21, 0)], 1).astype(np.int64)
    train = train[(tr[:, 0] < tr[:, 1]) & (tr[:, 1] < tr[:, 2])]
    tp = np.repeat(np.arange(len(pr)), 40)
    trc = np.concatenate([rng.choice([x for x in range(P) if x not in (a, b)], 40, replace=False) for a, b in pr.tolist()])
    rank, score, universe = eng.rank_per_pair(np.stack(thetas), np.stack(prs), cand, pr, train, tp, trc)
    tset = set(int(x) for x in train.tolist())
    for q, (a, b) in enumerate(pr.tolist()):
        a, b = sorted((a, b))
        c = np.array([x for x in range(P) if x not in (a, b)])
        tri = np.sort(np.stack([np.full(len(c), a), np.full(len(c), b), c], 1), 1)
        known = np.array([(int(x) << 42 | int(y) << 21 | int(z)) in tset for x, y, z in tri.tolist()])
        s = eng.score_sum(np.stack(thetas), np.stack(prs), cand[tri])
        c, s = c[~known], s[~known]
        order = np.lexsort((c, -s))
        c, s = c[order], s[order]
        first, last = near_tie_runs(s)
        where = {int(x): i for i, x in enumerate(c.tolist())}
        assert universe[q] == len(c)
        for j in np.flatnonzero(tp == q).tolist():
            if int(trc[j]) not in where:
                assert rank[j] == 0
                continue
            i = where[int(trc[j])]
            assert first[i] <= rank[j] <= last[i]
            assert abs(score[j] - s[i]) <= TOL * s[i]


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3])
def test_golden_base(torch_cuda, K):
    m = _trained_base_model(K)
    res = m.rank_held_out_per_pair()
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
def test_train_with_save_params_then_predict_cli_held_out_pairs(torch_cuda, tmp_path):
    from trigenicinteractionpredictor_b200 import Model, main
    from trigenicinteractionpredictor_b200.predict import main as predict_main
    out = str(tmp_path) + os.sep
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["-t", tr, "-e", te, "-k", "2", "-i", "300", "-f", "5", "-b", "10", "-n", "2", "-o", out,
                 "--seed", "1000", "--save-params"]) == 0
    params = [out + "Sample_0_K2.npz", out + "Sample_1_K2.npz"]
    mm = Model()
    mm.get_traintest(tr, te)
    for with_pairs in (False, True):
        pred = str(tmp_path / "held_pairs.tsv")
        argv = ["-t", tr, "-e", te, "-p", params[0], "-p", params[1], "--held-out-pairs", "-o", pred]
        pairs = None
        if with_pairs:
            keys = list(mm.test_links)[:5]
            pairs = [(mm.id_gene[int(k.split("_")[0])], mm.id_gene[int(k.split("_")[2])]) for k in keys]
            pairs = list(dict.fromkeys(pairs))
            (tmp_path / "pairs.txt").write_text("".join("%s+%s\n" % p for p in pairs))
            argv += ["-r", str(tmp_path / "pairs.txt")]
        assert predict_main(argv) == 0
        text = open(pred, encoding="utf-8").read().split("\n")
        hdr = text.index("Query pair\tRank\tPair universe\tPredicted Interaction\tReal Interaction\tID of genes\tGenes")
        summary = dict(line.split(":\t") for line in text[:hdr])
        want = mm.rank_held_out_per_pair(pairs, params=params)
        assert int(summary["Views"]) == want["views"] and int(summary["Positive views"]) == want["positives"]
        assert int(summary["Query pairs"]) == len(want["pairs"])
        assert summary["Hits at 20"] == str(want["hits_at"][20]["positives"]) or want["hits_at"][20]["positives"] is None
        body = [ln.split("\t") for ln in text[hdr + 1:] if ln]
        assert len(body) == len(want["rows"])
        for b, r in zip(body, want["rows"]):
            assert b[0] == r[0] and int(b[1]) == r[5] and int(b[2]) == r[6] and float(b[3]) == r[4]
            assert int(b[4]) == r[3] and b[5] == r[1] and b[6] == r[2]
