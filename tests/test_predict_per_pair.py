"""Prediction per query pair: for every pair of genes, the top-N unseen triplets that contain both (tip_top_triplets_per_pair,
EMEngine.top_triplets_per_pair, Model.predict_top_triplets_per_pair, predict -r).

The per-pair oracle is the exhaustive `top_triplets_np` of tests/test_predict.py (itself pinned to
oracle.mmsbm_oracle.predict_loops) over all triplets, filtered to the rows that contain both ranks of the pair."""
import ctypes
import itertools
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from tests.test_predict import BASE, TOL, _digested, _trained_base_model, check_against_oracle, pack_ranks, random_params, \
    top_triplets_np

MASK = np.uint64((1 << 21) - 1)


def all_triplets_oracle(thetas, prs, cand, known):
    """(ids, scores, rank triples [m][3]) of every unseen triplet, best first (score descending, packed ranks ascending)."""
    nc = len(cand)
    ids, sc, k = top_triplets_np(thetas, prs, cand, known, nc * (nc - 1) * (nc - 2) // 6)
    r = np.stack([(k >> np.uint64(42)) & MASK, (k >> np.uint64(21)) & MASK, k & MASK], 1).astype(np.int64)
    return ids, sc, r


def per_pair_oracle(allt, ra, rb):
    """The rows of the all-triplet oracle that contain both ranks, in its order."""
    ids, sc, r = allt
    has = (r == ra).any(axis=1) & (r == rb).any(axis=1)
    return ids[has], sc[has]


def _known(rng, P, m):
    kr = np.sort(rng.choice(P, size=(m, 3), replace=True), axis=1)
    kr = kr[(kr[:, 0] < kr[:, 1]) & (kr[:, 1] < kr[:, 2])]
    return np.unique(pack_ranks(kr[:, 0], kr[:, 1], kr[:, 2]))


def _n_known_of_pair(known, ra, rb):
    k = np.asarray(known, dtype=np.uint64)
    r = np.stack([(k >> np.uint64(42)) & MASK, (k >> np.uint64(21)) & MASK, k & MASK], 1).astype(np.int64)
    return int(((r == ra).any(axis=1) & (r == rb).any(axis=1)).sum())


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_filtered_oracle_equals_itertools_brute_force(S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(30 + S)
    P, K = 21, 3
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str))
    known = pack_ranks([0, 0, 3, 5], [1, 4, 10, 6], [7, 20, 20, 12])
    known_set = set(int(x) for x in known.tolist())
    tl, pl = [t.tolist() for t in thetas], [p.tolist() for p in prs]
    allt = all_triplets_oracle(thetas, prs, cand, known)
    # rank edges, adjacent ranks (no middle region), and a pair given in reverse order
    for a, b in [(0, 1), (0, P - 1), (P - 2, P - 1), (5, 6), (12, 3), (10, 20)]:
        o_ids, o_sc = per_pair_oracle(allt, min(a, b), max(a, b))
        rows = []
        for c in range(P):
            if c in (a, b):
                continue
            ra, rb, rc = sorted((a, b, c))
            pk = (ra << 42) | (rb << 21) | rc
            if pk in known_set:
                continue
            x, y, z = (int(cand[i]) for i in (ra, rb, rc))
            s = sum(orc.predict_loops(t, p, x, y, z) for t, p in zip(tl, pl)) / S
            rows.append((-s, c, (x, y, z)))
        rows.sort()
        assert len(rows) == len(o_sc) == P - 2 - _n_known_of_pair(known, min(a, b), max(a, b))
        assert np.max(np.abs(o_sc + np.array([x[0] for x in rows])) / o_sc) < TOL
        check_against_oracle(o_ids, o_sc, np.array([x[2] for x in rows]), -np.array([x[0] for x in rows]), len(rows))


def test_workspace_bytes_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_top_triplets_per_pair_workspace_bytes(100, 500, 10, 2, 0, 20, ctypes.byref(nb)) == 0 and nb.value > 0
    for args in [(100, 10, 10, 39, 0, 20),          # S K = 390 > 384
                 (1 << 21, 1 << 20, 2, 1, 0, 17),   # n_pairs N > 2^24
                 (100, -1, 2, 1, 0, 1), (100, 10, 2, 1, 0, -1), (-1, 10, 2, 1, 0, 1), (100, 10, 2, 1, -1, 1)]:
        assert lib.tip_top_triplets_per_pair_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"n_pairs*N <= 2^24" in lib.tip_last_error() and b"S*K <= 384" in lib.tip_last_error()
    assert lib.tip_top_triplets_per_pair_workspace_bytes(1 << 21, 1 << 20, 2, 1, 0, 16, ctypes.byref(nb)) == 0


def test_model_refusals():
    random.seed(2)
    m = _digested()
    m.initialize_parameters(2)
    g = [m.id_gene[i] for i in range(4)]
    for pairs, genes, msg in [([("NOPE", g[0])], None, "unknown gene names: NOPE"),
                              ([(g[0], "NOPE2")], [g[1], "NOPE3"], "NOPE2, NOPE3"),
                              ([(g[0], g[1]), (g[2], g[2])], None, "a pair of one gene: %s\\+%s" % (g[2], g[2])),
                              ([(g[0], g[1]), (g[2], g[3]), (g[1], g[0])], None, "duplicate pairs: "),
                              ([(g[0], g[1]), (g[0], g[1])], None, "duplicate pairs: "),
                              ([(g[0], g[1], g[2])], None, "a pair is not two gene names"),
                              ([], None, "pairs is empty")]:
        with pytest.raises(ValueError, match=msg):
            m.predict_top_triplets_per_pair(pairs, 5, genes=genes)
    with pytest.raises(ValueError, match="n must be >= 0"):
        m.predict_top_triplets_per_pair([(g[0], g[1])], -1)
    with pytest.raises(ValueError, match="predict_top_triplets_per_pair: params is empty"):
        m.predict_top_triplets_per_pair([(g[0], g[1])], 5, params=[])
    with pytest.raises(ValueError, match="predict_top_triplets_per_pair needs a model digested"):
        from trigenicinteractionpredictor_b200 import Model
        Model().predict_top_triplets_per_pair([(g[0], g[1])], 5)


def test_cli_pair_file_errors(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    base = ["-t", tr, "-e", te, "-p", good]
    g = [m.id_gene[i] for i in range(4)]
    assert main(base + ["-r", str(tmp_path / "missing.txt")]) == 2
    cases = {"empty": ("\n  \n", "names no pair"),
             "malformed_one": ("%s+%s\n%s\n" % (g[0], g[1], g[2]), "line 2"),
             "malformed_three": ("%s %s %s\n" % (g[0], g[1], g[2]), "line 1"),
             "malformed_plus": ("%s+%s+%s\n" % (g[0], g[1], g[2]), "line 1"),
             "malformed_empty_name": ("%s+\n" % g[0], "line 1"),
             "unknown": ("%s+NOPE1\nNOPE2 %s\n" % (g[0], g[1]), "NOPE1, NOPE2"),
             "one_gene": ("%s+%s\n%s+%s\n" % (g[0], g[1], g[2], g[2]), "a pair of one gene: %s+%s" % (g[2], g[2])),
             "twice": ("%s+%s\n%s %s\n%s+%s\n" % (g[0], g[1], g[2], g[3], g[1], g[0]), "pairs listed twice: %s+%s" % (g[1], g[0]))}
    for name, (text, msg) in cases.items():
        f = tmp_path / (name + ".txt")
        f.write_text(text)
        assert main(base + ["--pairs", str(f)]) == 2, name
        assert msg in capsys.readouterr().err, name
    pf, qf = tmp_path / "p.txt", tmp_path / "q.txt"
    pf.write_text("%s+%s\n" % (g[0], g[1]))
    qf.write_text("%s\n" % g[0])
    assert main(base + ["-r", str(pf), "-q", str(qf)]) == 2
    assert "exclude each other" in capsys.readouterr().err


def test_sass_pair_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    body = [f for f in out.split("Function : ") if f.split("\n", 1)[0].find("tip_pair_pass_kernel") >= 0]
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
def test_per_pair_matches_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(P * 100 + K * 10 + S + 11)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = _known(rng, P, 3000 if P == 130 else 400)
    if P == 40:
        pr = np.array(list(itertools.combinations(range(P), 2)), dtype=np.int32)
    else:
        edges = [(0, 1), (0, P - 1), (P - 2, P - 1), (1, 2), (64, 65), (77, 3), (P - 1, 0)]
        rand = rng.choice(P, size=(400, 2))
        rand = rand[rand[:, 0] != rand[:, 1]][:200]
        pr = np.array(edges + rand.tolist(), dtype=np.int32)
    pr = pr[rng.permutation(len(pr))]
    pr[::2] = pr[::2, ::-1]                      # either order
    allt = all_triplets_oracle(thetas, prs, cand, known)
    oracle = [per_pair_oracle(allt, min(a, b), max(a, b)) for a, b in pr.tolist()]
    eng = _engine(P, K)
    for n in (1, 7, P - 2):
        ids, sc, cnt = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, pr, known, n)
        assert ids.shape[:2] == sc.shape and len(cnt) == len(pr)
        for qi, (a, b) in enumerate(pr.tolist()):
            o_ids, o_sc = oracle[qi]
            assert cnt[qi] == min(n, len(o_sc))
            check_against_oracle(ids[qi, :cnt[qi]], sc[qi, :cnt[qi]], o_ids, o_sc, n)
            if n == P - 2:
                assert cnt[qi] == P - 2 - _n_known_of_pair(known, min(a, b), max(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("P,n", [(30, 40), (80, 1), (300, 10), (300, 298)],
                         ids=["fits_buffer", "selects_on_ranks", "large", "whole_row"])
def test_all_scores_tied_gives_rank_order(torch_cuda, P, n):
    """Identical theta rows and dyadic parameters: every score is the same number in any summation order.  At P = 80 and
    300 a pair's partners exceed its buffer (4 N + 64), so its threshold has to continue on rc."""
    K = 3
    theta = np.tile(np.array([0.5, 0.25, 0.25]), (P, 1))
    rng = np.random.default_rng(3)
    p1 = rng.integers(1, 4, size=(K, K, K)) / 4.0
    pr = np.stack([1.0 - p1, p1], axis=3)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    pairs = np.array([(0, 1), (1, 0), (0, P - 1), (P - 2, P - 1), (P // 3, P // 2), (P - 1, 5)], dtype=np.int32)
    ids, sc, cnt = _engine(P, K).top_triplets_per_pair(theta[None], pr[None], cand, pairs, np.empty(0, dtype=np.uint64), n)
    for qi, (a, b) in enumerate(pairs.tolist()):
        m = min(n, P - 2)
        assert cnt[qi] == m and np.all(sc[qi, :m] == sc[qi, 0])
        want = [tuple(cand[sorted((a, b, c))].tolist()) for c in range(P) if c not in (a, b)][:m]
        assert [tuple(x) for x in ids[qi, :m].tolist()] == want


@pytest.mark.gpu
def test_consistent_with_per_gene(torch_cuda):
    """The per-gene list of gene a over all its C(n - 1, 2) pairs, filtered to the rows that contain b, is the per-pair list
    of (a, b): same rows in the same order, scores within TOL."""
    P, K, S = 40, 4, 2
    rng = np.random.default_rng(44)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = _known(rng, P, 600)
    eng = _engine(P, K)
    qr = np.arange(P, dtype=np.int32)
    g_ids, g_sc, g_cnt = eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand, qr, known, (P - 1) * (P - 2) // 2)
    pairs = np.array([(a, b) for a in range(0, P, 3) for b in range(P) if b != a], dtype=np.int32)
    ids, sc, cnt = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, pairs, known, P - 2)
    for qi, (a, b) in enumerate(pairs.tolist()):
        gb = cand[b]
        rows = [(tuple(t), s) for t, s in zip(g_ids[a, :g_cnt[a]].tolist(), g_sc[a, :g_cnt[a]].tolist()) if gb in t]
        assert cnt[qi] == len(rows)
        assert [tuple(t) for t in ids[qi, :cnt[qi]].tolist()] == [t for t, _ in rows]
        assert np.all(np.abs(sc[qi, :cnt[qi]] - np.array([s for _, s in rows])) <= TOL * sc[qi, :cnt[qi]])


@pytest.mark.gpu
def test_bad_pair_ranks_are_refused(torch_cuda):
    torch = torch_cuda
    from trigenicinteractionpredictor_b200 import _cabi
    P, K = 50, 3
    rng = np.random.default_rng(8)
    thetas, prs = random_params(rng, P, K, 1)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    none = np.empty(0, dtype=np.uint64)
    for pr, msg in [([[3, 4], [1, 50]], "rank 50 of pair 1 is not in \\[0, 50\\)"), ([[-1, 2]], "rank -1 of pair 0"),
                    ([[4, 9], [7, 7]], "pair 1 has the same rank twice \\(7\\)")]:
        with pytest.raises(_cabi.TipLibraryError, match=msg):
            eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, np.array(pr, dtype=np.int32), none, 5)
        assert eng.lib.tip_top_triplets_per_pair_last_passes() == 0     # refused before any sweep
    torch.cuda.synchronize()
    ids, sc, cnt = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, np.array([[4, 9], [9, 4]], dtype=np.int32),
                                             none, 5)
    assert list(cnt) == [5, 5] and np.array_equal(ids[0], ids[1]) and np.array_equal(sc[0], sc[1])


@pytest.mark.gpu
def test_p1500_against_tip_score_and_sort(torch_cuda):
    """300 random pairs: every partner scored through tip_score, sorted by (score descending, rc ascending)."""
    torch = torch_cuda
    P, K, N = 1500, 4, 50
    rng = np.random.default_rng(151)
    thetas, prs = random_params(rng, P, K, 1)
    cand_np = np.array(sorted(range(P), key=str), dtype=np.int32)
    pr = rng.choice(P, size=(600, 2))
    pr = pr[pr[:, 0] != pr[:, 1]][:300].astype(np.int32)
    eng = _engine(P, K)
    ids, sc, cnt = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand_np, pr, np.empty(0, dtype=np.uint64), N)
    assert eng.lib.tip_top_triplets_per_pair_last_passes() <= 3     # two for continuous scores, a third for a rare overflow
    eng.set_params(thetas[0], prs[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)
    a = torch.from_numpy(pr.min(axis=1).astype(np.int64)).to(dev)[:, None].expand(-1, P - 2)
    b = torch.from_numpy(pr.max(axis=1).astype(np.int64)).to(dev)[:, None].expand(-1, P - 2)
    c = torch.arange(P - 2, device=dev)[None, :].expand(len(pr), -1)
    c = c + (c >= a).long()
    c = c + (c >= b).long()                      # every rank but a and b, ascending
    rr = torch.stack([a, b, c], 2).reshape(-1, 3).sort(dim=1).values
    g = cand[rr].to(torch.int32)
    g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
    out = torch.empty(rr.shape[0], dtype=torch.float64, device=dev)
    assert eng.lib.tip_score(P, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()), ctypes.c_void_p(g3.data_ptr()),
                             rr.shape[0], ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                             ctypes.c_void_p(out.data_ptr()), eng._stream()) == 0
    scores = out.reshape(len(pr), P - 2).cpu().numpy()
    gids = g.reshape(len(pr), P - 2, 3).cpu().numpy()
    for qi in range(len(pr)):
        order = np.argsort(-scores[qi], kind="stable")      # rc ascending within equal scores
        assert cnt[qi] == N
        check_against_oracle(ids[qi], sc[qi], gids[qi][order], scores[qi][order], N)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 10])
def test_golden_base_rows_are_do_prediction_of_their_keys(torch_cuda, K):
    m = _trained_base_model(K)
    rng = np.random.default_rng(K + 50)
    genes = rng.choice(m.P, size=24, replace=False).tolist()
    pairs = [(m.id_gene[genes[2 * i]], m.id_gene[genes[2 * i + 1]]) for i in range(12)]
    res = m.predict_top_triplets_per_pair(pairs, 30)
    assert list(res) == pairs
    known = set(m.links.keys()) | set(m.test_links.keys())
    for (qa, qb), rows in res.items():
        assert len(rows) == 30
        ida, idb = str(m.gene_id[qa]), str(m.gene_id[qb])
        prev = None
        for s, key, names in rows:
            a, b, c = key.split("_")
            assert ida in (a, b, c) and idb in (a, b, c)
            assert sorted([a, b, c]) == [a, b, c]
            assert key not in known
            assert abs(s - m.do_prediction(a, b, c)) <= TOL * s
            assert names == "_".join(sorted(m.id_gene[int(x)] for x in (a, b, c)))
            assert prev is None or s <= prev
            prev = s


@pytest.mark.gpu
def test_train_with_save_params_then_predict_cli_pairs(torch_cuda, tmp_path):
    from trigenicinteractionpredictor_b200 import Model, main
    from trigenicinteractionpredictor_b200.predict import main as predict_main
    out = str(tmp_path) + os.sep
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["-t", tr, "-e", te, "-k", "2", "-i", "300", "-f", "5", "-b", "10", "-n", "2", "-o", out,
                 "--seed", "1000", "--save-params"]) == 0
    models = []
    for s in (0, 1):
        mm = Model()
        mm.get_traintest(tr, te)
        mm.load_parameters(out + "Sample_%d_K2.npz" % s)
        models.append(mm)
    g = models[0].id_gene
    pairs = [(g[17], g[3]), (g[60], g[2]), (g[5], g[40])]
    pfile = tmp_path / "pairs.txt"
    pfile.write_text("%s+%s\n\n%s %s\n%s\t%s\n" % (pairs[0] + pairs[1] + pairs[2]))
    pred = str(tmp_path / "pred.tsv")
    assert predict_main(["-t", tr, "-e", te, "-p", out + "Sample_0_K2.npz", "--params", out + "Sample_1_K2.npz",
                         "-n", "15", "-r", str(pfile), "-o", pred]) == 0
    lines = open(pred, encoding="utf-8").read().split("\n")
    assert lines[0] == "Query pair\tPredicted Interaction\tID of genes\tGenes" and lines[-1] == ""
    assert len(lines) == 2 + 3 * 15
    assert [ln.split("\t")[0] for ln in lines[1:-1]] == [a + "+" + b for a, b in pairs for _ in range(15)]
    want = models[0].predict_top_triplets_per_pair(pairs, 15, params=[out + "Sample_0_K2.npz", out + "Sample_1_K2.npz"])
    got = [ln.split("\t") for ln in lines[1:-1]]
    exp = [(a + "+" + b, s, key, names) for a, b in pairs for s, key, names in want[(a, b)]]
    assert [(q, key, names) for q, _, key, names in got] == [(q, key, names) for q, _, key, names in exp]
    for (q, score, key, names), (_, s, _, _) in zip(got, exp):
        assert float(score) == s
        a, b, c = key.split("_")
        pa, pb = q.split("+")
        assert str(models[0].gene_id[pa]) in (a, b, c) and str(models[0].gene_id[pb]) in (a, b, c)
        mean = (models[0].do_prediction(a, b, c) + models[1].do_prediction(a, b, c)) / 2
        assert abs(float(score) - mean) <= TOL * mean
        assert key not in models[0].links and key not in models[0].test_links


@pytest.mark.gpu
@pytest.mark.parametrize("n", [20, 150])
def test_most_partners_score_zero(torch_cuda, n):
    """One-hot theta rows and a p with a single non-zero entry: most partners of a pair score exactly 0, far below the
    row's first counting range.  At N = 20 a pair's 198 partners exceed its buffer (4 N + 64), so the row starts by
    counting and has to count down to zero, then settle the run of zeros on rc; at N = 150 the whole row fits the buffer
    and the long run of zeros is ordered by rc.  Scores are dyadic, so exact."""
    P, K = 200, 3
    cls = np.arange(P) % K
    theta = np.eye(K)[cls]
    p1 = np.zeros((K, K, K))
    p1[0, 1, 2] = 0.5
    p1[1, 1, 0] = 0.25
    pr = np.stack([1.0 - p1, p1], axis=3)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    rng = np.random.default_rng(9)
    known = _known(rng, P, 3000)
    known_set = set(int(x) for x in known.tolist())
    pairs = np.array([(0, 1), (5, 7), (P - 1, 3), (10, 11), (40, 120), (2, 4)], dtype=np.int32)
    eng = _engine(P, K)
    ids, sc, cnt = eng.top_triplets_per_pair(theta[None], pr[None], cand, pairs, known, n)
    assert eng.lib.tip_top_triplets_per_pair_last_passes() <= 16
    for qi, (a, b) in enumerate(pairs.tolist()):
        rows = []
        for c in range(P):
            if c in (a, b):
                continue
            r = sorted((a, b, c))
            if (r[0] << 42) | (r[1] << 21) | r[2] in known_set:
                continue
            g = cand[r]
            rows.append((-p1[cls[g[0]], cls[g[1]], cls[g[2]]], c, tuple(g.tolist())))
        rows.sort()
        m = min(n, len(rows))
        assert cnt[qi] == m
        assert [tuple(t) for t in ids[qi, :m].tolist()] == [x[2] for x in rows[:m]]
        assert sc[qi, :m].tolist() == [-x[0] for x in rows[:m]]


@pytest.mark.gpu
def test_repeated_known_keys_count_once(torch_cuda):
    P, K = 60, 3
    rng = np.random.default_rng(12)
    thetas, prs = random_params(rng, P, K, 1)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = _known(rng, P, 800)
    pairs = np.array([(0, 1), (3, 40), (P - 1, 7)], dtype=np.int32)
    eng = _engine(P, K)
    want = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, pairs, known, P - 2)
    got = eng.top_triplets_per_pair(np.stack(thetas), np.stack(prs), cand, pairs, np.repeat(known, 3), P - 2)
    assert np.array_equal(want[2], got[2]) and np.array_equal(want[0], got[0]) and np.array_equal(want[1], got[1], equal_nan=True)
