"""Prediction per gene: for every query gene, the top-N unseen triplets that contain it (tip_top_triplets_per_gene,
EMEngine.top_triplets_per_gene, Model.predict_top_triplets_per_gene, predict -q).

The per-query oracle is the exhaustive `top_triplets_np` of tests/test_predict.py (itself pinned to
oracle.mmsbm_oracle.predict_loops) over all triplets, filtered to the rows that contain the query's rank."""
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


def per_query_oracle(thetas, prs, cand, known, r):
    """(ids, scores) of every unseen triplet containing rank r, best first (score descending, packed ranks ascending)."""
    nc = len(cand)
    ids, sc, k = top_triplets_np(thetas, prs, cand, known, nc * (nc - 1) * (nc - 2) // 6)
    ru = np.uint64(r)
    has = ((k >> np.uint64(42)) & MASK == ru) | ((k >> np.uint64(21)) & MASK == ru) | (k & MASK == ru)
    return ids[has], sc[has]


def n_pairs(m):
    return m * (m - 1) // 2


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_filtered_oracle_equals_itertools_brute_force(S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(20 + S)
    P, K = 21, 3
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str))
    known = pack_ranks([0, 1, 3], [4, 6, 10], [7, 19, 20])
    known_set = set(int(x) for x in known.tolist())
    tl, pl = [t.tolist() for t in thetas], [p.tolist() for p in prs]
    for r in (0, 1, 7, P - 2, P - 1):
        o_ids, o_sc = per_query_oracle(thetas, prs, cand, known, r)
        rows = []
        for x, y in itertools.combinations([i for i in range(P) if i != r], 2):
            ra, rb, rc = sorted((r, x, y))
            pk = (ra << 42) | (rb << 21) | rc
            if pk in known_set:
                continue
            a, b, c = (int(cand[i]) for i in (ra, rb, rc))
            s = sum(orc.predict_loops(t, p, a, b, c) for t, p in zip(tl, pl)) / S
            rows.append((-s, pk, (a, b, c)))
        rows.sort()
        assert len(rows) == len(o_sc) == n_pairs(P - 1) - sum(r in (ra, rb, rc) for ra, rb, rc in
                                                               [(0, 4, 7), (1, 6, 19), (3, 10, 20)])
        assert np.max(np.abs(o_sc + np.array([x[0] for x in rows])) / o_sc) < TOL
        check_against_oracle(o_ids, o_sc, np.array([x[2] for x in rows]), -np.array([x[0] for x in rows]), len(rows))


def test_workspace_bytes_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_top_triplets_per_gene_workspace_bytes(100, 50, 10, 2, 0, 20, ctypes.byref(nb)) == 0 and nb.value > 0
    for args in [(100, 101, 10, 1, 0, 20),          # n_query > n_cand
                 (100, 10, 10, 39, 0, 20),          # S K = 390 > 384
                 (1 << 21, 1 << 20, 2, 1, 0, 17),   # n_query N > 2^24
                 (100, -1, 2, 1, 0, 1), (100, 10, 2, 1, 0, -1)]:
        assert lib.tip_top_triplets_per_gene_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"n_query*N <= 2^24" in lib.tip_last_error() and b"S*K <= 384" in lib.tip_last_error()
    assert lib.tip_top_triplets_per_gene_workspace_bytes(1 << 21, 1 << 20, 2, 1, 0, 16, ctypes.byref(nb)) == 0


def test_model_refusals():
    random.seed(2)
    m = _digested()
    m.initialize_parameters(2)
    g = [m.id_gene[i] for i in range(4)]
    for queries, genes, msg in [(["NOPE"], None, "unknown gene names: NOPE"),
                                ([g[0], "NOPE2"], [g[1], "NOPE3"], "NOPE2, NOPE3"),
                                ([g[0], g[1], g[0]], None, "duplicate query genes: " + g[0]),
                                ([], None, "queries is empty")]:
        with pytest.raises(ValueError, match=msg):
            m.predict_top_triplets_per_gene(queries, 5, genes=genes)
    with pytest.raises(ValueError, match="n must be >= 0"):
        m.predict_top_triplets_per_gene(g[:2], -1)
    with pytest.raises(ValueError, match="predict_top_triplets_per_gene: params is empty"):
        m.predict_top_triplets_per_gene(g[:2], 5, params=[])
    with pytest.raises(ValueError, match="predict_top_triplets_per_gene needs a model digested"):
        from trigenicinteractionpredictor_b200 import Model
        Model().predict_top_triplets_per_gene(g[:2], 5)


def test_cli_query_file_errors(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    base = ["-t", tr, "-e", te, "-p", good]
    g = [m.id_gene[i] for i in range(3)]
    assert main(base + ["-q", str(tmp_path / "missing.txt")]) == 2
    cases = {"empty": ("\n  \n", "names no gene"),
             "unknown": ("%s\nNOPE1\n%s\nNOPE2\n" % (g[0], g[1]), "NOPE1, NOPE2"),
             "twice": ("%s\n%s\n%s\n%s\n" % (g[0], g[1], g[0], g[0]), "listed twice: " + g[0])}
    for name, (text, msg) in cases.items():
        f = tmp_path / (name + ".txt")
        f.write_text(text)
        assert main(base + ["--queries", str(f)]) == 2, name
        assert msg in capsys.readouterr().err


def test_sass_query_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    body = [f for f in out.split("Function : ") if f.split("\n", 1)[0].find("tip_query_pass_kernel") >= 0]
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


def _known(rng, P, m):
    kr = np.sort(rng.choice(P, size=(m, 3), replace=True), axis=1)
    kr = kr[(kr[:, 0] < kr[:, 1]) & (kr[:, 1] < kr[:, 2])]
    return np.unique(pack_ranks(kr[:, 0], kr[:, 1], kr[:, 2]))


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 3])
@pytest.mark.parametrize("K", [1, 2, 3, 4, 10, 32])
@pytest.mark.parametrize("P", [40, 130])
def test_per_gene_matches_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(P * 100 + K * 10 + S + 7)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = _known(rng, P, 400)
    qr = list(range(P)) if P == 40 else [0, 1, P // 2, P - 2, P - 1, 77]
    qr = rng.permutation(qr).astype(np.int32)
    oracle = {int(r): per_query_oracle(thetas, prs, cand, known, r) for r in qr}
    eng = _engine(P, K)
    allp = n_pairs(P - 1)
    for n in (1, 10, allp):
        ids, sc, cnt = eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand, qr, known, n)
        assert ids.shape[:2] == sc.shape and len(cnt) == len(qr)
        for qi, r in enumerate(qr.tolist()):
            o_ids, o_sc = oracle[r]
            assert cnt[qi] == min(n, len(o_sc))
            check_against_oracle(ids[qi, :cnt[qi]], sc[qi, :cnt[qi]], o_ids, o_sc, n)
            if n == allp:
                k_r = sum(1 for k in known.tolist() if r in ((k >> 42) & 0x1FFFFF, (k >> 21) & 0x1FFFFF, k & 0x1FFFFF))
                assert cnt[qi] == allp - k_r


@pytest.mark.gpu
@pytest.mark.parametrize("P,n", [(30, 406), (80, 10), (200, 40)], ids=["fits_buffer", "selects_on_ranks", "large"])
def test_all_scores_tied_gives_rank_order(torch_cuda, P, n):
    """Identical theta rows: every score is the same number.  At P = 80 and 200 a query's pairs (3 081, 19 701) exceed
    its buffer (4 N + 256), so its threshold has to continue on the packed rank triple."""
    K = 3
    rng = np.random.default_rng(1)
    theta = np.tile(rng.dirichlet(np.ones(K)), (P, 1))
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    qr = np.array([0, 1, P // 3, P - 2, P - 1], dtype=np.int32)
    ids, sc, cnt = _engine(P, K).top_triplets_per_gene(theta[None], pr[None], cand, qr, np.empty(0, dtype=np.uint64), n)
    for qi, r in enumerate(qr.tolist()):
        assert cnt[qi] == n and np.all(sc[qi] == sc[qi, 0])
        want = [tuple(cand[list(t)].tolist()) for t in itertools.islice(
            (t for t in itertools.combinations(range(P), 3) if r in t), n)]
        assert [tuple(x) for x in ids[qi].tolist()] == want


@pytest.mark.gpu
def test_consistent_with_global_top_triplets(torch_cuda):
    """Every gene a query: the global top M rows that contain a gene are in its list (M <= N) with the same score."""
    P, K, S, M, N = 130, 4, 2, 60, 60
    rng = np.random.default_rng(33)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    known = _known(rng, P, 2000)
    eng = _engine(P, K)
    g_ids, g_sc = eng.top_triplets(np.stack(thetas), np.stack(prs), cand, known, M)
    qr = np.arange(P, dtype=np.int32)
    ids, sc, cnt = eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand, qr, known, N)
    rank = {g: r for r, g in enumerate(cand.tolist())}
    seen = 0
    for qi in range(P):
        mine = {tuple(t): s for t, s in zip(ids[qi, :cnt[qi]].tolist(), sc[qi, :cnt[qi]].tolist())}
        for t, s in zip(g_ids.tolist(), g_sc.tolist()):
            if qi in (rank[t[0]], rank[t[1]], rank[t[2]]):
                assert abs(mine[tuple(t)] - s) <= 1e-12 * s
                seen += 1
    assert seen == 3 * M


@pytest.mark.gpu
def test_bad_query_ranks_are_refused(torch_cuda):
    torch = torch_cuda
    from trigenicinteractionpredictor_b200 import _cabi
    P, K = 50, 3
    rng = np.random.default_rng(8)
    thetas, prs = random_params(rng, P, K, 1)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    none = np.empty(0, dtype=np.uint64)
    for qr, msg in [([3, 50], "query rank 50 of query 1 is not in \\[0, 50\\)"), ([-1], "query rank -1"),
                    ([4, 9, 4], "query rank 4 appears twice")]:
        with pytest.raises(_cabi.TipLibraryError, match=msg):
            eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand, np.array(qr, dtype=np.int32), none, 5)
        assert eng.lib.tip_top_triplets_per_gene_last_passes() == 0     # refused before any sweep
    torch.cuda.synchronize()
    ids, sc, cnt = eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand, np.array([4, 9], dtype=np.int32), none, 5)
    assert list(cnt) == [5, 5]


@pytest.mark.gpu
def test_p1500_against_chunked_tip_score_and_topk(torch_cuda):
    """A few queries' 1.1e6 pairs each scored through tip_score, ranked with torch.topk."""
    torch = torch_cuda
    P, K, N = 1500, 4, 200
    rng = np.random.default_rng(150)
    thetas, prs = random_params(rng, P, K, 1)
    cand_np = np.array(sorted(range(P), key=str), dtype=np.int32)
    qr = np.array([0, 5, 731, P - 2, P - 1], dtype=np.int32)
    eng = _engine(P, K)
    ids, sc, cnt = eng.top_triplets_per_gene(np.stack(thetas), np.stack(prs), cand_np, qr, np.empty(0, dtype=np.uint64), N)
    eng.set_params(thetas[0], prs[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)
    for qi, r in enumerate(qr.tolist()):
        others = torch.tensor([i for i in range(P) if i != r], device=dev)
        X, Y = torch.meshgrid(others, others, indexing="ij")
        keep = X < Y
        rr = torch.stack([X[keep], Y[keep], torch.full_like(X[keep], r)], 1).sort(dim=1).values
        g = cand[rr].to(torch.int32)
        g1, g2, g3 = (g[:, i].contiguous() for i in range(3))
        out = torch.empty(rr.shape[0], dtype=torch.float64, device=dev)
        assert eng.lib.tip_score(P, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()),
                                 ctypes.c_void_p(g3.data_ptr()), rr.shape[0], ctypes.c_void_p(eng.theta.data_ptr()),
                                 ctypes.c_void_p(eng.p.data_ptr()), ctypes.c_void_p(out.data_ptr()), eng._stream()) == 0
        keys = (rr[:, 0] << 42) | (rr[:, 1] << 21) | rr[:, 2]
        v, i = torch.topk(out, N + 64)
        order = np.lexsort((keys[i].cpu().numpy(), -v.cpu().numpy()))
        o_sc = v.cpu().numpy()[order]
        k = keys[i].cpu().numpy()[order]
        m = (1 << 21) - 1
        o_ids = cand_np[np.stack([(k >> 42) & m, (k >> 21) & m, k & m], 1)]
        assert cnt[qi] == N
        check_against_oracle(ids[qi], sc[qi], o_ids, o_sc, N)


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 10])
def test_golden_base_rows_are_do_prediction_of_their_keys(torch_cuda, K):
    m = _trained_base_model(K)
    rng = np.random.default_rng(K)
    queries = [m.id_gene[i] for i in rng.choice(m.P, size=12, replace=False).tolist()]
    res = m.predict_top_triplets_per_gene(queries, 30)
    assert list(res) == queries
    known = set(m.links.keys()) | set(m.test_links.keys())
    for q, rows in res.items():
        assert len(rows) == 30
        qid = str(m.gene_id[q])
        prev = None
        for s, key, names in rows:
            a, b, c = key.split("_")
            assert qid in (a, b, c)
            assert sorted([a, b, c]) == [a, b, c]
            assert key not in known
            assert abs(s - m.do_prediction(a, b, c)) <= TOL * s
            assert names == "_".join(sorted(m.id_gene[int(x)] for x in (a, b, c)))
            assert prev is None or s <= prev
            prev = s


@pytest.mark.gpu
def test_train_with_save_params_then_predict_cli_queries(torch_cuda, tmp_path):
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
    queries = [models[0].id_gene[i] for i in (17, 3, 60)]
    qfile = tmp_path / "queries.txt"
    qfile.write_text("\n".join(queries) + "\n")
    pred = str(tmp_path / "pred.tsv")
    assert predict_main(["-t", tr, "-e", te, "-p", out + "Sample_0_K2.npz", "--params", out + "Sample_1_K2.npz",
                         "-n", "15", "-q", str(qfile), "-o", pred]) == 0
    lines = open(pred, encoding="utf-8").read().split("\n")
    assert lines[0] == "Query gene\tPredicted Interaction\tID of genes\tGenes" and lines[-1] == ""
    assert len(lines) == 2 + 3 * 15
    assert [ln.split("\t")[0] for ln in lines[1:-1]] == [q for q in queries for _ in range(15)]
    for line in lines[1:-1]:
        q, score, key, names = line.split("\t")
        a, b, c = key.split("_")
        assert str(models[0].gene_id[q]) in (a, b, c)
        want = (models[0].do_prediction(a, b, c) + models[1].do_prediction(a, b, c)) / 2
        assert abs(float(score) - want) <= TOL * want
        assert key not in models[0].links and key not in models[0].test_links
        assert names == "_".join(sorted(models[0].id_gene[int(x)] for x in (a, b, c)))
