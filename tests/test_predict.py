"""Prediction of unseen triplets: exhaustive top-N over all triplets of a gene set (tip_top_triplets,
Model.predict_top_triplets, the predict command line) and the kept parameters (.npz) it reads.

The NumPy restatement `top_triplets_np` below is the oracle: exhaustive, chunked by middle slot, and itself pinned to
`oracle.mmsbm_oracle.predict_loops` (the reference's do_prediction in its operation order).  Order rule of the result:
score descending, then ascending rank triple, where a gene's rank is its position in the decimal-string order of the
candidate ids.  Device rows may differ in order from the oracle's only where the oracle's neighbouring scores are within
1e-12 of each other."""
import itertools
import os
import random
import shutil
import subprocess

import numpy as np
import pytest

from tests.conftest import GOLDEN

BASE = os.path.join(GOLDEN, "base")
TOL = 1e-12


# ----------------------------------------------------------------------------------------------
# oracle
# ----------------------------------------------------------------------------------------------
def pack_ranks(ra, rb, rc):
    return (np.asarray(ra, dtype=np.uint64) << np.uint64(42)) | (np.asarray(rb, dtype=np.uint64) << np.uint64(21)) | \
        np.asarray(rc, dtype=np.uint64)


def top_triplets_np(thetas, prs, cand, known, n):
    """Exhaustive top-n of all triplets of distinct genes of `cand` (ids in decimal-string order) under the mean over the
    parameter sets of do_prediction; `known`: packed rank triples to leave out.  Returns (ids [m][3] in slot order,
    scores [m], packed ranks [m]), best first."""
    cand = np.asarray(cand, dtype=np.int64)
    nc = cand.shape[0]
    known = set(int(x) for x in np.asarray(known, dtype=np.uint64).tolist())
    all_s, all_k = [], []
    for j in range(1, nc - 1):
        a, c = np.arange(j), np.arange(j + 1, nc)
        acc = np.zeros((j, c.shape[0]))
        for th, pr in zip(thetas, prs):
            th = np.asarray(th, dtype=np.float64)
            acc += np.einsum("ax,y,cz,xyz->ac", th[cand[a]], th[cand[j]], th[cand[c]], np.asarray(pr)[..., 1], optimize=True)
        acc /= len(thetas)
        A, C = np.meshgrid(a, c, indexing="ij")
        all_s.append(acc.reshape(-1))
        all_k.append(pack_ranks(A.reshape(-1), np.full(A.size, j), C.reshape(-1)))
    if not all_s:
        return np.empty((0, 3), dtype=np.int64), np.empty(0), np.empty(0, dtype=np.uint64)
    s, k = np.concatenate(all_s), np.concatenate(all_k)
    if known:
        keep = ~np.isin(k, np.array(sorted(known), dtype=np.uint64))
        s, k = s[keep], k[keep]
    order = np.lexsort((k, -s))[:n]
    s, k = s[order], k[order]
    m = np.uint64((1 << 21) - 1)
    ranks = np.stack([(k >> np.uint64(42)) & m, (k >> np.uint64(21)) & m, k & m], axis=1).astype(np.int64)
    return cand[ranks], s, k


def check_against_oracle(ids, scores, o_ids, o_scores, n):
    """Same rows as the oracle's first n, scores within TOL; order free only inside runs of near-equal oracle scores
    (o_* may hold more than n rows so that a run crossing the cut is seen whole)."""
    m = min(n, len(o_scores))
    assert len(scores) == m
    if m == 0:
        return
    assert np.max(np.abs(scores - o_scores[:m]) / np.maximum(np.abs(o_scores[:m]), 1e-300)) < TOL
    got = [tuple(r) for r in np.asarray(ids).tolist()]
    exp = [tuple(r) for r in np.asarray(o_ids).tolist()]
    i = 0
    while i < m:
        hi = i + 1
        while hi < len(o_scores) and abs(o_scores[hi] - o_scores[hi - 1]) <= TOL * abs(o_scores[hi - 1]):
            hi += 1
        if hi - i == 1:
            assert got[i] == exp[i], "row %d" % i
        else:
            assert set(got[i:min(hi, m)]) <= set(exp[i:hi]), "rows %d..%d" % (i, hi)
        i = hi


def random_params(rng, P, K, S):
    thetas = [rng.dirichlet(np.ones(K), size=P) for _ in range(S)]
    prs = []
    for _ in range(S):
        pr = rng.random((K, K, K, 2))
        prs.append(pr / pr.sum(axis=3, keepdims=True))
    return thetas, prs


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
def test_rank_order_is_key_slot_order_brute_force():
    """Sorting the candidate ids by their decimal strings makes every i < j < k of positions the key's slot order."""
    cand = sorted(range(131), key=str)
    for i, j, k in itertools.combinations(range(len(cand)), 3):
        key = sorted([str(cand[i]), str(cand[j]), str(cand[k])])      # TIP.py:353
        assert key == [str(cand[i]), str(cand[j]), str(cand[k])]


@pytest.mark.parametrize("S", [1, 2])
@pytest.mark.parametrize("K", [1, 3])
def test_oracle_is_pinned_to_predict_loops(K, S):
    from oracle import mmsbm_oracle as orc
    rng = np.random.default_rng(10 * K + S)
    P = 25
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(rng.choice(P, size=22, replace=False).tolist(), key=str))
    known = pack_ranks([0, 1, 2], [5, 6, 3], [7, 9, 4])
    ids, sc, _ = top_triplets_np(thetas, prs, cand, known, 10 ** 6)
    assert len(sc) == 22 * 21 * 20 // 6 - 3
    tl = [t.tolist() for t in thetas]
    pl = [p.tolist() for p in prs]
    for (a, b, c), s in zip(ids[::7].tolist(), sc[::7].tolist()):
        assert sorted([str(a), str(b), str(c)]) == [str(a), str(b), str(c)]
        want = sum(orc.predict_loops(t, p, a, b, c) for t, p in zip(tl, pl)) / S
        assert abs(s - want) <= TOL * want
    assert np.all(sc[:-1] >= sc[1:])
    ranks = {g: r for r, g in enumerate(cand.tolist())}
    left = {(ranks[a], ranks[b], ranks[c]) for a, b, c in ids.tolist()}
    assert not left & {(0, 5, 7), (1, 6, 9), (2, 3, 4)}


def _digested(train="train1.dat", test="test1.dat"):
    from trigenicinteractionpredictor_b200 import Model
    m = Model()
    m.get_traintest(os.path.join(BASE, train), os.path.join(BASE, test))
    return m


def test_known_keys_are_packed_ranks_of_candidates():
    m = _digested()
    rng = np.random.default_rng(0)
    sub = rng.choice(m.P, size=60, replace=False).tolist()
    cand = np.array(sorted(sub, key=str), dtype=np.int32)
    got = m._known_packed(cand)
    rank = {g: r for r, g in enumerate(cand.tolist())}
    want = set()
    for key in list(m.links.keys()) + list(m.test_links.keys()):
        g = [int(x) for x in key.split("_")]
        if all(x in rank for x in g) and len(set(g)) == 3:
            r = [rank[x] for x in g]
            assert r == sorted(r)                     # slot order is rank order
            want.add((r[0] << 42) | (r[1] << 21) | r[2])
    assert got.dtype == np.uint64 and np.all(got[:-1] < got[1:])
    assert set(got.tolist()) == want and len(want) > 0


def test_parameters_round_trip_through_npz(tmp_path):
    random.seed(7)
    m = _digested()
    m.initialize_parameters(3)
    path = str(tmp_path / "params.bin")
    m.save_parameters(path)
    assert os.path.exists(path)                      # exactly the path given, no suffix added
    with np.load(path) as z:
        assert sorted(z.files) == ["K", "genes", "pr", "theta"] and int(z["K"]) == 3
        assert [str(g) for g in z["genes"]] == [m.id_gene[i] for i in range(m.P)]
    m2 = _digested()
    m2.load_parameters(path)
    assert m2.K == 3
    assert np.array_equal(np.array(m2.theta), np.array(m.theta)) and np.array_equal(np.array(m2.pr), np.array(m.pr))


def _save(path, theta, pr, K, genes):
    with open(path, "wb") as fh:
        np.savez(fh, theta=theta, pr=pr, K=np.int64(K), genes=np.array(genes, dtype=str))


def test_load_parameters_refusals(tmp_path):
    random.seed(3)
    m = _digested()
    m.initialize_parameters(2)
    th, pr = np.array(m.theta), np.array(m.pr)
    genes = [m.id_gene[i] for i in range(m.P)]
    cases = {
        "genes": (th, pr, 2, genes[::-1], "gene list"),
        "fewer_genes": (th[:-1], pr, 2, genes[:-1], "gene list"),
        "K": (np.full((m.P, 3), 1 / 3), np.full((3, 3, 3, 2), 0.5), 3, genes, "K = 3"),
        "nan": (np.where(np.arange(th.size).reshape(th.shape) == 5, np.nan, th), pr, 2, genes, "non-finite"),
        "inf": (th, np.where(np.arange(pr.size).reshape(pr.shape) == 1, np.inf, pr), 2, genes, "non-finite"),
        "negative": (th, -pr, 2, genes, "negative"),
        "shape": (th[:, :1], pr, 2, genes, "shapes"),
    }
    for name, (t, p, K, g, msg) in cases.items():
        path = str(tmp_path / (name + ".npz"))
        _save(path, t, p, K, g)
        fresh = _digested()
        fresh.initialize_parameters(2)
        with pytest.raises(ValueError, match=msg):
            fresh.load_parameters(path)
    bad = str(tmp_path / "not.npz")
    open(bad, "w").write("not an archive")
    with pytest.raises(ValueError):
        _digested().load_parameters(bad)


def test_predict_cli_argument_and_file_errors(tmp_path, capsys):
    from trigenicinteractionpredictor_b200.predict import main
    random.seed(5)
    m = _digested()
    m.initialize_parameters(2)
    good = str(tmp_path / "good.npz")
    m.save_parameters(good)
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["--bogus"]) == 2
    assert main(["-t", tr, "-e", te]) == 2                                        # no parameter file
    assert main(["-t", tr, "-e", te, "-p", str(tmp_path / "missing.npz")]) == 2
    assert main(["-t", str(tmp_path / "missing.dat"), "-e", te, "-p", good]) == 2
    assert main(["-t", tr, "-e", te, "-p", good, "-n", "zero"]) == 2
    with np.load(good) as z:
        genes = [str(g) for g in z["genes"]]
        genes[0], genes[1] = genes[1], genes[0]
        _save(str(tmp_path / "other.npz"), z["theta"], z["pr"], 2, genes)
    assert main(["-t", tr, "-e", te, "-p", good, "-p", str(tmp_path / "other.npz")]) == 2
    assert "gene list" in capsys.readouterr().err
    gfile = tmp_path / "genes.txt"
    gfile.write_text("G00001\nNOPE1\nG00002\nNOPE2\n")
    assert main(["-t", tr, "-e", te, "-p", good, "-g", str(gfile)]) == 2
    assert "NOPE1, NOPE2" in capsys.readouterr().err


def test_sass_scoring_kernel_runs_on_dmma():
    from trigenicinteractionpredictor_b200 import _cabi, build
    build.build()
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    funcs = out.split("Function : ")
    body = [f for f in funcs if f.split("\n", 1)[0].find("tip_predict_pass_kernel") >= 0]
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
def test_top_n_matches_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(P * 100 + K * 10 + S)
    thetas, prs = random_params(rng, P, K, S)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    total = P * (P - 1) * (P - 2) // 6
    kr = np.sort(rng.choice(P, size=(40, 3), replace=True), axis=1)
    kr = kr[(kr[:, 0] < kr[:, 1]) & (kr[:, 1] < kr[:, 2])]
    known = np.unique(pack_ranks(kr[:, 0], kr[:, 1], kr[:, 2]))
    o_ids, o_sc, _ = top_triplets_np(thetas, prs, cand, known, total)
    eng = _engine(P, K)
    for n in (1, 10, 500, total):
        ids, sc = eng.top_triplets(np.stack(thetas), np.stack(prs), cand, known, n)
        check_against_oracle(ids, sc, o_ids, o_sc, n)
    assert len(sc) == total - len(known)


@pytest.mark.gpu
@pytest.mark.parametrize("P,n", [(60, 700), (160, 100)], ids=["fits_buffer", "selects_on_ranks"])
def test_all_scores_tied_gives_rank_order(torch_cuda, P, n):
    """Identical theta rows: every score is the same number.  At P = 160 the 669 920 triplets exceed the selection
    buffer, so the threshold has to continue on the packed rank triple."""
    K = 3
    rng = np.random.default_rng(1)
    theta = np.tile(rng.dirichlet(np.ones(K)), (P, 1))
    pr = rng.random((K, K, K, 2))
    pr /= pr.sum(axis=3, keepdims=True)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    ids, sc = _engine(P, K).top_triplets(theta[None], pr[None], cand, np.empty(0, dtype=np.uint64), n)
    assert len(sc) == n and np.all(sc == sc[0])
    want = [tuple(cand[list(t)].tolist()) for t in itertools.islice(itertools.combinations(range(P), 3), n)]
    assert [tuple(r) for r in ids.tolist()] == want


def _trained_base_model(K, iters=5, seed=1000):
    from trigenicinteractionpredictor_b200 import Model
    m = Model()
    m.get_traintest(os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat"))
    random.seed(seed)
    m.initialize_parameters(K)
    for _ in range(iters):
        m.make_iteration()
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 10])
def test_golden_base_top50_are_do_prediction_of_their_keys(torch_cuda, K):
    m = _trained_base_model(K)
    rows = m.predict_top_triplets(50)
    assert len(rows) == 50
    known = set(m.links.keys()) | set(m.test_links.keys())
    for s, key, names in rows:
        a, b, c = key.split("_")
        assert sorted([a, b, c]) == [a, b, c]                           # key slot order
        assert key not in known
        assert abs(s - m.do_prediction(a, b, c)) <= TOL * s
        assert names == "_".join(sorted(m.id_gene[int(x)] for x in (a, b, c)))
    th, pr = np.array(m.theta), np.array(m.pr)
    cand = np.array(sorted(range(m.P), key=str))
    o_ids, o_sc, _ = top_triplets_np([th], [pr], cand, m._known_packed(cand.astype(np.int32)), 80)
    check_against_oracle(np.array([[int(x) for x in r[1].split("_")] for r in rows]), np.array([r[0] for r in rows]),
                         o_ids, o_sc, 50)
    # exclusion off: the known keys come back where the oracle puts them
    rows_all = m.predict_top_triplets(300, exclude_known=False)
    o_ids, o_sc, _ = top_triplets_np([th], [pr], cand, [], 330)
    check_against_oracle(np.array([[int(x) for x in r[1].split("_")] for r in rows_all]),
                         np.array([r[0] for r in rows_all]), o_ids, o_sc, 300)
    assert any(r[1] in known for r in rows_all)


@pytest.mark.gpu
def test_gene_subset_and_ensemble_of_parameter_sets(torch_cuda, tmp_path):
    m = _trained_base_model(3)
    rng = np.random.default_rng(4)
    names = [m.id_gene[i] for i in rng.choice(m.P, size=45, replace=False).tolist()]
    th1, pr1 = np.array(m.theta), np.array(m.pr)
    thetas, prs = random_params(rng, m.P, 3, 1)
    sets = [(th1, pr1), (thetas[0], prs[0])]
    p1 = str(tmp_path / "a.npz")
    m.save_parameters(p1)
    rows = m.predict_top_triplets(200, genes=names, params=[p1, sets[1]])
    ids = sorted(m.gene_id[g] for g in names)
    cand = np.array(sorted(ids, key=str))
    o_ids, o_sc, _ = top_triplets_np([s[0] for s in sets], [s[1] for s in sets], cand,
                                     m._known_packed(cand.astype(np.int32)), 230)
    got = np.array([[int(x) for x in r[1].split("_")] for r in rows])
    check_against_oracle(got, np.array([r[0] for r in rows]), o_ids, o_sc, 200)
    assert set(got.reshape(-1).tolist()) <= set(ids)


@pytest.mark.gpu
def test_p1500_against_chunked_tip_score_and_topk(torch_cuda):
    """5.6e8 triplets: the same set and order as a brute force of tip_score over every triplet on the device."""
    import ctypes
    torch = torch_cuda
    P, K, N = 1500, 4, 300
    rng = np.random.default_rng(15)
    thetas, prs = random_params(rng, P, K, 1)
    cand_np = np.array(sorted(range(P), key=str), dtype=np.int32)
    eng = _engine(P, K)
    ids, sc = eng.top_triplets(np.stack(thetas), np.stack(prs), cand_np, np.empty(0, dtype=np.uint64), N)
    eng.set_params(thetas[0], prs[0])
    dev = eng.device
    cand = torch.from_numpy(cand_np).to(dev)
    best_s = torch.empty(0, dtype=torch.float64, device=dev)
    best_k = torch.empty(0, dtype=torch.int64, device=dev)
    j = 1
    while j < P - 1:
        js, size = [], 0
        while j < P - 1 and size < 8_000_000:
            js.append(j)
            size += j * (P - 1 - j)
            j += 1
        parts = []
        for jj in js:
            a = torch.arange(jj, device=dev)
            c = torch.arange(jj + 1, P, device=dev)
            A, C = torch.meshgrid(a, c, indexing="ij")
            parts.append(torch.stack([A.reshape(-1), torch.full((A.numel(),), jj, device=dev), C.reshape(-1)], 1))
        r = torch.cat(parts)
        g = cand[r].to(torch.int32).contiguous()
        g1, g2, g3 = g[:, 0].contiguous(), g[:, 1].contiguous(), g[:, 2].contiguous()
        out = torch.empty(r.shape[0], dtype=torch.float64, device=dev)
        assert eng.lib.tip_score(P, K, ctypes.c_void_p(g1.data_ptr()), ctypes.c_void_p(g2.data_ptr()),
                                 ctypes.c_void_p(g3.data_ptr()), r.shape[0], ctypes.c_void_p(eng.theta.data_ptr()),
                                 ctypes.c_void_p(eng.p.data_ptr()), ctypes.c_void_p(out.data_ptr()), eng._stream()) == 0
        keys = (r[:, 0] << 42) | (r[:, 1] << 21) | r[:, 2]
        v, i = torch.topk(out, min(N + 64, out.numel()))
        best_s = torch.cat([best_s, v])
        best_k = torch.cat([best_k, keys[i]])
        v, i = torch.topk(best_s, min(N + 64, best_s.numel()))
        best_s, best_k = v, best_k[i]
    order = np.lexsort((best_k.cpu().numpy(), -best_s.cpu().numpy()))
    o_sc = best_s.cpu().numpy()[order]
    k = best_k.cpu().numpy()[order]
    m = (1 << 21) - 1
    o_ids = cand_np[np.stack([(k >> 42) & m, (k >> 21) & m, k & m], 1)]
    check_against_oracle(ids, sc, o_ids, o_sc, N)


@pytest.mark.gpu
def test_train_with_save_params_then_predict_cli(torch_cuda, tmp_path, capsys):
    """Training CLI with --save-params on the golden base files (two samples that converge), then the predict CLI on
    both .npz files: every printed score is the mean of the two models' do_prediction."""
    from trigenicinteractionpredictor_b200 import Model, main
    from trigenicinteractionpredictor_b200.predict import main as predict_main
    out = str(tmp_path) + os.sep
    tr, te = os.path.join(BASE, "train1.dat"), os.path.join(BASE, "test1.dat")
    assert main(["-t", tr, "-e", te, "-k", "2", "-i", "300", "-f", "5", "-b", "10", "-n", "2", "-o", out,
                 "--seed", "1000", "--save-params"]) == 0
    assert sorted(os.listdir(out)) == ["Sample_0_K2.csv", "Sample_0_K2.npz", "Sample_1_K2.csv", "Sample_1_K2.npz"]
    pred = str(tmp_path / "pred.tsv")
    assert predict_main(["-t", tr, "-e", te, "-p", out + "Sample_0_K2.npz", "--params", out + "Sample_1_K2.npz",
                         "-n", "40", "-o", pred]) == 0
    lines = open(pred, encoding="utf-8").read().split("\n")
    assert lines[0] == "Predicted Interaction\tID of genes\tGenes" and lines[-1] == "" and len(lines) == 42
    models = []
    for s in (0, 1):
        mm = Model()
        mm.get_traintest(tr, te)
        mm.load_parameters(out + "Sample_%d_K2.npz" % s)
        models.append(mm)
    prev = None
    for line in lines[1:-1]:
        score, key, names = line.split("\t")
        a, b, c = key.split("_")
        want = (models[0].do_prediction(a, b, c) + models[1].do_prediction(a, b, c)) / 2
        assert abs(float(score) - want) <= TOL * want
        assert key not in models[0].links and key not in models[0].test_links
        assert names == "_".join(sorted(models[0].id_gene[int(x)] for x in (a, b, c)))
        assert prev is None or float(score) <= prev
        prev = float(score)
