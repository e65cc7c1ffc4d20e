"""The digenic model past its training path (DESIGN §4.11): pair scores of the test set (tip_score_pairs), the N best
unseen gene pairs over all pairs (tip_top_pairs) and per query gene (tip_top_pairs_per_gene), the engine and
TrigenicInteractionPredictor_23.Model methods on top of them, the held-out likelihood, test-set tables and metrics, kept
parameters, and the two command lines.

Everything here is an addition defined by formulas, so the reference is the NumPy oracle below (pinned to an itertools
brute force), not the author's test-set code."""
import contextlib
import ctypes
import io
import itertools
import os
import random
import shutil
import subprocess
import sys

import numpy as np
import pytest

from tests.test_predict import TOL, check_against_oracle

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
DIGENIC = os.path.join(HERE, "golden", "digenic")
CHUNK = 1 << 21                     # TIP_PAIR_CHUNK of include/tip.h


# ----------------------------------------------------------------------------------------------
# NumPy oracle of DESIGN §4.11
# ----------------------------------------------------------------------------------------------
def pair_sums(thetas, qrs, cand):
    """M[ra][rb] = sum over the sets of the score of (cand[ra], cand[rb]) with cand[ra] in the first slot."""
    cand = np.asarray(cand, dtype=np.int64)
    M = 0.0
    for th, q in zip(thetas, qrs):
        t = np.asarray(th, dtype=np.float64)[cand]
        M = M + t @ np.asarray(q, dtype=np.float64)[:, :, 1] @ t.T
    return np.asarray(M, dtype=np.float64).reshape(len(cand), len(cand))


def top_pairs_np(thetas, qrs, cand, known, N):
    """(ids [m][2], mean scores [m], packed [m]) of the first N unseen pairs: sum descending, packed ranks ascending."""
    n = len(cand)
    if n < 2:
        return np.empty((0, 2), dtype=np.int64), np.empty(0), np.empty(0, dtype=np.uint64)
    M = pair_sums(thetas, qrs, cand)
    ra, rb = np.triu_indices(n, 1)
    pk = (ra.astype(np.uint64) << np.uint64(21)) | rb.astype(np.uint64)
    keep = ~np.isin(pk, np.asarray(known, dtype=np.uint64))
    ra, rb, pk, s = ra[keep], rb[keep], pk[keep], M[ra[keep], rb[keep]]
    order = np.lexsort((pk, -s))[:N]
    cand = np.asarray(cand)
    return np.stack([cand[ra[order]], cand[rb[order]]], axis=1), s[order] / len(thetas), pk[order]


def per_gene_np(thetas, qrs, cand, known, r, N, M=None):
    """(ids [m][2], mean scores [m]) of the first N unseen pairs of rank r with another candidate x: sum descending,
    then x ascending."""
    n = len(cand)
    M = pair_sums(thetas, qrs, cand) if M is None else M
    x = np.array([i for i in range(n) if i != r], dtype=np.int64)
    lo, hi = np.minimum(x, r), np.maximum(x, r)
    pk = (lo.astype(np.uint64) << np.uint64(21)) | hi.astype(np.uint64)
    keep = ~np.isin(pk, np.asarray(known, dtype=np.uint64))
    lo, hi, x, s = lo[keep], hi[keep], x[keep], M[lo[keep], hi[keep]]
    order = np.lexsort((x, -s))[:N]
    cand = np.asarray(cand)
    return np.stack([cand[lo[order]], cand[hi[order]]], axis=1), s[order] / len(thetas)


def random_sets(rng, P, K, S):
    thetas = [rng.dirichlet(np.ones(K), size=P) for _ in range(S)]
    qrs = []
    for _ in range(S):
        q = rng.random((K, K, 2))
        qrs.append(q / q.sum(axis=2, keepdims=True))
    return np.stack(thetas), np.stack(qrs)


def pack2(ra, rb):
    return (np.asarray(ra, dtype=np.uint64) << np.uint64(21)) | np.asarray(rb, dtype=np.uint64)


def _digested_model(device=None):
    from trigenicinteractionpredictor_b200.TrigenicInteractionPredictor_23 import Model
    m = Model(device=device)
    with contextlib.redirect_stdout(io.StringIO()):
        m.get_train_test(os.path.join(DIGENIC, "train_mixed.dat"), os.path.join(DIGENIC, "test_mixed.dat"))
    return m


# ----------------------------------------------------------------------------------------------
# CPU tests
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2])
def test_oracle_equals_itertools_brute_force(S):
    rng = np.random.default_rng(40 + S)
    P, K = 17, 3
    thetas, qrs = random_sets(rng, P, K, S)
    thetas[:, 5] = thetas[:, 9]                      # exact ties between pairs that differ in one gene
    thetas[:, 11] = thetas[:, 9]
    cand = np.array(sorted(range(P), key=str))
    known = np.sort(pack2([0, 2, 3], [1, 9, 16]))
    kset = set(int(k) for k in known.tolist())

    def score(a, b):
        return sum(sum(th[a][i] * th[b][j] * q[i][j][1] for i in range(K) for j in range(K)) for th, q in zip(thetas, qrs))

    rows = []
    for ra, rb in itertools.combinations(range(P), 2):
        pk = (ra << 21) | rb
        if pk not in kset:
            rows.append((-score(cand[ra], cand[rb]), pk, (int(cand[ra]), int(cand[rb]))))
    rows.sort()
    ids, sc, _ = top_pairs_np(thetas, qrs, cand, known, len(rows) + 5)
    assert len(sc) == len(rows) == P * (P - 1) // 2 - 3
    check_against_oracle(ids, sc, np.array([r[2] for r in rows]), -np.array([r[0] for r in rows]) / S, len(rows))
    for r in (0, 1, 9, P - 1):
        prow = []
        for x in range(P):
            if x == r:
                continue
            lo, hi = min(x, r), max(x, r)
            if ((lo << 21) | hi) in kset:
                continue
            prow.append((-score(cand[lo], cand[hi]), x, (int(cand[lo]), int(cand[hi]))))
        prow.sort()
        gi, gs = per_gene_np(thetas, qrs, cand, known, r, P)
        check_against_oracle(gi, gs, np.array([p[2] for p in prow]), -np.array([p[0] for p in prow]) / S, len(prow))


def test_workspace_bytes_and_abi_refusals():
    from trigenicinteractionpredictor_b200 import _cabi
    lib = _cabi.load()
    nb = ctypes.c_size_t(0)
    assert lib.tip_top_pairs_workspace_bytes(6000, 10, 10, 1000, ctypes.byref(nb)) == 0
    # O(n S K + N + chunk), independent of n^2
    assert nb.value < 2 * 6000 * 100 * 8 + 4 * 8 * (1000 + CHUNK) + (64 << 20)
    for args in [(100, 10, 39, 10), ((1 << 21) + 1, 2, 1, 10), (100, 33, 1, 10), (100, 2, 1, 1 << 28), (100, 2, 1, -1)]:
        assert lib.tip_top_pairs_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"S*K <= 384" in lib.tip_last_error() and b"N < 2^28" in lib.tip_last_error()
    assert lib.tip_top_pairs_per_gene_workspace_bytes(6000, 6000, 10, 10, 20, ctypes.byref(nb)) == 0
    assert nb.value < 4 * 6000 * 100 * 8 + 24 * CHUNK + (64 << 20)
    for args in [(100, 101, 2, 1, 1), (100, 10, 10, 39, 1), ((1 << 21), 1 << 20, 2, 1, 17), (100, -1, 2, 1, 1)]:
        assert lib.tip_top_pairs_per_gene_workspace_bytes(*args, ctypes.byref(nb)) == -1
        assert b"n_query*N <= 2^24" in lib.tip_last_error()
    assert lib.tip_top_pairs_per_gene_workspace_bytes(1 << 21, 1 << 20, 2, 1, 16, ctypes.byref(nb)) == 0
    # refused before any device work
    n_out = ctypes.c_int64(7)
    assert lib.tip_top_pairs(10, 2, 200, None, None, None, 5, None, 0, 3, None, 0, None, None, ctypes.byref(n_out), None) == -1
    assert b"tip_top_pairs: bad arguments" in lib.tip_last_error()
    assert lib.tip_score_pairs(10, 40, None, None, None, None, 3, None, None) == -1
    assert b"tip_score_pairs: bad arguments" in lib.tip_last_error()
    assert lib.tip_score_pairs(10, 2, None, None, None, None, 3, None, None) == -1
    assert b"null pointer" in lib.tip_last_error()


def test_model_refusals():
    from trigenicinteractionpredictor_b200.TrigenicInteractionPredictor_23 import Model
    with pytest.raises(ValueError, match="digested"):
        Model().predict_top_pairs(5)
    m = _digested_model()
    with pytest.raises(ValueError, match="initialize_parameters"):
        m.predict_top_pairs(5)
    random.seed(1)
    m.initialize_parameters(3)
    with pytest.raises(ValueError, match="unknown gene names: nope"):
        m.predict_top_pairs(5, genes=["nope"])
    with pytest.raises(ValueError, match="n must be >= 0"):
        m.predict_top_pairs(-1)
    with pytest.raises(ValueError, match="queries is empty"):
        m.predict_top_pairs_per_gene([], 5)
    g = m.id_gene[0]
    with pytest.raises(ValueError, match="duplicate query genes: " + g):
        m.predict_top_pairs_per_gene([g, g], 5)
    with pytest.raises(ValueError, match="unknown gene names: nope"):
        m.predict_top_pairs_per_gene([g, "nope"], 5)
    with pytest.raises(ValueError, match="n must be >= 0"):
        m.predict_top_pairs_per_gene([g], -2)
    th = np.full((m.P, 3), 1 / 3)
    with pytest.raises(ValueError, match="params is empty"):
        m.predict_top_pairs(5, params=[])
    with pytest.raises(ValueError, match="K = 2, the model has K = 3"):
        m.predict_top_pairs(5, params=[(np.full((m.P, 2), 0.5), np.full((2, 2, 2), 0.5))])
    with pytest.raises(ValueError, match="negative"):
        m.predict_top_pairs(5, params=[(th, -np.ones((3, 3, 2)))])
    with pytest.raises(ValueError, match="shapes"):
        m.predict_top_pairs(5, params=[(th, np.ones((3, 2, 2)))])


def test_parameter_file_round_trip_and_refusals(tmp_path):
    from trigenicinteractionpredictor_b200 import TrigenicInteractionPredictor as tip
    m = _digested_model()
    random.seed(7)
    m.initialize_parameters(3)
    path = str(tmp_path / "S0.npz")
    m.save_parameters(path)
    th, pr, qr = m.check_parameters_file(path)
    assert np.array_equal(th, np.array(m.theta)) and np.array_equal(pr, np.array(m.pr)) and np.array_equal(qr, np.array(m.qr))
    m2 = _digested_model()
    m2.load_parameters(path)
    assert m2.K == 3 and np.array_equal(np.array(m2.qr), qr) and np.array_equal(np.array(m2.theta), th)
    with np.load(path) as z:
        base = {k: z[k] for k in z.files}

    def write(name, **over):
        d = dict(base)
        d.update(over)
        d = {k: v for k, v in d.items() if v is not None}
        p = str(tmp_path / name)
        with open(p, "wb") as fh:
            np.savez(fh, **d)
        return p

    cases = [(write("genes.npz", genes=base["genes"][::-1]), "gene list"),
             (write("k.npz", K=np.int64(4)), "K = 4"),
             (write("shape.npz", qr=base["qr"][:2]), "shapes"),
             (write("nan.npz", qr=np.where(np.arange(18).reshape(3, 3, 2) == 4, np.nan, base["qr"])), "non-finite"),
             (write("neg.npz", theta=-base["theta"]), "negative"),
             (write("tri.npz", qr=None), "trigenic parameter file")]
    for p, why in cases:
        with pytest.raises(ValueError, match=why):
            m.check_parameters_file(p)
    with pytest.raises(ValueError, match="not a parameter file"):
        m.check_parameters_file(str(tmp_path / "missing.npz"))
    # a trigenic model refuses nothing it needs from a digenic file, and a digenic model refuses a trigenic file
    t = tip.Model()
    tri = str(tmp_path / "tri_model.npz")
    t.P, t.K, t.id_gene = m.P, 3, dict(m.id_gene)
    t._theta_host, t._pr_host, t._params_on, t._host_valid = np.array(m.theta), np.array(m.pr), "host", True
    t.save_parameters(tri)
    with pytest.raises(ValueError, match="no qr"):
        m.check_parameters_file(tri)


def test_dmma_in_the_pair_kernels():
    from trigenicinteractionpredictor_b200 import _cabi  # noqa: F401  (the build below is the package's)
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    obj = os.path.join(ROOT, "trigenicinteractionpredictor_b200", "csrc", "_obj", "tip_predict.o")
    if not os.path.exists(cuobjdump) or not os.path.exists(obj):
        pytest.skip("cuobjdump or the build's objects not available")
    out = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True).stdout
    for kernel in ("tip_top_pairs_pass_kernel", "tip_top_pairs_gene_kernel"):
        start = out.index("Function : ", out.index(kernel) - 200)
        body = out[start:out.find("Function : ", start + 20)]
        assert kernel in body[:400] and "DMMA.8x8x4" in body, kernel


def _run(mod, *args, cwd=None):
    return subprocess.run([sys.executable, "-m", "trigenicinteractionpredictor_b200." + mod, *args], capture_output=True,
                          text=True, cwd=cwd or ROOT, env=dict(os.environ, PYTHONPATH=ROOT))


def test_cli_argument_errors(tmp_path):
    tr, te = os.path.join(DIGENIC, "train_mixed.dat"), os.path.join(DIGENIC, "test_mixed.dat")
    r = _run("predict_pairs", "-t", tr, "-e", te)
    assert r.returncode == 2 and "at least one -p/--params" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", str(tmp_path / "none.npz"))
    assert r.returncode == 2 and "does not exist" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", tr, "-n", "0")
    assert r.returncode == 2 and "--top must be positive" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", tr, "-n", "x")
    assert r.returncode == 2 and "--top must be an integer" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", tr, "--bogus")
    assert r.returncode == 2 and "argument error" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", tr, "-o", str(tmp_path / "no" / "out.tsv"))
    assert r.returncode == 2 and "directory" in r.stderr
    bad = tmp_path / "bad.npz"
    with open(bad, "wb") as fh:
        np.savez(fh, theta=np.ones((2, 2)))
    q = tmp_path / "q.txt"
    q.write_text("G00019\nG00019\n")
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", str(bad), "-q", str(q))
    assert r.returncode == 2 and "query genes listed twice: G00019" in r.stderr
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", str(bad))
    assert r.returncode == 2 and "has no qr" in r.stderr and "READ DATA" not in r.stdout
    r = _run("TrigenicInteractionPredictor_23", "-t", tr)
    assert r.returncode == 2 and "Argument error" in r.stdout
    r = _run("TrigenicInteractionPredictor_23", "-t", tr, "-e", te, "-k", "0")
    assert r.returncode == 2
    r = _run("TrigenicInteractionPredictor_23", "-t", tr, "-e", te, "--dist", "links")
    assert r.returncode == 2 and "Argument error" in r.stdout


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
def test_both_modes_against_the_oracle(torch_cuda, P, K, S):
    rng = np.random.default_rng(1000 * P + 10 * K + S)
    thetas, qrs = random_sets(rng, P, K, S)
    eng = _engine(P, K)
    for subset in (False, True):
        ids = sorted(rng.choice(P, size=P * 2 // 3, replace=False).tolist()) if subset else list(range(P))
        cand = np.array(sorted(ids, key=str), dtype=np.int32)
        n = len(cand)
        M = pair_sums(thetas, qrs, cand)
        for with_known in (False, True):
            known = np.empty(0, dtype=np.uint64)
            if with_known:
                ra = rng.integers(0, n - 1, size=n)
                rb = ra + 1 + rng.integers(0, n - 1 - ra)
                known = np.unique(pack2(ra, rb))
            o_ids, o_sc, _ = top_pairs_np(thetas, qrs, cand, known, n * n)      # whole runs of tied scores
            for N in (1, 7, 50, n * (n - 1) // 2 + 3):
                g_ids, g_sc = eng.top_pairs(thetas, qrs, cand, known, N)
                check_against_oracle(g_ids, g_sc, o_ids, o_sc, N)
            queries = np.array([0, n - 1] + rng.choice(np.arange(1, n - 1), size=5, replace=False).tolist(), dtype=np.int32)
            for N in (1, 9, n + 2):
                g_ids, g_sc, cnt = eng.top_pairs_per_gene(thetas, qrs, cand, queries, known, N)
                for qi, r in enumerate(queries.tolist()):
                    o_ids, o_sc = per_gene_np(thetas, qrs, cand, known, r, n, M)
                    assert cnt[qi] == min(N, len(o_sc))
                    check_against_oracle(g_ids[qi, :cnt[qi]], g_sc[qi, :cnt[qi]], o_ids, o_sc, N)


@pytest.mark.gpu
def test_ties_and_degenerate_universes(torch_cuda):
    P, K = 50, 3
    rng = np.random.default_rng(5)
    eng = _engine(P, K)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    q = rng.random((1, K, K, 2))
    th = np.tile(rng.dirichlet(np.ones(K)), (1, P, 1))          # all-equal theta rows: equal scores, packed order
    ids, sc = eng.top_pairs(th, q, cand, np.empty(0, np.uint64), 30)
    exp = [(int(cand[a]), int(cand[b])) for a, b in itertools.islice(itertools.combinations(range(P), 2), 30)]
    assert [tuple(r) for r in ids.tolist()] == exp and len(set(sc.tolist())) == 1
    gi, gs, cnt = eng.top_pairs_per_gene(th, q, cand, np.array([7, 0, 49], np.int32), np.empty(0, np.uint64), 60)
    assert cnt.tolist() == [49, 49, 49]
    for qi, r in enumerate((7, 0, 49)):
        exp = [(int(cand[min(x, r)]), int(cand[max(x, r)])) for x in range(P) if x != r]
        assert [tuple(v) for v in gi[qi, :49].tolist()] == exp
    z = q.copy()
    z[..., 1] = 0.0                                                # exact-zero scores
    th2 = random_sets(rng, P, K, 1)[0]
    ids, sc = eng.top_pairs(th2, z, cand, np.empty(0, np.uint64), 10)
    assert np.all(sc == 0) and [tuple(r) for r in ids.tolist()] == \
        [(int(cand[a]), int(cand[b])) for a, b in itertools.islice(itertools.combinations(range(P), 2), 10)]
    # repeated known keys count once
    known = np.sort(np.concatenate([pack2([0, 0, 3], [1, 1, 9])] * 2))
    ids, sc = eng.top_pairs(th2, q, cand, known, 10 ** 6)
    assert len(sc) == P * (P - 1) // 2 - 2
    o_ids, o_sc, _ = top_pairs_np(th2, q, cand, known, 10 ** 6)
    check_against_oracle(ids, sc, o_ids, o_sc, 10 ** 6)
    gi, gs, cnt = eng.top_pairs_per_gene(th2, q, cand, np.array([0], np.int32), known, 100)
    assert cnt.tolist() == [P - 2]
    # universes of 0, 1 and 2 candidates
    for nc in (0, 1, 2):
        c = cand[:nc]
        ids, sc = eng.top_pairs(th2, q, c, np.empty(0, np.uint64), 5)
        assert len(sc) == (1 if nc == 2 else 0)
        if nc:
            gi, gs, cnt = eng.top_pairs_per_gene(th2, q, c, np.arange(nc, dtype=np.int32), np.empty(0, np.uint64), 5)
            assert cnt.tolist() == [nc - 1] * nc
    ids, sc = eng.top_pairs(th2, q, cand[:2], pack2([0], [1]), 5)
    assert len(sc) == 0
    # refusals before any device work
    from trigenicinteractionpredictor_b200 import _cabi
    with pytest.raises(_cabi.TipLibraryError, match="appears twice"):
        eng.top_pairs_per_gene(th2, q, cand, np.array([3, 3], np.int32), np.empty(0, np.uint64), 5)
    with pytest.raises(_cabi.TipLibraryError, match="is not in"):
        eng.top_pairs_per_gene(th2, q, cand, np.array([P], np.int32), np.empty(0, np.uint64), 5)


@pytest.mark.gpu
def test_chunk_merging(torch_cuda):
    """C(n, 2) over several chunks (global) and more queries than one chunk holds (per gene), at K = 2."""
    from trigenicinteractionpredictor_b200 import _cabi
    P, K = 2600, 2
    rng = np.random.default_rng(11)
    thetas, qrs = random_sets(rng, P, K, 1)
    eng = _engine(P, K)
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    M = pair_sums(thetas, qrs, cand)
    ra = rng.integers(0, P - 1, size=3000)
    known = np.unique(pack2(ra, ra + 1 + rng.integers(0, P - 1 - ra)))
    for N in (1000, 40000):
        ids, sc = eng.top_pairs(thetas, qrs, cand, known, N)
        assert eng.lib.tip_top_pairs_last_chunks() >= 2
        o_ids, o_sc, _ = top_pairs_np(thetas, qrs, cand, known, N + 64)
        check_against_oracle(ids, sc, o_ids, o_sc, N)
    queries = rng.permutation(P).astype(np.int32)
    gi, gs, cnt = eng.top_pairs_per_gene(thetas, qrs, cand, queries, known, 20)
    assert eng.lib.tip_top_pairs_per_gene_last_chunks() == -(-P // (CHUNK // (P - 1)))
    for qi in rng.choice(P, size=60, replace=False).tolist() + [int(np.argmin(queries)), int(np.argmax(queries))]:
        o_ids, o_sc = per_gene_np(thetas, qrs, cand, known, int(queries[qi]), 84, M)
        check_against_oracle(gi[qi, :cnt[qi]], gs[qi, :cnt[qi]], o_ids, o_sc, 20)
    assert _cabi is not None


@pytest.mark.gpu
def test_1500_genes_against_score_pairs_and_a_sort(torch_cuda):
    import torch
    P, K = 1500, 10
    rng = np.random.default_rng(15)
    thetas, qrs = random_sets(rng, P, K, 1)
    eng = _engine(P, K)
    eng.set_params(thetas[0], np.zeros((K, K, K, 2)))
    eng.set_q(qrs[0])
    cand = np.array(sorted(range(P), key=str), dtype=np.int32)
    ra, rb = np.triu_indices(P, 1)
    s = eng.score_pairs(cand[ra], cand[rb])
    order = torch.sort(-s, stable=True).indices.cpu().numpy()
    sc_all = s.cpu().numpy()
    N = 5000
    ids, sc = eng.top_pairs(thetas, qrs, cand, np.empty(0, np.uint64), N)
    o_ids = np.stack([cand[ra[order]], cand[rb[order]]], axis=1)
    check_against_oracle(ids, sc, o_ids, sc_all[order], N)
    # tip_score_pairs itself against the oracle
    M = pair_sums(thetas, qrs, cand)
    assert np.max(np.abs(sc_all - M[ra, rb]) / M[ra, rb]) < TOL


def _trained_golden(K, iterations=5):
    from oracle import digenic_oracle as dg
    m = _digested_model()
    random.seed(2300 + K)
    m.initialize_parameters(K)
    for _ in range(iterations):
        m.make_iteration()
    lines = open(os.path.join(DIGENIC, "train_mixed.dat"), encoding="utf-8").read().splitlines()
    l3, l2, _ = dg.digest_mixed(lines)
    return m, l3, l2


@pytest.mark.gpu
@pytest.mark.parametrize("K", [2, 3, 10])
def test_test_set_evaluation_against_the_oracle(torch_cuda, K):
    from oracle import digenic_oracle as dg
    from oracle import mmsbm_oracle as base
    m, _, _ = _trained_golden(K)
    th, pr, qr = np.array(m.theta), np.array(m.pr), np.array(m.qr)
    # the test lines, each counted once
    t3, t2 = {}, {}
    for line in open(os.path.join(DIGENIC, "test_mixed.dat"), encoding="utf-8"):
        f = line.strip().split("\t")
        ids = sorted(str(m.gene_id[g]) for g in f[0].split("_") if g != "hoΔ")
        (t3 if len(ids) == 3 else t2).setdefault("_".join(ids), [0, 0])[int(f[1])] += 1
    ids3 = np.array([[int(x) for x in k.split("_")] for k in t3], dtype=np.int64).reshape(-1, 3)
    ids2 = np.array([[int(x) for x in k.split("_")] for k in t2], dtype=np.int64).reshape(-1, 2)
    cnt3, cnt2 = np.array(list(t3.values())).reshape(-1, 2), np.array(list(t2.values())).reshape(-1, 2)
    assert len(t3) and len(t2)
    ll = m.compute_likelihood("test")
    assert ll == pytest.approx(dg.loglik_23_np(th, pr, qr, ids3, cnt3, ids2, cnt2), rel=1e-12)
    assert m.heldoutlikelihood == ll and m.likelihood == 0
    assert all(c % 2 == 0 for k, c2 in m.test_links.items() if k.count("_") == 2 for c in c2)   # test_links unchanged
    m.calculate_test_set_results()
    # triplet scores equal the trigenic tip_score of the same parameters, bit for bit
    keys3 = [r[1] for r in m.results]
    ref = m._engine.score_sum(th[None], pr[None], [[int(x) for x in k.split("_")] for k in keys3])
    assert [r[0] for r in m.results] == ref.tolist()
    assert sorted(keys3) == sorted(t3) and [r[2] for r in m.results] == [0 if t3[k][0] else 1 for k in keys3]
    for sc, key, _ in m.results:
        a, b, c = (int(x) for x in key.split("_"))
        assert sc == pytest.approx(base.predict_loops(th.tolist(), pr.tolist(), a, b, c), rel=TOL)
    # pair scores
    assert len(m.dresults) == len(t2)
    for sc, key, label in m.dresults:
        a, b = (int(x) for x in key.split("_"))
        assert abs(sc - th[a] @ qr[:, :, 1] @ th[b]) <= TOL * abs(sc)
        assert label == (0 if t2[key][0] else 1)
    assert [r[0] for r in m.dresults] == sorted((r[0] for r in m.dresults), reverse=True)
    # metrics against the quadratic loop of TIP.py:583-637
    for fn, train, rows in ((m.calculate_metrics, m.links, m.results), (m.calculate_pair_metrics, m.dlinks, m.dresults)):
        try:
            want = base.metrics_quadratic(rows, train, len(rows))
        except ZeroDivisionError:
            with pytest.raises(ZeroDivisionError):
                fn()
            continue
        assert fn() == want


@pytest.mark.gpu
def test_end_to_end_cli(torch_cuda, tmp_path):
    tr, te = os.path.join(DIGENIC, "train_mixed.dat"), os.path.join(DIGENIC, "test_mixed.dat")
    out = str(tmp_path) + os.sep
    r = _run("TrigenicInteractionPredictor_23", "-t", tr, "-e", te, "-k", "3", "-i", "400", "-n", "2", "-f", "10", "-b", "0",
             "--seed", "4", "--save-params", "-o", out)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.count("Likelihood has converged") == 2, r.stdout
    for s in (0, 1):
        assert os.path.isfile(out + "Sample_%d_K3.csv" % s) and os.path.isfile(out + "Sample_%d_K3.npz" % s)
    text = open(out + "Sample_0_K3.csv", encoding="utf-8").read()
    assert "Held-out Likelihood:\t" in text and "\nNumber of pair links:\t" in text and "\nPair test set:" in text
    before = os.path.getmtime(out + "Sample_0_K3.csv")
    r = _run("TrigenicInteractionPredictor_23", "-t", tr, "-e", te, "-k", "3", "-i", "30", "-n", "1", "--seed", "4", "-o", out)
    assert r.returncode == 0 and os.path.getmtime(out + "Sample_0_K3.csv") == before      # skip-if-exists
    p0, p1 = out + "Sample_0_K3.npz", out + "Sample_1_K3.npz"
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", p0, "-p", p1, "-n", "15")
    assert r.returncode == 0, r.stderr
    lines = r.stdout.splitlines()
    assert lines[0] == "Predicted Interaction\tID of genes\tGenes" and len(lines) == 16 and "READ DATA" in r.stderr
    m = _digested_model()
    sets = [m.check_parameters_file(p) for p in (p0, p1)]
    cand = np.array(sorted(range(m.P), key=str))
    o_ids, o_sc, _ = top_pairs_np([s[0] for s in sets], [s[2] for s in sets], cand, m._known_pairs(cand), 15 + 64)
    got = [(int(x.split("\t")[1].split("_")[0]), int(x.split("\t")[1].split("_")[1])) for x in lines[1:]]
    check_against_oracle(np.array(got), np.array([float(x.split("\t")[0]) for x in lines[1:]]), o_ids, o_sc, 15)
    for x in lines[1:]:
        s, key, names = x.split("\t")
        assert names == "_".join(sorted(m.id_gene[int(i)] for i in key.split("_")))
    q = tmp_path / "q.txt"
    names = [m.id_gene[3], m.id_gene[0]]
    q.write_text("\n".join(names) + "\n")
    r = _run("predict_pairs", "-t", tr, "-e", te, "-p", p0, "-n", "4", "-q", str(q), "-o", str(tmp_path / "o.tsv"))
    assert r.returncode == 0, r.stderr
    lines = open(tmp_path / "o.tsv", encoding="utf-8").read().splitlines()
    assert lines[0] == "Query gene\tPredicted Interaction\tID of genes\tGenes" and len(lines) == 9
    assert [x.split("\t")[0] for x in lines[1:]] == [names[0]] * 4 + [names[1]] * 4
    per = m.predict_top_pairs_per_gene(names, 4, params=[p0])
    assert [x.split("\t", 1)[1] for x in lines[1:]] == ["%r\t%s\t%s" % (s, k, nm) for g in names for s, k, nm in per[g]]
