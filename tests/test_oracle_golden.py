"""Pin the CPU oracle to vectors produced by the unmodified reference (oracle/gen_golden.py)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import fetch_ref
from oracle import mmsbm_oracle as orc
from tests.conftest import GOLDEN, read_lines

BASE = os.path.join(GOLDEN, "base")
DUPS = os.path.join(GOLDEN, "dups")


def _digest(case_dir, train="train1.dat", test="test1.dat"):
    return orc.digest_traintest(read_lines(os.path.join(case_dir, train)), read_lines(os.path.join(case_dir, test)))


def _check_digest(dg, rec):
    assert dg.P == rec["P"]
    assert [dg.id_gene[i] for i in range(dg.P)] == rec["genes_in_id_order"]
    assert [dg.uniqueg[i] for i in range(dg.P)] == rec["uniqueg"]
    assert list(dg.links.keys()) == rec["link_keys"]
    assert [list(v) for v in dg.links.values()] == rec["link_counts"]
    assert list(dg.nlinks.keys()) == rec["nlink_keys"]
    assert list(dg.test_links.keys()) == rec["test_keys"]
    assert [list(v) for v in dg.test_links.values()] == rec["test_counts"]


def test_digest_bit_exact_base():
    _check_digest(_digest(BASE), json.load(open(os.path.join(BASE, "digest.json"))))


def test_digest_bit_exact_dups_and_string_sort_trap():
    dg = _digest(DUPS, "train.dat", "test.dat")
    rec = json.load(open(os.path.join(DUPS, "digest.json")))
    _check_digest(dg, rec)
    # the trap itself: some key must be out of numeric order (e.g. "10_11_9")
    assert any([int(t) for t in k.split("_")] != sorted(int(t) for t in k.split("_")) for k in dg.links)
    assert any(max(v) > 1 for v in dg.links.values())          # duplicates counted
    assert any(v[0] and v[1] for v in dg.links.values())       # conflicting labels kept


def test_digest_testonly_gene_gets_id():
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    dg = _digest(os.path.join(GOLDEN, "testonly"), "train.dat", "test.dat")
    _check_digest(dg, man["testonly"]["digest"])
    assert man["testonly"]["exception"] == "ZeroDivisionError"
    ids, cnt = orc.links_to_arrays(dg.links)
    random.seed(5)
    th, pr = orc.init_params(dg.P, 2)
    with pytest.raises(ZeroDivisionError):
        orc.em_step_np(th, pr, ids, cnt)
    with pytest.raises(ZeroDivisionError):
        orc.em_step_loops(th.tolist(), pr.tolist(), ids.tolist(), cnt.tolist())
    with pytest.raises(ZeroDivisionError):
        orc.em_step_c(th, pr, ids, cnt)


def test_fold_files_bit_exact():
    """get_input is outside the oracle; the fold is replayed from the links the reference built."""
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))
    # rebuild the get_input state: ids in first-appearance order over (query1, query2, array)
    gene_id, id_gene, links = {}, {}, {}
    for line in read_lines(os.path.join(BASE, "input_s2.tsv"))[1:]:
        f = line.split("\t")
        names = f[1].split("+") + [f[3]]
        r = 1 if (float(f[6]) < 0.05 and float(f[5]) < -0.08) else 0
        ids = []
        for nm in names:
            if nm not in gene_id:
                gene_id[nm] = len(gene_id)
                id_gene[gene_id[nm]] = nm
            ids.append(str(gene_id[nm]))
        ids.sort()
        links.setdefault("_".join(ids), [0, 0])[r] += 1
    assert [id_gene[i] for i in range(len(id_gene))] == man["base"]["get_input"]["genes_in_id_order"]
    assert list(links)[:50] == man["base"]["get_input"]["link_keys_head"]
    np.random.seed(2)
    tests, trains = orc.fold_texts(links, id_gene, 0.2)
    for i in range(5):
        assert tests[i] == open(os.path.join(BASE, "test%d.dat" % i), encoding="utf-8").read()
        assert trains[i] == open(os.path.join(BASE, "train%d.dat" % i), encoding="utf-8").read()


@pytest.mark.parametrize("K", [1, 2, 3, 10])
def test_init_bit_exact(K):
    dg = _digest(BASE)
    tr = np.load(os.path.join(BASE, "trace_K%d.npz" % K))
    random.seed(1000)
    th, pr = orc.init_params(dg.P, K)
    assert np.array_equal(th, tr["theta0"])
    assert np.array_equal(pr, tr["pr0"])
    assert random.random() == tr["after_init_random"][0]      # same number of draws consumed


def _trace_check(case_dir, K, train, test, seed, iters, stepper, rtol):
    dg = _digest(case_dir, train, test)
    tr = np.load(os.path.join(case_dir, "trace_K%d.npz" % K))
    ids, cnt = orc.links_to_arrays(dg.links)
    tids, tcnt = orc.links_to_arrays(dg.test_links)
    th, pr = tr["theta0"], tr["pr0"]
    assert orc.loglik_np(th, pr, ids, cnt) == pytest.approx(tr["loglik"][0], rel=rtol)
    for it in range(iters):
        th, pr = stepper(th, pr, ids, cnt)
        np.testing.assert_allclose(th, tr["theta%d" % (it + 1)], rtol=rtol, atol=1e-300)
        np.testing.assert_allclose(pr, tr["pr%d" % (it + 1)], rtol=rtol, atol=1e-300)
        assert orc.loglik_np(th, pr, ids, cnt) == pytest.approx(tr["loglik"][it + 1], rel=rtol)
    assert orc.loglik_np(th, pr, tids, tcnt) == pytest.approx(tr["heldout"][0], rel=rtol)
    return dg, tr, th, pr, tids


@pytest.mark.parametrize("K", [1, 2, 3, 10])
def test_em_trace_numpy(K):
    dg, tr, th, pr, tids = _trace_check(BASE, K, "train1.dat", "test1.dat", 1000, 5, orc.em_step_np, 1e-12)
    sc = orc.scores_np(th, pr, tids)
    np.testing.assert_allclose(sc, tr["scores_test_order"], rtol=1e-12)
    # results order and metrics from the REFERENCE's own scores (ordering is exact given equal scores)
    res = orc.test_results(tr["scores_test_order"], dg.test_links)
    assert [r[1] for r in res] == tr["result_keys"].tolist()
    assert [r[2] for r in res] == tr["result_labels"].tolist()
    assert np.array_equal(np.array([r[0] for r in res]), tr["result_scores"])
    m = orc.metrics(res, dg.links, len(dg.test_links))
    assert m == tr["metrics"].tolist()
    assert orc.metrics_quadratic(res, dg.links, len(dg.test_links)) == tr["metrics"].tolist()


def test_em_trace_dups_numpy():
    _trace_check(DUPS, 3, "train.dat", "test.dat", 1001, 3, orc.em_step_np, 1e-12)


KUZMIN = os.path.join(GOLDEN, "kuzmin")


@pytest.mark.parametrize("K,iters", [(3, 5), (10, 3)])
def test_em_trace_kuzmin_hub_shaped(K, iters):
    """Hub-shaped data (query pair x array gene, oracle/gen_golden_kuzmin.py): digestion bit-exact incl. where the
    hubs land under the decimal-string slot order, EM trace / scores / metrics of the unmodified reference."""
    info = json.load(open(os.path.join(KUZMIN, "info.json")))
    _check_digest(_digest(KUZMIN), json.load(open(os.path.join(KUZMIN, "digest.json"))))
    dg, tr, th, pr, tids = _trace_check(KUZMIN, K, "train1.dat", "test1.dat", 1000, iters, orc.em_step_np, 1e-12)
    ids, _ = orc.links_to_arrays(dg.links)
    deg = [np.bincount(ids[:, s], minlength=dg.P) for s in range(3)]
    assert [int(d.max()) for d in deg] == info["max_degree_per_slot"]
    assert min(info["max_degree_per_slot"]) > 100           # hubs in every slot
    np.testing.assert_allclose(orc.scores_np(th, pr, tids), tr["scores_test_order"], rtol=1e-12)
    res = orc.test_results(tr["scores_test_order"], dg.test_links)
    assert [r[1] for r in res] == tr["result_keys"].tolist()
    assert orc.metrics(res, dg.links, len(dg.test_links)) == tr["metrics"].tolist()


@pytest.mark.parametrize("K", [2, 3])
def test_em_trace_c_bit_exact(K):
    """The literal-order C restatement reproduces CPython's doubles bit for bit."""
    dg = _digest(BASE)
    tr = np.load(os.path.join(BASE, "trace_K%d.npz" % K))
    ids, cnt = orc.links_to_arrays(dg.links)
    th, pr = tr["theta0"], tr["pr0"]
    for it in range(5):
        th, pr = orc.em_step_c(th, pr, ids, cnt)
        assert np.array_equal(th, tr["theta%d" % (it + 1)])
        assert np.array_equal(pr, tr["pr%d" % (it + 1)])
        assert orc.loglik_c(th, pr, ids, cnt) == tr["loglik"][it + 1]


def test_em_trace_c_K10_and_dups():
    _trace_check(BASE, 10, "train1.dat", "test1.dat", 1000, 5, orc.em_step_c, 1e-15)
    _trace_check(DUPS, 3, "train.dat", "test.dat", 1001, 3, orc.em_step_c, 1e-15)


def test_em_loops_match_one_iteration():
    dg = _digest(BASE)
    tr = np.load(os.path.join(BASE, "trace_K2.npz"))
    ids, cnt = orc.links_to_arrays(dg.links)
    th, pr = orc.em_step_loops(tr["theta0"].tolist(), tr["pr0"].tolist(), ids.tolist(), cnt.tolist())
    assert np.array_equal(np.array(th), tr["theta1"])
    assert np.array_equal(np.array(pr), tr["pr1"])
    assert orc.loglik_loops(th, pr, ids.tolist(), cnt.tolist()) == tr["loglik"][1]
    k0 = [int(t) for t in next(iter(dg.test_links)).split("_")]
    th5, pr5 = tr["theta5"].tolist(), tr["pr5"].tolist()
    assert orc.predict_loops(th5, pr5, *k0) == tr["predict_by_name"][0] == tr["predict_by_name"][1]


def test_c_multithreaded_stats_sum_to_single_thread():
    dg = _digest(BASE)
    tr = np.load(os.path.join(BASE, "trace_K3.npz"))
    ids, cnt = orc.links_to_arrays(dg.links)
    nt, npr = orc.em_stats_c_mt(tr["theta0"], tr["pr0"], ids, cnt, threads=4)
    nt1, npr1, deg = orc.em_step_np(tr["theta0"], tr["pr0"], ids, cnt, return_stats=True)
    np.testing.assert_allclose(nt, nt1, rtol=1e-12)
    np.testing.assert_allclose(npr, npr1, rtol=1e-12)
    th, pr = orc.normalise_np(nt, npr, deg)
    np.testing.assert_allclose(th, tr["theta1"], rtol=1e-12)


def test_training_loop_semantics():
    man = json.load(open(os.path.join(GOLDEN, "manifest.json")))["base"]["loop"]
    dg = _digest(BASE)
    ids, cnt = orc.links_to_arrays(dg.links)
    random.seed(1000)
    th, pr = orc.init_params(dg.P, man["K"])
    th, pr, conv, done, like, trace = orc.train_sample_np(th, pr, ids, cnt, man["iterations"], man["fcheck"],
                                                          man["bcheck"])
    assert conv and done - 1 == man["converged_at_iteration"]
    np.testing.assert_allclose(trace, man["checks"], rtol=1e-11)


@pytest.mark.skipif(not os.path.exists(fetch_ref.DST),
                    reason="needs the original TrigenicInteractionPredictor.py in oracle/_ref/ (python oracle/fetch_ref.py)")
@pytest.mark.parametrize("seed", range(4))
def test_oracle_against_the_live_reference_on_random_files(tmp_path, monkeypatch, seed):
    """The unmodified reference, loaded from its sha256-checked copy in oracle/_ref/, digests random files (unsorted
    names, duplicates, conflicts, test-only genes, ids of different digit counts), folds them and runs two EM
    iterations; the oracle must agree - dictionaries and fold files exactly, theta / p / log-likelihood to 1e-12."""
    import contextlib
    import io
    import random
    ref = fetch_ref.load_reference_module()
    assert ref is not None, "oracle/_ref/ holds a file whose sha256 is not the pinned reference's"
    rng = np.random.default_rng(500 + seed)
    P = int(rng.integers(10, 60))
    names = ["G%d" % v for v in rng.permutation(3000)[:P]]

    def triple():
        t = [names[i] for i in rng.choice(P, size=3, replace=False)]
        rng.shuffle(t)
        return "_".join(t)
    train = [triple() + "\t" + str(int(rng.random() < 0.3)) + "\n" for _ in range(int(rng.integers(60, 250)))]
    train += [names[i] + "_" + names[(i + 1) % P] + "_" + names[(i + 2) % P] + "\t0\n" for i in range(P)]   # coverage
    train += [train[i] for i in rng.integers(0, len(train), size=len(train) // 6)]
    train += [train[i].rsplit("\t", 1)[0] + "\t" + ("0" if train[i].strip().endswith("1") else "1") + "\n"
              for i in rng.integers(0, len(train), size=len(train) // 8)]
    test = [triple() + "\t" + str(int(rng.random() < 0.3)) + "\n" for _ in range(30)]
    tr, te = tmp_path / "train.dat", tmp_path / "test.dat"
    tr.write_text("".join(train))
    te.write_text("".join(test))
    m = ref.Model()
    with contextlib.redirect_stdout(io.StringIO()):
        m.get_traintest(str(tr), str(te))
    dg = orc.digest_traintest(train, test)
    assert (m.P, m.gene_id, m.id_gene, m.uniqueg) == (dg.P, dg.gene_id, dg.id_gene, dg.uniqueg)
    for mine, ours in ((m.links, dg.links), (m.nlinks, dg.nlinks), (m.test_links, dg.test_links)):
        assert list(mine.items()) == list(ours.items())
    monkeypatch.chdir(tmp_path)
    np.random.seed(9 + seed)
    with contextlib.redirect_stdout(io.StringIO()):
        m.fold()
    np.random.seed(9 + seed)
    test_txt, train_txt = orc.fold_texts(dg.links, dg.id_gene)
    for i in range(5):
        assert (tmp_path / ("test%d.dat" % i)).read_text() == test_txt[i]
        assert (tmp_path / ("train%d.dat" % i)).read_text() == train_txt[i]
    K = 3
    random.seed(40 + seed)
    m.initialize_parameters(K)
    random.seed(40 + seed)
    theta, pr = orc.init_params(dg.P, K)
    ids, cnt = orc.links_to_arrays(dg.links)
    tids, tcnt = orc.links_to_arrays(dg.test_links)
    for _ in range(2):
        m.make_iteration()
        theta, pr = orc.em_step_np(theta, pr, ids, cnt)
    np.testing.assert_allclose(np.array(m.theta), theta, rtol=1e-12)
    np.testing.assert_allclose(np.array(m.pr), pr, rtol=1e-12)
    assert m.compute_likelihood() == pytest.approx(orc.loglik_np(theta, pr, ids, cnt), rel=1e-12)
    assert m.compute_likelihood("test") == pytest.approx(orc.loglik_np(theta, pr, tids, tcnt), rel=1e-12)


# ---------------------------------------------------------------------------------------------- digenic extension (f-4)
DIGENIC = os.path.join(GOLDEN, "digenic")


@pytest.mark.parametrize("K", [2, 3, 10])
def test_digenic_oracle_and_host_model_against_the_patched_reference(K):
    """tests/golden/digenic was produced by the author's TrigenicInteractionPredictor_23.py made importable by the
    two-token recipe of oracle/gen_golden_23.py.  The oracle restatement and the host side of the drop-in class must
    give its ids, counts and initial parameters exactly (RNG position included) and its iterations to 1e-12."""
    import contextlib
    import io
    import random
    from oracle import digenic_oracle as dg
    from trigenicinteractionpredictor_b200.TrigenicInteractionPredictor_23 import Model
    tr = np.load(os.path.join(DIGENIC, "trace23_K%d.npz" % K))
    lines = open(os.path.join(DIGENIC, "train_mixed.dat"), encoding="utf-8").read().splitlines()
    l3, l2, P = dg.digest_mixed(lines)
    ids3 = np.array([[int(t) for t in k.split("_")] for k in l3])
    ids2 = np.array([[int(t) for t in k.split("_")] for k in l2])
    cnt3, cnt2 = np.array(list(l3.values())), np.array(list(l2.values()))
    assert P == int(tr["P"])
    for got, want in ((ids3, "ids3"), (cnt3, "cnt3"), (ids2, "ids2"), (cnt2, "cnt2")):
        assert np.array_equal(got, tr[want]), want
    random.seed(2300 + K)
    th, p, q = dg.init_params_23(P, K)
    assert np.array_equal(th, tr["theta0"]) and np.array_equal(p, tr["pr0"]) and np.array_equal(q, tr["qr0"])
    assert random.random() == float(tr["rng_next"])
    assert dg.loglik_23_np(th, p, q, ids3, cnt3, ids2, cnt2) == pytest.approx(tr["loglik"][0], rel=1e-12)
    for it in range(len(tr["loglik"]) - 1):
        th, p, q = dg.em_step_23_np(th, p, q, ids3, cnt3, ids2, cnt2)
        np.testing.assert_allclose(th, tr["theta%d" % (it + 1)], rtol=1e-12)
        np.testing.assert_allclose(p, tr["pr%d" % (it + 1)], rtol=1e-12)
        np.testing.assert_allclose(q, tr["qr%d" % (it + 1)], rtol=1e-12)
        assert dg.loglik_23_np(th, p, q, ids3, cnt3, ids2, cnt2) == pytest.approx(tr["loglik"][it + 1], rel=1e-12)
    # the product's host side: digestion and initialisation (no GPU needed)
    m = Model()
    with contextlib.redirect_stdout(io.StringIO()):
        m.get_train_test(os.path.join(DIGENIC, "train_mixed.dat"), os.path.join(DIGENIC, "test_mixed.dat"))
    random.seed(2300 + K)
    m.initialize_parameters(K)
    a3, c3 = Model._arrays(m.links, 3)
    a2, c2 = Model._arrays(m.dlinks, 2)
    assert m.P == P and np.array_equal(a3, ids3) and np.array_equal(c3, cnt3) and np.array_equal(a2, ids2) and np.array_equal(c2, cnt2)
    assert np.array_equal(np.array(m.theta), tr["theta0"]) and np.array_equal(np.array(m.pr), tr["pr0"])
    assert np.array_equal(np.array(m.qr), tr["qr0"]) and random.random() == float(tr["rng_next"])
