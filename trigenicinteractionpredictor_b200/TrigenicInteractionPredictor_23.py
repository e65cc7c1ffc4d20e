#!/usr/bin/env python3
"""Drop-in `Model` for the DIGENIC extension of the reference, src/TrigenicInteractionPredictor_23.py (`_23.py`): the
trigenic model plus links between two genes (`dlinks`) that share theta and have their own rating tensor `qr[K][K][R]`.

Scope (SURVEY f-4): the training path - `get_train_test` (mixed train files: a line with two gene names is a pair,
_23.py:393-450), `initialize_parameters` (_23.py:123-217: theta rows, pr cells, then qr cells from the same
`random.random()` stream), `make_iteration` (_23.py:1572-1687) and `compute_likelihood` (_23.py:1534-1562).  Same method
names, attributes (`theta`, `pr`, `qr`, `links`, `dlinks`, `test_links`, `dtest_links`, `gene_id`, `id_gene`,
`gene_num_aparitions`, `likelihood`, `K`, `P`, `R`, `eps`) and error behaviour as the author's class; the numerics run on
the device: the triplet term through the same E-step kernels as the trigenic `Model`, the pair term through
`tip_pairs_step` / `tip_pairs_normalise` / `tip_pairs_loglik` (csrc/tip_pairs.cu).  The author's file does not run as
shipped (an enum member is misspelled); oracle/gen_golden_23.py documents the two-token recipe that makes it importable
and froze the vectors this class is tested against.

Past the training path the author's file cannot run as shipped, so the rest is an ADDITION defined in DESIGN §4.11 and
held to a NumPy oracle, not to the author's test-set code: `make_iterations`, the held-out likelihood, the test-set
tables of triplets (`results`) and pairs (`dresults`) with their metrics, the report (`to_string` / `to_file`), kept
parameters (`save_parameters`, `check_parameters_file`, `load_parameters`: the trigenic .npz plus `qr`), and the N best
unseen gene pairs (`predict_top_pairs`, `predict_top_pairs_per_gene`).  The command line

    python -m trigenicinteractionpredictor_b200.TrigenicInteractionPredictor_23 -t train_mixed.dat -e test_mixed.dat \\
        [-i -n -s -f -b -o -k --seed --device --save-params]

trains as the trigenic command line does (same flags, defaults, Sample_{s}_K{k}.csv / .npz naming, skip-if-exists).

There is no CPU fallback: without libtip.so and a CUDA device the numeric methods raise."""
from __future__ import annotations

import codecs
import collections
import getopt
import os
import random
import re
import sys

import numpy as np

__all__ = ["Model"]


class Model:
    def __init__(self, device=None, flags: int | None = None):
        self.id_gene, self.gene_id = {}, {}
        self.links, self.nLinks = {}, {}
        self.dlinks, self.ndlinks = {}, {}
        self.test_links, self.dtest_links = {}, {}
        self.gene_num_aparitions = {}
        self.results, self.dresults = [], []
        self.likelihood = 0
        self.heldoutlikelihood = 0
        self.likelihoodVector = []
        self.R, self.K, self.P = 2, 0, 0
        self.eps = 1e-10
        self._device, self._flags = device, flags
        self._engine = None
        self._theta, self._pr, self._qr = [], [], []
        self._on_device = False

    # ---------------------------------------------------------------- parameters (host mirrors, lists like the reference's)
    def _pull(self):
        if self._on_device:
            th, pr = self._engine.get_params()
            self._theta, self._pr, self._qr = th.tolist(), pr.tolist(), self._engine.get_q().tolist()
            self._on_device = False

    @property
    def theta(self):
        self._pull()
        return self._theta

    @property
    def pr(self):
        self._pull()
        return self._pr

    @property
    def qr(self):
        self._pull()
        return self._qr

    def initialize_parameters(self, k=2, interaction=None):
        try:
            self.K = int(k)
        except ValueError:
            self.K = 2
        self.dataType = interaction
        self.likelihoodVector = []
        K, R, rnd = self.K, self.R, random.random
        # draw order of _23.py:137-172: every theta row, every pr cell (i, j, k, r), then every qr cell (i, j, r)
        theta = [[rnd() for _ in range(K)] for _ in range(self.P)]
        pr = [[[[rnd() for _ in range(R)] for _ in range(K)] for _ in range(K)] for _ in range(K)]
        qr = [[[rnd() for _ in range(R)] for _ in range(K)] for _ in range(K)]
        for g in range(self.P):
            acc = 0.0
            for v in theta[g]:
                acc += v
            if acc < self.eps:                               # _23.py:180-182
                theta[g] = [rnd() for _ in range(K)]
            total = sum(theta[g])
            row = theta[g]
            for kk in range(K):
                try:
                    row[kk] /= total
                except ZeroDivisionError:
                    row[kk] /= (total + self.eps)
        for cells in ([c for plane in pr for line in plane for c in line], [c for line in qr for c in line]):
            for cell in cells:
                acc = 0.0
                for r in range(R):
                    acc += cell[r]
                for r in range(R):
                    try:
                        cell[r] /= acc
                    except ZeroDivisionError:
                        cell[r] /= (acc + self.eps)
        self._theta, self._pr, self._qr = theta, pr, qr
        self._on_device = False
        self._uploaded = False

    # ---------------------------------------------------------------- digestion (_23.py:393-560)
    def _register(self, names, next_id):
        ids = []
        for name in names:
            gid = self.gene_id.get(name)
            if gid is None:
                gid = next_id
                next_id += 1
                self.gene_id[name] = gid
                self.id_gene[gid] = name
                self.gene_num_aparitions[gid] = 0
            self.gene_num_aparitions[gid] += 1
            ids.append(str(gid))
        return ids, next_id

    @staticmethod
    def _bump(table, key, r):
        cell = table.get(key)
        if cell is None:
            cell = table[key] = [0, 0]
        cell[r] += 1

    def get_train_test(self, train_file_path, test_file_path):
        try:
            next_id = 0
            with codecs.open(train_file_path, encoding='utf-8', mode='r') as fh:
                for line in fh.readlines():
                    fields = line.strip().split('\t')
                    names = fields[0].split('_')
                    if 'hoΔ' in names:
                        names.remove('hoΔ')
                    rating = int(fields[1])
                    ids, next_id = self._register(names, next_id)
                    names.sort()
                    ids.sort()                               # STRING sort of the decimal ids (_23.py:427)
                    if len(names) == 3:
                        self._bump(self.links, '_'.join(ids), rating)
                        self._bump(self.nLinks, '_'.join(names), rating)
                    if len(names) == 2:
                        self._bump(self.dlinks, '_'.join(ids), rating)
                        self._bump(self.ndlinks, '_'.join(names), rating)
                self.P = len(self.id_gene)
            print('number of triplets, pairs', len(self.links), len(self.dlinks))
            with codecs.open(test_file_path, encoding='utf-8', mode='r') as fh:
                for line in fh.readlines():
                    fields = re.split(r'\t+', line)
                    names = fields[0].split('_')
                    if 'hoΔ' in names:
                        names.remove('hoΔ')
                    rating = int(fields[1])
                    ids, next_id = self._register(names, next_id)
                    names.sort()
                    ids.sort()
                    key = '_'.join(ids)
                    self._bump(self.test_links, key, rating)          # every line, and once more for a triplet (_23.py:502-516)
                    if len(names) == 3:
                        self._bump(self.test_links, key, rating)
                    if len(names) == 2:
                        self._bump(self.dtest_links, key, rating)
                self.P = len(self.id_gene)
        except ValueError as error:
            print(error)
        except IOError as error:
            print('Error, file does not exist or can\'t be read')
            print(error)
        print('READ DATA train', len(self.links), len(self.nLinks))
        print('READ DATA train', len(self.dlinks), len(self.ndlinks))
        print('READ DATA test', len(self.test_links))
        self._engine = None

    # ---------------------------------------------------------------- device
    @staticmethod
    def _arrays(table, width):
        n = len(table)
        if n == 0:
            return np.empty((0, width), dtype=np.int32), np.empty((0, 2), dtype=np.int32)
        ids = np.array("_".join(table.keys()).split("_"), dtype=np.int64).astype(np.int32).reshape(n, width)
        cnt = np.fromiter((c for pair in table.values() for c in pair), dtype=np.int32, count=2 * n).reshape(n, 2)
        return ids, cnt

    def _ready(self):
        from .engine import EMEngine
        if self.K < 1 or self.P < 1:
            raise ValueError("initialize_parameters() and get_train_test() must run before numeric methods")
        if self._engine is None or self._engine.K != self.K or self._engine.P != self.P:
            eng = EMEngine(self.P, self.K, device=self._device, flags=self._flags)
            ids3, cnt3 = self._arrays(self.links, 3)
            ids2, cnt2 = self._arrays(self.dlinks, 2)
            eng.set_train_links(ids3[:, 0], ids3[:, 1], ids3[:, 2], cnt3[:, 0], cnt3[:, 1])
            eng.set_pair_links(ids2[:, 0], ids2[:, 1], cnt2[:, 0], cnt2[:, 1])
            deg = np.bincount(np.concatenate([ids3.ravel(), ids2.ravel()]), minlength=self.P)
            self._deg_zero = bool((deg[: self.P] == 0).any())
            self._engine = eng
            self._uploaded = False
        if not self._uploaded:
            self._engine.set_params(np.asarray(self._theta, dtype=np.float64), np.asarray(self._pr, dtype=np.float64))
            self._engine.set_q(np.asarray(self._qr, dtype=np.float64))
            self._uploaded = True
        return self._engine

    def make_iteration(self):
        eng = self._ready()
        if self._deg_zero:
            raise ZeroDivisionError("float division by zero")     # _23.py:1643, a gene that has no training link
        eng.em_iteration()
        self._on_device = True

    def make_iterations(self, n):
        """n x make_iteration, the iteration body (triplet and pair terms) replayed from a CUDA graph (addition)."""
        eng = self._ready()
        if self._deg_zero:
            raise ZeroDivisionError("float division by zero")
        eng.em_iterations(int(n))
        self._on_device = True

    def compute_likelihood(self, selected_set='train'):
        """'train' (the default, _23.py:1534-1562) sets `likelihood`.  Anything else sets `heldoutlikelihood`: the same
        sum over the held-out links, the triplet keys of `test_links` through tip_loglik and `dtest_links` through
        tip_pairs_loglik.  get_train_test adds every triplet test line to `test_links` twice (_23.py:502-516); the
        held-out likelihood counts each test line once, so it uses half of those counts.  `test_links` is not changed."""
        eng = self._ready()
        if selected_set == 'train':
            self.likelihood = eng.loglik("train")
            return self.likelihood
        self._test_ready()
        if eng.test is None and eng.test_pairs is None:
            self.heldoutlikelihood = 0.0
        else:
            self.heldoutlikelihood = eng.loglik("test")
        return self.heldoutlikelihood

    # ---------------------------------------------------------------- held-out links, test-set tables and metrics (additions)
    def _test_triplets(self):
        """(keys, ids [T][3], counts [T][2] per test line) of the triplet keys of test_links."""
        keys = [k for k in self.test_links if k.count('_') == 2]
        if not keys:
            return keys, np.empty((0, 3), dtype=np.int32), np.empty((0, 2), dtype=np.int32)
        ids = np.array("_".join(keys).split("_"), dtype=np.int64).astype(np.int32).reshape(-1, 3)
        cnt = np.array([self.test_links[k] for k in keys], dtype=np.int32).reshape(-1, 2) // 2
        return keys, ids, cnt

    def _test_ready(self):
        eng = self._ready()
        if getattr(eng, "_digenic_test_set", False):
            return eng
        _, ids3, cnt3 = self._test_triplets()
        if ids3.shape[0]:
            eng.set_test_links(ids3[:, 0], ids3[:, 1], ids3[:, 2], cnt3[:, 0], cnt3[:, 1])
        ids2, cnt2 = self._arrays(self.dtest_links, 2)
        if ids2.shape[0]:
            eng.set_test_pair_links(ids2[:, 0], ids2[:, 1], cnt2[:, 0], cnt2[:, 1])
        eng._digenic_test_set = True
        return eng

    @staticmethod
    def _sorted_rows(eng, scores, keys, labels):
        """[[score, key, label], ...] in the order of list.sort(); reverse() (TIP.py:568-569), as the trigenic
        _build_results: the device sorts the scores, rows with EQUAL scores are put in list order on the host."""
        if len(keys) == 0:
            return []
        order, sorted_scores = eng.sort_scores(scores)
        rows = [[s, keys[i], labels[i]] for s, i in zip(sorted_scores.tolist(), order.tolist())]
        ties = np.flatnonzero(sorted_scores[1:] == sorted_scores[:-1])
        if ties.size:
            starts = ties[np.concatenate([[True], np.diff(ties) > 1])]
            for lo in starts.tolist():
                hi = lo + 1
                while hi < len(rows) and rows[hi][0] == rows[lo][0]:
                    hi += 1
                rows[lo:hi] = sorted(rows[lo:hi], reverse=True)
        return rows

    def calculate_test_set_results(self):
        """`results`: [score, "a_b_c", label] of every triplet key of test_links (do_prediction, tip_score); `dresults`:
        [score, "a_b", label] of every key of dtest_links (the pair score of DESIGN §4.11, tip_score_pairs).  Both sorted
        descending as the trigenic report sorts them; a label is 0 when the key has a negative sighting, else 1."""
        import torch
        eng = self._test_ready()
        keys3, ids3, _ = self._test_triplets()
        self._scores3 = eng.scores() if ids3.shape[0] else torch.empty(0, dtype=torch.float64, device=eng.device)
        self._labels3 = [0 if self.test_links[k][0] else 1 for k in keys3]
        self.results = self._sorted_rows(eng, self._scores3, keys3, self._labels3)
        keys2 = list(self.dtest_links.keys())
        ids2, _ = self._arrays(self.dtest_links, 2)
        self._scores2 = eng.score_pairs(ids2[:, 0], ids2[:, 1])
        self._labels2 = [0 if self.dtest_links[k][0] else 1 for k in keys2]
        self.dresults = self._sorted_rows(eng, self._scores2, keys2, self._labels2)

    def _metrics(self, train, scores, labels):
        """TIP.py:583-637: positives_fraction from the train keys with exactly one positive sighting, strict '>' AUC,
        the same ZeroDivisionError cases."""
        import torch
        hits = 0
        for n in train.values():
            if n[1] == 1:
                hits += 1
        positives_fraction = hits / len(train)
        positives_number = int(positives_fraction * len(labels))
        if scores is None or int(scores.numel()) == 0:
            wins = npos = nneg = tp = fp = fn = tn = 0
        else:
            lab = torch.tensor(labels, dtype=torch.int32, device=scores.device)
            c = self._engine.metric_counts(scores, positives_number, labels=lab)
            wins, npos, nneg = c["wins"], c["n_pos"], c["n_neg"]
            tp, fp, fn, tn = c["tp"], c["fp"], c["fn"], c["tn"]
        auc = wins / (npos * nneg)
        precision = tp / (tp + fp)
        recall = tp / (tp + fn)
        fallout = fp / (fp + tn)
        return [precision, recall, fallout, auc]

    def calculate_metrics(self):
        """[precision, recall, fallout, auc] of the triplet test table (calculate_test_set_results first), by TIP's rules
        with `links` as the train set and the triplet keys of test_links as the test set."""
        return self._metrics(self.links, getattr(self, "_scores3", None), getattr(self, "_labels3", []))

    def calculate_pair_metrics(self):
        """The same for the pair test table, with `dlinks` as the train set and `dtest_links` as the test set."""
        return self._metrics(self.dlinks, getattr(self, "_scores2", None), getattr(self, "_labels2", []))

    def to_string(self):
        """The trigenic report (TIP.py:793-904) of the triplet part, then, when the model has held-out pair links, the
        number of pair links, the pair metrics and the pair test table."""
        out = ["Max Likelihood:\t", str(self.likelihood), "\n",
               "Held-out Likelihood:\t", str(self.compute_likelihood('test')), "\n",
               "Number of genes (P):\t", str(self.P), "\n",
               "Number of links:\t", str(len(self.links)), "\n",
               "Number of groups of genes (K):\n", str(self.K), "\n",
               "Number of possible ratings (R):\n", str(self.R), "\n\n"]
        self.calculate_test_set_results()
        m = self.calculate_metrics()
        out.append("\nMetrics:\nPrecision\tRecall\tFallout\tAUC\n")
        out.append(str(m[0]) + "\t" + str(m[1]) + "\t" + str(m[2]) + "\t" + str(m[3]))
        out.append("\nTest set:")
        out.append('\nPredicted Interaction\tID of genes\tReal Interaction\n')
        for score, key, label in self.results:
            out.append(str(score) + '\t' + str(key) + '\t' + str(label) + '\n')
        if self.dtest_links:
            d = self.calculate_pair_metrics()
            out.append("\nNumber of pair links:\t" + str(len(self.dlinks)) + "\n")
            out.append("\nPair metrics:\nPrecision\tRecall\tFallout\tAUC\n")
            out.append(str(d[0]) + "\t" + str(d[1]) + "\t" + str(d[2]) + "\t" + str(d[3]))
            out.append("\nPair test set:")
            out.append('\nPredicted Interaction\tID of genes\tReal Interaction\n')
            for score, key, label in self.dresults:
                out.append(str(score) + '\t' + str(key) + '\t' + str(label) + '\n')
        return ''.join(out)

    def to_file(self, name_file=None):
        try:
            if name_file is None:
                name_file = "out.txt"
            with codecs.open(name_file, encoding='utf-8', mode="w+") as fh:
                fh.write(self.to_string())
        except IOError:
            print("I/O error")

    # ---------------------------------------------------------------- kept parameters (additions)
    def _genes_in_id_order(self):
        return [self.id_gene[i] for i in range(self.P)]

    def save_parameters(self, path):
        """Write theta, pr, qr, K and the gene names in id order to an .npz file at exactly `path`."""
        theta = np.asarray(self.theta, dtype=np.float64).reshape(self.P, self.K)
        pr = np.asarray(self.pr, dtype=np.float64).reshape(self.K, self.K, self.K, self.R)
        qr = np.asarray(self.qr, dtype=np.float64).reshape(self.K, self.K, self.R)
        with open(path, "wb") as fh:
            np.savez(fh, theta=theta, pr=pr, qr=qr, K=np.int64(self.K), genes=np.array(self._genes_in_id_order(), dtype=str))

    def check_parameters_file(self, path):
        """(theta [P][K], pr [K][K][K][2], qr [K][K][2]) of an .npz written by save_parameters, checked against this
        model's digestion: the same genes in the same id order, the model's K (when it has one), the shapes, finite
        non-negative values.  A trigenic file (no qr) is refused.  Raises ValueError with the reason.  Host only."""
        try:
            with np.load(path, allow_pickle=False) as z:
                if "qr" not in z.files:
                    raise ValueError("%s has no qr: a trigenic parameter file, not one of the digenic model" % path)
                theta, pr, qr, K = z["theta"], z["pr"], z["qr"], int(z["K"])
                genes = [str(g) for g in z["genes"]]
        except (OSError, KeyError) as exc:
            raise ValueError("%s is not a parameter file of save_parameters (%s)" % (path, exc)) from exc
        except ValueError as exc:
            if "trigenic parameter file" in str(exc):
                raise
            raise ValueError("%s is not a parameter file of save_parameters (%s)" % (path, exc)) from exc
        return self._check_parameters(theta, pr, qr, K, genes, str(path))

    def _check_parameters(self, theta, pr, qr, K, genes, what):
        theta = np.asarray(theta, dtype=np.float64)
        pr = None if pr is None else np.asarray(pr, dtype=np.float64)
        qr = np.asarray(qr, dtype=np.float64)
        if genes is not None and genes != self._genes_in_id_order():
            raise ValueError("%s: its gene list (%d genes) differs from the model's digestion (%d genes)"
                             % (what, len(genes), self.P))
        if self.K and K != self.K:
            raise ValueError("%s: K = %d, the model has K = %d" % (what, K, self.K))
        if theta.shape != (self.P, K) or qr.shape != (K, K, self.R) or (pr is not None and pr.shape != (K, K, K, self.R)):
            raise ValueError("%s: theta %s / pr %s / qr %s do not have the shapes (%d, %d) / (%d, %d, %d, %d) / (%d, %d, %d)"
                             % (what, theta.shape, None if pr is None else pr.shape, qr.shape, self.P, K, K, K, K, self.R,
                                K, K, self.R))
        arrays = [a for a in (theta, pr, qr) if a is not None]
        if not all(np.isfinite(a).all() for a in arrays):
            raise ValueError("%s: theta, pr or qr holds a non-finite value" % what)
        if any((a < 0).any() for a in arrays):
            raise ValueError("%s: theta, pr or qr holds a negative value" % what)
        return theta, pr, qr

    def load_parameters(self, path):
        """Make the parameters of an .npz written by save_parameters the model's current theta / pr / qr (see
        check_parameters_file for what is refused)."""
        theta, pr, qr = self.check_parameters_file(path)
        self.K = theta.shape[1]
        self._theta, self._pr, self._qr = theta.tolist(), pr.tolist(), qr.tolist()
        self._on_device = False
        self._uploaded = False

    # ---------------------------------------------------------------- the N best unseen gene pairs (additions, DESIGN §4.11)
    def _pair_sets(self, params, who):
        """The checked (theta, qr) sets a prediction averages over: the current theta / qr, or `params` (.npz paths of
        save_parameters or (theta, qr) pairs).  Raises ValueError (messages prefixed with `who`)."""
        if self.P < 1 or len(self.id_gene) != self.P:
            raise ValueError(who + " needs a model digested from train / test files")
        if params is None:
            if self.K < 1 or not self._theta and not self._on_device:
                raise ValueError(who + ": initialize_parameters() or load_parameters() must run first")
            th, _, q = self._check_parameters(self.theta, None, self.qr, self.K, None, "the model's parameters")
            return [(th, q)]
        sets = []
        for item in params:
            if isinstance(item, (str, bytes, os.PathLike)):
                th, _, q = self.check_parameters_file(item)
            else:
                th, q = item
                th, _, q = self._check_parameters(th, None, q, np.asarray(th).shape[-1], None, "a (theta, qr) pair")
            sets.append((th, q))
        if not sets:
            raise ValueError(who + ": params is empty")
        Ks = {th.shape[1] for th, _ in sets}
        if len(Ks) != 1:
            raise ValueError(who + ": the parameter sets have different K (%s)" % sorted(Ks))
        return sets

    def _pair_engine(self, K):
        from .engine import EMEngine
        if self._engine is not None and self._engine.K == K and self._engine.P == self.P:
            return self._engine
        return EMEngine(self.P, K, device=self._device, flags=self._flags)

    def _known_pairs(self, cand):
        """Sorted packed rank pairs (ra << 21 | rb) of the keys of dlinks and dtest_links whose two genes are both
        candidates."""
        rank = np.full(self.P, -1, dtype=np.int64)
        rank[cand] = np.arange(cand.shape[0], dtype=np.int64)
        parts = []
        for table in (self.dlinks, self.dtest_links):
            ids, _ = self._arrays(table, 2)
            if ids.shape[0] == 0:
                continue
            r = np.sort(rank[ids.astype(np.int64)], axis=1)
            r = r[(r[:, 0] >= 0) & (r[:, 0] < r[:, 1])]
            parts.append((r[:, 0] << 21) | r[:, 1])
        if not parts:
            return np.empty(0, dtype=np.uint64)
        return np.unique(np.concatenate(parts)).astype(np.uint64)

    def _pair_rows(self, ids, scores):
        rows = []
        for (a, b), s in zip(ids.tolist(), scores.tolist()):
            rows.append([s, "%d_%d" % (a, b), "_".join(sorted((self.id_gene[a], self.id_gene[b])))])
        return rows

    def predict_top_pairs(self, n, genes=None, exclude_known=True, params=None):
        """The `n` most likely interacting pairs of distinct genes among `genes` (names; default all P genes), by the pair
        score (DESIGN §4.11) of the current theta / qr, or by the mean over the parameter sets in `params` (.npz paths of
        save_parameters or (theta, qr) pairs).  With exclude_known the keys of dlinks and dtest_links are left out.
        Exhaustive over C(n_genes, 2) pairs on the device.  Returns [[score, "a_b", "nameA_nameB"], ...], best first;
        equal scores in ascending order of the pairs' positions in the decimal-string order of the candidate ids."""
        sets = self._pair_sets(params, "predict_top_pairs")
        K = sets[0][0].shape[1]
        if int(n) < 0:
            raise ValueError("predict_top_pairs: n must be >= 0 (got %d)" % int(n))
        if genes is None:
            ids = list(range(self.P))
        else:
            missing = [g for g in genes if g not in self.gene_id]
            if missing:
                raise ValueError("unknown gene names: %s" % ", ".join(missing))
            ids = sorted({self.gene_id[g] for g in genes})
        cand = np.array(sorted(ids, key=str), dtype=np.int32)
        known = self._known_pairs(cand) if exclude_known else np.empty(0, dtype=np.uint64)
        eng = self._pair_engine(K)
        out_ids, scores = eng.top_pairs(np.stack([th for th, _ in sets]), np.stack([q for _, q in sets]), cand, known, int(n))
        return self._pair_rows(out_ids, scores)

    def predict_top_pairs_per_gene(self, queries, n, genes=None, exclude_known=True, params=None):
        """For every gene of `queries` (names, distinct): the `n` most likely interacting pairs that contain it, its
        partner a distinct gene of `genes` + `queries` (names; default all P genes; the queries are always candidates),
        scored as in predict_top_pairs.  With exclude_known the keys of dlinks and dtest_links are left out.  Returns
        {query name: [[score, "a_b", "nameA_nameB"], ...]} in the order of `queries`, each list best first with ties in
        ascending order of the partner's rank; a list is shorter than n when the gene has fewer unseen pairs."""
        sets = self._pair_sets(params, "predict_top_pairs_per_gene")
        K = sets[0][0].shape[1]
        queries = list(queries)
        if not queries:
            raise ValueError("predict_top_pairs_per_gene: queries is empty")
        names = queries + (list(genes) if genes is not None else [])
        missing = [g for g in names if g not in self.gene_id]
        if missing:
            raise ValueError("unknown gene names: %s" % ", ".join(dict.fromkeys(missing)))
        twice = [g for g, c in collections.Counter(queries).items() if c > 1]
        if twice:
            raise ValueError("predict_top_pairs_per_gene: duplicate query genes: %s" % ", ".join(twice))
        if int(n) < 0:
            raise ValueError("predict_top_pairs_per_gene: n must be >= 0 (got %d)" % int(n))
        ids = set(range(self.P)) if genes is None else {self.gene_id[g] for g in names}
        cand = np.array(sorted(ids, key=str), dtype=np.int32)
        rank = {g: r for r, g in enumerate(cand.tolist())}
        qr = np.array([rank[self.gene_id[q]] for q in queries], dtype=np.int32)
        known = self._known_pairs(cand) if exclude_known else np.empty(0, dtype=np.uint64)
        eng = self._pair_engine(K)
        out_ids, scores, counts = eng.top_pairs_per_gene(np.stack([th for th, _ in sets]), np.stack([q for _, q in sets]),
                                                         cand, qr, known, int(n))
        return {q: self._pair_rows(out_ids[qi, :counts[qi]], scores[qi, :counts[qi]]) for qi, q in enumerate(queries)}


# ----------------------------------------------------------------------------------------------
# command line: the trigenic flags that apply to the digenic model (TrigenicInteractionPredictor.main), driving the same
# train_sample
# ----------------------------------------------------------------------------------------------
def main(argv=None):
    from .TrigenicInteractionPredictor import train_sample
    argv = sys.argv[1:] if argv is None else argv
    iterations, num_samples, sample_ini, fcheck, bcheck = 10000, 100, 0, 25, 100
    train = test = None
    outpath, argk = "", 1
    seed, device, save_params = None, None, False
    try:
        opts, rest = getopt.getopt(argv, "hi:n:s:f:b:o:t:e:k:",
                                   ["help", "num_iterations=", "num_samples=", "sample_ini=", "fcheck=", "bcheck=",
                                    "out=", "train=", "test=", "k=", "seed=", "device=", "save-params"])
        if rest:
            print("Argument error. Aborting")
            return 2
        for opt, arg in opts:
            if opt in ("-h", "--help"):
                print(__doc__)
                return 0
            elif opt in ("-i", "--num_iterations"):
                if int(arg) < 1:
                    print("\n\nERROR: Number of num_iterations should be a integer positive number!")
                    raise ValueError
                iterations = int(arg)
            elif opt in ("-n", "--num_samples"):
                if int(arg) < 1:
                    print("\n\nERROR: Number of samples should be a integer positive number")
                    raise ValueError
                num_samples = int(arg)
            elif opt in ("-s", "--sample_ini"):
                if int(arg) < 0:
                    print("\n\nERROR: Number of samples should be a integer positive number!")
                    raise ValueError
                sample_ini = int(arg)
            elif opt in ("-f", "--fcheck"):
                if int(arg) < 0:
                    print("\n\nERROR: frequency of checking should be a integer positive number or 0!")
                    raise ValueError
                fcheck = iterations + 1 if int(arg) == 0 else int(arg)
            elif opt in ("-b", "--bcheck"):
                if int(arg) < 0:
                    print("\n\nERROR: Threshold to start checking likelihood should be a integer positive number or 0!")
                    raise ValueError
                bcheck = int(arg)
            elif opt in ("-o", "--out"):
                if not os.path.exists(str(arg)):
                    print("\n\nERROR: The selected path does not exist.")
                    raise ValueError
                outpath = arg
            elif opt in ("-t", "--train"):
                if not os.path.isfile(arg):
                    print("\n\nERROR: The selected file does not exist.")
                    raise ValueError
                train = arg
            elif opt in ("-e", "--test"):
                if not os.path.isfile(arg):
                    print("\n\nERROR: The selected file does not exist.")
                    raise ValueError
                test = arg
            elif opt in ("-k", "--k"):
                if int(arg) < 1:
                    print("\n\nERROR: Number of groups should be a positive integer number different from 0")
                    raise ValueError
                argk = int(arg)
            elif opt == "--seed":
                seed = int(arg)
            elif opt == "--device":
                device = arg
            elif opt == "--save-params":
                save_params = True
    except getopt.GetoptError:
        print("Argument error. Aborting")
        return 2
    except ValueError:
        return 2
    if train is None or test is None:
        print("Argument error. Aborting")
        return 2
    random.seed(os.getpid() if seed is None else seed)
    print("\n*******************************************\n* Digenic Interaction Predictor (B200) *\n"
          "*******************************************\n\nDoing " + str(num_samples) + " samples of " + str(iterations) +
          " num_iterations.\nTrain-file is " + str(train) + "\n Test-file is " + str(test) +
          "\n Output directory is " + str(outpath) + "\nK value (number of groups) is " + str(argk) +
          ".\nLikelihood will be computed every " + str(fcheck) + " num_iterations after iteration number " + str(bcheck))
    model = Model(device=device)
    model.get_train_test(train, test)
    print("\nStarting algorithm...")
    for sample in range(sample_ini, sample_ini + int(num_samples)):
        outfile = outpath + 'Sample_' + str(sample) + '_K' + str(argk) + '.csv'
        if os.path.isfile(outfile):
            continue
        print("Sample " + str(sample) + ":")
        if seed is not None:
            random.seed(seed + sample)
        params = outpath + 'Sample_' + str(sample) + '_K' + str(argk) + '.npz' if save_params else None
        train_sample(model, argk, iterations, fcheck, bcheck, outfile=outfile, params_file=params)
    return 0


if __name__ == "__main__":
    sys.exit(main())
