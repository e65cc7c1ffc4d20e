#!/usr/bin/env python3
"""Drop-in `Model` for AleixMT/TrigenicInteractionPredictor with the numerics on a B200.

Same class surface as the reference's src/TrigenicInteractionPredictor.py (TIP.py:33-1067): same
method names, arguments, attributes, printed messages and error behaviour.  What differs is where
the work happens: links are digested once into int32 arrays and packed on the device, and
make_iteration / compute_likelihood / do_prediction / calculate_test_set_results /
calculate_metrics run as CUDA kernels behind the C ABI in include/tip.h.  Host code keeps only what
must be bit-identical to CPython: gene-id assignment, the string-sorted link key, np.random.shuffle
in fold(), and the random.random() stream of initialize_parameters().

There is no CPU fallback: without libtip.so and a CUDA device the numeric methods raise.

CLI (same flags as TIP.py:1166-1167):
    python -m trigenicinteractionpredictor_b200.TrigenicInteractionPredictor \
        --train train0.dat --test test0.dat --k 10 --num_samples 10 --out results/
"""
from __future__ import annotations

import codecs
import getopt
import math
import os
import random
import re
import sys

import numpy as np

__all__ = ["Model", "SoALinks", "main"]


def _nested(arr: np.ndarray):
    return arr.tolist()


def _is_torch(x) -> bool:
    return type(x).__module__.split(".")[0] == "torch"


class SoALinks:
    """Links handed over already digested (Model.set_links_soa): int32 arrays g1, g2, g3 in key slot order plus the
    counts per rating, behind the read-only part of the dict interface the reference's `links` / `test_links` have
    (len, iteration in order, keys "a_b_c" -> [n0, n1]).  Keys are formatted on demand, never stored: 1e8 links are
    1.6 GB as arrays and would not fit a Python dict."""

    def __init__(self, g1, g2, g3, n0, n1):
        self.g = [x if _is_torch(x) else np.ascontiguousarray(x, dtype=np.int32) for x in (g1, g2, g3)]
        self.n = [x if _is_torch(x) else np.ascontiguousarray(x, dtype=np.int32) for x in (n0, n1)]

    def __len__(self):
        return int(self.g[0].shape[0])

    def _host(self):
        return [x.cpu().numpy() if _is_torch(x) else x for x in self.g + self.n]

    def keys(self):
        a, b, c, _, _ = self._host()
        for i in range(len(self)):
            yield "%d_%d_%d" % (a[i], b[i], c[i])

    __iter__ = keys

    def values(self):
        _, _, _, n0, n1 = self._host()
        for i in range(len(self)):
            yield [int(n0[i]), int(n1[i])]

    def items(self):
        return zip(self.keys(), self.values())

    def count_single_positive(self):
        """#{links with n1 == 1} (TIP.py:588)."""
        n1 = self.n[1]
        return int((n1 == 1).sum())


class Model:
    """State and methods of the MMSBM predictor (TIP.py:33).  `device`/`group`/`flags` are additions:
    the CUDA device to use, a torch.distributed group for link-sharded training, and TIP_EM_* flags."""

    def __init__(self, device=None, group=None, flags: int | None = None):
        # --- reference attributes (TIP.py:39-88) ---
        self.id_gene = {}
        self.gene_id = {}
        self.nlinks = {}
        self.links = {}
        self.test_links = {}
        self.uniqueg = {}
        self.likelihood = 0
        self.heldoutlikelihood = 0
        self.vlikelihood = []
        self.R = 2
        self.K = 0
        self.P = 0
        self.eps = 1e-10
        # --- device plumbing ---
        self._device = device
        self._group = group
        self._flags = flags
        self._engine = None
        self._engine_key = None
        self._links_version = 0          # bumped when links / test_links change
        self._packed_version = -1
        self._theta_host = []            # list[P][K]
        self._pr_host = []               # list[K][K][K][R]
        self._params_on = "host"         # which copy is authoritative: "host" | "device"
        self._host_valid = True          # host lists mirror the device
        self._exposed = False            # a host list was handed out since the last upload
        self._scores = None              # device scores of the test set (test order)
        self._results = []
        self._results_stale = False
        self._deg_zero = None

    # ------------------------------------------------------------------------------------------
    # host mirrors of theta / pr
    # ------------------------------------------------------------------------------------------
    def _pull(self):
        if self._params_on == "device" and not self._host_valid:
            th, pr = self._engine.get_params()
            self._theta_host, self._pr_host = _nested(th), _nested(pr)
            self._host_valid = True

    @property
    def theta(self):
        self._pull()
        self._exposed = True
        if isinstance(self._theta_host, np.ndarray):
            self._theta_host = self._theta_host.tolist()
        return self._theta_host

    @theta.setter
    def theta(self, value):
        self._pull()
        self._theta_host = value
        self._params_on, self._host_valid = "host", True

    @property
    def pr(self):
        self._pull()
        self._exposed = True
        if isinstance(self._pr_host, np.ndarray):
            self._pr_host = self._pr_host.tolist()
        return self._pr_host

    @pr.setter
    def pr(self, value):
        self._pull()
        self._pr_host = value
        self._params_on, self._host_valid = "host", True

    @property
    def ntheta(self):
        """Scratch of the reference; always zero between iterations (TIP.py:1038-1039)."""
        return [[0.0] * self.K for _ in range(self.P)]

    @ntheta.setter
    def ntheta(self, value):
        pass

    @property
    def npr(self):
        return [[[[0.0] * self.R for _ in range(self.K)] for _ in range(self.K)] for _ in range(self.K)]

    @npr.setter
    def npr(self, value):
        pass

    @property
    def results(self):
        if self._results_stale:
            self._build_results()
        return self._results

    @results.setter
    def results(self, value):
        self._results, self._results_stale = value, False

    # ------------------------------------------------------------------------------------------
    # initialisation (host RNG stream must match the reference draw for draw)   TIP.py:106-170
    # ------------------------------------------------------------------------------------------
    def initialize_parameters(self, k_value=10):
        try:
            self.K = int(k_value)
        except ValueError:
            self.K = 10
        self.vlikelihood = []
        K, R = self.K, self.R
        theta, pr = self._draw_parameters_fast(K, R)
        if theta is None:
            theta, pr = self._draw_parameters_loops(K, R)
        self._theta_host, self._pr_host = theta, pr
        self._params_on, self._host_valid, self._exposed = "host", True, False

    def _draw_parameters_loops(self, K, R):
        """The reference's loops, one random.random() per cell (TIP.py:117-170)."""
        rnd = random.random
        # draw order: all theta rows, then p cells in (i, j, k, r) order (TIP.py:117-139)
        theta = [[rnd() for _ in range(K)] for _ in range(self.P)]
        pr = [[[[rnd() for _ in range(R)] for _ in range(K)] for _ in range(K)] for _ in range(K)]
        for g in range(self.P):
            acc = 0.0
            for k in range(K):
                acc += theta[g][k]
            if acc < self.eps:                       # TIP.py:147-149
                theta[g] = [rnd() for _ in range(K)]
            total = sum(theta[g])                    # builtin sum, like TIP.py:151
            row = theta[g]
            for k in range(K):
                try:
                    row[k] /= total
                except ZeroDivisionError:
                    row[k] /= (total + self.eps)
        for plane in pr:
            for line in plane:
                for cell in line:
                    acc = 0.0
                    for r in range(R):
                        acc += cell[r]
                    for r in range(R):
                        try:
                            cell[r] /= acc
                        except ZeroDivisionError:
                            cell[r] /= (acc + self.eps)
        return theta, pr

    def _draw_parameters_fast(self, K, R):
        """The same numbers without a Python call per draw: `random.random()` is MT19937's 53-bit output, exactly what
        numpy's legacy RandomState.random_sample produces from the same state, so the whole block of P*K + K^3*R draws
        is taken from a RandomState seeded with the `random` module's state, and that module's state is then moved to
        where the loops would have left it (consecutive samples continue one stream, TIP.py:1149).  Row totals are the
        builtin sum() of TIP.py:151 restated (compensated since Python 3.12, so not numpy's pairwise sum); divisions are
        elementwise IEEE either way.  Returns arrays (the list mirrors are made when a caller reads theta / pr), or
        (None, None) in the cases the loops treat specially (a row summing to < eps is redrawn, a zero total divides by
        total + eps): the caller then runs the loops from the untouched state.  tests/test_host_model.py holds the two
        paths bit-identical, RNG position included."""
        state = random.getstate()
        if state[0] != 3 or R != 2:
            return None, None
        rs = np.random.RandomState()
        rs.set_state(("MT19937", np.array(state[1][:-1], dtype=np.uint32), state[1][-1], 0, 0.0))
        th = rs.random_sample(self.P * K).reshape(self.P, K)
        pp = rs.random_sample(K * K * K * R).reshape(K, K, K, R)
        # builtin sum() over a row, as CPython >= 3.12 computes it (Neumaier-compensated), all rows at once
        f = np.zeros(self.P)
        c = np.zeros(self.P)
        for k in range(K):
            x = th[:, k]
            t = f + x
            c += np.where(np.abs(f) >= np.abs(x), (f - t) + x, (x - t) + f)
            f = t
        totals = f + c if sys.version_info >= (3, 12) else None
        if totals is None:
            totals = np.array([sum(row) for row in th.tolist()], dtype=np.float64)
        cell_tot = (0.0 + pp[..., 0]) + pp[..., 1]
        # the loops redraw a row whose sequential sum is < eps and divide by total + eps when a total is zero
        if float(totals.min()) < 1e-6 or (cell_tot == 0.0).any():
            return None, None
        ns = rs.get_state()
        random.setstate((3, tuple(int(x) for x in ns[1]) + (int(ns[2]),), state[2]))
        return th / totals[:, None], pp / cell_tot[..., None]

    # ------------------------------------------------------------------------------------------
    # link digestion
    # ------------------------------------------------------------------------------------------
    def _ids_for(self, names, next_id):
        """Dense ids in order of first appearance; every appearance counts in uniqueg (TIP.py:336-349)."""
        out = []
        for name in names:
            gid = self.gene_id.get(name)
            if gid is None:
                gid = next_id
                next_id += 1
                self.gene_id[name] = gid
                self.id_gene[gid] = name
                self.uniqueg[gid] = 0
            self.uniqueg[gid] += 1
            out.append(str(gid))
        return out, next_id

    @staticmethod
    def _bump(table, key, r):
        cell = table.get(key)
        if cell is None:
            cell = table[key] = [0, 0]
        cell[r] += 1

    def get_input(self, argfilename, selectedinteractiontype="trigenic", cutoffvalue=-0.08, discard=0,
                  interactions='ALL'):
        """Digest a raw Kuzmin-2018 table (TIP.py:218-318): 12 columns (S1; column 6 dropped) or 8 (S2)."""
        try:
            next_id = 0
            if selectedinteractiontype not in ('trigenic', 'digenic', '*'):
                raise ValueError("argument 2 selectedInteractionType must be trigenic, digenic or *")
            with codecs.open(argfilename, encoding='utf-8', mode='r') as fh:
                header = re.split(r'\t+', fh.readline())
                raw = len(header) == 12
                for line in fh.readlines():
                    f = re.split(r'\t+', line)
                    if raw:
                        f.pop(5)
                    if selectedinteractiontype != "*" and f[4] != selectedinteractiontype:
                        continue
                    if interactions == 'ALL':
                        r = 1 if (float(f[6]) < 0.05 and float(f[5]) < cutoffvalue) else 0
                    else:
                        if float(f[6]) >= 0.05:
                            continue
                        if float(f[5]) < cutoffvalue:
                            r = 1
                        elif discard:
                            continue
                        else:
                            r = 0
                    names = f[1].split('+')
                    names.append(f[3])
                    ids, next_id = self._ids_for(names, next_id)
                    names.sort()
                    ids.sort()                      # STRING sort of decimal ids (TIP.py:294)
                    self._bump(self.links, '_'.join(ids), r)
                    self._bump(self.nlinks, '_'.join(names), r)
                self.P = len(self.id_gene)
        except ValueError as error:
            print(error)
        except IOError as error:
            print('Error, file does not exist or can\'t be read')
            print(error)
        self._links_version += 1

    def get_traintest(self, trainfile, testfile):
        """Read `name_name_name<TAB>rating` train and test files (TIP.py:321-423)."""
        try:
            next_id = 0
            with codecs.open(trainfile, encoding='utf-8', mode='r') as fh:
                for line in fh.readlines():
                    f = line.strip().split('\t')
                    names = f[0].split('_')
                    r = int(f[1])
                    ids, next_id = self._ids_for(names, next_id)
                    names.sort()
                    ids.sort()
                    self._bump(self.links, '_'.join(ids), r)
                    self._bump(self.nlinks, '_'.join(names), r)
                self.P = len(self.id_gene)
            with codecs.open(testfile, encoding='utf-8', mode='r') as fh:
                for line in fh.readlines():
                    f = re.split(r'\t+', line)
                    names = f[0].split('_')
                    r = int(f[1])
                    ids, next_id = self._ids_for(names, next_id)
                    ids.sort()
                    self._bump(self.test_links, '_'.join(ids), r)
                self.P = len(self.id_gene)
        except ValueError as error:
            print(error)
        except IOError as error:
            print('Error, file does not exist or can\'t be read')
            print(error)
            exit(1)
        self._links_version += 1
        print('READ DATA train', len(self.links), len(self.nlinks))
        print('READ DATA test', len(self.test_links))

    def set_links_soa(self, train, test=None, P=None):
        """Addition (not in the reference): take links that are ALREADY digested - `train` / `test` = (g1, g2, g3, n0, n1)
        int32 arrays (numpy, or torch tensors already on the device) of dense gene ids in the key's slot order (the
        decimal-string order of TIP.py:353) and the counts per rating (TIP.py:361-368).  This is how BASELINE configs
        3 and 4 enter the drop-in: 1e8 triplets cannot pass through the reference's dict of strings.  `links` and
        `test_links` become read-only views with the dict's len / keys / values / items."""
        self.links = SoALinks(*train)
        self.test_links = SoALinks(*test) if test is not None else {}
        if P is None:
            tops = [int(x.max()) for x in self.links.g] + ([int(x.max()) for x in self.test_links.g] if test is not None else [])
            P = max(tops) + 1
        self.P = int(P)
        self.id_gene = {}
        self.gene_id = {}
        self._links_version += 1

    # ------------------------------------------------------------------------------------------
    # 5-fold split (TIP.py:447-523) - bit-exact files, same global numpy stream
    # ------------------------------------------------------------------------------------------
    def fold(self, fraction=0.2):
        per_fold = int(len(self.links) * fraction)
        n_folds = int(1 / fraction)
        order = list(self.links.keys())
        np.random.shuffle(order)                     # legacy global RandomState, like TIP.py:455
        parts = [order[per_fold * i: per_fold * (i + 1)] for i in range(n_folds)]
        parts[n_folds - 1] += order[per_fold * n_folds:]   # remainder joins the last fold

        def text_of(keys):
            chunks = []
            for key in keys:
                rating = 0 if self.links[key][0] else 1
                names = sorted(self.id_gene[int(t)] for t in key.split("_"))
                chunks.append('_'.join(names) + '\t' + str(rating) + '\n')
            return ''.join(chunks)

        for i in range(n_folds):
            with codecs.open('test' + str(i) + '.dat', encoding='utf-8', mode="w+") as fh:
                fh.write(text_of(parts[i]))
        for i in range(n_folds):
            rest = []
            for j in range(n_folds):
                if j != i:
                    rest.extend(parts[j])
            with codecs.open('train' + str(i) + '.dat', encoding='utf-8', mode="w+") as fh:
                fh.write(text_of(rest))

    # ------------------------------------------------------------------------------------------
    # device state
    # ------------------------------------------------------------------------------------------
    @staticmethod
    def _soa(table):
        """dict {"a_b_c": [n0, n1]} (insertion order) -> int32 arrays g1,g2,g3,n0,n1."""
        if isinstance(table, SoALinks):
            return (*table.g, *table.n)
        n = len(table)
        if n == 0:
            z = np.empty(0, dtype=np.int32)
            return z, z.copy(), z.copy(), z.copy(), z.copy()
        # one pass in C instead of a Python loop per link: all keys joined, split once, parsed by numpy
        ids = np.array("_".join(table.keys()).split("_"), dtype=np.int64).astype(np.int32).reshape(n, 3)
        cnt = np.fromiter((c for pair in table.values() for c in pair), dtype=np.int32, count=2 * n).reshape(n, 2)
        return ids[:, 0].copy(), ids[:, 1].copy(), ids[:, 2].copy(), cnt[:, 0].copy(), cnt[:, 1].copy()

    def _ready(self, need_params=True):
        """Make the device copy of links and parameters current; returns the engine."""
        from .engine import EMEngine
        from . import dist as _dist
        key = (self.P, self.K)
        if self._engine is None or self._engine_key != key:
            if self.K < 1 or self.P < 1:
                raise ValueError("initialize_parameters() and link digestion must run before numeric methods")
            self._engine = EMEngine(self.P, self.K, device=self._device, group=self._group, flags=self._flags)
            self._engine_key = key
            self._packed_version = -1
            if self._params_on == "device":          # engine replaced: host copy must be authoritative
                self._params_on = "host"
        eng = self._engine
        if self._packed_version != self._links_version:
            g1, g2, g3, n0, n1 = self._soa(self.links)
            if _is_torch(g1):
                import torch
                deg = torch.bincount(torch.cat([g1, g2, g3]).to(torch.int64), minlength=self.P).to(torch.int32)
            else:
                deg = np.bincount(np.concatenate([g1, g2, g3]), minlength=self.P).astype(np.int32)
            self._deg_zero = bool((deg[: self.P] == 0).any())
            if self._group is not None:
                world, rk = _dist.world_size(self._group), _dist.rank(self._group)
            else:
                world, rk = 1, 0
            lo, hi = _dist.shard_bounds(len(g1), rk, world)
            eng.set_train_links(g1[lo:hi], g2[lo:hi], g3[lo:hi], n0[lo:hi], n1[lo:hi], global_deg=deg)
            eng.set_test_links(*self._soa(self.test_links))
            self._packed_version = self._links_version
        if need_params and (self._params_on == "host" or self._exposed):
            eng.set_params(np.asarray(self._theta_host, dtype=np.float64), np.asarray(self._pr_host, dtype=np.float64))
            self._params_on, self._host_valid, self._exposed = "device", True, False
        return eng

    # ------------------------------------------------------------------------------------------
    # EM iteration, likelihood (TIP.py:984-1043, 952-974)
    # ------------------------------------------------------------------------------------------
    def make_iteration(self):
        eng = self._ready()
        if self._deg_zero:
            # a gene with no training link: the reference divides by float(0) at TIP.py:1018
            raise ZeroDivisionError("float division by zero")
        eng.em_iteration()
        self._host_valid = False

    def make_iterations(self, n):
        """n x make_iteration with the iteration body replayed from a CUDA graph (addition)."""
        eng = self._ready()
        if self._deg_zero:
            raise ZeroDivisionError("float division by zero")
        eng.em_iterations(int(n))
        self._host_valid = False

    def compute_likelihood(self, selected_set='train'):
        eng = self._ready()
        value = eng.loglik('train' if selected_set == 'train' else 'test')
        if selected_set == 'train':
            self.likelihood = value
        else:
            self.heldoutlikelihood = value
        return value

    # ------------------------------------------------------------------------------------------
    # prediction, held-out table, metrics (TIP.py:530-637)
    # ------------------------------------------------------------------------------------------
    def do_prediction(self, id1, id2, id3):
        try:
            a, b, c = int(id1), int(id2), int(id3)
        except ValueError:
            a, b, c = self.gene_id[id1], self.gene_id[id2], self.gene_id[id3]
        import ctypes
        import torch
        from . import _cabi
        eng = self._ready()
        ids = torch.tensor([a, b, c], dtype=torch.int32, device=eng.device)
        out = torch.empty(1, dtype=torch.float64, device=eng.device)
        _cabi.check(eng.lib.tip_score(self.P, self.K, ctypes.c_void_p(ids[0:1].data_ptr()),
                                      ctypes.c_void_p(ids[1:2].data_ptr()), ctypes.c_void_p(ids[2:3].data_ptr()), 1,
                                      ctypes.c_void_p(eng.theta.data_ptr()), ctypes.c_void_p(eng.p.data_ptr()),
                                      ctypes.c_void_p(out.data_ptr()), eng._stream()), "tip_score")
        eng.launches += 1
        return float(out.item())

    def calculate_test_set_results(self):
        eng = self._ready()
        self._scores = eng.scores()
        self._results, self._results_stale = [], True

    def _build_results(self):
        """[[score, "a_b_c", label], ...] sorted descending like list.sort(); reverse() (TIP.py:568-569).  The order
        comes from the device (tip_sort_scores: stable descending radix sort of the fp64 scores); only rows whose scores
        are EQUAL - where the reference's list comparison falls through to the key string and the label - are put in
        their reference order on the host."""
        order, sorted_scores = self._engine.sort_scores(self._scores)
        keys = list(self.test_links.keys())
        labels = [0 if n[0] else 1 for n in self.test_links.values()]
        rows = [[s, keys[i], labels[i]] for s, i in zip(sorted_scores.tolist(), order.tolist())]
        ties = np.flatnonzero(sorted_scores[1:] == sorted_scores[:-1])
        if ties.size:
            starts = ties[np.concatenate([[True], np.diff(ties) > 1])]
            for lo in starts.tolist():
                hi = lo + 1
                while hi < len(rows) and rows[hi][0] == rows[lo][0]:
                    hi += 1
                rows[lo:hi] = sorted(rows[lo:hi], reverse=True)
        self._results, self._results_stale = rows, False

    def calculate_metrics(self):
        n_train = len(self.links)
        if isinstance(self.links, SoALinks):
            hits = self.links.count_single_positive()
        else:
            hits = 0
            for n in self.links.values():
                if n[1] == 1:                        # exactly one positive sighting (TIP.py:588)
                    hits += 1
        positives_fraction = hits / n_train
        positives_number = int(positives_fraction * len(self.test_links))
        if self._scores is None or int(self._scores.numel()) == 0:
            wins = npos = nneg = tp = fp = fn = tn = 0
        else:
            c = self._engine.metric_counts(self._scores, positives_number)
            wins, npos, nneg = c["wins"], c["n_pos"], c["n_neg"]
            tp, fp, fn, tn = c["tp"], c["fp"], c["fn"], c["tn"]
        auc = wins / (npos * nneg)                   # Python int division: same rounding and same
        precision = tp / (tp + fp)                   # ZeroDivisionError as TIP.py:615, 633-635
        recall = tp / (tp + fn)
        fallout = fp / (fp + tn)
        return [precision, recall, fallout, auc]

    # ------------------------------------------------------------------------------------------
    # kept parameters and prediction of unseen triplets (additions: the reference's loader, get_data, opens its file
    # with "w+" and never reads one)
    # ------------------------------------------------------------------------------------------
    def _genes_in_id_order(self):
        return [self.id_gene[i] for i in range(self.P)]

    def save_parameters(self, path):
        """Write theta, pr, K and the gene names in id order to an .npz file at exactly `path`."""
        theta = np.asarray(self.theta, dtype=np.float64)
        pr = np.asarray(self.pr, dtype=np.float64)
        with open(path, "wb") as fh:
            np.savez(fh, theta=theta, pr=pr, K=np.int64(self.K), genes=np.array(self._genes_in_id_order(), dtype=str))

    def check_parameters_file(self, path):
        """(theta [P][K], pr [K][K][K][2]) of an .npz written by save_parameters, checked against this model's digestion:
        the same genes in the same id order, the model's K (when it has one), finite non-negative values.  Raises
        ValueError with the reason otherwise.  Host only."""
        try:
            with np.load(path, allow_pickle=False) as z:
                theta, pr, K, genes = z["theta"], z["pr"], int(z["K"]), [str(g) for g in z["genes"]]
        except (OSError, KeyError, ValueError) as exc:
            raise ValueError("%s is not a parameter file of save_parameters (%s)" % (path, exc)) from exc
        return self._check_parameters(theta, pr, K, genes, str(path))

    def _check_parameters(self, theta, pr, K, genes, what):
        theta = np.asarray(theta, dtype=np.float64)
        pr = np.asarray(pr, dtype=np.float64)
        if genes is not None and genes != self._genes_in_id_order():
            raise ValueError("%s: its gene list (%d genes) differs from the model's digestion (%d genes)"
                             % (what, len(genes), self.P))
        if self.K and K != self.K:
            raise ValueError("%s: K = %d, the model has K = %d" % (what, K, self.K))
        if theta.shape != (self.P, K) or pr.shape != (K, K, K, self.R):
            raise ValueError("%s: theta %s / pr %s do not have the shapes (%d, %d) / (%d, %d, %d, %d)"
                             % (what, theta.shape, pr.shape, self.P, K, K, K, K, self.R))
        if not (np.isfinite(theta).all() and np.isfinite(pr).all()):
            raise ValueError("%s: theta or pr holds a non-finite value" % what)
        if (theta < 0).any() or (pr < 0).any():
            raise ValueError("%s: theta or pr holds a negative value" % what)
        return theta, pr

    def load_parameters(self, path):
        """Make the parameters of an .npz written by save_parameters the model's current theta / pr (see
        check_parameters_file for what is refused)."""
        with np.load(path, allow_pickle=False) as z:
            K = int(z["K"]) if "K" in z.files else 0
        theta, pr = self.check_parameters_file(path)
        self.K = K
        self._theta_host, self._pr_host = theta, pr
        self._params_on, self._host_valid, self._exposed = "host", True, False

    def predict_top_triplets(self, n, genes=None, exclude_known=True, params=None):
        """The `n` most likely interacting triplets of distinct genes among `genes` (names; default all P genes), by
        do_prediction (TIP.py:530-547) of the current theta / pr, or by the mean over the parameter sets in `params`
        (.npz paths of save_parameters or (theta, pr) pairs).  With exclude_known the keys of links and test_links are
        left out.  Exhaustive over C(n_genes, 3) triplets on the device.  Returns [[score, "a_b_c", "nameA_nameB_nameC"],
        ...], best first; equal scores in ascending order of the triplets' positions in the decimal-string order of the
        candidate ids.  The id key is the report's "ID of genes" column; names are sorted as in the fold files (TIP.py:486)."""
        if self.P < 1 or len(self.id_gene) != self.P:
            raise ValueError("predict_top_triplets needs a model digested from train / test files")
        if params is None:
            if self.K < 1:
                raise ValueError("predict_top_triplets: initialize_parameters() or load_parameters() must run first")
            sets = [self._check_parameters(self.theta, self.pr, self.K, None, "the model's parameters")]
        else:
            sets = []
            for item in params:
                if isinstance(item, (str, bytes, os.PathLike)):
                    sets.append(self.check_parameters_file(item))
                else:
                    th, pr = item
                    sets.append(self._check_parameters(th, pr, np.asarray(th).shape[-1], None, "a (theta, pr) pair"))
            if not sets:
                raise ValueError("predict_top_triplets: params is empty")
            Ks = {th.shape[1] for th, _ in sets}
            if len(Ks) != 1:
                raise ValueError("predict_top_triplets: the parameter sets have different K (%s)" % sorted(Ks))
        K = sets[0][0].shape[1]
        if genes is None:
            ids = list(range(self.P))
        else:
            missing = [g for g in genes if g not in self.gene_id]
            if missing:
                raise ValueError("unknown gene names: %s" % ", ".join(missing))
            ids = sorted({self.gene_id[g] for g in genes})
        cand = np.array(sorted(ids, key=str), dtype=np.int32)
        known = np.empty(0, dtype=np.uint64)
        if exclude_known:
            known = self._known_packed(cand)
        from .engine import EMEngine
        eng = self._engine if (self._engine is not None and self._engine_key == (self.P, K)) else None
        if eng is None:
            eng = EMEngine(self.P, K, device=self._device, flags=self._flags)
        out_ids, scores = eng.top_triplets(np.stack([th for th, _ in sets]), np.stack([pr for _, pr in sets]), cand, known, int(n))
        rows = []
        for (a, b, c), s in zip(out_ids.tolist(), scores.tolist()):
            names = sorted((self.id_gene[a], self.id_gene[b], self.id_gene[c]))
            rows.append([s, "%d_%d_%d" % (a, b, c), "_".join(names)])
        return rows

    def _known_packed(self, cand):
        """Sorted packed rank triples (ra << 42 | rb << 21 | rc) of the keys of links and test_links whose three genes
        are all candidates."""
        rank = np.full(self.P, -1, dtype=np.int64)
        rank[cand] = np.arange(cand.shape[0], dtype=np.int64)
        parts = []
        for table in (self.links, self.test_links):
            if len(table) == 0:
                continue
            g = [np.asarray(x.cpu().numpy() if _is_torch(x) else x, dtype=np.int64) for x in self._soa(table)[:3]]
            r = np.stack([rank[g[0]], rank[g[1]], rank[g[2]]], axis=1)
            r = r[(r >= 0).all(axis=1)]
            r.sort(axis=1)
            r = r[(r[:, 0] < r[:, 1]) & (r[:, 1] < r[:, 2])]
            parts.append((r[:, 0] << 42) | (r[:, 1] << 21) | r[:, 2])
        if not parts:
            return np.empty(0, dtype=np.uint64)
        return np.unique(np.concatenate(parts)).astype(np.uint64)

    # ------------------------------------------------------------------------------------------
    # report (TIP.py:793-904)
    # ------------------------------------------------------------------------------------------
    def to_string(self):
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
        return ''.join(out)

    def to_file(self, name_file=None):
        try:
            if name_file is None:
                name_file = "out.txt"
            with codecs.open(name_file, encoding='utf-8', mode="w+") as fh:
                fh.write(self.to_string())
        except IOError:
            print("I/O error")

    # ------------------------------------------------------------------------------------------
    # dataset audit helpers (TIP.py:915-942, 1053-1067) - host-only set differences
    # ------------------------------------------------------------------------------------------
    def compare_links(self, arg_model):
        return [k for k in self.nlinks if k not in arg_model.nlinks]

    def compare_genes(self, arg_model):
        return [g for g in self.gene_id if g not in arg_model.gene_id]

    def compare_dataset(self, arg_model):
        links_ok = not self.compare_links(arg_model)
        print("First dataset is subgraph of second dataset for links" if links_ok
              else "First dataset is not subgraph of second dataset for links")
        genes_ok = not self.compare_genes(arg_model)
        print("First dataset is subgraph of second dataset for nodes" if genes_ok
              else "First dataset is not subgraph of second dataset for nodes")
        return int(genes_ok) and int(links_ok)


# ----------------------------------------------------------------------------------------------
# command line: same flags, defaults, file naming, skip-if-exists and convergence rule as
# TIP.py:1148-1279.  Additions: --seed (instead of os.getpid()), --device, --dist samples|links, --reducible (append the
# gene list block so that the sample files feed testResultsReducer directly),
# --mode auto|slots|fp64|segmented|fp32 (E-step formulation: slot-segmented 4K^2 per link without per-link atomics - the
# default for K >= 4 -, K^3 per link, gene-segmented 2K^2 per link - all the same results to rounding -, or
# fp32-compute / fp64-accumulate within 1e-5), --save-params (write Sample_{s}_K{k}.npz, the trained theta / pr, next to each
# report written; `python -m trigenicinteractionpredictor_b200.predict` ranks unseen triplets with them).
# ----------------------------------------------------------------------------------------------
def train_sample(model, k, iterations, fcheck, bcheck, outfile=None, verbose=True, log=print, reducible=False,
                 params_file=None):
    """One random restart (TIP.py:1260-1279).  Returns (converged, iterations_done, checks).  reducible: append the
    LIST OF REGISTERED GENES block (TIP.py:863-867, commented out in the reference) that testResultsReducer parses.
    params_file: where the report is written, also write the trained parameters there (Model.save_parameters)."""
    model.initialize_parameters(k)
    if verbose:
        log("Parameters have been initialized")
    like0 = model.compute_likelihood()
    if verbose:
        log("· Initial Likelihood is " + str(like0))
    checks = [like0]
    it = 0
    while it < iterations:
        # iterations between two likelihood checks run back to back on the device
        nxt = it
        while nxt < iterations and not (nxt % fcheck == 0 and nxt > bcheck):
            nxt += 1
        run = min(nxt, iterations - 1) - it + 1
        model.make_iterations(run)
        it += run
        last = it - 1
        if last % fcheck == 0 and last > bcheck:
            like = model.compute_likelihood()
            checks.append(like)
            if verbose:
                log("· Likelihood " + str(last + 1) + " is " + str(like))
            if math.fabs((like - like0) / like0) < 0.01:
                if verbose:
                    log("\n\t**************************\n\t* Likelihood has converged *\n\t**************************")
                if outfile is not None:
                    model.to_file(outfile)
                    if reducible:
                        from .testResultsReducer import gene_list_block
                        with codecs.open(outfile, encoding='utf-8', mode="a") as fh:
                            fh.write(gene_list_block(model))
                    if params_file is not None:
                        model.save_parameters(params_file)
                return True, it, checks
            like0 = like
    return False, it, checks


def main(argv=None):
    argv = sys.argv[1:] if argv is None else argv
    iterations, num_samples, sample_ini, fcheck, bcheck = 10000, 100, 0, 25, 100
    train = test = None
    outpath, argk = "", 1
    seed, device, dist_mode, mode_flags, reducible, save_params = None, None, "none", None, False, False
    try:
        opts, _ = getopt.getopt(argv, "hi:n:s:f:b:o:t:e:k:",
                                ["help", "num_iterations=", "num_samples=", "sample_ini=", "fcheck=", "bcheck=",
                                 "out=", "train=", "test=", "k=", "seed=", "device=", "dist=", "mode=", "reducible",
                                 "save-params"])
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
                fcheck = iterations + 1 if int(arg) == 0 else int(arg)   # order-dependent, as in TIP.py:1192-1193
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
            elif opt == "--dist":
                if arg not in ("none", "samples", "links"):
                    raise ValueError
                dist_mode = arg
            elif opt == "--reducible":
                reducible = True
            elif opt == "--save-params":
                save_params = True
            elif opt == "--mode":
                if arg not in ("auto", "slots", "fp64", "segmented", "fp32"):
                    raise ValueError
                mode_flags = {"auto": None, "slots": 32, "fp64": 0, "segmented": 8, "fp32": 2}[arg]   # TIP_EM_* of include/tip.h
    except getopt.GetoptError:
        print("Argument error. Aborting")
        return 2
    except ValueError:
        return 2
    if train is None or test is None:
        print("Argument error. Aborting")
        return 2

    from . import dist as _dist
    rk, world, local = (0, 1, 0)
    if dist_mode != "none":
        rk, world, local = _dist.init_from_env()
        if device is None:
            device = "cuda:%d" % local
    if seed is None and dist_mode == "links":
        # link shards are replicas of ONE model: every rank must draw the same initial theta / p (TIP.py:1149 seeds
        # with the pid, which differs per rank) - rank 0's pid is the seed of the whole job
        seed_all = _dist.broadcast_int(os.getpid())
        random.seed(seed_all)
    else:
        random.seed(os.getpid() if seed is None else seed)

    print("\n****************************************\n* Trigenic Interaction Predictor (B200) *\n"
          "****************************************\n\nDoing " + str(num_samples) + " samples of " + str(iterations) +
          " num_iterations.\nTrain-file is " + str(train) + "\n Test-file is " + str(test) +
          "\n Output directory is " + str(outpath) + "\nK value (number of groups) is " + str(argk) +
          ".\nLikelihood will be computed every " + str(fcheck) + " num_iterations after iteration number " + str(bcheck))

    model = Model(device=device, group=None if dist_mode != "links" else _dist.td.group.WORLD, flags=mode_flags)
    model.get_traintest(train, test)
    print("\nStarting algorithm...")
    samples = range(sample_ini, sample_ini + int(num_samples))
    if dist_mode == "samples":
        samples = _dist.samples_for_rank(sample_ini, int(num_samples), rk, world)
    for sample in samples:
        outfile = outpath + 'Sample_' + str(sample) + '_K' + str(argk) + '.csv'
        if os.path.isfile(outfile):                  # resume-by-skip (TIP.py:1256-1257)
            continue
        print("Sample " + str(sample) + ":")
        if seed is not None:
            random.seed(seed + sample)
        write = outfile if (dist_mode != "links" or rk == 0) else None
        params = outpath + 'Sample_' + str(sample) + '_K' + str(argk) + '.npz' if (save_params and write) else None
        train_sample(model, argk, iterations, fcheck, bcheck, outfile=write, reducible=reducible, params_file=params)
    return 0


if __name__ == "__main__":
    sys.exit(main())
