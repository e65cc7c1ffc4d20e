"""The prediction, ranking and gene-pair kernels of tip_predict.cu at the sizes their limits accept, against an exact
reference that needs no enumeration of the universe.

Every entry point accepts n_cand <= 2^21 and packs ranks into 21-bit fields; the other test files stop at n = 1 500,
where no rank has more than 11 bits, no shared 32-bit histogram bin comes near its flush and no universe passes 2^32.
The problems here are planted so that the exact answer at any n is cheap:

* dead genes: almost every candidate has a theta row of exact zeros in every set, so every triplet or pair that holds one
  scores exactly +0.0 whatever the contraction order;
* live genes: a few hundred candidates, placed at chosen ranks (0, 1, n - 2, n - 1, ranks with the top bits set), have
  dyadic rows (multiples of 2^-3 in [0, 1], none all zero) and p, q entries are multiples of 2^-4 in (0, 1], so every
  product and partial sum is an integer multiple of 2^-13 (triplets) or 2^-10 (pairs) far below 2^53: the reference
  scores the live triplets in int64 and every summation order gives the same bits;
* ties at zero in closed form: past the positive scores the order is the packed key (or the partner's rank), so top-N rows
  come from a generator of the smallest keys that are neither live nor known, a rank from the positives ahead plus a
  count of the zero keys below it (`count_below`, O(n) per query), and the histogram's zero bin from C(n, 3).

Ranks are positions in the decimal-string order of the ids, so at n = 2^21 most ids differ from their ranks and the
id <-> rank mapping is exercised at high ids.  Where the universe of a query is O(n) (per pair, digenic per gene) a
random-parameter case at full n is also compared with an exhaustive NumPy reference, tie-aware to 1e-12.

The reference is pinned without a GPU at n <= 40 against the exhaustive oracles of the other test files.
SCALE_COVERAGE maps every kernel of tip_predict.cu to the test here that runs it at scale, or to why it is left out.
"""
import itertools
from math import comb

import numpy as np
import pytest

from tests.test_digenic_predict import pack2, per_gene_np, top_pairs_np
from tests.test_kernel_coverage import CSRC, _kernels_in
from tests.test_predict import check_against_oracle, pack_ranks, top_triplets_np
from tests.test_rank_per_gene import gene_oracle
from tests.test_rank_per_pair import pair_oracle

M21 = np.uint64((1 << 21) - 1)
TH_UNIT, P_UNIT = 8, 16            # theta entries are multiples of 1/8, p and q entries of 1/16
TRIPLET_ULP = 2.0 ** -13           # theta^3 p
PAIR_ULP = 2.0 ** -10              # theta^2 q
MAX_N = 1 << 21

# ---------------------------------------------------------------------------------------------------------------------
# coverage: every __global__ kernel of tip_predict.cu -> the tests here that run it at scale, or why it is left out
# ---------------------------------------------------------------------------------------------------------------------
_TT = ["test_top_triplets_past_the_shared_bin_flush", "test_top_triplets_known_keys_at_2_22"]
_PG = ["test_top_triplets_per_gene_universe_past_2_33", "test_top_triplets_per_gene_at_2_21",
       "test_top_triplets_per_gene_buffers_at_2_24"]
_PP = ["test_top_triplets_per_pair_at_2_21", "test_top_triplets_per_pair_buffers_at_2_24"]
_RP = ["test_rank_per_pair_at_2_21", "test_rank_per_pair_2_22_pairs_2_26_known"]
_RG = ["test_rank_per_gene_past_2_32", "test_rank_per_gene_at_2_21"]
_TP = ["test_top_pairs_past_4000_chunks", "test_top_pairs_ranks_past_2_20"]
_GP = ["test_top_pairs_per_gene_at_2_21", "test_top_pairs_per_gene_buffers_at_2_24"]
SCALE_COVERAGE = {
    "tip_predict_prep_kernel": _TT + ["test_score_histogram_total_past_2_42"],
    "tip_predict_sample_kernel": _TT,
    "tip_predict_pass_kernel": _TT,
    "tip_predict_finish_kernel": _TT,
    "tip_query_prep_kernel": _PG + _PP + _RP + _RG,
    "tip_query_rowsum_kernel": _PG + _PP + ["test_score_histogram_total_past_2_42"],
    "tip_query_bound_kernel": _PG,
    "tip_query_sample_kernel": _PG,
    "tip_query_pass_kernel": _PG,
    "tip_query_finish_kernel": _PG,
    "tip_pair_keys_kernel": _PP + _RP,
    "tip_pair_split_kernel": _PP + _RP,
    "tip_pair_known_kernel": _PP,
    "tip_pair_vec_kernel": _PP + _RP,
    "tip_pair_init_kernel": _PP,
    "tip_pair_pass_kernel": _PP,
    "tip_pair_segments_kernel": _PP,
    "tip_pair_finish_kernel": _PP,
    "tip_hist_bound_kernel": ["test_score_histogram_total_past_2_42"],
    "tip_hist_pass_kernel": ["test_score_histogram_total_past_2_42"],
    "tip_rank_inverse_kernel": _RP,
    "tip_rank_test_keys_kernel": _RP,
    "tip_rank_train_kernel": _RP,
    "tip_rank_rows_kernel": _RP,
    "tip_rank_iota_kernel": _RP + _RG,
    "tip_rank_pass_kernel": _RP,
    "tip_rank_finish_kernel": _RP,
    "tip_gene_rank_pass_kernel": _RG,
    "tip_gene_test_keys_kernel": _RG,
    "tip_gene_train_kernel": _RG,
    "tip_gene_offsets_kernel": _RG,
    "tip_gene_items_kernel": _RG,
    "tip_gene_flags_kernel": _RG,
    "tip_gene_compact_kernel": _RG,
    "tip_gene_universe_kernel": _RG,
    "tip_gene_finish_kernel": _RG,
    "tip_pair_prep_kernel": _TP + _GP,
    "tip_top_pairs_pass_kernel": _TP,
    "tip_top_pairs_finish_kernel": _TP,
    "tip_top_pairs_gene_kernel": _GP,
    "tip_top_pairs_gene_finish_kernel": _GP,
    "tip_pair_offsets_kernel": _GP,
    "tip_score_pairs_kernel": ["test_score_pairs_at_high_ids"],
}
SCALE_LEFT_OUT = {}


def test_every_predict_kernel_has_a_scale_row():
    kernels = _kernels_in(CSRC + "/tip_predict.cu")
    rows = set(SCALE_COVERAGE) | set(SCALE_LEFT_OUT)
    problems = ["%s has no row" % k for k in sorted(kernels - rows)]
    problems += ["the row %s names no kernel" % k for k in sorted(rows - kernels)]
    for k, tests in SCALE_COVERAGE.items():
        problems += ["%s names a missing test %s" % (k, t) for t in tests if not callable(globals().get(t))]
    assert not problems, "; ".join(problems)


# ---------------------------------------------------------------------------------------------------------------------
# the planted problem and its exact reference
# ---------------------------------------------------------------------------------------------------------------------
def cand_of(n):
    """ids 0 .. n-1 in decimal-string order: cand[rank] = id"""
    return np.array(sorted(range(n), key=str), dtype=np.int32)


def unpack(k):
    k = np.asarray(k, dtype=np.uint64)
    return np.stack([(k >> np.uint64(42)) & M21, (k >> np.uint64(21)) & M21, k & M21], 1).astype(np.int64)


def in_sorted(sorted_keys, x):
    x = np.asarray(x, dtype=np.uint64)
    if len(sorted_keys) == 0:
        return np.zeros(x.shape, dtype=bool)
    i = np.searchsorted(sorted_keys, x).clip(max=len(sorted_keys) - 1)
    return sorted_keys[i] == x


class Planted:
    """n candidates, ids 0 .. n-1 ranked in decimal-string order; the ranks `live` have dyadic theta rows (integers
    `ti` / 8), every other row is zero; p[..., 1] = pi / 16 and q[..., 1] = qi / 16 with pi, qi in 1 .. 16."""

    def __init__(self, n, live, K, S, seed):
        rng = np.random.default_rng(seed)
        self.n, self.K, self.S = n, K, S
        self.cand = cand_of(n)
        self.live = np.unique(np.asarray(live, dtype=np.int64))
        L = len(self.live)
        ti = rng.integers(0, TH_UNIT + 1, size=(S, L, K))
        ti[ti.sum(axis=2) == 0, 0] = 1 + rng.integers(0, TH_UNIT)
        self.ti = ti.astype(np.int64)
        self.pi = rng.integers(1, P_UNIT + 1, size=(S, K, K, K)).astype(np.int64)
        self.qi = rng.integers(1, P_UNIT + 1, size=(S, K, K)).astype(np.int64)
        self.is_live = np.zeros(n, dtype=bool)
        self.is_live[self.live] = True
        self.lpos = np.full(n, -1, dtype=np.int64)
        self.lpos[self.live] = np.arange(L)
        self._live_triplets = None

    # ---- parameters as the kernels take them
    def thetas(self):
        th = np.zeros((self.S, self.n, self.K))
        th[:, self.cand[self.live]] = self.ti / TH_UNIT
        return th

    def prs(self):
        p1 = self.pi / P_UNIT
        return np.stack([1.0 - p1, p1], axis=-1)

    def qs(self):
        q1 = self.qi / P_UNIT
        return np.stack([1.0 - q1, q1], axis=-1)

    # ---- exact integer scores (sum over the sets, in units of TRIPLET_ULP / PAIR_ULP)
    def _rows(self, r):
        r = np.asarray(r, dtype=np.int64)
        out = np.zeros((self.S, len(r), self.K), dtype=np.int64)
        live = self.is_live[r]
        out[:, live] = self.ti[:, self.lpos[r[live]]]
        return out

    def triplet_int(self, tri):
        """integer score sums of rank triples [m][3] in slot order"""
        tri = np.asarray(tri, dtype=np.int64).reshape(-1, 3)
        a, b, c = (self._rows(tri[:, i]) for i in range(3))
        return np.einsum("six,siy,siz,sxyz->i", a, b, c, self.pi)

    def pair_int(self, ra, rb):
        """integer score sums of rank pairs, ra in the first slot"""
        return np.einsum("six,siy,sxy->i", self._rows(ra), self._rows(rb), self.qi)

    def live_triplets(self):
        """(packed keys ascending, integer score sums) of every triplet of live ranks"""
        if self._live_triplets is None:
            L = len(self.live)
            keys, scs = [], []
            for j in range(1, L - 1):
                W = np.einsum("sy,sxyz->sxz", self.ti[:, j], self.pi)
                Q = np.einsum("sax,sxz->asz", self.ti[:, :j], W)
                s = np.einsum("asz,scz->ac", Q, self.ti[:, j + 1:])
                A, C = np.meshgrid(np.arange(j), np.arange(j + 1, L), indexing="ij")
                keys.append(pack_ranks(self.live[A.ravel()], np.full(A.size, self.live[j]), self.live[C.ravel()]))
                scs.append(s.ravel())
            k = np.concatenate(keys) if keys else np.empty(0, np.uint64)
            s = np.concatenate(scs) if scs else np.empty(0, np.int64)
            o = np.argsort(k)
            self._live_triplets = (k[o], s[o])
        return self._live_triplets

    def live_triplets_of(self, r):
        """(keys, integer sums) of the live triplets that contain rank r"""
        k, s = self.live_triplets()
        if not self.is_live[r]:
            return k[:0], s[:0]
        has = (unpack(k) == r).any(axis=1)
        return k[has], s[has]

    def ids(self, keys):
        return self.cand[unpack(keys)]


def best_first(keys, s):
    """(-s, key) order"""
    o = np.lexsort((keys, -s))
    return keys[o], s[o]


def zero_keys(prob, blocks, known, need):
    """the first `need` keys of `blocks` (rank triples in ascending key order) that are neither live nor known"""
    out, got = [], 0
    for a, b, c in blocks:
        if got >= need:
            break
        a, b, c = np.broadcast_arrays(a, b, c)
        k = pack_ranks(a, b, c)
        keep = ~(prob.is_live[a] & prob.is_live[b] & prob.is_live[c]) & ~in_sorted(known, k)
        k = k[keep][:need - got]
        out.append(k)
        got += len(k)
    return np.concatenate(out) if out else np.empty(0, np.uint64)


def all_blocks(n):
    for a in range(n - 2):
        for b in range(a + 1, n - 1):
            yield a, b, np.arange(b + 1, n)


def gene_blocks(n, r):
    """the rank triples that contain r, in key order"""
    for a in range(r):
        yield a, np.arange(a + 1, r), r
        yield a, r, np.arange(r + 1, n)
    for b in range(r + 1, n - 1):
        yield r, b, np.arange(b + 1, n)


def ref_top(prob, known, N):
    """(keys, integer sums) of tip_top_triplets' first N rows"""
    k, s = prob.live_triplets()
    keep = ~in_sorted(known, k)
    k, s = best_first(k[keep], s[keep])
    if N <= len(k):
        return k[:N], s[:N]
    z = zero_keys(prob, all_blocks(prob.n), known, N - len(k))
    return np.concatenate([k, z]), np.concatenate([s, np.zeros(len(z), np.int64)])


def ref_top_gene(prob, r, known, N):
    """(keys, integer sums) of the first N rows of query rank r"""
    k, s = prob.live_triplets_of(r)
    keep = ~in_sorted(known, k)
    k, s = best_first(k[keep], s[keep])
    if N <= len(k):
        return k[:N], s[:N]
    z = zero_keys(prob, gene_blocks(prob.n, r), known, N - len(k))
    return np.concatenate([k, z]), np.concatenate([s, np.zeros(len(z), np.int64)])


def pair_partners(prob, ra, rb, known):
    """every partner rank of the pair, its triplet key, integer sum and whether it is unseen, in rank order"""
    n = prob.n
    c = np.arange(n)
    c = c[(c != ra) & (c != rb)]
    tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
    keys = pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2])
    s = np.zeros(len(c), np.int64)
    live = prob.is_live[c] & prob.is_live[ra] & prob.is_live[rb]
    s[live] = prob.triplet_int(tri[live])
    return c, keys, s, ~in_sorted(known, keys)


def ref_top_pair(prob, ra, rb, known, N):
    """(partner ranks, integer sums) of the first N rows of the pair: score descending, partner rank ascending"""
    c, _, s, unseen = pair_partners(prob, ra, rb, known)
    c, s = c[unseen], s[unseen]
    o = np.lexsort((c, -s))[:N]
    return c[o], s[o]


def ref_rank_pair(prob, ra, rb, known, rcs):
    """(ranks, integer sums, universe) of test partners rcs of the pair; rank 0 for a known triplet"""
    c, keys, s, unseen = pair_partners(prob, ra, rb, known)
    cu, su = c[unseen], s[unseen]
    o = np.lexsort((cu, -su))
    pos = np.zeros(prob.n, np.int64)
    pos[cu[o]] = np.arange(1, len(o) + 1)
    rcs = np.asarray(rcs, dtype=np.int64)
    tri = np.sort(np.stack([np.full(len(rcs), ra), np.full(len(rcs), rb), rcs], 1), 1)
    return pos[rcs], prob.triplet_int(tri), int(unseen.sum())


def count_below(n, r, t):
    """number of rank triples (slot order) that contain r and whose key is below the triple t = (a, b, c)"""
    a, b, c = (int(x) for x in t)
    x = np.arange(n, dtype=np.int64)
    lo, hi = x[x < r], x[x > r]
    cnt = 0
    # x < r, y in (x, r): (x, y, r)
    cnt += int((r - lo[lo < a] - 1).sum())
    if a < r:
        cnt += max(0, min(b, r) - a - 1) + int(a < b < r and r < c)
    # x < r, y > r: (x, r, y)
    cnt += (n - r - 1) * int((lo < a).sum())
    if a < r:
        cnt += (n - r - 1) if r < b else (max(0, c - r - 1) if r == b else 0)
    # x > r: (r, x, y), y > x
    if r < a:
        cnt += int((n - hi - 1).sum())
    elif r == a:
        cnt += int((n - hi[hi < b] - 1).sum())
        if b > r:
            cnt += max(0, c - b - 1)
    return cnt


def ref_rank_gene(prob, r, known, tests):
    """(ranks, integer sums, universe) of test pairs (u, v) of query rank r; rank 0 for a known triplet"""
    kk = np.asarray(known, dtype=np.uint64)
    kr = kk[(unpack(kk) == r).any(axis=1)] if len(kk) else kk
    universe = comb(prob.n - 1, 2) - len(kr)
    lk, ls = prob.live_triplets_of(r)
    unseen = ~in_sorted(kr, lk)
    pk, ps = lk[unseen], ls[unseen]
    kr_zero = kr[~in_sorted(lk, kr)]
    ranks, sums = [], []
    for u, v in tests:
        t = sorted((r, int(u), int(v)))
        key = (t[0] << 42) | (t[1] << 21) | t[2]
        s = int(prob.triplet_int([t])[0])
        sums.append(s)
        if in_sorted(kr, [key])[0]:
            ranks.append(0)
        elif s > 0:
            ranks.append(1 + int(((ps > s) | ((ps == s) & (pk < np.uint64(key)))).sum()))
        else:
            ranks.append(len(pk) + count_below(prob.n, r, t) - int((lk < np.uint64(key)).sum())
                         - int((kr_zero < np.uint64(key)).sum()) + 1)
    return np.array(ranks, dtype=np.int64), np.array(sums, dtype=np.int64), universe


def ref_histogram(prob, layout):
    """counts of tip_score_histogram: the live sums by the host bin function, the rest at zero"""
    _, s = prob.live_triplets()
    h = np.bincount(layout.bins(s * TRIPLET_ULP), minlength=layout.n_bins).astype(np.int64)
    h[layout.bins(np.zeros(1))[0]] += comb(prob.n, 3) - len(s)
    return h


def live_pairs(prob):
    """(packed pairs ascending, integer sums) of every pair of live ranks"""
    i, j = np.triu_indices(len(prob.live), 1)
    ra, rb = prob.live[i], prob.live[j]
    return pack2(ra, rb), prob.pair_int(ra, rb)


def ref_top_pairs(prob, known, N):
    k, s = live_pairs(prob)
    keep = ~in_sorted(known, k)
    k, s = best_first(k[keep], s[keep])
    if N <= len(k):
        return k[:N], s[:N]
    out, got = [k], len(k)
    for a in range(prob.n - 1):
        if got >= N:
            break
        b = np.arange(a + 1, prob.n)
        z = pack2(np.full(len(b), a), b)
        z = z[~(prob.is_live[a] & prob.is_live[b]) & ~in_sorted(known, z)][:N - got]
        out.append(z)
        got += len(z)
    z = np.concatenate(out)
    return z, np.concatenate([s, np.zeros(len(z) - len(s), np.int64)])


def ref_top_pairs_gene(prob, r, known, N):
    """(partner ranks, integer sums) of the first N pairs of query rank r: sum descending, partner rank ascending"""
    x = np.arange(prob.n)
    x = x[x != r]
    lo, hi = np.minimum(x, r), np.maximum(x, r)
    keep = ~in_sorted(known, pack2(lo, hi))
    x, lo, hi = x[keep], lo[keep], hi[keep]
    s = np.zeros(len(x), np.int64)
    live = prob.is_live[x] & prob.is_live[r]
    s[live] = prob.pair_int(lo[live], hi[live])
    o = np.lexsort((x, -s))[:N]
    return x[o], s[o]


def unpack2(k):
    k = np.asarray(k, dtype=np.uint64)
    return np.stack([k >> np.uint64(21), k & M21], 1).astype(np.int64)


def bits(x):
    return np.ascontiguousarray(x, dtype=np.float64).view(np.uint64)


def small_problem(n, S, seed):
    live = sorted({0, 1, n - 2, n - 1} | set(np.random.default_rng(seed).choice(n, size=n // 3, replace=False).tolist()))
    return Planted(n, live, 2, S, seed)


def small_known(prob, rng):
    """some live triplets and some of the first zero keys"""
    k, _ = prob.live_triplets()
    z = zero_keys(prob, all_blocks(prob.n), np.empty(0, np.uint64), 40)
    return np.unique(np.concatenate([rng.choice(k, size=len(k) // 4, replace=False), z[::3],
                                     pack_ranks([0], [prob.n - 2], [prob.n - 1])]))


# ---------------------------------------------------------------------------------------------------------------------
# the reference pinned to the exhaustive oracles (no GPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("S", [1, 2, 4])
def test_dyadic_scores_are_the_same_bits_in_two_orders(S):
    prob = small_problem(40, S, 3 + S)
    th, pr = prob.thetas(), prob.prs()
    k, si = prob.live_triplets()
    g = prob.cand[unpack(k)]
    # (th_a . W_b) . th_c with W_b = th_b . p, summed over the sets last, against the plain sum over x, y, z, s reversed
    first = np.zeros(len(k))
    for s in range(S):
        W = np.einsum("iy,xyz->ixz", th[s][g[:, 1]], pr[s][..., 1])
        first += np.einsum("ix,ixz,iz->i", th[s][g[:, 0]], W, th[s][g[:, 2]])
    second = np.zeros(len(k))
    for s in reversed(range(S)):
        for z, y, x in itertools.product(reversed(range(2)), repeat=3):
            second += th[s][g[:, 2], z] * th[s][g[:, 1], y] * th[s][g[:, 0], x] * pr[s][x, y, z, 1]
    assert np.array_equal(bits(first), bits(second))
    assert np.array_equal(bits(first), bits(si * TRIPLET_ULP))
    assert np.all(si > 0) and len(si) == comb(len(prob.live), 3)


@pytest.mark.parametrize("S", [1, 2])
def test_reference_top_rows_and_histogram_against_the_oracle(S):
    from trigenicinteractionpredictor_b200.engine import BinLayout
    rng = np.random.default_rng(50 + S)
    prob = small_problem(40, S, 10 + S)
    known = small_known(prob, rng)
    total = comb(prob.n, 3)
    o_ids, o_sc, o_k = top_triplets_np(prob.thetas(), prob.prs(), prob.cand, known, total)
    for N in (1, 7, len(prob.live_triplets()[0]) - 3, total - len(known), total):
        k, s = ref_top(prob, known, N)
        assert np.array_equal(k, o_k[:N]) and np.array_equal(bits(s * TRIPLET_ULP / S), bits(o_sc[:N]))
    _, sums, _ = top_triplets_np(prob.thetas(), prob.prs(), prob.cand, [], total)
    sums = sums * S
    for top in (0, 2, 5):
        layout = BinLayout(3, 8, 1023 + top)
        want = np.bincount(layout.bins(sums), minlength=layout.n_bins)
        got = ref_histogram(prob, layout)
        assert np.array_equal(got, want) and got.sum() == total


@pytest.mark.parametrize("S", [1, 2])
def test_reference_per_gene_and_per_pair_rows_against_the_oracle(S):
    rng = np.random.default_rng(60 + S)
    prob = small_problem(37, S, 20 + S)
    n = prob.n
    known = small_known(prob, rng)
    o_ids, o_sc, o_k = top_triplets_np(prob.thetas(), prob.prs(), prob.cand, known, comb(n, 3))
    o_r = unpack(o_k)
    dead = int(np.flatnonzero(~prob.is_live)[0])
    for r in (0, 1, int(prob.live[len(prob.live) // 2]), dead, n - 2, n - 1):
        has = (o_r == r).any(axis=1)
        for N in (3, int(has.sum()), int(has.sum()) + 4):
            k, s = ref_top_gene(prob, r, known, N)
            assert np.array_equal(k, o_k[has][:N]) and np.array_equal(bits(s * TRIPLET_ULP / S), bits(o_sc[has][:N]))
    for ra, rb in ((0, n - 1), (n - 2, n - 1), (0, 1), (0, dead), (dead, n - 1)):
        has = (o_r == ra).any(axis=1) & (o_r == rb).any(axis=1)
        want_c = o_r[has].sum(axis=1) - ra - rb
        c, s = ref_top_pair(prob, ra, rb, known, n)
        assert np.array_equal(c, want_c) and np.array_equal(bits(s * TRIPLET_ULP / S), bits(o_sc[has]))


def test_count_below_against_enumeration():
    n = 13
    for r in range(n):
        triples = sorted(tuple(sorted((r, x, y))) for x, y in itertools.combinations([i for i in range(n) if i != r], 2))
        for i, t in enumerate(triples):
            assert count_below(n, r, t) == i, (r, t)
        for t in itertools.combinations(range(n), 3):          # keys of other triples too
            assert count_below(n, r, t) == sum(u < t for u in triples), (r, t)
    assert count_below(n, 0, (0, 1, 2)) == 0 and count_below(n, n - 1, (n - 3, n - 2, n - 1)) == comb(n - 1, 2) - 1


@pytest.mark.parametrize("S", [1, 2])
def test_reference_ranks_against_the_oracles(S):
    rng = np.random.default_rng(70 + S)
    prob = small_problem(31, S, 30 + S)
    n = prob.n
    known = small_known(prob, rng)
    th, pr = prob.thetas(), prob.prs()
    dead = int(np.flatnonzero(~prob.is_live)[0])
    for r in (0, int(prob.live[3]), dead, n - 1):
        packed, s = gene_oracle(th, pr, prob.cand, known, r)
        others = [x for x in range(n) if x != r]
        tests = list(itertools.combinations(others, 2))
        rank, sums, universe = ref_rank_gene(prob, r, known, tests)
        assert universe == len(packed)
        where = {int(x): i for i, x in enumerate(packed.tolist())}
        for (u, v), rk, sm in zip(tests, rank.tolist(), sums.tolist()):
            t = sorted((r, u, v))
            key = (t[0] << 42) | (t[1] << 21) | t[2]
            if key in where:
                assert rk == where[key] + 1 and sm * TRIPLET_ULP / S == s[where[key]]
            else:
                assert rk == 0 and key in set(known.tolist())
    for ra, rb in ((0, n - 1), (n - 2, n - 1), (int(prob.live[2]), int(prob.live[5])), (dead, n - 1)):
        c, s = pair_oracle(th, pr, prob.cand, known, ra, rb)
        rcs = [x for x in range(n) if x not in (ra, rb)]
        rank, sums, universe = ref_rank_pair(prob, ra, rb, known, rcs)
        assert universe == len(c)
        where = {int(x): i for i, x in enumerate(c.tolist())}
        for x, rk, sm in zip(rcs, rank.tolist(), sums.tolist()):
            assert rk == (where[x] + 1 if x in where else 0)
            if x in where:
                assert sm * TRIPLET_ULP / S == s[where[x]]


@pytest.mark.parametrize("S", [1, 2])
def test_reference_pairs_against_the_oracle(S):
    rng = np.random.default_rng(80 + S)
    prob = small_problem(38, S, 40 + S)
    n = prob.n
    th, qs = prob.thetas(), prob.qs()
    lk, _ = live_pairs(prob)
    z = pack2(np.zeros(5, np.int64), np.arange(1, 6))
    known = np.unique(np.concatenate([rng.choice(lk, size=len(lk) // 4, replace=False), z, pack2([n - 2], [n - 1])]))
    total = comb(n, 2)
    o_ids, o_sc, o_k = top_pairs_np(th, qs, prob.cand, known, total)
    for N in (1, len(lk) - 2, total):
        k, s = ref_top_pairs(prob, known, N)
        assert np.array_equal(k, o_k[:N]) and np.array_equal(bits(s * PAIR_ULP / S), bits(o_sc[:N]))
    dead = int(np.flatnonzero(~prob.is_live)[0])
    for r in (0, dead, int(prob.live[4]), n - 1):
        o_ids, o_sc = per_gene_np(th, qs, prob.cand, known, r, n)
        x, s = ref_top_pairs_gene(prob, r, known, n)
        lo, hi = np.minimum(x, r), np.maximum(x, r)
        assert np.array_equal(prob.cand[np.stack([lo, hi], 1)], o_ids)
        assert np.array_equal(bits(s * PAIR_ULP / S), bits(o_sc))


# ---------------------------------------------------------------------------------------------------------------------
# GPU cases
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch


def need_memory(torch, gib):
    free, _ = torch.cuda.mem_get_info()
    if free < gib * 2 ** 30:
        pytest.skip("needs %.1f GiB of free device memory, %.1f GiB free (%.1f GiB short)" %
                    (gib, free / 2 ** 30, gib - free / 2 ** 30))


def _engine(P, K):
    from trigenicinteractionpredictor_b200.engine import EMEngine
    return EMEngine(P, K, device="cuda:0")


def live_ranks(n, extra, seed, top_bit):
    """0, 1, 2, n - 2, n - 1, some ranks with `top_bit` set and `extra` random ones"""
    rng = np.random.default_rng(seed)
    hi = [r for r in ((1 << top_bit), (1 << top_bit) + 1, (1 << top_bit) | ((1 << top_bit) - 1), n - 3) if r < n]
    rand = rng.choice(n, size=extra, replace=False).tolist()
    return np.unique([0, 1, 2, n - 2, n - 1] + hi + rand)


def assert_rows(prob, ids, sc, keys, sums):
    assert len(sc) == len(keys)
    assert np.array_equal(ids, prob.ids(keys))
    assert np.array_equal(bits(sc), bits(sums * TRIPLET_ULP / prob.S))


# Passes of the unmutated build (measured on a B200): a wrapped shared bin may cost passes without changing the rows, so
# the pass count is part of the result.
TOP_TRIPLETS_PASSES = {"within_positives": 3, "known": 5}


def _top_triplets_cases(torch, n, cases, prob):
    import time
    eng = _engine(n, prob.K)
    th, pr = prob.thetas(), prob.prs()
    for name, (kn, N) in cases.items():
        t0 = time.time()
        ids, sc = eng.top_triplets(th, pr, prob.cand, kn, N)
        passes = eng.lib.tip_top_triplets_last_passes()
        print("tip_top_triplets n=%d %s: %d passes, %.1f s" % (n, name, passes, time.time() - t0), flush=True)
        keys, sums = ref_top(prob, kn, N)
        assert_rows(prob, ids, sc, keys, sums)
        assert passes == TOP_TRIPLETS_PASSES[name], (name, passes)


@pytest.mark.gpu
def test_top_triplets_past_the_shared_bin_flush(torch_cuda):
    """n = 2^15: the first pass lets all C(n, 3) = 5.9e12 scores through, ~1e10 per CTA into 32-bit shared bins, so the
    flush runs; N within the 2.4e6 positive scores.  The rows and the pass count cannot show a missing flush: a bin that
    wraps still sums, over the hundreds of CTAs, to ~10^11 or more, far above the buffer capacity and N (< 2^30) that the
    narrowing compares it with, so every narrowing decision is the same.  (N into the zero tie at this n takes minutes
    of passes: the tie is narrowed on the packed ranks in test_top_triplets_known_keys_at_2_22.)"""
    need_memory(torch_cuda, 2)
    n = 1 << 15
    prob = Planted(n, live_ranks(n, 240, 1, 14), 2, 2, 1)
    _top_triplets_cases(torch_cuda, n, {"within_positives": (np.empty(0, np.uint64), 5000)}, prob)


@pytest.mark.gpu
def test_top_triplets_known_keys_at_2_22(torch_cuda):
    """n = 2^12, 2^22 known keys: half of the live triplets and the first zero keys, N 10^5 past them, so the selection
    ends in the zero tie and is narrowed on packed ranks over a 54-bit range."""
    need_memory(torch_cuda, 2)
    n = 1 << 12
    prob = Planted(n, live_ranks(n, 240, 2, 11), 2, 2, 2)
    lk, _ = prob.live_triplets()
    rng = np.random.default_rng(2)
    planted = rng.choice(lk, size=len(lk) // 2, replace=False)
    first = zero_keys(prob, all_blocks(n), np.empty(0, np.uint64), (1 << 22) - len(planted))
    known = np.unique(np.concatenate([planted, first]))
    assert len(known) == 1 << 22
    _top_triplets_cases(torch_cuda, n, {"known": (known, len(lk) - len(planted) + 100_000)}, prob)


@pytest.mark.gpu
def test_score_histogram_total_past_2_42(torch_cuda):
    """n = 2^15: every one of the C(n, 3) > 2^42 scores is counted once; the zero bin and the live bins are exact."""
    need_memory(torch_cuda, 1)
    n, K, S = 1 << 15, 2, 2
    prob = Planted(n, live_ranks(n, 200, 3, 14), K, S, 3)
    layout, hist = _engine(n, K).score_histogram(prob.thetas(), prob.prs(), prob.cand)
    want = ref_histogram(prob, layout)
    assert int(hist.sum()) == comb(n, 3) > 1 << 42
    assert np.array_equal(hist, want)


@pytest.mark.gpu
def test_top_triplets_per_gene_universe_past_2_33(torch_cuda):
    """n = 2^17 + 3: C(n - 1, 2) = 8.6e9 pairs per query; queries at ranks 0 and n - 1, a live and a dead one, N past the
    positives into the zero tie, known keys among the live triplets and the first zero keys of query 0."""
    need_memory(torch_cuda, 2)
    n, K, S = (1 << 17) + 3, 2, 1
    prob = Planted(n, live_ranks(n, 180, 4, 16), K, S, 4)
    eng = _engine(n, K)
    dead = int(np.flatnonzero(~prob.is_live[1000:])[0]) + 1000
    live = int(prob.live[len(prob.live) // 2])
    queries = [0, n - 1, live, dead]
    lk, _ = prob.live_triplets()
    rng = np.random.default_rng(5)
    known = np.unique(np.concatenate([rng.choice(lk, size=len(lk) // 3, replace=False),
                                      zero_keys(prob, gene_blocks(n, 0), np.empty(0, np.uint64), 30_000)[::2]]))
    N = 60_000
    ids, sc, counts = eng.top_triplets_per_gene(prob.thetas(), prob.prs(), prob.cand, queries, known, N)
    assert np.array_equal(counts, [N] * 4)
    for i, r in enumerate(queries):
        keys, sums = ref_top_gene(prob, r, known, N)
        assert_rows(prob, ids[i], sc[i], keys, sums)
    print("tip_top_triplets_per_gene passes:", eng.lib.tip_top_triplets_per_gene_last_passes())


@pytest.mark.gpu
def test_top_triplets_per_gene_at_2_21(torch_cuda):
    """n_cand = 2^21, the limit: one live query at rank n - 1 (every bit of the 21-bit fields set), 2.2e12 pairs."""
    need_memory(torch_cuda, 2)
    n, K, S = MAX_N, 2, 1
    prob = Planted(n, live_ranks(n, 150, 6, 20), K, S, 6)
    N = 2000
    ids, sc, counts = _engine(n, K).top_triplets_per_gene(prob.thetas(), prob.prs(), prob.cand, [n - 1],
                                                          np.empty(0, np.uint64), N)
    keys, sums = ref_top_gene(prob, n - 1, np.empty(0, np.uint64), N)
    assert counts[0] == N and np.all(sums > 0)
    assert_rows(prob, ids[0], sc[0], keys, sums)


def _pairs_at_the_edges(prob):
    n = prob.n
    dead = np.flatnonzero(~prob.is_live)
    lv = prob.live
    return [(0, n - 1), (n - 1, n - 2), (int(lv[3]), int(lv[-4])), (int(dead[5]), int(dead[-7])), (int(lv[6]), int(dead[9]))]


@pytest.mark.gpu
def test_top_triplets_per_pair_at_2_21(torch_cuda):
    """n_cand = 2^21: pairs (0, n - 1), (n - 2, n - 1), live, dead and mixed; N past the positives into the zero tie
    (partner rank order) with known partners; then random parameters against an exhaustive NumPy reference."""
    need_memory(torch_cuda, 2)
    n, K, S = MAX_N, 2, 2
    prob = Planted(n, live_ranks(n, 150, 7, 20), K, S, 7)
    eng = _engine(n, K)
    pairs = _pairs_at_the_edges(prob)
    known = []
    for ra, rb in pairs:
        c = np.array([x for x in list(range(2, 400, 3)) + [n - 3] if x not in (ra, rb)])
        tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
        known.append(pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2]))
    known = np.unique(np.concatenate(known))
    N = 1500
    ids, sc, counts = eng.top_triplets_per_pair(prob.thetas(), prob.prs(), prob.cand, pairs, known, N)
    for i, (ra, rb) in enumerate(pairs):
        c, sums = ref_top_pair(prob, min(ra, rb), max(ra, rb), known, N)
        assert counts[i] == N
        tri = np.sort(np.stack([np.full(N, ra), np.full(N, rb), c], 1), 1)
        assert np.array_equal(ids[i], prob.cand[tri])
        assert np.array_equal(bits(sc[i]), bits(sums * TRIPLET_ULP / S))
    # random parameters: exhaustive over the 2^21 partners of each pair
    rng = np.random.default_rng(8)
    th = rng.dirichlet(np.ones(K), size=n)[None]
    pr = rng.random((1, K, K, K, 2))
    cand = prob.cand.astype(np.int64)
    ids, sc, counts = eng.top_triplets_per_pair(th, pr, prob.cand, pairs[:3], np.empty(0, np.uint64), N)
    for i, (ra, rb) in enumerate(pairs[:3]):
        c = np.arange(n)
        c = c[(c != ra) & (c != rb)]
        tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
        g = th[0][cand[tri]]
        s = np.einsum("ix,iy,iz,xyz->i", g[:, 0], g[:, 1], g[:, 2], pr[0][..., 1], optimize=True)
        o = np.lexsort((c, -s))[:N + 64]
        check_against_oracle(ids[i], sc[i], cand[tri[o]], s[o], N)


@pytest.mark.gpu
def test_rank_per_pair_at_2_21(torch_cuda):
    """n_cand = 2^21: test partners at rc = n - 1, live, and deep in the zero tie with train partners interleaved
    (every other partner of two pairs: 2^21 known keys); ranks up to 2^21 - 3."""
    need_memory(torch_cuda, 2)
    n, K, S = MAX_N, 2, 1
    prob = Planted(n, live_ranks(n, 150, 9, 20), K, S, 9)
    eng = _engine(n, K)
    lv = prob.live
    dead = np.flatnonzero(~prob.is_live)
    pairs = [(0, 1), (int(lv[3]), int(lv[-4])), (int(dead[5]), int(dead[-7])), (n - 2, int(lv[5]))]
    known = []
    for ra, rb in pairs[:2]:
        c = np.arange(0, n, 2)
        c = c[(c != ra) & (c != rb)]
        tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
        known.append(pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2]))
    known = np.unique(np.concatenate(known))
    assert len(known) > (1 << 21) - 8
    rng = np.random.default_rng(10)
    tp, trc = [], []
    for p, (ra, rb) in enumerate(pairs):
        cs = set(rng.choice(n, size=40).tolist()) | {n - 1, n - 3, 2, 3, 4, 5} | set(lv[::10].tolist())
        cs = sorted(c for c in cs if c not in (ra, rb))
        tp += [p] * len(cs)
        trc += cs
    tp, trc = np.array(tp), np.array(trc)
    rank, score, universe = eng.rank_per_pair(prob.thetas(), prob.prs(), prob.cand, pairs, known, tp, trc)
    for p, (ra, rb) in enumerate(pairs):
        sel = tp == p
        want_rank, want_sum, want_u = ref_rank_pair(prob, min(ra, rb), max(ra, rb), known, trc[sel])
        assert universe[p] == want_u
        assert np.array_equal(rank[sel], want_rank), p
        seen = want_rank > 0
        assert np.array_equal(bits(score[sel][seen]), bits(want_sum[seen] * TRIPLET_ULP / S))
    assert rank.max() > (1 << 21) - 64


@pytest.mark.gpu
def test_rank_per_gene_past_2_32(torch_cuda):
    """n = 2^17 + 3: zero-score test triplets near the end of the packed order (ranks and universes > 2^32), train
    triplets ahead of them subtracted, live test triplets, and a query with 2 049 test entries (two count rounds)."""
    need_memory(torch_cuda, 2)
    n, K, S = (1 << 17) + 3, 2, 2
    prob = Planted(n, live_ranks(n, 180, 11, 16), K, S, 11)
    eng = _engine(n, K)
    lv = prob.live
    dead = int(np.flatnonzero(~prob.is_live[1000:])[0]) + 1000
    queries = [0, n - 1, int(lv[len(lv) // 2]), dead]
    rng = np.random.default_rng(12)
    lk, _ = prob.live_triplets()
    tail = [(n - 3, n - 2), (n - 4, n - 1), (n - 2, n - 1), (1, 2), (5, n - 1)]
    tests = {0: tail + [(int(lv[3]), int(lv[7]))], 1: [(0, 1), (n - 4, n - 3), (n - 5, n - 2), (int(lv[4]), int(lv[9]))],
             3: tail[:3] + [(0, 1), (dead + 1, dead + 2)]}
    others = np.array([x for x in lv.tolist() if x != queries[2]])
    uv = set()
    while len(uv) < 2049:
        u, v = sorted(rng.choice(n, size=2, replace=False).tolist()) if len(uv) % 3 else sorted(rng.choice(others, 2, False))
        if queries[2] not in (u, v):
            uv.add((u, v))
    tests[2] = sorted(uv)
    known = [rng.choice(lk, size=len(lk) // 3, replace=False)]
    for qi, q in enumerate(queries):
        # train triplets of the query ahead of its tail tests and among its first keys
        tr = [sorted((q, n - 5 - i, n - 4 - i)) for i in range(3, 40)] + [sorted((q, x, x + 1)) for x in range(3, 60, 2)]
        tr = [t for t in tr if len(set(t)) == 3]
        known.append(pack_ranks(*np.array(tr).T))
    known = np.unique(np.concatenate(known))
    tq, tu, tv = [], [], []
    for qi, q in enumerate(queries):
        for u, v in tests[qi]:
            if q not in (u, v) and u != v:
                tq.append(qi)
                tu.append(u)
                tv.append(v)
    tq, tu, tv = np.array(tq), np.array(tu), np.array(tv)
    rank, score, universe = eng.rank_per_gene(prob.thetas(), prob.prs(), prob.cand, queries, known, tq, tu, tv)
    for qi, q in enumerate(queries):
        sel = tq == qi
        want_rank, want_sum, want_u = ref_rank_gene(prob, q, known, zip(tu[sel], tv[sel]))
        assert universe[qi] == want_u > 1 << 32
        assert np.array_equal(rank[sel], want_rank), q
        seen = want_rank > 0
        assert np.array_equal(bits(score[sel][seen]), bits(want_sum[seen] * TRIPLET_ULP / S))
    assert rank.max() > 1 << 32


@pytest.mark.gpu
def test_rank_per_gene_at_2_21(torch_cuda):
    """n_cand = 2^21, one query: the count sweep over the largest per-query universe (C(2^21 - 1, 2) = 2.2e12)."""
    need_memory(torch_cuda, 2)
    n, K, S = MAX_N, 2, 1
    prob = Planted(n, live_ranks(n, 120, 13, 20), K, S, 13)
    lv = prob.live
    q = n - 1
    tests = [(n - 3, n - 2), (0, 1), (int(lv[3]), int(lv[8])), (1 << 20, (1 << 20) + 5), (n - 7, n - 2)]
    known = np.sort(pack_ranks([n - 5, 0], [n - 4, 2], [n - 1, n - 1]))
    tu, tv = np.array([t[0] for t in tests]), np.array([t[1] for t in tests])
    rank, score, universe = _engine(n, K).rank_per_gene(prob.thetas(), prob.prs(), prob.cand, [q], known,
                                                        np.zeros(len(tests), np.int32), tu, tv)
    want_rank, want_sum, want_u = ref_rank_gene(prob, q, known, tests)
    assert universe[0] == want_u
    assert np.array_equal(rank, want_rank)
    assert np.array_equal(bits(score), bits(want_sum * TRIPLET_ULP / S))
    assert rank.max() > 1 << 40


@pytest.mark.gpu
def test_top_pairs_past_4000_chunks(torch_cuda):
    """n = 2^17 + 5: 8.6e9 pairs in more than 4 000 chunks, live ranks with bit 17 set, N = 2^20 into the zero tie."""
    need_memory(torch_cuda, 2)
    n, K, S = (1 << 17) + 5, 2, 2
    prob = Planted(n, live_ranks(n, 200, 14, 17), K, S, 14)
    eng = _engine(n, K)
    lk, _ = live_pairs(prob)
    rng = np.random.default_rng(15)
    known = np.unique(np.concatenate([rng.choice(lk, size=len(lk) // 3, replace=False),
                                      pack2(np.zeros(300, np.int64), np.arange(7, 1207, 4))]))
    N = 1 << 20
    ids, sc = eng.top_pairs(prob.thetas(), prob.qs(), prob.cand, known, N)
    assert eng.lib.tip_top_pairs_last_chunks() > 4000
    keys, sums = ref_top_pairs(prob, known, N)
    assert len(sc) == N
    assert np.array_equal(ids, prob.cand[unpack2(keys)])
    assert np.array_equal(bits(sc), bits(sums * PAIR_ULP / S))


@pytest.mark.gpu
def test_top_pairs_per_gene_at_2_21(torch_cuda):
    """n_cand = 2^21: one query per chunk; queries 0, n - 1, live and dead, N past the positives into the zero tie; then
    random parameters against NumPy."""
    need_memory(torch_cuda, 2)
    n, K, S = MAX_N, 2, 2
    prob = Planted(n, live_ranks(n, 300, 16, 20), K, S, 16)
    eng = _engine(n, K)
    dead = int(np.flatnonzero(~prob.is_live)[3])
    queries = [0, n - 1, int(prob.live[100]), dead]
    known = np.unique(pack2([0, 0, 5, n - 2, dead], [1, 3, n - 1, n - 1, dead + 1]))
    N = 1000
    ids, sc, counts = eng.top_pairs_per_gene(prob.thetas(), prob.qs(), prob.cand, queries, known, N)
    assert eng.lib.tip_top_pairs_per_gene_last_chunks() == len(queries)
    for i, r in enumerate(queries):
        x, sums = ref_top_pairs_gene(prob, r, known, N)
        lo, hi = np.minimum(x, r), np.maximum(x, r)
        assert counts[i] == N
        assert np.array_equal(ids[i], prob.cand[np.stack([lo, hi], 1)])
        assert np.array_equal(bits(sc[i]), bits(sums * PAIR_ULP / S))
    rng = np.random.default_rng(17)
    th = rng.dirichlet(np.ones(K), size=n)[None]
    q = rng.random((1, K, K, 2))
    cand = prob.cand.astype(np.int64)
    ids, sc, counts = eng.top_pairs_per_gene(th, q, prob.cand, [0, n - 1], np.empty(0, np.uint64), N)
    t = th[0][cand]
    for i, r in enumerate([0, n - 1]):
        x = np.arange(n)
        x = x[x != r]
        lo, hi = np.minimum(x, r), np.maximum(x, r)
        s = np.einsum("ix,xy,iy->i", t[lo], q[0][..., 1], t[hi])
        o = np.lexsort((x, -s))[:N + 64]
        check_against_oracle(ids[i], sc[i], cand[np.stack([lo[o], hi[o]], 1)], s[o], N)


@pytest.mark.gpu
def test_score_pairs_at_high_ids(torch_cuda):
    """P = 2^21: tip_score and tip_score_pairs of live ids up to 2^21 - 1, bit-equal to the dyadic reference."""
    need_memory(torch_cuda, 1)
    n, K, S = MAX_N, 3, 1
    prob = Planted(n, live_ranks(n, 60, 18, 20), K, S, 18)
    eng = _engine(n, K)
    th, pr, q = prob.thetas(), prob.prs(), prob.qs()
    rank_of = np.empty(n, np.int64)
    rank_of[prob.cand] = np.arange(n)
    live_ids = np.sort(prob.cand[prob.live])
    extra = [i for i in (n - 1, n - 2, (1 << 20) + 1) if i not in set(live_ids[-40:].tolist())]
    ids = np.concatenate([live_ids[-40:], extra]).astype(np.int64)
    assert len(set(ids.tolist())) == len(ids)
    trip = np.array([t for t in itertools.combinations(ids[-12:].tolist(), 3)])
    got = eng.score_sum(th, pr, trip)
    want = prob.triplet_int(rank_of[trip]) * TRIPLET_ULP
    assert np.array_equal(bits(got), bits(want)) and np.count_nonzero(want) > 0
    eng.set_params(th[0], pr[0])
    eng.set_q(q[0])
    a, b = np.array(list(itertools.permutations(ids[-15:].tolist(), 2))).T
    got = eng.score_pairs(a, b).cpu().numpy()
    want = prob.pair_int(rank_of[a], rank_of[b]) * PAIR_ULP
    assert np.array_equal(bits(got), bits(want)) and np.count_nonzero(want) > 0


@pytest.mark.gpu
def test_top_pairs_ranks_past_2_20(torch_cuda):
    """n = 2^20 + 2^12: pair keys whose low rank field has bit 20 set (100 live ranks lie past 2^20), N within the
    positives, a third of the live pairs known.  The first chunk (rows below 64, columns below 2^15) holds more than N
    positive pairs, so the running threshold leaves the zero tie after it and the 2.6e5 chunks after it stay cheap."""
    need_memory(torch_cuda, 2)
    n, K, S = (1 << 20) + (1 << 12), 2, 2
    rng = np.random.default_rng(19)
    live = np.concatenate([live_ranks(n, 20, 19, 20), rng.choice(64, size=40, replace=False),
                           rng.choice(np.arange(64, 1 << 15), size=100, replace=False),
                           rng.choice(np.arange(1 << 20, n), size=100, replace=False)])
    prob = Planted(n, live, K, S, 19)
    eng = _engine(n, K)
    lk, _ = live_pairs(prob)
    known = np.unique(rng.choice(lk, size=len(lk) // 3, replace=False))
    N = 2000
    ids, sc = eng.top_pairs(prob.thetas(), prob.qs(), prob.cand, known, N)
    keys, sums = ref_top_pairs(prob, known, N)
    assert np.all(sums > 0) and (unpack2(keys)[:, 1] >= 1 << 20).sum() > 100
    assert len(sc) == N
    assert np.array_equal(ids, prob.cand[unpack2(keys)])
    assert np.array_equal(bits(sc), bits(sums * PAIR_ULP / S))


@pytest.mark.gpu
def test_top_triplets_per_gene_buffers_at_2_24(torch_cuda):
    """n_query * N = 2^24, the limit: every one of n = 4 096 ranks is a query (in a shuffled order), N = 4 096, with
    known keys among the live triplets; every query's rows exact."""
    need_memory(torch_cuda, 2)
    n, K, S = 1 << 12, 2, 2
    prob = Planted(n, live_ranks(n, 100, 20, 11), K, S, 20)
    rng = np.random.default_rng(21)
    queries = rng.permutation(n)
    lk, _ = prob.live_triplets()
    known = np.unique(rng.choice(lk, size=len(lk) // 3, replace=False))
    N = 1 << 12
    ids, sc, counts = _engine(n, K).top_triplets_per_gene(prob.thetas(), prob.prs(), prob.cand, queries, known, N)
    assert np.array_equal(counts, np.full(n, N))
    for i, r in enumerate(queries.tolist()):
        keys, sums = ref_top_gene(prob, r, known, N)
        assert_rows(prob, ids[i], sc[i], keys, sums)


@pytest.mark.gpu
def test_top_triplets_per_pair_buffers_at_2_24(torch_cuda):
    """n_pairs * N = 2^24, the limit: 4 096 pairs (live, dead, mixed, the edges of the rank range) with N = 4 096 of the
    n - 2 = 4 198 partners each, so every pair's rows run deep into its zero tie, with known partners."""
    need_memory(torch_cuda, 2)
    n, K, S = 4200, 2, 1
    prob = Planted(n, live_ranks(n, 120, 22, 12), K, S, 22)
    rng = np.random.default_rng(23)
    lv = prob.live
    pairs = {(0, n - 1), (n - 2, n - 1), (0, 1)} | {tuple(sorted(rng.choice(lv, 2, replace=False).tolist())) for _ in range(500)}
    while len(pairs) < 4096:
        a, b = sorted(rng.choice(n, 2, replace=False).tolist())
        pairs.add((a, b))
    pairs = [p if i % 2 else p[::-1] for i, p in enumerate(sorted(pairs))]
    known = []
    for ra, rb in pairs[::7]:
        c = np.array([x for x in range(1, n, 97) if x not in (ra, rb)])
        tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
        known.append(pack_ranks(tri[:, 0], tri[:, 1], tri[:, 2]))
    known = np.unique(np.concatenate(known))
    N = 1 << 12
    ids, sc, counts = _engine(n, K).top_triplets_per_pair(prob.thetas(), prob.prs(), prob.cand, pairs, known, N)
    for i, (ra, rb) in enumerate(pairs):
        c, sums = ref_top_pair(prob, min(ra, rb), max(ra, rb), known, N)
        assert counts[i] == len(c)
        tri = np.sort(np.stack([np.full(len(c), ra), np.full(len(c), rb), c], 1), 1)
        assert np.array_equal(ids[i][:len(c)], prob.cand[tri]), (ra, rb)
        assert np.array_equal(bits(sc[i][:len(c)]), bits(sums * TRIPLET_ULP / S))


@pytest.mark.gpu
def test_top_pairs_per_gene_buffers_at_2_24(torch_cuda):
    """n_query * N = 2^24, the limit: 4 096 queries of n = 8 192 (0 and n - 1 among them, shuffled), N = 4 096."""
    need_memory(torch_cuda, 2)
    n, K, S = 1 << 13, 2, 2
    prob = Planted(n, live_ranks(n, 150, 24, 12), K, S, 24)
    rng = np.random.default_rng(25)
    inner = np.unique(np.concatenate([prob.live, rng.choice(n, 6000, replace=False)]))
    inner = rng.permutation(inner[(inner > 0) & (inner < n - 1)])[:4094]
    queries = rng.permutation(np.concatenate([[0, n - 1], inner]))
    lk, _ = live_pairs(prob)
    known = np.unique(np.concatenate([rng.choice(lk, size=len(lk) // 3, replace=False), pack2([0, 0, 7], [1, n - 1, n - 2])]))
    N = 1 << 12
    ids, sc, counts = _engine(n, K).top_pairs_per_gene(prob.thetas(), prob.qs(), prob.cand, queries, known, N)
    assert len(queries) == 4096 and np.array_equal(counts, np.full(4096, N))
    for i, r in enumerate(queries.tolist()):
        x, sums = ref_top_pairs_gene(prob, r, known, N)
        lo, hi = np.minimum(x, r), np.maximum(x, r)
        assert np.array_equal(ids[i], prob.cand[np.stack([lo, hi], 1)]), r
        assert np.array_equal(bits(sc[i]), bits(sums * PAIR_ULP / S))


@pytest.mark.gpu
def test_rank_per_pair_2_22_pairs_2_26_known(torch_cuda):
    """n_pairs = 2^22 and n_known = 2^26: every pair (i, j) with i < 2 048 <= j < 4 096 of n = 4 112 candidates, the 16
    highest ranks F a known partner of every pair, one test partner per pair (in F for some: rank 0).  A pair with a
    dead gene has no positive partner, so its rank is 1 + the partners below it outside {i, j} (F lies above them all);
    the pairs of two live genes take the exhaustive per-pair reference."""
    torch = torch_cuda
    need_memory(torch, 6)
    n, K, S = 4096 + 16, 2, 1
    prob = Planted(n, live_ranks(n, 100, 26, 11), K, S, 26)
    F = np.arange(4096, n, dtype=np.uint64)
    i, j = np.meshgrid(np.arange(2048), np.arange(2048, 4096), indexing="ij")
    i, j = i.ravel(), j.ravel()
    known = ((i.astype(np.uint64)[:, None] << np.uint64(42)) | (j.astype(np.uint64)[:, None] << np.uint64(21)) | F).ravel()
    assert len(known) == 1 << 26 and np.all(known[1:] > known[:-1])
    pairs = np.stack([i, j], 1)
    pairs[1::2] = pairs[1::2, ::-1]
    c = (i * 7 + j * 13) % n
    while True:
        bad = (c == i) | (c == j)
        if not bad.any():
            break
        c[bad] = (c[bad] + 1) % n
    tp = np.arange(len(i))
    rank, score, universe = _engine(n, K).rank_per_pair(prob.thetas(), prob.prs(), prob.cand, pairs, known, tp, c)
    del known
    assert np.all(universe == n - 2 - 16)
    both = prob.is_live[i] & prob.is_live[j]
    want = np.where(c >= 4096, 0, 1 + c - (i < c) - (j < c))
    assert np.array_equal(rank[~both], want[~both])
    assert np.all(score[~both] == 0)
    known_F = lambda a, b: pack_ranks(np.full(16, a), np.full(16, b), np.arange(4096, n))  # noqa: E731
    for p in np.flatnonzero(both).tolist():
        want_rank, want_sum, _ = ref_rank_pair(prob, int(i[p]), int(j[p]), known_F(i[p], j[p]), [c[p]])
        assert rank[p] == want_rank[0], p
        if want_rank[0]:
            assert bits(score[p:p + 1])[0] == bits(want_sum * TRIPLET_ULP / S)[0]
    assert both.sum() > 100
