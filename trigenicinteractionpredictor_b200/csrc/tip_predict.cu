// Exact top-N of all unordered triplets of a candidate gene list (tip_top_triplets, include/tip.h).
//
// The candidates are relabelled by rank, their position in the decimal-string order of their ids, so that every triple of
// ranks i < j < k is already in the reference's key slot order (a, b, c) (TIP.py:353).  Fixing the middle slot b = j:
//     W_b[x][z]        = sum_y th_b[y] p[x][y][z][1]                        (tip_predict_prep_kernel, K^3 per gene)
//     Q_b[i][z]        = sum_x th_i[x] W_b[x][z]            for i < j        (scoring kernel, in shared memory)
//     score(i, j, k)   = sum_z Q_b[i][z] th_k[z]            for k > j        (scoring kernel, DMMA m8n8k4)
// and with S parameter sets the contraction index runs over (s, z): the ensemble sum is the same product, S K long.
// One sweep is C(n, 3) * 2 S K flop on the fp64 tensor path; nothing is stored per triplet.
//
// Selection by recomputation.  Every pass recomputes all scores (same kernel, same contraction order, so bit-identical
// numbers in every pass) and only the ones that clear a threshold leave the registers: they are counted, histogrammed
// in shared memory and appended to a bounded buffer.  The host picks the first threshold from a deterministic sample of
// triplets, then narrows it with the histogram until the buffer holds between N and its capacity; under ties the threshold
// continues on the packed rank triple, so the result is exact whatever the scores are.  The buffer is then sorted by
// (score descending, packed ranks ascending) and the first N rows are written out.  Known triplets are dropped in the
// epilogue (binary search in the sorted known keys), so they never count towards N.
//
// Per query gene (tip_top_triplets_per_gene): the pairs of a query of rank r split into three regions by r's slot, each a
// product th_x^T M th_y with a K x K matrix of the query (tip_query_pass_kernel, which shares the Q tile, the DMMA block
// loop and the epilogue with tip_predict_pass_kernel).  Each query has its own threshold, survivor count, histogram and
// buffer; its first threshold is the best score of a per-query sample, and sweeps after the first score only the queries
// whose threshold has not settled.  A segmented sort orders every query's buffer.
//
// Histogram of all scores (tip_score_histogram): the same sweep as tip_top_triplets, counting every score into a fixed
// log-spaced histogram of its bits (tip_hist_pass_kernel); the ranks of held-out triplets among all triplets follow from it.
//
// Ranks per query pair (tip_rank_per_pair): the tiles and column phases of tip_top_triplets_per_pair, swept once to record
// the scores of the held-out partners and once to count, per pair, the scores ahead of each of them (tip_rank_pass_kernel).
//
// Ranks per query gene (tip_rank_per_gene): the work items, Q tiles and column blocks of tip_top_triplets_per_gene, swept
// once to record the scores of the held-out and train triplets of the queries and once to count, per query, the scores
// ahead of each held-out one (tip_gene_rank_pass_kernel); the train triplets ahead are subtracted.
//
// The digenic model's gene pairs (tip_top_pairs, tip_top_pairs_per_gene, tip_score_pairs): see the last section.
#include <algorithm>
#include <cmath>
#include <vector>

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_segmented_sort.cuh>
#include <cub/device/device_select.cuh>

#include "tip_common.cuh"

namespace tip {
namespace {

constexpr int kPredRows = 64;         // rows (slot a) of a work item
constexpr int kPredThreads = 128;     // 4 warps: 2 row halves x 2 column halves of a 64 x 64 block
constexpr int kPredBins = 2048;       // histogram bins; bin kPredBins counts the entries ranked ahead of the range
constexpr int kPredSample = 1 << 20;  // triplets in the sample that places the first threshold
constexpr int kPredMaxSK = 384;       // S * K: the Q tile of 64 rows must fit shared memory
constexpr int kRankBits = 21;
constexpr unsigned long long kInfBits = 0x7FF0000000000000ull;

// shared-memory row stride of the Q tile: == 4 (mod 16) doubles, so that the fragment loads (8 rows x 4 columns) touch
// every bank pair the minimum number of times
__host__ __device__ inline int q_stride(int skp) { return (skp + 11) / 16 * 16 + 4; }

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// items before middle rank j: sum_{i=1}^{j-1} ceil(i / 64)
__host__ __device__ inline long long items_before(long long j)
{
    const long long m = j - 1;
    if (m <= 0) return 0;
    const long long q = m / kPredRows, r = m % kPredRows;
    return kPredRows * q * (q + 1) / 2 + r * (q + 1);
}

// threshold state of one selection (one per call of tip_top_triplets, one per query of tip_top_triplets_per_gene)
struct Sel {
    int mode;                       // 0: keep bits >= lo; 1: keep bits > v, or bits == v and packed <= rhi
    int shift;
    unsigned long long lo, hi;      // mode 0: histogram range of score bits (bin 0 = highest)
    unsigned long long v, rlo, rhi; // mode 1: tied score bits and the histogram range of packed ranks (bin 0 = lowest)
};

// where the scores of a work item sit: row ra and column rc are a triplet when ra < row_end, rc < col_end and (tri) rc > ra;
// its packed rank triple is (ra << sh_r) | (rc << sh_c) | fixed
struct TileMap {
    int row_end, col_end;
    bool tri;
    int sh_r, sh_c;
    unsigned long long fixed;
};

struct PassArgs {
    int n, S, K, SK, SKP;
    const double *tcat;             // [n_pad][SKP] theta of every model, rank order, zero padded
    const double *W;                // [S][n][K][K]
    const unsigned long long *known;  // sorted packed rank triples
    long long n_known;
    long long n_items;
    Sel sel;
    unsigned long long *counter;    // [0] entries kept, [1] work-item cursor
    unsigned long long *hist;       // [kPredBins + 1]
    unsigned long long *out_bits, *out_packed;
    long long cap;
};

__device__ __noinline__ bool is_known(const unsigned long long *known, long long n, unsigned long long key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        const unsigned long long k = __ldg(known + mid);
        if (k < key) lo = mid + 1; else hi = mid;
    }
    return lo < n && __ldg(known + lo) == key;
}

// tcat[r][s K + k] = theta_s of candidate r, zero padded to n_pad rows and SKP columns
__device__ __forceinline__ double tcat_entry(long long t, int S, int P, int K, int n, int SKP, const double *theta,
                                             const int32_t *cand)
{
    const int r = (int)(t / SKP), col = (int)(t % SKP);
    if (r >= n || col >= S * K) return 0.0;
    const int s = col / K, k = col % K;
    return theta[((long long)s * P + cand[r]) * K + k];
}

__global__ void tip_predict_prep_kernel(int S, int P, int K, int n, int n_pad, int SKP, const double *__restrict__ theta,
                                        const double *__restrict__ p, const int32_t *__restrict__ cand, double *__restrict__ tcat,
                                        double *__restrict__ W)
{
    const long long n_t = (long long)n_pad * SKP, KK = (long long)K * K, n_w = (long long)S * n * KK;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_t + n_w; t += (long long)gridDim.x * blockDim.x) {
        if (t < n_t) {
            tcat[t] = tcat_entry(t, S, P, K, n, SKP, theta, cand);
        } else {
            const long long u = t - n_t;
            const int s = (int)(u / ((long long)n * KK));
            const long long rem = u % ((long long)n * KK);
            const int r = (int)(rem / KK), x = (int)(rem % KK) / K, z = (int)(rem % KK) % K;
            const double *th = theta + ((long long)s * P + cand[r]) * K;
            const double *ps = p + (long long)s * 2 * K * K * K;
            double acc = 0.0;
            for (int y = 0; y < K; ++y) acc = fma(th[y], ps[(((long long)x * K + y) * K + z) * 2 + 1], acc);
            W[u] = acc;
        }
    }
}

// deterministic uniform sample of triplets (three distinct ranks), scored with the same factors as the passes
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__global__ void tip_predict_sample_kernel(int n, int S, int K, int SKP, const double *__restrict__ tcat,
                                          const double *__restrict__ W, int n_sample, unsigned long long *__restrict__ out)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_sample) return;
    unsigned long long h = splitmix64((unsigned long long)t * 3 + 0x1234567ull);
    int r[3];
    for (int d = 0; d < 3;) {
        h = splitmix64(h);
        const int x = (int)(h % (unsigned long long)n);
        bool dup = false;
        for (int e = 0; e < d; ++e) dup |= (r[e] == x);
        if (!dup) r[d++] = x;
    }
    int a = min(r[0], min(r[1], r[2])), c = max(r[0], max(r[1], r[2]));
    int b = r[0] + r[1] + r[2] - a - c;
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
        const double *Wb = W + ((long long)s * n + b) * K * K;
        for (int x = 0; x < K; ++x) {
            double q = 0.0;
            for (int z = 0; z < K; ++z) q = fma(Wb[x * K + z], tcat[(long long)c * SKP + s * K + z], q);
            acc = fma(tcat[(long long)a * SKP + s * K + x], q, acc);
        }
    }
    out[t] = (unsigned long long)__double_as_longlong(acc);
}

// ---- pieces of a scoring pass, shared by tip_predict_pass_kernel and tip_query_pass_kernel ----

// Q tile: Q[i][s K + z] = sum_x th_{a0+i}[s K + x] M[s][x][z] (M of set s at M + s * m_stride); pad rows / columns are zero
__device__ __forceinline__ void form_q_tile(double *Q, int qs, const double *tcat, int SKP, int SK, int K, int a0, int rows,
                                            const double *M, long long m_stride)
{
    for (int e = threadIdx.x; e < kPredRows * SKP; e += kPredThreads) {
        const int i = e / SKP, col = e % SKP;
        double acc = 0.0;
        if (i < rows && col < SK) {
            const int s = col / K, z = col % K;
            const double *th = tcat + (long long)(a0 + i) * SKP + s * K;
            const double *Wb = M + s * m_stride + z;
            for (int x = 0; x < K; ++x) acc = fma(__ldg(th + x), __ldg(Wb + x * K), acc);
        }
        Q[i * qs + col] = acc;
    }
}

// a warp's 32 x 32 block of scores: acc[mi][ni][e] = row gq + 8 mi of Qw times column 8 ni + 2 tq + e of Bw
__device__ __forceinline__ void dmma_block(double (&acc)[4][4][2], const double *Qw, int qs, const double *Bw, int SKP)
{
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
#pragma unroll 2
    for (int kk = 0; kk < SKP; kk += 4) {
        double af[4], bf[4];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) af[mi] = Qw[mi * 8 * qs + kk];
#pragma unroll
        for (int ni = 0; ni < 4; ++ni) bf[ni] = __ldg(Bw + (long long)ni * 8 * SKP + kk);
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int ni = 0; ni < 4; ++ni) dmma884(acc[mi][ni][0], acc[mi][ni][1], af[mi], bf[ni]);
    }
}

// epilogue of a block (ra0 = the lane's first row, rc0 = its first column): the threshold test runs in registers; only
// survivors go further: known keys are dropped, the rest are histogrammed in sh_hist and appended to out_* (counted past cap)
__device__ __forceinline__ void select_block(const double (&acc)[4][4][2], const Sel sel, const TileMap tm, int lane, int ra0,
                                             int rc0, const unsigned long long *known, long long n_known, unsigned *sh_hist,
                                             unsigned long long *counter, unsigned long long *out_bits,
                                             unsigned long long *out_packed, long long cap)
{
    unsigned keep = 0;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
                const bool pass = sel.mode == 0 ? bits >= sel.lo : bits >= sel.v;
                keep |= (pass ? 1u : 0u) << ((mi * 4 + ni) * 2 + e);
            }
    if (!__any_sync(0xffffffffu, keep != 0)) return;
#pragma unroll
    for (int f = 0; f < 32; ++f) {
        const int mi = f >> 3, ni = (f >> 1) & 3, e = f & 1;
        const int ra = ra0 + mi * 8, rc = rc0 + ni * 8 + e;
        const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
        const unsigned long long packed = ((unsigned long long)ra << tm.sh_r) | ((unsigned long long)rc << tm.sh_c) | tm.fixed;
        bool q = ((keep >> f) & 1u) && ra < tm.row_end && rc < tm.col_end && (!tm.tri || rc > ra);
        if (q && sel.mode == 1) q = bits > sel.v || packed <= sel.rhi;
        if (q && n_known > 0) q = !is_known(known, n_known, packed);
        int bin = kPredBins;
        if (q) {
            if (sel.mode == 0) {
                if (bits <= sel.hi) bin = (int)((sel.hi - bits) >> sel.shift);
            } else if (bits == sel.v && packed >= sel.rlo) {
                bin = (int)((packed - sel.rlo) >> sel.shift);
            }
            atomicAdd(sh_hist + bin, 1u);
        }
        const unsigned m = __ballot_sync(0xffffffffu, q);
        if (m == 0) continue;
        unsigned long long base = 0;
        if (lane == __ffs(m) - 1) base = atomicAdd(counter, (unsigned long long)__popc(m));
        base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
        if (q) {
            const unsigned long long idx = base + __popc(m & ((1u << lane) - 1u));
            if ((long long)idx < cap) {
                out_bits[idx] = bits;
                out_packed[idx] = packed;
            }
        }
    }
}

// add the CTA's shared bins to hist and clear them (all threads, between barriers)
__device__ __forceinline__ void flush_hist(unsigned *sh_hist, unsigned long long *hist)
{
    for (int i = threadIdx.x; i <= kPredBins; i += kPredThreads) {
        if (sh_hist[i]) atomicAdd(hist + i, (unsigned long long)sh_hist[i]);
        sh_hist[i] = 0;
    }
}

__global__ void __launch_bounds__(kPredThreads) tip_predict_pass_kernel(PassArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP);
    double *Q = reinterpret_cast<double *>(smem);                                   // [64][qs]
    unsigned *sh_hist = reinterpret_cast<unsigned *>(Q + (size_t)kPredRows * qs);  // [kPredBins + 1]
    __shared__ long long sh_item;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    for (int i = tid; i <= kPredBins; i += kPredThreads) sh_hist[i] = 0;
    double since_flush = 0.0;   // upper bound of the entries added to sh_hist since it was last flushed (CTA-uniform)
    const int n = A.n, SKP = A.SKP, K = A.K;

    for (;;) {
        __syncthreads();   // Q and sh_item of the previous item are no longer read
        if (tid == 0) sh_item = (long long)atomicAdd(A.counter + 1, 1ull);
        __syncthreads();
        const long long item = sh_item;
        if (item >= A.n_items) break;
        // item -> (middle rank j, row tile): items are numbered by ascending j, the heaviest (longest rows of c) first
        int jl = 1, jh = n - 2;
        while (jl < jh) {
            const int mid = (jl + jh + 1) >> 1;
            if (items_before(mid) <= item) jl = mid; else jh = mid - 1;
        }
        const int j = jl;
        const int a0 = (int)(item - items_before(j)) * kPredRows;
        const int rows = min(kPredRows, j - a0);
        const int n_c = n - 1 - j;

        form_q_tile(Q, qs, A.tcat, SKP, A.SK, K, a0, rows, A.W + (long long)j * K * K, (long long)n * K * K);
        __syncthreads();

        const TileMap tm{j, n, false, 2 * kRankBits, 0, (unsigned long long)j << kRankBits};
        if (wr * 32 < rows) {
            const double *Qw = Q + (wr * 32 + gq) * qs + tq;
            for (int c0 = j + 1 + wc * 32; c0 < n; c0 += 64) {
                double acc[4][4][2];
                dmma_block(acc, Qw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                select_block(acc, A.sel, tm, lane, a0 + wr * 32 + gq, c0 + 2 * tq, A.known, A.n_known, sh_hist, A.counter,
                             A.out_bits, A.out_packed, A.cap);
            }
        }
        // shared bins are 32-bit: flush before they could overflow
        since_flush += (double)rows * n_c;
        if (since_flush > 2.0e9) {
            __syncthreads();
            flush_hist(sh_hist, A.hist);
            since_flush = 0.0;
        }
    }
    flush_hist(sh_hist, A.hist);
}

// ---- per query (tip_top_triplets_per_gene) ----
// The pairs x < y of a query of rank r (both != r) fall into three regions by the query's slot; g = 0: x < y < r (slot c),
// g = 1: x < r < y (slot b), g = 2: r < x < y (slot a).  In each the score is th_x^T M_g th_y with, per set,
//     M_0[u][v] = sum_w th_q[w] p[u][v][w][1],   M_1[u][w] = sum_v th_q[v] p[u][v][w][1] (= W),   M_2[v][w] = sum_u th_q[u] p[u][v][w][1]
// Regions 0 and 2 are triangles (y > x); region 1 is the rectangle tip_predict_pass_kernel sweeps for middle rank r.

// tcat as tip_predict_prep_kernel writes it, and Mq[query][g][s][K][K]
__global__ void tip_query_prep_kernel(int S, int P, int K, int n, int n_pad, int SKP, int n_query, const double *__restrict__ theta,
                                      const double *__restrict__ p, const int32_t *__restrict__ cand,
                                      const int32_t *__restrict__ qrank, double *__restrict__ tcat, double *__restrict__ Mq)
{
    const long long n_t = (long long)n_pad * SKP, KK = (long long)K * K, n_m = (long long)n_query * 3 * S * KK;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_t + n_m; t += (long long)gridDim.x * blockDim.x) {
        if (t < n_t) {
            tcat[t] = tcat_entry(t, S, P, K, n, SKP, theta, cand);
        } else {
            const long long u = t - n_t;
            const int qi = (int)(u / (3 * S * KK)), g = (int)(u / (S * KK) % 3), s = (int)(u / KK % S);
            const int x = (int)(u % KK) / K, z = (int)(u % KK) % K;
            const double *th = theta + ((long long)s * P + cand[qrank[qi]]) * K;
            const double *ps = p + (long long)s * 2 * K * K * K;
            // index of p[.][.][.][1] with the query's group y in slot (2 - g) and (x, z) in the other two, in order
            const long long step = g == 0 ? 1 : g == 1 ? K : KK;
            const long long base = g == 0 ? ((long long)x * K + z) * K : g == 1 ? (long long)x * KK + z : (long long)x * K + z;
            double acc = 0.0;
            for (int y = 0; y < K; ++y) acc = fma(th[y], ps[(base + y * step) * 2 + 1], acc);
            Mq[u] = acc;
        }
    }
}

// T[s] = bits of the largest row sum of theta_s over the candidates (T zeroed by the caller)
__global__ void tip_query_rowsum_kernel(int n, int S, int K, int SKP, const double *__restrict__ tcat, unsigned long long *T)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    for (int s = 0; s < S; ++s) {
        double sum = 0.0;
        for (int k = 0; k < K; ++k) sum += tcat[(long long)r * SKP + s * K + k];
        atomicMax(T + s, (unsigned long long)__double_as_longlong(sum));
    }
}

// bound[q] >= every sum over the sets of a query's scores (non-negative parameters): th_x^T M th_y <= max(M) |th_x|_1 |th_y|_1
__global__ void tip_query_bound_kernel(int n_query, int S, int K, const double *__restrict__ Mq, const unsigned long long *T,
                                       double *__restrict__ bound)
{
    const int qi = blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= n_query) return;
    const long long KK = (long long)K * K;
    double best = 0.0;
    for (int g = 0; g < 3; ++g) {
        double b = 0.0;
        for (int s = 0; s < S; ++s) {
            const double *m = Mq + (((long long)qi * 3 + g) * S + s) * KK;
            double mx = 0.0;
            for (long long e = 0; e < KK; ++e) mx = fmax(mx, m[e]);
            const double t = __longlong_as_double((long long)T[s]);
            b += mx * t * t;
        }
        best = fmax(best, b);
    }
    bound[qi] = best;
}

// best[q] = bits of the largest of n_samp scores (summed over the sets) of deterministic random pairs of query q; with
// about pairs / n_samp scores above it, it places the query's first threshold (best zeroed by the caller)
__global__ void tip_query_sample_kernel(int n, int S, int K, int SKP, int n_query, int n_samp, const int32_t *__restrict__ qrank,
                                        const double *__restrict__ tcat, const double *__restrict__ Mq,
                                        unsigned long long *__restrict__ best)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (long long)n_query * n_samp) return;
    const int qi = (int)(t / n_samp), r = qrank[qi];
    unsigned long long h = splitmix64((unsigned long long)t * 3 + 0x7654321ull);
    int x, y;
    do {
        h = splitmix64(h);
        x = (int)(h % (unsigned long long)n);
        h = splitmix64(h);
        y = (int)(h % (unsigned long long)n);
    } while (x == y || x == r || y == r);
    if (x > y) { const int z = x; x = y; y = z; }
    const int g = y < r ? 0 : x < r ? 1 : 2;
    const long long KK = (long long)K * K;
    double acc = 0.0;
    for (int s = 0; s < S; ++s) {
        const double *m = Mq + (((long long)qi * 3 + g) * S + s) * KK;
        for (int u = 0; u < K; ++u) {
            double q = 0.0;
            for (int v = 0; v < K; ++v) q = fma(m[u * K + v], tcat[(long long)y * SKP + s * K + v], q);
            acc = fma(tcat[(long long)x * SKP + s * K + u], q, acc);
        }
    }
    atomicMax(best + qi, (unsigned long long)__double_as_longlong(acc));
}

// tiles of the three regions of the query of rank r: tc (g = 0, rows 0 .. r-2), tb (g = 1, rows 0 .. r-1, only when
// r <= n-2), ta (g = 2, rows r+1 .. n-2)
__host__ __device__ inline void query_tiles(int n, int r, int &tc, int &tb, int &ta)
{
    tc = (max(r - 1, 0) + kPredRows - 1) / kPredRows;
    tb = r <= n - 2 ? (r + kPredRows - 1) / kPredRows : 0;
    ta = (max(n - 2 - r, 0) + kPredRows - 1) / kPredRows;
}

struct QueryPassArgs {
    int n, S, K, SK, SKP;
    const double *tcat;               // [n_pad][SKP]
    const double *Mq;                 // [n_query][3][S][K][K]
    const int32_t *qrank;             // [n_query]
    const int32_t *active;            // [n_active] queries this pass sweeps, ascending
    const long long *item_start;      // [n_active + 1] first work item of each
    long long n_items;
    const Sel *sel;                   // [n_query]
    const unsigned long long *known;  // sorted packed rank triples
    long long n_known;
    int n_active;
    unsigned long long *counter;      // [n_query] entries kept
    unsigned long long *cursor;       // work-item cursor
    unsigned long long *hist;         // [n_active][kPredBins + 1]
    unsigned long long *out_bits, *out_packed;   // [n_query][cap]
    long long cap;
};

// work items are (query, region, 64-row tile), query-major, so a CTA flushes its shared histogram when the query changes
__global__ void __launch_bounds__(kPredThreads, 4) tip_query_pass_kernel(QueryPassArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP);
    double *Q = reinterpret_cast<double *>(smem);                                   // [64][qs]
    unsigned *sh_hist = reinterpret_cast<unsigned *>(Q + (size_t)kPredRows * qs);  // [kPredBins + 1]
    __shared__ long long sh_item;
    __shared__ Sel sh_sel;       // the item's threshold and geometry: CTA-uniform, read from shared memory in the epilogue
    __shared__ TileMap sh_tm;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    for (int i = tid; i <= kPredBins; i += kPredThreads) sh_hist[i] = 0;
    double since_flush = 0.0;   // as in tip_predict_pass_kernel
    int cur = -1;               // active slot whose entries sh_hist holds (CTA-uniform)
    const int n = A.n, SKP = A.SKP, K = A.K;
    const long long KK = (long long)K * K;

    for (;;) {
        __syncthreads();   // Q, sh_item and sh_hist of the previous item are no longer used
        if (tid == 0) sh_item = (long long)atomicAdd(A.cursor, 1ull);
        __syncthreads();
        const long long item = sh_item;
        if (item >= A.n_items) break;
        int al = 0, ah = A.n_active - 1;
        while (al < ah) {
            const int mid = (al + ah + 1) >> 1;
            if (A.item_start[mid] <= item) al = mid; else ah = mid - 1;
        }
        if (al != cur || since_flush > 2.0e9) {
            if (cur >= 0) flush_hist(sh_hist, A.hist + (long long)cur * (kPredBins + 1));
            cur = al;
            since_flush = 0.0;
        }
        const int qi = A.active[al], r = A.qrank[qi];
        int tc, tb, ta;
        query_tiles(n, r, tc, tb, ta);
        int t = (int)(item - A.item_start[al]);
        int g, a0, col0;
        TileMap tm;
        if (t < tc) {
            g = 0; a0 = t * kPredRows; col0 = a0 + 1;
            tm = TileMap{r - 1, r, true, 2 * kRankBits, kRankBits, (unsigned long long)r};
        } else if ((t -= tc) < tb) {
            g = 1; a0 = t * kPredRows; col0 = r + 1;
            tm = TileMap{r, n, false, 2 * kRankBits, 0, (unsigned long long)r << kRankBits};
        } else {
            t -= tb;
            g = 2; a0 = r + 1 + t * kPredRows; col0 = a0 + 1;
            tm = TileMap{n - 1, n, true, kRankBits, 0, (unsigned long long)r << (2 * kRankBits)};
        }
        const int rows = min(kPredRows, tm.row_end - a0);
        if (tid == 0) {
            sh_sel = A.sel[qi];
            sh_tm = tm;
        }

        form_q_tile(Q, qs, A.tcat, SKP, A.SK, K, a0, rows, A.Mq + ((long long)qi * 3 + g) * A.S * KK, KK);
        __syncthreads();

        if (wr * 32 < rows) {
            const double *Qw = Q + (wr * 32 + gq) * qs + tq;
            for (int c0 = col0 + wc * 32; c0 < tm.col_end; c0 += 64) {
                double acc[4][4][2];
                dmma_block(acc, Qw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                select_block(acc, sh_sel, sh_tm, lane, a0 + wr * 32 + gq, c0 + 2 * tq, A.known, A.n_known, sh_hist, A.counter + qi,
                             A.out_bits + (long long)qi * A.cap, A.out_packed + (long long)qi * A.cap, A.cap);
            }
        }
        since_flush += (double)rows * (tm.col_end - col0);
    }
    if (cur >= 0) flush_hist(sh_hist, A.hist + (long long)cur * (kPredBins + 1));
}

__global__ void tip_query_finish_kernel(int n_query, int N, long long cap, int S, const long long *__restrict__ m_rows,
                                        const unsigned long long *__restrict__ bits, const unsigned long long *__restrict__ packed,
                                        const int32_t *__restrict__ cand, int32_t *__restrict__ out_ids, double *__restrict__ out_scores)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_query * N) return;
    const long long qi = i / N, t = i % N;
    if (t >= m_rows[qi]) return;
    const long long src = qi * cap + t;
    const unsigned long long pk = packed[src], mask = (1ull << kRankBits) - 1;
    out_ids[3 * i + 0] = cand[(pk >> (2 * kRankBits)) & mask];
    out_ids[3 * i + 1] = cand[(pk >> kRankBits) & mask];
    out_ids[3 * i + 2] = cand[pk & mask];
    out_scores[i] = __longlong_as_double((long long)bits[src]) / (double)S;
}


__global__ void tip_predict_finish_kernel(long long m, int S, const unsigned long long *__restrict__ bits,
                                          const unsigned long long *__restrict__ packed, const int32_t *__restrict__ cand,
                                          int32_t *__restrict__ out_ids, double *__restrict__ out_scores)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const unsigned long long pk = packed[i], mask = (1ull << kRankBits) - 1;
    out_ids[3 * i + 0] = cand[(pk >> (2 * kRankBits)) & mask];
    out_ids[3 * i + 1] = cand[(pk >> kRankBits) & mask];
    out_ids[3 * i + 2] = cand[pk & mask];
    out_scores[i] = __longlong_as_double((long long)bits[i]) / (double)S;
}

inline size_t a256(size_t b) { return (b + 255) / 256 * 256; }

long long n_triplets(long long n) { return n < 3 ? 0 : n * (n - 1) / 2 * (n - 2) / 3; }

long long capacity(long long n, long long N)
{
    const long long total = n_triplets(n);
    const long long want = 4 * N + (1ll << 18);
    return std::max(1ll, std::min(total, want));
}

struct Layout {
    size_t o_tcat, o_W, o_samp, o_samp2, o_bits, o_pk, o_bits2, o_pk2, o_hist, o_cnt, o_cub, cub_bytes, total;
    int n_pad, SKP;
    long long cap;
};

Layout layout(int n, int K, int S, long long N)
{
    Layout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.cap = capacity(n, N);
    size_t cb1 = 0, cb2 = 0, cb3 = 0;
    cub::DeviceRadixSort::SortKeysDescending(nullptr, cb1, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                             kPredSample, 0, 64, (cudaStream_t)0);
    cub::DeviceRadixSort::SortPairs(nullptr, cb2, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)std::min<long long>(L.cap, 1ll << 30),
                                    0, 64, (cudaStream_t)0);
    cub::DeviceRadixSort::SortPairsDescending(nullptr, cb3, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                              (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                              (int)std::min<long long>(L.cap, 1ll << 30), 0, 64, (cudaStream_t)0);
    L.cub_bytes = std::max(cb1, std::max(cb2, cb3));
    size_t off = 0;
    L.o_tcat = off; off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_W = off;    off += a256((size_t)S * n * K * K * 8);
    L.o_samp = off; off += a256((size_t)kPredSample * 8);
    L.o_samp2 = off; off += a256((size_t)kPredSample * 8);
    L.o_bits = off; off += a256((size_t)L.cap * 8);
    L.o_pk = off;   off += a256((size_t)L.cap * 8);
    L.o_bits2 = off; off += a256((size_t)L.cap * 8);
    L.o_pk2 = off;  off += a256((size_t)L.cap * 8);
    L.o_hist = off; off += a256((size_t)(kPredBins + 1) * 8);
    L.o_cnt = off;  off += 256;
    L.o_cub = off;  off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

int shift_for(unsigned long long span)
{
    int s = 0;
    while (s < 64 && (span >> s) >= (unsigned long long)kPredBins) ++s;
    return s;
}

// One narrowing step after a pass that kept more than cap entries, at least M of them needed: walk the pass's histogram in
// result order to the bin where the count reaches M and set the next pass's threshold from it.  Under ties (a bin one score
// wide that still holds too many) the selection continues on the packed ranks.  false: the histogram does not reach M.
bool narrow(Sel &sel, long long M, long long cap, const unsigned long long *hist, unsigned long long max_packed)
{
    long long cum = (long long)hist[kPredBins];
    if (sel.mode == 0 && cum >= M) {
        // everything needed lies above the histogram's range
        sel.lo = sel.hi + 1;
        sel.hi = kInfBits;
        sel.shift = shift_for(sel.hi - sel.lo);
        return true;
    }
    int b = 0;
    for (; b < kPredBins; ++b) {
        cum += (long long)hist[b];
        if (cum >= M) break;
    }
    if (b == kPredBins) return false;
    if (sel.mode == 0) {
        const unsigned long long top = sel.hi - ((unsigned long long)b << sel.shift);
        const unsigned long long width = (sel.shift >= 64) ? ~0ull : (1ull << sel.shift);
        const unsigned long long bottom = (top - sel.lo + 1 <= width) ? sel.lo : top - width + 1;
        if (cum <= cap) {
            sel.lo = bottom;
        } else if (bottom == top) {
            // every remaining candidate has the same score: continue on the packed ranks
            sel.mode = 1;
            sel.v = top;
            sel.rlo = 0;
            sel.rhi = max_packed;
        } else {
            sel.lo = bottom;
            sel.hi = top;
        }
    } else {
        const unsigned long long lo_b = sel.rlo + ((unsigned long long)b << sel.shift);
        const unsigned long long hi_b = std::min(sel.rhi, lo_b + ((sel.shift >= 64) ? ~0ull : (1ull << sel.shift) - 1));
        if (cum <= cap) {
            sel.rhi = hi_b;
        } else {
            sel.rlo = lo_b;
            sel.rhi = hi_b;
        }
    }
    sel.shift = sel.mode == 0 ? shift_for(sel.hi - sel.lo) : shift_for(sel.rhi - sel.rlo);
    return true;
}

}  // namespace
}  // namespace tip

using namespace tip;

static thread_local int g_last_passes = 0;

static bool predict_args_ok(int n_cand, int K, int S, int64_t n_known, int64_t N)
{
    return n_cand >= 0 && n_cand <= (1 << kRankBits) && K >= 1 && K <= TIP_MAX_K && S >= 1 && (long long)S * K <= kPredMaxSK &&
           n_known >= 0 && N >= 0 && N < (1ll << 28);
}

extern "C" int tip_top_triplets_workspace_bytes(int n_cand, int K, int S, int64_t n_known, int64_t N, size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && predict_args_ok(n_cand, K, S, n_known, N),
                "tip_top_triplets_workspace_bytes: bad arguments (n_cand <= 2^21, 1 <= K <= %d, S >= 1, S*K <= %d, "
                "0 <= N < 2^28)", TIP_MAX_K, kPredMaxSK);
    *bytes = layout(n_cand, K, S, N).total;
    return 0;
}

extern "C" int tip_top_triplets(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand,
                                int n_cand, const uint64_t *d_known, int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes,
                                int32_t *d_out_ids, double *d_out_scores, int64_t *h_n_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && predict_args_ok(n_cand, K, S, n_known, N) && h_n_out != nullptr,
                "tip_top_triplets: bad arguments (P > 0, n_cand <= min(P, 2^21), 1 <= K <= %d, S >= 1, S*K <= %d, "
                "n_known >= 0, 0 <= N < 2^28)", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && (d_known || n_known == 0) &&
                    (N == 0 || (d_out_ids && d_out_scores)),
                "tip_top_triplets: null pointer");
    *h_n_out = 0;
    g_last_passes = 0;
    const int n = n_cand;
    const long long total = n_triplets(n);
    TIP_REQUIRE(n_known <= total, "tip_top_triplets: more known keys (%lld) than candidate triplets (%lld)",
                (long long)n_known, total);
    long long M = std::min<long long>(N, total - n_known);
    if (M <= 0) return 0;
    const Layout L = layout(n, K, S, N);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_top_triplets: workspace too small (%zu < %zu)", ws_bytes, L.total);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *W = reinterpret_cast<double *>(base + L.o_W);
    auto *samp = reinterpret_cast<unsigned long long *>(base + L.o_samp), *samp2 = reinterpret_cast<unsigned long long *>(base + L.o_samp2);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits), *pk = reinterpret_cast<unsigned long long *>(base + L.o_pk);
    auto *bits2 = reinterpret_cast<unsigned long long *>(base + L.o_bits2), *pk2 = reinterpret_cast<unsigned long long *>(base + L.o_pk2);
    auto *hist = reinterpret_cast<unsigned long long *>(base + L.o_hist), *cnt = reinterpret_cast<unsigned long long *>(base + L.o_cnt);
    void *cub_tmp = base + L.o_cub;

    {
        const long long work = (long long)L.n_pad * L.SKP + (long long)S * n * K * K;
        const long long want = (work + 255) / 256;
        tip_predict_prep_kernel<<<(int)std::min<long long>(want, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, d_theta, d_p, d_cand, tcat, W);
        TIP_CHECK_CUDA(cudaGetLastError());
    }

    // a pass: recompute every score, keep those the threshold lets through
    const size_t smem = (size_t)kPredRows * q_stride(L.SKP) * 8 + (size_t)(kPredBins + 1) * 4;
    static int smem_set = 0;
    if ((int)smem > smem_set && smem > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_predict_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = (int)smem;
    }
    int per_sm = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tip_predict_pass_kernel, kPredThreads, smem));
    TIP_REQUIRE(per_sm > 0, "tip_top_triplets: S*K = %d does not fit one block's shared memory", S * K);
    PassArgs A{};
    A.n = n; A.S = S; A.K = K; A.SK = S * K; A.SKP = L.SKP;
    A.tcat = tcat; A.W = W; A.known = reinterpret_cast<const unsigned long long *>(d_known); A.n_known = n_known;
    A.n_items = items_before(n - 1);   // middle ranks 1 .. n-2
    A.counter = cnt; A.hist = hist; A.out_bits = bits; A.out_packed = pk; A.cap = L.cap;
    const long long grid_l = std::min<long long>((long long)sm_count() * per_sm, A.n_items);
    std::vector<unsigned long long> h_hist(kPredBins + 1);
    unsigned long long h_cnt[2];
    auto run_pass = [&]() -> int {
        TIP_CHECK_CUDA(cudaMemsetAsync(cnt, 0, 16, st));
        TIP_CHECK_CUDA(cudaMemsetAsync(hist, 0, (kPredBins + 1) * 8, st));
        tip_predict_pass_kernel<<<(int)grid_l, kPredThreads, smem, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_cnt, cnt, 16, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_hist.data(), hist, (kPredBins + 1) * 8, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    };

    // first threshold: everything when it fits the buffer, else a quantile of a deterministic sample
    A.sel.mode = 0;
    A.sel.hi = kInfBits;
    A.sel.lo = 0;
    long long samp_idx = -1;
    unsigned long long *samp_sorted = samp2;
    auto sample_at = [&](long long idx, unsigned long long *v) -> int {
        TIP_CHECK_CUDA(cudaMemcpyAsync(v, samp_sorted + idx, 8, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    };
    if (total > L.cap) {
        tip_predict_sample_kernel<<<(kPredSample + 255) / 256, 256, 0, st>>>(n, S, K, L.SKP, tcat, W, kPredSample, samp);
        TIP_CHECK_CUDA(cudaGetLastError());
        size_t cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortKeysDescending(cub_tmp, cb, samp, samp2, kPredSample, 0, 64, st));
        // expected survivors ~2 M: well inside the buffer (4 N + 2^18)
        samp_idx = (long long)((double)(2 * M) / (double)total * kPredSample);
        if (samp_idx < kPredSample) {
            int rc = sample_at(samp_idx, &A.sel.lo);
            if (rc) return rc;
            rc = sample_at(0, &A.sel.hi);
            if (rc) return rc;
        }
    }
    A.sel.shift = shift_for(A.sel.hi - A.sel.lo);

    const unsigned long long max_packed = ((unsigned long long)(n - 1) << (2 * kRankBits)) | ((unsigned long long)(n - 1) << kRankBits) |
                                          (unsigned long long)(n - 1);
    long long kept = -1;
    for (int pass = 0; pass < 200; ++pass) {
        int rc = run_pass();
        if (rc) return rc;
        ++g_last_passes;
        const long long C = (long long)h_cnt[0];
        if (C >= M && C <= L.cap) { kept = C; break; }
        if (C < M) {
            if (A.sel.mode == 0 && A.sel.lo == 0) { M = C; kept = C; break; }   // every candidate is in the buffer
            // the sample placed the threshold too high: lower it to a sample value below it, or to zero
            unsigned long long v = A.sel.lo;
            while (v >= A.sel.lo) {
                samp_idx = samp_idx < 0 ? 0 : samp_idx * 4 + 16;
                if (samp_idx >= kPredSample) { v = 0; break; }
                if ((rc = sample_at(samp_idx, &v))) return rc;
            }
            A.sel.lo = v;
            A.sel.shift = shift_for(A.sel.hi - A.sel.lo);
            continue;
        }
        // too many for the buffer
        TIP_REQUIRE(narrow(A.sel, M, L.cap, h_hist.data(), max_packed),
                    "tip_top_triplets: histogram does not reach N (internal error)");
    }
    TIP_REQUIRE(kept >= 0, "tip_top_triplets: the threshold did not converge (internal error)");
    if (M <= 0) return 0;
    // order: packed ranks ascending, then (stable) score descending
    size_t cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, pk, pk2, bits, bits2, (int)kept, 0, 64, st));
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(cub_tmp, cb, bits2, bits, pk2, pk, (int)kept, 0, 64, st));
    tip_predict_finish_kernel<<<(int)((M + 255) / 256), 256, 0, st>>>(M, S, bits, pk, d_cand, d_out_ids, d_out_scores);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    *h_n_out = M;
    return 0;
}

extern "C" int tip_top_triplets_last_passes(void) { return g_last_passes; }

// ---- tip_top_triplets_per_gene ----
namespace tip {
namespace {

constexpr long long kQueryMaxRows = 1ll << 24;   // n_query * N

long long n_pairs(long long m) { return m < 2 ? 0 : m * (m - 1) / 2; }

// buffer of a query: room for 4 N survivors plus slack, never more than its pairs
long long query_capacity(int n, long long N) { return std::max(1ll, std::min(n_pairs(n - 1), 4 * N + 256)); }

struct QueryLayout {
    size_t o_tcat, o_M, o_T, o_bound, o_best, o_sel, o_active, o_start, o_cnt, o_mrows, o_beg, o_end, o_hist, o_bits, o_pk, o_bits2,
        o_pk2, o_cub, cub_bytes, total;
    int n_pad, SKP;
    long long cap;
};

QueryLayout query_layout(int n, int n_query, int K, int S, long long N)
{
    QueryLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.cap = query_capacity(n, N);
    const long long items = (long long)n_query * L.cap;
    size_t cb1 = 0, cb2 = 0;
    cub::DeviceSegmentedSort::StableSortPairs(nullptr, cb1, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                              (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)items,
                                              n_query, (const int *)nullptr, (const int *)nullptr, (cudaStream_t)0);
    cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, cb2, (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (int)items, n_query, (const int *)nullptr,
                                                        (const int *)nullptr, (cudaStream_t)0);
    L.cub_bytes = std::max(cb1, cb2);
    const size_t nq = (size_t)n_query;
    size_t off = 0;
    L.o_tcat = off;   off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_M = off;      off += a256(nq * 3 * S * K * K * 8);
    L.o_T = off;      off += a256((size_t)S * 8);
    L.o_bound = off;  off += a256(nq * 8);
    L.o_best = off;   off += a256(nq * 8);
    L.o_sel = off;    off += a256(nq * sizeof(Sel));
    L.o_active = off; off += a256(nq * 4);
    L.o_start = off;  off += a256((nq + 1) * 8);
    L.o_cnt = off;    off += a256((nq + 1) * 8);
    L.o_mrows = off;  off += a256(nq * 8);
    L.o_beg = off;    off += a256(nq * 4);
    L.o_end = off;    off += a256(nq * 4);
    L.o_hist = off;   off += a256(nq * (kPredBins + 1) * 8);
    L.o_bits = off;   off += a256((size_t)items * 8);
    L.o_pk = off;     off += a256((size_t)items * 8);
    L.o_bits2 = off;  off += a256((size_t)items * 8);
    L.o_pk2 = off;    off += a256((size_t)items * 8);
    L.o_cub = off;    off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

}  // namespace
}  // namespace tip

static thread_local int g_last_query_passes = 0;

static bool per_gene_args_ok(int n_cand, int n_query, int K, int S, int64_t n_known, int64_t N)
{
    return predict_args_ok(n_cand, K, S, n_known, N) && n_query >= 0 && n_query <= n_cand &&
           (long long)n_query * N <= kQueryMaxRows;
}

extern "C" int tip_top_triplets_per_gene_workspace_bytes(int n_cand, int n_query, int K, int S, int64_t n_known, int64_t N,
                                                         size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && per_gene_args_ok(n_cand, n_query, K, S, n_known, N),
                "tip_top_triplets_per_gene_workspace_bytes: bad arguments (n_cand <= 2^21, 0 <= n_query <= n_cand, "
                "1 <= K <= %d, S >= 1, S*K <= %d, N >= 0, n_query*N <= 2^24)", TIP_MAX_K, kPredMaxSK);
    *bytes = query_layout(n_cand, n_query, K, S, N).total;
    return 0;
}

extern "C" int tip_top_triplets_per_gene(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand,
                                         int n_cand, const int32_t *d_query_ranks, int n_query, const uint64_t *d_known,
                                         int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes, int32_t *d_out_ids,
                                         double *d_out_scores, int64_t *h_n_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && per_gene_args_ok(n_cand, n_query, K, S, n_known, N) && (h_n_out || n_query == 0),
                "tip_top_triplets_per_gene: bad arguments (P > 0, n_cand <= min(P, 2^21), 0 <= n_query <= n_cand, "
                "1 <= K <= %d, S >= 1, S*K <= %d, n_known >= 0, N >= 0, n_query*N <= 2^24)", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && (d_query_ranks || n_query == 0) && (d_known || n_known == 0) &&
                    (N == 0 || n_query == 0 || (d_out_ids && d_out_scores)),
                "tip_top_triplets_per_gene: null pointer");
    g_last_query_passes = 0;
    if (n_query == 0) return 0;
    const int n = n_cand, nq = n_query;
    // the query ranks are checked on the host before any device work
    std::vector<int32_t> qr(nq);
    TIP_CHECK_CUDA(cudaMemcpyAsync(qr.data(), d_query_ranks, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    {
        std::vector<char> seen(n, 0);
        for (int i = 0; i < nq; ++i) {
            TIP_REQUIRE(qr[i] >= 0 && qr[i] < n, "tip_top_triplets_per_gene: query rank %d of query %d is not in [0, %d)", qr[i],
                        i, n);
            TIP_REQUIRE(!seen[qr[i]], "tip_top_triplets_per_gene: query rank %d appears twice", qr[i]);
            seen[qr[i]] = 1;
        }
    }
    for (int i = 0; i < nq; ++i) h_n_out[i] = 0;
    const long long pairs = n_pairs(n - 1);
    if (N == 0 || pairs == 0) return 0;
    const QueryLayout L = query_layout(n, nq, K, S, N);
    // sample size per query: about 4 N of its pairs score above the sample's best, at most 4096 samples
    const int n_samp = (int)std::max(1ll, std::min(4096ll, pairs / (4 * std::min<long long>(N, pairs))));
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_top_triplets_per_gene: workspace too small (%zu < %zu)", ws_bytes,
                L.total);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *Mq = reinterpret_cast<double *>(base + L.o_M);
    auto *T = reinterpret_cast<unsigned long long *>(base + L.o_T);
    double *bound = reinterpret_cast<double *>(base + L.o_bound);
    auto *best = reinterpret_cast<unsigned long long *>(base + L.o_best);
    Sel *d_sel = reinterpret_cast<Sel *>(base + L.o_sel);
    auto *d_active = reinterpret_cast<int32_t *>(base + L.o_active);
    auto *d_start = reinterpret_cast<long long *>(base + L.o_start);
    auto *cnt = reinterpret_cast<unsigned long long *>(base + L.o_cnt);
    auto *d_mrows = reinterpret_cast<long long *>(base + L.o_mrows);
    auto *d_beg = reinterpret_cast<int *>(base + L.o_beg), *d_end = reinterpret_cast<int *>(base + L.o_end);
    auto *hist = reinterpret_cast<unsigned long long *>(base + L.o_hist);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits), *pk = reinterpret_cast<unsigned long long *>(base + L.o_pk);
    auto *bits2 = reinterpret_cast<unsigned long long *>(base + L.o_bits2), *pk2 = reinterpret_cast<unsigned long long *>(base + L.o_pk2);
    void *cub_tmp = base + L.o_cub;

    {
        const long long work = (long long)L.n_pad * L.SKP + (long long)nq * 3 * S * K * K;
        const long long want = (work + 255) / 256;
        tip_query_prep_kernel<<<(int)std::min<long long>(want, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, nq, d_theta, d_p, d_cand, d_query_ranks, tcat, Mq);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaMemsetAsync(T, 0, (size_t)S * 8, st));
        tip_query_rowsum_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, S, K, L.SKP, tcat, T);
        TIP_CHECK_CUDA(cudaGetLastError());
        tip_query_bound_kernel<<<(nq + 127) / 128, 128, 0, st>>>(nq, S, K, Mq, T, bound);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaMemsetAsync(best, 0, (size_t)nq * 8, st));
        if (pairs > L.cap) {
            const long long work = (long long)nq * n_samp;
            tip_query_sample_kernel<<<(int)((work + 255) / 256), 256, 0, st>>>(n, S, K, L.SKP, nq, n_samp, d_query_ranks, tcat,
                                                                                 Mq, best);
            TIP_CHECK_CUDA(cudaGetLastError());
        }
    }
    std::vector<double> h_bound(nq);
    std::vector<unsigned long long> h_best(nq);
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_bound.data(), bound, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_best.data(), best, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));

    const size_t smem = (size_t)kPredRows * q_stride(L.SKP) * 8 + (size_t)(kPredBins + 1) * 4;
    static int smem_set = 0;
    if ((int)smem > smem_set && smem > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_query_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = (int)smem;
    }
    int per_sm = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tip_query_pass_kernel, kPredThreads, smem));
    TIP_REQUIRE(per_sm > 0, "tip_top_triplets_per_gene: S*K = %d does not fit one block's shared memory", S * K);

    // first threshold of each query: everything when its pairs fit its buffer; else the best score of its sample, with the
    // histogram spanning up to an upper bound of its scores.  Neither has to be right: entries above the bound are counted
    // ahead of the range, and a threshold that keeps fewer than N moves down in a later pass; they set how many passes it
    // takes, not the result
    std::vector<Sel> sel(nq);
    std::vector<long long> M(nq), kept(nq, -1);
    for (int i = 0; i < nq; ++i) {
        Sel &q = sel[i];
        q = Sel{};
        q.hi = kInfBits;
        M[i] = std::min<long long>(N, pairs);
        if (pairs > L.cap) {
            const double hb = h_bound[i] * (1.0 + 1e-9);
            q.hi = std::min<unsigned long long>((unsigned long long)__builtin_bit_cast(long long, hb), kInfBits);
            q.lo = std::min(h_best[i], q.hi);
        }
        q.shift = shift_for(q.hi - q.lo);
    }
    const unsigned long long max_packed = ((unsigned long long)(n - 1) << (2 * kRankBits)) | ((unsigned long long)(n - 1) << kRankBits) |
                                          (unsigned long long)(n - 1);
    QueryPassArgs A{};
    A.n = n; A.S = S; A.K = K; A.SK = S * K; A.SKP = L.SKP;
    A.tcat = tcat; A.Mq = Mq; A.qrank = d_query_ranks; A.active = d_active; A.item_start = d_start; A.sel = d_sel;
    A.known = reinterpret_cast<const unsigned long long *>(d_known); A.n_known = n_known;
    A.counter = cnt; A.cursor = cnt + nq; A.hist = hist; A.out_bits = bits; A.out_packed = pk; A.cap = L.cap;
    std::vector<int32_t> active;
    std::vector<long long> start;
    std::vector<unsigned long long> h_cnt(nq), h_hist;
    for (int pass = 0;; ++pass) {
        active.clear();
        start.assign(1, 0);
        for (int i = 0; i < nq; ++i) {
            if (kept[i] >= 0) continue;
            int tc, tb, ta;
            query_tiles(n, qr[i], tc, tb, ta);
            active.push_back(i);
            start.push_back(start.back() + tc + tb + ta);
        }
        if (active.empty()) break;
        TIP_REQUIRE(pass < 200, "tip_top_triplets_per_gene: the threshold did not converge (internal error)");
        const int na = (int)active.size();
        A.n_active = na;
        A.n_items = start.back();
        TIP_CHECK_CUDA(cudaMemcpyAsync(d_sel, sel.data(), (size_t)nq * sizeof(Sel), cudaMemcpyHostToDevice, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(d_active, active.data(), (size_t)na * 4, cudaMemcpyHostToDevice, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(d_start, start.data(), (size_t)(na + 1) * 8, cudaMemcpyHostToDevice, st));
        TIP_CHECK_CUDA(cudaMemsetAsync(cnt, 0, (size_t)(nq + 1) * 8, st));
        TIP_CHECK_CUDA(cudaMemsetAsync(hist, 0, (size_t)na * (kPredBins + 1) * 8, st));
        const long long grid_l = std::min<long long>((long long)sm_count() * per_sm, A.n_items);
        tip_query_pass_kernel<<<(int)grid_l, kPredThreads, smem, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
        h_hist.resize((size_t)na * (kPredBins + 1));
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_cnt.data(), cnt, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_hist.data(), hist, h_hist.size() * 8, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        ++g_last_query_passes;
        for (int a = 0; a < na; ++a) {
            const int i = active[a];
            Sel &q = sel[i];
            const long long C = (long long)h_cnt[i];
            if (C >= M[i] && C <= L.cap) { kept[i] = C; continue; }
            if (C < M[i]) {
                if (q.mode == 0 && q.lo == 0) { M[i] = C; kept[i] = C; continue; }   // every candidate is in the buffer
                // the threshold was too high: move it 16 binades down (to zero below the normal range)
                q.lo = q.lo > (16ull << 52) ? q.lo - (16ull << 52) : 0;
                q.shift = shift_for(q.hi - q.lo);
                continue;
            }
            TIP_REQUIRE(narrow(q, M[i], L.cap, h_hist.data() + (size_t)a * (kPredBins + 1), max_packed),
                        "tip_top_triplets_per_gene: histogram does not reach N (internal error)");
        }
    }
    // order: per query, packed ranks ascending, then (stable) score descending
    std::vector<int> beg(nq), end(nq);
    for (int i = 0; i < nq; ++i) {
        beg[i] = (int)((long long)i * L.cap);
        end[i] = beg[i] + (int)kept[i];
    }
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_beg, beg.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_end, end.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_mrows, M.data(), (size_t)nq * 8, cudaMemcpyHostToDevice, st));
    const int items = (int)((long long)nq * L.cap);
    size_t cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceSegmentedSort::StableSortPairs(cub_tmp, cb, pk, pk2, bits, bits2, items, nq, d_beg, d_end, st));
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(
        cub::DeviceSegmentedSort::StableSortPairsDescending(cub_tmp, cb, bits2, bits, pk2, pk, items, nq, d_beg, d_end, st));
    const long long rows = (long long)nq * N;
    tip_query_finish_kernel<<<(int)((rows + 255) / 256), 256, 0, st>>>(nq, (int)N, L.cap, S, d_mrows, bits, pk, d_cand,
                                                                         d_out_ids, d_out_scores);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < nq; ++i) h_n_out[i] = M[i];
    return 0;
}

extern "C" int tip_top_triplets_per_gene_last_passes(void) { return g_last_query_passes; }

// ---- tip_top_triplets_per_pair ----
// A query pair of ranks ra < rb and a partner of rank rc: the triplet's slots follow from rc (rc < ra: (c, a, b); ra < rc < rb:
// (a, c, b); rc > rb: (a, b, c)), and its score is th_c . V_g with, per set (M_0, M_1 of gene b as tip_query_prep_kernel forms
// them, so K^2 per pair and vector entry)
//     V_0[x] = sum_y M_0[x][y] th_a[y],   V_1[y] = sum_x th_a[x] M_0[x][y],   V_2[z] = sum_x th_a[x] M_1[x][z]
// The pairs are sorted by (ra, rb) on the device; a work item is a tile of 64 of them, swept over the columns in three phases,
// one per region, each loading that region's V rows as the A tile of dmma_block; the epilogue masks each row to its region.
// A CTA owns its rows for the whole sweep, so selection is CTA-local: each row's histogram lives in shared memory, and at the
// end of the tile the CTA sets the row's next threshold from it.  First sweep: count every score in a range just below the
// row's upper bound (known triplets included: the row's count of known triplets is added to what it needs).  Second: keep
// the unknown scores at or above the boundary bin, appended to the row's slice of a buffer.  A row whose slice overflows
// narrows as narrow() does, continuing on rc under ties, and is swept again.
namespace tip {
namespace {

constexpr long long kPairMaxRows = 1ll << 24;           // n_pairs * N
constexpr unsigned long long kPairSpan = 4ull << 52;    // first histogram range: 4 binades below the row's bound

// selection state of one pair
struct PairSel {
    int state;                      // 0: count bits in [lo, hi] (histogram only); 1: keep bits >= lo; 2: keep bits > v, or
                                    // bits == v and rc <= rhi; 3: resolved
    int shift;
    int rlo, rhi;                   // state 2: histogram range of rc (bin 0 = lowest)
    unsigned long long lo, hi, v;   // states 0, 1: histogram range of score bits (bin 0 = highest); state 2: tied score bits
};

__host__ __device__ inline int pair_shift(unsigned long long span, int nb)
{
    int s = 0;
    while (s < 64 && (span >> s) >= (unsigned long long)nb) ++s;
    return s;
}

// sort keys (ra << 21) | rb with ra < rb, and the caller's index
__global__ void tip_pair_keys_kernel(long long n_pairs, const int32_t *__restrict__ pr, unsigned long long *__restrict__ key,
                                     int32_t *__restrict__ idx)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    const int a = min(pr[2 * i], pr[2 * i + 1]), b = max(pr[2 * i], pr[2 * i + 1]);
    key[i] = ((unsigned long long)a << kRankBits) | (unsigned long long)b;
    idx[i] = (int32_t)i;
}

// per sorted pair: its ranks; active[i] = i lists every tile for the first sweep (there are fewer tiles than pairs)
__global__ void tip_pair_split_kernel(long long n_pairs, const unsigned long long *__restrict__ key, int32_t *__restrict__ ra,
                                      int32_t *__restrict__ rb, int32_t *__restrict__ active)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs) return;
    ra[i] = (int32_t)(key[i] >> kRankBits);
    rb[i] = (int32_t)(key[i] & ((1ull << kRankBits) - 1));
    active[i] = (int32_t)i;
}

// per sorted pair: its count of distinct known triplets (a known triple adds one to every pair it contains)
__global__ void tip_pair_known_kernel(long long n_known, const unsigned long long *__restrict__ known, long long n_pairs,
                                      const unsigned long long *__restrict__ key, unsigned long long *__restrict__ krow)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_known || (i > 0 && known[i] == known[i - 1])) return;   // a repeated key counts once
    const unsigned long long k = known[i], m = (1ull << kRankBits) - 1;
    const unsigned long long r0 = (k >> (2 * kRankBits)) & m, r1 = (k >> kRankBits) & m, r2 = k & m;
    const unsigned long long want[3] = {(r0 << kRankBits) | r1, (r0 << kRankBits) | r2, (r1 << kRankBits) | r2};
    for (int w = 0; w < 3; ++w) {
        long long lo = 0, hi = n_pairs;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (key[mid] < want[w]) lo = mid + 1; else hi = mid;
        }
        for (; lo < n_pairs && key[lo] == want[w]; ++lo) atomicAdd(krow + lo, 1ull);
    }
}

// V[pair][g][s K + x] for the pairs whose gene b is one of the chunk's genes [c0, c1) (Mq of the chunk, local index)
__global__ void tip_pair_vec_kernel(long long n_pairs, int S, int K, int SKP, int c0, int c1, const int32_t *__restrict__ bidx,
                                    const int32_t *__restrict__ ra, const int32_t *__restrict__ rb, const double *__restrict__ tcat,
                                    const double *__restrict__ Mq, double *__restrict__ V)
{
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_pairs * 3 * SKP) return;
    const long long p = t / (3 * SKP);
    const int g = (int)(t / SKP % 3), col = (int)(t % SKP);
    const int u = bidx[rb[p]];
    if (u < c0 || u >= c1) return;
    double acc = 0.0;
    if (col < S * K) {
        const int s = col / K, x = col % K;
        const long long KK = (long long)K * K;
        const double *th = tcat + (long long)ra[p] * SKP + s * K;
        const double *M = Mq + (((long long)(u - c0) * 3 + (g == 2 ? 1 : 0)) * S + s) * KK;
        if (g == 0) {
            for (int y = 0; y < K; ++y) acc = fma(M[x * K + y], th[y], acc);
        } else {
            for (int y = 0; y < K; ++y) acc = fma(th[y], M[y * K + x], acc);
        }
    }
    V[t] = acc;
}

// first state of every pair: rows to select (M) and to count (M + known triplets), and the first histogram range, up to
// an upper bound of the row's scores: th_c . V_s <= max(V_s) |th_c|_1 <= max(V_s) T[s] (non-negative parameters)
__global__ void tip_pair_init_kernel(long long n_pairs, int n, int S, int K, int SKP, long long N, long long cap, int nb,
                                     const double *__restrict__ V, const unsigned long long *__restrict__ T,
                                     const unsigned long long *__restrict__ krow, PairSel *__restrict__ sel,
                                     long long *__restrict__ need0, long long *__restrict__ m_rows, long long *__restrict__ kept)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const long long k = (long long)krow[p];
    const long long M = max(0ll, min(N, (long long)(n - 2) - k));
    m_rows[p] = M;
    need0[p] = M + k;
    kept[p] = 0;
    PairSel q{};
    q.hi = kInfBits;
    if (M == 0) {
        q.state = 3;
    } else if (n - 2 <= cap) {
        q.state = 1;   // every partner fits the row's slice
    } else {
        double best = 0.0;
        for (int g = 0; g < 3; ++g) {
            double b = 0.0;
            for (int s = 0; s < S; ++s) {
                double mx = 0.0;
                for (int x = 0; x < K; ++x) mx = fmax(mx, V[(p * 3 + g) * SKP + s * K + x]);
                b += mx * __longlong_as_double((long long)T[s]);
            }
            best = fmax(best, b);
        }
        q.hi = min((unsigned long long)__double_as_longlong(best * (1.0 + 1e-9)), kInfBits);
        q.lo = q.hi >= kPairSpan ? q.hi - kPairSpan + 1 : 0;
    }
    q.shift = pair_shift(q.hi - q.lo, nb);
    sel[p] = q;
}

// is_known for the pair kernel: a second call site of is_known changes the code generated for it inside the two scoring
// kernels above, so the pair kernel has its own copy
__device__ __noinline__ bool pair_is_known(const unsigned long long *known, long long n, unsigned long long key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(known + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo < n && __ldg(known + lo) == key;
}

struct PairPassArgs {
    int n, SKP, nb;
    const double *tcat;               // [n_pad][SKP]
    const double *V;                  // [n_pairs][3][SKP], sorted pair order
    const int32_t *ra, *rb;           // [n_pairs] sorted
    const int32_t *active;            // [n_active] tiles this sweep scores (tile t = sorted pairs 64 t .. 64 t + 63), ascending
    int n_active, n_pairs;
    const unsigned long long *known;  // sorted packed rank triples
    long long n_known;
    PairSel *sel;                     // [n_pairs]
    const long long *need0;           // [n_pairs] rows state 0 must reach (M + known triplets of the pair)
    long long *m_rows, *kept;         // [n_pairs]
    char *again;                      // [n_active] 1: a row of the tile is swept again
    unsigned long long *ctl;          // [0] tile cursor, [1] rows not resolved, [2] internal errors
    unsigned long long *out_bits, *out_rc;   // [n_pairs][cap]
    long long cap;
};

// epilogue of a block for phase g (i0 = the lane's first row in the tile, rc0 = its first column)
__device__ __forceinline__ void pair_select_block(const double (&acc)[4][4][2], int g, int i0, int rc0, const PairPassArgs &A,
                                                  const PairSel *sh_sel, const int *sh_ra, const int *sh_rb, const int *sh_p,
                                                  unsigned *sh_cnt, unsigned *sh_hist)
{
    const int nb = A.nb;
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) {
        const int i = i0 + mi * 8;
        const PairSel q = sh_sel[i];
        if (q.state == 3) continue;
        const int ra = sh_ra[i], rb = sh_rb[i];
        const int lo_c = g == 0 ? 0 : g == 1 ? ra + 1 : rb + 1, hi_c = g == 0 ? ra : g == 1 ? rb : A.n;
        unsigned *h = sh_hist + i * (nb + 1);
#pragma unroll
        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int rc = rc0 + ni * 8 + e;
                if (rc < lo_c || rc >= hi_c) continue;
                const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
                if (q.state == 0) {
                    if (bits >= q.lo) atomicAdd(h + (bits > q.hi ? nb : (int)((q.hi - bits) >> q.shift)), 1u);
                    continue;
                }
                if (!(q.state == 1 ? bits >= q.lo : (bits > q.v || (bits == q.v && rc <= q.rhi)))) continue;
                if (A.n_known > 0) {
                    const unsigned long long a = ra, b = rb, c = rc;
                    const unsigned long long packed = g == 0 ? (c << 42) | (a << 21) | b
                                                    : g == 1 ? (a << 42) | (c << 21) | b : (a << 42) | (b << 21) | c;
                    if (pair_is_known(A.known, A.n_known, packed)) continue;
                }
                int bin = nb;
                if (q.state == 1) {
                    if (bits <= q.hi) bin = (int)((q.hi - bits) >> q.shift);
                } else if (bits == q.v && rc >= q.rlo) {
                    bin = (rc - q.rlo) >> q.shift;
                }
                atomicAdd(h + bin, 1u);
                const unsigned idx = atomicAdd(sh_cnt + i, 1u);
                if ((long long)idx < A.cap) {
                    const long long o = (long long)sh_p[i] * A.cap + idx;
                    A.out_bits[o] = bits;
                    A.out_rc[o] = (unsigned long long)rc;
                }
            }
    }
}

// next state of a row after a sweep counted C kept entries into its histogram h: 1 resolved, 0 swept again, -1 error.
// States 1 and 2 follow narrow(); state 0 places the boundary where the count reaches need0, or, when the range does not
// reach it, counts everything below the range in the next sweep.
__device__ int narrow_pair(PairSel &q, long long C, long long need0, long long &M, long long cap, const unsigned *h, int nb, int n)
{
    const unsigned long long width = q.shift >= 64 ? ~0ull : (1ull << q.shift);
    if (q.state == 1 || q.state == 2) {
        if (C >= M && C <= cap) return 1;
        if (C < M) {
            if (q.state == 2) return -1;
            if (q.lo == 0) { M = C; return 1; }   // every unknown partner is in the slice
            q.state = 0;                          // count again, everything below this range
            q.hi = q.lo - 1;
            q.lo = 0;
            q.shift = pair_shift(q.hi - q.lo, nb);
            return 0;
        }
    }
    if (q.state == 0) {
        long long cum = h[nb];
        int b = 0;
        if (cum < need0)
            for (; b < nb; ++b)
                if ((cum += h[b]) >= need0) break;
        if (cum < need0 || b == nb) {
            if (q.lo == 0) return -1;
            q.hi = q.lo - 1;   // the range missed: the next one reaches down to zero
            q.lo = 0;
        } else if (h[nb] >= need0) {
            q.state = 1;
            q.lo = q.hi + 1;
            q.hi = kInfBits;
        } else {
            const unsigned long long top = q.hi - ((unsigned long long)b << q.shift);
            q.state = 1;
            q.lo = (top - q.lo + 1 <= width) ? q.lo : top - width + 1;
        }
        q.shift = pair_shift(q.hi - q.lo, nb);
        return 0;
    }
    // too many for the slice: the histogram holds exactly the kept entries
    long long cum = h[nb];
    if (q.state == 1 && cum >= M) {
        q.lo = q.hi + 1;
        q.hi = kInfBits;
        q.shift = pair_shift(q.hi - q.lo, nb);
        return 0;
    }
    int b = 0;
    for (; b < nb; ++b)
        if ((cum += h[b]) >= M) break;
    if (b == nb) return -1;
    if (q.state == 1) {
        const unsigned long long top = q.hi - ((unsigned long long)b << q.shift);
        const unsigned long long bottom = (top - q.lo + 1 <= width) ? q.lo : top - width + 1;
        if (cum <= cap) {
            q.lo = bottom;
        } else if (bottom == top) {
            q.state = 2;   // one score value holds too many: continue on rc
            q.v = top;
            q.rlo = 0;
            q.rhi = n - 1;
        } else {
            q.lo = bottom;
            q.hi = top;
        }
    } else {
        const long long lo_b = q.rlo + ((long long)b << q.shift);
        const int hi_b = (int)min((long long)q.rhi, lo_b + (long long)width - 1);
        if (cum > cap) q.rlo = (int)lo_b;
        q.rhi = hi_b;
    }
    q.shift = q.state == 1 ? pair_shift(q.hi - q.lo, nb) : pair_shift((unsigned long long)(q.rhi - q.rlo), nb);
    return 0;
}

// work items are the active tiles of 64 sorted pairs; every tile sweeps the columns of each region of its rows.  A tile
// holds the same rows in every sweep (resolved rows are skipped in the epilogue), so every score is computed at the same
// place in the same DMMA fragment, with the same contraction order, in every sweep
__global__ void __launch_bounds__(kPredThreads) tip_pair_pass_kernel(PairPassArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP), nb = A.nb;
    double *At = reinterpret_cast<double *>(smem);                                        // [64][qs]
    PairSel *sh_sel = reinterpret_cast<PairSel *>(At + (size_t)kPredRows * qs);          // [64]
    int *sh_ra = reinterpret_cast<int *>(sh_sel + kPredRows), *sh_rb = sh_ra + kPredRows, *sh_p = sh_rb + kPredRows;
    unsigned *sh_cnt = reinterpret_cast<unsigned *>(sh_p + kPredRows);                   // [64]
    unsigned *sh_hist = sh_cnt + kPredRows;                                                // [64][nb + 1]
    __shared__ long long sh_item;
    __shared__ int sh_range[4];   // min ra, max ra, min rb, max rb of the tile
    __shared__ int sh_again;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    const int n = A.n, SKP = A.SKP;

    for (;;) {
        __syncthreads();   // the previous tile is no longer read
        if (tid == 0) sh_item = (long long)atomicAdd(A.ctl, 1ull);
        __syncthreads();
        const long long item = sh_item;
        if (item >= A.n_active) break;
        const int t0 = A.active[item] * kPredRows, rows = min(kPredRows, A.n_pairs - t0);
        if (tid == 0) sh_again = 0;
        if (tid < kPredRows) {
            const int p = t0 + (tid < rows ? tid : 0);
            sh_p[tid] = p;
            sh_ra[tid] = A.ra[p];
            sh_rb[tid] = A.rb[p];
            PairSel q = A.sel[p];
            if (tid >= rows) q.state = 3;
            sh_sel[tid] = q;
            sh_cnt[tid] = 0;
        }
        for (int i = tid; i < kPredRows * (nb + 1); i += kPredThreads) sh_hist[i] = 0;
        __syncthreads();
        if (tid == 0) {
            int r0 = n, r1 = 0, r2 = n, r3 = 0;
            for (int i = 0; i < rows; ++i) {
                r0 = min(r0, sh_ra[i]); r1 = max(r1, sh_ra[i]);
                r2 = min(r2, sh_rb[i]); r3 = max(r3, sh_rb[i]);
            }
            sh_range[0] = r0; sh_range[1] = r1; sh_range[2] = r2; sh_range[3] = r3;
        }
        __syncthreads();

        for (int g = 0; g < 3; ++g) {
            const int col0 = g == 0 ? 0 : g == 1 ? sh_range[0] + 1 : sh_range[2] + 1;
            const int col_end = g == 0 ? sh_range[1] : g == 1 ? sh_range[3] : n;
            if (col0 >= col_end) continue;
            __syncthreads();   // the previous phase's A tile is no longer read
            for (int e = tid; e < kPredRows * SKP; e += kPredThreads) {
                const int i = e / SKP, col = e % SKP;
                At[i * qs + col] = i < rows ? __ldg(A.V + ((long long)sh_p[i] * 3 + g) * SKP + col) : 0.0;
            }
            __syncthreads();
            if (wr * 32 < rows) {
                const double *Aw = At + (wr * 32 + gq) * qs + tq;
                for (int c0 = col0 + wc * 32; c0 < col_end; c0 += 64) {
                    double acc[4][4][2];
                    dmma_block(acc, Aw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                    pair_select_block(acc, g, wr * 32 + gq, c0 + 2 * tq, A, sh_sel, sh_ra, sh_rb, sh_p, sh_cnt, sh_hist);
                }
            }
        }
        __syncthreads();
        if (tid < rows) {
            const int p = sh_p[tid];
            PairSel q = sh_sel[tid];
            long long M = A.m_rows[p];
            const long long C = sh_cnt[tid];
            int r = 1;
            if (q.state != 3) r = narrow_pair(q, C, A.need0[p], M, A.cap, sh_hist + tid * (nb + 1), nb, n);
            if (r < 0) {
                atomicAdd(A.ctl + 2, 1ull);
                r = 1;
            }
            if (r == 1 && q.state != 3) {
                q.state = 3;
                A.kept[p] = C;
                A.m_rows[p] = M;
            }
            A.sel[p] = q;
            if (r == 0) {
                sh_again = 1;
                atomicAdd(A.ctl + 1, 1ull);
            }
        }
        __syncthreads();
        if (tid == 0) A.again[item] = (char)sh_again;
    }
}

__global__ void tip_pair_segments_kernel(long long n_pairs, long long cap, const long long *__restrict__ kept, int *__restrict__ beg,
                                         int *__restrict__ end)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    beg[p] = (int)(p * cap);
    end[p] = (int)(p * cap + kept[p]);
}

// row t of sorted pair p goes to the caller's pair perm[p]; ids in slot order (ranks ascending)
__global__ void tip_pair_finish_kernel(long long n_pairs, long long N, long long cap, int S, const int32_t *__restrict__ perm,
                                       const int32_t *__restrict__ ra, const int32_t *__restrict__ rb,
                                       const long long *__restrict__ m_rows, const unsigned long long *__restrict__ bits,
                                       const unsigned long long *__restrict__ rc, const int32_t *__restrict__ cand,
                                       int32_t *__restrict__ out_ids, double *__restrict__ out_scores, int64_t *__restrict__ counts)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pairs * N) return;
    const long long p = i / N, t = i % N, o = (long long)perm[p] * N + t;
    if (t == 0) counts[perm[p]] = m_rows[p];
    if (t >= m_rows[p]) return;
    const long long src = p * cap + t;
    const int a = ra[p], b = rb[p], c = (int)rc[src];
    const int x = min(c, a), z = max(c, b), y = a + b + c - x - z;
    out_ids[3 * o + 0] = cand[x];
    out_ids[3 * o + 1] = cand[y];
    out_ids[3 * o + 2] = cand[z];
    out_scores[o] = __longlong_as_double((long long)bits[src]) / (double)S;
}

// room for 4 N survivors plus slack in a row's slice, never more than its partners
long long pair_capacity(int n, long long N) { return std::max(1ll, std::min((long long)n - 2, 4 * N + 64)); }

struct PairLayout {
    size_t o_tcat, o_M, o_T, o_key, o_key2, o_idx, o_perm, o_ra, o_rb, o_bidx, o_ub, o_krow, o_V, o_sel, o_need, o_mrows, o_kept,
        o_again, o_act, o_act2, o_nsel, o_ctl, o_beg, o_end, o_counts, o_bits, o_rc, o_bits2, o_rc2, o_cub, cub_bytes, total;
    int n_pad, SKP, chunk;
    long long cap;
};

PairLayout pair_layout(int n, long long n_pairs, int K, int S, long long N)
{
    PairLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.cap = pair_capacity(n, N);
    // genes b whose K x K matrices are formed at a time: about n S K doubles
    L.chunk = (int)std::max(1ll, std::min((long long)n, (long long)L.n_pad * L.SKP / (3ll * S * K * K)));
    const long long items = n_pairs * L.cap;
    const int np = (int)n_pairs;
    size_t cb[5] = {0, 0, 0, 0, 0};
    cub::DeviceRadixSort::SortPairs(nullptr, cb[0], (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, np, 0, 2 * kRankBits, (cudaStream_t)0);
    cub::DeviceSelect::Flagged(nullptr, cb[1], (const int32_t *)nullptr, (const char *)nullptr, (int32_t *)nullptr, (int *)nullptr,
                               np, (cudaStream_t)0);
    cub::DeviceSegmentedSort::StableSortPairs(nullptr, cb[2], (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                              (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)items, np,
                                              (const int *)nullptr, (const int *)nullptr, (cudaStream_t)0);
    cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, cb[3], (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (int)items, np, (const int *)nullptr,
                                                        (const int *)nullptr, (cudaStream_t)0);
    L.cub_bytes = *std::max_element(cb, cb + 5);
    const size_t q = (size_t)n_pairs;
    size_t off = 0;
    L.o_tcat = off;   off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_M = off;      off += a256((size_t)L.chunk * 3 * S * K * K * 8);
    L.o_T = off;      off += a256((size_t)S * 8);
    L.o_key = off;    off += a256(q * 8);
    L.o_key2 = off;   off += a256(q * 8);
    L.o_idx = off;    off += a256(q * 4);
    L.o_perm = off;   off += a256(q * 4);
    L.o_ra = off;     off += a256(q * 4);
    L.o_rb = off;     off += a256(q * 4);
    L.o_bidx = off;   off += a256((size_t)n * 4);
    L.o_ub = off;     off += a256((size_t)n * 4);
    L.o_krow = off;   off += a256(q * 8);
    L.o_V = off;      off += a256(q * 3 * L.SKP * 8);
    L.o_sel = off;    off += a256(q * sizeof(PairSel));
    L.o_need = off;   off += a256(q * 8);
    L.o_mrows = off;  off += a256(q * 8);
    L.o_kept = off;   off += a256(q * 8);
    L.o_again = off;  off += a256(q);
    L.o_act = off;    off += a256(q * 4);
    L.o_act2 = off;   off += a256(q * 4);
    L.o_nsel = off;   off += 256;
    L.o_ctl = off;    off += 256;
    L.o_beg = off;    off += a256(q * 4);
    L.o_end = off;    off += a256(q * 4);
    L.o_counts = off; off += a256(q * 8);
    L.o_bits = off;   off += a256((size_t)items * 8);
    L.o_rc = off;     off += a256((size_t)items * 8);
    L.o_bits2 = off;  off += a256((size_t)items * 8);
    L.o_rc2 = off;    off += a256((size_t)items * 8);
    L.o_cub = off;    off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

// bins per row of the shared histograms: the most of 256, 128, 64 that fit beside the A tile
size_t pair_smem(int SKP, int nb)
{
    return (size_t)kPredRows * q_stride(SKP) * 8 + (size_t)kPredRows * (sizeof(PairSel) + 16) + (size_t)kPredRows * (nb + 1) * 4;
}

}  // namespace
}  // namespace tip

static thread_local int g_last_pair_passes = 0;

static bool per_pair_args_ok(int n_cand, int64_t n_pairs, int K, int S, int64_t n_known, int64_t N)
{
    return predict_args_ok(n_cand, K, S, n_known, N) && n_pairs >= 0 && n_pairs <= kPairMaxRows &&
           (N == 0 || n_pairs <= kPairMaxRows / N);
}

extern "C" int tip_top_triplets_per_pair_workspace_bytes(int n_cand, int64_t n_pairs, int K, int S, int64_t n_known, int64_t N,
                                                         size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && per_pair_args_ok(n_cand, n_pairs, K, S, n_known, N),
                "tip_top_triplets_per_pair_workspace_bytes: bad arguments (n_cand <= 2^21, n_pairs >= 0, 1 <= K <= %d, S >= 1, "
                "S*K <= %d, N >= 0, n_pairs*N <= 2^24)", TIP_MAX_K, kPredMaxSK);
    *bytes = pair_layout(n_cand, n_pairs, K, S, N).total;
    return 0;
}

extern "C" int tip_top_triplets_per_pair(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand,
                                         int n_cand, const int32_t *d_pair_ranks, int64_t n_pairs, const uint64_t *d_known,
                                         int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes, int32_t *d_out_ids,
                                         double *d_out_scores, int64_t *h_n_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && per_pair_args_ok(n_cand, n_pairs, K, S, n_known, N) && (h_n_out || n_pairs == 0),
                "tip_top_triplets_per_pair: bad arguments (P > 0, n_cand <= min(P, 2^21), n_pairs >= 0, 1 <= K <= %d, S >= 1, "
                "S*K <= %d, n_known >= 0, N >= 0, n_pairs*N <= 2^24)", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && (d_pair_ranks || n_pairs == 0) && (d_known || n_known == 0) &&
                    (N == 0 || n_pairs == 0 || (d_out_ids && d_out_scores)),
                "tip_top_triplets_per_pair: null pointer");
    g_last_pair_passes = 0;
    if (n_pairs == 0) return 0;
    const int n = n_cand;
    const long long Q = n_pairs;
    // the pair ranks are checked on the host before any device work
    std::vector<int32_t> pr((size_t)Q * 2);
    TIP_CHECK_CUDA(cudaMemcpyAsync(pr.data(), d_pair_ranks, (size_t)Q * 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> bidx(std::max(n, 1), -1), ub;
    for (long long i = 0; i < Q; ++i) {
        for (int e = 0; e < 2; ++e)
            TIP_REQUIRE(pr[2 * i + e] >= 0 && pr[2 * i + e] < n, "tip_top_triplets_per_pair: rank %d of pair %lld is not in [0, %d)",
                        pr[2 * i + e], i, n);
        TIP_REQUIRE(pr[2 * i] != pr[2 * i + 1], "tip_top_triplets_per_pair: pair %lld has the same rank twice (%d)", i, pr[2 * i]);
        bidx[std::max(pr[2 * i], pr[2 * i + 1])] = 0;
    }
    for (long long i = 0; i < Q; ++i) h_n_out[i] = 0;
    if (N == 0 || n < 3) return 0;
    for (int r = 0; r < n; ++r)
        if (bidx[r] == 0) {
            bidx[r] = (int32_t)ub.size();
            ub.push_back(r);
        }
    const PairLayout L = pair_layout(n, Q, K, S, N);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_top_triplets_per_pair: workspace too small (%zu < %zu)", ws_bytes,
                L.total);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *Mq = reinterpret_cast<double *>(base + L.o_M);
    auto *T = reinterpret_cast<unsigned long long *>(base + L.o_T);
    auto *key = reinterpret_cast<unsigned long long *>(base + L.o_key), *key2 = reinterpret_cast<unsigned long long *>(base + L.o_key2);
    auto *idx = reinterpret_cast<int32_t *>(base + L.o_idx), *perm = reinterpret_cast<int32_t *>(base + L.o_perm);
    auto *ra = reinterpret_cast<int32_t *>(base + L.o_ra), *rb = reinterpret_cast<int32_t *>(base + L.o_rb);
    auto *d_bidx = reinterpret_cast<int32_t *>(base + L.o_bidx), *d_ub = reinterpret_cast<int32_t *>(base + L.o_ub);
    auto *krow = reinterpret_cast<unsigned long long *>(base + L.o_krow);
    double *V = reinterpret_cast<double *>(base + L.o_V);
    PairSel *sel = reinterpret_cast<PairSel *>(base + L.o_sel);
    auto *need0 = reinterpret_cast<long long *>(base + L.o_need), *m_rows = reinterpret_cast<long long *>(base + L.o_mrows);
    auto *kept = reinterpret_cast<long long *>(base + L.o_kept);
    char *again = base + L.o_again;
    auto *act = reinterpret_cast<int32_t *>(base + L.o_act), *act2 = reinterpret_cast<int32_t *>(base + L.o_act2);
    auto *nsel = reinterpret_cast<int *>(base + L.o_nsel);
    auto *ctl = reinterpret_cast<unsigned long long *>(base + L.o_ctl);
    auto *d_beg = reinterpret_cast<int *>(base + L.o_beg), *d_end = reinterpret_cast<int *>(base + L.o_end);
    auto *counts = reinterpret_cast<int64_t *>(base + L.o_counts);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits), *rcs = reinterpret_cast<unsigned long long *>(base + L.o_rc);
    auto *bits2 = reinterpret_cast<unsigned long long *>(base + L.o_bits2), *rcs2 = reinterpret_cast<unsigned long long *>(base + L.o_rc2);
    void *cub_tmp = base + L.o_cub;
    const int g1 = (int)((Q + 255) / 256);

    // pairs sorted by (ra, rb), with the permutation back to the caller's order
    tip_pair_keys_kernel<<<g1, 256, 0, st>>>(Q, d_pair_ranks, key, idx);
    TIP_CHECK_CUDA(cudaGetLastError());
    size_t cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, key, key2, idx, perm, (int)Q, 0, 2 * kRankBits, st));
    tip_pair_split_kernel<<<g1, 256, 0, st>>>(Q, key2, ra, rb, act);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaMemsetAsync(krow, 0, (size_t)Q * 8, st));
    if (n_known > 0) {
        tip_pair_known_kernel<<<(int)((n_known + 255) / 256), 256, 0, st>>>(n_known, reinterpret_cast<const unsigned long long *>(d_known),
                                                                              Q, key2, krow);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    // V of every pair, from the matrices of its gene b, a chunk of genes at a time
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_bidx, bidx.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_ub, ub.data(), ub.size() * 4, cudaMemcpyHostToDevice, st));
    const int n_ub = (int)ub.size();
    for (int c0 = 0; c0 < n_ub; c0 += L.chunk) {
        const int c1 = std::min(n_ub, c0 + L.chunk);
        const long long work = (long long)L.n_pad * L.SKP + (long long)(c1 - c0) * 3 * S * K * K;
        tip_query_prep_kernel<<<(int)std::min<long long>((work + 255) / 256, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, c1 - c0, d_theta, d_p, d_cand, d_ub + c0, tcat, Mq);
        TIP_CHECK_CUDA(cudaGetLastError());
        tip_pair_vec_kernel<<<(int)((Q * 3 * L.SKP + 255) / 256), 256, 0, st>>>(Q, S, K, L.SKP, c0, c1, d_bidx, ra, rb, tcat, Mq, V);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    TIP_CHECK_CUDA(cudaMemsetAsync(T, 0, (size_t)S * 8, st));
    tip_query_rowsum_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, S, K, L.SKP, tcat, T);
    TIP_CHECK_CUDA(cudaGetLastError());

    int dev = 0, optin = 0;
    TIP_CHECK_CUDA(cudaGetDevice(&dev));
    TIP_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    int nb = 256;
    while (nb > 64 && pair_smem(L.SKP, nb) + 1024 > (size_t)optin) nb /= 2;
    const size_t smem = pair_smem(L.SKP, nb);
    static int smem_set = 0;
    if ((int)smem > smem_set && smem > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_pair_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = (int)smem;
    }
    int per_sm = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tip_pair_pass_kernel, kPredThreads, smem));
    TIP_REQUIRE(per_sm > 0, "tip_top_triplets_per_pair: S*K = %d does not fit one block's shared memory", S * K);

    tip_pair_init_kernel<<<g1, 256, 0, st>>>(Q, n, S, K, L.SKP, N, L.cap, nb, V, T, krow, sel, need0, m_rows, kept);
    TIP_CHECK_CUDA(cudaGetLastError());

    PairPassArgs A{};
    A.n = n; A.SKP = L.SKP; A.nb = nb;
    A.tcat = tcat; A.V = V; A.ra = ra; A.rb = rb; A.active = act; A.n_active = (int)((Q + kPredRows - 1) / kPredRows);
    A.n_pairs = (int)Q;
    A.known = reinterpret_cast<const unsigned long long *>(d_known); A.n_known = n_known;
    A.sel = sel; A.need0 = need0; A.m_rows = m_rows; A.kept = kept; A.again = again; A.ctl = ctl;
    A.out_bits = bits; A.out_rc = rcs; A.cap = L.cap;
    unsigned long long h_ctl[3];
    for (int pass = 0;; ++pass) {
        TIP_REQUIRE(pass < 200, "tip_top_triplets_per_pair: the threshold did not converge (internal error)");
        TIP_CHECK_CUDA(cudaMemsetAsync(ctl, 0, 24, st));
        tip_pair_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm, A.n_active), kPredThreads, smem, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
        ++g_last_pair_passes;
        // the tiles that hold a row not yet resolved, in order
        int32_t *next = A.active == act ? act2 : act;
        cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceSelect::Flagged(cub_tmp, cb, A.active, again, next, nsel, A.n_active, st));
        int h_nsel = 0;
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_ctl, ctl, 24, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(&h_nsel, nsel, 4, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        TIP_REQUIRE(h_ctl[2] == 0, "tip_top_triplets_per_pair: the histogram does not reach N (internal error)");
        if (h_nsel == 0) break;
        A.active = next;
        A.n_active = h_nsel;
    }
    // order: per pair, rc ascending, then (stable) score descending
    tip_pair_segments_kernel<<<g1, 256, 0, st>>>(Q, L.cap, kept, d_beg, d_end);
    TIP_CHECK_CUDA(cudaGetLastError());
    const int items = (int)(Q * L.cap);
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceSegmentedSort::StableSortPairs(cub_tmp, cb, rcs, rcs2, bits, bits2, items, (int)Q, d_beg, d_end, st));
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(
        cub::DeviceSegmentedSort::StableSortPairsDescending(cub_tmp, cb, bits2, bits, rcs2, rcs, items, (int)Q, d_beg, d_end, st));
    tip_pair_finish_kernel<<<(int)((Q * N + 255) / 256), 256, 0, st>>>(Q, N, L.cap, S, perm, ra, rb, m_rows, bits, rcs, d_cand,
                                                                         d_out_ids, d_out_scores, counts);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_n_out, counts, (size_t)Q * 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    return 0;
}

extern "C" int tip_top_triplets_per_pair_last_passes(void) { return g_last_pair_passes; }

// ---- tip_score_histogram ----
// Every triplet of the candidates is scored by the same work items, Q tiles and DMMA block loop as tip_predict_pass_kernel,
// and counted into a fixed log-spaced histogram of the bits of its ensemble sum; no score is stored.  With B = 2^log2_bins
// bins per binade, key(x) = bits(x) >> (52 - log2_bins) (the biased exponent and the top log2_bins mantissa bits) and
// key_top = ((top_exp + 1) << log2_bins) - 1, the bin of a score is
//     0                   when key > key_top (above the range)
//     1 + key_top - key   when key_top - key < n_binades B
//     n_binades B + 1     otherwise (below the range, down to exact zeros)
// so bin 0 holds the highest scores, every bin is an interval of score bits, and the host bins any double the same way.
namespace tip {
namespace {

constexpr int kHistMaxLog2Bins = 10;
constexpr long long kHistMaxRange = 1ll << 14;   // n_binades * B: shared bins beside the Q tile

__host__ __device__ inline int hist_bin(unsigned long long bits, int shift, unsigned long long key_top, unsigned long long n_range)
{
    const unsigned long long key = bits >> shift;
    if (key > key_top) return 0;
    const unsigned long long d = key_top - key;
    return d < n_range ? (int)d + 1 : (int)n_range + 1;
}

// bound[0] = sum_s max(p_s[.][.][.][1]) T_s^3 >= every ensemble sum of scores (non-negative parameters, T_s the largest
// row sum of theta_s over the candidates); one block
__global__ void tip_hist_bound_kernel(int S, int K, const double *__restrict__ p, const unsigned long long *__restrict__ T,
                                      double *__restrict__ bound)
{
    __shared__ double sh_max[256];
    const long long KKK = (long long)K * K * K;
    double sum = 0.0;
    for (int s = 0; s < S; ++s) {
        double mx = 0.0;
        for (long long e = threadIdx.x; e < KKK; e += blockDim.x) mx = fmax(mx, p[((long long)s * KKK + e) * 2 + 1]);
        sh_max[threadIdx.x] = mx;
        __syncthreads();
        for (int w = blockDim.x / 2; w > 0; w >>= 1) {
            if ((int)threadIdx.x < w) sh_max[threadIdx.x] = fmax(sh_max[threadIdx.x], sh_max[threadIdx.x + w]);
            __syncthreads();
        }
        const double t = __longlong_as_double((long long)T[s]);
        sum += sh_max[0] * t * t * t;
        __syncthreads();
    }
    if (threadIdx.x == 0) bound[0] = sum;
}

struct HistPassArgs {
    int n, SK, SKP, K;
    const double *tcat;             // [n_pad][SKP]
    const double *W;                // [S][n][K][K]
    long long n_items;
    int shift;                      // 52 - log2_bins
    unsigned long long key_top, n_range;
    int n_bins;                     // n_range + 2
    unsigned long long *cursor;     // work-item cursor
    unsigned long long *hist;       // [n_bins]
};

// epilogue of a block: every valid score into its shared bin, one shared atomic per distinct bin of the warp
__device__ __forceinline__ void hist_block(const double (&acc)[4][4][2], int lane, int ra0, int rc0, int row_end, int n,
                                           const HistPassArgs &A, unsigned *sh_hist)
{
#pragma unroll
    for (int f = 0; f < 32; ++f) {
        const int mi = f >> 3, ni = (f >> 1) & 3, e = f & 1;
        const int ra = ra0 + mi * 8, rc = rc0 + ni * 8 + e;
        const int bin = (ra < row_end && rc < n)
                            ? hist_bin((unsigned long long)__double_as_longlong(acc[mi][ni][e]), A.shift, A.key_top, A.n_range)
                            : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin >= 0 && lane == __ffs(peers) - 1) atomicAdd(sh_hist + bin, (unsigned)__popc(peers));
    }
}

__device__ __forceinline__ void hist_flush(unsigned *sh_hist, unsigned long long *hist, int n_bins)
{
    for (int i = threadIdx.x; i < n_bins; i += kPredThreads) {
        if (sh_hist[i]) atomicAdd(hist + i, (unsigned long long)sh_hist[i]);
        sh_hist[i] = 0;
    }
}

// the sweep of tip_predict_pass_kernel (same items, Q tiles and DMMA blocks) with a counting epilogue
__global__ void __launch_bounds__(kPredThreads) tip_hist_pass_kernel(HistPassArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP);
    double *Q = reinterpret_cast<double *>(smem);                                   // [64][qs]
    unsigned *sh_hist = reinterpret_cast<unsigned *>(Q + (size_t)kPredRows * qs);  // [n_bins]
    __shared__ long long sh_item;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    for (int i = tid; i < A.n_bins; i += kPredThreads) sh_hist[i] = 0;
    double since_flush = 0.0;   // as in tip_predict_pass_kernel
    const int n = A.n, SKP = A.SKP, K = A.K;

    for (;;) {
        __syncthreads();
        if (tid == 0) sh_item = (long long)atomicAdd(A.cursor, 1ull);
        __syncthreads();
        const long long item = sh_item;
        if (item >= A.n_items) break;
        int jl = 1, jh = n - 2;
        while (jl < jh) {
            const int mid = (jl + jh + 1) >> 1;
            if (items_before(mid) <= item) jl = mid; else jh = mid - 1;
        }
        const int j = jl;
        const int a0 = (int)(item - items_before(j)) * kPredRows;
        const int rows = min(kPredRows, j - a0);
        const int n_c = n - 1 - j;

        form_q_tile(Q, qs, A.tcat, SKP, A.SK, K, a0, rows, A.W + (long long)j * K * K, (long long)n * K * K);
        __syncthreads();

        if (wr * 32 < rows) {
            const double *Qw = Q + (wr * 32 + gq) * qs + tq;
            for (int c0 = j + 1 + wc * 32; c0 < n; c0 += 64) {
                double acc[4][4][2];
                dmma_block(acc, Qw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                hist_block(acc, lane, a0 + wr * 32 + gq, c0 + 2 * tq, j, n, A, sh_hist);
            }
        }
        since_flush += (double)rows * n_c;
        if (since_flush > 2.0e9) {
            __syncthreads();
            hist_flush(sh_hist, A.hist, A.n_bins);
            since_flush = 0.0;
        }
    }
    hist_flush(sh_hist, A.hist, A.n_bins);
}

struct HistLayout {
    size_t o_tcat, o_W, o_T, o_bound, o_cursor, total;
    int n_pad, SKP;
};

HistLayout hist_layout(int n, int K, int S)
{
    HistLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    size_t off = 0;
    L.o_tcat = off;   off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_W = off;      off += a256((size_t)S * n * K * K * 8);
    L.o_T = off;      off += a256((size_t)S * 8);
    L.o_bound = off;  off += 256;
    L.o_cursor = off; off += 256;
    L.total = off + 256;
    return L;
}

size_t hist_smem(int SKP, long long n_bins) { return (size_t)kPredRows * q_stride(SKP) * 8 + (size_t)n_bins * 4; }

}  // namespace
}  // namespace tip

static bool hist_args_ok(int n_cand, int K, int S, int log2_bins, int n_binades)
{
    return predict_args_ok(n_cand, K, S, 0, 0) && log2_bins >= 0 && log2_bins <= kHistMaxLog2Bins && n_binades >= 1 &&
           ((long long)n_binades << log2_bins) <= kHistMaxRange;
}

#define TIP_HIST_LIMITS "n_cand <= 2^21, 1 <= K <= %d, S >= 1, S*K <= %d, 0 <= log2_bins <= %d, n_binades >= 1, " \
                        "n_binades * 2^log2_bins <= %lld"

extern "C" int tip_score_histogram_workspace_bytes(int n_cand, int K, int S, int log2_bins, int n_binades, size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && hist_args_ok(n_cand, K, S, log2_bins, n_binades),
                "tip_score_histogram_workspace_bytes: bad arguments (" TIP_HIST_LIMITS ")", TIP_MAX_K, kPredMaxSK,
                kHistMaxLog2Bins, kHistMaxRange);
    *bytes = hist_layout(n_cand, K, S).total;
    return 0;
}

extern "C" int tip_score_histogram(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand,
                                   int n_cand, int log2_bins, int n_binades, int *h_top_exp, uint64_t *d_hist_out, void *d_ws,
                                   size_t ws_bytes, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && hist_args_ok(n_cand, K, S, log2_bins, n_binades) && h_top_exp != nullptr,
                "tip_score_histogram: bad arguments (P > 0, n_cand <= P, " TIP_HIST_LIMITS ")", TIP_MAX_K, kPredMaxSK,
                kHistMaxLog2Bins, kHistMaxRange);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && d_hist_out, "tip_score_histogram: null pointer");
    const int n = n_cand;
    const HistLayout L = hist_layout(n, K, S);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_score_histogram: workspace too small (%zu < %zu)", ws_bytes, L.total);
    const long long n_range = (long long)n_binades << log2_bins, n_bins = n_range + 2;
    const size_t smem = hist_smem(L.SKP, n_bins);
    int dev = 0, optin = 0;
    TIP_CHECK_CUDA(cudaGetDevice(&dev));
    TIP_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    TIP_REQUIRE(smem + 64 <= (size_t)optin,
                "tip_score_histogram: the Q tile of S*K = %d and %lld bins need %zu bytes of shared memory (the device has %d)",
                S * K, n_bins, smem, optin);
    static int smem_set = 0;
    if ((int)smem > smem_set && smem > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_hist_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        smem_set = (int)smem;
    }
    int per_sm = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tip_hist_pass_kernel, kPredThreads, smem));
    TIP_REQUIRE(per_sm > 0, "tip_score_histogram: S*K = %d does not fit one block's shared memory", S * K);

    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *W = reinterpret_cast<double *>(base + L.o_W);
    auto *T = reinterpret_cast<unsigned long long *>(base + L.o_T);
    double *bound = reinterpret_cast<double *>(base + L.o_bound);
    auto *cursor = reinterpret_cast<unsigned long long *>(base + L.o_cursor);
    TIP_CHECK_CUDA(cudaMemsetAsync(d_hist_out, 0, (size_t)n_bins * 8, st));
    *h_top_exp = 0;
    if (n < 3) {
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    }
    {
        const long long work = (long long)L.n_pad * L.SKP + (long long)S * n * K * K;
        tip_predict_prep_kernel<<<(int)std::min<long long>((work + 255) / 256, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, d_theta, d_p, d_cand, tcat, W);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaMemsetAsync(T, 0, (size_t)S * 8, st));
        tip_query_rowsum_kernel<<<(n + 255) / 256, 256, 0, st>>>(n, S, K, L.SKP, tcat, T);
        TIP_CHECK_CUDA(cudaGetLastError());
        tip_hist_bound_kernel<<<1, 256, 0, st>>>(S, K, d_p, T, bound);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    double h_bound = 0.0;
    TIP_CHECK_CUDA(cudaMemcpyAsync(&h_bound, bound, 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    // the range's top binade holds the bound (with a margin for its rounding); a score above it lands in bin 0
    const double hb = h_bound * (1.0 + 1e-9);
    const int top_exp = std::isfinite(hb) ? (int)((unsigned long long)__builtin_bit_cast(long long, hb) >> 52) & 0x7FF : 2046;
    *h_top_exp = std::min(top_exp, 2046);

    HistPassArgs A{};
    A.n = n; A.SK = S * K; A.SKP = L.SKP; A.K = K;
    A.tcat = tcat; A.W = W;
    A.n_items = items_before(n - 1);
    A.shift = 52 - log2_bins;
    A.key_top = (((unsigned long long)*h_top_exp + 1) << log2_bins) - 1;
    A.n_range = (unsigned long long)n_range;
    A.n_bins = (int)n_bins;
    A.cursor = cursor; A.hist = reinterpret_cast<unsigned long long *>(d_hist_out);
    TIP_CHECK_CUDA(cudaMemsetAsync(cursor, 0, 8, st));
    tip_hist_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm, A.n_items), kPredThreads, smem, st>>>(A);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ---- tip_rank_per_pair ----
// The exact rank of every held-out partner among its query pair's unseen partners.  The sorted pairs, their V rows, the
// tiles of 64 sorted pairs, the three column phases and dmma_block are those of tip_top_triplets_per_pair, so every score is
// computed at the same fragment position, with the same contraction order, as there.  Test entries (pair, rc) are sorted by
// (sorted pair, rc); the train partners of a pair (the distinct known keys that contain it) by (the first sorted position
// of the pair, rc).
// Capture sweep: each warp jumps to the column blocks that hold a test partner of one of its rows and records its bits.
// Count sweep: a tile's entries sit in shared memory, per row in the order (bits descending, rc ascending), at most e_max of
// them per round (a tile with more is swept once per round).  Every score of a row is tested in registers against the
// row's weakest entry of the round; train partners, found by a cursor that walks the row's sorted train list along the
// columns, are skipped; a score that passes is placed among the entries by binary search and counted at its slot (the
// scores ahead of every entry of the round in a register per row).  rank = 1 + the slot counts up to the entry.
namespace tip {
namespace {

constexpr int kRankMaxEntries = 2048;             // entries of a count round in shared memory, 16 bytes each
constexpr int kRankMinEntries = 256;              // fewer beside the A tile: refused (bounds the rounds in the workspace)
constexpr int kRankKeyBits = kRankBits + 24;      // (sorted pair << 21) | rc, n_pairs <= 2^24
constexpr unsigned long long kRcMask = (1ull << kRankBits) - 1;

struct RankPassArgs {
    int n, SKP, n_pairs, mode;          // mode 0: capture the bits of the test entries; 1: count
    const double *tcat;                 // [n_pad][SKP]
    const double *V;                    // [n_pairs][3][SKP], sorted pair order
    const int32_t *ra, *rb;             // [n_pairs] sorted
    const int4 *items;                  // {tile, g0, g1, 0}: the count sweep ranks the entries [g0, g1) of the tile
    int n_items;
    const int32_t *te_off;              // [n_pairs + 1] test entries of sorted pair p: [te_off[p], te_off[p + 1])
    const unsigned long long *te_key;   // [n_test] (p << 21) | rc, ascending
    const int32_t *tr_beg, *tr_end;     // [n_pairs] train partners of sorted pair p in tr_key
    const unsigned long long *tr_key;   // (first sorted position of the pair << 21) | rc, ascending
    unsigned long long *te_bits;        // capture: [n_test] score bits, te_key order
    const unsigned long long *ord_bits; // count: [n_test] score bits, per pair in the order (bits descending, rc ascending)
    const int32_t *ord_pos;             // count: [n_test] the te_key position of each entry of that order
    const int32_t *te_idx;              // [n_test] the caller's index of each te_key entry
    int64_t *rank;                      // count: [n_test] caller's order
    unsigned long long *ctl;            // [0] item cursor
};

__device__ __forceinline__ long long lower_bound_u64(const unsigned long long *a, long long n, unsigned long long key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (a[mid] < key) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// per caller's pair: its sorted position
__global__ void tip_rank_inverse_kernel(long long n_pairs, const int32_t *__restrict__ perm, int32_t *__restrict__ inv)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p < n_pairs) inv[perm[p]] = (int32_t)p;
}

__global__ void tip_rank_test_keys_kernel(long long n_test, const int32_t *__restrict__ test_pair, const int32_t *__restrict__ test_rc,
                                          const int32_t *__restrict__ inv, unsigned long long *__restrict__ key,
                                          int32_t *__restrict__ idx)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_test) return;
    key[j] = ((unsigned long long)inv[test_pair[j]] << kRankBits) | (unsigned long long)test_rc[j];
    idx[j] = (int32_t)j;
}

// the train partners: per distinct known key (ascending ranks, all < n) and each of its three pairs that is listed, the
// key's third rank, tagged with the pair's first sorted position
__global__ void tip_rank_train_kernel(long long n_known, const unsigned long long *__restrict__ known, int n, long long n_pairs,
                                      const unsigned long long *__restrict__ key, unsigned long long *__restrict__ tr_key,
                                      unsigned long long *n_tr)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_known || (i > 0 && known[i] == known[i - 1])) return;   // a repeated key counts once
    const unsigned long long k = known[i];
    const unsigned long long r0 = (k >> (2 * kRankBits)) & kRcMask, r1 = (k >> kRankBits) & kRcMask, r2 = k & kRcMask;
    if (!(r0 < r1 && r1 < r2 && r2 < (unsigned long long)n)) return;
    const unsigned long long want[3] = {(r0 << kRankBits) | r1, (r0 << kRankBits) | r2, (r1 << kRankBits) | r2};
    const unsigned long long third[3] = {r2, r1, r0};
    for (int w = 0; w < 3; ++w) {
        const long long pos = lower_bound_u64(key, n_pairs, want[w]);
        if (pos < n_pairs && key[pos] == want[w])
            tr_key[atomicAdd(n_tr, 1ull)] = ((unsigned long long)pos << kRankBits) | third[w];
    }
}

// per sorted pair: its test entries, its train partners and |U| (in the caller's order)
__global__ void tip_rank_rows_kernel(long long n_pairs, int n, const unsigned long long *__restrict__ key, const int32_t *__restrict__ perm,
                                     long long n_test, const unsigned long long *__restrict__ te_key, long long n_tr,
                                     const unsigned long long *__restrict__ tr_key, int32_t *__restrict__ te_off,
                                     int32_t *__restrict__ rep, int32_t *__restrict__ tr_beg, int32_t *__restrict__ tr_end,
                                     int64_t *__restrict__ universe)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_pairs) return;
    const unsigned long long r = (unsigned long long)lower_bound_u64(key, n_pairs, key[p]);
    te_off[p] = (int32_t)lower_bound_u64(te_key, n_test, (unsigned long long)p << kRankBits);
    if (p == n_pairs - 1) te_off[n_pairs] = (int32_t)n_test;
    const long long b = lower_bound_u64(tr_key, n_tr, r << kRankBits), e = lower_bound_u64(tr_key, n_tr, (r + 1) << kRankBits);
    rep[p] = (int32_t)r;
    tr_beg[p] = (int32_t)b;
    tr_end[p] = (int32_t)e;
    universe[perm[p]] = max(0ll, (long long)n - 2 - (e - b));
}

__global__ void tip_rank_iota_kernel(long long m, int32_t *__restrict__ out)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j < m) out[j] = (int32_t)j;
}

// the lane's score at column offset off (from the lane's first column) of row mi of its block, if the lane holds it
__device__ __forceinline__ bool lane_score(const double (&acc)[4][4][2], int mi, int off, double &v)
{
    bool hit = false;
#pragma unroll
    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
        for (int e = 0; e < 2; ++e)
            if (off == ni * 8 + e) {
                v = acc[mi][ni][e];
                hit = true;
            }
    return hit;
}

// work items are tiles of 64 sorted pairs (the tiles of tip_pair_pass_kernel, swept over the same column ranges)
__global__ void __launch_bounds__(kPredThreads) tip_rank_pass_kernel(RankPassArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP);
    double *At = reinterpret_cast<double *>(smem);                                                     // [64][qs]
    const bool count = A.mode == 1;
    unsigned long long *sh_eb = reinterpret_cast<unsigned long long *>(At + (size_t)kPredRows * qs);  // count: entry bits
    int *sh_erc = nullptr;                                                                             // entry rc
    unsigned *sh_cnt = nullptr;                                                                        // slot counts
    __shared__ int sh_ra[kPredRows], sh_rb[kPredRows], sh_lb[kPredRows], sh_le[kPredRows], sh_elo[kPredRows], sh_ehi[kPredRows];
    __shared__ long long sh_item;
    __shared__ int sh_range[4];   // min ra, max ra, min rb, max rb of the tile
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    const int n = A.n, SKP = A.SKP;
    const unsigned long long *list = count ? A.tr_key : A.te_key;   // the column lists the cursors walk

    for (;;) {
        __syncthreads();   // the previous tile is no longer read
        if (tid == 0) sh_item = (long long)atomicAdd(A.ctl, 1ull);
        __syncthreads();
        const long long item = sh_item;
        if (item >= A.n_items) break;
        const int4 it = A.items[item];
        const int t0 = it.x * kPredRows, rows = min(kPredRows, A.n_pairs - t0), n_e = it.z - it.y;
        sh_erc = reinterpret_cast<int *>(sh_eb + n_e);
        sh_cnt = reinterpret_cast<unsigned *>(sh_erc + n_e);
        if (tid < kPredRows) {
            const int p = t0 + (tid < rows ? tid : 0);
            sh_ra[tid] = A.ra[p];
            sh_rb[tid] = A.rb[p];
            const int b = A.te_off[p], e = A.te_off[p + 1];
            const bool in = tid < rows;
            sh_lb[tid] = !in ? 0 : count ? A.tr_beg[p] : b;
            sh_le[tid] = !in ? 0 : count ? A.tr_end[p] : e;
            const int elo = max(b, it.y) - it.y, ehi = min(e, it.z) - it.y;
            sh_elo[tid] = in && count ? elo : 0;
            sh_ehi[tid] = in && count ? max(elo, ehi) : 0;
        }
        if (count)
            for (int e = tid; e < n_e; e += kPredThreads) {
                const int g = it.y + e;
                sh_eb[e] = A.ord_bits[g];
                sh_erc[e] = (int)(A.te_key[A.ord_pos[g]] & kRcMask);
                sh_cnt[e] = 0;
            }
        __syncthreads();
        if (tid == 0) {
            int r0 = n, r1 = 0, r2 = n, r3 = 0;
            for (int i = 0; i < rows; ++i) {
                r0 = min(r0, sh_ra[i]); r1 = max(r1, sh_ra[i]);
                r2 = min(r2, sh_rb[i]); r3 = max(r3, sh_rb[i]);
            }
            sh_range[0] = r0; sh_range[1] = r1; sh_range[2] = r2; sh_range[3] = r3;
        }
        __syncthreads();

        for (int g = 0; g < 3; ++g) {
            const int col0 = g == 0 ? 0 : g == 1 ? sh_range[0] + 1 : sh_range[2] + 1;
            const int col_end = g == 0 ? sh_range[1] : g == 1 ? sh_range[3] : n;
            if (col0 >= col_end) continue;
            __syncthreads();   // the previous phase's A tile is no longer read
            for (int e = tid; e < kPredRows * SKP; e += kPredThreads) {
                const int i = e / SKP, col = e % SKP;
                At[i * qs + col] = i < rows ? __ldg(A.V + ((long long)(t0 + i) * 3 + g) * SKP + col) : 0.0;
            }
            __syncthreads();
            if (wr * 32 >= rows) continue;
            const int ib = wr * 32 + gq;   // the lane's first row
            int cur[4], lim[4];
            unsigned ahead[4] = {0u, 0u, 0u, 0u};   // count: scores ahead of every entry of the round, per row
            bool any = false;
#pragma unroll
            for (int mi = 0; mi < 4; ++mi) {
                const int i = ib + mi * 8;
                const bool act = !count || sh_elo[i] < sh_ehi[i];
                cur[mi] = act ? sh_lb[i] : 0;
                lim[mi] = act ? sh_le[i] : 0;
                any |= count ? act : cur[mi] < lim[mi];
            }
            if (!__any_sync(0xffffffffu, any)) continue;
            const double *Aw = At + ib * qs + tq;
            const int cbase = col0 + wc * 32;
            for (int c0 = cbase; c0 < col_end; c0 += 64) {
                if (!count) {
                    // the warp's next column, at or after c0, that holds a test partner of one of its rows in the row's region
                    int nxt = INT_MAX;
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) {
                        const int i = ib + mi * 8, ra = sh_ra[i], rb = sh_rb[i];
                        const int lo_c = g == 0 ? 0 : g == 1 ? ra + 1 : rb + 1, hi_c = g == 0 ? ra : g == 1 ? rb : n;
                        const int from = max(c0, lo_c);
                        while (cur[mi] < lim[mi] && (int)(__ldg(list + cur[mi]) & kRcMask) < from) ++cur[mi];
                        if (cur[mi] < lim[mi]) {
                            const int r = (int)(__ldg(list + cur[mi]) & kRcMask);
                            if (r < hi_c) nxt = min(nxt, r);
                        }
                    }
                    nxt = __reduce_min_sync(0xffffffffu, nxt);
                    if (nxt >= col_end) break;
                    const int c1 = cbase + (nxt - cbase) / 64 * 64;
                    c0 = c1;
                    if (nxt - c1 >= 32) continue;   // in the other column half: look again from the next block
                }
                double acc[4][4][2];
                dmma_block(acc, Aw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                const int rc0 = c0 + 2 * tq;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    const int i = ib + mi * 8, ra = sh_ra[i], rb = sh_rb[i];
                    const int lo_c = g == 0 ? 0 : g == 1 ? ra + 1 : rb + 1, hi_c = g == 0 ? ra : g == 1 ? rb : n;
                    if (!count) {
                        // the row's test partners in this block (the cursor is at the first at or after max(c0, lo_c))
                        while (cur[mi] < lim[mi]) {
                            const int r = (int)(__ldg(list + cur[mi]) & kRcMask);
                            if (r >= c0 + 32 || r >= hi_c) break;
                            double v = 0.0;
                            if (lane_score(acc, mi, r - rc0, v)) A.te_bits[cur[mi]] = (unsigned long long)__double_as_longlong(v);
                            ++cur[mi];
                        }
                        continue;
                    }
                    const int elo = sh_elo[i], ehi = sh_ehi[i];
                    if (elo == ehi) continue;
                    // the row's train partners among the lane's columns of this block
                    unsigned skip = 0;
                    while (cur[mi] < lim[mi]) {
                        const int r = (int)(__ldg(list + cur[mi]) & kRcMask);
                        if (r >= c0 + 32) break;
                        const int off = r - rc0;
#pragma unroll
                        for (int f = 0; f < 8; ++f)
                            if (off == (f >> 1) * 8 + (f & 1)) skip |= 1u << f;
                        ++cur[mi];
                    }
                    const unsigned long long wb = sh_eb[ehi - 1], fb = sh_eb[elo];
                    const int wrc = sh_erc[ehi - 1], frc = sh_erc[elo];
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const int rc = rc0 + ni * 8 + e;
                            if (rc < lo_c || rc >= hi_c || ((skip >> (ni * 2 + e)) & 1u)) continue;
                            const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
                            if (!(bits > wb || (bits == wb && rc < wrc))) continue;   // not ahead of the weakest entry
                            if (bits > fb || (bits == fb && rc < frc)) {
                                ++ahead[mi];
                                continue;
                            }
                            // the first entry in (elo, ehi) the score is ahead of
                            int lo = elo + 1, hi = ehi - 1;
                            while (lo < hi) {
                                const int mid = (lo + hi) >> 1;
                                const unsigned long long mb = sh_eb[mid];
                                if (bits > mb || (bits == mb && rc < sh_erc[mid])) hi = mid; else lo = mid + 1;
                            }
                            atomicAdd(sh_cnt + lo, 1u);
                        }
                }
            }
            if (count) {
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    unsigned a = ahead[mi];
                    a += __shfl_xor_sync(0xffffffffu, a, 1);
                    a += __shfl_xor_sync(0xffffffffu, a, 2);
                    const int i = ib + mi * 8;
                    if (tq == 0 && a) atomicAdd(sh_cnt + sh_elo[i], a);
                }
            }
        }
        __syncthreads();
        if (count && tid < rows) {
            long long run = 0;
            for (int s = sh_elo[tid]; s < sh_ehi[tid]; ++s) {
                run += sh_cnt[s];
                A.rank[A.te_idx[A.ord_pos[it.y + s]]] = (int64_t)(1 + run);
            }
        }
    }
}

// per test entry (te_key order): the mean score, and rank 0 when its triplet is a train partner of its pair
__global__ void tip_rank_finish_kernel(long long n_test, int S, const unsigned long long *__restrict__ te_key,
                                       const int32_t *__restrict__ te_idx, const unsigned long long *__restrict__ bits,
                                       const int32_t *__restrict__ rep, long long n_tr, const unsigned long long *__restrict__ tr_key,
                                       int64_t *__restrict__ rank, double *__restrict__ score)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_test) return;
    const unsigned long long k = te_key[j];
    const unsigned long long want = ((unsigned long long)rep[k >> kRankBits] << kRankBits) | (k & kRcMask);
    const long long at = lower_bound_u64(tr_key, n_tr, want);
    const int o = te_idx[j];
    score[o] = __longlong_as_double((long long)bits[j]) / (double)S;
    if (at < n_tr && tr_key[at] == want) rank[o] = 0;
}

struct RankLayout {
    size_t o_tcat, o_M, o_key, o_key2, o_idx, o_perm, o_inv, o_ra, o_rb, o_act, o_bidx, o_ub, o_V, o_tk, o_tk2, o_ti, o_ti2,
        o_bits, o_obits, o_opos0, o_opos, o_toff, o_rep, o_trb, o_tre, o_trk, o_trk2, o_ntr, o_ctl, o_items, o_cub, cub_bytes,
        total;
    int n_pad, SKP, chunk;
    long long max_items;
};

RankLayout rank_layout(int n, long long n_pairs, int K, int S, long long n_known, long long n_test)
{
    RankLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.chunk = (int)std::max(1ll, std::min((long long)n, (long long)L.n_pad * L.SKP / (3ll * S * K * K)));
    const long long tiles = (n_pairs + kPredRows - 1) / kPredRows;
    L.max_items = 2 * tiles + n_test / kRankMinEntries + 1;   // the capture items, then the count rounds
    const int np = (int)n_pairs, nt = (int)n_test, ntr = (int)(3 * n_known);
    size_t cb[5] = {0, 0, 0, 0, 0};
    cub::DeviceRadixSort::SortPairs(nullptr, cb[0], (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, np, 0, 2 * kRankBits, (cudaStream_t)0);
    cub::DeviceRadixSort::SortPairs(nullptr, cb[1], (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, nt, 0, kRankKeyBits, (cudaStream_t)0);
    cub::DeviceRadixSort::SortKeys(nullptr, cb[2], (const unsigned long long *)nullptr, (unsigned long long *)nullptr, ntr, 0,
                                   kRankKeyBits, (cudaStream_t)0);
    cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, cb[3], (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (const int32_t *)nullptr, (int32_t *)nullptr,
                                                        nt, np, (const int *)nullptr, (const int *)nullptr, (cudaStream_t)0);
    L.cub_bytes = *std::max_element(cb, cb + 5);
    const size_t q = (size_t)n_pairs, t = (size_t)n_test;
    size_t off = 0;
    L.o_tcat = off;   off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_M = off;      off += a256((size_t)L.chunk * 3 * S * K * K * 8);
    L.o_key = off;    off += a256(q * 8);
    L.o_key2 = off;   off += a256(q * 8);
    L.o_idx = off;    off += a256(q * 4);
    L.o_perm = off;   off += a256(q * 4);
    L.o_inv = off;    off += a256(q * 4);
    L.o_ra = off;     off += a256(q * 4);
    L.o_rb = off;     off += a256(q * 4);
    L.o_act = off;    off += a256(q * 4);
    L.o_bidx = off;   off += a256((size_t)n * 4);
    L.o_ub = off;     off += a256((size_t)n * 4);
    L.o_V = off;      off += a256(q * 3 * L.SKP * 8);
    L.o_tk = off;     off += a256(t * 8);
    L.o_tk2 = off;    off += a256(t * 8);
    L.o_ti = off;     off += a256(t * 4);
    L.o_ti2 = off;    off += a256(t * 4);
    L.o_bits = off;   off += a256(t * 8);
    L.o_obits = off;  off += a256(t * 8);
    L.o_opos0 = off;  off += a256(t * 4);
    L.o_opos = off;   off += a256(t * 4);
    L.o_toff = off;   off += a256((q + 1) * 4);
    L.o_rep = off;    off += a256(q * 4);
    L.o_trb = off;    off += a256(q * 4);
    L.o_tre = off;    off += a256(q * 4);
    L.o_trk = off;    off += a256((size_t)n_known * 3 * 8);
    L.o_trk2 = off;   off += a256((size_t)n_known * 3 * 8);
    L.o_ntr = off;    off += 256;
    L.o_ctl = off;    off += 256;
    L.o_items = off;  off += a256((size_t)L.max_items * sizeof(int4));
    L.o_cub = off;    off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

size_t rank_smem(int SKP, int e_max) { return (size_t)kPredRows * q_stride(SKP) * 8 + (size_t)e_max * 16; }

}  // namespace
}  // namespace tip

static bool rank_args_ok(int n_cand, int64_t n_pairs, int K, int S, int64_t n_known, int64_t n_test)
{
    return predict_args_ok(n_cand, K, S, n_known, 0) && n_pairs >= 0 && n_pairs <= kPairMaxRows && n_known <= (1ll << 29) &&
           n_test >= 0 && n_test < (1ll << 31);
}

#define TIP_RANK_LIMITS "n_cand <= 2^21, 1 <= K <= %d, S >= 1, S*K <= %d, 0 <= n_pairs <= 2^24, 0 <= n_known <= 2^29, " \
                        "0 <= n_test < 2^31"

extern "C" int tip_rank_per_pair_workspace_bytes(int n_cand, int64_t n_pairs, int K, int S, int64_t n_known, int64_t n_test,
                                                 size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && rank_args_ok(n_cand, n_pairs, K, S, n_known, n_test),
                "tip_rank_per_pair_workspace_bytes: bad arguments (" TIP_RANK_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    *bytes = rank_layout(n_cand, n_pairs, K, S, n_known, n_test).total;
    return 0;
}

extern "C" int tip_rank_per_pair(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand, int n_cand,
                                 const int32_t *d_pair_ranks, int64_t n_pairs, const uint64_t *d_known, int64_t n_known,
                                 const int32_t *d_test_pair, const int32_t *d_test_rc, int64_t n_test, void *d_ws, size_t ws_bytes,
                                 int64_t *d_rank_out, double *d_score_out, int64_t *d_universe_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && rank_args_ok(n_cand, n_pairs, K, S, n_known, n_test),
                "tip_rank_per_pair: bad arguments (P > 0, n_cand <= P, " TIP_RANK_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && (d_known || n_known == 0) &&
                    (n_pairs == 0 || (d_pair_ranks && d_universe_out)) &&
                    (n_test == 0 || (d_test_pair && d_test_rc && d_rank_out && d_score_out)),
                "tip_rank_per_pair: null pointer");
    const int n = n_cand;
    const long long Q = n_pairs, T = n_test;
    // pair ranks and test entries are checked on the host before any device work
    std::vector<int32_t> pr((size_t)Q * 2), tp((size_t)T), trc((size_t)T);
    if (Q) TIP_CHECK_CUDA(cudaMemcpyAsync(pr.data(), d_pair_ranks, (size_t)Q * 8, cudaMemcpyDeviceToHost, st));
    if (T) {
        TIP_CHECK_CUDA(cudaMemcpyAsync(tp.data(), d_test_pair, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(trc.data(), d_test_rc, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
    }
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> bidx(std::max(n, 1), -1), ub;
    for (long long i = 0; i < Q; ++i) {
        for (int e = 0; e < 2; ++e)
            TIP_REQUIRE(pr[2 * i + e] >= 0 && pr[2 * i + e] < n, "tip_rank_per_pair: rank %d of pair %lld is not in [0, %d)",
                        pr[2 * i + e], i, n);
        TIP_REQUIRE(pr[2 * i] != pr[2 * i + 1], "tip_rank_per_pair: pair %lld has the same rank twice (%d)", i, pr[2 * i]);
        bidx[std::max(pr[2 * i], pr[2 * i + 1])] = 0;
    }
    for (long long j = 0; j < T; ++j) {
        TIP_REQUIRE(tp[j] >= 0 && tp[j] < Q, "tip_rank_per_pair: test entry %lld names pair %d, not in [0, %lld)", j, tp[j], Q);
        const int32_t a = pr[2 * (size_t)tp[j]], b = pr[2 * (size_t)tp[j] + 1];
        TIP_REQUIRE(trc[j] >= 0 && trc[j] < n && trc[j] != a && trc[j] != b,
                    "tip_rank_per_pair: test entry %lld has partner rank %d, not a rank in [0, %d) other than its pair's (%d, %d)",
                    j, trc[j], n, a, b);
    }
    if (Q == 0) return 0;
    for (int r = 0; r < n; ++r)
        if (bidx[r] == 0) {
            bidx[r] = (int32_t)ub.size();
            ub.push_back(r);
        }
    const RankLayout L = rank_layout(n, Q, K, S, n_known, T);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_rank_per_pair: workspace too small (%zu < %zu)", ws_bytes, L.total);
    int dev = 0, optin = 0;
    TIP_CHECK_CUDA(cudaGetDevice(&dev));
    TIP_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa{};
    TIP_CHECK_CUDA(cudaFuncGetAttributes(&fa, tip_rank_pass_kernel));
    const long long room = ((long long)optin - 1024 - (long long)fa.sharedSizeBytes - (long long)rank_smem(L.SKP, 0)) / 16;
    const int e_max = (int)std::min<long long>(kRankMaxEntries, room);
    TIP_REQUIRE(e_max >= kRankMinEntries, "tip_rank_per_pair: S*K = %d leaves room for %d entries beside the A tile (internal error)",
                S * K, e_max);

    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *Mq = reinterpret_cast<double *>(base + L.o_M);
    auto *key = reinterpret_cast<unsigned long long *>(base + L.o_key), *key2 = reinterpret_cast<unsigned long long *>(base + L.o_key2);
    auto *idx = reinterpret_cast<int32_t *>(base + L.o_idx), *perm = reinterpret_cast<int32_t *>(base + L.o_perm);
    auto *inv = reinterpret_cast<int32_t *>(base + L.o_inv);
    auto *ra = reinterpret_cast<int32_t *>(base + L.o_ra), *rb = reinterpret_cast<int32_t *>(base + L.o_rb);
    auto *act = reinterpret_cast<int32_t *>(base + L.o_act);
    auto *d_bidx = reinterpret_cast<int32_t *>(base + L.o_bidx), *d_ub = reinterpret_cast<int32_t *>(base + L.o_ub);
    double *V = reinterpret_cast<double *>(base + L.o_V);
    auto *tk = reinterpret_cast<unsigned long long *>(base + L.o_tk), *tk2 = reinterpret_cast<unsigned long long *>(base + L.o_tk2);
    auto *ti = reinterpret_cast<int32_t *>(base + L.o_ti), *ti2 = reinterpret_cast<int32_t *>(base + L.o_ti2);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits);
    auto *obits = reinterpret_cast<unsigned long long *>(base + L.o_obits);
    auto *opos0 = reinterpret_cast<int32_t *>(base + L.o_opos0), *opos = reinterpret_cast<int32_t *>(base + L.o_opos);
    auto *toff = reinterpret_cast<int32_t *>(base + L.o_toff), *rep = reinterpret_cast<int32_t *>(base + L.o_rep);
    auto *trb = reinterpret_cast<int32_t *>(base + L.o_trb), *tre = reinterpret_cast<int32_t *>(base + L.o_tre);
    auto *trk = reinterpret_cast<unsigned long long *>(base + L.o_trk), *trk2 = reinterpret_cast<unsigned long long *>(base + L.o_trk2);
    auto *ntr = reinterpret_cast<unsigned long long *>(base + L.o_ntr), *ctl = reinterpret_cast<unsigned long long *>(base + L.o_ctl);
    auto *items = reinterpret_cast<int4 *>(base + L.o_items);
    void *cub_tmp = base + L.o_cub;
    const int g1 = (int)((Q + 255) / 256), gt = (int)((T + 255) / 256);
    size_t cb = 0;

    // pairs sorted by (ra, rb) as tip_top_triplets_per_pair sorts them, with the permutation back to the caller's order
    tip_pair_keys_kernel<<<g1, 256, 0, st>>>(Q, d_pair_ranks, key, idx);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, key, key2, idx, perm, (int)Q, 0, 2 * kRankBits, st));
    tip_pair_split_kernel<<<g1, 256, 0, st>>>(Q, key2, ra, rb, act);
    TIP_CHECK_CUDA(cudaGetLastError());
    tip_rank_inverse_kernel<<<g1, 256, 0, st>>>(Q, perm, inv);
    TIP_CHECK_CUDA(cudaGetLastError());
    // test entries by (sorted pair, rc)
    if (T) {
        tip_rank_test_keys_kernel<<<gt, 256, 0, st>>>(T, d_test_pair, d_test_rc, inv, tk, ti);
        TIP_CHECK_CUDA(cudaGetLastError());
        cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, tk, tk2, ti, ti2, (int)T, 0, kRankKeyBits, st));
    }
    // train partners by (first sorted position of the pair, rc)
    TIP_CHECK_CUDA(cudaMemsetAsync(ntr, 0, 8, st));
    if (n_known > 0) {
        tip_rank_train_kernel<<<(int)((n_known + 255) / 256), 256, 0, st>>>(
            n_known, reinterpret_cast<const unsigned long long *>(d_known), n, Q, key2, trk, ntr);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    unsigned long long h_ntr = 0;
    TIP_CHECK_CUDA(cudaMemcpyAsync(&h_ntr, ntr, 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    const long long NT = (long long)h_ntr;
    if (NT) {
        cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortKeys(cub_tmp, cb, trk, trk2, (int)NT, 0, kRankKeyBits, st));
    }
    tip_rank_rows_kernel<<<g1, 256, 0, st>>>(Q, n, key2, perm, T, tk2, NT, trk2, toff, rep, trb, tre, d_universe_out);
    TIP_CHECK_CUDA(cudaGetLastError());
    if (T == 0) {
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    }

    // V of every pair, from the matrices of its gene b, a chunk of genes at a time (as tip_top_triplets_per_pair)
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_bidx, bidx.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_ub, ub.data(), ub.size() * 4, cudaMemcpyHostToDevice, st));
    const int n_ub = (int)ub.size();
    for (int c0 = 0; c0 < n_ub; c0 += L.chunk) {
        const int c1 = std::min(n_ub, c0 + L.chunk);
        const long long work = (long long)L.n_pad * L.SKP + (long long)(c1 - c0) * 3 * S * K * K;
        tip_query_prep_kernel<<<(int)std::min<long long>((work + 255) / 256, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, c1 - c0, d_theta, d_p, d_cand, d_ub + c0, tcat, Mq);
        TIP_CHECK_CUDA(cudaGetLastError());
        tip_pair_vec_kernel<<<(int)((Q * 3 * L.SKP + 255) / 256), 256, 0, st>>>(Q, S, K, L.SKP, c0, c1, d_bidx, ra, rb, tcat, Mq, V);
        TIP_CHECK_CUDA(cudaGetLastError());
    }

    // work items: the tiles that hold a test entry (capture), then each of them in rounds of at most e_max entries (count)
    std::vector<int32_t> h_off((size_t)Q + 1);
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_off.data(), toff, ((size_t)Q + 1) * 4, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    std::vector<int4> h_items;
    const long long tiles = (Q + kPredRows - 1) / kPredRows;
    for (long long t = 0; t < tiles; ++t) {
        const int b = h_off[(size_t)(t * kPredRows)], e = h_off[(size_t)std::min(Q, (t + 1) * kPredRows)];
        if (e > b) h_items.push_back(make_int4((int)t, b, e, 0));
    }
    const int n_capture = (int)h_items.size();
    for (int k = 0; k < n_capture; ++k)
        for (int b = h_items[k].y; b < h_items[k].z; b += e_max)
            h_items.push_back(make_int4(h_items[k].x, b, std::min(h_items[k].z, b + e_max), 0));
    const int n_count = (int)h_items.size() - n_capture;
    TIP_REQUIRE((long long)h_items.size() <= L.max_items, "tip_rank_per_pair: %zu work items (internal error)", h_items.size());
    TIP_CHECK_CUDA(cudaMemcpyAsync(items, h_items.data(), h_items.size() * sizeof(int4), cudaMemcpyHostToDevice, st));

    const size_t smem0 = rank_smem(L.SKP, 0), smem1 = rank_smem(L.SKP, e_max);
    static int smem_set = 0;
    if ((int)smem1 > smem_set && smem1 > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_rank_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        smem_set = (int)smem1;
    }
    int per_sm0 = 0, per_sm1 = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm0, tip_rank_pass_kernel, kPredThreads, smem0));
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm1, tip_rank_pass_kernel, kPredThreads, smem1));
    TIP_REQUIRE(per_sm0 > 0 && per_sm1 > 0, "tip_rank_per_pair: S*K = %d does not fit one block's shared memory", S * K);

    RankPassArgs A{};
    A.n = n; A.SKP = L.SKP; A.n_pairs = (int)Q;
    A.tcat = tcat; A.V = V; A.ra = ra; A.rb = rb;
    A.te_off = toff; A.te_key = tk2; A.tr_beg = trb; A.tr_end = tre; A.tr_key = trk2;
    A.te_bits = bits; A.ord_bits = obits; A.ord_pos = opos; A.te_idx = ti2; A.rank = d_rank_out; A.ctl = ctl;
    // capture sweep
    A.mode = 0; A.items = items; A.n_items = n_capture;
    TIP_CHECK_CUDA(cudaMemsetAsync(ctl, 0, 8, st));
    tip_rank_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm0, n_capture), kPredThreads, smem0, st>>>(A);
    TIP_CHECK_CUDA(cudaGetLastError());
    // per pair: entries in the order (bits descending, rc ascending): a stable sort of the (pair, rc) order
    tip_rank_iota_kernel<<<gt, 256, 0, st>>>(T, opos0);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceSegmentedSort::StableSortPairsDescending(cub_tmp, cb, bits, obits, opos0, opos, (int)T, (int)Q, toff,
                                                                      toff + 1, st));
    // count sweep
    A.mode = 1; A.items = items + n_capture; A.n_items = n_count;
    TIP_CHECK_CUDA(cudaMemsetAsync(ctl, 0, 8, st));
    tip_rank_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm1, n_count), kPredThreads, smem1, st>>>(A);
    TIP_CHECK_CUDA(cudaGetLastError());
    tip_rank_finish_kernel<<<gt, 256, 0, st>>>(T, S, tk2, ti2, bits, rep, NT, trk2, d_rank_out, d_score_out);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ---- tip_rank_per_gene ----
// The exact rank of every held-out triplet among its query gene's unseen triplets.  The work items (query, region, 64-row
// tile) of query_tiles, the Q tiles that form_q_tile builds from the Mq of tip_query_prep_kernel, the column blocks from
// col0 + wc 32 in steps of 64 and dmma_block are those of tip_query_pass_kernel, so every score is computed at the same
// fragment position, with the same contraction order, as tip_top_triplets_per_gene computes it.  In a triplet {q, u, v}
// with u < v the row is u and the column v.  Entries are keyed (query index << 42) | (u << 21) | v; for a fixed query this
// order is the packed order of the triplets.  They are the test entries and the train entries: per distinct known key, each
// of its genes that is a query.
// Capture sweep: only the tiles that hold an entry; each warp jumps to the column blocks that hold an entry of one of its rows
// and the lane that holds the score writes its bits.  A segmented stable sort then orders each query's entries by (bits
// descending, key ascending), and a scan of the test flags gives every test entry its place among the query's test entries
// and the number of train entries ahead of it.
// Count sweep: items (query, round, region, tile), query-major; a round is at most e_max of the query's test entries, held in
// shared memory.  Every score is tested in registers against the round's weakest entry, then its first; the scores between
// them are placed by binary search and counted at their slot with a shared atomic.  Slot counts go to global memory, one
// atomic per slot, when the CTA's (query, round) changes.  rank = 1 + the round's slot counts up to the entry - the train
// entries ahead of it: train triplets are counted like any other score and subtracted, not skipped.
namespace tip {
namespace {

constexpr int kGeneEntryBytes = 20;                      // a count round's entry in shared memory: bits, key, slot count
constexpr unsigned long long kUvMask = (1ull << (2 * kRankBits)) - 1;

struct GeneRankArgs {
    int n, S, K, SK, SKP, mode;           // mode 0: capture the bits of the entries; 1: count
    const double *tcat;                   // [n_pad][SKP]
    const double *Mq;                     // [n_query][3][S][K][K]
    const int32_t *qrank;                 // [n_query]
    const long long *seg_start;           // capture: [n_query + 1] first item of each query; count: [n_seg + 1] of each round
    const int4 *seg;                      // count: [n_seg] {query, first, end, 0}: the round's entries in the t_* arrays
    int n_seg;
    const long long *items;               // capture: [n_items] the item ids that hold an entry
    long long n_items;
    int e_max;                            // count: entries of a round in shared memory
    const unsigned long long *key;        // capture: [n_entries] sorted entry keys
    const int32_t *q_off;                 // capture: [n_query + 1] each query's entries in key
    unsigned long long *bits;             // capture: [n_entries] score bits, key order
    const unsigned long long *t_bits;     // count: test entries per query in the order (bits descending, key ascending)
    const unsigned long long *t_uv;       // count: (u << 21) | v of each
    unsigned long long *t_cnt;            // count: slot counts
    unsigned long long *ctl;              // [0] item cursor
};

__device__ __forceinline__ unsigned long long lane_bits(double v) { return (unsigned long long)__double_as_longlong(v); }

__global__ void __launch_bounds__(kPredThreads) tip_gene_rank_pass_kernel(GeneRankArgs A)
{
    extern __shared__ __align__(16) unsigned char smem[];
    const int qs = q_stride(A.SKP);
    double *Q = reinterpret_cast<double *>(smem);                                                  // [64][qs]
    unsigned long long *sh_eb = reinterpret_cast<unsigned long long *>(Q + (size_t)kPredRows * qs);  // count: entry bits
    unsigned long long *sh_ek = sh_eb + A.e_max;                                                   // entry (u << 21) | v
    unsigned *sh_cnt = reinterpret_cast<unsigned *>(sh_ek + A.e_max);                              // slot counts
    __shared__ long long sh_item;
    __shared__ long long sh_lb[kPredRows], sh_le[kPredRows];   // capture: each row's entries in key
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    const int n = A.n, SKP = A.SKP, K = A.K;
    const long long KK = (long long)K * K;
    const bool count = A.mode == 1;
    int cur_seg = -1, ne = 0;   // count: the round whose entries and slot counts shared memory holds (CTA-uniform)
    double since_flush = 0.0;   // as in tip_predict_pass_kernel: the 32-bit slot counts are flushed before they could overflow

    for (;;) {
        __syncthreads();   // Q, the entries and sh_item of the previous item are no longer read
        if (tid == 0) sh_item = (long long)atomicAdd(A.ctl, 1ull);
        __syncthreads();
        const long long it = sh_item;
        if (it >= A.n_items) break;
        const long long item = count ? it : A.items[it];
        int sl = 0, sh = A.n_seg - 1;
        while (sl < sh) {
            const int mid = (sl + sh + 1) >> 1;
            if (A.seg_start[mid] <= item) sl = mid; else sh = mid - 1;
        }
        const int qi = count ? A.seg[sl].x : sl, r = A.qrank[qi];
        if (count && (sl != cur_seg || since_flush > 2.0e9)) {
            // the same thread flushes, clears and reloads an index: no barrier between the loops
            for (int e = tid; e < ne; e += kPredThreads) {
                if (sh_cnt[e]) atomicAdd(A.t_cnt + A.seg[cur_seg].y + e, (unsigned long long)sh_cnt[e]);
                sh_cnt[e] = 0;
            }
            if (sl != cur_seg) {
                const int4 s = A.seg[sl];
                ne = s.z - s.y;
                for (int e = tid; e < ne; e += kPredThreads) {
                    sh_eb[e] = A.t_bits[s.y + e];
                    sh_ek[e] = A.t_uv[s.y + e];
                    sh_cnt[e] = 0;
                }
                cur_seg = sl;
            }
            since_flush = 0.0;
        }
        int tc, tb, ta;
        query_tiles(n, r, tc, tb, ta);
        int t = (int)(item - A.seg_start[sl]);
        int g, a0, col0, row_end;
        bool tri;
        if (t < tc) {
            g = 0; a0 = t * kPredRows; col0 = a0 + 1; row_end = r - 1; tri = true;
        } else if ((t -= tc) < tb) {
            g = 1; a0 = t * kPredRows; col0 = r + 1; row_end = r; tri = false;
        } else {
            t -= tb;
            g = 2; a0 = r + 1 + t * kPredRows; col0 = a0 + 1; row_end = n - 1; tri = true;
        }
        const int col_end = g == 0 ? r : n;
        const int rows = min(kPredRows, row_end - a0);
        if (!count && tid < kPredRows) {
            long long b = 0, e = 0;
            if (tid < rows) {
                const long long qb = A.q_off[qi], qe = A.q_off[qi + 1];
                const unsigned long long k0 = ((unsigned long long)qi << (2 * kRankBits)) | ((unsigned long long)(a0 + tid) << kRankBits);
                b = qb + lower_bound_u64(A.key + qb, qe - qb, k0);
                e = b + lower_bound_u64(A.key + b, qe - b, k0 + (1ull << kRankBits));
            }
            sh_lb[tid] = b;
            sh_le[tid] = e;
        }

        form_q_tile(Q, qs, A.tcat, SKP, A.SK, K, a0, rows, A.Mq + ((long long)qi * 3 + g) * A.S * KK, KK);
        __syncthreads();

        if (wr * 32 < rows) {
            const int ib = wr * 32 + gq;   // the lane's first row in the tile
            const double *Qw = Q + ib * qs + tq;
            const int cbase = col0 + wc * 32;
            if (!count) {
                long long cur[4], lim[4];
                bool any = false;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi) {
                    cur[mi] = sh_lb[ib + mi * 8];
                    lim[mi] = sh_le[ib + mi * 8];
                    any |= cur[mi] < lim[mi];
                }
                const bool warp_any = __any_sync(0xffffffffu, any);
                for (int c0 = cbase; warp_any && c0 < col_end; c0 += 64) {
                    // the warp's next column, at or after c0, that holds an entry of one of its rows in this region
                    int nxt = INT_MAX;
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi) {
                        const int ra = a0 + ib + mi * 8;
                        const int from = max(c0, tri ? ra + 1 : col0);
                        while (cur[mi] < lim[mi] && (int)(__ldg(A.key + cur[mi]) & kRcMask) < from) ++cur[mi];
                        if (cur[mi] < lim[mi]) {
                            const int v = (int)(__ldg(A.key + cur[mi]) & kRcMask);
                            if (v < col_end) nxt = min(nxt, v);
                        }
                    }
                    nxt = __reduce_min_sync(0xffffffffu, nxt);
                    if (nxt >= col_end) break;
                    c0 = cbase + (nxt - cbase) / 64 * 64;
                    if (nxt - c0 >= 32) continue;   // in the other column half: look again from the next block
                    double acc[4][4][2];
                    dmma_block(acc, Qw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                    const int rc0 = c0 + 2 * tq;
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
                        while (cur[mi] < lim[mi]) {
                            const int v = (int)(__ldg(A.key + cur[mi]) & kRcMask);
                            if (v >= c0 + 32 || v >= col_end) break;
                            double s = 0.0;
                            if (lane_score(acc, mi, v - rc0, s)) A.bits[cur[mi]] = lane_bits(s);
                            ++cur[mi];
                        }
                }
            } else {
                const unsigned long long wb = sh_eb[ne - 1], wk = sh_ek[ne - 1], fb = sh_eb[0], fk = sh_ek[0];
                const int ra0 = a0 + ib;
                unsigned ahead = 0;   // scores ahead of every entry of the round
                for (int c0 = cbase; c0 < col_end; c0 += 64) {
                    double acc[4][4][2];
                    dmma_block(acc, Qw, qs, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
                    const int rc0 = c0 + 2 * tq;
#pragma unroll
                    for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                        for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                            for (int e = 0; e < 2; ++e) {
                                const int ra = ra0 + mi * 8, rc = rc0 + ni * 8 + e;
                                if (ra >= row_end || rc >= col_end || (tri && rc <= ra)) continue;
                                const unsigned long long b = lane_bits(acc[mi][ni][e]);
                                const unsigned long long k = ((unsigned long long)ra << kRankBits) | (unsigned long long)rc;
                                if (!(b > wb || (b == wb && k < wk))) continue;   // not ahead of the weakest entry
                                if (b > fb || (b == fb && k < fk)) {
                                    ++ahead;
                                    continue;
                                }
                                // the first entry in (0, ne - 1] the score is ahead of
                                int lo = 1, hi = ne - 1;
                                while (lo < hi) {
                                    const int mid = (lo + hi) >> 1;
                                    const unsigned long long mb = sh_eb[mid];
                                    if (b > mb || (b == mb && k < sh_ek[mid])) hi = mid; else lo = mid + 1;
                                }
                                atomicAdd(sh_cnt + lo, 1u);
                            }
                }
                ahead = __reduce_add_sync(0xffffffffu, ahead);
                if (lane == 0 && ahead) atomicAdd(sh_cnt, ahead);
            }
        }
        since_flush += (double)rows * (col_end - col0);
    }
    if (count)
        for (int e = tid; e < ne; e += kPredThreads)
            if (sh_cnt[e]) atomicAdd(A.t_cnt + A.seg[cur_seg].y + e, (unsigned long long)sh_cnt[e]);
}

// entries: test entry j is ((query << 42) | (min(u, v) << 21) | max(u, v), j)
__global__ void tip_gene_test_keys_kernel(long long n_test, const int32_t *__restrict__ tq, const int32_t *__restrict__ tu,
                                          const int32_t *__restrict__ tv, unsigned long long *__restrict__ key,
                                          int32_t *__restrict__ idx)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_test) return;
    const unsigned long long u = (unsigned long long)min(tu[j], tv[j]), v = (unsigned long long)max(tu[j], tv[j]);
    key[j] = ((unsigned long long)tq[j] << (2 * kRankBits)) | (u << kRankBits) | v;
    idx[j] = (int32_t)j;
}

// the train entries: per distinct known key (ascending ranks, all < n) and each of its genes that is a query, the key's other
// two ranks, appended after the n_test test entries with an index >= n_test
__global__ void tip_gene_train_kernel(long long n_known, const unsigned long long *__restrict__ known, int n,
                                      const int32_t *__restrict__ qidx, long long n_test, unsigned long long *__restrict__ key,
                                      int32_t *__restrict__ idx, unsigned long long *n_tr)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_known || (i > 0 && known[i] == known[i - 1])) return;   // a repeated key counts once
    const unsigned long long k = known[i];
    const unsigned long long r0 = (k >> (2 * kRankBits)) & kRcMask, r1 = (k >> kRankBits) & kRcMask, r2 = k & kRcMask;
    if (!(r0 < r1 && r1 < r2 && r2 < (unsigned long long)n)) return;
    const unsigned long long self[3] = {r0, r1, r2};
    const unsigned long long other[3] = {(r1 << kRankBits) | r2, (r0 << kRankBits) | r2, (r0 << kRankBits) | r1};
    for (int w = 0; w < 3; ++w) {
        const int q = qidx[self[w]];
        if (q < 0) continue;
        const long long at = n_test + (long long)atomicAdd(n_tr, 1ull);
        key[at] = ((unsigned long long)q << (2 * kRankBits)) | other[w];
        idx[at] = (int32_t)at;
    }
}

// per query: its first entry in the sorted keys
__global__ void tip_gene_offsets_kernel(int n_query, long long n_entries, const unsigned long long *__restrict__ key,
                                        int32_t *__restrict__ off)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q > n_query) return;
    off[q] = (int32_t)lower_bound_u64(key, n_entries, (unsigned long long)q << (2 * kRankBits));
}

// per sorted entry: the work item (query_tiles numbering from item_start[query]) that holds its score
__global__ void tip_gene_items_kernel(long long n_entries, int n, const unsigned long long *__restrict__ key,
                                      const int32_t *__restrict__ qrank, const long long *__restrict__ item_start,
                                      unsigned long long *__restrict__ item)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n_entries) return;
    const unsigned long long k = key[p];
    const int q = (int)(k >> (2 * kRankBits)), u = (int)((k >> kRankBits) & kRcMask), v = (int)(k & kRcMask), r = qrank[q];
    int tc, tb, ta;
    query_tiles(n, r, tc, tb, ta);
    const int t = v < r ? u / kPredRows : u < r ? tc + u / kPredRows : tc + tb + (u - r - 1) / kPredRows;
    item[p] = (unsigned long long)(item_start[q] + t);
}

// per entry in the query order (bits descending, key ascending): 1 when it is a test entry
__global__ void tip_gene_flags_kernel(long long n_entries, const int32_t *__restrict__ ord_pos, const int32_t *__restrict__ idx,
                                      long long n_test, int32_t *__restrict__ flag)
{
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o < n_entries) flag[o] = idx[ord_pos[o]] < n_test ? 1 : 0;
}

// the test entries of each query in that order (tscan: exclusive scan of the flags), with the train entries ahead of each,
// -1 when its triplet is a train entry itself (the last entry of its key's run is then a train entry)
__global__ void tip_gene_compact_kernel(long long n_entries, long long n_test, const unsigned long long *__restrict__ key,
                                        const int32_t *__restrict__ idx, const int32_t *__restrict__ q_off,
                                        const unsigned long long *__restrict__ ord_bits, const int32_t *__restrict__ ord_pos,
                                        const int32_t *__restrict__ tscan, unsigned long long *__restrict__ t_bits,
                                        unsigned long long *__restrict__ t_uv, int32_t *__restrict__ t_idx,
                                        int32_t *__restrict__ t_train)
{
    const long long o = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= n_entries) return;
    const long long p = ord_pos[o];
    if (idx[p] >= n_test) return;
    const unsigned long long k = key[p];
    const int q = (int)(k >> (2 * kRankBits));
    const long long qb = q_off[q], qe = q_off[q + 1];
    const long long last = p + lower_bound_u64(key + p, qe - p, k + 1) - 1;
    const int t = tscan[o];
    t_bits[t] = ord_bits[o];
    t_uv[t] = k & kUvMask;
    t_idx[t] = idx[p];
    t_train[t] = idx[last] >= n_test ? -1 : (int32_t)((o - qb) - (t - tscan[qb]));
}

// per query: its first test entry in the t_* arrays and |U| = C(n - 1, 2) - its train entries
__global__ void tip_gene_universe_kernel(int n_query, long long n_entries, long long n_test, long long pairs,
                                         const int32_t *__restrict__ q_off, const int32_t *__restrict__ tscan,
                                         int32_t *__restrict__ t_off, int64_t *__restrict__ universe)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q > n_query) return;
    auto tests_before = [&](long long o) -> long long { return n_test == 0 ? 0 : o < n_entries ? tscan[o] : n_test; };
    t_off[q] = (int32_t)tests_before(q_off[q]);
    if (q == n_query) return;
    const long long train = (q_off[q + 1] - q_off[q]) - (tests_before(q_off[q + 1]) - tests_before(q_off[q]));
    universe[q] = pairs - train;
}

// per round: rank = 1 + the round's slot counts up to the entry - the train entries ahead of it (0 for a train triplet)
__global__ void tip_gene_finish_kernel(int n_seg, int S, const int4 *__restrict__ seg, const unsigned long long *__restrict__ t_cnt,
                                       const unsigned long long *__restrict__ t_bits, const int32_t *__restrict__ t_idx,
                                       const int32_t *__restrict__ t_train, int64_t *__restrict__ rank, double *__restrict__ score)
{
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    long long run = 0;
    for (int k = seg[s].y; k < seg[s].z; ++k) {
        run += (long long)t_cnt[k];
        const int j = t_idx[k];
        score[j] = __longlong_as_double((long long)t_bits[k]) / (double)S;
        rank[j] = t_train[k] < 0 ? 0 : 1 + run - t_train[k];
    }
}

struct GeneRankLayout {
    size_t o_tcat, o_M, o_qidx, o_istart, o_qoff, o_toff, o_key, o_key2, o_idx, o_idx2, o_bits, o_obits, o_opos0, o_opos, o_flag,
        o_scan, o_item, o_item2, o_uitem, o_tbits, o_tuv, o_tcnt, o_tidx, o_ttr, o_seg, o_sstart, o_cnt, o_cub, cub_bytes, total;
    int n_pad, SKP;
    long long max_seg;
};

GeneRankLayout gene_rank_layout(int n, int n_query, int K, int S, long long n_known, long long n_test)
{
    GeneRankLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.max_seg = n_query + n_test / kRankMinEntries + 1;
    const long long e_all = n_test + 3 * n_known;
    const int ne = (int)std::min<long long>(e_all, INT_MAX), nq = std::max(n_query, 1);
    size_t cb[5] = {0, 0, 0, 0, 0};
    cub::DeviceRadixSort::SortPairs(nullptr, cb[0], (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, ne, 0, 64, (cudaStream_t)0);
    cub::DeviceRadixSort::SortKeys(nullptr, cb[1], (const unsigned long long *)nullptr, (unsigned long long *)nullptr, ne, 0, 64,
                                   (cudaStream_t)0);
    cub::DeviceSelect::Unique(nullptr, cb[2], (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int *)nullptr, ne,
                              (cudaStream_t)0);
    cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, cb[3], (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (const int32_t *)nullptr, (int32_t *)nullptr,
                                                        ne, nq, (const int *)nullptr, (const int *)nullptr, (cudaStream_t)0);
    cub::DeviceScan::ExclusiveSum(nullptr, cb[4], (const int32_t *)nullptr, (int32_t *)nullptr, ne, (cudaStream_t)0);
    L.cub_bytes = *std::max_element(cb, cb + 5);
    const size_t e = (size_t)e_all, t = (size_t)n_test, q = (size_t)n_query;
    size_t off = 0;
    L.o_tcat = off;   off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_M = off;      off += a256(q * 3 * S * K * K * 8);
    L.o_qidx = off;   off += a256((size_t)n * 4);
    L.o_istart = off; off += a256((q + 1) * 8);
    L.o_qoff = off;   off += a256((q + 1) * 4);
    L.o_toff = off;   off += a256((q + 1) * 4);
    L.o_key = off;    off += a256(e * 8);
    L.o_key2 = off;   off += a256(e * 8);
    L.o_idx = off;    off += a256(e * 4);
    L.o_idx2 = off;   off += a256(e * 4);
    L.o_bits = off;   off += a256(e * 8);
    L.o_obits = off;  off += a256(e * 8);
    L.o_opos0 = off;  off += a256(e * 4);
    L.o_opos = off;   off += a256(e * 4);
    L.o_flag = off;   off += a256(e * 4);
    L.o_scan = off;   off += a256(e * 4);
    L.o_item = off;   off += a256(e * 8);
    L.o_item2 = off;  off += a256(e * 8);
    L.o_uitem = off;  off += a256(e * 8);
    L.o_tbits = off;  off += a256(t * 8);
    L.o_tuv = off;    off += a256(t * 8);
    L.o_tcnt = off;   off += a256(t * 8);
    L.o_tidx = off;   off += a256(t * 4);
    L.o_ttr = off;    off += a256(t * 4);
    L.o_seg = off;    off += a256((size_t)L.max_seg * sizeof(int4));
    L.o_sstart = off; off += a256(((size_t)L.max_seg + 1) * 8);
    L.o_cnt = off;    off += 256;
    L.o_cub = off;    off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

size_t gene_rank_smem(int SKP, int e_max) { return (size_t)kPredRows * q_stride(SKP) * 8 + (size_t)e_max * kGeneEntryBytes; }

int bits_for(long long x)
{
    int b = 0;
    while (b < 63 && (1ll << b) <= x) ++b;
    return b;
}

}  // namespace
}  // namespace tip

static bool gene_rank_args_ok(int n_cand, int n_query, int K, int S, int64_t n_known, int64_t n_test)
{
    return predict_args_ok(n_cand, K, S, n_known, 0) && n_query >= 0 && n_query <= n_cand && n_known <= (1ll << 29) &&
           n_test >= 0 && n_test < (1ll << 31);
}

#define TIP_GENE_RANK_LIMITS "n_cand <= 2^21, 1 <= K <= %d, S >= 1, S*K <= %d, 0 <= n_query <= n_cand, 0 <= n_known <= 2^29, " \
                             "0 <= n_test < 2^31"

extern "C" int tip_rank_per_gene_workspace_bytes(int n_cand, int n_query, int K, int S, int64_t n_known, int64_t n_test,
                                                 size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && gene_rank_args_ok(n_cand, n_query, K, S, n_known, n_test),
                "tip_rank_per_gene_workspace_bytes: bad arguments (" TIP_GENE_RANK_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    *bytes = gene_rank_layout(n_cand, n_query, K, S, n_known, n_test).total;
    return 0;
}

extern "C" int tip_rank_per_gene(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand, int n_cand,
                                 const int32_t *d_query_ranks, int n_query, const uint64_t *d_known, int64_t n_known,
                                 const int32_t *d_test_query, const int32_t *d_test_u, const int32_t *d_test_v, int64_t n_test,
                                 void *d_ws, size_t ws_bytes, int64_t *d_rank_out, double *d_score_out, int64_t *d_universe_out,
                                 void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && gene_rank_args_ok(n_cand, n_query, K, S, n_known, n_test),
                "tip_rank_per_gene: bad arguments (P > 0, n_cand <= P, " TIP_GENE_RANK_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_p && (d_cand || n_cand == 0) && (d_known || n_known == 0) &&
                    (n_query == 0 || (d_query_ranks && d_universe_out)) &&
                    (n_test == 0 || (d_test_query && d_test_u && d_test_v && d_rank_out && d_score_out)),
                "tip_rank_per_gene: null pointer");
    const int n = n_cand, nq = n_query;
    const long long T = n_test;
    // query ranks and test entries are checked on the host before any device work
    std::vector<int32_t> qr(nq), tq((size_t)T), tu((size_t)T), tv((size_t)T);
    if (nq) TIP_CHECK_CUDA(cudaMemcpyAsync(qr.data(), d_query_ranks, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    if (T) {
        TIP_CHECK_CUDA(cudaMemcpyAsync(tq.data(), d_test_query, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(tu.data(), d_test_u, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(tv.data(), d_test_v, (size_t)T * 4, cudaMemcpyDeviceToHost, st));
    }
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    std::vector<int32_t> qidx(std::max(n, 1), -1);
    for (int i = 0; i < nq; ++i) {
        TIP_REQUIRE(qr[i] >= 0 && qr[i] < n, "tip_rank_per_gene: query rank %d of query %d is not in [0, %d)", qr[i], i, n);
        TIP_REQUIRE(qidx[qr[i]] < 0, "tip_rank_per_gene: query rank %d appears twice", qr[i]);
        qidx[qr[i]] = i;
    }
    for (long long j = 0; j < T; ++j) {
        TIP_REQUIRE(tq[j] >= 0 && tq[j] < nq, "tip_rank_per_gene: test entry %lld names query %d, not in [0, %d)", j, tq[j], nq);
        const int32_t r = qr[tq[j]];
        TIP_REQUIRE(tu[j] >= 0 && tu[j] < n && tv[j] >= 0 && tv[j] < n && tu[j] != r && tv[j] != r && tu[j] != tv[j],
                    "tip_rank_per_gene: test entry %lld has ranks (%d, %d), not two distinct ranks in [0, %d) other than its "
                    "query's (%d)", j, tu[j], tv[j], n, r);
    }
    if (nq == 0) return 0;
    const GeneRankLayout L = gene_rank_layout(n, nq, K, S, n_known, T);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_rank_per_gene: workspace too small (%zu < %zu)", ws_bytes, L.total);
    int dev = 0, optin = 0;
    TIP_CHECK_CUDA(cudaGetDevice(&dev));
    TIP_CHECK_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    cudaFuncAttributes fa{};
    TIP_CHECK_CUDA(cudaFuncGetAttributes(&fa, tip_gene_rank_pass_kernel));
    const long long room =
        ((long long)optin - 1024 - (long long)fa.sharedSizeBytes - (long long)gene_rank_smem(L.SKP, 0)) / kGeneEntryBytes;
    const int e_max = (int)std::min<long long>(kRankMaxEntries, room);
    TIP_REQUIRE(e_max >= kRankMinEntries, "tip_rank_per_gene: S*K = %d leaves room for %d entries beside the Q tile (internal error)",
                S * K, e_max);

    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *Mq = reinterpret_cast<double *>(base + L.o_M);
    auto *d_qidx = reinterpret_cast<int32_t *>(base + L.o_qidx);
    auto *istart = reinterpret_cast<long long *>(base + L.o_istart);
    auto *qoff = reinterpret_cast<int32_t *>(base + L.o_qoff), *toff = reinterpret_cast<int32_t *>(base + L.o_toff);
    auto *key = reinterpret_cast<unsigned long long *>(base + L.o_key), *key2 = reinterpret_cast<unsigned long long *>(base + L.o_key2);
    auto *idx = reinterpret_cast<int32_t *>(base + L.o_idx), *idx2 = reinterpret_cast<int32_t *>(base + L.o_idx2);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits);
    auto *obits = reinterpret_cast<unsigned long long *>(base + L.o_obits);
    auto *opos0 = reinterpret_cast<int32_t *>(base + L.o_opos0), *opos = reinterpret_cast<int32_t *>(base + L.o_opos);
    auto *flag = reinterpret_cast<int32_t *>(base + L.o_flag), *tscan = reinterpret_cast<int32_t *>(base + L.o_scan);
    auto *item = reinterpret_cast<unsigned long long *>(base + L.o_item);
    auto *item2 = reinterpret_cast<unsigned long long *>(base + L.o_item2);
    auto *uitem = reinterpret_cast<unsigned long long *>(base + L.o_uitem);
    auto *t_bits = reinterpret_cast<unsigned long long *>(base + L.o_tbits), *t_uv = reinterpret_cast<unsigned long long *>(base + L.o_tuv);
    auto *t_cnt = reinterpret_cast<unsigned long long *>(base + L.o_tcnt);
    auto *t_idx = reinterpret_cast<int32_t *>(base + L.o_tidx), *t_tr = reinterpret_cast<int32_t *>(base + L.o_ttr);
    auto *seg = reinterpret_cast<int4 *>(base + L.o_seg);
    auto *sstart = reinterpret_cast<long long *>(base + L.o_sstart);
    auto *cnt = reinterpret_cast<unsigned long long *>(base + L.o_cnt);   // [0] train entries, [1] item cursor, [2] unique items
    void *cub_tmp = base + L.o_cub;
    size_t cb = 0;

    // the work items of every query, numbered as tip_query_pass_kernel numbers them, query after query
    std::vector<long long> h_istart((size_t)nq + 1, 0);
    for (int i = 0; i < nq; ++i) {
        int tc, tb, ta;
        query_tiles(n, qr[i], tc, tb, ta);
        h_istart[i + 1] = h_istart[i] + tc + tb + ta;
    }
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_qidx, qidx.data(), (size_t)n * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(istart, h_istart.data(), ((size_t)nq + 1) * 8, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemsetAsync(cnt, 0, 3 * 8, st));
    // entries: the test entries, then the train entries of the queries; sorted by (query, u, v)
    if (T) {
        tip_gene_test_keys_kernel<<<(int)((T + 255) / 256), 256, 0, st>>>(T, d_test_query, d_test_u, d_test_v, key, idx);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    if (n_known > 0) {
        tip_gene_train_kernel<<<(int)((n_known + 255) / 256), 256, 0, st>>>(
            n_known, reinterpret_cast<const unsigned long long *>(d_known), n, d_qidx, T, key, idx, cnt);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    unsigned long long h_ntr = 0;
    TIP_CHECK_CUDA(cudaMemcpyAsync(&h_ntr, cnt, 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    const long long E = T + (long long)h_ntr;
    TIP_REQUIRE(E < (1ll << 31), "tip_rank_per_gene: %lld test and train entries, more than 2^31 - 1", E);
    const int end_bit = 2 * kRankBits + bits_for(nq - 1);
    if (E) {
        cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, key, key2, idx, idx2, (int)E, 0, end_bit, st));
    }
    tip_gene_offsets_kernel<<<(nq + 256) / 256, 256, 0, st>>>(nq, E, key2, qoff);
    TIP_CHECK_CUDA(cudaGetLastError());
    const long long pairs = n_pairs(n - 1);
    if (T == 0) {
        tip_gene_universe_kernel<<<(nq + 256) / 256, 256, 0, st>>>(nq, E, 0, pairs, qoff, tscan, toff, d_universe_out);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        return 0;
    }

    // tcat and the query matrices as tip_top_triplets_per_gene forms them
    {
        const long long work = (long long)L.n_pad * L.SKP + (long long)nq * 3 * S * K * K;
        tip_query_prep_kernel<<<(int)std::min<long long>((work + 255) / 256, (long long)sm_count() * 16), 256, 0, st>>>(
            S, P, K, n, L.n_pad, L.SKP, nq, d_theta, d_p, d_cand, d_query_ranks, tcat, Mq);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    // capture items: the distinct items that hold an entry
    const int ge = (int)((E + 255) / 256);
    tip_gene_items_kernel<<<ge, 256, 0, st>>>(E, n, key2, d_query_ranks, istart, item);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortKeys(cub_tmp, cb, item, item2, (int)E, 0, std::max(1, bits_for(h_istart[nq])), st));
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceSelect::Unique(cub_tmp, cb, item2, uitem, reinterpret_cast<int *>(cnt + 2), (int)E, st));
    int n_capture = 0;
    TIP_CHECK_CUDA(cudaMemcpyAsync(&n_capture, cnt + 2, 4, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));

    const size_t smem0 = gene_rank_smem(L.SKP, 0), smem1 = gene_rank_smem(L.SKP, e_max);
    static int smem_set = 0;
    if ((int)smem1 > smem_set && smem1 > 48 * 1024) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(tip_gene_rank_pass_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        smem_set = (int)smem1;
    }
    int per_sm0 = 0, per_sm1 = 0;
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm0, tip_gene_rank_pass_kernel, kPredThreads, smem0));
    TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm1, tip_gene_rank_pass_kernel, kPredThreads, smem1));
    TIP_REQUIRE(per_sm0 > 0 && per_sm1 > 0, "tip_rank_per_gene: S*K = %d does not fit one block's shared memory", S * K);

    GeneRankArgs A{};
    A.n = n; A.S = S; A.K = K; A.SK = S * K; A.SKP = L.SKP;
    A.tcat = tcat; A.Mq = Mq; A.qrank = d_query_ranks; A.ctl = cnt + 1;
    // capture sweep
    A.mode = 0; A.seg_start = istart; A.n_seg = nq; A.items = reinterpret_cast<const long long *>(uitem); A.n_items = n_capture;
    A.key = key2; A.q_off = qoff; A.bits = bits;
    if (n_capture > 0) {
        tip_gene_rank_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm0, n_capture), kPredThreads, smem0, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    // per query: entries in the order (bits descending, key ascending), a stable sort of the key order; the test entries
    // of that order with the train entries ahead of each
    tip_rank_iota_kernel<<<ge, 256, 0, st>>>(E, opos0);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceSegmentedSort::StableSortPairsDescending(cub_tmp, cb, bits, obits, opos0, opos, (int)E, nq, qoff,
                                                                      qoff + 1, st));
    tip_gene_flags_kernel<<<ge, 256, 0, st>>>(E, opos, idx2, T, flag);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = L.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(cub_tmp, cb, flag, tscan, (int)E, st));
    tip_gene_compact_kernel<<<ge, 256, 0, st>>>(E, T, key2, idx2, qoff, obits, opos, tscan, t_bits, t_uv, t_idx, t_tr);
    TIP_CHECK_CUDA(cudaGetLastError());
    tip_gene_universe_kernel<<<(nq + 256) / 256, 256, 0, st>>>(nq, E, T, pairs, qoff, tscan, toff, d_universe_out);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaMemsetAsync(t_cnt, 0, (size_t)T * 8, st));

    // count items: every tile of every query with a test entry, once per round of at most e_max of its test entries
    std::vector<int32_t> h_toff((size_t)nq + 1);
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_toff.data(), toff, ((size_t)nq + 1) * 4, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    std::vector<int4> h_seg;
    std::vector<long long> h_sstart(1, 0);
    for (int i = 0; i < nq; ++i)
        for (int b = h_toff[i]; b < h_toff[i + 1]; b += e_max) {
            h_seg.push_back(make_int4(i, b, std::min(h_toff[i + 1], b + e_max), 0));
            h_sstart.push_back(h_sstart.back() + (h_istart[i + 1] - h_istart[i]));
        }
    const int n_seg = (int)h_seg.size();
    TIP_REQUIRE(n_seg <= L.max_seg, "tip_rank_per_gene: %d rounds (internal error)", n_seg);
    TIP_CHECK_CUDA(cudaMemcpyAsync(seg, h_seg.data(), (size_t)n_seg * sizeof(int4), cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(sstart, h_sstart.data(), ((size_t)n_seg + 1) * 8, cudaMemcpyHostToDevice, st));
    // count sweep
    A.mode = 1; A.seg_start = sstart; A.seg = seg; A.n_seg = n_seg; A.items = nullptr; A.n_items = h_sstart.back();
    A.e_max = e_max; A.t_bits = t_bits; A.t_uv = t_uv; A.t_cnt = t_cnt;
    TIP_CHECK_CUDA(cudaMemsetAsync(cnt + 1, 0, 8, st));
    if (A.n_items > 0) {
        tip_gene_rank_pass_kernel<<<(int)std::min<long long>((long long)sm_count() * per_sm1, A.n_items), kPredThreads, smem1, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    tip_gene_finish_kernel<<<(n_seg + 127) / 128, 128, 0, st>>>(n_seg, S, seg, t_cnt, t_bits, t_idx, t_tr, d_rank_out, d_score_out);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    return 0;
}

// ---- the digenic model: top-N gene pairs (tip_top_pairs, tip_top_pairs_per_gene) and test-set pair scores ----
// A pair of ranks a < b (already in key slot order) scores
//     score(a, b) = sum_ij th_a[i] qr[i][j][1] th_b[j] = V[a] . tcat[b],   V[x][s K + j] = sum_i th_x[s K + i] qr_s[i][j][1]
// (tip_pair_prep_kernel), the ensemble sum being the same dot product, S K long.  The pair universe is C(n, 2), so every score
// is computed once, in chunks of at most TIP_PAIR_CHUNK pairs, each scored into a bounded buffer and merged:
//   global    items of 64 rows x 128 columns of the upper triangle (tip_top_pairs_pass_kernel); a chunk keeps the scores at or
//             above the N-th best so far, appends them behind the running best N, and two stable radix sorts (packed ranks
//             ascending, then bits descending) put the running best N first again;
//   per gene  a chunk of queries x (n - 1) partners (tip_top_pairs_gene_kernel: the query's V row against the partners'
//             theta for x > r, the partners' V rows against the query's theta for x < r), then a stable segmented sort
//             by bits descending of the partners in ascending order, and the first N of every segment.
namespace tip {
namespace {

constexpr int kTpRows = 64;                 // rows of a global item (2 warps x 32)
constexpr int kTpCols = 128;                // columns of a global item (2 warps x 2 x 32)
constexpr long long kTpItemPairs = (long long)kTpRows * kTpCols;
constexpr long long kTpChunk = TIP_PAIR_CHUNK;
constexpr int kTpMaxRows = 1 << 24;         // per gene: n_query * N

// tcat[r] = theta rows of candidate r (tcat_entry), V[r] = its rows times qr[..][1]; Tq / Vq: the same rows of the queries,
// in the order of qsorted (per gene only)
__global__ void tip_pair_prep_kernel(int S, int P, int K, int n, int n_pad, int SKP, const double *__restrict__ theta,
                                     const double *__restrict__ q, const int32_t *__restrict__ cand, int n_q, int nq_pad,
                                     const int32_t *__restrict__ qsorted, double *__restrict__ tcat, double *__restrict__ V,
                                     double *__restrict__ Tq, double *__restrict__ Vq)
{
    const long long n_t = (long long)n_pad * SKP, n_qt = (long long)nq_pad * SKP;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < 2 * n_t + 2 * n_qt;
         t += (long long)gridDim.x * blockDim.x) {
        const bool is_q = t >= 2 * n_t;
        const long long u = is_q ? t - 2 * n_t : t, m = is_q ? n_qt : n_t;
        const bool is_v = u >= m;
        const long long e = is_v ? u - m : u;
        long long row = e / SKP;
        const int col = (int)(e % SKP);
        if (is_q) row = row < n_q ? qsorted[row] : n;         // pad rows map to a zero row
        double val = 0.0;
        if (row < n && col < S * K) {
            const int s = col / K, j = col % K;
            const double *th = theta + ((long long)s * P + cand[row]) * K;
            if (is_v) {
                const double *qs = q + (long long)s * 2 * K * K;
                for (int i = 0; i < K; ++i) val = fma(th[i], qs[((long long)i * K + j) * 2 + 1], val);
            } else {
                val = th[j];
            }
        }
        double *out = is_q ? (is_v ? Vq : Tq) : (is_v ? V : tcat);
        out[e] = val;
    }
}

__device__ __forceinline__ bool pair_key_known(const unsigned long long *known, long long n, unsigned long long key)
{
    long long lo = 0, hi = n;
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (__ldg(known + mid) < key) lo = mid + 1; else hi = mid;
    }
    return lo < n && __ldg(known + lo) == key;
}

struct TopPairArgs {
    int n, SKP;
    const double *V, *tcat;             // [n_pad][SKP]
    const unsigned long long *known;    // sorted packed pairs (ra << 21) | rb
    long long n_known;
    const long long *tile_item;         // [n_tiles + 1] first item of every row tile
    int n_tiles;
    long long item0;                    // first item of the chunk
    const unsigned long long *thr;      // [0]: bits of the N-th best so far (0: keep everything)
    unsigned long long *counter;        // entries appended
    unsigned long long *out_bits, *out_packed;
};

// an item is 64 rows a0.. of one row tile and 128 columns c0..; pairs b > a only
__global__ void __launch_bounds__(kPredThreads) tip_top_pairs_pass_kernel(TopPairArgs A)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    const long long item = A.item0 + blockIdx.x;
    int tl = 0, th = A.n_tiles - 1;
    while (tl < th) {
        const int mid = (tl + th + 1) >> 1;
        if (A.tile_item[mid] <= item) tl = mid; else th = mid - 1;
    }
    const int a0 = tl * kTpRows + wr * 32;
    const int cs = tl * kTpRows + (int)(item - A.tile_item[tl]) * kTpCols;
    const int n = A.n, SKP = A.SKP;
    const unsigned long long thr = *A.thr;
    if (a0 >= n - 1) return;
    for (int h = 0; h < 2; ++h) {
        const int c0 = cs + h * 64 + wc * 32;
        if (c0 >= n || c0 + 31 <= a0) continue;       // outside the candidates, or wholly on or below the diagonal
        double acc[4][4][2];
        dmma_block(acc, A.V + (long long)(a0 + gq) * SKP + tq, SKP, A.tcat + (long long)(c0 + gq) * SKP + tq, SKP);
#pragma unroll
        for (int f = 0; f < 32; ++f) {
            const int mi = f >> 3, ni = (f >> 1) & 3, e = f & 1;
            const int ra = a0 + gq + mi * 8, rb = c0 + 2 * tq + ni * 8 + e;
            const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
            const unsigned long long packed = ((unsigned long long)ra << kRankBits) | (unsigned long long)rb;
            bool keep = rb < n && rb > ra && bits >= thr;
            if (keep && A.n_known > 0) keep = !pair_key_known(A.known, A.n_known, packed);
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            if (m == 0) continue;
            unsigned long long base = 0;
            if (lane == __ffs(m) - 1) base = atomicAdd(A.counter, (unsigned long long)__popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            if (keep) {
                const unsigned long long idx = base + __popc(m & ((1u << lane) - 1u));
                A.out_bits[idx] = bits;
                A.out_packed[idx] = packed;
            }
        }
    }
}

__global__ void tip_top_pairs_finish_kernel(long long m, int S, const unsigned long long *__restrict__ bits,
                                            const unsigned long long *__restrict__ packed, const int32_t *__restrict__ cand,
                                            int32_t *__restrict__ out_ids, double *__restrict__ out_scores)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const unsigned long long pk = packed[i], mask = (1ull << kRankBits) - 1;
    out_ids[2 * i + 0] = cand[(pk >> kRankBits) & mask];
    out_ids[2 * i + 1] = cand[pk & mask];
    out_scores[i] = __longlong_as_double((long long)bits[i]) / (double)S;
}

struct GenePairArgs {
    int n, SKP, n_q;
    const double *V, *tcat;             // [n_pad][SKP]
    const double *Vq, *Tq;              // [nq_pad][SKP] rows of the chunk's queries
    const int32_t *qrank;               // [n_q] ranks of the chunk's queries, ascending
    const unsigned long long *known;
    long long n_known;
    unsigned long long *key;            // [n_q][n - 1]: bits + 1 of partner x at x - (x > r); 0 for a known pair
    int32_t *part;                      // [n_q][n - 1]: x
};

// a CTA: 64 queries (blockIdx.y) x 128 partners (blockIdx.x); per warp block, x > r takes Vq[q] . tcat[x] and x < r takes
// Tq[q] . V[x], each product run only when the block holds such a partner
__global__ void __launch_bounds__(kPredThreads, 4) tip_top_pairs_gene_kernel(GenePairArgs A)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wr = warp & 1, wc = warp >> 1;
    const int gq = lane >> 2, tq = lane & 3;
    const int q0 = blockIdx.y * kTpRows + wr * 32;
    const int n = A.n, SKP = A.SKP;
    if (q0 >= A.n_q) return;
    const int rmin = A.qrank[q0], rmax = A.qrank[min(q0 + 31, A.n_q - 1)];
    int r[4];
#pragma unroll
    for (int mi = 0; mi < 4; ++mi) r[mi] = q0 + gq + mi * 8 < A.n_q ? A.qrank[q0 + gq + mi * 8] : -1;
    const long long stride = n - 1;
    for (int h = 0; h < 2; ++h) {
        const int c0 = blockIdx.x * kTpCols + h * 64 + wc * 32;
        if (c0 >= n) continue;
        for (int side = 0; side < 2; ++side) {         // 0: partners x > r, 1: partners x < r
            if (side == 0 ? c0 + 31 <= rmin : c0 >= rmax) continue;
            double acc[4][4][2];
            const double *Aq = side == 0 ? A.Vq : A.Tq, *Bx = side == 0 ? A.tcat : A.V;
            dmma_block(acc, Aq + (long long)(q0 + gq) * SKP + tq, SKP, Bx + (long long)(c0 + gq) * SKP + tq, SKP);
#pragma unroll
            for (int f = 0; f < 32; ++f) {
                const int mi = f >> 3, ni = (f >> 1) & 3, e = f & 1;
                const int x = c0 + 2 * tq + ni * 8 + e, rq = r[mi];
                if (rq < 0 || x >= n || (side == 0 ? x <= rq : x >= rq)) continue;
                const unsigned long long packed = side == 0 ? ((unsigned long long)rq << kRankBits) | (unsigned long long)x
                                                            : ((unsigned long long)x << kRankBits) | (unsigned long long)rq;
                const bool known = A.n_known > 0 && pair_key_known(A.known, A.n_known, packed);
                const long long pos = (long long)(q0 + gq + mi * 8) * stride + x - (side == 0 ? 1 : 0);
                A.key[pos] = known ? 0ull : (unsigned long long)__double_as_longlong(acc[mi][ni][e]) + 1ull;
                A.part[pos] = x;
            }
        }
    }
}

// the first min(N, n - 1) entries of every sorted segment that are not known pairs; out row of query qi: oq[qi]
__global__ void tip_top_pairs_gene_finish_kernel(int n_q, int n, long long N, int S, const unsigned long long *__restrict__ key,
                                                 const int32_t *__restrict__ part, const int32_t *__restrict__ qrank,
                                                 const int32_t *__restrict__ oq, const int32_t *__restrict__ cand,
                                                 unsigned long long *__restrict__ n_out, int32_t *__restrict__ out_ids,
                                                 double *__restrict__ out_scores)
{
    const long long m = N < n - 1 ? N : n - 1;
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)n_q * m) return;
    const long long qi = i / m, t = i % m;
    const unsigned long long k = key[qi * (n - 1) + t];
    if (k == 0) return;
    const int x = part[qi * (n - 1) + t], r = qrank[qi];
    const long long o = (long long)oq[qi] * N + t;
    out_ids[2 * o + 0] = cand[x < r ? x : r];
    out_ids[2 * o + 1] = cand[x < r ? r : x];
    out_scores[o] = __longlong_as_double((long long)(k - 1)) / (double)S;
    atomicAdd(n_out + oq[qi], 1ull);
}

// the test-set pair score of one parameter set (do_prediction's pair counterpart, rating 1, no eps)
__global__ void tip_score_pairs_kernel(int K, const int32_t *__restrict__ a, const int32_t *__restrict__ b, long long T,
                                       const double *__restrict__ theta, const double *__restrict__ q, double *__restrict__ out)
{
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < T; t += (long long)gridDim.x * blockDim.x) {
        const double *ta = theta + (long long)a[t] * K, *tb = theta + (long long)b[t] * K;
        double acc = 0.0;
        for (int i = 0; i < K; ++i) {
            double v = 0.0;
            for (int j = 0; j < K; ++j) v = fma(q[(i * K + j) * 2 + 1], tb[j], v);
            acc = fma(ta[i], v, acc);
        }
        out[t] = acc;
    }
}

// rows of the global sweep: row tiles of 64 over ranks 0 .. n-2, each with ceil((n - a0) / 128) column items
int tp_tiles(int n) { return n < 2 ? 0 : (n - 1 + kTpRows - 1) / kTpRows; }

struct TopPairLayout {
    size_t o_tcat, o_V, o_tile, o_thr, o_cnt, o_bits, o_pk, o_bits2, o_pk2, o_cub, cub_bytes, total;
    int n_pad, SKP;
    long long cap;
};

TopPairLayout top_pair_layout(int n, int K, int S, long long N)
{
    TopPairLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.cap = N + kTpChunk;
    size_t cb1 = 0, cb2 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cb1, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                    (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)L.cap, 0,
                                    2 * kRankBits, (cudaStream_t)0);
    cub::DeviceRadixSort::SortPairsDescending(nullptr, cb2, (const unsigned long long *)nullptr, (unsigned long long *)nullptr,
                                              (const unsigned long long *)nullptr, (unsigned long long *)nullptr, (int)L.cap, 0,
                                              63, (cudaStream_t)0);
    L.cub_bytes = std::max(cb1, cb2);
    size_t off = 0;
    L.o_tcat = off;  off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_V = off;     off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_tile = off;  off += a256(((size_t)tp_tiles(n) + 1) * 8);
    L.o_thr = off;   off += 256;
    L.o_cnt = off;   off += 256;
    L.o_bits = off;  off += a256((size_t)L.cap * 8);
    L.o_pk = off;    off += a256((size_t)L.cap * 8);
    L.o_bits2 = off; off += a256((size_t)L.cap * 8);
    L.o_pk2 = off;   off += a256((size_t)L.cap * 8);
    L.o_cub = off;   off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

// queries per chunk: as many whole segments of n - 1 partners as TIP_PAIR_CHUNK holds, at least one
int gp_chunk_queries(int n, int n_query)
{
    return (int)std::max(1ll, std::min<long long>(n_query, kTpChunk / std::max(1, n - 1)));
}

struct GenePairLayout {
    size_t o_tcat, o_V, o_Tq, o_Vq, o_qs, o_oq, o_off, o_nout, o_key, o_part, o_key2, o_part2, o_cub, cub_bytes, total;
    int n_pad, nq_pad, SKP, qc;
};

GenePairLayout gene_pair_layout(int n, int n_query, int K, int S)
{
    GenePairLayout L{};
    L.n_pad = (n + 63) / 64 * 64 + 64;
    L.nq_pad = (n_query + 63) / 64 * 64 + 64;
    L.SKP = (S * K + 3) / 4 * 4;
    L.qc = gp_chunk_queries(n, n_query);
    const long long items = (long long)L.qc * std::max(1, n - 1);
    size_t cb = 0;
    cub::DeviceSegmentedSort::StableSortPairsDescending(nullptr, cb, (const unsigned long long *)nullptr,
                                                        (unsigned long long *)nullptr, (const int32_t *)nullptr, (int32_t *)nullptr,
                                                        (int)items, L.qc, (const int *)nullptr, (const int *)nullptr, (cudaStream_t)0);
    L.cub_bytes = cb;
    size_t off = 0;
    L.o_tcat = off;  off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_V = off;     off += a256((size_t)L.n_pad * L.SKP * 8);
    L.o_Tq = off;    off += a256((size_t)L.nq_pad * L.SKP * 8);
    L.o_Vq = off;    off += a256((size_t)L.nq_pad * L.SKP * 8);
    L.o_qs = off;    off += a256((size_t)std::max(n_query, 1) * 4);
    L.o_oq = off;    off += a256((size_t)std::max(n_query, 1) * 4);
    L.o_off = off;   off += a256(((size_t)L.qc + 1) * 4);
    L.o_nout = off;  off += a256((size_t)std::max(n_query, 1) * 8);
    L.o_key = off;   off += a256((size_t)items * 8);
    L.o_part = off;  off += a256((size_t)items * 4);
    L.o_key2 = off;  off += a256((size_t)items * 8);
    L.o_part2 = off; off += a256((size_t)items * 4);
    L.o_cub = off;   off += a256(L.cub_bytes);
    L.total = off + 256;
    return L;
}

__global__ void tip_pair_offsets_kernel(int m, int len, int *__restrict__ off)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= m) off[i] = i * len;
}

int launch_pair_prep(int S, int P, int K, int n, int n_pad, int SKP, const double *theta, const double *q, const int32_t *cand,
                     int n_q, int nq_pad, const int32_t *qsorted, double *tcat, double *V, double *Tq, double *Vq, cudaStream_t st)
{
    const long long work = 2 * ((long long)n_pad + (n_q > 0 ? nq_pad : 0)) * SKP;
    const long long want = (work + 255) / 256;
    tip_pair_prep_kernel<<<(int)std::max(1ll, std::min<long long>(want, (long long)sm_count() * 16)), 256, 0, st>>>(
        S, P, K, n, n_pad, SKP, theta, q, cand, n_q, n_q > 0 ? nq_pad : 0, qsorted, tcat, V, Tq, Vq);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace
}  // namespace tip

static thread_local int g_last_pair_chunks = 0;
static thread_local int g_last_gene_pair_chunks = 0;

static bool top_pairs_args_ok(int n_cand, int K, int S, int64_t N)
{
    return n_cand >= 0 && n_cand <= (1 << kRankBits) && K >= 1 && K <= TIP_MAX_K && S >= 1 && (long long)S * K <= kPredMaxSK &&
           N >= 0 && N < (1ll << 28);
}

#define TIP_TOP_PAIRS_LIMITS "n_cand <= 2^21, 1 <= K <= %d, S >= 1, S*K <= %d, 0 <= N < 2^28"
#define TIP_GENE_PAIRS_LIMITS "n_cand <= 2^21, 0 <= n_query <= n_cand, 1 <= K <= %d, S >= 1, S*K <= %d, N >= 0, n_query*N <= 2^24"

extern "C" int tip_score_pairs(int P, int K, const double *d_theta, const double *d_q, const int32_t *d_a, const int32_t *d_b,
                               int64_t T, double *d_out, void *stream)
{
    TIP_REQUIRE(P > 0 && K >= 1 && K <= TIP_MAX_K && T >= 0, "tip_score_pairs: bad arguments (P > 0, 1 <= K <= %d, T >= 0)",
                TIP_MAX_K);
    TIP_REQUIRE(d_theta && d_q && (T == 0 || (d_a && d_b && d_out)), "tip_score_pairs: null pointer");
    if (T == 0) return 0;
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    const long long want = (T + 255) / 256;
    tip_score_pairs_kernel<<<(int)std::min<long long>(want, (long long)sm_count() * 32), 256, 0, st>>>(K, d_a, d_b, T, d_theta,
                                                                                                     d_q, d_out);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

extern "C" int tip_top_pairs_workspace_bytes(int n_cand, int K, int S, int64_t N, size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && top_pairs_args_ok(n_cand, K, S, N),
                "tip_top_pairs_workspace_bytes: bad arguments (" TIP_TOP_PAIRS_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    *bytes = top_pair_layout(n_cand, K, S, N).total;
    return 0;
}

extern "C" int tip_top_pairs(int P, int K, int S, const double *d_theta, const double *d_q, const int32_t *d_cand, int n_cand,
                             const uint64_t *d_known, int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes, int32_t *d_out_ids,
                             double *d_out_scores, int64_t *h_n_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && top_pairs_args_ok(n_cand, K, S, N) && n_known >= 0 && h_n_out != nullptr,
                "tip_top_pairs: bad arguments (P > 0, n_known >= 0, " TIP_TOP_PAIRS_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_q && (d_cand || n_cand == 0) && (d_known || n_known == 0) && (N == 0 || (d_out_ids && d_out_scores)),
                "tip_top_pairs: null pointer");
    *h_n_out = 0;
    g_last_pair_chunks = 0;
    const int n = n_cand;
    if (N == 0 || n < 2) return 0;
    const TopPairLayout L = top_pair_layout(n, K, S, N);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_top_pairs: workspace too small (%zu < %zu)", ws_bytes, L.total);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *V = reinterpret_cast<double *>(base + L.o_V);
    auto *tile = reinterpret_cast<long long *>(base + L.o_tile);
    auto *thr = reinterpret_cast<unsigned long long *>(base + L.o_thr), *cnt = reinterpret_cast<unsigned long long *>(base + L.o_cnt);
    auto *bits = reinterpret_cast<unsigned long long *>(base + L.o_bits), *pk = reinterpret_cast<unsigned long long *>(base + L.o_pk);
    auto *bits2 = reinterpret_cast<unsigned long long *>(base + L.o_bits2), *pk2 = reinterpret_cast<unsigned long long *>(base + L.o_pk2);
    void *cub_tmp = base + L.o_cub;

    if (int rc = launch_pair_prep(S, P, K, n, L.n_pad, L.SKP, d_theta, d_q, d_cand, 0, 0, nullptr, tcat, V, nullptr, nullptr, st))
        return rc;
    // items: row tile t holds ceil((n - 64 t) / 128) of them
    const int n_tiles = tp_tiles(n);
    std::vector<long long> h_tile((size_t)n_tiles + 1, 0);
    for (int t = 0; t < n_tiles; ++t) h_tile[t + 1] = h_tile[t] + (n - t * kTpRows + kTpCols - 1) / kTpCols;
    const long long n_items = h_tile[n_tiles];
    TIP_CHECK_CUDA(cudaMemcpyAsync(tile, h_tile.data(), ((size_t)n_tiles + 1) * 8, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemsetAsync(thr, 0, 8, st));

    TopPairArgs A{};
    A.n = n; A.SKP = L.SKP; A.V = V; A.tcat = tcat;
    A.known = reinterpret_cast<const unsigned long long *>(d_known); A.n_known = n_known;
    A.tile_item = tile; A.n_tiles = n_tiles; A.thr = thr; A.counter = cnt;
    const long long per_chunk = kTpChunk / kTpItemPairs;
    long long have = 0;          // running best, sorted, at bits[0, have) / pk[0, have)
    for (long long i0 = 0; i0 < n_items; i0 += per_chunk) {
        const long long items = std::min(per_chunk, n_items - i0);
        TIP_CHECK_CUDA(cudaMemsetAsync(cnt, 0, 8, st));
        A.item0 = i0; A.out_bits = bits + have; A.out_packed = pk + have;
        tip_top_pairs_pass_kernel<<<(int)items, kPredThreads, 0, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
        unsigned long long h_cnt = 0;
        TIP_CHECK_CUDA(cudaMemcpyAsync(&h_cnt, cnt, 8, cudaMemcpyDeviceToHost, st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(st));
        ++g_last_pair_chunks;
        if (h_cnt == 0) continue;
        const int total = (int)(have + (long long)h_cnt);
        // packed ranks ascending, then (stable) bits descending: the running best N come first
        size_t cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(cub_tmp, cb, pk, pk2, bits, bits2, total, 0, 2 * kRankBits, st));
        cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(cub_tmp, cb, bits2, bits, pk2, pk, total, 0, 63, st));
        have = std::min<long long>(N, total);
        if (have == N) TIP_CHECK_CUDA(cudaMemcpyAsync(thr, bits + N - 1, 8, cudaMemcpyDeviceToDevice, st));
    }
    if (have > 0) {
        tip_top_pairs_finish_kernel<<<(int)((have + 255) / 256), 256, 0, st>>>(have, S, bits, pk, d_cand, d_out_ids, d_out_scores);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    *h_n_out = have;
    return 0;
}

extern "C" int tip_top_pairs_last_chunks(void) { return g_last_pair_chunks; }

static bool gene_pairs_args_ok(int n_cand, int n_query, int K, int S, int64_t N)
{
    return n_cand >= 0 && n_cand <= (1 << kRankBits) && K >= 1 && K <= TIP_MAX_K && S >= 1 && (long long)S * K <= kPredMaxSK &&
           n_query >= 0 && n_query <= n_cand && N >= 0 && (long long)n_query * N <= kTpMaxRows;
}

extern "C" int tip_top_pairs_per_gene_workspace_bytes(int n_cand, int n_query, int K, int S, int64_t N, size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && gene_pairs_args_ok(n_cand, n_query, K, S, N),
                "tip_top_pairs_per_gene_workspace_bytes: bad arguments (" TIP_GENE_PAIRS_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    *bytes = gene_pair_layout(n_cand, n_query, K, S).total;
    return 0;
}

extern "C" int tip_top_pairs_per_gene(int P, int K, int S, const double *d_theta, const double *d_q, const int32_t *d_cand,
                                      int n_cand, const int32_t *d_query_ranks, int n_query, const uint64_t *d_known,
                                      int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes, int32_t *d_out_ids,
                                      double *d_out_scores, int64_t *h_n_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && n_cand <= P && gene_pairs_args_ok(n_cand, n_query, K, S, N) && n_known >= 0 && (h_n_out || n_query == 0),
                "tip_top_pairs_per_gene: bad arguments (P > 0, n_known >= 0, " TIP_GENE_PAIRS_LIMITS ")", TIP_MAX_K, kPredMaxSK);
    TIP_REQUIRE(d_theta && d_q && (d_cand || n_cand == 0) && (d_query_ranks || n_query == 0) && (d_known || n_known == 0) &&
                    (N == 0 || n_query == 0 || (d_out_ids && d_out_scores)),
                "tip_top_pairs_per_gene: null pointer");
    g_last_gene_pair_chunks = 0;
    if (n_query == 0) return 0;
    const int n = n_cand, nq = n_query;
    // the query ranks are checked on the host before any device work
    std::vector<int32_t> qr(nq);
    TIP_CHECK_CUDA(cudaMemcpyAsync(qr.data(), d_query_ranks, (size_t)nq * 4, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    {
        std::vector<char> seen(n, 0);
        for (int i = 0; i < nq; ++i) {
            TIP_REQUIRE(qr[i] >= 0 && qr[i] < n, "tip_top_pairs_per_gene: query rank %d of query %d is not in [0, %d)", qr[i], i, n);
            TIP_REQUIRE(!seen[qr[i]], "tip_top_pairs_per_gene: query rank %d appears twice", qr[i]);
            seen[qr[i]] = 1;
        }
    }
    for (int i = 0; i < nq; ++i) h_n_out[i] = 0;
    if (N == 0 || n < 2) return 0;
    const GenePairLayout L = gene_pair_layout(n, nq, K, S);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= L.total, "tip_top_pairs_per_gene: workspace too small (%zu < %zu)", ws_bytes,
                L.total);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    double *tcat = reinterpret_cast<double *>(base + L.o_tcat), *V = reinterpret_cast<double *>(base + L.o_V);
    double *Tq = reinterpret_cast<double *>(base + L.o_Tq), *Vq = reinterpret_cast<double *>(base + L.o_Vq);
    auto *qs = reinterpret_cast<int32_t *>(base + L.o_qs), *oq = reinterpret_cast<int32_t *>(base + L.o_oq);
    auto *off = reinterpret_cast<int *>(base + L.o_off);
    auto *n_out = reinterpret_cast<unsigned long long *>(base + L.o_nout);
    auto *key = reinterpret_cast<unsigned long long *>(base + L.o_key), *key2 = reinterpret_cast<unsigned long long *>(base + L.o_key2);
    auto *part = reinterpret_cast<int32_t *>(base + L.o_part), *part2 = reinterpret_cast<int32_t *>(base + L.o_part2);
    void *cub_tmp = base + L.o_cub;

    // queries in ascending rank order, so that a warp's rows span a short range of ranks; oq maps them back
    std::vector<int32_t> order(nq);
    for (int i = 0; i < nq; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return qr[a] < qr[b]; });
    std::vector<int32_t> h_qs(nq);
    for (int i = 0; i < nq; ++i) h_qs[i] = qr[order[i]];
    TIP_CHECK_CUDA(cudaMemcpyAsync(qs, h_qs.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(oq, order.data(), (size_t)nq * 4, cudaMemcpyHostToDevice, st));
    TIP_CHECK_CUDA(cudaMemsetAsync(n_out, 0, (size_t)nq * 8, st));
    if (int rc = launch_pair_prep(S, P, K, n, L.n_pad, L.SKP, d_theta, d_q, d_cand, nq, L.nq_pad, qs, tcat, V, Tq, Vq, st))
        return rc;
    tip_pair_offsets_kernel<<<(L.qc + 256) / 256, 256, 0, st>>>(L.qc, n - 1, off);
    TIP_CHECK_CUDA(cudaGetLastError());

    GenePairArgs A{};
    A.n = n; A.SKP = L.SKP; A.V = V; A.tcat = tcat;
    A.known = reinterpret_cast<const unsigned long long *>(d_known); A.n_known = n_known;
    A.key = key; A.part = part;
    const int col_tiles = (n + kTpCols - 1) / kTpCols;
    const long long m = std::min<long long>(N, n - 1);
    for (int c = 0; c < nq; c += L.qc) {
        const int cq = std::min(L.qc, nq - c);
        A.n_q = cq; A.qrank = qs + c; A.Vq = Vq + (long long)c * L.SKP; A.Tq = Tq + (long long)c * L.SKP;
        tip_top_pairs_gene_kernel<<<dim3(col_tiles, (cq + kTpRows - 1) / kTpRows), kPredThreads, 0, st>>>(A);
        TIP_CHECK_CUDA(cudaGetLastError());
        const int items = cq * (n - 1);
        size_t cb = L.cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceSegmentedSort::StableSortPairsDescending(cub_tmp, cb, key, key2, part, part2, items, cq, off,
                                                                          off + 1, st));
        const long long rows = (long long)cq * m;
        tip_top_pairs_gene_finish_kernel<<<(int)((rows + 255) / 256), 256, 0, st>>>(cq, n, N, S, key2, part2, qs + c, oq + c, d_cand,
                                                                                   n_out, d_out_ids, d_out_scores);
        TIP_CHECK_CUDA(cudaGetLastError());
        ++g_last_gene_pair_chunks;
    }
    std::vector<unsigned long long> h_out(nq);
    TIP_CHECK_CUDA(cudaMemcpyAsync(h_out.data(), n_out, (size_t)nq * 8, cudaMemcpyDeviceToHost, st));
    TIP_CHECK_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < nq; ++i) h_n_out[i] = (int64_t)h_out[i];
    return 0;
}

extern "C" int tip_top_pairs_per_gene_last_chunks(void) { return g_last_gene_pair_chunks; }
