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
#include <algorithm>
#include <vector>

#include <cub/device/device_radix_sort.cuh>

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

struct PassArgs {
    int n, S, K, SK, SKP;
    const double *tcat;             // [n_pad][SKP] theta of every model, rank order, zero padded
    const double *W;                // [S][n][K][K]
    const unsigned long long *known;  // sorted packed rank triples
    long long n_known;
    long long n_items;
    int mode;                       // 0: keep bits >= lo; 1: keep bits > v, or bits == v and packed <= rhi
    unsigned long long lo, hi;      // mode 0: histogram range of score bits (bin 0 = highest)
    unsigned long long v, rlo, rhi; // mode 1: tied score bits and the histogram range of packed ranks (bin 0 = lowest)
    int shift;
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

__global__ void tip_predict_prep_kernel(int S, int P, int K, int n, int n_pad, int SKP, const double *__restrict__ theta,
                                        const double *__restrict__ p, const int32_t *__restrict__ cand, double *__restrict__ tcat,
                                        double *__restrict__ W)
{
    const long long n_t = (long long)n_pad * SKP, KK = (long long)K * K, n_w = (long long)S * n * KK;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_t + n_w; t += (long long)gridDim.x * blockDim.x) {
        if (t < n_t) {
            const int r = (int)(t / SKP), col = (int)(t % SKP);
            double v = 0.0;
            if (r < n && col < S * K) {
                const int s = col / K, k = col % K;
                v = theta[((long long)s * P + cand[r]) * K + k];
            }
            tcat[t] = v;
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

        // Q tile: Q[i][s K + z] = sum_x th_{a0+i}[s K + x] W[s][j][x][z]; pad columns are zero
        for (int e = tid; e < kPredRows * SKP; e += kPredThreads) {
            const int i = e / SKP, col = e % SKP;
            double acc = 0.0;
            if (i < rows && col < A.SK) {
                const int s = col / K, z = col % K;
                const double *th = A.tcat + (long long)(a0 + i) * SKP + s * K;
                const double *Wb = A.W + ((long long)s * n + j) * K * K + z;
                for (int x = 0; x < K; ++x) acc = fma(__ldg(th + x), __ldg(Wb + x * K), acc);
            }
            Q[i * qs + col] = acc;
        }
        __syncthreads();

        const bool warp_rows = wr * 32 < rows;
        if (warp_rows) {
            const double *Qw = Q + (wr * 32 + gq) * qs + tq;
            for (int c0 = j + 1 + wc * 32; c0 < n; c0 += 64) {
                double acc[4][4][2];
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni) acc[mi][ni][0] = acc[mi][ni][1] = 0.0;
                const double *Bw = A.tcat + (long long)(c0 + gq) * SKP + tq;
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
                // epilogue: the threshold test runs in registers; only survivors go further
                unsigned keep = 0;
#pragma unroll
                for (int mi = 0; mi < 4; ++mi)
#pragma unroll
                    for (int ni = 0; ni < 4; ++ni)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
                            const bool pass = A.mode == 0 ? bits >= A.lo : bits >= A.v;
                            keep |= (pass ? 1u : 0u) << ((mi * 4 + ni) * 2 + e);
                        }
                if (!__any_sync(0xffffffffu, keep != 0)) continue;
#pragma unroll
                for (int f = 0; f < 32; ++f) {
                    const int mi = f >> 3, ni = (f >> 1) & 3, e = f & 1;
                    const int ra = a0 + wr * 32 + mi * 8 + gq, rc = c0 + ni * 8 + 2 * tq + e;
                    const unsigned long long bits = (unsigned long long)__double_as_longlong(acc[mi][ni][e]);
                    const unsigned long long packed = ((unsigned long long)ra << (2 * kRankBits)) |
                                                      ((unsigned long long)j << kRankBits) | (unsigned long long)rc;
                    bool q = ((keep >> f) & 1u) && ra < j && rc < n;
                    if (q && A.mode == 1) q = bits > A.v || packed <= A.rhi;
                    if (q && A.n_known > 0) q = !is_known(A.known, A.n_known, packed);
                    int bin = kPredBins;
                    if (q) {
                        if (A.mode == 0) {
                            if (bits <= A.hi) bin = (int)((A.hi - bits) >> A.shift);
                        } else if (bits == A.v && packed >= A.rlo) {
                            bin = (int)((packed - A.rlo) >> A.shift);
                        }
                        atomicAdd(sh_hist + bin, 1u);
                    }
                    const unsigned m = __ballot_sync(0xffffffffu, q);
                    if (m == 0) continue;
                    unsigned long long base = 0;
                    if (lane == __ffs(m) - 1) base = atomicAdd(A.counter, (unsigned long long)__popc(m));
                    base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
                    if (q) {
                        const unsigned long long idx = base + __popc(m & ((1u << lane) - 1u));
                        if ((long long)idx < A.cap) {
                            A.out_bits[idx] = bits;
                            A.out_packed[idx] = packed;
                        }
                    }
                }
            }
        }
        // shared bins are 32-bit: flush before they could overflow
        since_flush += (double)rows * n_c;
        if (since_flush > 2.0e9) {
            __syncthreads();
            for (int i = tid; i <= kPredBins; i += kPredThreads) {
                if (sh_hist[i]) atomicAdd(A.hist + i, (unsigned long long)sh_hist[i]);
                sh_hist[i] = 0;
            }
            since_flush = 0.0;
        }
    }
    for (int i = tid; i <= kPredBins; i += kPredThreads)
        if (sh_hist[i]) atomicAdd(A.hist + i, (unsigned long long)sh_hist[i]);
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
    A.mode = 0;
    A.hi = kInfBits;
    A.lo = 0;
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
            int rc = sample_at(samp_idx, &A.lo);
            if (rc) return rc;
            rc = sample_at(0, &A.hi);
            if (rc) return rc;
        }
    }
    A.shift = shift_for(A.hi - A.lo);

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
            if (A.mode == 0 && A.lo == 0) { M = C; kept = C; break; }   // every candidate is in the buffer
            // the sample placed the threshold too high: lower it to a sample value below it, or to zero
            unsigned long long v = A.lo;
            while (v >= A.lo) {
                samp_idx = samp_idx < 0 ? 0 : samp_idx * 4 + 16;
                if (samp_idx >= kPredSample) { v = 0; break; }
                if ((rc = sample_at(samp_idx, &v))) return rc;
            }
            A.lo = v;
            A.shift = shift_for(A.hi - A.lo);
            continue;
        }
        // too many for the buffer: walk the histogram in result order to the bin where the count reaches M
        long long cum = (long long)h_hist[kPredBins];
        if (A.mode == 0 && cum >= M) {
            // everything needed lies above the histogram's range
            A.lo = A.hi + 1;
            A.hi = kInfBits;
            A.shift = shift_for(A.hi - A.lo);
            continue;
        }
        int b = 0;
        for (; b < kPredBins; ++b) {
            cum += (long long)h_hist[b];
            if (cum >= M) break;
        }
        TIP_REQUIRE(b < kPredBins, "tip_top_triplets: histogram does not reach N (internal error)");
        if (A.mode == 0) {
            const unsigned long long top = A.hi - ((unsigned long long)b << A.shift);
            const unsigned long long width = (A.shift >= 64) ? ~0ull : (1ull << A.shift);
            const unsigned long long bottom = (top - A.lo + 1 <= width) ? A.lo : top - width + 1;
            if (cum <= L.cap) {
                A.lo = bottom;
            } else if (bottom == top) {
                // every remaining candidate has the same score: continue on the packed ranks
                A.mode = 1;
                A.v = top;
                A.rlo = 0;
                A.rhi = max_packed;
            } else {
                A.lo = bottom;
                A.hi = top;
            }
        } else {
            const unsigned long long lo_b = A.rlo + ((unsigned long long)b << A.shift);
            const unsigned long long hi_b = std::min(A.rhi, lo_b + ((A.shift >= 64) ? ~0ull : (1ull << A.shift) - 1));
            if (cum <= L.cap) {
                A.rhi = hi_b;
            } else {
                A.rlo = lo_b;
                A.rhi = hi_b;
            }
        }
        A.shift = A.mode == 0 ? shift_for(A.hi - A.lo) : shift_for(A.rhi - A.rlo);
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
