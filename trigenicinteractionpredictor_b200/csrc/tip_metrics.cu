// Integer part of Model.calculate_metrics (TIP.py:583-637) on the device: the strict-greater pair
// count behind the AUC and the confusion counts at the rank-cut threshold.
//
// The reference's O(pos*neg) loop (TIP.py:611-615) counts pairs with score_pos > score_neg.  With the
// scores sorted ascending, a positive at rank i beats exactly the negatives that lie before the first
// element equal to it, so  wins = sum_{i: label=1} negatives_before[lower_bound(score_i)].
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "tip_common.cuh"

namespace tip {

__global__ void neg_flag_kernel(const int32_t *__restrict__ labels, int64_t T, int32_t *__restrict__ neg)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T; i += (int64_t)gridDim.x * blockDim.x)
        neg[i] = labels[i] ? 0 : 1;
}

// out: {wins, n_pos, n_neg, tp, fp, fn, tn, cut bits}
__global__ void metrics_count_kernel(const double *__restrict__ sorted, const int32_t *__restrict__ labels,
                                     const int64_t *__restrict__ neg_before, int64_t T, int64_t positives_number,
                                     unsigned long long *__restrict__ out)
{
    const double cut = positives_number < T ? sorted[T - 1 - positives_number] : 0.0;  // TIP.py:595-599
    unsigned long long wins = 0, npos = 0, nneg = 0, tp = 0, fp = 0, fn = 0, tn = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < T; i += (int64_t)gridDim.x * blockDim.x) {
        const double s = sorted[i];
        const bool pos = labels[i] != 0;
        if (pos) {
            int64_t lo = 0, hi = i;  // first index with sorted[idx] >= s, known to be <= i
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if (sorted[mid] < s) lo = mid + 1; else hi = mid;
            }
            wins += (unsigned long long)neg_before[lo];
            ++npos;
        } else {
            ++nneg;
        }
        if (s >= cut) {                       // TIP.py:622
            if (pos) ++tp; else ++fp;
        } else {
            if (pos) ++fn; else ++tn;
        }
    }
    unsigned long long v[7] = {wins, npos, nneg, tp, fp, fn, tn};
#pragma unroll
    for (int k = 0; k < 7; ++k) {
        unsigned long long x = v[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
        if ((threadIdx.x & 31) == 0 && x) atomicAdd(out + k, x);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[7] = (unsigned long long)__double_as_longlong(cut);
}

struct MetWs {
    double *keys_out;
    int32_t *labels_out, *neg;
    int64_t *neg_before;
    void *cub_tmp;
    size_t cub_bytes;
};

static size_t a256(size_t x) { return (x + 255) / 256 * 256; }

static size_t metrics_layout(int64_t T, void *base, MetWs *ws)
{
    size_t sort_bytes = 0, scan_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, (const double *)nullptr, (double *)nullptr,
                                    (const int32_t *)nullptr, (int32_t *)nullptr, T, 0, 64, (cudaStream_t)0);
    cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, (const int32_t *)nullptr, (int64_t *)nullptr, T, (cudaStream_t)0);
    const size_t cub_bytes = sort_bytes > scan_bytes ? sort_bytes : scan_bytes;
    size_t off = 0;
    auto take = [&](size_t b) { size_t o = off; off += a256(b); return o; };
    const size_t o_k = take((size_t)T * 8), o_l = take((size_t)T * 4), o_n = take((size_t)T * 4),
                 o_b = take((size_t)T * 8), o_c = take(cub_bytes);
    if (ws) {
        char *b = reinterpret_cast<char *>(base);
        ws->keys_out = reinterpret_cast<double *>(b + o_k);
        ws->labels_out = reinterpret_cast<int32_t *>(b + o_l);
        ws->neg = reinterpret_cast<int32_t *>(b + o_n);
        ws->neg_before = reinterpret_cast<int64_t *>(b + o_b);
        ws->cub_tmp = b + o_c;
        ws->cub_bytes = cub_bytes;
    }
    return off + 256;
}

__global__ void iota_kernel(int32_t *v, int64_t n)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) v[i] = (int32_t)i;
}

static size_t sort_scores_layout(int64_t T, size_t *o_idx, size_t *o_cub, size_t *cub_bytes)
{
    size_t cb = 0;
    cub::DeviceRadixSort::SortPairsDescending(nullptr, cb, (const double *)nullptr, (double *)nullptr, (const int32_t *)nullptr,
                                              (int32_t *)nullptr, T, 0, 64, (cudaStream_t)0);
    *o_idx = 0;
    *o_cub = a256((size_t)T * 4);
    *cub_bytes = cb;
    return *o_cub + a256(cb) + 256;
}

}  // namespace tip

using namespace tip;

extern "C" int tip_sort_scores_workspace_bytes(int64_t T, size_t *bytes)
{
    TIP_REQUIRE(T >= 0 && bytes != nullptr, "tip_sort_scores_workspace_bytes: bad arguments");
    size_t a, b, c;
    *bytes = sort_scores_layout(T < 1 ? 1 : T, &a, &b, &c);
    return 0;
}

extern "C" int tip_sort_scores(const double *d_scores, int64_t T, void *d_ws, size_t ws_bytes, int32_t *d_order,
                               double *d_sorted, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(T >= 0 && T < (1ll << 31), "tip_sort_scores: T out of range");
    if (T == 0) return 0;
    size_t o_idx, o_cub, cub_bytes;
    const size_t need = sort_scores_layout(T, &o_idx, &o_cub, &cub_bytes);
    TIP_REQUIRE(d_scores && d_order && d_sorted && d_ws && ws_bytes >= need, "tip_sort_scores: workspace too small (%zu < %zu)",
                ws_bytes, need);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    int32_t *idx = reinterpret_cast<int32_t *>(base + o_idx);
    const int64_t want = (T + 255) / 256;
    iota_kernel<<<(int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8), 256, 0, st>>>(idx, T);
    TIP_CHECK_CUDA(cudaGetLastError());
    size_t cb = cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(base + o_cub, cb, d_scores, d_sorted, idx, d_order, T, 0, 64, st));
    return 0;
}

extern "C" int tip_metrics_workspace_bytes(int64_t T, size_t *bytes)
{
    TIP_REQUIRE(T >= 0 && bytes != nullptr, "tip_metrics_workspace_bytes: bad arguments");
    *bytes = metrics_layout(T < 1 ? 1 : T, nullptr, nullptr);
    return 0;
}

extern "C" int tip_metrics(const double *d_scores, const int32_t *d_labels, int64_t T, int64_t positives_number,
                           void *d_ws, size_t ws_bytes, int64_t *d_out, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(T > 0, "tip_metrics: empty test set (the reference raises ZeroDivisionError; the caller handles it)");
    // the exclusive scan of the int32 negative flags accumulates in int32 (CUB takes the input type), so neg_before
    // would wrap past 2^31 - 1 negatives
    TIP_REQUIRE(T < (1ll << 31), "tip_metrics: T = %lld; need T < 2^31", (long long)T);
    TIP_REQUIRE(positives_number >= 0, "tip_metrics: negative positives_number");
    const size_t need = metrics_layout(T, nullptr, nullptr);
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= need, "tip_metrics: workspace too small (%zu < %zu)", ws_bytes, need);
    uintptr_t basep = (reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256;
    MetWs ws;
    metrics_layout(T, reinterpret_cast<void *>(basep), &ws);
    size_t cb = ws.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(ws.cub_tmp, cb, d_scores, ws.keys_out, d_labels, ws.labels_out, T, 0, 64, st));
    const int threads = 256;
    int64_t want = (T + threads - 1) / threads;
    int grid = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
    neg_flag_kernel<<<grid, threads, 0, st>>>(ws.labels_out, T, ws.neg);
    TIP_CHECK_CUDA(cudaGetLastError());
    cb = ws.cub_bytes;
    TIP_CHECK_CUDA(cub::DeviceScan::ExclusiveSum(ws.cub_tmp, cb, ws.neg, ws.neg_before, T, st));
    TIP_CHECK_CUDA(cudaMemsetAsync(d_out, 0, 8 * sizeof(int64_t), st));
    metrics_count_kernel<<<grid, threads, 0, st>>>(ws.keys_out, ws.labels_out, ws.neg_before, T, positives_number,
                                                  reinterpret_cast<unsigned long long *>(d_out));
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}
