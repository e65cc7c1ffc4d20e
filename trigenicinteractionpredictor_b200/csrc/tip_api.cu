// extern "C" surface of libtip.so (see include/tip.h), the host-buffer entry and the peak probes.
#include <stdarg.h>
#include <string.h>

#include <chrono>

#include "tip_common.cuh"

namespace tip {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

static bool valid_K(int K) { return K >= 1 && K <= TIP_MAX_K; }
// K-specialised kernels: K <= 10 always; K = 11..16 in plain fp64 mode (no by-product, no fp32 mode);
// K = 17..32 in the gene-segmented formulation (the only specialised one there)
static bool uses_tuned(int K, unsigned flags)
{
    if (flags & TIP_EM_FORCE_GENERIC) return false;
    if (K <= 10) return true;
    return !(flags & (TIP_EM_WITH_LOGLIK | TIP_EM_FP32_COMPUTE));
}
static bool seg_flag(unsigned flags) { return (flags & TIP_EM_GENE_SEGMENTED) != 0; }
static bool seg3_flag(unsigned flags) { return (flags & TIP_EM_SLOT_SEGMENTED) != 0; }

}  // namespace tip

using namespace tip;

extern "C" int tip_abi_version(void) { return TIP_ABI_VERSION; }
extern "C" const char *tip_last_error(void) { return g_err; }

extern "C" int64_t tip_stats_len(int P, int K) { return (int64_t)P * K + 2ll * K * K * K + 1; }

extern "C" int tip_em_workspace_bytes(int P, int K, int64_t n_rows, unsigned flags, size_t *bytes)
{
    TIP_REQUIRE(bytes != nullptr && P > 0 && valid_K(K) && n_rows >= 0, "tip_em_workspace_bytes: bad arguments");
    if (seg3_flag(flags)) {
        *bytes = em_seg3_workspace_bytes(P, K, n_rows);
        return 0;
    }
    *bytes = uses_tuned(K, flags) ? em_tuned_workspace_bytes(P, K, seg_flag(flags))
                                  : (size_t)(n_rows < 1 ? 1 : n_rows) * sizeof(double);
    return 0;
}

extern "C" int tip_em_step(int P, int K, const void *d_rows, int64_t n_rows, int64_t n_rows_r0, const double *d_theta,
                           const double *d_p, double *d_stats, void *d_ws, size_t ws_bytes, unsigned flags, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && valid_K(K), "tip_em_step: need P > 0 and 1 <= K <= %d (got P=%d K=%d)", TIP_MAX_K, P, K);
    TIP_REQUIRE(n_rows >= 0 && n_rows % 32 == 0 && n_rows_r0 >= 0 && n_rows_r0 <= n_rows && n_rows_r0 % 32 == 0,
                "tip_em_step: n_rows (%lld) and n_rows_r0 (%lld) must be multiples of 32 from tip_pack_rows",
                (long long)n_rows, (long long)n_rows_r0);
    TIP_REQUIRE(d_theta && d_p && d_stats && (d_rows || n_rows == 0), "tip_em_step: null pointer");
    TIP_REQUIRE(!(flags & TIP_EM_FP32_COMPUTE) || (K <= 10 && !(flags & (TIP_EM_FORCE_GENERIC | TIP_EM_WITH_LOGLIK))),
                "tip_em_step: TIP_EM_FP32_COMPUTE exists for the K <= 10 kernels only, without FORCE_GENERIC / WITH_LOGLIK");
    TIP_REQUIRE(!seg_flag(flags) || !(flags & (TIP_EM_FORCE_GENERIC | TIP_EM_WITH_LOGLIK | TIP_EM_FP32_COMPUTE)),
                "tip_em_step: TIP_EM_GENE_SEGMENTED cannot be combined with other mode flags");
    TIP_REQUIRE(!seg3_flag(flags) || (flags & ~(TIP_EM_SLOT_SEGMENTED | TIP_EM_GATHER_L1)) == 0,
                "tip_em_step: TIP_EM_SLOT_SEGMENTED combines with TIP_EM_GATHER_L1 only");
    TIP_REQUIRE(seg3_flag(flags) || !(flags & TIP_EM_GATHER_L1), "tip_em_step: TIP_EM_GATHER_L1 needs TIP_EM_SLOT_SEGMENTED");
    TIP_CHECK_CUDA(cudaMemsetAsync(d_stats, 0, sizeof(double) * (size_t)tip_stats_len(P, K), st));
    if (n_rows == 0) return 0;
    const int4 *rows = reinterpret_cast<const int4 *>(d_rows);
    if (seg3_flag(flags)) {
        const size_t need = em_seg3_workspace_bytes(P, K, n_rows);
        TIP_REQUIRE(d_ws != nullptr && ws_bytes >= need,
                    "tip_em_step: the slot-segmented mode needs %zu bytes of workspace (got %zu), see tip_em_workspace_bytes",
                    need, ws_bytes);
        return launch_em_seg3(P, K, rows, n_rows, n_rows_r0, d_theta, d_p, d_stats, reinterpret_cast<double *>(d_ws),
                              (flags & TIP_EM_GATHER_L1) != 0, st);
    }
    if (uses_tuned(K, flags)) {
        const size_t need = em_tuned_workspace_bytes(P, K, seg_flag(flags));
        TIP_REQUIRE(need == 0 || (d_ws != nullptr && ws_bytes >= need),
                    "tip_em_step: K=%d needs %zu bytes of workspace (got %zu), see tip_em_workspace_bytes", K, need, ws_bytes);
        bool handled = false;
        int rc = launch_em_tuned(P, K, rows, n_rows, n_rows_r0, d_theta, d_p, d_stats, reinterpret_cast<double *>(d_ws),
                                 (flags & TIP_EM_WITH_LOGLIK) != 0, (flags & TIP_EM_FP32_COMPUTE) != 0, seg_flag(flags), st,
                                 &handled);
        if (rc != 0 || handled) return rc;
    }
    TIP_REQUIRE(d_ws != nullptr && ws_bytes >= (size_t)n_rows * sizeof(double),
                "tip_em_step: the any-K path needs %zu bytes of workspace (got %zu)", (size_t)n_rows * sizeof(double), ws_bytes);
    return launch_em_generic(P, K, rows, n_rows, n_rows_r0, d_theta, d_p, d_stats, reinterpret_cast<double *>(d_ws), st);
}

extern "C" int tip_em_step_host_rows(int P, int K, const void *h_rows, int64_t n_rows, int64_t n_rows_r0, unsigned row_flags,
                                     void *d_rows_dev, const double *d_theta, const double *d_p, double *d_stats, void *d_ws,
                                     size_t ws_bytes, unsigned *d_err, void *stream, void *copy_stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream), cs = reinterpret_cast<cudaStream_t>(copy_stream);
    TIP_REQUIRE(P > 0 && valid_K(K) && em_streamed_available(K, false, false, false),
                "tip_em_step_host_rows: the streamed E-step exists for the plain fp64 K <= 10 kernels (got K=%d); copy the "
                "rows and call tip_em_step", K);
    TIP_REQUIRE(n_rows > 0 && n_rows % 32 == 0 && n_rows_r0 >= 0 && n_rows_r0 <= n_rows && n_rows_r0 % 32 == 0,
                "tip_em_step_host_rows: n_rows (%lld) and n_rows_r0 (%lld) must be multiples of 32 from tip_pack_rows",
                (long long)n_rows, (long long)n_rows_r0);
    TIP_REQUIRE(h_rows && d_rows_dev && d_theta && d_p && d_stats && d_err && cs != st && (row_flags & ~TIP_ROWS_COMPACT8) == 0,
                "tip_em_step_host_rows: bad arguments (two distinct streams are required)");
    const size_t need = em_tuned_workspace_bytes(P, K, false);
    TIP_REQUIRE(need == 0 || (d_ws != nullptr && ws_bytes >= need),
                "tip_em_step_host_rows: K=%d needs %zu bytes of workspace (got %zu), see tip_em_workspace_bytes", K, need, ws_bytes);
    static cudaEvent_t ev_free = nullptr, ev_filled = nullptr, ev_done = nullptr;
    if (!ev_free) {
        TIP_CHECK_CUDA(cudaEventCreateWithFlags(&ev_free, cudaEventDisableTiming));
        TIP_CHECK_CUDA(cudaEventCreateWithFlags(&ev_filled, cudaEventDisableTiming));
        TIP_CHECK_CUDA(cudaEventCreateWithFlags(&ev_done, cudaEventDisableTiming));
    }
    const bool compact = (row_flags & TIP_ROWS_COMPACT8) != 0;
    const size_t bytes = (size_t)n_rows * (compact ? 8 : 16);
    // the copy stream may not touch d_rows_dev before everything already queued on `stream` (an earlier E-step that
    // reads it) is done; then: sentinel fill, ONE copy of all rows, and the kernel starts as soon as the fill is over
    TIP_CHECK_CUDA(cudaEventRecord(ev_free, st));
    TIP_CHECK_CUDA(cudaStreamWaitEvent(cs, ev_free, 0));
    TIP_CHECK_CUDA(cudaMemsetAsync(d_rows_dev, 0xFF, bytes, cs));
    TIP_CHECK_CUDA(cudaEventRecord(ev_filled, cs));
    TIP_CHECK_CUDA(cudaMemcpyAsync(d_rows_dev, h_rows, bytes, cudaMemcpyHostToDevice, cs));
    TIP_CHECK_CUDA(cudaEventRecord(ev_done, cs));
    TIP_CHECK_CUDA(cudaMemsetAsync(d_stats, 0, sizeof(double) * (size_t)tip_stats_len(P, K), st));
    bool handled = false;
    int rc = launch_em_tuned(P, K, nullptr, 0, 0, d_theta, d_p, d_stats, reinterpret_cast<double *>(d_ws), false, false, false,
                             st, &handled, 1);
    if (rc) return rc;
    TIP_CHECK_CUDA(cudaStreamWaitEvent(st, ev_filled, 0));
    unsigned long long *chk = reinterpret_cast<unsigned long long *>(d_err) + 4;   // bytes 32..63 of the error block
    rc = launch_em_streamed(P, K, d_rows_dev, n_rows, n_rows_r0, d_theta, d_stats, reinterpret_cast<double *>(d_ws), d_err, chk,
                            compact, st);
    if (rc) return rc;
    rc = launch_em_tuned(P, K, nullptr, 0, 0, d_theta, d_p, d_stats, reinterpret_cast<double *>(d_ws), false, false, false, st,
                         &handled, 4);
    if (rc) return rc;
    // the copy is complete: what the kernel consumed must be what landed (d_err[0] = 2 otherwise)
    TIP_CHECK_CUDA(cudaStreamWaitEvent(st, ev_done, 0));
    return launch_stream_verify(d_rows_dev, n_rows, compact, chk, d_err, st);
}

extern "C" int tip_normalise(int P, int K, const double *d_stats, const int32_t *d_deg, double *d_theta, double *d_p,
                             void *stream)
{
    TIP_REQUIRE(P > 0 && valid_K(K) && d_stats && d_deg && d_theta && d_p, "tip_normalise: bad arguments");
    return launch_normalise(P, K, d_stats, d_deg, d_theta, d_p, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" size_t tip_loglik_workspace_bytes(int P, int K) { return loglik_ws_bytes(P, K); }

extern "C" int tip_loglik(int P, int K, const void *d_rows, int64_t n_rows, int64_t n_rows_r0, const double *d_theta,
                          const double *d_p, double *d_out, void *d_ws, unsigned flags, void *stream)
{
    cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
    TIP_REQUIRE(P > 0 && valid_K(K) && d_theta && d_p && d_out && d_ws && n_rows >= 0 && n_rows % 32 == 0 &&
                    n_rows_r0 >= 0 && n_rows_r0 <= n_rows && n_rows_r0 % 32 == 0,
                "tip_loglik: bad arguments");
    if (n_rows == 0) {
        TIP_CHECK_CUDA(cudaMemsetAsync(d_out, 0, sizeof(double), st));
        return 0;
    }
    return launch_loglik(P, K, reinterpret_cast<const int4 *>(d_rows), n_rows, n_rows_r0, d_theta, d_p, d_out, d_ws,
                         (flags & TIP_EM_FORCE_GENERIC) != 0, st);
}

extern "C" int tip_score(int P, int K, const int32_t *d_g1, const int32_t *d_g2, const int32_t *d_g3, int64_t T,
                         const double *d_theta, const double *d_p, double *d_scores, void *stream)
{
    TIP_REQUIRE(P > 0 && valid_K(K) && T >= 0 && d_theta && d_p && (T == 0 || (d_g1 && d_g2 && d_g3 && d_scores)),
                "tip_score: bad arguments");
    return launch_score(K, d_g1, d_g2, d_g3, T, d_theta, d_p, d_scores, reinterpret_cast<cudaStream_t>(stream));
}

// ---------------------------------------------------------------------------------------------
// host-buffer entry (grow-only device scratch, released with the process)
// ---------------------------------------------------------------------------------------------
namespace {
constexpr int kHostChunks = 8;  // row chunks of the first iteration: H2D of chunk i+1 overlaps the E-step of chunk i
struct HostPool {
    void *rows = nullptr, *rows8 = nullptr, *theta = nullptr, *p = nullptr, *stats = nullptr, *deg = nullptr, *ws = nullptr;
    size_t rows_b = 0, rows8_b = 0, theta_b = 0, p_b = 0, stats_b = 0, deg_b = 0, ws_b = 0;
    cudaStream_t st = nullptr, copy = nullptr;
    cudaEvent_t ev[kHostChunks] = {};
    // streamed first iteration: error word on the device and its read-back in pinned host memory
    unsigned *err = nullptr, *h_err = nullptr;
    unsigned long long *chk = nullptr;   // device: checksums of the streamed step and its "do not trust" flag
    void *order_ws = nullptr, *order_ws2 = nullptr;
    size_t order_ws_b = 0, order_ws2_b = 0;
    cudaEvent_t ev_rows = nullptr, ev_ordered = nullptr;
};
HostPool g_pool;

int ensure(void **ptr, size_t *have, size_t need)
{
    if (*have >= need && *ptr) return 0;
    if (*ptr) TIP_CHECK_CUDA(cudaFree(*ptr));
    *ptr = nullptr;
    *have = 0;
    TIP_CHECK_CUDA(cudaMalloc(ptr, need < 256 ? 256 : need));
    *have = need;
    return 0;
}

// 8-byte rows (TIP_ROWS_COMPACT8): c | b << 20 | a << 40 | rating << 60 | count << 61  ->  int4 {a, b, c, count << 1 | rating}
constexpr int kCompactGeneBits = 20;
constexpr int kCompactMaxCount = 7;

__global__ void rows_expand_kernel(const unsigned long long *__restrict__ in, int4 *__restrict__ out, int64_t n)
{
    const unsigned long long mask = (1ull << kCompactGeneBits) - 1;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long v = in[i];
        out[i] = make_int4((int)((v >> (2 * kCompactGeneBits)) & mask), (int)((v >> kCompactGeneBits) & mask), (int)(v & mask),
                           (int)(((v >> 61) << 1) | ((v >> 60) & 1ull)));
    }
}

int launch_rows_expand(const void *in8, void *out16, int64_t n, cudaStream_t st)
{
    if (n <= 0) return 0;
    const int64_t want = (n + 255) / 256;
    const int grid = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
    rows_expand_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const unsigned long long *>(in8), reinterpret_cast<int4 *>(out16), n);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}
}  // namespace

extern "C" int tip_rows_expand(const void *d_rows8, void *d_rows, int64_t n_rows, void *stream)
{
    TIP_REQUIRE(n_rows >= 0 && (n_rows == 0 || (d_rows8 && d_rows)), "tip_rows_expand: bad arguments");
    return launch_rows_expand(d_rows8, d_rows, n_rows, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int tip_rows_compact_host(const void *h_rows, int64_t n_rows, uint64_t *h_rows8)
{
    TIP_REQUIRE(n_rows >= 0 && (n_rows == 0 || (h_rows && h_rows8)), "tip_rows_compact_host: bad arguments");
    const int32_t *r = reinterpret_cast<const int32_t *>(h_rows);
    for (int64_t i = 0; i < n_rows; ++i) {
        const int32_t a = r[4 * i], b = r[4 * i + 1], c = r[4 * i + 2], w = r[4 * i + 3];
        TIP_REQUIRE(a >= 0 && b >= 0 && c >= 0 && ((a | b | c) >> kCompactGeneBits) == 0 && w >= 0 && (w >> 1) <= kCompactMaxCount,
                    "tip_rows_compact_host: row %lld does not fit 8 bytes (gene ids < 2^%d, count <= %d); use the 16-byte rows",
                    (long long)i, kCompactGeneBits, kCompactMaxCount);
        h_rows8[i] = (uint64_t)c | ((uint64_t)b << kCompactGeneBits) | ((uint64_t)a << (2 * kCompactGeneBits)) |
                     ((uint64_t)(w & 1) << 60) | ((uint64_t)(w >> 1) << 61);
        TIP_REQUIRE(h_rows8[i] != ~0ull, "tip_rows_compact_host: row %lld encodes to the arrival sentinel; use the 16-byte rows",
                    (long long)i);
    }
    return 0;
}

extern "C" int tip_em_iterations_host(int P, int K, const void *h_rows, int64_t n_rows, int64_t n_rows_r0,
                                      const int32_t *h_deg, double *h_theta, double *h_p, int n_iter, unsigned flags)
{
    TIP_REQUIRE(P > 0 && valid_K(K) && h_rows && h_deg && h_theta && h_p && n_iter >= 0 && n_rows >= 0,
                "tip_em_iterations_host: bad arguments");
    HostPool &g = g_pool;
    if (!g.st) {
        TIP_CHECK_CUDA(cudaStreamCreateWithFlags(&g.st, cudaStreamNonBlocking));
        TIP_CHECK_CUDA(cudaStreamCreateWithFlags(&g.copy, cudaStreamNonBlocking));
        for (int c = 0; c < kHostChunks; ++c) TIP_CHECK_CUDA(cudaEventCreateWithFlags(&g.ev[c], cudaEventDisableTiming));
        // the error word of the streamed kernel lives in mapped pinned host memory: written (only on a timeout)
        // straight from the kernel, read by the host after the synchronisation - no device-to-host copy per call
        TIP_CHECK_CUDA(cudaHostAlloc(reinterpret_cast<void **>(&g.h_err), 256, cudaHostAllocMapped));
        memset(g.h_err, 0, 256);
        TIP_CHECK_CUDA(cudaHostGetDevicePointer(reinterpret_cast<void **>(&g.err), g.h_err, 0));
        TIP_CHECK_CUDA(cudaEventCreateWithFlags(&g.ev_rows, cudaEventDisableTiming));
        TIP_CHECK_CUDA(cudaEventCreateWithFlags(&g.ev_ordered, cudaEventDisableTiming));
        TIP_CHECK_CUDA(cudaMalloc(reinterpret_cast<void **>(&g.chk), 256));
        TIP_CHECK_CUDA(cudaMemset(g.chk, 0, 256));
    }
    const size_t nth = (size_t)P * K * 8, np = (size_t)2 * K * K * K * 8, nst = (size_t)tip_stats_len(P, K) * 8;
    size_t wsb = 0;
    if (tip_em_workspace_bytes(P, K, n_rows, flags, &wsb) != 0) return -1;
    int rc = 0;
    const bool compact = (flags & TIP_ROWS_COMPACT8) != 0;
    flags &= ~TIP_ROWS_COMPACT8;
    const size_t row_b = compact ? 8 : 16;  // bytes per row in the HOST buffer
    if (compact && (rc = ensure(&g.rows8, &g.rows8_b, (size_t)n_rows * 8))) return rc;
    // slot-segmented iterations need the rows in three orders plus the tile schedules: ordered on the device once the
    // rows have landed (the first, streamed iteration runs the K^3-per-link kernel, which needs order a only)
    const bool seg3 = seg3_flag(flags);
    size_t order_b = 0;
    if (seg3 && tip_order_rows_workspace_bytes(n_rows, &order_b) != 0) return -1;
    if (seg3 && ((rc = ensure(&g.order_ws, &g.order_ws_b, order_b)) || (rc = ensure(&g.order_ws2, &g.order_ws2_b, order_b)))) return rc;
    if ((rc = ensure(&g.rows, &g.rows_b, (size_t)n_rows * 16 + (seg3 ? (size_t)tip_order_rows_out_bytes(n_rows) : 0))) || (rc = ensure(&g.theta, &g.theta_b, nth)) ||
        (rc = ensure(&g.p, &g.p_b, np)) || (rc = ensure(&g.stats, &g.stats_b, nst)) ||
        (rc = ensure(&g.deg, &g.deg_b, (size_t)P * 4)) || (rc = ensure(&g.ws, &g.ws_b, wsb)))
        return rc;
    if (seg3 && n_iter > 0 && n_rows >= 32 && getenv("TIP_HOST_SEG3_AFTER_STREAM") == nullptr) {
        // Slot-segmented kernels for EVERY iteration.  The rows land first (they are needed in three orders, so nothing
        // can follow the DMA front); then pass A of the first iteration runs on the main stream while the copy stream
        // sorts the rows into orders b and c, which only passes B and C need.
        TIP_CHECK_CUDA(cudaMemcpyAsync(g.theta, h_theta, nth, cudaMemcpyHostToDevice, g.st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(g.p, h_p, np, cudaMemcpyHostToDevice, g.st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(compact ? g.rows8 : g.rows, h_rows, (size_t)n_rows * row_b, cudaMemcpyHostToDevice, g.st));
        if (compact && (rc = launch_rows_expand(g.rows8, g.rows, n_rows, g.st))) return rc;
        TIP_CHECK_CUDA(cudaEventRecord(g.ev_rows, g.st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(g.deg, h_deg, (size_t)P * 4, cudaMemcpyHostToDevice, g.st));
        char *rows_bc = (char *)g.rows + (size_t)n_rows * 16;
        TIP_CHECK_CUDA(cudaStreamWaitEvent(g.copy, g.ev_rows, 0));
        if ((rc = order_rows_parts(g.rows, n_rows, n_rows_r0, g.order_ws2, g.order_ws2_b, rows_bc, g.copy, 2, P))) return rc;
        TIP_CHECK_CUDA(cudaEventRecord(g.ev_ordered, g.copy));
        if ((rc = order_rows_parts(g.rows, n_rows, n_rows_r0, g.order_ws, g.order_ws_b, rows_bc, g.st, 1, P))) return rc;
        for (int it = 0; it < n_iter; ++it) {
            if (it == 0) seg3_wait_before_bc(g.ev_ordered);
            rc = tip_em_step(P, K, g.rows, n_rows, n_rows_r0, (const double *)g.theta, (const double *)g.p, (double *)g.stats,
                             g.ws, g.ws_b, flags, g.st);
            if (rc) return rc;
            rc = launch_normalise(P, K, (const double *)g.stats, (const int32_t *)g.deg, (double *)g.theta, (double *)g.p, g.st);
            if (rc) return rc;
        }
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_theta, g.theta, nth, cudaMemcpyDeviceToHost, g.st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_p, g.p, np, cudaMemcpyDeviceToHost, g.st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(g.st));
        return 0;
    }
    const bool tuned = uses_tuned(K, flags & ~(TIP_EM_SLOT_SEGMENTED | TIP_EM_GATHER_L1));
    const bool streamed = tuned && n_iter > 0 && n_rows >= 32 * kHostChunks &&
                          em_streamed_available(K, (flags & TIP_EM_WITH_LOGLIK) != 0, (flags & TIP_EM_FP32_COMPUTE) != 0,
                                                seg_flag(flags)) && getenv("TIP_HOST_NO_STREAM") == nullptr;
    char *s_dst = compact ? (char *)g.rows8 : (char *)g.rows;
    // the small parameter copies are queued FIRST: one host-to-device engine serves every stream in submission order,
    // and behind the rows they would hold the kernel back until the whole transfer is over (measured)
    TIP_CHECK_CUDA(cudaMemcpyAsync(g.theta, h_theta, nth, cudaMemcpyHostToDevice, g.st));
    TIP_CHECK_CUDA(cudaMemcpyAsync(g.p, h_p, np, cudaMemcpyHostToDevice, g.st));
    if (!streamed) TIP_CHECK_CUDA(cudaMemcpyAsync(g.deg, h_deg, (size_t)P * 4, cudaMemcpyHostToDevice, g.st));
    if (streamed) {
        // sentinel fill, then ONE copy of all rows; the kernel (launched below, after the fill) follows the DMA front
        TIP_CHECK_CUDA(cudaMemsetAsync(s_dst, 0xFF, (size_t)n_rows * row_b, g.copy));
        TIP_CHECK_CUDA(cudaEventRecord(g.ev[0], g.copy));
        TIP_CHECK_CUDA(cudaMemcpyAsync(s_dst, h_rows, (size_t)n_rows * row_b, cudaMemcpyHostToDevice, g.copy));
        // only the M-step needs the degrees: their copy goes behind the rows, off the kernel's critical path
        TIP_CHECK_CUDA(cudaMemcpyAsync(g.deg, h_deg, (size_t)P * 4, cudaMemcpyHostToDevice, g.copy));
        TIP_CHECK_CUDA(cudaEventRecord(g.ev[1], g.copy));
    }
    int it0 = 0;
    if (streamed) {
        // first iteration: ONE launch of the fused kernel consumes the rows as they land (StreamArrive in tip_em.cu)
        bool handled = false;
        TIP_CHECK_CUDA(cudaMemsetAsync(g.stats, 0, nst, g.st));
        rc = launch_em_tuned(P, K, nullptr, 0, 0, (const double *)g.theta, (const double *)g.p, (double *)g.stats,
                             (double *)g.ws, false, false, false, g.st, &handled, 1);
        if (rc) return rc;
        TIP_CHECK_CUDA(cudaStreamWaitEvent(g.st, g.ev[0], 0));
        rc = launch_em_streamed(P, K, s_dst, n_rows, n_rows_r0, (const double *)g.theta, (double *)g.stats, (double *)g.ws,
                                g.err, g.chk, compact, g.st);
        if (rc) return rc;
        rc = launch_em_tuned(P, K, nullptr, 0, 0, (const double *)g.theta, (const double *)g.p, (double *)g.stats,
                             (double *)g.ws, false, false, false, g.st, &handled, 4);
        if (rc) return rc;
        TIP_CHECK_CUDA(cudaStreamWaitEvent(g.st, g.ev[1], 0));
        // the copy is complete: check that the kernel consumed exactly what landed; if not, the flag g.chk[3] makes every
        // M-step of this call a no-op (theta / p stay as uploaded) and the iterations are repeated below from resident rows
        rc = launch_stream_verify(s_dst, n_rows, compact, g.chk, g.err, g.st);
        if (rc) return rc;
        rc = launch_normalise(P, K, (const double *)g.stats, (const int32_t *)g.deg, (double *)g.theta, (double *)g.p, g.st,
                              g.chk + 3);
        if (rc) return rc;
        if (compact && n_iter > 1 && (rc = launch_rows_expand(g.rows8, g.rows, n_rows, g.st))) return rc;
        it0 = 1;
    } else
    if (tuned && n_iter > 0 && n_rows >= 32 * kHostChunks) {
        // first iteration: rows arrive in chunks on the copy stream, the fused kernel consumes each chunk as
        // soon as it has landed (statistics accumulate across the chunk launches)
        const int4 *rows = reinterpret_cast<const int4 *>(g.rows);
        const bool ll = (flags & TIP_EM_WITH_LOGLIK) != 0, f32 = (flags & TIP_EM_FP32_COMPUTE) != 0, sg = seg_flag(flags);
        bool handled = false;
        TIP_CHECK_CUDA(cudaMemsetAsync(g.stats, 0, nst, g.st));
        rc = launch_em_tuned(P, K, rows, 0, 0, (const double *)g.theta, (const double *)g.p, (double *)g.stats,
                             (double *)g.ws, ll, f32, sg, g.st, &handled, 1);
        if (rc) return rc;
        const int64_t n_tiles = n_rows / 32, per = (n_tiles + kHostChunks - 1) / kHostChunks;
        for (int c = 0; c < kHostChunks; ++c) {
            const int64_t t0 = per * c, t1 = (t0 + per < n_tiles) ? t0 + per : n_tiles;
            if (t0 >= t1) break;
            char *dst = compact ? (char *)g.rows8 : (char *)g.rows;
            TIP_CHECK_CUDA(cudaMemcpyAsync(dst + t0 * 32 * row_b, (const char *)h_rows + t0 * 32 * row_b,
                                           (size_t)(t1 - t0) * 32 * row_b, cudaMemcpyHostToDevice, g.copy));
            TIP_CHECK_CUDA(cudaEventRecord(g.ev[c], g.copy));
            TIP_CHECK_CUDA(cudaStreamWaitEvent(g.st, g.ev[c], 0));
            if (compact && (rc = launch_rows_expand((char *)g.rows8 + t0 * 256, (char *)g.rows + t0 * 512, (t1 - t0) * 32, g.st)))
                return rc;
            int64_t r0 = n_rows_r0 / 32 - t0;
            r0 = r0 < 0 ? 0 : (r0 > t1 - t0 ? t1 - t0 : r0);
            rc = launch_em_tuned(P, K, rows + t0 * 32, (t1 - t0) * 32, r0 * 32, (const double *)g.theta, (const double *)g.p,
                                 (double *)g.stats, (double *)g.ws, ll, f32, sg, g.st, &handled, 2);
            if (rc) return rc;
        }
        rc = launch_em_tuned(P, K, rows, 0, 0, (const double *)g.theta, (const double *)g.p, (double *)g.stats, (double *)g.ws,
                             ll, f32, sg, g.st, &handled, 4);
        if (rc) return rc;
        rc = tip_normalise(P, K, (const double *)g.stats, (const int32_t *)g.deg, (double *)g.theta, (double *)g.p, g.st);
        if (rc) return rc;
        it0 = 1;
    } else {
        TIP_CHECK_CUDA(cudaMemcpyAsync(compact ? g.rows8 : g.rows, h_rows, (size_t)n_rows * row_b, cudaMemcpyHostToDevice, g.st));
        if (compact && (rc = launch_rows_expand(g.rows8, g.rows, n_rows, g.st))) return rc;
    }
    auto run_resident = [&](int first) -> int {
        if (seg3 && first < n_iter) {
            int rc2 = tip_order_rows_by_gene(g.rows, n_rows, n_rows_r0, P, g.order_ws, g.order_ws_b, (char *)g.rows + (size_t)n_rows * 16, g.st);
            if (rc2) return rc2;
        }
        for (int it = first; it < n_iter; ++it) {
            int rc2 = tip_em_step(P, K, g.rows, n_rows, n_rows_r0, (const double *)g.theta, (const double *)g.p, (double *)g.stats,
                                  g.ws, g.ws_b, flags, g.st);
            if (rc2) return rc2;
            rc2 = launch_normalise(P, K, (const double *)g.stats, (const int32_t *)g.deg, (double *)g.theta, (double *)g.p, g.st,
                                   streamed ? g.chk + 3 : nullptr);
            if (rc2) return rc2;
        }
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_theta, g.theta, nth, cudaMemcpyDeviceToHost, g.st));
        TIP_CHECK_CUDA(cudaMemcpyAsync(h_p, g.p, np, cudaMemcpyDeviceToHost, g.st));
        TIP_CHECK_CUDA(cudaStreamSynchronize(g.st));
        return 0;
    };
    if ((rc = run_resident(it0))) return rc;
    if (streamed && g.h_err[0] == 2u) {
        // the streamed kernel consumed a word that was not what finally landed: nothing was normalised (theta / p on the
        // device are still the uploaded ones) - repeat every iteration from the rows that are now resident
        g.h_err[0] = 0;
        TIP_CHECK_CUDA(cudaMemsetAsync(g.chk, 0, 32, g.st));
        if (compact && n_iter <= 1 && (rc = launch_rows_expand(g.rows8, g.rows, n_rows, g.st))) return rc;
        if ((rc = run_resident(0))) return rc;
    }
    if (streamed && g.h_err[0] != 0) {
        TIP_CHECK_CUDA(cudaStreamSynchronize(g.copy));
        g.h_err[0] = 0;
        set_error("tip_em_iterations_host: the rows did not arrive on the device within 5 s (copy stream stalled)");
        return -3;
    }
    return 0;
}

// ---------------------------------------------------------------------------------------------
// peak probes (roofline denominators are measured, not assumed)
// ---------------------------------------------------------------------------------------------
namespace {

constexpr int kProbeChains = 8;

template <typename T>
__global__ void __launch_bounds__(256) fma_probe_kernel(T *out, int iters, T a, T b)
{
    T acc[kProbeChains];
#pragma unroll
    for (int i = 0; i < kProbeChains; ++i) acc[i] = (T)(threadIdx.x + i);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < kProbeChains; ++i) acc[i] = fma(acc[i], a, b);
    }
    T s = 0;
#pragma unroll
    for (int i = 0; i < kProbeChains; ++i) s += acc[i];
    if (s == (T)123456.789) out[0] = s;
}

__device__ __forceinline__ void dmma_m8n8k4(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// mode 0: DMMA only; mode 1: DMMA + DFMA interleaved (same number of each instruction)
template <int MODE>
__global__ void __launch_bounds__(256) dmma_probe_kernel(double *out, int iters, double a, double b)
{
    double c[8];
    double f[4];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = threadIdx.x + i;
#pragma unroll
    for (int i = 0; i < 4; ++i) f[i] = threadIdx.x - i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            dmma_m8n8k4(c[2 * i], c[2 * i + 1], a, b);
            if (MODE == 1) f[i] = fma(f[i], a, b);
        }
    }
    double s = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) s += f[i];
    if (s == 123456.789) out[0] = s;
}

__global__ void __launch_bounds__(256) red_probe_kernel(double *buf, int64_t n_addr, int mode, int iters)
{
    unsigned long long x = (blockIdx.x * 256ull + threadIdx.x) * 0x9E3779B97F4A7C15ull + 12345;
    const int lane = threadIdx.x & 31;
    for (int it = 0; it < iters; ++it) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        int64_t addr;
        if (mode == 0) {
            addr = (int64_t)(x % (unsigned long long)n_addr);
        } else {
            // groups of 10 lanes share one random row of 10 doubles (lanes 30,31 idle), like theta rows at K=10
            unsigned long long xr = __shfl_sync(0xffffffffu, x, (lane / 10) * 10);
            const int64_t rows = n_addr / 10;
            addr = (int64_t)(xr % (unsigned long long)rows) * 10 + lane % 10;
            if (lane >= 30) continue;
        }
        asm volatile("red.global.add.f64 [%0], %1;" ::"l"(buf + addr), "d"(1.0) : "memory");
    }
}

// random rows of a small (L2-resident) table, `vecs` 16-byte loads each, L2 only (ld.global.cg): the gather pattern of the
// slot-segmented passes (theta rows of 8K bytes on 128-byte lines)
__global__ void __launch_bounds__(256) gather_probe_kernel(const double2 *__restrict__ table, int n_rows_table, int row_vecs,
                                                           int vecs, int iters, double *out)
{
    unsigned long long x = (blockIdx.x * 256ull + threadIdx.x) * 0x9E3779B97F4A7C15ull + 777;
    double acc = 0.0;
    for (int it = 0; it < iters; ++it) {
        x ^= x << 13; x ^= x >> 7; x ^= x << 17;
        const double2 *row = table + (size_t)(x % (unsigned long long)n_rows_table) * row_vecs;
        for (int v = 0; v < vecs; ++v) {
            double2 d;
            asm volatile("ld.global.cg.v2.f64 {%0, %1}, [%2];" : "=d"(d.x), "=d"(d.y) : "l"(row + v));
            acc += d.x + d.y;
        }
    }
    if (acc == 123456.789) out[0] = acc;
}

template <typename F>
int time_kernel(F launch, double *ms_out)
{
    cudaEvent_t e0, e1;
    TIP_CHECK_CUDA(cudaEventCreate(&e0));
    TIP_CHECK_CUDA(cudaEventCreate(&e1));
    launch();  // warm-up
    TIP_CHECK_CUDA(cudaDeviceSynchronize());
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
        TIP_CHECK_CUDA(cudaEventRecord(e0));
        launch();
        TIP_CHECK_CUDA(cudaEventRecord(e1));
        TIP_CHECK_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        TIP_CHECK_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best) best = ms;
    }
    TIP_CHECK_CUDA(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    *ms_out = best;
    return 0;
}

}  // namespace

extern "C" int tip_measure_fma_peak(int kind, double *tflops)
{
    TIP_REQUIRE(tflops != nullptr && kind >= 0 && kind <= 3, "tip_measure_fma_peak: kind must be 0..3");
    double *d_out = nullptr;
    TIP_CHECK_CUDA(cudaMalloc(&d_out, 256));
    const int blocks = sm_count() * 8, threads = 256;
    double ms = 0, flops = 0;
    int rc = 0;
    if (kind == 0) {
        const int iters = 1 << 15;
        rc = time_kernel([&] { fma_probe_kernel<double><<<blocks, threads>>>(d_out, iters, 1.0000001, 1e-9); }, &ms);
        flops = 2.0 * kProbeChains * (double)iters * blocks * threads;
    } else if (kind == 1) {
        const int iters = 1 << 16;
        rc = time_kernel([&] { fma_probe_kernel<float><<<blocks, threads>>>(reinterpret_cast<float *>(d_out), iters, 1.0000001f, 1e-9f); }, &ms);
        flops = 2.0 * kProbeChains * (double)iters * blocks * threads;
    } else if (kind == 2) {
        const int iters = 1 << 13;
        rc = time_kernel([&] { dmma_probe_kernel<0><<<blocks, threads>>>(d_out, iters, 1.0000001, 1e-9); }, &ms);
        flops = 2.0 * 256.0 * 4 * (double)iters * blocks * (threads / 32);  // m8n8k4 = 256 FMA per warp instruction
    } else {
        const int iters = 1 << 13;
        rc = time_kernel([&] { dmma_probe_kernel<1><<<blocks, threads>>>(d_out, iters, 1.0000001, 1e-9); }, &ms);
        flops = (2.0 * 256.0 * 4 * (threads / 32) + 2.0 * 4 * threads) * (double)iters * blocks;
    }
    cudaFree(d_out);
    if (rc) return rc;
    *tflops = flops / (ms * 1e-3) / 1e12;
    return 0;
}

extern "C" int tip_measure_l2_gather(int n_rows_table, int row_bytes, double *gbs)
{
    TIP_REQUIRE(gbs != nullptr && n_rows_table >= 1 && row_bytes >= 16 && row_bytes % 16 == 0 && row_bytes <= 1024,
                "tip_measure_l2_gather: row_bytes must be a multiple of 16 up to 1024");
    const int row_stride = (row_bytes + 127) / 128 * 128;
    double2 *table = nullptr;
    double *d_out = nullptr;
    TIP_CHECK_CUDA(cudaMalloc(&table, (size_t)n_rows_table * row_stride));
    TIP_CHECK_CUDA(cudaMemset(table, 0, (size_t)n_rows_table * row_stride));
    TIP_CHECK_CUDA(cudaMalloc(&d_out, 256));
    const int blocks = sm_count() * 8, threads = 256, iters = 512;
    double ms = 0;
    int rc = time_kernel([&] { gather_probe_kernel<<<blocks, threads>>>(table, n_rows_table, row_stride / 16, row_bytes / 16, iters, d_out); }, &ms);
    cudaFree(table);
    cudaFree(d_out);
    if (rc) return rc;
    // bytes that cross the L2 -> SM crossbar: whole 32-byte sectors of every row
    const double sectors = (row_bytes + 31) / 32;
    *gbs = sectors * 32.0 * (double)blocks * threads * iters / (ms * 1e-3) / 1e9;
    return 0;
}

extern "C" int tip_measure_red_f64(int64_t n_addr, int mode, double *gops)
{
    TIP_REQUIRE(gops != nullptr && n_addr >= 10 && (mode == 0 || mode == 1), "tip_measure_red_f64: bad arguments");
    double *buf = nullptr;
    TIP_CHECK_CUDA(cudaMalloc(&buf, (size_t)n_addr * 8));
    TIP_CHECK_CUDA(cudaMemset(buf, 0, (size_t)n_addr * 8));
    const int blocks = sm_count() * 8, threads = 256, iters = 2048;
    double ms = 0;
    int rc = time_kernel([&] { red_probe_kernel<<<blocks, threads>>>(buf, n_addr, mode, iters); }, &ms);
    cudaFree(buf);
    if (rc) return rc;
    const double lanes = mode == 0 ? 32.0 : 30.0;
    *gops = lanes / 32.0 * (double)blocks * threads * iters / (ms * 1e-3) / 1e9;
    return 0;
}
