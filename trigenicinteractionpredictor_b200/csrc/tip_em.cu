// K-specialised fused E-step for sm_100a (K = 1..16): the hot kernel of Model.make_iteration
// (TIP.py:987-1012).  fp64 CUDA-core FMA bound.
//
// Persistent single-warp CTAs (12 resident per SM): every control decision depends only on
// blockIdx / kernel parameters, which lets ptxas prove warp-uniformity and keep the p operand on the
// uniform datapath.  A warp walks tiles of 32 packed rows (all one rating, see tip.h):
//
//   gather   cp.async the three theta rows of each of the 32 links into a [link][th_a|th_b|th_c]
//            shared-memory stage (16-byte copies, whole rows per request).
//   phase A  lane = link.  th_b, th_c and the accumulators v[K], w[K] live in registers;
//            p[.][.][.][r] comes from the constant bank on the uniform datapath (see c_pem).
//              q[ab]  = sum_c p[abc] th_c[c]              K^3 DFMA
//              w[c]  += th_a[a] th_b[b] p[abc]            K^3 DFMA
//              u[a]  += th_b[b] q[ab],  v[b] += th_a[a] q[ab]
//            d = eps + sum_a th_a[a] u[a];  s = count / d.
//            Slot-b/c contributions s*th_b*v, s*th_c*w go to a [link][3K] shared buffer and from there
//            to the statistics with one bulk add-reduction (TMA unit) per theta row; s*th_c overwrites
//            th_c in the stage.
//   phase B  Rows are sorted by slot-a gene g, so th_a is constant over a run of links and everything
//            that multiplies th_a can be accumulated per gene first (gene-segmented factorisation):
//              M_g[b][c] += th_b[b] * (s th_c[c])         per link   K^2 DFMA (lanes = cells of M)
//            and, once per iteration in em_finalize_kernel,
//              Ntheta[g][a] += th_g[a] * sum_bc p[abc] M_g[b][c]      (the slot-a statistic)
//              S[a][b][c]   += th_g[a] * M_g[b][c]                    (the p statistic, npr = p * S)
//            so the p statistic costs K^2 per link + 2 K^3 per (gene, rating) instead of K^3 per link,
//            and the slot-a scatter disappears.  M_g lives in the workspace (2*P*K^2 doubles).
//   K <= 4   K^3 <= 64: S is thread-private (registers) and updated in phase A; slot-a contributions are
//            pre-reduced over runs of equal gene; no workspace.
#include <stdlib.h>

#include "tip_common.cuh"

namespace tip {

// p in the E-step layout [r][ab][c] (c padded to KP), read through the constant bank: the index is
// warp-uniform, so ptxas keeps p on the uniform datapath (LDCU.64 -> UR operand of DFMA) and the
// 1000 values per link never touch the vector register file or the shared-memory pipe.  Measured on
// B200 (tools/probes/probe_operand_paths.cu): shared-memory broadcast saturates at 75 % of the DFMA
// peak whatever the occupancy; the constant path reaches 84 % at 8 warps/SM and 89 % at 20.
// Capacity: 63 KB of the 64 KB user constant bank.  K <= 10 needs 2*K*K*KP <= 2000 doubles for both ratings and
// rotates over three 2000-double slots (so launches on neighbouring streams do not collide); K = 11..14 fits both
// ratings once; K = 15, 16 fits ONE rating (K*K*KP <= 4096 doubles), so the E-step is launched per rating block.
constexpr int kPSlots = 3;
constexpr int kPSlotDoubles = 2000;
constexpr int kPBankDoubles = 8064;
constexpr int kMaxTunedK = 32;      // K = 17..32: gene-segmented formulation only
__constant__ double c_pem[kPBankDoubles];
__device__ double g_pstage[kPBankDoubles];

template <int K>
struct EmCfg {
    static constexpr int KP = K + (K & 1);                   // sub-row length (even)
    static constexpr int S3 = 3 * KP;
    static constexpr int RS = S3 + ((S3 % 4 == 2) ? 0 : 2);  // row stride == 2 (mod 4): conflict-free 128-bit rows
    static constexpr int K3 = K * K * K;
    static constexpr bool kPrivateS = (K <= 4);              // S thread-private, no gene segmentation
    // phase B lane mapping: lane -> (b = lane % K, c-group = lane / K), a group covers CB values of c
    static constexpr int NG = (32 / K) < K ? (32 / K) : K;
    static constexpr int CB = (K + NG - 1) / NG;
    static constexpr int NGU = (K + CB - 1) / CB;            // groups actually needed
    // contribution buffer row: [ca|cb|cc] for K <= 4, [cb|cc] otherwise (slot a comes from M_g); stride == 2 (mod 4)
    static constexpr int CSLOTS = kPrivateS ? 3 : 2;
    static constexpr int CA = kPrivateS ? KP : 0;            // offset of cb inside a row
    static constexpr int RC = CSLOTS * KP + (((CSLOTS * KP) % 4 == 2) ? 0 : 2);
    // shared memory of one warp-CTA: theta stage + contribution buffer (doubles), then ids (32 int4)
    static constexpr int WARP_DBL = 32 * RS + 32 * RC;
    static constexpr size_t SMEM = (size_t)WARP_DBL * 8 + 32 * 16;
};

// p[abc][r] (reference layout) -> [r][ab][c padded] staging copy (fp64, or fp32 for the fp32-compute mode),
// then memcpy to the constant bank.  Ratings r_lo .. r_lo + n_r - 1 are staged.
template <typename T>
__global__ void stage_p_kernel(int K, int KP, int r_lo, int n_r, const double *__restrict__ p, T *__restrict__ out)
{
    const int n = n_r * K * K * KP;
    for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < n; e += gridDim.x * blockDim.x) {
        const int r = e / (K * K * KP), rem = e - r * (K * K * KP);
        const int pair = rem / KP, c = rem - pair * KP;
        out[e] = (c < K) ? (T)p[((int64_t)pair * K + c) * 2 + r_lo + r] : (T)0;
    }
}

// Row gather: LPI links per warp instruction, each link's three theta rows copied as U units of
// UNIT doubles (16-byte cp.async when K is even).  Which (link-in-group, slot, unit) a lane serves is
// fixed for the whole kernel, so an iteration costs one id load, two address computations and the copy.
template <int K>
struct GatherMap {
    static constexpr int UNIT = (K % 2 == 0) ? 2 : 1;
    static constexpr int U = K / UNIT;
    static constexpr int LPI = (3 * U <= 32) ? 32 / (3 * U) : 1;   // links per warp instruction
    static constexpr int ITERS = (32 + LPI - 1) / LPI;
    static constexpr int UP = (3 * U + 31) / 32;                    // instructions per link when 3U > 32 (odd K >= 11)
};

template <int K, int RS, int KP>
__device__ __forceinline__ void gather_tile(const double *__restrict__ theta, const int4 *ids, double *stage, int lane)
{
    using G = GatherMap<K>;
    if constexpr (3 * G::U > 32) {
        // a link's 3U units do not fit one warp instruction: UP instructions per link
        const int *idw = reinterpret_cast<const int *>(ids);
#pragma unroll 2
        for (int l = 0; l < 32; ++l) {
#pragma unroll
            for (int j = 0; j < G::UP; ++j) {
                const int u = lane + 32 * j;
                if (u < 3 * G::U) {
                    const int slot = u / G::U, k0 = (u - slot * G::U) * G::UNIT;
                    const int g = idw[l * 4 + slot];
                    if (G::UNIT == 2)
                        cp_async_16(stage + l * RS + slot * KP + k0, theta + (int64_t)g * K + k0);
                    else
                        cp_async_8(stage + l * RS + slot * KP + k0, theta + (int64_t)g * K + k0);
                }
            }
        }
        return;
    }
    const int sub = lane / (3 * G::U), rem = lane - sub * (3 * G::U);
    const int slot = rem / G::U, k0 = (rem - slot * G::U) * G::UNIT;
    const bool active = sub < G::LPI;
    const int *idp = reinterpret_cast<const int *>(ids) + sub * 4 + slot;
    double *dst = stage + sub * RS + slot * KP + k0;
    const double *src0 = theta + k0;
#pragma unroll 4
    for (int it = 0; it < G::ITERS; ++it) {
        if (active && (32 % G::LPI == 0 || it * G::LPI + sub < 32)) {
            const int g = *idp;
            if (G::UNIT == 2)
                cp_async_16(dst, src0 + (int64_t)g * K);
            else
                cp_async_8(dst, src0 + (int64_t)g * K);
        }
        idp += G::LPI * 4;
        dst += G::LPI * RS;
    }
}

// fire-and-forget fp64 reduction, skipped when the value is exactly zero (padding rows)
__device__ __forceinline__ void red_add_f64_nz(double *addr, double v)
{
    asm volatile("{ .reg .pred p; setp.neu.f64 p, %1, 0d0000000000000000; @p red.global.add.f64 [%0], %1; }" ::"l"(addr),
                 "d"(v)
                 : "memory");
}

// Bulk asynchronous add-reduction of `bytes` (multiple of 16) contiguous doubles from shared memory into
// global memory (SASS: UBLKRED.G.S.ADD.F64): one request to the TMA unit per theta row instead of K
// per-lane red.global.add.f64 (which cost the LSU ~1.3 cycles per lane).
__device__ __forceinline__ void bulk_red_add_f64(double *gdst, const double *ssrc, int bytes)
{
    const unsigned sa = static_cast<unsigned>(__cvta_generic_to_shared(ssrc));
    asm volatile("cp.reduce.async.bulk.global.shared::cta.bulk_group.add.f64 [%0], [%1], %2;" ::"l"(gdst), "r"(sa),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Scatter of slot-b / slot-c contributions with per-lane reductions (odd K, where a row is not a multiple
// of 16 bytes): the flat index i*32+lane over 32 links x 2K values repeats its (link offset, slot, k)
// pattern every PER warp instructions, so the PER offsets a lane needs are computed once per kernel.
template <int K>
struct ScatterMap {
    static constexpr int gcd(int a, int b) { return b == 0 ? a : gcd(b, a % b); }
    static constexpr int V = 2 * K;     // values per link
    static constexpr int G = gcd(32, V);
    static constexpr int PER = V / G;   // warp instructions per period
    static constexpr int LPP = 32 / G;  // links per period
    static constexpr int NPERIOD = G;   // periods per tile (32 / LPP)
};

// T = double: the fp64 path (1e-9 parity).  T = float: fp32-compute / fp64-accumulate mode (TIP_EM_FP32_COMPUTE):
// only the two K^3 contractions of phase A run in fp32 (FFMA, p as fp32 in the constant bank); the normaliser,
// s, every contribution that leaves the thread, M_g and all statistics stay fp64 (1e-5 parity).
//
// SEG = true (TIP_EM_GENE_SEGMENTED, K >= 5): the gene-segmented factorisation applied to phase A as well.  p is
// contracted with th_a once per (gene, rating) by seg_prep_kernel, Z_g[b][c] = sum_a th_g[a] p[abc], and a link then
// costs 2 K^2 DFMA instead of 2 K^3:   y[b] = sum_c Z_g[b][c] th_c[c],   w[c] = sum_b th_b[b] Z_g[b][c],
// d = eps + sum_b th_b[b] y[b].  Lanes read Z of their own slot-a gene through L1 (one address per run of equal
// gene, so a warp instruction touches one or two lines).  The kernel is then bound by the theta gather and the
// slot-b/c reductions, not by the FMA pipe; bench.py reports it separately from the headline kernel.
//
// STREAM = true (host-buffer entry, tip_em_iterations_host): the rows are still arriving from the host while the
// kernel runs.  The device buffer is filled with a sentinel (all ones, never a valid row) before ONE host-to-device
// copy of all rows is queued on a copy stream; a warp polls the rows of its next tile (ld.cv) until none of them is
// the sentinel.  Rows are written once, so an 8-byte word that is not the sentinel is final: no flags, no chunking,
// one launch and one copy, and the kernel follows the DMA front tile by tile.  sa.compact: the rows are the 8-byte
// host format (tip_rows_compact_host), decoded on load.  A warp that waits longer than sa.timeout_ns sets *sa.err and
// treats every later row as padding (count 0), so a stalled host cannot hang the GPU.
// The CUDA memory model does not promise that a kernel racing a DMA sees whole, final 8-byte words, so the kernel PROVES
// what it consumed: every warp adds the words it accepted into sa.chk[0] (wrapping 64-bit sum), and once the copy is
// complete stream_verify_kernel sums the buffer itself into sa.chk[1]; a difference (a torn or stale word was consumed)
// sets the error word to 2 and a device flag that makes the M-step leave theta / p untouched - the caller then repeats the
// iteration from the resident rows.  Detection and repair instead of trust.
struct StreamArrive {
    unsigned long long *chk;  // device: {consumed sum, buffer sum, blocks done, mismatch flag}
    unsigned *err;
    int compact;
    unsigned long long timeout_ns;
};
constexpr unsigned long long kRowSentinel = ~0ull;

__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// MINB resident warp-CTAs per SM: the register budget is stated with __maxnreg__ (65536 / (32 MINB), multiple of 8)
// because __launch_bounds__(32, MINB) makes ptxas fall back to 128 registers for every MINB above 12.
constexpr int em_max_regs(int minb)
{
    const int r = 65536 / (32 * minb) / 8 * 8;
    return r > 255 ? 255 : r;
}

template <int K, int MINB, bool LL, typename T, bool SEG, bool STREAM = false>
__global__ void __launch_bounds__(32) __maxnreg__(em_max_regs(MINB))
    em_fused_kernel(int P, const int4 *__restrict__ rows, int n_tiles, int n_tiles_r0, const double *__restrict__ theta,
                    int p_off0, int p_off1, double *__restrict__ stats, double *__restrict__ Mg,
                    const double *__restrict__ Zg, StreamArrive sa)
{
    using C = EmCfg<K>;
    constexpr int KP = C::KP, RS = C::RS, K3 = C::K3, CB = C::CB, RC = C::RC, CA = C::CA;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x;
    double *stage = reinterpret_cast<double *>(smem_raw);    // [32][RS]
    double *cbuf = stage + 32 * RS;                          // [32][RC]
    int4 *ids = reinterpret_cast<int4 *>(cbuf + 32 * RC);    // [32]

    // Tile bookkeeping (t, W, the rating of a tile, the p index) must stay on the uniform datapath.
    // ptxas gives every value ONE home: a single per-lane use of %ctaid.x / %nctaid.x (the row pointers
    // below) moves the tile counter - and with it the p index - to the vector register file, and the p
    // loads degrade from LDCU (uniform) to per-lane LDC.64, measured 1.4x slower than even the
    // shared-memory version.  volatile asm, a round trip through shared memory and shuffles do not
    // separate the copies (the store or shuffle is itself a vector use).  What does: the per-lane side
    // reads %clusterid.x / %nclusterid.x, which equal %ctaid.x / %nctaid.x for this non-cluster launch
    // but are different special registers to the compiler.
    const int W = gridDim.x;
    const int w0 = blockIdx.x;
    unsigned bx_v, gx_v;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(bx_v));
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(gx_v));
    const int4 *rp = rows + (int64_t)bx_v * 32 + lane;  // next tile of rows this lane will fetch
    const int64_t rstride = (int64_t)gx_v * 32;
    // (Tried: staggering the start of the co-resident warp-CTAs of an SM by 0.3-5 us each, in case the 12 warps run
    // their phases in lockstep - no effect at 800 k or 10 M links, so the phases already interleave.)
    // STREAM: per-lane tile index of the next fetch
    unsigned tile_v = bx_v;
    bool stream_dead = false;
    unsigned long long consumed = 0;
    auto next_rows = [&]() -> int4 {
        int4 v;
        if constexpr (STREAM) {
            const unsigned long long *src =
                sa.compact ? reinterpret_cast<const unsigned long long *>(rows) + (int64_t)tile_v * 32 + lane
                           : reinterpret_cast<const unsigned long long *>(rp);
            unsigned long long q0 = 0, q1 = 0, t_start = 0;
            unsigned spins = 0;
            for (;;) {
                if (!stream_dead) {
                    q0 = __ldcv(src);
                    q1 = sa.compact ? 0ull : __ldcv(src + 1);
                }
                const bool ok = stream_dead || (q0 != kRowSentinel && q1 != kRowSentinel);
                if (__all_sync(0xffffffffu, ok)) break;
                if (spins == 0) t_start = global_timer_ns();
                __nanosleep(100);
                if (((++spins & 255u) == 0 || sa.timeout_ns == 0) && global_timer_ns() - t_start >= sa.timeout_ns) {
                    stream_dead = true;
                    *sa.err = 1u;
                }
            }
            stream_dead = __any_sync(0xffffffffu, stream_dead);
            if (!stream_dead) consumed += q0 + q1;
            if (stream_dead) {
                v = make_int4(0, 0, 0, 0);
            } else if (sa.compact) {
                const unsigned long long mask = (1ull << 20) - 1;
                v = make_int4((int)((q0 >> 40) & mask), (int)((q0 >> 20) & mask), (int)(q0 & mask),
                              (int)(((q0 >> 61) << 1) | ((q0 >> 60) & 1ull)));
            } else {
                v = make_int4((int)(unsigned)q0, (int)(q0 >> 32), (int)(unsigned)q1, (int)(q1 >> 32));
            }
            tile_v += gx_v;
        } else {
            v = *rp;
        }
        rp += rstride;
        return v;
    };

    // phase B lane mapping
    const int b_lane = lane % K;
    int grp = lane / K;
    const bool b_active = grp < C::NGU;
    if (grp >= C::NGU) grp = 0;
    const int c0 = grp * CB;

    // odd K: scatter pattern of this lane, (value offset in cbuf | id offset << 16 | k << 24) per phase
    unsigned sc_pack[ScatterMap<K>::PER];
#pragma unroll
    for (int ph = 0; ph < ScatterMap<K>::PER; ++ph) {
        const int idx = ph * 32 + lane;
        const int l = idx / (2 * K), rem = idx - l * (2 * K);
        const int slot = 1 + rem / K, kk = rem % K;
        sc_pack[ph] = (unsigned)(l * RC + CA + (slot - 1) * KP + kk) | ((unsigned)(l * 4 + slot) << 16) | ((unsigned)kk << 24);
    }

    // K <= 4 only: thread-private S
    constexpr int NS = C::kPrivateS ? K3 : 1;
    double Sacc[NS];
#pragma unroll
    for (int i = 0; i < NS; ++i) Sacc[i] = 0.0;
    int cur_r = -1;
    double ll = 0.0;
    double *Sg = stats + stats_off_S(P, K);

    auto flush_S = [&](int r) {
        if (r < 0) return;
        double *dst = Sg + r * K3;
#pragma unroll
        for (int i = 0; i < NS; ++i) {
            const double t = warp_sum(Sacc[i]);
            if (lane == 0 && t != 0.0) red_add_f64(dst + i, t);
            Sacc[i] = 0.0;
        }
    };

    // the rows of the next tile are loaded while the current tile is gathered
    int4 ids_next = make_int4(0, 0, 0, 0);
    if (w0 < n_tiles) ids_next = next_rows();

    for (int t = w0; t < n_tiles; t += W) {
        ids[lane] = ids_next;
        __syncwarp();
        gather_tile<K, RS, KP>(theta, ids, stage, lane);
        cp_async_commit();
        if (t + W < n_tiles) ids_next = next_rows();
        cp_async_wait<0>();
        __syncwarp();

        const int4 me = ids[lane];
        // the rating is the same for the whole tile and follows from the tile index alone, which keeps
        // the p index below provably warp-uniform (uniform datapath)
        const int r = t >= n_tiles_r0 ? 1 : 0;
        // per-lane copy of the rating taken from the row data (same value for the whole tile), so that
        // r itself never enters the vector register file
        const int r_v = row_rating(me.w);
        const double cnt = (double)row_count(me.w);
        if constexpr (C::kPrivateS) {
            if (r_v != cur_r) {
                flush_S(cur_r);
                cur_r = r_v;
            }
        }

        // ================= phase A: lane = link =================
        {
            if constexpr (K % 2 == 0) bulk_wait_read();  // the previous tile's bulk reductions have read cbuf
            double *row = stage + lane * RS;
            double *crow = cbuf + lane * RC;
            // p index (units of T) of this tile's rating inside the constant bank
            const int pbase = r ? p_off1 : p_off0;
            const T *cp = reinterpret_cast<const T *>(c_pem);
            // registers: th_b / v only on the K^3 path; the gene-segmented path reads th_b[b] from the stage as
            // it goes and parks the unscaled slot-b contribution in cbuf, so it needs 2K doubles of state (K <= 32)
            T tb[SEG ? 2 : KP], tc[KP], v[SEG ? 1 : K], w[KP];
#pragma unroll
            for (int k = 0; k < KP; k += 2) {
                const double2 c2 = *reinterpret_cast<const double2 *>(row + 2 * KP + k);
                tc[k] = (T)c2.x; tc[k + 1] = (T)c2.y;
                w[k] = (T)0; w[k + 1] = (T)0;
                if constexpr (!SEG) {
                    const double2 b2 = *reinterpret_cast<const double2 *>(row + KP + k);
                    tb[k] = (T)b2.x; tb[k + 1] = (T)b2.y;
                }
            }
            if constexpr (!SEG) {
#pragma unroll
                for (int k = 0; k < K; ++k) v[k] = (T)0;
            }
            T dsum = (T)0;
            if constexpr (SEG) {
                // Z of this link's slot-a gene and rating.  Most tiles lie inside one run of equal slot-a gene (runs are
                // ~4 tiles long at cfg2): then Z_g is staged once, coalesced, into the th_a slots of the stage - which
                // this formulation never reads - as zs[b * RS + c], and every lane takes it from there as a shared-memory
                // broadcast instead of 50 dependent-latency L2 loads per link (long-scoreboard stalls were 41 % of this
                // kernel, profiles/r1_em_fused_k10_gene_segmented_before_zstage_summary.txt).  Mixed tiles read Z through L1 as before.
                const double *Zrow = Zg + ((int64_t)r_v * P + me.x) * (K * K);
                const int g0 = __shfl_sync(0xffffffffu, me.x, 0);
                const bool one_gene = __all_sync(0xffffffffu, me.x == g0 && cnt != 0.0);
                if (one_gene) {
#pragma unroll
                    for (int e = lane; e < K * K; e += 32) {
                        const int zb = e / K, zc = e - zb * K;
                        stage[zb * RS + zc] = __ldg(Zrow + e);
                    }
                    __syncwarp();
                }
                auto seg_phase_a = [&](auto zpair) {
#pragma unroll 2
                    for (int b = 0; b < K; ++b) {
                        const T tbb = (T)row[KP + b];
                        T y0 = (T)0, y1 = (T)0;
#pragma unroll
                        for (int c = 0; c < K; c += 2) {
                            const double2 z = zpair(b, c);   // z.y is not used for the last column of an odd K
                            y0 = fma((T)z.x, tc[c], y0);
                            w[c] = fma(tbb, (T)z.x, w[c]);
                            if (c + 1 < K) {
                                y1 = fma((T)z.y, tc[c + 1], y1);
                                w[c + 1] = fma(tbb, (T)z.y, w[c + 1]);
                            }
                        }
                        const T tby = tbb * (y0 + y1);
                        dsum += tby;
                        crow[CA + b] = (double)tby;  // unscaled slot-b contribution, multiplied by s below
                    }
                };
                if (one_gene) {
                    seg_phase_a([&](int b, int c) {
                        if constexpr (K % 2 == 0) {
                            return *reinterpret_cast<const double2 *>(stage + b * RS + c);
                        } else {
                            return make_double2(stage[b * RS + c], (c + 1 < K) ? stage[b * RS + c + 1] : 0.0);
                        }
                    });
                } else {
                    seg_phase_a([&](int b, int c) {
                        if constexpr (K % 2 == 0) {
                            return __ldg(reinterpret_cast<const double2 *>(Zrow + b * K + c));
                        } else {
                            return make_double2(__ldg(Zrow + b * K + c), (c + 1 < K) ? __ldg(Zrow + b * K + c + 1) : 0.0);
                        }
                    });
                }
            }
            const double *ta_p = row;  // walked separately so that `a` only ever indexes the constant bank
            double *tt_p = crow;
            // (A per-lane ld.const prefetch of the next a-slice was tried against the 88 % constant-cache hit rate
            // ncu reports: the divergent constant access serialises and costs 35 % - not kept.  88 % is exactly one
            // miss per 64-byte line of 8 doubles: the 8 KB table of a rating is streamed once per tile and nothing
            // survives until the next walk.  What those misses cost was measured by aliasing every a-slab onto the
            // first one (wrong results, timing only): 0.254 -> 0.230 ms at 800 k links, 2.45 -> 2.15 ms at 10 M,
            // i.e. 10-12 %.  A uniform prefetch needs uniform registers, which are what limits the load lookahead
            // already; unrolling the a-loop by 2 changed nothing.)
            if constexpr (!SEG)
#pragma unroll 1
            for (int a = 0; a < K; ++a) {
                const T ta = (T)(*ta_p++);
                const int pa = pbase + a * (K * KP);
                T u = (T)0;
#pragma unroll
                for (int b = 0; b < K; ++b) {
                    const T ab = ta * tb[b];
                    T q0 = (T)0, q1 = (T)0;
#pragma unroll
                    for (int c = 0; c < K; c += 2) {
                        // (pa + b*KP + c) is even: one uniform load feeds four FMA
                        const T p0 = cp[pa + b * KP + c];
                        q0 = fma(p0, tc[c], q0);
                        w[c] = fma(ab, p0, w[c]);
                        if (c + 1 < K) {
                            const T p1 = cp[pa + b * KP + c + 1];
                            q1 = fma(p1, tc[c + 1], q1);
                            w[c + 1] = fma(ab, p1, w[c + 1]);
                        }
                    }
                    const T q = q0 + q1;
                    u = fma(tb[b], q, u);
                    v[b] = fma(ta, q, v[b]);
                }
                const T tt = ta * u;
                dsum += tt;
                if constexpr (C::kPrivateS) *tt_p++ = (double)tt;  // slot-a contribution (K >= 5: from M_g in em_finalize_kernel)
            }
            (void)ta_p; (void)tt_p; (void)cp; (void)pbase;
            const double d = TIP_EPS + (double)dsum;
            // s = cnt / d.  d lies in [1e-10, ~1]: an fp32 reciprocal seed and two Newton steps give 1/d to the
            // last ulp or two (far inside the 1e-9 budget) in ~8 instructions instead of the ~30 of an IEEE divide
            double rd = (double)__frcp_rn((float)d);
            rd = rd * fma(-d, rd, 2.0);
            rd = rd * fma(-d, rd, 2.0);
            const double s = cnt * rd;
            if constexpr (LL) ll += cnt * log(d);  // by-product, only on request (TIP_EM_WITH_LOGLIK)
            // contributions of slot b and slot c; s*th_c into the stage for phase B
#pragma unroll
            for (int k = 0; k < KP; k += 2) {
                if constexpr (C::kPrivateS) {
                    double2 ca = *reinterpret_cast<double2 *>(crow + k);
                    ca.x *= s; ca.y *= s;
                    *reinterpret_cast<double2 *>(crow + k) = ca;
                }
                // theta values re-read in fp64 from the stage (T = float only rounded them for the contractions)
                const double2 c2 = *reinterpret_cast<const double2 *>(row + 2 * KP + k);
                if constexpr (SEG) {
                    double2 cb2 = *reinterpret_cast<double2 *>(crow + CA + k);
                    cb2.x *= s;
                    cb2.y = (k + 1 < K) ? cb2.y * s : 0.0;
                    *reinterpret_cast<double2 *>(crow + CA + k) = cb2;
                } else {
                    const double2 b2 = *reinterpret_cast<const double2 *>(row + KP + k);
                    const double vb1 = (k + 1 < K) ? (double)v[k + 1] : 0.0;
                    *reinterpret_cast<double2 *>(crow + CA + k) = make_double2(s * b2.x * (double)v[k], s * b2.y * vb1);
                }
                const double sc0 = s * c2.x, sc1 = s * c2.y;
                *reinterpret_cast<double2 *>(crow + CA + KP + k) = make_double2(sc0 * (double)w[k], sc1 * (double)w[k + 1]);
                *reinterpret_cast<double2 *>(row + 2 * KP + k) = make_double2(sc0, sc1);
            }
            if constexpr (C::kPrivateS) {
                // thread-private S += th_a th_b (s th_c)
#pragma unroll
                for (int a = 0; a < K; ++a) {
                    const double ta = row[a];
#pragma unroll
                    for (int b = 0; b < K; ++b) {
                        const double sab = s * ta * (double)tb[b];
#pragma unroll
                        for (int c = 0; c < K; ++c)
                            Sacc[(a * K + b) * K + c] = fma(sab, (double)tc[c], Sacc[(a * K + b) * K + c]);
                    }
                }
            }
        }
        __syncwarp();

        // ================= scatter theta statistics =================
        {
            const int *idw = reinterpret_cast<const int *>(ids);
            if constexpr (C::kPrivateS) {
                // slot a: run-length pre-reduction.  lane -> (k = lane % K, part = lane / K); each part
                // walks a contiguous range of the 32 links and emits one reduction per run of equal gene.
                constexpr int NPART = 32 / K > 4 ? 4 : (32 / K);
                constexpr int LPP = (32 + NPART - 1) / NPART;
                const int k = lane % K, part = lane / K;
                if (part < NPART) {
                    const int l0 = part * LPP;
                    const int l1 = (l0 + LPP < 32) ? l0 + LPP : 32;
                    double acc = 0.0;
                    int g = idw[l0 * 4];
                    for (int l = l0; l < l1; ++l) {
                        const int gl = idw[l * 4];
                        if (gl != g) {
                            red_add_f64_nz(stats + (int64_t)g * K + k, acc);
                            acc = 0.0;
                            g = gl;
                        }
                        acc += cbuf[l * RC + k];
                    }
                    red_add_f64_nz(stats + (int64_t)g * K + k, acc);
                }
            }
            // slots b, c
            // (Tried: all 64 bulk reductions of a tile issued by lane 0 in an unrolled loop over the links, instead of
            // two per lane - ptxas wraps the uniform-datapath UBLKRED of each lane in an elect-one-lane loop, 16 % of
            // the kernel in the round-1 capture.  The single-lane loop still gets a one-trip elect loop per
            // instruction and serialises the address set-up: 0.274 vs 0.258 ms at 800 k links - not kept.
            // Per-lane REDs for even K as well measured equal to the bulk path within noise at K = 10.)
            if constexpr (K % 2 == 0) {
                // one bulk add-reduction per (link, slot): the 8K-byte row goes to the TMA unit
                fence_async_smem();
                if (cnt != 0.0) {
                    const double *crow = cbuf + lane * RC + CA;
                    bulk_red_add_f64(stats + (int64_t)me.y * K, crow, K * 8);
                    bulk_red_add_f64(stats + (int64_t)me.z * K, crow + KP, K * 8);
                }
                bulk_commit();
            } else {
                using SM = ScatterMap<K>;
                const double *cb = cbuf;
                const int *ib = idw;
#pragma unroll 1
                for (int per = 0; per < SM::NPERIOD; ++per) {
#pragma unroll
                    for (int ph = 0; ph < SM::PER; ++ph) {
                        const unsigned pk = sc_pack[ph];
                        const double val = cb[pk & 0xffffu];
                        const int g = ib[(pk >> 16) & 0xffu];
                        red_add_f64_nz(stats + (int64_t)g * K + (pk >> 24), val);
                    }
                    cb += SM::LPP * RC;
                    ib += SM::LPP * 4;
                }
            }
        }

        // ====== phase B: M_g[b][c] += th_b[b] * (s th_c[c]), flushed per run of equal slot-a gene ======
        if constexpr (!C::kPrivateS) {
            const int *idw = reinterpret_cast<const int *>(ids);
            double M[CB];
#pragma unroll
            for (int j = 0; j < CB; ++j) M[j] = 0.0;
            double *Mr = Mg + (int64_t)r_v * P * (K * K) + b_lane * K + c0;  // this lane's cells of M_g, gene 0
            auto flush_M = [&](int g) {
                double *dst = Mr + (int64_t)g * (K * K);
#pragma unroll
                for (int j = 0; j < CB; ++j) {
                    if (b_active && c0 + j < K) red_add_f64_nz(dst + j, M[j]);
                    M[j] = 0.0;
                }
            };
            int a_prev = idw[0];
#pragma unroll 4
            for (int l = 0; l < 32; ++l) {
                const double *rw = stage + l * RS;
                const int a_l = idw[l * 4];  // same address for every lane: the branch is warp-uniform
                if (a_l != a_prev) {
                    flush_M(a_prev);
                    a_prev = a_l;
                }
                const double tb = rw[KP + b_lane];
                double sc[CB];
                if constexpr (CB % 2 == 0) {
#pragma unroll
                    for (int j = 0; j < CB; j += 2) {
                        const double2 t2 = *reinterpret_cast<const double2 *>(rw + 2 * KP + c0 + j);
                        sc[j] = t2.x; sc[j + 1] = t2.y;
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < CB; ++j) sc[j] = rw[2 * KP + c0 + j];
                }
#pragma unroll
                for (int j = 0; j < CB; ++j) M[j] = fma(tb, sc[j], M[j]);
            }
            flush_M(a_prev);
        }
        __syncwarp();
    }
    if constexpr (C::kPrivateS) flush_S(cur_r);
    if constexpr (LL) {
        ll = warp_sum(ll);
        if (lane == 0 && ll != 0.0) red_add_f64(stats + stats_off_ll(P, K), ll);
    }
    if constexpr (STREAM) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) consumed += __shfl_xor_sync(0xffffffffu, consumed, o);
        if (lane == 0) atomicAdd(sa.chk, consumed);
    }
}

// sum of the 8-byte words of the landed buffer against what the streamed kernel consumed (see StreamArrive)
__global__ void __launch_bounds__(256) stream_verify_kernel(const unsigned long long *__restrict__ words, int64_t n_words,
                                                            unsigned long long *chk, unsigned *err)
{
    unsigned long long s = 0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (int64_t)gridDim.x * blockDim.x) s += words[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(chk + 1, s);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned long long done = atomicAdd(chk + 2, 1ull) + 1;
        if (done == gridDim.x) {
            __threadfence();
            const unsigned long long a = atomicAdd(chk, 0ull), b = atomicAdd(chk + 1, 0ull);
            if (a != b && *err == 0u) {       // (a timed-out step, err == 1, consumed less by construction)
                chk[3] = 1ull;
                *err = 2u;
            }
        }
    }
}

int launch_stream_verify(const void *rows, int64_t n_rows, bool compact, unsigned long long *chk, unsigned *err, cudaStream_t st)
{
    const int64_t n_words = n_rows * (compact ? 1 : 2);
    // TIP_STREAM_INJECT_FAULT (tests): pretend the kernel consumed something else, to exercise detection and repair
    if (getenv("TIP_STREAM_INJECT_FAULT")) TIP_CHECK_CUDA(cudaMemsetAsync(chk, 0x5A, sizeof(unsigned long long), st));
    int64_t want = (n_words + 256 * 8 - 1) / (256 * 8);
    const int grid = (int)(want < 1 ? 1 : (want > (int64_t)sm_count() * 4 ? (int64_t)sm_count() * 4 : want));
    stream_verify_kernel<<<grid, 256, 0, st>>>(reinterpret_cast<const unsigned long long *>(rows), n_words, chk, err);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// Z[r][g][bc] = sum_a theta[g][a] * p[a][bc][r]   (TIP_EM_GENE_SEGMENTED; 2*P*K^3 FMA per iteration in total)
__global__ void seg_prep_kernel(int P, int K, const double *__restrict__ theta, const double *__restrict__ p,
                                double *__restrict__ Zg)
{
    const int KK = K * K;
    const int64_t n = 2ll * P * KK;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        const int r = (int)(e / ((int64_t)P * KK));
        const int64_t rem = e - (int64_t)r * P * KK;
        const int g = (int)(rem / KK), bc = (int)(rem - (int64_t)g * KK);
        double z = 0.0;
        for (int a = 0; a < K; ++a) z = fma(__ldg(theta + (int64_t)g * K + a), __ldg(p + ((int64_t)a * KK + bc) * 2 + r), z);
        Zg[e] = z;
    }
}

// ---------------------------------------------------------------------------------------------
// Per-gene finish of the gene-segmented factorisation (K >= 5), once per iteration:
//   Ntheta[g][a] += th_g[a] * sum_r sum_bc p[a][b][c][r] M_{r,g}[b][c]
//   S[r][a][b][c] += sum_g th_g[a] * M_{r,g}[b][c]
// One CTA per chunk of genes; thread = cell (a, b, c) for S, thread = (gene, a) for Ntheta.
// ---------------------------------------------------------------------------------------------
constexpr int kFinThreads = 512;   // 16 warps; two CTAs per SM (grid = 2 x SMs): the kernel is latency-bound, see DESIGN 4.2
constexpr int kFinWarps = kFinThreads / 32;
// genes staged in shared memory per pass (both ratings): as many as fit beside p in ~200 KB, at most 48
template <int K>
constexpr int fin_chunk()
{
    const long avail = 100 * 1024 - 16L * K * K * K;  // two CTAs per SM
    const long per_gene = 16L * K * K + 8L * K;
    const long n = avail / per_gene;
    return n > 48 ? 48 : (n < 1 ? 1 : (int)n);
}

template <int K>
__global__ void __launch_bounds__(kFinThreads, 2)
    em_finalize_kernel(int P, const double *__restrict__ theta, const double *__restrict__ p,
                       const double *__restrict__ Mg, double *__restrict__ stats)
{
    constexpr int KK = K * K, K3 = K * K * K;
    constexpr int CPT = (K3 + kFinThreads - 1) / kFinThreads;  // S cells per thread
    constexpr int BPL = (KK + 31) / 32;                        // (b,c) pairs per lane
    constexpr int kFinChunk = fin_chunk<K>();
    extern __shared__ __align__(16) double fsm[];
    double *sP = fsm;                         // [2][K3]   p[r][a][bc]
    double *sT = sP + 2 * K3;                 // [kFinChunk][K]
    double *sM = sT + kFinChunk * K;          // [2][kFinChunk][KK]
    const int tid = threadIdx.x, warp = tid / 32, lane = tid % 32;
    const int per = (P + gridDim.x - 1) / gridDim.x;
    const int g_lo = blockIdx.x * per, g_hi = (g_lo + per < P) ? g_lo + per : P;
    for (int e = tid; e < 2 * K3; e += kFinThreads) sP[(e & 1) * K3 + (e >> 1)] = p[e];
    int ca[CPT], cbc[CPT];
    double acc0[CPT], acc1[CPT];
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
        int cell = tid + i * kFinThreads;
        if (cell >= K3) cell = K3 - 1;
        ca[i] = cell / KK;
        cbc[i] = cell - ca[i] * KK;
        acc0[i] = acc1[i] = 0.0;
    }
    for (int g0 = g_lo; g0 < g_hi; g0 += kFinChunk) {
        const int ng = (g_hi - g0 < kFinChunk) ? g_hi - g0 : kFinChunk;
        __syncthreads();
        // stage this chunk: all loads independent, so one memory round trip covers the lot
        const int nM = ng * KK;
#pragma unroll 8
        for (int e = tid; e < nM; e += kFinThreads) {
            sM[e] = __ldg(Mg + (int64_t)g0 * KK + e);
            sM[kFinChunk * KK + e] = __ldg(Mg + ((int64_t)P + g0) * KK + e);
        }
        for (int e = tid; e < ng * K; e += kFinThreads) sT[e] = __ldg(theta + (int64_t)g0 * K + e);
        __syncthreads();
        // p statistic: thread = cells of S
        for (int gi = 0; gi < ng; ++gi) {
#pragma unroll
            for (int i = 0; i < CPT; ++i) {
                const double th = sT[gi * K + ca[i]];
                acc0[i] = fma(th, sM[gi * KK + cbc[i]], acc0[i]);
                acc1[i] = fma(th, sM[(kFinChunk + gi) * KK + cbc[i]], acc1[i]);
            }
        }
        // slot-a statistic: warp = gene, lanes split the (b,c) pairs, K interleaved butterfly reductions
        for (int gi = warp; gi < ng; gi += kFinWarps) {
            double t[K];
#pragma unroll
            for (int a = 0; a < K; ++a) t[a] = 0.0;
#pragma unroll
            for (int i = 0; i < BPL; ++i) {
                const int bc = lane + 32 * i;
                if (bc < KK) {
                    const double m0 = sM[gi * KK + bc], m1 = sM[(kFinChunk + gi) * KK + bc];
#pragma unroll
                    for (int a = 0; a < K; ++a) t[a] = fma(sP[K3 + a * KK + bc], m1, fma(sP[a * KK + bc], m0, t[a]));
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1)
#pragma unroll
                for (int a = 0; a < K; ++a) t[a] += __shfl_xor_sync(0xffffffffu, t[a], o);
#pragma unroll
            for (int a = 0; a < K; ++a)
                if (lane == a) red_add_f64_nz(stats + (int64_t)(g0 + gi) * K + a, sT[gi * K + a] * t[a]);
        }
    }
    double *S = stats + stats_off_S(P, K);
#pragma unroll
    for (int i = 0; i < CPT; ++i) {
        const int cell = tid + i * kFinThreads;
        if (cell < K3) {
            red_add_f64_nz(S + cell, acc0[i]);
            red_add_f64_nz(S + K3 + cell, acc1[i]);
        }
    }
}

template <int K>
constexpr size_t fin_smem_bytes()
{
    return sizeof(double) * (2 * K * K * K + fin_chunk<K>() * K + 2 * fin_chunk<K>() * K * K);
}

// ---------------------------------------------------------------------------------------------
// Per-gene finish for K > 16 (run-time K, gene-segmented mode only): the same two contractions as
// em_finalize_kernel, shaped as small tiled GEMMs because p (2*K^3 doubles) no longer fits shared memory.
//   fin_S_generic_kernel   S[r][a][bc]  += sum_g theta[g][a] * M_r[g][bc]          thread = bc, K accumulators
//   fin_A_generic_kernel   Ntheta[g][a] += theta[g][a] * sum_r sum_bc p[a][bc][r] * M_r[g][bc]   thread = (gene, a)
// ---------------------------------------------------------------------------------------------
constexpr int kFinGChunkGenes = 32;

__global__ void __launch_bounds__(128)
    fin_S_generic_kernel(int P, int K, int genes_per_cta, const double *__restrict__ theta, const double *__restrict__ Mg,
                         double *__restrict__ stats)
{
    __shared__ double sT[kFinGChunkGenes][TIP_MAX_K];
    const int KK = K * K, K3 = KK * K;
    const int r = blockIdx.z;
    const int bc = blockIdx.x * 128 + threadIdx.x;
    const int g_lo = blockIdx.y * genes_per_cta, g_hi = (g_lo + genes_per_cta < P) ? g_lo + genes_per_cta : P;
    double acc[TIP_MAX_K];
#pragma unroll
    for (int a = 0; a < TIP_MAX_K; ++a) acc[a] = 0.0;
    const double *Mr = Mg + (int64_t)r * P * KK;
    for (int g0 = g_lo; g0 < g_hi; g0 += kFinGChunkGenes) {
        const int ng = (g_hi - g0 < kFinGChunkGenes) ? g_hi - g0 : kFinGChunkGenes;
        __syncthreads();
        for (int e = threadIdx.x; e < ng * K; e += 128) sT[e / K][e % K] = __ldg(theta + (int64_t)g0 * K + e);
        __syncthreads();
        if (bc < KK) {
#pragma unroll 4
            for (int gi = 0; gi < ng; ++gi) {
                const double m = __ldg(Mr + (int64_t)(g0 + gi) * KK + bc);
#pragma unroll
                for (int a = 0; a < TIP_MAX_K; ++a)
                    if (a < K) acc[a] = fma(sT[gi][a], m, acc[a]);
            }
        }
    }
    if (bc < KK) {
        double *S = stats + stats_off_S(P, K) + (int64_t)r * K3;
#pragma unroll
        for (int a = 0; a < TIP_MAX_K; ++a)
            if (a < K) red_add_f64_nz(S + (int64_t)a * KK + bc, acc[a]);
    }
}

constexpr int kFinAGenes = 8, kFinATile = 64;

__global__ void __launch_bounds__(kFinAGenes *TIP_MAX_K)
    fin_A_generic_kernel(int P, int K, const double *__restrict__ theta, const double *__restrict__ p,
                         const double *__restrict__ Mg, double *__restrict__ stats)
{
    __shared__ double sP[kFinATile][2][TIP_MAX_K];      // p[a][bc][r] tile, a contiguous
    __shared__ double sM[kFinAGenes][kFinATile][2];     // M_r[g][bc] tile
    const int KK = K * K;
    const int a = threadIdx.x % TIP_MAX_K, gi = threadIdx.x / TIP_MAX_K;
    const int g = blockIdx.x * kFinAGenes + gi;
    const int nthreads = kFinAGenes * TIP_MAX_K;
    double t = 0.0;
    for (int bc0 = 0; bc0 < KK; bc0 += kFinATile) {
        const int nb = (KK - bc0 < kFinATile) ? KK - bc0 : kFinATile;
        __syncthreads();
        for (int e = threadIdx.x; e < nb * 2 * K; e += nthreads) {
            const int aa = e / (nb * 2), rem = e - aa * (nb * 2), j = rem >> 1, rr = rem & 1;   // p[aa][bc0+j][rr] contiguous in (j, rr)
            sP[j][rr][aa] = __ldg(p + ((int64_t)aa * KK + bc0 + j) * 2 + rr);
        }
        for (int e = threadIdx.x; e < kFinAGenes * nb * 2; e += nthreads) {
            const int gg = e / (nb * 2), rem = e - gg * (nb * 2), rr = rem / nb, j = rem - rr * nb;
            const int gene = blockIdx.x * kFinAGenes + gg;
            sM[gg][j][rr] = gene < P ? __ldg(Mg + ((int64_t)rr * P + gene) * KK + bc0 + j) : 0.0;
        }
        __syncthreads();
        if (a < K) {
#pragma unroll 8
            for (int j = 0; j < nb; ++j) t = fma(sP[j][1][a], sM[gi][j][1], fma(sP[j][0][a], sM[gi][j][0], t));
        }
    }
    if (a < K && g < P) red_add_f64_nz(stats + (int64_t)g * K + a, __ldg(theta + (int64_t)g * K + a) * t);
}

static int launch_finalize_generic(int P, int K, const double *theta, const double *p, const double *Mg, double *stats,
                                   cudaStream_t st)
{
    const int KK = K * K;
    const int chunks = 24;
    const int genes_per_cta = (P + chunks - 1) / chunks;
    fin_S_generic_kernel<<<dim3((KK + 127) / 128, (P + genes_per_cta - 1) / genes_per_cta, 2), 128, 0, st>>>(
        P, K, genes_per_cta, theta, Mg, stats);
    TIP_CHECK_CUDA(cudaGetLastError());
    fin_A_generic_kernel<<<(P + kFinAGenes - 1) / kFinAGenes, kFinAGenes * TIP_MAX_K, 0, st>>>(P, K, theta, p, Mg, stats);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

static int g_slot_counter = 0;

template <int K, int MINB, bool LL, typename T = double, bool SEG = false, bool STREAM = false>
static int launch_variant(int P, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, int p_off0,
                          int p_off1, double *stats, double *Mg, cudaStream_t st, StreamArrive sa = StreamArrive{})
{
    using C = EmCfg<K>;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(em_fused_kernel<K, MINB, LL, T, SEG, STREAM>,
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
        TIP_CHECK_CUDA(cudaFuncSetAttribute(em_fused_kernel<K, MINB, LL, T, SEG, STREAM>,
                                            cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int nb = 0;
        TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, em_fused_kernel<K, MINB, LL, T, SEG, STREAM>, 32,
                                                                     C::SMEM));
        TIP_REQUIRE(nb >= 1, "em_fused_kernel<%d> does not fit on an SM (smem %zu)", K, C::SMEM);
        blocks_per_sm = nb;
    }
    const int64_t n_tiles = n_rows / 32;
    TIP_REQUIRE(n_tiles < (1ll << 31), "tip_em_step: more than 2^31 tiles in one shard");
    int64_t cap = (int64_t)sm_count() * blocks_per_sm;
    int grid = (int)(n_tiles < cap ? n_tiles : cap);
    if (grid < 1) grid = 1;
    em_fused_kernel<K, MINB, LL, T, SEG, STREAM><<<grid, 32, C::SMEM, st>>>(
        P, rows, (int)n_tiles, (int)(n_rows_r0 / 32), theta, p_off0, p_off1, stats, Mg,
        SEG ? Mg + 2 * (size_t)P * K * K : nullptr, sa);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

size_t em_tuned_workspace_bytes(int P, int K, bool seg)
{
    if (K <= 4 || K > kMaxTunedK) return 0;
    // M_g[r][gene][b][c], followed by Z_g[r][gene][b][c] in the gene-segmented mode (always for K > 16)
    return sizeof(double) * 2 * (size_t)P * K * K * ((seg || K > 16) ? 2 : 1);
}

// ratings [r_lo, r_lo + n_r) of p -> E-step layout -> constant bank at double-offset base_d (stream-ordered)
static int upload_p_const(int K, const double *p, int r_lo, int n_r, int base_d, bool f32, cudaStream_t st)
{
    const int KP = K + (K & 1);
    static double *stage_ptr = nullptr;
    if (!stage_ptr) TIP_CHECK_CUDA(cudaGetSymbolAddress(reinterpret_cast<void **>(&stage_ptr), g_pstage));
    const int n = n_r * K * K * KP;
    double *dst = stage_ptr + base_d;
    if (f32)
        stage_p_kernel<float><<<(n + 255) / 256, 256, 0, st>>>(K, KP, r_lo, n_r, p, reinterpret_cast<float *>(dst));
    else
        stage_p_kernel<double><<<(n + 255) / 256, 256, 0, st>>>(K, KP, r_lo, n_r, p, dst);
    TIP_CHECK_CUDA(cudaGetLastError());
    TIP_CHECK_CUDA(cudaMemcpyToSymbolAsync(c_pem, dst, (f32 ? sizeof(float) : sizeof(double)) * n, sizeof(double) * base_d,
                                           cudaMemcpyDeviceToDevice, st));
    return 0;
}

// both ratings of a K <= 10 table into the next rotating slot; returns the slot's double-offset
static int upload_p_slot(int K, const double *p, bool f32, cudaStream_t st, int *base_d)
{
    *base_d = ((g_slot_counter++) % kPSlots) * kPSlotDoubles;
    return upload_p_const(K, p, 0, 2, *base_d, f32, st);
}

// phases: 1 = begin (p -> constant bank, clear M_g), 2 = run the fused kernel over `rows`, 4 = end (per-gene
// finish).  tip_em_step runs all three; the host-buffer entry runs "2" once per row chunk as the chunks arrive.
constexpr int kPhaseBegin = 1, kPhaseRun = 2, kPhaseEnd = 4;
static int g_phase_off0 = 0, g_phase_off1 = 0;

template <int K, int MINB, bool LL, typename T>
static int run_rows(int P, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, const double *p,
                    double *stats, double *ws, cudaStream_t st)
{
    constexpr int KP = K + (K & 1), TBL = K * K * KP;
    if constexpr (2 * TBL <= kPBankDoubles) {
        return launch_variant<K, MINB, LL, T>(P, rows, n_rows, n_rows_r0, theta, g_phase_off0, g_phase_off1, stats, ws,
                                              st);
    } else {
        // one rating fits the bank at a time: upload p_r, run that rating block, in stream order
        for (int r = 0; r < 2; ++r) {
            const int64_t lo = r == 0 ? 0 : n_rows_r0, hi = r == 0 ? n_rows_r0 : n_rows;
            if (hi <= lo) continue;
            int rc = upload_p_const(K, p, r, 1, 0, sizeof(T) == 4, st);
            if (rc != 0) return rc;
            rc = launch_variant<K, MINB, LL, T>(P, rows + lo, hi - lo, r == 0 ? hi - lo : 0, theta, 0, 0, stats, ws, st);
            if (rc != 0) return rc;
        }
        return 0;
    }
}

template <int K>
static int launch_em_fused(int P, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta,
                           const double *p, double *stats, double *ws, bool with_ll, bool f32, bool seg, int phases,
                           cudaStream_t st)
{
    constexpr int KP = K + (K & 1), TBL = K * K * KP;
    const int tscale = f32 ? 2 : 1;  // offsets are in units of T
    if (K <= 4) seg = false;         // thread-private S path: nothing to segment
    if (phases & kPhaseBegin) {
        if (seg) {
            // Z_g = theta_g . p  for every (gene, rating), into the second half of the workspace
            const int64_t n = 2ll * P * K * K;
            const int threads = 256;
            int64_t want = (n + threads - 1) / threads;
            const int grid = (int)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
            seg_prep_kernel<<<grid, threads, 0, st>>>(P, K, theta, p, ws + 2 * (size_t)P * K * K);
            TIP_CHECK_CUDA(cudaGetLastError());
        } else if constexpr (2 * TBL <= kPSlotDoubles) {
            int base = 0;
            const int rc0 = upload_p_slot(K, p, f32, st, &base);
            if (rc0 != 0) return rc0;
            g_phase_off0 = base * tscale;
            g_phase_off1 = base * tscale + TBL;
        } else if constexpr (2 * TBL <= kPBankDoubles) {
            const int rc0 = upload_p_const(K, p, 0, 2, 0, f32, st);
            if (rc0 != 0) return rc0;
            g_phase_off0 = 0;
            g_phase_off1 = TBL;
        }
        if (K > 4) TIP_CHECK_CUDA(cudaMemsetAsync(ws, 0, em_tuned_workspace_bytes(P, K, false), st));  // M_g only
    }
    int rc = 0;
    if (!(phases & kPhaseRun) || n_rows == 0) {
        rc = 0;
    } else if (seg) {
        if constexpr (K > 4)
            rc = launch_variant<K, 16, false, double, true>(P, rows, n_rows, n_rows_r0, theta, 0, 0, stats, ws, st);
    } else if constexpr (K > 10) {
        // K >= 14 prefers 10 resident warps with ~198 registers and no spills (1e7 links: K=16 8.16 vs 8.96 ms,
        // K=14 6.10 vs 6.27 ms); K = 11..13 stay at 12.
        rc = run_rows<K, (K >= 14) ? 10 : 12, false, double>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, st);
    } else if (f32) {
        rc = run_rows<K, 16, false, float>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, st);
    } else if (with_ll) {
        rc = run_rows<K, 12, true, double>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, st);
    } else {
        // resident warp-CTAs per SM (register budget 65536 / (32 MINB)): measured at 1e7 links, K = 10 gains 6-7 % and
        // K = 8 2.6 % from 16 (128 registers, ~90 bytes of spills) over 12 (158 registers); K = 9 loses 1 %, K <= 6
        // does not care.
        rc = run_rows<K, (K == 10 || K == 8) ? 16 : 12, false, double>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, st);
    }
    if (rc != 0) return rc;
    if (!(phases & kPhaseEnd)) return 0;
    if constexpr (K > 4) {
        static bool fin_attr = false;
        if (!fin_attr) {
            TIP_CHECK_CUDA(cudaFuncSetAttribute(em_finalize_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                (int)fin_smem_bytes<K>()));
            fin_attr = true;
        }
        int grid = 2 * sm_count();
        if (grid > P) grid = P;
        em_finalize_kernel<K><<<grid, kFinThreads, fin_smem_bytes<K>(), st>>>(P, theta, p, ws, stats);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    return 0;
}

// K = 17..32: only the gene-segmented formulation exists (p does not fit the constant bank, and 4K doubles of
// per-link state do not fit the register file); same phases as launch_em_fused
template <int K>
static int launch_em_seg_large(int P, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta,
                               const double *p, double *stats, double *ws, int phases, cudaStream_t st)
{
    if (phases & kPhaseBegin) {
        const int64_t n = 2ll * P * K * K;
        const int threads = 256;
        int64_t want = (n + threads - 1) / threads;
        const int grid = (int)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16);
        seg_prep_kernel<<<grid, threads, 0, st>>>(P, K, theta, p, ws + 2 * (size_t)P * K * K);
        TIP_CHECK_CUDA(cudaGetLastError());
        TIP_CHECK_CUDA(cudaMemsetAsync(ws, 0, sizeof(double) * 2 * (size_t)P * K * K, st));
    }
    if ((phases & kPhaseRun) && n_rows > 0) {
        const int rc = launch_variant<K, 8, false, double, true>(P, rows, n_rows, n_rows_r0, theta, 0, 0, stats, ws, st);
        if (rc != 0) return rc;
    }
    if (phases & kPhaseEnd) return launch_finalize_generic(P, K, theta, p, ws, stats, st);
    return 0;
}

// ---------------------------------------------------------------------------------------------
// Model.compute_likelihood on the same machinery (K <= 10): lane = link, only the normaliser
//   d = eps + sum_a th_a[a] sum_b th_b[b] sum_c p[abc] th_c[c]        (K^3 + K^2 DFMA per link)
// Per-CTA partial sums land in `partials`; the last CTA to finish adds them in index order, so the
// result does not depend on scheduling.
// ---------------------------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(32, 16)
    loglik_fused_kernel(const int4 *__restrict__ rows, int n_tiles, int n_tiles_r0, const double *__restrict__ theta,
                        int p_slot, double *__restrict__ partials, unsigned *__restrict__ counter, double *__restrict__ out)
{
    using C = EmCfg<K>;
    constexpr int KP = C::KP, RS = C::RS;
    __shared__ __align__(16) double stage[32 * RS];
    __shared__ __align__(16) int4 ids_sm[32];
    const int lane = threadIdx.x;
    unsigned bx_v, gx_v;  // per-lane copies of the block coordinates, see em_fused_kernel
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(bx_v));
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(gx_v));
    const int4 *rp = rows + (int64_t)bx_v * 32 + lane;
    const int64_t rstride = (int64_t)gx_v * 32;
    double ll = 0.0;
    for (int t = blockIdx.x; t < n_tiles; t += gridDim.x) {
        __syncwarp();
        ids_sm[lane] = *rp;
        rp += rstride;
        __syncwarp();
        gather_tile<K, RS, KP>(theta, ids_sm, stage, lane);
        cp_async_commit();
        cp_async_wait<0>();
        __syncwarp();
        const double cnt = (double)row_count(ids_sm[lane].w);
        const int r = t >= n_tiles_r0 ? 1 : 0;
        const int pbase = p_slot * kPSlotDoubles + r * (K * K * KP);
        const double *row = stage + lane * RS;
        double tb[KP], tc[KP];
#pragma unroll
        for (int k = 0; k < KP; k += 2) {
            const double2 b2 = *reinterpret_cast<const double2 *>(row + KP + k);
            const double2 c2 = *reinterpret_cast<const double2 *>(row + 2 * KP + k);
            tb[k] = b2.x; tb[k + 1] = b2.y;
            tc[k] = c2.x; tc[k + 1] = c2.y;
        }
        double dsum = 0.0;
        const double *ta_p = row;
#pragma unroll 1
        for (int a = 0; a < K; ++a) {
            const double ta = *ta_p++;
            const int pa = pbase + a * (K * KP);
            double u = 0.0;
#pragma unroll
            for (int b = 0; b < K; ++b) {
                double q0 = 0.0, q1 = 0.0;
#pragma unroll
                for (int c = 0; c < K; c += 2) {
                    q0 = fma(c_pem[pa + b * KP + c], tc[c], q0);
                    if (c + 1 < K) q1 = fma(c_pem[pa + b * KP + c + 1], tc[c + 1], q1);
                }
                u = fma(tb[b], q0 + q1, u);
            }
            dsum = fma(ta, u, dsum);
        }
        if (cnt != 0.0) ll += cnt * log(TIP_EPS + dsum);
    }
    ll = warp_sum(ll);
    __shared__ bool last;
    if (lane == 0) {
        partials[bx_v] = ll;  // per-lane uses go through the clusterid copies (see em_fused_kernel)
        __threadfence();
        last = (atomicAdd(counter, 1u) == gx_v - 1);
    }
    __syncwarp();
    if (last) {
        __threadfence();
        // fixed-order sum of the partials: lanes take strided slices, then a butterfly
        double t = 0.0;
        for (unsigned i = lane; i < gx_v; i += 32) t += reinterpret_cast<volatile double *>(partials)[i];
        t = warp_sum(t);
        if (lane == 0) {
            *out = t;
            *counter = 0;
        }
    }
}

template <int K>
static int launch_loglik_fused(const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, const double *p,
                               double *out, double *partials, unsigned *counter, int max_blocks, cudaStream_t st)
{
    int base = 0;
    {
        const int rc0 = upload_p_slot(K, p, false, st, &base);
        if (rc0 != 0) return rc0;
    }
    const int slot = base / kPSlotDoubles;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        int nb = 0;
        TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, loglik_fused_kernel<K>, 32, 0));
        blocks_per_sm = nb < 1 ? 1 : nb;
    }
    const int64_t n_tiles = n_rows / 32;
    int64_t cap = (int64_t)sm_count() * blocks_per_sm;
    if (cap > max_blocks) cap = max_blocks;
    int grid = (int)(n_tiles < cap ? n_tiles : cap);
    if (grid < 1) grid = 1;
    loglik_fused_kernel<K><<<grid, 32, 0, st>>>(rows, (int)n_tiles, (int)(n_rows_r0 / 32), theta, slot, partials, counter, out);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

int launch_loglik_tuned(int K, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, const double *p,
                        double *out, double *partials, unsigned *counter, int max_blocks, cudaStream_t st, bool *handled)
{
    *handled = true;
    switch (K) {
        case 1: return launch_loglik_fused<1>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 2: return launch_loglik_fused<2>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 3: return launch_loglik_fused<3>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 4: return launch_loglik_fused<4>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 5: return launch_loglik_fused<5>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 6: return launch_loglik_fused<6>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 7: return launch_loglik_fused<7>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 8: return launch_loglik_fused<8>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 9: return launch_loglik_fused<9>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        case 10: return launch_loglik_fused<10>(rows, n_rows, n_rows_r0, theta, p, out, partials, counter, max_blocks, st);
        default: *handled = false; return 0;
    }
}

// ---------------------------------------------------------------------------------------------
// Model.compute_likelihood for K = 11..32 in the gene-segmented formulation (run-time K):
//   Z_g = theta_g . p  (seg_prep_kernel),   d = eps + sum_b th_b[b] sum_c Z_a[b][c] th_c[c]     (K^2 FMA per link)
// Same deterministic reduction of per-CTA partials as loglik_fused_kernel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32, 16)
    loglik_seg_kernel(int P, int K, const int4 *__restrict__ rows, int n_tiles, const double *__restrict__ theta,
                      const double *__restrict__ Zg, double *__restrict__ partials, unsigned *__restrict__ counter,
                      double *__restrict__ out)
{
    extern __shared__ __align__(16) double lsm[];   // [32][2K+1]: th_b | th_c per link (odd stride: conflict-free)
    const int lane = threadIdx.x, RSL = 2 * K + 1, KK = K * K;
    unsigned bx_v, gx_v;
    asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(bx_v));
    asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(gx_v));
    double ll = 0.0;
    for (unsigned t = bx_v; t < (unsigned)n_tiles; t += gx_v) {
        const int4 me = rows[(int64_t)t * 32 + lane];
        __syncwarp();
        // gather th_b and th_c of the 32 links (row-contiguous: consecutive lanes read consecutive doubles)
        for (int e = lane; e < 32 * 2 * K; e += 32) {
            const int l = e / (2 * K), rem = e - l * 2 * K, slot = rem / K, k = rem - slot * K;
            // (the shuffled value is evaluated in the SOURCE lane: fetch both slots, select by this lane's slot)
            const int gb = __shfl_sync(0xffffffffu, me.y, l), gc = __shfl_sync(0xffffffffu, me.z, l);
            const int gsrc = slot == 0 ? gb : gc;
            lsm[l * RSL + rem] = __ldg(theta + (int64_t)gsrc * K + k);
        }
        __syncwarp();
        const int cnt = row_count(me.w);
        const double *Zrow = Zg + ((int64_t)row_rating(me.w) * P + me.x) * KK;
        const double *tb = lsm + lane * RSL, *tc = tb + K;
        double dsum = 0.0;
        for (int b = 0; b < K; ++b) {
            double y0 = 0.0, y1 = 0.0;
            int c = 0;
            for (; c + 1 < K; c += 2) {
                y0 = fma(__ldg(Zrow + b * K + c), tc[c], y0);
                y1 = fma(__ldg(Zrow + b * K + c + 1), tc[c + 1], y1);
            }
            if (c < K) y0 = fma(__ldg(Zrow + b * K + c), tc[c], y0);
            dsum = fma(tb[b], y0 + y1, dsum);
        }
        if (cnt != 0) ll += (double)cnt * log(TIP_EPS + dsum);
    }
    ll = warp_sum(ll);
    __shared__ bool last;
    if (lane == 0) {
        partials[bx_v] = ll;
        __threadfence();
        last = (atomicAdd(counter, 1u) == gx_v - 1);
    }
    __syncwarp();
    if (last) {
        __threadfence();
        double t = 0.0;
        for (unsigned i = lane; i < gx_v; i += 32) t += reinterpret_cast<volatile double *>(partials)[i];
        t = warp_sum(t);
        if (lane == 0) {
            *out = t;
            *counter = 0;
        }
    }
}

size_t loglik_seg_workspace_bytes(int P, int K) { return K > 10 ? sizeof(double) * 2 * (size_t)P * K * K : 0; }

int launch_loglik_seg(int P, int K, const int4 *rows, int64_t n_rows, const double *theta, const double *p, double *out,
                      double *partials, unsigned *counter, int max_blocks, double *Zws, cudaStream_t st)
{
    const int64_t n = 2ll * P * K * K;
    int64_t want = (n + 255) / 256;
    seg_prep_kernel<<<(int)(want < (int64_t)sm_count() * 16 ? want : (int64_t)sm_count() * 16), 256, 0, st>>>(P, K, theta, p, Zws);
    TIP_CHECK_CUDA(cudaGetLastError());
    const int64_t n_tiles = n_rows / 32;
    int64_t cap = (int64_t)sm_count() * 16;
    if (cap > max_blocks) cap = max_blocks;
    const int grid = (int)(n_tiles < cap ? (n_tiles < 1 ? 1 : n_tiles) : cap);
    const size_t smem = sizeof(double) * 32 * (2 * K + 1);
    loglik_seg_kernel<<<grid, 32, smem, st>>>(P, K, rows, (int)n_tiles, theta, Zws, partials, counter, out);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// The "run" phase of the plain fp64 K <= 10 E-step over rows that are still arriving from the host (see StreamArrive).
// Between launch_em_tuned(phases = kPhaseBegin) and (phases = kPhaseEnd) on the same stream.
bool em_streamed_available(int K, bool with_ll, bool f32, bool seg) { return K >= 1 && K <= 10 && !with_ll && !f32 && !seg; }

template <int K>
static int launch_streamed_k(int P, const void *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, double *stats,
                             double *ws, StreamArrive sa, cudaStream_t st)
{
    constexpr int MINB = (K == 10 || K == 8) ? 16 : 12;  // as in launch_em_fused
    return launch_variant<K, MINB, false, double, false, true>(P, reinterpret_cast<const int4 *>(rows), n_rows, n_rows_r0, theta,
                                                                  g_phase_off0, g_phase_off1, stats, ws, st, sa);
}

int launch_em_streamed(int P, int K, const void *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, double *stats,
                       double *ws, unsigned *err, unsigned long long *chk, bool compact, cudaStream_t st)
{
    StreamArrive sa;
    sa.chk = chk;
    TIP_CHECK_CUDA(cudaMemsetAsync(chk, 0, 4 * sizeof(unsigned long long), st));
    sa.err = err;
    sa.compact = compact ? 1 : 0;
    // 5 s: a host that stopped feeding the copy stream must not hang the GPU (TIP_STREAM_TIMEOUT_US overrides it, so
    // that the give-up path can be exercised in tests)
    const char *to = getenv("TIP_STREAM_TIMEOUT_US");
    sa.timeout_ns = to ? 1000ull * strtoull(to, nullptr, 10) : 5000000000ull;
    switch (K) {
        case 1: return launch_streamed_k<1>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 2: return launch_streamed_k<2>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 3: return launch_streamed_k<3>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 4: return launch_streamed_k<4>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 5: return launch_streamed_k<5>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 6: return launch_streamed_k<6>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 7: return launch_streamed_k<7>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 8: return launch_streamed_k<8>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 9: return launch_streamed_k<9>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        case 10: return launch_streamed_k<10>(P, rows, n_rows, n_rows_r0, theta, stats, ws, sa, st);
        default: set_error("launch_em_streamed: K = %d has no streamed kernel", K); return -1;
    }
}

int launch_em_tuned(int P, int K, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta,
                    const double *p, double *stats, double *ws, bool with_ll, bool f32, bool seg, cudaStream_t st,
                    bool *handled, int phases)
{
    *handled = true;
    switch (K) {
        case 1: return launch_em_fused<1>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 2: return launch_em_fused<2>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 3: return launch_em_fused<3>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 4: return launch_em_fused<4>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 5: return launch_em_fused<5>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 6: return launch_em_fused<6>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 7: return launch_em_fused<7>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 8: return launch_em_fused<8>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 9: return launch_em_fused<9>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 10: return launch_em_fused<10>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 11: return launch_em_fused<11>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 12: return launch_em_fused<12>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 13: return launch_em_fused<13>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 14: return launch_em_fused<14>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 15: return launch_em_fused<15>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 16: return launch_em_fused<16>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, with_ll, f32, seg, phases, st);
        case 17: return launch_em_seg_large<17>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 18: return launch_em_seg_large<18>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 19: return launch_em_seg_large<19>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 20: return launch_em_seg_large<20>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 21: return launch_em_seg_large<21>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 22: return launch_em_seg_large<22>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 23: return launch_em_seg_large<23>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 24: return launch_em_seg_large<24>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 25: return launch_em_seg_large<25>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 26: return launch_em_seg_large<26>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 27: return launch_em_seg_large<27>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 28: return launch_em_seg_large<28>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 29: return launch_em_seg_large<29>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 30: return launch_em_seg_large<30>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 31: return launch_em_seg_large<31>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        case 32: return launch_em_seg_large<32>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, phases, st);
        default: *handled = false; return 0;
    }
}

}  // namespace tip
