// Slot-segmented E-step (TIP_EM_SLOT_SEGMENTED) for sm_100a: every theta statistic of Model.make_iteration
// (TIP.py:1009-1011) and the p statistic (TIP.py:1012) are accumulated per RUN OF EQUAL GENE, in three sort orders of
// the same links, so that no statistic is ever scattered with per-link atomics - a hub gene (a Kuzmin query gene
// sits in tens of thousands of triplets) costs the same as any other.
//
// For a link (a, b, c) of rating r with count n:   d = eps + sum_abc th_a th_b th_c p_abc,r ,  s = n / d.
//   pass A (rows ordered by slot-a gene g):  Z_g[b][c] = sum_a th_g[a] p[a][b][c][r]       (once per gene, seg3_prep_kernel)
//                                            d = eps + sum_bc th_b[b] th_c[c] Z_g[b][c]    K^2 DFMA, lane = link
//                                            s -> sbuf[position of the link in order a]
//                                            M0_g[b][c] += s th_b[b] th_c[c]               K^2, tensor pipe (DMMA)
//   pass B (rows ordered by slot-b gene g):  M1_g[a][c] += s th_a[a] th_c[c]               s read back from sbuf
//   pass C (rows ordered by slot-c gene g):  M2_g[a][b] += s th_a[a] th_b[b]
//   finish (once per iteration, per gene):   Ntheta[g][k] = th_g[k] * sum_{slot, r} sum_xy P_slot[r][k][xy] M_slot,r,g[xy]
//                                            S[r][a][bc]  = sum_g th_g[a] M0_r,g[bc]        (npr = p * S)
// A link costs 4 K^2 FMA instead of 3 K^3; what bounds the kernels is the gather of six theta rows per link from
// L2 (6 x 96 bytes at K = 10) and instruction issue, not the FMA pipe.
//
// The M accumulation of a 32-link tile is a [K x 32] . [32 x K] product: it runs on the fp64 tensor path
// (mma.sync.m8n8k4.f64, SASS DMMA - same pipe as DFMA, a quarter of the issue slots).  Operands are staged
// TRANSPOSED in shared memory ([component][link], stride 36 doubles: fragment loads and the lane = link stores are
// both conflict-free).  Accumulator fragments stay in registers across tiles and are flushed (red.global.add.f64)
// only where the run of equal gene ends or the warp's chunk of tiles ends: atomics per iteration ~ K^2 x (#runs +
// #chunks) instead of 2 K x #links.
//
// Scheduling.  A tile's cost grows with the number of runs it holds (every run end is a flush and a Z fetch), and
// hub-shaped links put tiles with 20-30 one-link runs (array genes that appear once or twice in a slot) next to thousands
// of tiles inside one hub run: handing out consecutive tiles left a few warps with ten such tiles each and the SMs idle
// for 70 % of the kernel (ncu: 354k cycles elapsed, 100k active).  tip_order_rows therefore writes a SCHEDULE per
// launch - chunks of up to four consecutive tiles, tiles with many runs on their own, sorted by descending cost, single
// tiles at the very end - and the single-warp CTAs draw chunk after chunk from one atomic counter (longest processing time
// first; two draws in flight per warp).
//
// Overlap of the two pass launches.  A warp needs ~7 us per tile and handles only ~10 tiles per launch, so the last tiles
// of a launch leave most SMs idle for 15-20 us (ncu: sm__cycles_active min 84k / max 134k of 140k elapsed).  Pass B + C is
// therefore launched with the programmatic-dependent-launch attribute and pass A releases it at once
// (griddepcontrol.launch_dependents): its CTAs move in as pass-A CTAs retire and work on the tiles whose s values are
// there.  sbuf starts every iteration as NaN (written by seg3_prep_kernel); pass A publishes s with st.relaxed.gpu, pass
// B + C checks the s it gathered and re-reads (ld.relaxed.gpu) the ones still NaN.  Every pass-A tile has been drawn by
// a resident warp before the first pass-B tile can be (A's grid is one resident wave), so the wait is bounded; a wait of
// more than ~2 s poisons the statistics with NaN instead of hanging.
#include <cub/device/device_radix_sort.cuh>

#include "tip_common.cuh"

namespace tip {

__device__ __forceinline__ void dmma884(double &c0, double &c1, double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

__device__ __forceinline__ void red_add_f64_nz3(double *addr, double v)
{
    asm volatile("{ .reg .pred p; setp.neu.f64 p, %1, 0d0000000000000000; @p red.global.add.f64 [%0], %1; }" ::"l"(addr),
                 "d"(v)
                 : "memory");
}

__device__ __forceinline__ void st_relaxed_gpu_f64(double *addr, double v)
{
    asm volatile("st.relaxed.gpu.global.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ double ld_relaxed_gpu_f64(const double *addr)
{
    double v;
    asm volatile("ld.relaxed.gpu.global.f64 %0, [%1];" : "=d"(v) : "l"(addr) : "memory");
    return v;
}

template <int K>
struct S3 {
    static constexpr int KK = K * K;
    static constexpr int NB = (K + 7) / 8;    // 8 x 8 accumulator blocks per dimension of M
    static constexpr int NKG = (K + 3) / 4;   // k-steps of the d contraction
    // stage row [th_x | th_y] of a link, stride == 4 (mod 16) doubles: the two fragment access patterns of this kernel -
    // (row = link, col = component) and (row = component, col = link) - both hit every bank pair exactly twice
    static constexpr int RS = ((2 * K + 11) / 16) * 16 + 4;
    static constexpr size_t BUF_BYTES = (size_t)32 * RS * 8 + 32 * 8 + 32 * 16;   // stage | s | ids
    static constexpr int UNIT = (K % 2 == 0) ? 2 : 1;                  // doubles per cp.async
    static constexpr int U = K / UNIT;                                 // copies per theta row
    static constexpr int LPI = (2 * U <= 32) ? 32 / (2 * U) : 0;       // whole links per gather instruction (0: flat mapping)
    static constexpr int ITERS = LPI ? (32 + LPI - 1) / LPI : 2 * U;
    static constexpr bool HOIST_Z = NB * NKG <= 12;                    // Z fragments of a run kept in registers
    static constexpr int TP = (K + 15) / 16 * 16;                      // row stride of the gather copy of theta: rows start on
                                                                       // 128-byte lines (one tag request and ceil(8K/32) sectors each)
};

constexpr int kS3Groups = 64;                 // chunk ranges / counters per launch
constexpr int kS3CounterDoubles = 2 * kS3Groups * 16;   // two launches x groups x one 128-byte line, as doubles

struct S3Args {
    int P;
    const int4 *rows;        // pass A: order a.  pass BC: order b followed by order c
    int n_tiles;             // tiles this launch walks (tiles_per_order, or 2 x tiles_per_order)
    int tiles_per_order;
    int n_tiles_r0;          // rating-0 tiles of an order
    int slot0;               // first slot of this launch (0 or 1)
    const double *theta;     // [P][TP]: the 128-byte-aligned copy seg3_prep_kernel writes
    const double *Zg;        // [2][P][KK]            (pass A)
    double *sbuf;            // [tiles_per_order * 32] (written by pass A, read by pass BC)
    double *Mg;              // [3][2][P][KK]
    unsigned *counter;       // schedule position counter of this launch, zero on entry
    const int *sched;        // chunks of this launch: (first tile << 3) | tiles, by descending cost; 0 = end of the list
    int n_sched;             // entries in sched (real chunks first, zeros behind them)
};

__device__ __forceinline__ void cp_async_16_ca(void *smem_dst, const void *gmem_src)
{
    unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem_src) : "memory");
}
// 8 bytes, or zeros when src_bytes == 0 (the source is then not read)
__device__ __forceinline__ void cp_async_8_zfill(void *smem_dst, const void *gmem_src, int src_bytes)
{
    unsigned s = static_cast<unsigned>(__cvta_generic_to_shared(smem_dst));
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(s), "l"(gmem_src), "r"(src_bytes) : "memory");
}

// theta rows of the 32 links of a tile -> stage[link][th_x | th_y].  K even: 16-byte copies, whole links per warp
// instruction (a row is never split over two instructions, so its sectors are requested once).  CA: through L1
// (cp.async.ca) - what hub-shaped links need, the few hub rows then stay in L1 instead of hammering a handful of L2
// slices from every SM; .cg (L2 only) otherwise.  The gene ids are read first, then the copies are issued back to back.
template <int K, bool CA>
__device__ __forceinline__ void s3_gather(const double *__restrict__ theta, const int4 *ids_sm, double *stage, int lane)
{
    using C = S3<K>;
    const int *idw = reinterpret_cast<const int *>(ids_sm);
    auto copy = [&](int g, int l, int slot, int k0) {
        double *dst = stage + l * C::RS + slot * K + k0;
        const double *src = theta + (int64_t)g * C::TP + k0;
        if (C::UNIT == 2) {
            if (CA)
                cp_async_16_ca(dst, src);
            else
                cp_async_16(dst, src);
        } else {
            cp_async_8(dst, src);
        }
    };
    if constexpr (C::LPI > 0) {
        const int sub = lane / (2 * C::U), rem = lane - sub * (2 * C::U);
        const int slot = rem / C::U, k0 = (rem - slot * C::U) * C::UNIT;
        if (sub < C::LPI) {
            int g[C::ITERS];
#pragma unroll
            for (int it = 0; it < C::ITERS; ++it) {
                const int l = it * C::LPI + sub;
                g[it] = (32 % C::LPI == 0 || l < 32) ? idw[l * 4 + 1 + slot] : 0;
            }
#pragma unroll
            for (int it = 0; it < C::ITERS; ++it) {
                const int l = it * C::LPI + sub;
                if (32 % C::LPI == 0 || l < 32) copy(g[it], l, slot, k0);
            }
        }
    } else {
#pragma unroll 4
        for (int it = 0; it < C::ITERS; ++it) {
            const int u = it * 32 + lane;
            const int l = u / (2 * C::U), rem = u - l * (2 * C::U);
            const int slot = rem / C::U;
            copy(idw[l * 4 + 1 + slot], l, slot, (rem - slot * C::U) * C::UNIT);
        }
    }
}

// Two stage buffers: the gather of the next tile is in flight while a tile is computed
template <int K, bool FIRST, bool CA>
__global__ void __launch_bounds__(32, K <= 16 ? (FIRST ? 16 : 18) : 1) seg3_pass_kernel(const S3Args a)
{
    using C = S3<K>;
    constexpr int KK = C::KK, NB = C::NB, NKG = C::NKG, RS = C::RS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x, li = lane & 3, ri = lane >> 2;
    if constexpr (FIRST) {
        // pass A is itself a programmatic dependent of the prep kernel (its CTAs are resident and past their launch latency
        // when the prep kernel ends): wait for the prep kernel's results FIRST, then let pass B + C move in behind us - in
        // that order, so that pass B + C can never start before the prep kernel is complete
        asm volatile("griddepcontrol.wait;" ::: "memory");
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }
    auto stage_of = [&](int b) { return reinterpret_cast<double *>(smem_raw + (size_t)b * C::BUF_BYTES); };
    auto ids_of = [&](int b) { return reinterpret_cast<int4 *>(stage_of(b) + 32 * RS + 32); };
    // fragment coordinates of this lane: component i*8 + ri of an 8 x 8 block (rows/cols >= K read as zero)
    int xo[NB];
    bool xv[NB];
#pragma unroll
    for (int i = 0; i < NB; ++i) {
        xv[i] = i * 8 + ri < K;
        xo[i] = xv[i] ? i * 8 + ri : 0;
    }

    double acc[NB][NB][2];
#pragma unroll
    for (int i = 0; i < NB; ++i)
#pragma unroll
        for (int j = 0; j < NB; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
    auto flush = [&](int mrow) {
        double *dst = a.Mg + (int64_t)mrow * KK;
#pragma unroll
        for (int i = 0; i < NB; ++i)
#pragma unroll
            for (int j = 0; j < NB; ++j) {
                const int x = i * 8 + ri, y = j * 8 + 2 * li;
                if (x < K && y < K) red_add_f64_nz3(dst + x * K + y, acc[i][j][0]);
                if (x < K && y + 1 < K) red_add_f64_nz3(dst + x * K + y + 1, acc[i][j][1]);
                acc[i][j][0] = acc[i][j][1] = 0.0;
            }
    };
    auto mbase_of = [&](int tt) {   // a launch walks one order (pass A) or two (pass B + C): no division needed
        const int so = tt >= a.tiles_per_order ? 1 : 0, tl = tt - (so ? a.tiles_per_order : 0);
        return ((a.slot0 + so) * 2 + (tl >= a.n_tiles_r0 ? 1 : 0)) * a.P;
    };

    // ---- tile sequence of this warp: chunks of the schedule, drawn from one atomic counter.  Lane 0 keeps one schedule
    // entry loaded (`ent`, the next chunk) and one position drawn ahead (`pos2`): the counter's round trip and the entry's
    // load both have a whole chunk of compute to return.
    int gen_t = 0, gen_end = 0;
    bool gen_done = false;
    unsigned pos2 = 0;
    int ent = 0;
    if (lane == 0) {
        // the first two chunks of every warp are fixed (positions w and w + #warps: the heaviest tiles, which head the
        // list, are spread one per warp, and nobody queues at the counter before doing any work); the counter starts at
        // 2 x #warps (written by seg3_prep_kernel)
        const unsigned p0 = blockIdx.x;
        pos2 = blockIdx.x + gridDim.x;
        ent = p0 < (unsigned)a.n_sched ? __ldg(a.sched + p0) : 0;
    }
    auto next_tile = [&]() -> int {
        if (gen_t < gen_end) return gen_t++;
        if (gen_done) return -1;
        const int e = __shfl_sync(0xffffffffu, ent, 0);
        if (e == 0) {
            gen_done = true;
            return -1;
        }
        if (lane == 0) {
            ent = pos2 < (unsigned)a.n_sched ? __ldg(a.sched + pos2) : 0;
            pos2 = atomicAdd(a.counter, 1u);
        }
        gen_t = e >> 3;
        gen_end = gen_t + (e & 7);
        return gen_t++;
    };
    auto issue_gather = [&](int buf, const int4 &me) {
        int4 *ids = ids_of(buf);
        double *st = stage_of(buf);
        ids[lane] = me;
        __syncwarp();
        s3_gather<K, CA>(a.theta, ids, st, lane);
        if constexpr (!FIRST) cp_async_8_zfill(st + 32 * RS + lane, a.sbuf + (me.w >= 0 ? me.w : 0), me.w >= 0 ? 8 : 0);
    };

    // tq[0]: tile computed this iteration (gathered into buffer cb); tq[1 .. RQ]: rows held in registers
    // (the rows come from HBM: RQ tiles of lookahead hide that latency)
    constexpr int RQ = 2;
    int tq[1 + RQ];
    int4 meq[RQ];
    tq[0] = next_tile();
    if (tq[0] >= 0) issue_gather(0, a.rows[(int64_t)tq[0] * 32 + lane]);
    cp_async_commit();
#pragma unroll
    for (int j = 0; j < RQ; ++j) {
        tq[1 + j] = next_tile();
        meq[j] = make_int4(0, 0, 0, 0);
        if (tq[1 + j] >= 0) meq[j] = a.rows[(int64_t)tq[1 + j] * 32 + lane];
    }

    int cb = 0;    // buffer of tq[0]
    int cur = -1;  // run the accumulators belong to (-1: none)
    int zcur = -1; // run whose Z fragments are in registers
    int znext = -1; // run whose Z fragments were requested ahead (the first run of the next tile)
    double zf[C::HOIST_Z ? NB : 1][C::HOIST_Z ? NKG : 1], zn[C::HOIST_Z ? NB : 1][C::HOIST_Z ? NKG : 1];
    (void)zcur; (void)zf; (void)znext; (void)zn;
    auto load_z = [&](double (&dst)[C::HOIST_Z ? NB : 1][C::HOIST_Z ? NKG : 1], int mrow_z) {
        const double *Zr = a.Zg + (int64_t)mrow_z * KK;
#pragma unroll
        for (int j = 0; j < (C::HOIST_Z ? NB : 1); ++j)
#pragma unroll
            for (int kg = 0; kg < (C::HOIST_Z ? NKG : 1); ++kg)
                dst[j][kg] = (xv[j] && 4 * kg + li < K) ? __ldg(Zr + xo[j] * K + 4 * kg + li) : 0.0;
    };

    while (tq[0] >= 0) {
        // ---- A: gather of the next tile into the other buffer; B: rows of the tile after it ----
        if (tq[1] >= 0) issue_gather(cb ^ 1, meq[0]);
        cp_async_commit();
        const int tn = next_tile();
#pragma unroll
        for (int j = 0; j + 1 < RQ; ++j) meq[j] = meq[j + 1];
        if (tn >= 0) meq[RQ - 1] = a.rows[(int64_t)tn * 32 + lane];
        cp_async_wait<1>();
        __syncwarp();

        const int t = tq[0];
        double *st = stage_of(cb);
        double *ssm = st + 32 * RS;
        const int4 *ids = ids_of(cb);
        const int mrow = mbase_of(t) + ids[lane].x;
        int prev = __shfl_up_sync(0xffffffffu, mrow, 1);
        if (cur < 0) cur = __shfl_sync(0xffffffffu, mrow, 0);
        if (lane == 0) prev = cur;
        const unsigned bm = __ballot_sync(0xffffffffu, mrow != prev);  // bit l: link l starts a new run

        if constexpr (!FIRST) {
            // s of this tile's links was gathered while pass A may still have been running: NaN = not published yet
            const int w = ids[lane].w;
            double sv = ssm[lane];
            bool pending = w >= 0 && sv != sv;
            if (__any_sync(0xffffffffu, pending)) {
                unsigned spins = 0;
                do {
                    if (pending) {
                        sv = ld_relaxed_gpu_f64(a.sbuf + w);
                        pending = sv != sv;
                        if (!pending) ssm[lane] = sv;
                    }
                    if (++spins > (1u << 23)) break;     // ~2 s: leave the NaN in place, the statistics become NaN (loud)
                    if (pending) __nanosleep(200);
                } while (__any_sync(0xffffffffu, pending));
                __syncwarp();
            }
        }

        if constexpr (FIRST) {
            // ---- Y[link][b] = sum_c th_c[c] Z_g[b][c], one masked tensor product per run of equal gene ----
            double Y[4][NB][2];
#pragma unroll
            for (int rb = 0; rb < 4; ++rb)
#pragma unroll
                for (int j = 0; j < NB; ++j) Y[rb][j][0] = Y[rb][j][1] = 0.0;
            int l0 = 0;
            while (l0 < 32) {
                const unsigned rest = (l0 < 31) ? (bm & ~((2u << l0) - 1u)) : 0u;  // run starts after l0
                const int l1 = rest ? __ffs(rest) - 1 : 32;
                const int mseg = __shfl_sync(0xffffffffu, mrow, l0);
                const double *Zr = a.Zg + (int64_t)mseg * KK;
                if constexpr (C::HOIST_Z) {
                    if (mseg != zcur) {
                        if (mseg == znext) {
#pragma unroll
                            for (int j = 0; j < NB; ++j)
#pragma unroll
                                for (int kg = 0; kg < NKG; ++kg) zf[j][kg] = zn[j][kg];
                        } else {
                            load_z(zf, mseg);
                        }
                        zcur = mseg;
                    }
                    if (l1 < 32) {
                        // the next run of this tile: its Z fragments travel while this run is contracted
                        const int mnext = __shfl_sync(0xffffffffu, mrow, l1);
                        if (mnext != znext) {
                            load_z(zn, mnext);
                            znext = mnext;
                        }
                    }
                }
#pragma unroll
                for (int rb = 0; rb < 4; ++rb) {
                    if (rb * 8 < l1 && rb * 8 + 8 > l0) {
                        const int lr = rb * 8 + ri;
                        const bool in = lr >= l0 && lr < l1;
#pragma unroll
                        for (int kg = 0; kg < NKG; ++kg) {
                            const double av = (in && 4 * kg + li < K) ? st[lr * RS + K + 4 * kg + li] : 0.0;
#pragma unroll
                            for (int j = 0; j < NB; ++j) {
                                double zv;
                                if constexpr (C::HOIST_Z)
                                    zv = zf[j][kg];
                                else
                                    zv = (xv[j] && 4 * kg + li < K) ? __ldg(Zr + xo[j] * K + 4 * kg + li) : 0.0;
                                dmma884(Y[rb][j][0], Y[rb][j][1], av, zv);
                            }
                        }
                    }
                }
                l0 = l1;
            }
            // ---- d = eps + sum_b th_b[b] Y[b];  s = count / d for link li * 8 + ri ----
            double dsel = 1.0;
#pragma unroll
            for (int rb = 0; rb < 4; ++rb) {
                double part = 0.0;
#pragma unroll
                for (int j = 0; j < NB; ++j) {
                    const int b0 = j * 8 + 2 * li;
                    if (b0 < K) {  // (same for every use of this lane: no divergence cost beyond predication)
                        const double2 tb = *reinterpret_cast<const double2 *>(st + (rb * 8 + ri) * RS + b0);
                        part = fma(tb.x, Y[rb][j][0], part);
                        if (b0 + 1 < K) part = fma(tb.y, Y[rb][j][1], part);
                    }
                }
                part += __shfl_xor_sync(0xffffffffu, part, 1);
                part += __shfl_xor_sync(0xffffffffu, part, 2);
                if (li == rb) dsel = TIP_EPS + part;
            }
            if constexpr (C::HOIST_Z) {
                // Z fragments of the next tile's first run, requested now so that they land during the M phase below
                if (tq[1] >= 0) {
                    const int mnext = mbase_of(tq[1]) + ids_of(cb ^ 1)[0].x;
                    if (mnext != zcur && mnext != znext) {
                        load_z(zn, mnext);
                        znext = mnext;
                    }
                }
            }
            const int L = li * 8 + ri;
            // 1/d: fp32 reciprocal seed and three Newton steps (d lies in [1e-10, ~1]; last-ulp accuracy, see tip_em.cu)
            double rd = (double)__frcp_rn((float)dsel);
            rd = rd * fma(-dsel, rd, 2.0);
            rd = rd * fma(-dsel, rd, 2.0);
            rd = rd * fma(-dsel, rd, 2.0);
            const double s = (double)row_count(ids[L].w) * rd;
            ssm[L] = s;
            st_relaxed_gpu_f64(a.sbuf + (int64_t)t * 32 + L, s);
            __syncwarp();
        }

        // ---- M += (s th_x)^T . th_y over the runs of equal gene in this tile ----
        if (bm == 0u) {
            // the whole tile continues the current run: eight unconditional k-steps
#pragma unroll 4
            for (int ks = 0; ks < 8; ++ks) {
                const double *lrow = st + (4 * ks + li) * RS;
                const double sv = ssm[4 * ks + li];
                double av[NB], bv[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    av[i] = xv[i] ? lrow[xo[i]] * sv : 0.0;
                    bv[i] = xv[i] ? lrow[K + xo[i]] : 0.0;
                }
#pragma unroll
                for (int i = 0; i < NB; ++i)
#pragma unroll
                    for (int j = 0; j < NB; ++j) dmma884(acc[i][j][0], acc[i][j][1], av[i], bv[j]);
            }
        } else {
#pragma unroll 1
            for (int ks = 0; ks < 8; ++ks) {
                const unsigned nib = (bm >> (4 * ks)) & 15u;
                const double *lrow = st + (4 * ks + li) * RS;
                const double sv = ssm[4 * ks + li];
                double av[NB], bv[NB];
#pragma unroll
                for (int i = 0; i < NB; ++i) {
                    av[i] = xv[i] ? lrow[xo[i]] * sv : 0.0;
                    bv[i] = xv[i] ? lrow[K + xo[i]] : 0.0;
                }
                if (nib == 0) {
#pragma unroll
                    for (int i = 0; i < NB; ++i)
#pragma unroll
                        for (int j = 0; j < NB; ++j) dmma884(acc[i][j][0], acc[i][j][1], av[i], bv[j]);
                } else {
                    // a run ends inside these four links: one masked product per segment
                    int j0 = 0;
                    while (j0 < 4) {
                        if ((nib >> j0) & 1u) {
                            flush(cur);
                            cur = __shfl_sync(0xffffffffu, mrow, 4 * ks + j0);
                        }
                        const unsigned higher = nib >> (j0 + 1);
                        const int len = higher ? __ffs(higher) : 4 - j0;
                        const bool mine = li >= j0 && li < j0 + len;
#pragma unroll
                        for (int i = 0; i < NB; ++i)
#pragma unroll
                            for (int j = 0; j < NB; ++j) dmma884(acc[i][j][0], acc[i][j][1], mine ? av[i] : 0.0, bv[j]);
                        j0 += len;
                    }
                }
            }
        }
        if (tq[1] != t + 1) {  // the warp's chunk ends here
            flush(cur);
            cur = -1;
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < RQ; ++j) tq[j] = tq[j + 1];
        tq[RQ] = tn;
        cb ^= 1;
    }
}

// Z[r][g][b][c] = sum_a theta[g][a] p[a][b][c][r]  (one CTA per group of genes, p staged in shared memory), and the three
// orientations of p the finish contracts with:
//   PT[slot][r][k][e]:  slot 0: k = a, e = (b, c);  slot 1: k = b, e = (a, c);  slot 2: k = c, e = (a, b)
constexpr int kPrepGenes = 16;
__global__ void __launch_bounds__(256) seg3_prep_kernel(int P, int K, const double *__restrict__ theta,
                                                        const double *__restrict__ p, double *__restrict__ Zg,
                                                        double *__restrict__ PT, double *__restrict__ thpad, int TP,
                                                        double2 *__restrict__ zero2, int64_t n_zero2,
                                                        double2 *__restrict__ nan2, int64_t n_nan2,
                                                        unsigned *__restrict__ cnt_a, unsigned cnt_a0,
                                                        unsigned *__restrict__ cnt_bc, unsigned cnt_bc0)
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");   // pass A may become resident (it waits for this grid)
    if (blockIdx.x == 0 && threadIdx.x == 0) {   // schedule positions 0 .. 2 x #warps - 1 are taken statically
        *cnt_a = cnt_a0;
        *cnt_bc = cnt_bc0;
    }
    extern __shared__ double psm[];  // [2][K^3]  p[r][a][bc]  (K <= 20), then theta of this CTA's genes [kPrepGenes][K]
    const int KK = K * K, K3 = KK * K;
    const bool staged = K <= 20;
    double *tsm = psm + (staged ? 2 * K3 : 0);
    const int g0 = blockIdx.x * kPrepGenes;
    const int ng = (P - g0 < kPrepGenes) ? P - g0 : kPrepGenes;
    // the loads of this CTA's operands go out FIRST (eight of p per thread and its theta value: one L2 round trip instead
    // of eight dependent ones - the staging store was the hottest line, long-scoreboard, of the first version) ...
    constexpr int PB = 8;
    double pv[PB];
    const int e_th = threadIdx.x;
    double tv = 0.0;
    if (e_th < ng * K) tv = __ldg(theta + (int64_t)g0 * K + e_th);
    if (staged) {
#pragma unroll
        for (int j = 0; j < PB; ++j) {
            const int e = threadIdx.x + j * 256;
            pv[j] = e < 2 * K3 ? __ldg(p + e) : 0.0;
        }
    }
    // ... and travel while the fills are issued: the accumulators M start every E-step from zero, sbuf from NaN ("not
    // published") - fire-and-forget stores spread over the CTAs instead of two memset launches
    {
        const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, nth = (int64_t)gridDim.x * blockDim.x;
        for (int64_t i = tid; i < n_zero2; i += nth) zero2[i] = make_double2(0.0, 0.0);
        const double qn = __longlong_as_double(-1ll);
        for (int64_t i = tid; i < n_nan2; i += nth) nan2[i] = make_double2(qn, qn);
    }
    if (staged) {
#pragma unroll
        for (int j = 0; j < PB; ++j) {
            const int e = threadIdx.x + j * 256;
            if (e < 2 * K3) psm[(e & 1) * K3 + (e >> 1)] = pv[j];
        }
        for (int e = threadIdx.x + PB * 256; e < 2 * K3; e += blockDim.x) psm[(e & 1) * K3 + (e >> 1)] = __ldg(p + e);
    }
    for (int e = threadIdx.x; e < ng * K; e += blockDim.x) {
        const double v = e == e_th ? tv : __ldg(theta + (int64_t)g0 * K + e);
        tsm[e] = v;
        const int gi = e / K;
        thpad[(int64_t)(g0 + gi) * TP + (e - gi * K)] = v;   // the gather copy of theta: rows on 128-byte lines
    }
    __syncthreads();
    // thread = (rating, b, c); the genes of the CTA in the inner loop
    for (int rbc = threadIdx.x; rbc < 2 * KK; rbc += blockDim.x) {
        const int r = rbc >= KK ? 1 : 0, bc = rbc - r * KK;
        double *out = Zg + ((int64_t)r * P + g0) * KK + bc;
        if (staged && K <= 16) {
            // the K values of p of this cell are the same for every gene: once into registers (halves the shared-memory
            // loads of the loop - the kernel was issue-bound on LDS + address arithmetic, ncu r2_seg3_prep_k10_final_summary)
            double pk[16];
#pragma unroll
            for (int q = 0; q < 16; ++q) pk[q] = q < K ? psm[r * K3 + q * KK + bc] : 0.0;
            for (int gi = 0; gi < ng; ++gi) {
                double z = 0.0;
#pragma unroll
                for (int q = 0; q < 16; ++q)
                    if (q < K) z = fma(tsm[gi * K + q], pk[q], z);
                out[(int64_t)gi * KK] = z;
            }
            continue;
        }
        for (int gi = 0; gi < ng; ++gi) {
            double z = 0.0;
            if (staged)
                for (int q = 0; q < K; ++q) z = fma(tsm[gi * K + q], psm[r * K3 + q * KK + bc], z);
            else
                for (int q = 0; q < K; ++q) z = fma(tsm[gi * K + q], __ldg(p + ((int64_t)q * KK + bc) * 2 + r), z);
            out[(int64_t)gi * KK] = z;
        }
    }
    // the transposed copies of p: spread over the CTAs
    for (int f = blockIdx.x * blockDim.x + threadIdx.x; f < 6 * K3; f += gridDim.x * blockDim.x) {
        const int slot = f / (2 * K3), rem = f - slot * 2 * K3;
        const int r = rem / K3, ke = rem - r * K3, k = ke / KK, xy = ke - k * KK, x = xy / K, y = xy - x * K;
        int i, j, l;
        if (slot == 0) { i = k; j = x; l = y; }
        else if (slot == 1) { i = x; j = k; l = y; }
        else { i = x; j = y; l = k; }
        PT[f] = __ldg(p + (((int64_t)i * K + j) * K + l) * 2 + r);
    }
}

// Per-gene finish.  Warp tasks, both as small fp64 tensor products straight out of L2 (no shared memory):
//   kind 1, task (group of 8 genes):  Ntheta[g][k] = th_g[k] * sum_slot sum_r sum_e M_slot,r,g[e] PT[slot][r][k][e]
//   kind 2, task (r, block of 8 (b,c) cells, chunk of genes):  S[r][a][bc] += sum_g th_g[a] M_0,r,g[bc]
// A kind-1 task owns its eight rows of Ntheta (all three slots, both ratings): plain stores, no atomics - and, for link
// shards, the SAME values stored straight into this rank's slot of every peer's inbox (S3Push): the statistics travel
// over NVLink while the rest of the finish is still computing, and the exchange kernel that follows only has the 2 K^3
// doubles of S left to send before it signals (tip_peer_push_mstep with theta_pushed = 1).
constexpr int kFin3Threads = 96;    // three warps: one per slot of a gene group (kind 1), or three kind-2 tasks
constexpr int kFin3GeneChunk = 96;  // genes per kind-2 task
constexpr int kS3MaxPeers = 16;

struct S3Push {
    int n;                        // number of peer destinations (0: single GPU)
    double *dst[kS3MaxPeers];     // this rank's slot in the inbox of each peer (the own rank is not listed)
};

template <int K>
__global__ void __launch_bounds__(kFin3Threads) seg3_finish_kernel(int P, const double *__restrict__ theta,
                                                                     const double *__restrict__ PT,
                                                                     const double *__restrict__ Mg, double *__restrict__ stats,
                                                                     const S3Push push)
{
    constexpr int KK = K * K, K3 = KK * K, NB = (K + 7) / 8, NBC = (KK + 7) / 8;
    const int lane = threadIdx.x & 31, li = lane & 3, ri = lane >> 2, warp = threadIdx.x >> 5;
    const int n_groups = (P + 7) / 8;
    const int n_chunks = (P + kFin3GeneChunk - 1) / kFin3GeneChunk, n_kind2 = 2 * NBC * n_chunks;
    __shared__ double csm[2][NB * 2][32];
    if ((int)blockIdx.x < n_groups) {
        // kind 1: the CTA owns eight rows of Ntheta; warp w contracts slot w (both ratings: two batches of loads in a
        // row, as short a dependency chain as the per-slot tasks of the first version), warp 0 adds the three and stores
        const int slot = warp, g = blockIdx.x * 8 + ri;
        const bool gv = g < P;
        double c[NB][2];
#pragma unroll
        for (int i = 0; i < NB; ++i) c[i][0] = c[i][1] = 0.0;
        constexpr int NE = (KK + 3) / 4;          // k-steps over the cells of M
        constexpr int EB = NE < 32 ? NE : 32;     // loads in flight per batch
        for (int r = 0; r < 2; ++r) {
            const double *Mrow = Mg + ((int64_t)(slot * 2 + r) * P + (gv ? g : 0)) * KK;
            const double *Pr = PT + (int64_t)(slot * 2 + r) * K3;
            for (int eb = 0; eb < NE; eb += EB) {
                double av[EB];
#pragma unroll
                for (int q = 0; q < EB; ++q) {
                    const int e = (eb + q) * 4 + li;
                    av[q] = (gv && e < KK) ? __ldg(Mrow + e) : 0.0;
                }
#pragma unroll
                for (int q = 0; q < EB; ++q) {
                    const int e = (eb + q) * 4 + li;
                    if (eb + q < NE) {
#pragma unroll
                        for (int i = 0; i < NB; ++i) {
                            const int k = i * 8 + ri;
                            const double bv = (k < K && e < KK) ? __ldg(Pr + k * KK + e) : 0.0;
                            dmma884(c[i][0], c[i][1], av[q], bv);
                        }
                    }
                }
            }
        }
        if (warp > 0) {
#pragma unroll
            for (int i = 0; i < NB; ++i) {
                csm[warp - 1][2 * i][lane] = c[i][0];
                csm[warp - 1][2 * i + 1][lane] = c[i][1];
            }
        }
        __syncthreads();
        if (warp == 0) {
            // the eight rows of this CTA are 8 K consecutive doubles of Ntheta: put them together in shared memory and write
            // them out as one contiguous burst of 16-byte stores per destination (8-byte stores scattered over the lanes made
            // the remote copies 15 us slower than a separate bulk copy at n = 8: 420 k small NVLink writes per iteration)
            __shared__ __align__(16) double rowbuf[8 * K + 2];
            if (gv) {
#pragma unroll
                for (int i = 0; i < NB; ++i)
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int k = i * 8 + 2 * li + h;
                        if (k < K)
                            rowbuf[ri * K + k] = __ldg(theta + (int64_t)g * K + k) *
                                                 ((c[i][h] + csm[0][2 * i + h][lane]) + csm[1][2 * i + h][lane]);
                    }
            }
            __syncwarp();
            const int g0 = blockIdx.x * 8, ng = (P - g0 < 8) ? P - g0 : 8, nd = ng * K;   // doubles to write
            const int64_t at0 = (int64_t)g0 * K;                                            // multiple of 8: 16-byte aligned
            for (int q = -1; q < push.n; ++q) {
                double *dst = (q < 0 ? stats : push.dst[q]) + at0;
                for (int i = lane; i < nd / 2; i += 32) reinterpret_cast<double2 *>(dst)[i] = reinterpret_cast<const double2 *>(rowbuf)[i];
                if ((nd & 1) && lane == 0) dst[nd - 1] = rowbuf[nd - 1];
            }
        }
        return;
    }
    const int wt = ((int)blockIdx.x - n_groups) * (kFin3Threads / 32) + warp;
    if (wt < n_kind2) {
        const int w2 = wt;
        const int chunk = w2 / (2 * NBC), rem = w2 - chunk * (2 * NBC), r = rem / NBC, bcb = rem - r * NBC;
        const int g_lo = chunk * kFin3GeneChunk, g_hi = (g_lo + kFin3GeneChunk < P) ? g_lo + kFin3GeneChunk : P;
        const int bc = bcb * 8 + ri;
        const double *Mr = Mg + (int64_t)r * P * KK;  // slot 0
        double c[NB][2];
#pragma unroll
        for (int i = 0; i < NB; ++i) c[i][0] = c[i][1] = 0.0;
#pragma unroll 4
        for (int g0 = g_lo; g0 < g_hi; g0 += 4) {
            const int g = g0 + li;
            const bool gv = g < g_hi;
            const double bv = (gv && bc < KK) ? __ldg(Mr + (int64_t)g * KK + bc) : 0.0;
#pragma unroll
            for (int i = 0; i < NB; ++i) {
                const int al = i * 8 + ri;
                const double av = (gv && al < K) ? __ldg(theta + (int64_t)g * K + al) : 0.0;
                dmma884(c[i][0], c[i][1], av, bv);
            }
        }
        double *S = stats + stats_off_S(P, K) + (int64_t)r * K3;
#pragma unroll
        for (int i = 0; i < NB; ++i)
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int al = i * 8 + ri, cell = bcb * 8 + 2 * li + h;
                if (al < K && cell < KK) red_add_f64_nz3(S + (int64_t)al * KK + cell, c[i][h]);
            }
    }
}

// ---------------------------------------------------------------------------------------------
// workspace:  M[3][2][P][KK] | chunk counters | Z[2][P][ZK] | PT[3][2][K^3] | sbuf[n_rows]
// ---------------------------------------------------------------------------------------------
struct S3Layout {
    size_t off_M, off_cnt, off_Z, off_PT, off_T, off_s, total;  // in doubles
};
static S3Layout s3_layout(int P, int K, int64_t n_rows)
{
    const size_t KK = (size_t)K * K;
    S3Layout l;
    l.off_M = 0;
    l.off_cnt = 6 * (size_t)P * KK;
    l.off_Z = l.off_cnt + kS3CounterDoubles;
    l.off_PT = l.off_Z + 2 * (size_t)P * KK;
    l.off_PT = (l.off_PT + 1) / 2 * 2;
    l.off_T = l.off_PT + 6 * KK * K;
    l.off_T = (l.off_T + 15) / 16 * 16;                       // 128-byte aligned rows (the workspace base is)
    l.off_s = l.off_T + (size_t)P * ((K + 15) / 16 * 16);
    l.total = l.off_s + (size_t)(n_rows < 32 ? 32 : n_rows);
    return l;
}

size_t em_seg3_workspace_bytes(int P, int K, int64_t n_rows) { return s3_layout(P, K, n_rows).total * sizeof(double); }

// Per-kernel timing of one E-step (tip_seg3_timing): CUDA events recorded on the launching stream between the five
// stages.  Off by default (event records cannot be captured in a CUDA graph); bench.py switches it on around the
// un-graphed steps it uses for the roofline of the dominant kernel.
static bool g_s3_timing = false;
static cudaEvent_t g_s3_ev[6] = {};
static int s3_mark(int i, cudaStream_t st)
{
    if (!g_s3_timing) return 0;
    if (!g_s3_ev[0])
        for (int j = 0; j < 6; ++j) TIP_CHECK_CUDA(cudaEventCreate(&g_s3_ev[j]));
    TIP_CHECK_CUDA(cudaEventRecord(g_s3_ev[i], st));
    return 0;
}

template <int K, bool FIRST, bool CA>
static int s3_launch_pass_ca(const S3Args &a, bool plain, cudaStream_t st, int *grid_only)
{
    using C = S3<K>;
    constexpr size_t smem = C::BUF_BYTES * 2;
    static int blocks_per_sm = 0;
    if (blocks_per_sm == 0) {
        TIP_CHECK_CUDA(cudaFuncSetAttribute(seg3_pass_kernel<K, FIRST, CA>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        TIP_CHECK_CUDA(cudaFuncSetAttribute(seg3_pass_kernel<K, FIRST, CA>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                            cudaSharedmemCarveoutMaxShared));
        int nb = 0;
        TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, seg3_pass_kernel<K, FIRST, CA>, 32, smem));
        TIP_REQUIRE(nb >= 1, "seg3_pass_kernel<%d> does not fit on an SM (smem %zu)", K, smem);
        blocks_per_sm = nb;
    }
    const int64_t cap = (int64_t)sm_count() * blocks_per_sm;
    int grid = (int)(a.n_tiles < cap ? a.n_tiles : cap);
    if (grid < 1) grid = 1;
    if (grid_only != nullptr) {
        *grid_only = grid;
        return 0;
    }
    if (!g_s3_timing && !plain) {
        // pass B + C may start while pass A drains (see the header comment); it never waits for the grid dependency,
        // only for the s values it needs.  Pass A is launched the same way behind the prep kernel and DOES wait
        // (griddepcontrol.wait at its top): what it gains is its launch latency and CTA ramp
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid);
        cfg.blockDim = dim3(32);
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        TIP_CHECK_CUDA(cudaLaunchKernelEx(&cfg, seg3_pass_kernel<K, FIRST, CA>, a));
        return 0;
    }
    seg3_pass_kernel<K, FIRST, CA><<<grid, 32, smem, st>>>(a);
    TIP_CHECK_CUDA(cudaGetLastError());
    return 0;
}

// gather_l1: gather through L1 (cp.async.ca) instead of L2 only (.cg).  plain: launch without the programmatic dependency
// on the previous kernel.  grid_only != nullptr: only report the grid the launch would use (the prep kernel presets the
// schedule counters with it)
template <int K, bool FIRST>
static int s3_launch_pass(const S3Args &a, bool gather_l1, bool plain, cudaStream_t st, int *grid_only = nullptr)
{
    return gather_l1 ? s3_launch_pass_ca<K, FIRST, true>(a, plain, st, grid_only)
                     : s3_launch_pass_ca<K, FIRST, false>(a, plain, st, grid_only);
}

static S3Push g_s3_push = {};

template <int K>
static int launch_em_seg3_k(int P, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, const double *p,
                            double *stats, double *ws, bool gather_l1, cudaStream_t st)
{
    // the one-shot settings of this E-step (push targets of the finish kernel, event pass B + C has to wait for) are taken
    // - and cleared - before anything can fail, so that an error below cannot leave them behind for a later call
    const S3Push push = g_s3_push;
    g_s3_push.n = 0;
    const cudaEvent_t bc_wait = seg3_take_bc_wait();
    const S3Layout l = s3_layout(P, K, n_rows);
    const int KK = K * K;
    TIP_REQUIRE(n_rows / 32 < (1ll << 27), "tip_em_step: too many tiles in one shard for the slot-segmented kernels");
    S3Args a;
    a.P = P;
    a.rows = rows;
    a.tiles_per_order = (int)(n_rows / 32);
    a.n_tiles_r0 = (int)(n_rows_r0 / 32);
    a.theta = ws + l.off_T;
    a.Zg = ws + l.off_Z;
    a.sbuf = ws + l.off_s;
    a.Mg = ws + l.off_M;
    a.n_tiles = a.tiles_per_order;
    a.slot0 = 0;
    a.counter = reinterpret_cast<unsigned *>(ws + l.off_cnt);
    const int *sched = reinterpret_cast<const int *>(rows + 3 * n_rows);   // written by tip_order_rows behind the three orders
    a.sched = sched;
    a.n_sched = a.tiles_per_order;
    S3Args bc = a;
    bc.rows = rows + n_rows;
    bc.n_tiles = 2 * a.tiles_per_order;
    bc.slot0 = 1;
    bc.counter = reinterpret_cast<unsigned *>(ws + l.off_cnt) + kS3Groups * 32;
    bc.sched = sched + a.tiles_per_order;
    bc.n_sched = 2 * a.tiles_per_order;
    int grid_a = 0, grid_bc = 0;
    int rc = s3_launch_pass<K, true>(a, gather_l1, false, st, &grid_a);
    if (rc) return rc;
    rc = s3_launch_pass<K, false>(bc, gather_l1, false, st, &grid_bc);
    if (rc) return rc;
    // M starts every E-step from zero, sbuf from NaN ("not published"), the schedule counters behind the statically
    // assigned positions: all written by the prep kernel (no memset launches)
    if (s3_mark(0, st)) return -2;
    if (s3_mark(1, st)) return -2;
    {
        const size_t smem = sizeof(double) * ((K <= 20 ? 2 * KK * K : 0) + kPrepGenes * K);
        static bool attr = false;
        if (!attr && smem > 48 * 1024) {
            TIP_CHECK_CUDA(cudaFuncSetAttribute(seg3_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 128 * 1024));
            attr = true;
        }
        seg3_prep_kernel<<<(P + kPrepGenes - 1) / kPrepGenes, 256, smem, st>>>(
            P, K, theta, p, ws + l.off_Z, ws + l.off_PT, ws + l.off_T, S3<K>::TP, reinterpret_cast<double2 *>(ws + l.off_M),
            (int64_t)l.off_cnt / 2, reinterpret_cast<double2 *>(ws + l.off_s), (n_rows < 32 ? 32 : n_rows) / 2, a.counter,
            2u * (unsigned)grid_a, bc.counter, 2u * (unsigned)grid_bc);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    if (s3_mark(2, st)) return -2;
    rc = s3_launch_pass<K, true>(a, gather_l1, false, st);
    if (rc) return rc;
    if (s3_mark(3, st)) return -2;
    // (host-buffer entry) orders b and c are still being produced on another stream: a plain launch behind the wait
    // (no programmatic dependency on pass A)
    if (bc_wait) TIP_CHECK_CUDA(cudaStreamWaitEvent(st, bc_wait, 0));
    rc = s3_launch_pass<K, false>(bc, gather_l1, bc_wait != nullptr, st);
    if (rc) return rc;
    if (s3_mark(4, st)) return -2;
    {
        constexpr int NBC = (K * K + 7) / 8;
        const int n_kind2 = 2 * NBC * ((P + kFin3GeneChunk - 1) / kFin3GeneChunk);
        const int wpc = kFin3Threads / 32;
        seg3_finish_kernel<K><<<(P + 7) / 8 + (n_kind2 + wpc - 1) / wpc, kFin3Threads, 0, st>>>(P, theta, ws + l.off_PT, ws + l.off_M,
                                                                                             stats, push);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    if (s3_mark(5, st)) return -2;
    return 0;
}

// rows: order a | order b | order c, n_rows rows each, then the two schedules (tip_order_rows); stats zeroed by the caller
int launch_em_seg3(int P, int K, const int4 *rows, int64_t n_rows, int64_t n_rows_r0, const double *theta, const double *p,
                   double *stats, double *ws, bool gather_l1, cudaStream_t st)
{
    switch (K) {
#define TIP_S3_CASE(k) \
    case k: return launch_em_seg3_k<k>(P, rows, n_rows, n_rows_r0, theta, p, stats, ws, gather_l1, st);
        TIP_S3_CASE(1) TIP_S3_CASE(2) TIP_S3_CASE(3) TIP_S3_CASE(4) TIP_S3_CASE(5) TIP_S3_CASE(6) TIP_S3_CASE(7) TIP_S3_CASE(8)
        TIP_S3_CASE(9) TIP_S3_CASE(10) TIP_S3_CASE(11) TIP_S3_CASE(12) TIP_S3_CASE(13) TIP_S3_CASE(14) TIP_S3_CASE(15)
        TIP_S3_CASE(16) TIP_S3_CASE(17) TIP_S3_CASE(18) TIP_S3_CASE(19) TIP_S3_CASE(20) TIP_S3_CASE(21) TIP_S3_CASE(22)
        TIP_S3_CASE(23) TIP_S3_CASE(24) TIP_S3_CASE(25) TIP_S3_CASE(26) TIP_S3_CASE(27) TIP_S3_CASE(28) TIP_S3_CASE(29)
        TIP_S3_CASE(30) TIP_S3_CASE(31) TIP_S3_CASE(32)
#undef TIP_S3_CASE
        default: set_error("launch_em_seg3: K = %d out of range", K); return -1;
    }
}

// ---------------------------------------------------------------------------------------------
// tip_order_rows: the order-b and order-c copies of the packed rows
// ---------------------------------------------------------------------------------------------
constexpr unsigned kOrderPadBit = 1u << 20, kOrderRatingShift = 21;

__global__ void order_keys_kernel(const int4 *__restrict__ rows, int64_t n_rows, int64_t n_rows_r0, int slot,
                                  unsigned *__restrict__ keys, int32_t *__restrict__ vals)
{
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x) {
        const int4 v = rows[i];
        const unsigned r = i >= n_rows_r0 ? 1u : 0u;
        const unsigned g = (unsigned)(slot == 1 ? v.y : v.z);
        keys[i] = (r << kOrderRatingShift) | (row_count(v.w) > 0 ? g : kOrderPadBit);
        vals[i] = (int32_t)i;
    }
}

__global__ void order_emit_kernel(const int4 *__restrict__ rows, const int32_t *__restrict__ vals, int64_t n_rows, int slot,
                                  int4 *__restrict__ out)
{
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_rows; j += (int64_t)gridDim.x * blockDim.x) {
        const int src = vals[j];
        const int4 v = rows[src];
        int4 o = make_int4(0, 0, 0, -1);
        if (row_count(v.w) > 0) o = slot == 1 ? make_int4(v.y, v.x, v.z, src) : make_int4(v.z, v.x, v.y, src);
        out[j] = o;
    }
}

// ---- counting sort by (rating, gene) for callers that know P (tip_order_rows_by_gene, the host-buffer entry): the keys have
// only 2 (P + 1) values, so a histogram in shared memory, one scan and one scatter with warp-aggregated cursors replace the
// three-pass radix sort (15 us instead of 78 us per slot at 800 k rows).  NOT stable: the order of the links inside a
// gene's run is whatever the cursors hand out - the statistics are sums over the run, so only their rounding moves.
constexpr int kCountMaxBins = 12288;   // 48 KB of shared-memory counters

__device__ __forceinline__ int order_bucket(const int4 &v, bool r1, int slot, int P)
{
    const int g = slot == 1 ? v.y : v.z;
    return (r1 ? P + 1 : 0) + (row_count(v.w) > 0 ? g : P);
}

__global__ void __launch_bounds__(256) order_hist_kernel(const int4 *__restrict__ rows, int64_t n_rows, int64_t n_rows_r0, int slot,
                                                         int P, int nb, unsigned *__restrict__ hist)
{
    extern __shared__ unsigned sh_cnt[];
    for (int b = threadIdx.x; b < nb; b += blockDim.x) sh_cnt[b] = 0u;
    __syncthreads();
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_rows; i += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(&sh_cnt[order_bucket(rows[i], i >= n_rows_r0, slot, P)], 1u);
    __syncthreads();
    for (int b = threadIdx.x; b < nb; b += blockDim.x)
        if (sh_cnt[b]) atomicAdd(hist + b, sh_cnt[b]);
}

// exclusive prefix sum of nb <= kCountMaxBins counters, in place, one CTA of 1024 threads
__global__ void __launch_bounds__(1024) order_scan_kernel(unsigned *__restrict__ hist, int nb)
{
    __shared__ unsigned part[1024];
    const int per = (nb + 1023) / 1024, lo = threadIdx.x * per, hi = (lo + per < nb) ? lo + per : nb;
    unsigned s = 0;
    for (int b = lo; b < hi; ++b) s += hist[b];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const unsigned v = threadIdx.x >= o ? part[threadIdx.x - o] : 0u;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned run = threadIdx.x ? part[threadIdx.x - 1] : 0u;
    for (int b = lo; b < hi; ++b) {
        const unsigned c = hist[b];
        hist[b] = run;
        run += c;
    }
}

__global__ void __launch_bounds__(256) order_scatter_kernel(const int4 *__restrict__ rows, int64_t n_rows, int64_t n_rows_r0,
                                                            int slot, int P, unsigned *__restrict__ cursor, int4 *__restrict__ out)
{
    const int lane = threadIdx.x & 31;
    const int64_t n32 = (n_rows + 31) / 32 * 32;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n32; i += (int64_t)gridDim.x * blockDim.x) {
        const bool in = i < n_rows;
        const int4 v = in ? rows[i] : make_int4(0, 0, 0, 0);
        const int b = in ? order_bucket(v, i >= n_rows_r0, slot, P) : -1;
        const unsigned peers = __match_any_sync(0xffffffffu, b);
        const int leader = __ffs(peers) - 1, rank = __popc(peers & ((1u << lane) - 1u));
        unsigned base = 0;
        if (in && lane == leader) base = atomicAdd(cursor + b, (unsigned)__popc(peers));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (in) {
            int4 o = make_int4(0, 0, 0, -1);
            if (row_count(v.w) > 0) o = slot == 1 ? make_int4(v.y, v.x, v.z, (int)i) : make_int4(v.z, v.x, v.y, (int)i);
            out[base + rank] = o;
        }
    }
}

// ---- the schedule of a launch (see the header comment).  One warp per group of kSchedGroup consecutive tiles of the
// launch's tile sequence (order a; or order b followed by order c).  A tile's cost = 1 + run ends inside it, where a run
// ends wherever (slot, rating, gene) changes - exactly what the pass kernel compares.  Every group owns kSchedGroup
// slots of the (key, entry) arrays: a light group fills one (the whole group as one chunk), a group with a heavy tile,
// or one of the groups set aside for the end of the list, fills one per tile; unused slots stay (0, 0).  The arrays are
// then sorted by descending key: heavy tiles first (longest processing time first), chunks by cost, single tiles last.
constexpr int kSchedGroup = 4;        // tiles per chunk (an entry holds the count in 3 bits)
constexpr int kSchedHeavy = 6;        // a tile with at least this many run ends is scheduled on its own
constexpr int kSchedTailTiles = 8 * 148 * 16;   // about this many tiles are handed out one by one at the end

__global__ void __launch_bounds__(128) sched_build_kernel(const int4 *__restrict__ rows, int n_tiles, int tiles_per_order,
                                                          int n_tiles_r0, int tail_stride, unsigned *__restrict__ keys,
                                                          int *__restrict__ vals)
{
    const int lane = threadIdx.x & 31;
    const int n_groups = (n_tiles + kSchedGroup - 1) / kSchedGroup;
    for (int g = blockIdx.x * 4 + (threadIdx.x >> 5); g < n_groups; g += gridDim.x * 4) {
        int cost[kSchedGroup];
        int heavy = 0, total = 0, nt = 0;
#pragma unroll
        for (int j = 0; j < kSchedGroup; ++j) {
            const int t = g * kSchedGroup + j;
            cost[j] = 0;
            if (t < n_tiles) {
                auto key_of = [&](int64_t row) -> long long {
                    const int tt = (int)(row >> 5);
                    const int so = tt >= tiles_per_order ? 1 : 0, tl = tt - (so ? tiles_per_order : 0);
                    return ((long long)(so * 2 + (tl >= n_tiles_r0 ? 1 : 0)) << 32) | (unsigned)rows[row].x;
                };
                const int64_t row = (int64_t)t * 32 + lane;
                const long long k = key_of(row);
                const long long kp = row > 0 ? key_of(row - 1) : k;
                const int b = __popc(__ballot_sync(0xffffffffu, k != kp));
                cost[j] = 1 + b;
                total += b;
                heavy |= b >= kSchedHeavy;
                ++nt;
            }
        }
        if (lane == 0) {
            const bool tail = (g % tail_stride) == tail_stride - 1;
#pragma unroll
            for (int j = 0; j < kSchedGroup; ++j) {
                unsigned key = 0;
                int val = 0;
                const int t = g * kSchedGroup + j;
                if (heavy) {
                    if (j < nt) { key = 128u + (unsigned)cost[j]; val = (t << 3) | 1; }
                } else if (tail) {
                    if (j < nt) { key = (unsigned)cost[j]; val = (t << 3) | 1; }
                } else if (j == 0) {
                    key = 64u + (unsigned)(1 + total);
                    val = ((g * kSchedGroup) << 3) | nt;
                }
                keys[g * kSchedGroup + j] = key;
                vals[g * kSchedGroup + j] = val;
            }
        }
    }
}

static size_t order_layout(int64_t n, size_t *o_ki, size_t *o_ko, size_t *o_vi, size_t *o_vo, size_t *o_cub, size_t *cub_bytes)
{
    size_t cb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, cb, (const unsigned *)nullptr, (unsigned *)nullptr, (const int32_t *)nullptr,
                                    (int32_t *)nullptr, n, 0, 22, (cudaStream_t)0);
    auto al = [](size_t x) { return (x + 255) / 256 * 256; };
    size_t off = 0;
    *o_ki = off; off += al((size_t)n * 4);
    *o_ko = off; off += al((size_t)n * 4);
    *o_vi = off; off += al((size_t)n * 4);
    *o_vo = off; off += al((size_t)n * 4);
    *o_cub = off; off += al(cb);
    *cub_bytes = cb;
    return off + 256;
}

}  // namespace tip

using namespace tip;

extern "C" int tip_em_set_push_targets(void *const *h_inbox_ptrs, int rank, int nranks, int64_t n_pad)
{
    TIP_REQUIRE(nranks >= 1 && nranks <= kS3MaxPeers && rank >= 0 && rank < nranks && (nranks == 1 || h_inbox_ptrs != nullptr) &&
                    n_pad >= 0,
                "tip_em_set_push_targets: bad arguments (nranks <= %d)", kS3MaxPeers);
    g_s3_push.n = 0;
    for (int q = 0; q < nranks; ++q)
        if (q != rank) g_s3_push.dst[g_s3_push.n++] = reinterpret_cast<double *>(h_inbox_ptrs[q]) + (int64_t)rank * n_pad;
    return 0;
}

extern "C" int tip_seg3_timing(int enable)
{
    g_s3_timing = enable != 0;
    return 0;
}

extern "C" int tip_seg3_last_timing(float *h_ms5)
{
    TIP_REQUIRE(h_ms5 != nullptr && g_s3_ev[0] != nullptr, "tip_seg3_last_timing: no timed slot-segmented E-step has run");
    TIP_CHECK_CUDA(cudaEventSynchronize(g_s3_ev[5]));
    for (int i = 0; i < 5; ++i) TIP_CHECK_CUDA(cudaEventElapsedTime(h_ms5 + i, g_s3_ev[i], g_s3_ev[i + 1]));
    return 0;
}

extern "C" int tip_order_rows_workspace_bytes(int64_t n_rows, size_t *bytes)
{
    TIP_REQUIRE(n_rows >= 0 && bytes != nullptr, "tip_order_rows_workspace_bytes: bad arguments");
    size_t a, b, c, d, e, f;
    *bytes = order_layout(n_rows < 32 ? 32 : n_rows, &a, &b, &c, &d, &e, &f);
    return 0;
}

extern "C" int tip_order_rows(const void *d_rows, int64_t n_rows, int64_t n_rows_r0, void *d_ws, size_t ws_bytes,
                              void *d_rows_bc, void *stream)
{
    return order_rows_parts(d_rows, n_rows, n_rows_r0, d_ws, ws_bytes, d_rows_bc, reinterpret_cast<cudaStream_t>(stream), 3, 0);
}

extern "C" int tip_order_rows_by_gene(const void *d_rows, int64_t n_rows, int64_t n_rows_r0, int P, void *d_ws, size_t ws_bytes,
                                      void *d_rows_bc, void *stream)
{
    TIP_REQUIRE(P > 0, "tip_order_rows_by_gene: P must be positive");
    return order_rows_parts(d_rows, n_rows, n_rows_r0, d_ws, ws_bytes, d_rows_bc, reinterpret_cast<cudaStream_t>(stream), 3, P);
}

namespace tip {
// parts: 1 = the schedule of the order-a launch (needs the packed rows only), 2 = orders b and c and their schedule;
// the host-buffer entry runs the two parts on different streams (each with its own workspace), so that pass A starts
// while the rows are still being sorted for passes B and C
int order_rows_parts(const void *d_rows, int64_t n_rows, int64_t n_rows_r0, void *d_ws, size_t ws_bytes, void *d_rows_bc,
                     cudaStream_t st, int parts, int P)
{
    TIP_REQUIRE(n_rows >= 0 && n_rows % 32 == 0 && n_rows_r0 >= 0 && n_rows_r0 <= n_rows && n_rows < (1ll << 31),
                "tip_order_rows: n_rows (%lld) must be a multiple of 32 below 2^31", (long long)n_rows);
    if (n_rows == 0) return 0;
    TIP_REQUIRE(d_rows && d_rows_bc && d_ws, "tip_order_rows: null pointer");
    size_t o_ki, o_ko, o_vi, o_vo, o_cub, cub_bytes;
    const size_t need = order_layout(n_rows, &o_ki, &o_ko, &o_vi, &o_vo, &o_cub, &cub_bytes);
    TIP_REQUIRE(ws_bytes >= need, "tip_order_rows: workspace too small (%zu < %zu)", ws_bytes, need);
    char *base = reinterpret_cast<char *>((reinterpret_cast<uintptr_t>(d_ws) + 255) / 256 * 256);
    unsigned *ki = reinterpret_cast<unsigned *>(base + o_ki), *ko = reinterpret_cast<unsigned *>(base + o_ko);
    int32_t *vi = reinterpret_cast<int32_t *>(base + o_vi), *vo = reinterpret_cast<int32_t *>(base + o_vo);
    const int4 *rows = reinterpret_cast<const int4 *>(d_rows);
    int4 *out = reinterpret_cast<int4 *>(d_rows_bc);
    const int64_t want = (n_rows + 255) / 256;
    const int grid = (int)(want < (int64_t)sm_count() * 8 ? want : (int64_t)sm_count() * 8);
    // P known and the (rating, gene) keys few enough for shared-memory counters: counting sort (not stable)
    const int nb = 2 * (P + 1);
    const bool counting = P > 0 && nb <= kCountMaxBins && nb <= n_rows;
    for (int slot = 1; slot <= 2 && (parts & 2) && counting; ++slot) {
        static bool attr = false;
        if (!attr) {
            TIP_CHECK_CUDA(cudaFuncSetAttribute(order_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kCountMaxBins * 4));
            attr = true;
        }
        TIP_CHECK_CUDA(cudaMemsetAsync(ki, 0, sizeof(unsigned) * (size_t)nb, st));
        const int hgrid = grid < sm_count() * 2 ? grid : sm_count() * 2;
        order_hist_kernel<<<hgrid, 256, sizeof(unsigned) * (size_t)nb, st>>>(rows, n_rows, n_rows_r0, slot, P, nb, ki);
        TIP_CHECK_CUDA(cudaGetLastError());
        order_scan_kernel<<<1, 1024, 0, st>>>(ki, nb);
        TIP_CHECK_CUDA(cudaGetLastError());
        order_scatter_kernel<<<grid, 256, 0, st>>>(rows, n_rows, n_rows_r0, slot, P, ki, out + (slot - 1) * n_rows);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    for (int slot = 1; slot <= 2 && (parts & 2) && !counting; ++slot) {
        order_keys_kernel<<<grid, 256, 0, st>>>(rows, n_rows, n_rows_r0, slot, ki, vi);
        TIP_CHECK_CUDA(cudaGetLastError());
        size_t cb = cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairs(base + o_cub, cb, ki, ko, vi, vo, n_rows, 0, 22, st));
        order_emit_kernel<<<grid, 256, 0, st>>>(rows, vo, n_rows, slot, out + (slot - 1) * n_rows);
        TIP_CHECK_CUDA(cudaGetLastError());
    }
    // the schedules of the two launches, behind the orders: [T] for order a, [2T] for orders b + c
    const int T = (int)(n_rows / 32), r0 = (int)(n_rows_r0 / 32);
    int *sched = reinterpret_cast<int *>(out + 2 * n_rows);
    for (int launch = 0; launch < 2; ++launch) {
        if (!(parts & (1 << launch))) continue;
        const int nt = launch == 0 ? T : 2 * T;
        const int n_groups = (nt + kSchedGroup - 1) / kSchedGroup, n_slots = n_groups * kSchedGroup;
        int tail_stride = n_groups / (kSchedTailTiles / kSchedGroup);
        if (tail_stride < 4) tail_stride = 4;
        const int want_b = (n_groups + 3) / 4;
        sched_build_kernel<<<want_b < sm_count() * 16 ? want_b : sm_count() * 16, 128, 0, st>>>(
            launch == 0 ? rows : out, nt, T, r0, tail_stride, ki, vi);
        TIP_CHECK_CUDA(cudaGetLastError());
        size_t cb = cub_bytes;
        TIP_CHECK_CUDA(cub::DeviceRadixSort::SortPairsDescending(base + o_cub, cb, ki, ko, vi, vo, n_slots, 0, 8, st));
        // the first nt sorted entries hold every real chunk (there are at most nt of them); zeros follow
        TIP_CHECK_CUDA(cudaMemcpyAsync(sched + (launch == 0 ? 0 : T), vo, sizeof(int) * (size_t)nt, cudaMemcpyDeviceToDevice, st));
    }
    return 0;
}

static cudaEvent_t g_s3_bc_wait = nullptr;
// the next slot-segmented E-step waits for `ev` between pass A and pass B + C (one-shot)
void seg3_wait_before_bc(cudaEvent_t ev) { g_s3_bc_wait = ev; }
cudaEvent_t seg3_take_bc_wait()
{
    cudaEvent_t ev = g_s3_bc_wait;
    g_s3_bc_wait = nullptr;
    return ev;
}
}  // namespace tip

extern "C" int64_t tip_order_rows_out_bytes(int64_t n_rows)
{
    if (n_rows < 0) return -1;
    return 2 * n_rows * 16 + 3 * (n_rows / 32) * 4 + 16;
}
