/* tip.h - C ABI of libtip.so: the B200 (sm_100a) implementation of the MMSBM EM hot path of
 * AleixMT/TrigenicInteractionPredictor.
 *
 * The reference has no FFI of its own: the hot path is the Python class `Model` in
 * src/TrigenicInteractionPredictor.py (TIP.py).  Each entry point below replaces the arithmetic
 * of one `Model` method; the Python `Model` in trigenicinteractionpredictor_b200/ binds them
 * with ctypes (see INTEGRATION.md for the stub a reference maintainer would add).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error; tip_last_error() gives the message
 *     (thread-local).  Nothing here ever falls back to the CPU.
 *   - pointers named d_* are DEVICE pointers owned by the caller (PyTorch tensors on the Python
 *     side); h_* are HOST pointers.  No ownership is transferred, no device memory is allocated
 *     by the d_* functions: scratch is passed in (`*_workspace_bytes` tells how much).
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream).  All d_* functions are
 *     asynchronous on that stream and CUDA-graph capturable unless stated otherwise.
 *   - doubles are IEEE fp64.  Layouts follow the reference: theta[P][K], p[K][K][K][2] row-major.
 *
 * Link rows ("packed rows"): one int4 per (link, rating) with a non-zero count:
 *     {a, b, c, (count << 1) | rating}   a,b,c = gene ids in the reference's key slot order
 * (decimal-string sort, TIP.py:353).  Rows are ordered rating 0 first, then rating 1, each block
 * sorted by slot-a gene and padded with zero-count rows to a multiple of 32, so that every warp
 * tile of 32 rows has one rating.  16 bytes per link-update is the algorithmic HBM traffic.
 *
 * Statistics buffer ("stats"), tip_stats_len(P,K) doubles - the quantity that is summed across
 * link shards (one NCCL allreduce per EM iteration):
 *     [0, P*K)                 Ntheta[g][k]   = sum over links/slots of omega * n     (TIP.py:1009-1011)
 *     [P*K, P*K + 2*K^3)       S[r][a][b][c]  = sum_l n_lr/d_lr * th_a th_b th_c     (npr = p * S, TIP.py:1012)
 *     [P*K + 2*K^3]            sum_l n_lr * log(d_lr) of the parameters the step STARTED from
 *                              (only with TIP_EM_WITH_LOGLIK or on the any-K path; 0 otherwise)
 */
#ifndef TIP_H_
#define TIP_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TIP_ABI_VERSION 1
#define TIP_EPS 1e-10 /* TIP.py:88 */
#define TIP_R 2       /* TIP.py:79 */
#define TIP_MAX_K 32

/* flags for tip_em_step */
#define TIP_EM_DEFAULT 0u
#define TIP_EM_FORCE_GENERIC 1u /* use the any-K kernels even where a K-specialised kernel exists */
#define TIP_EM_FP32_COMPUTE 2u  /* K <= 10: the two K^3 contractions of the E-step in fp32 (FFMA), everything that
                                   is accumulated across links in fp64; results within 1e-5 of the fp64 mode */
#define TIP_EM_GENE_SEGMENTED 8u /* K >= 5, fp64: contract p with theta once per (gene, rating) so that a link costs
                                   2K^2 instead of 2K^3 FMA (same results to rounding); the kernel is then bound by
                                   the theta gather and the reductions, not by the FMA pipe.  K = 17..32 always
                                   runs this formulation (its only specialised kernel) */
#define TIP_EM_SLOT_SEGMENTED 32u /* any K, fp64: all three theta statistics and the p statistic accumulated per run of
                                   equal gene, in three sort orders of the links (4K^2 FMA per link, no per-link atomics:
                                   hub genes cost nothing extra).  d_rows then holds the three orders back to back, n_rows
                                   rows each, and the tile schedules behind them: the packed rows, then tip_order_rows'
                                   output (tip_order_rows_out_bytes) */
#define TIP_EM_GATHER_L1 64u     /* with TIP_EM_SLOT_SEGMENTED: gather the theta rows through L1 (cp.async.ca) instead of L2
                                   only.  For hub-shaped links (a few genes in most triplets): the hub rows then stay in
                                   L1 instead of being requested from a handful of L2 slices by every SM (measured 0.31 ->
                                   0.24 ms at 800k Kuzmin-shaped links); costs ~4 % on uniform links */
#define TIP_EM_WITH_LOGLIK 4u   /* also accumulate the log-likelihood by-product (last stats slot); off by
                                   default because the log costs ~2 % of a K=10 step and the training loop only
                                   needs the likelihood every `fcheck` iterations (tip_loglik) */

/* flag for tip_em_iterations_host only: h_rows holds the 8-byte rows of tip_rows_compact_host */
#define TIP_ROWS_COMPACT8 16u

int tip_abi_version(void);
const char *tip_last_error(void);

/* number of doubles in the statistics buffer */
int64_t tip_stats_len(int P, int K);

/* ---- link digestion on the device (replaces the per-iteration key parsing of TIP.py:987-989) ----
 * in : d_g1,d_g2,d_g3 [L] gene ids in key slot order; d_n0,d_n1 [L] counts per rating (TIP.py:361-368)
 * out: d_rows [>= tip_rows_capacity(L)] packed rows; *h_n_rows = padded row count (multiple of 32);
 *      h_part[0..2] = {rows in the rating-0 block (padded), rows in the rating-1 block (padded),
 *                      real (unpadded) rows};  d_deg [P] int32 = distinct links touching each gene
 *      (the `counter` of TIP.py:986-994).  d_deg may be NULL.
 * Synchronises the stream (it returns counts to the host); digestion time, not iteration time. */
int64_t tip_rows_capacity(int64_t L);
int tip_pack_rows_workspace_bytes(int64_t L, size_t *bytes);
int tip_pack_rows(const int32_t *d_g1, const int32_t *d_g2, const int32_t *d_g3, const int32_t *d_n0,
                  const int32_t *d_n1, int64_t L, int P, void *d_ws, size_t ws_bytes, void *d_rows,
                  int64_t *h_n_rows, int64_t *h_part, int32_t *d_deg, void *stream);

/* ---- the slot-b and slot-c orders of the packed rows (TIP_EM_SLOT_SEGMENTED) ----
 * in : d_rows [n_rows] packed rows of tip_pack_rows (ordered by rating, then slot-a gene)
 * out: d_rows_bc [2 * n_rows]: the same links ordered by (rating, slot-b gene), then by (rating, slot-c gene); a row is
 *      {gene of the ordering slot, slot-a gene (or slot-a for c), the remaining gene, position of the link in d_rows},
 *      i.e. {b, a, c, pos} and {c, a, b, pos}; padding rows are {0, 0, 0, -1}.  The rating blocks keep their sizes, so
 *      n_rows and n_rows_r0 describe all three orders.  Stable: links of one gene stay in slot-a order.
 *      Behind the two orders, 3 * n_rows / 32 int32: the SCHEDULES of the two E-step launches (order a; orders b + c) -
 *      chunks of up to four consecutive 32-row tiles, (first tile << 3) | tiles, sorted by descending cost (a tile costs
 *      1 + the runs of equal gene that end in it; tiles with many runs stand alone and come first, single tiles close
 *      the list), 0-terminated.  Hub-shaped links put tiles with 20-30 one-link runs next to thousands of tiles inside
 *      one run; the schedule is what keeps every SM busy to the end of a launch.
 *      d_rows_bc must hold tip_order_rows_out_bytes(n_rows) bytes and MUST directly follow the packed rows in memory
 *      (d_rows_bc == d_rows + n_rows rows): tip_em_step takes one pointer to all of it.
 * Asynchronous on `stream`; digestion time, not iteration time. */
int tip_order_rows_workspace_bytes(int64_t n_rows, size_t *bytes);
int64_t tip_order_rows_out_bytes(int64_t n_rows);
/* The same orders and schedules for callers that know P: with few enough (rating, gene) keys (2 (P + 1) <= 12288 and
 * <= n_rows) a counting sort - shared-memory histogram, scan, scatter with warp-aggregated cursors - replaces the radix
 * sort (5x faster at 800k rows).  NOT stable: the order of the links inside a gene's run is unspecified (the statistics
 * are sums over the run; only their rounding moves).  Falls back to tip_order_rows' sort otherwise.  Same workspace and
 * output sizes.  Used by tip_em_iterations_host, where the ordering is inside the timed region. */
int tip_order_rows_by_gene(const void *d_rows, int64_t n_rows, int64_t n_rows_r0, int P, void *d_ws, size_t ws_bytes,
                           void *d_rows_bc, void *stream);
int tip_order_rows(const void *d_rows, int64_t n_rows, int64_t n_rows_r0, void *d_ws, size_t ws_bytes, void *d_rows_bc,
                   void *stream);

/* ---- Model.make_iteration, E-step half (TIP.py:987-1012) ----
 * Zeroes d_stats, then accumulates the statistics of `n_rows` packed rows under (d_theta, d_p).
 * n_rows_r0 = rows in the rating-0 block (h_part[0] of tip_pack_rows); both are multiples of 32.
 * d_ws: tip_em_workspace_bytes() bytes of scratch (per-gene M matrices for K = 5..16, per-row s on the any-K
 *       path; 0 for K <= 4, where it may be NULL). */
int tip_em_workspace_bytes(int P, int K, int64_t n_rows, unsigned flags, size_t *bytes);
int tip_em_step(int P, int K, const void *d_rows, int64_t n_rows, int64_t n_rows_r0, const double *d_theta,
                const double *d_p, double *d_stats, void *d_ws, size_t ws_bytes, unsigned flags, void *stream);

/* ---- E-step over rows that are still in HOST memory (the same statistics as tip_em_step) ----
 * h_rows: pinned host rows, 16 bytes each (row_flags = 0) or 8 bytes each (row_flags = TIP_ROWS_COMPACT8).
 * d_rows_dev: n_rows * 16 (or * 8) bytes of device memory that receives them.  The function fills d_rows_dev with a
 * sentinel and queues ONE host-to-device copy on `copy_stream`; the fused kernel, launched on `stream`, polls the
 * rows of each tile until they have landed, so the E-step follows the DMA front instead of waiting for the copy
 * (one launch, no chunking).  Queue small parameter copies BEFORE this call: the host-to-device engine serves all
 * streams in submission order.  d_err: 256 bytes of device memory, zero on entry; word 0 is set to 1 when a tile waited
 * more than 5 s (the statistics are then incomplete) and to 2 when the words the kernel consumed do not add up to the
 * words that finally landed (checked by a verification kernel once the copy is complete: a kernel racing a DMA has no
 * memory-model guarantee of seeing whole words, so the race is PROVEN harmless per call) - in both cases discard the
 * statistics and call tip_em_step on d_rows_dev, which then holds the rows.  Plain fp64 kernels for K <= 10 only (-1 otherwise: copy the rows
 * and call tip_em_step).  `stream` and `copy_stream` must differ.  Not capturable in a CUDA graph. */
int tip_em_step_host_rows(int P, int K, const void *h_rows, int64_t n_rows, int64_t n_rows_r0, unsigned row_flags,
                          void *d_rows_dev, const double *d_theta, const double *d_p, double *d_stats, void *d_ws,
                          size_t ws_bytes, unsigned *d_err, void *stream, void *copy_stream);

/* ---- Model.make_iteration, M-step half (TIP.py:1016-1043) ----
 * theta[g][k] = Ntheta[g][k] / deg[g];  npr = p*S;  p = npr / (eps + npr0 + npr1).  In place on d_p.
 * Genes with deg == 0 produce inf/nan like a float division would; the Python Model raises
 * ZeroDivisionError before launching, as TIP.py:1018 does. */
int tip_normalise(int P, int K, const double *d_stats, const int32_t *d_deg, double *d_theta, double *d_p,
                  void *stream);

/* ---- Model.compute_likelihood (TIP.py:952-974) ----
 * *d_out = sum_rows count * log(eps + sum_abc th th th p_r).  Deterministic summation order.
 * Rows as packed by tip_pack_rows (n_rows_r0 = h_part[0]); flags: TIP_EM_FORCE_GENERIC selects the any-K kernel.
 * d_ws: tip_loglik_workspace_bytes(P, K) bytes of scratch (per-CTA partials; for K > 10 also the per-gene
 *       contraction Z = theta . p of the gene-segmented formulation). */
size_t tip_loglik_workspace_bytes(int P, int K);
int tip_loglik(int P, int K, const void *d_rows, int64_t n_rows, int64_t n_rows_r0, const double *d_theta,
               const double *d_p, double *d_out, void *d_ws, unsigned flags, void *stream);

/* ---- Model.do_prediction over a whole test set (TIP.py:530-547, 564-565) ----
 * d_scores[t] = sum_abc th[g1[t]][a] th[g2[t]][b] th[g3[t]][c] p[a][b][c][1]   (no eps). */
int tip_score(int P, int K, const int32_t *d_g1, const int32_t *d_g2, const int32_t *d_g3, int64_t T,
              const double *d_theta, const double *d_p, double *d_scores, void *stream);

/* ---- Model.calculate_metrics (TIP.py:583-637), integer part ----
 * d_out[8] int64 = {auc_wins (#(pos,neg) with score_pos > score_neg, strict), n_pos, n_neg,
 *                   tp, fp, fn, tn, bit pattern of cut_value}
 * positives_number = int(positives_fraction * T) computed by the caller (TIP.py:592); cut_value is
 * the positives_number-th largest score, or 0.0 when positives_number >= T (TIP.py:595-599).
 * The ratios are formed by the caller in Python so ZeroDivisionError behaves as in the reference. */
int tip_metrics_workspace_bytes(int64_t T, size_t *bytes);
int tip_metrics(const double *d_scores, const int32_t *d_labels, int64_t T, int64_t positives_number,
                void *d_ws, size_t ws_bytes, int64_t *d_out, void *stream);

/* ---- Model.calculate_test_set_results, the ordering (TIP.py:568-569: results.sort(); results.reverse()) ----
 * d_sorted[T] = the scores in descending order, d_order[T] = the test-set index of each (stable: equal scores keep their
 * test order; the caller puts runs of EQUAL scores into the reference's (key string, label) order on the host - only
 * those need the strings). */
int tip_sort_scores_workspace_bytes(int64_t T, size_t *bytes);
int tip_sort_scores(const double *d_scores, int64_t T, void *d_ws, size_t ws_bytes, int32_t *d_order, double *d_sorted,
                    void *stream);

/* ---- prediction: the N highest-scoring unseen triplets of a candidate gene list, exhaustively ----
 * Candidates are all triplets of distinct genes of d_cand[n_cand] (gene ids, distinct, in decimal-string order: position =
 * rank).  A triplet's slots are its ranks in ascending order, which is the reference's key slot order (TIP.py:353); its
 * score is do_prediction (TIP.py:530-547, rating 1, no eps) averaged over the S parameter sets
 * d_theta[S][P][K], d_p[S][K][K][K][2].  d_known[n_known]: sorted, distinct packed rank triples
 * (ra << 42) | (rb << 21) | rc, ra < rb < rc, of triplets never to return (the known links among the candidates).
 * Out: the first min(N, C(n_cand, 3) - n_known) triplets in the order (score descending, (ra, rb, rc) ascending), exact
 * under any ties: d_out_ids[N][3] gene ids in slot order, d_out_scores[N], *h_n_out rows.
 * Every score is recomputed in each pass on the fp64 tensor path (C(n, 3) * 2 S K flop per pass, no per-triplet storage);
 * only scores above a threshold leave registers, and the host narrows the threshold between passes.  Synchronises the
 * stream (the host decides how many passes to run); not capturable in a CUDA graph.  Limits: n_cand <= 2^21, S * K <= 384,
 * N < 2^28.  Precondition: finite, non-negative parameters.  d_ws: tip_top_triplets_workspace_bytes() bytes. */
int tip_top_triplets_workspace_bytes(int n_cand, int K, int S, int64_t n_known, int64_t N, size_t *bytes);
int tip_top_triplets(int P, int K, int S, const double *d_theta, const double *d_p, const int32_t *d_cand, int n_cand,
                     const uint64_t *d_known, int64_t n_known, int64_t N, void *d_ws, size_t ws_bytes, int32_t *d_out_ids,
                     double *d_out_scores, int64_t *h_n_out, void *stream);
/* scoring passes (full sweeps) the last tip_top_triplets of this thread ran (measurement) */
int tip_top_triplets_last_passes(void);

/* ---- testResultsReducer.py:160-184: mean / median / standard deviation of every test triplet across samples ----
 * d_scores[S][T]: score of triplet t in sample j at [j * T + t]; d_n[t] (or NULL = S) = how many leading samples of
 * triplet t are valid.  mean = sequential sum in sample order / n; median = the reference's rule (ascending sort;
 * odd n: element round-half-even(n / 2), even n: mean of the two centre elements); std = sqrt(sum over the sorted
 * values of (x - mean)^2 / n).  Every operation is a separately rounded IEEE operation in the reference's order, so
 * mean and median are bit-identical to CPython.  d_sorted[S][T]: scratch, returns the ascending values per triplet.
 * The AUC / precision / recall / fallout of the mean scores then come from tip_metrics. */
int tip_reduce_samples(int S, int64_t T, const double *d_scores, const int32_t *d_n, double *d_sorted, double *d_mean,
                       double *d_median, double *d_std, void *stream);

/* ---- host-buffer entry: n_iter full make_iteration()s with HOST inputs and outputs ----
 * Copies rows/deg/theta/p to the device, runs n_iter x (E-step, M-step), copies theta/p back and
 * synchronises.  Keeps grow-only device scratch for the life of the process (the only function that allocates).
 * This is the call bench.py times for the end-to-end number.
 * Plain fp64, K <= 10: the first iteration is STREAMED - one copy of all rows on a side stream, the E-step kernel
 * polls each tile's rows until they have landed and so follows the DMA front (see tip_em_step_host_rows).  If the
 * rows do not arrive within 5 s (a platform that cannot run the copy beside the kernel) the call returns -3 and
 * h_theta / h_p are undefined; if the words the kernel consumed do not add up to the words that landed (verified on the
 * device after the copy) no M-step of the call takes effect and all iterations are repeated from the resident rows
 * before the call returns - the result is then still exact, only slower; the environment variable TIP_HOST_NO_STREAM=1 (read on every call) selects the
 * copy-in-chunks-then-compute path instead.  With TIP_EM_SLOT_SEGMENTED in `flags` the rows are ordered on the device
 * (tip_order_rows) once they have landed and iterations 2..n_iter run the slot-segmented kernels.
 * One call at a time per process (the scratch is shared). */
int tip_em_iterations_host(int P, int K, const void *h_rows, int64_t n_rows, int64_t n_rows_r0,
                           const int32_t *h_deg, double *h_theta, double *h_p, int n_iter, unsigned flags);

/* 8-byte host rows for the entry above (flags | TIP_ROWS_COMPACT8): halves the host->device traffic, which is what
 * bounds a single host-buffer iteration.  row = c | b << 20 | a << 40 | rating << 60 | count << 61; the device
 * expands them to the 16-byte rows as each chunk lands.  Pure host code (no CUDA call).  Fails (-1) when a gene id
 * needs more than 20 bits or a count exceeds 7 (duplicated input lines, TIP.py:361-368): use the 16-byte rows then. */
int tip_rows_compact_host(const void *h_rows, int64_t n_rows, uint64_t *h_rows8);
/* device side of the same format: d_rows8[n_rows] (8 B each) -> d_rows[n_rows] (16 B each), for callers that do
 * their own host->device copies (bench.py's link-sharded end-to-end leg) */
int tip_rows_expand(const void *d_rows8, void *d_rows, int64_t n_rows, void *stream);

/* ---- the digenic extension (src/TrigenicInteractionPredictor_23.py): PAIR links sharing theta, rating tensor q[K][K][2] ----
 * d_pairs: n_pairs rows int4 {a, b, n0, n1} (gene ids in the key's string-sorted order, counts per rating; no padding,
 * no ordering required).  For a pair: d_r = eps + sum_ij th_a[i] th_b[j] q_ij,r, s_r = n_r / d_r (_23.py:1617-1620).
 *   tip_pairs_step       adds the pair terms of Ntheta (_23.py:1629-1630) INTO d_stats[0, P*K) - call it after tip_em_step
 *                        (which zeroes and fills the statistics of the triplets) and before tip_normalise, with a degree
 *                        vector that counts appearances in distinct triplets AND pairs (_23.py:1584-1586, 1615-1616) -
 *                        and writes d_sq[2][K*K] = sum_l s_r th_a[i] th_b[j] (nqr = q * Sq, _23.py:1631)
 *   tip_pairs_normalise  q <- nqr / (eps + nqr_0 + nqr_1), in place (_23.py:1653-1659)
 *   tip_pairs_loglik     *d_out += sum_pairs n_r log d_r (_23.py:1551-1560; add it to tip_loglik's value) */
int tip_pairs_step(int P, int K, const void *d_pairs, int64_t n_pairs, const double *d_theta, const double *d_q, double *d_stats,
                   double *d_sq, void *stream);
int tip_pairs_normalise(int K, const double *d_sq, double *d_q, void *stream);
int tip_pairs_loglik(int P, int K, const void *d_pairs, int64_t n_pairs, const double *d_theta, const double *d_q, double *d_out,
                     void *stream);

/* ---- link shards over NVLink peer memory (replaces the NCCL allreduce between E-step and M-step) ----
 * One process per GPU.  Each rank shares its statistics buffers and a flag array with its peers:
 *   tip_ipc_export(d_ptr, handle[64], &offset)    on the owner; handle+offset travel over any host channel
 *   tip_ipc_import(handle, offset, &d_peer_ptr)   on each peer: a pointer usable in kernels (P2P over NVLink)
 * Per iteration i (statistics double-buffered by the caller, buffer i & 1):
 *   tip_em_step(... d_stats = own buffer i&1 ...)
 *   tip_peer_barrier(h_flag_ptrs, d_epoch, rank, nranks)   every rank has finished writing buffer i&1
 *   tip_normalise_peers(P, K, h_stats_ptrs, nranks, ...)   M-step of the sum, in rank order, of all buffers i&1
 * h_flag_ptrs[r] / h_stats_ptrs[r]: HOST arrays of nranks DEVICE pointers (own memory at index `rank`);
 * a flag array is nranks uint64 initialised to 0; d_epoch is one local uint64 initialised to 0.
 * The barrier kernel spins on flags written by other GPUs: run one rank per GPU, never two ranks on one GPU. */
int tip_ipc_export(const void *d_ptr, void *h_handle64, int64_t *h_offset);
int tip_ipc_import(const void *h_handle64, int64_t offset, void **d_ptr_out);
int tip_peer_barrier(void *const *h_flag_ptrs, void *d_epoch, int rank, int nranks, void *stream);
int tip_normalise_peers(int P, int K, void *const *h_stats_ptrs, int nranks, const int32_t *d_deg, double *d_theta,
                        double *d_p, void *stream);
/* The same exchange as reduce-scatter + all-gather, in ONE kernel (the default of the Python engine):
 *   every rank signals that its statistics are complete and waits for its peers; rank r then sums slice r of the n
 *   statistics buffers in rank order, normalises it and STORES the new theta / p values of that slice into the theta / p
 *   arrays of every rank; the last CTA signals "delivered" and waits for the peers' signals, so that on return (in
 *   stream order) this rank's theta and p are complete and nobody reads its statistics any more - no double buffering.
 * Per rank and iteration 1/n of the statistics is read from each peer and 1/n of the parameters written to each.
 * h_theta_ptrs[r] / h_p_ptrs[r]: the theta [P*K] and p [2*K^3] arrays of rank r (peer-mapped; they must live in
 * IPC-shared memory); h_flag_ptrs[r]: 2 * nranks uint64 of rank r, zero-initialised; d_sync: three local uint64, zero.
 * A peer that does not show up for ~10 s poisons d_sync[0] (~0) for good; the caller checks it when it synchronises. */
int tip_peer_mstep(int P, int K, void *const *h_stats_ptrs, void *const *h_theta_ptrs, void *const *h_p_ptrs,
                   void *const *h_flag_ptrs, void *d_sync, int rank, int nranks, const int32_t *d_deg, void *stream);
/* Push-based exchange (the default of the Python engine): ONE kernel, ONE handshake.  Every rank stores its statistics
 * into its slot of every peer's inbox (remote stores over NVLink), then signals; once every peer's statistics have
 * arrived it adds the n buffers in rank order (its own statistics in place of its own slot) and runs the M-step of all
 * of theta and p locally.  The data travels before the barrier, while slower ranks are still in their E-step, so what
 * follows the last arrival is one flag latency and a local sum.  Replicas stay bit-identical (same numbers, same order).
 * h_inbox_ptrs[q]: inbox of rank q FOR THIS PARITY, [nranks][n_pad] doubles (double-buffer the inboxes: iteration i uses
 * inbox i & 1); h_flag_ptrs[q]: nranks uint64 of rank q, zero-initialised; d_sync: four local uint64, zero;
 * n_pad: slot stride in doubles (even, >= tip_stats_len).  Timeout (~10 s) poisons d_sync[0] (~0) for good.
 * theta_pushed != 0: the Ntheta part of the statistics is already in the peers' inboxes - the E-step stored it there
 * itself (tip_em_set_push_targets) - and only the 2 K^3 + 1 doubles behind it are sent here. */
int tip_peer_push_mstep(int P, int K, const double *d_own_stats, void *const *h_inbox_ptrs, void *const *h_flag_ptrs,
                        void *d_sync, int rank, int nranks, int64_t n_pad, int theta_pushed, const int32_t *d_deg,
                        double *d_theta, double *d_p, void *stream);
/* Fused compute + transfer for link shards: the NEXT tip_em_step(TIP_EM_SLOT_SEGMENTED) on this thread's process stores
 * every row of Ntheta, as its finish kernel produces it, into this rank's slot of every peer's inbox as well (remote
 * stores over NVLink that overlap the rest of the finish), so that tip_peer_push_mstep(theta_pushed = 1) has almost nothing
 * left to send before it signals.  One-shot: consumed by that E-step.  h_inbox_ptrs / n_pad as for tip_peer_push_mstep. */
int tip_em_set_push_targets(void *const *h_inbox_ptrs, int rank, int nranks, int64_t n_pad);

/* ---- roofline denominators: measured FMA peak of this GPU ----
 * kind 0: fp64 DFMA, 1: fp32 FFMA, 2: fp64 mma.sync (DMMA m8n8k4), 3: DFMA and DMMA interleaved.
 * Returns TFLOP/s (2 flops per FMA) in *tflops; runs on the current device, synchronous. */
int tip_measure_fma_peak(int kind, double *tflops);
/* scattered fp64 red.global.add throughput over `n_addr` doubles: G atomics/s in *gops.
 * mode 0: one random address per lane; mode 1: row-contiguous runs of 10 doubles. */
int tip_measure_red_f64(int64_t n_addr, int mode, double *gops);

/* gather bandwidth out of L2: random rows of `row_bytes` bytes (on 128-byte lines) of a table of n_rows_table rows, read
 * with 16-byte L2-only loads by 2048 threads per SM - the access pattern of the slot-segmented passes.  GB/s of whole
 * 32-byte sectors delivered in *gbs; the roofline denominator of those kernels. */
int tip_measure_l2_gather(int n_rows_table, int row_bytes, double *gbs);

/* ---- per-kernel timing of the slot-segmented E-step (measurement only) ----
 * tip_seg3_timing(1): every following tip_em_step(TIP_EM_SLOT_SEGMENTED) records CUDA events on its stream between its
 * five stages (not capturable in a CUDA graph while on); tip_seg3_last_timing waits for the last such step and returns
 * the milliseconds of {workspace memset, prep kernel, pass A, pass B + C, finish kernel}. */
int tip_seg3_timing(int enable);
int tip_seg3_last_timing(float *h_ms5);

#ifdef __cplusplus
}
#endif
#endif /* TIP_H_ */
