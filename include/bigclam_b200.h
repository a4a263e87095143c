/*
 * bigclam_b200.h — C ABI of the B200-native BigCLAM F-gradient / line-search step.
 *
 * The reference (thangdnsf/BigCLAM-ApacheSpark) has no FFI or plugin interface; its boundary is
 * the implicit signature of one spark-shell function and the globals it touches:
 *
 *     def backtrackingLineSearchs(uset: List[Long]): Double      codes/bigclam4-7.scala:152
 *       reads   collectNeighbor / Neightborbc (adjacency)         codes/bigclam4-7.scala:50-51
 *               K, liststepSizeRDD, alpha, MIN_P_/MAX_P_/MIN_F_/MAX_F_   :134,:28-34,:22,:39-43
 *       reads+writes  F (N x K affiliation rows), sumF (K)        codes/bigclam4-7.scala:36,38,190,192
 *       returns the log-likelihood after the update               codes/bigclam4-7.scala:196-222
 *
 * Every entry point below names the reference lines it replaces.  A JVM binding (JNI) that the
 * Scala driver would use is shown in INTEGRATION.md; the Python ctypes binding used by the tests
 * lives in bigclam_apachespark_b200/_lib.py.
 *
 * Conventions: plain C, no exceptions cross the boundary.  Every function returns 0 on success
 * and a negative BIGCLAM_E* code on failure; bigclam_last_error() gives the message.  The caller
 * owns all host buffers; the context owns all device memory.  A context is driven by one thread
 * at a time; distinct contexts are independent.  All calls are synchronous on return unless noted.
 * There is NO CPU fallback: creating a context without a usable CUDA device fails.
 */
#ifndef BIGCLAM_B200_H
#define BIGCLAM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BIGCLAM_OK            0
#define BIGCLAM_EINVAL      (-1)   /* bad argument */
#define BIGCLAM_ECUDA       (-2)   /* CUDA runtime / driver error, or no device */
#define BIGCLAM_ENOMEM      (-3)   /* host or device allocation failed */
#define BIGCLAM_EIO         (-4)   /* edge-list file unreadable / malformed */
#define BIGCLAM_EUNSUPPORTED (-5)  /* parameter combination the kernels do not cover */

typedef struct bigclam_ctx bigclam_ctx;

/* Script-level variables of the reference, one field each. */
typedef struct {
    int32_t k;           /* K.value: number of communities            bigclam4-7.scala:134,249 */
    int32_t max_inter;   /* MaxInter = 15 -> 16 step sizes            bigclam4-7.scala:26-34   */
    double  alpha;       /* 0.05  Armijo slope                        bigclam4-7.scala:22      */
    double  beta;        /* 0.1   step shrink factor                  bigclam4-7.scala:24      */
    double  min_p;       /* MIN_P_ = 0.0001                           bigclam4-7.scala:40      */
    double  max_p;       /* MAX_P_ = 0.9999                           bigclam4-7.scala:41      */
    double  min_f;       /* MIN_F_ = 0.0                              bigclam4-7.scala:42      */
    double  max_f;       /* MAX_F_ = 1000.0                           bigclam4-7.scala:43      */
    int32_t device;      /* CUDA ordinal; -1 = the calling thread's current device */
    int32_t flags;       /* BIGCLAM_F_* */
} bigclam_params;

#define BIGCLAM_F_TIME_KERNELS   1   /* record CUDA events around every step-kernel launch */
#define BIGCLAM_F_RECORD_ACCEPTED 2  /* keep the accepted step index per node (diagnostics/tests) */
#define BIGCLAM_F_SPARSE_ROWS     4  /* keep F as sparse rows on the device (like the reference's BSV[Double],
                                        bigclam4-7.scala:97-104): k <= 1024, min_f == 0, n < 2^28.  The dense entry
                                        points still work (bigclam_set_F / bigclam_get_F convert on the device);
                                        bigclam_set_F_csr / bigclam_get_F_csr never build a dense image. */

#define BIGCLAM_F_LS_EXHAUSTIVE   8  /* sparse rows: evaluate all max_inter+1 candidates of every node like the reference
                                        does (bigclam4-7.scala:172-181).  Default: a candidate that a bound on the node's
                                        objective proves unable to pass the Armijo test (:181) is not evaluated — same
                                        accepted steps, same rows, same LLH bits (DESIGN.md (d), tests/test_gpu_prune.py). */

/* Fills *p with the reference's constants for a given K. */
int bigclam_default_params(bigclam_params *p, int32_t k);

/* The 16 candidate step sizes, built by repeated `*= beta` exactly as bigclam4-7.scala:28-34
 * (out[0] = 1.0, out[j] = out[j-1]*beta; max_inter+1 values). */
int bigclam_step_sizes(double beta, int32_t max_inter, double *out);

/*
 * Context = the hot path's resident state: CSR adjacency (collectNeighbor, :50-51), F double
 * buffer, sumF.  rowptr has n+1 entries, col has rowptr[n] entries in [0,n); neighbour lists are
 * taken as given (multiplicity and order preserved, like collectNeighborIds(Either)).
 * Replaces: Neightborbc broadcast (:51) and the per-call Fbc broadcast (:154).
 */
int bigclam_create(bigclam_ctx **out, int64_t n, const int64_t *rowptr, const int32_t *col,
                   const bigclam_params *params);
void bigclam_destroy(bigclam_ctx *ctx);
const char *bigclam_last_error(const bigclam_ctx *ctx);   /* ctx may be NULL: last create error */

/* F <- host row-major n x k; sumF <- exact column sums (initNeighborComF, :105-107). */
int bigclam_set_F(bigclam_ctx *ctx, const double *F);
/* Optional: inject a sumF that has drifted from colsum(F) (the reference never recomputes it, :192). */
int bigclam_set_sumF(bigclam_ctx *ctx, const double *sumF);
int bigclam_get_F(bigclam_ctx *ctx, double *F_out);        /* n x k row-major */
int bigclam_get_sumF(bigclam_ctx *ctx, double *sumF_out);  /* k */

/*
 * One call of backtrackingLineSearchs(uset)  (bigclam4-7.scala:152-223): PRE (:157-169), 16-candidate
 * Armijo line search keeping the max passing step (:172-184), Jacobi row swap + incremental sumF
 * (:186-193), LLH with the new F and sumF (:196-219, returned).  node_mask: NULL = all vertices
 * (the reference always passes all, :227); otherwise n bytes, u is in uset iff node_mask[u] != 0.
 * Nodes with an empty neighbour list are never updated (the reference would throw, see DESIGN.md).
 * The returned LLH is the PRE sum of the next call, so the next call's step kernel (same uset) is launched
 * speculatively to obtain it; a following bigclam_step with the same uset just commits that result.  Every
 * other entry point that reads or writes the state sees exactly the state after this call.
 */
int bigclam_step(bigclam_ctx *ctx, const uint8_t *node_mask, double *llh_out, int64_t *n_updated_out);

/* loglikelihood() (bigclamv3-7.scala:106-120, Bigclamv2.scala:187-200) on the current F, sumF. */
int bigclam_loglikelihood(bigclam_ctx *ctx, double *llh_out);

/*
 * Outer loop on the device, LLH of step t taken from step t+1's PRE pass (they are the same sum).
 *   variant 4: SGDFindC  (bigclam4-7.scala:225-243)  LLHold = first step; returns LLHold as coded at :242
 *   variant 3: MBSGD     (bigclamv3-7.scala:206-222) LLHold = 0.0
 *   variant 2: MBSGD     (Bigclamv2.scala:203-219)   LLHold = loglikelihood()
 * Stops when |1 - new/old| < rel_tol (:237) or after max_outer hot-path calls (0 = unbounded, like
 * the reference).  llh_trace (optional, trace_cap doubles) receives every call's returned LLH.
 * On return F/sumF are exactly the state after `*calls_out` calls.
 */
int bigclam_run(bigclam_ctx *ctx, int32_t variant, double rel_tol, int64_t max_outer,
                double *llh_out, int64_t *calls_out, double *llh_trace, int64_t trace_cap);

/* Diagnostics (BIGCLAM_F_RECORD_ACCEPTED): index of the accepted step size per node for the
 * most recent step, -1 = row unchanged. */
int bigclam_get_accepted(bigclam_ctx *ctx, int8_t *accepted_out);

/* Timing of the most recent bigclam_step / bigclam_run (BIGCLAM_F_TIME_KERNELS), CUDA events on
 * the context's stream: total device ms of the step kernels and how many were launched. */
int bigclam_get_kernel_time(bigclam_ctx *ctx, double *step_kernel_ms_sum, int64_t *step_kernel_launches,
                            int64_t *all_kernel_launches);

/* Interop with the host framework's plumbing (torch streams / NCCL buffers): use an existing
 * cudaStream_t, and expose device pointers of the current F (n x ld doubles, ld = row pitch) and sumF. */
/* Sparse rows (BIGCLAM_F_SPARSE_ROWS): how the small nodes were processed since the
 * context was created / the counters were last read — tiles done on the tile path, tiles that did not fit the
 * warp's shared memory and went node by node through the general path; the tile layout of the current order
 * (tiles, nodes on the general path, split hubs).  The two counters count from the previous read. */
int bigclam_get_tile_stats(bigclam_ctx *ctx, int64_t *tiles_done, int64_t *tiles_fallback, int64_t *n_tiles,
                           int64_t *n_general_nodes, int64_t *n_split_hubs);

/* Sparse rows, line search by bounds: of the nodes that asked for a line search since the previous read (split hubs not
 * counted), how many had at least one candidate that the bounds could not exclude (and were therefore evaluated). */
int bigclam_get_ls_stats(bigclam_ctx *ctx, int64_t *nodes_asked, int64_t *nodes_searched);

/*
 * Held-out pairs, for choosing K by held-out likelihood (BigCLAM, Yang & Leskovec; the thesis p.20).  Symmetric lists
 * ho_rowptr[n+1] / ho_col: the held-out partners of every node; ho_is_edge[e] = 1 for a held-out edge, 0 for a held-out
 * non-edge.  No self pairs, no pair twice in a list, no pair that is also in the context's neighbour lists.  From now
 * on bigclam_step / bigclam_run / bigclam_loglikelihood use the masked objective: every held-out pair is left out of
 * both the edge term and the non-edge term, i.e. llh_u gains sum_{v in HO(u)} Fu.Fv and grad_u gains sum_{v in HO(u)} Fv
 * (DESIGN.md (f) f-5).  NULL ho_rowptr clears the lists and restores the unmasked behaviour exactly.  Sparse-rows
 * contexts on one GPU only: BIGCLAM_EUNSUPPORTED for a dense context, one that owns a node range or set, or one with
 * peers open; any input error is BIGCLAM_EINVAL and leaves the context as it was.
 */
int bigclam_set_holdout(bigclam_ctx *ctx, const int64_t *ho_rowptr, const int32_t *ho_col, const uint8_t *ho_is_edge);
/* L_HO of the current F over every held-out pair once: sum of log(1 - p) over held-out edges plus sum of log(p) over
 * held-out non-edges, p = clamp(exp(-Fu.Fv), min_p, max_p) (bigclam4-7.scala:166).  n_pairs_out (optional) = number
 * of unordered pairs scored.  Same bits on every run. */
int bigclam_holdout_loglikelihood(bigclam_ctx *ctx, double *llh_out, int64_t *n_pairs_out);

/* Sparse rows: re-cut the tiles of small nodes for the current average row size (rows grow or shrink while the solver
 * runs; bigclam_run does this by itself between its batches, bigclam_set_F* always).  Synchronises the stream. */
int bigclam_retile(bigclam_ctx *ctx);

int bigclam_set_stream(bigclam_ctx *ctx, void *cuda_stream);
int bigclam_device_state(bigclam_ctx *ctx, void **F_dev, void **F_next_dev, void **sumF_dev, int64_t *ld);
/* Device pointer of the per-node accepted-step index (int8, n entries; BIGCLAM_F_RECORD_ACCEPTED):
 * lets a multi-GPU caller exchange only the rows that changed. */
int bigclam_device_accepted(bigclam_ctx *ctx, void **accepted_dev);

/*
 * Multi-GPU (node-partitioned) pieces: a context created with an owned node range only updates
 * rows [lo,hi); rows outside are halo (read-only copies refreshed by the caller's collective).
 * See DESIGN.md (e).  bigclam_step_local runs PRE+LS+row swap for owned rows and leaves the partial
 * reductions [sum(old-new) (ld) | unused (ld) | llh_pre | n_updated] in a device buffer of 2*ld+2 doubles
 * (ld = row pitch, see bigclam_device_state) that
 * the caller all-reduces; bigclam_finish_local applies the reduced values (sumF update, :192).
 */
int bigclam_set_owned_range(bigclam_ctx *ctx, int64_t lo, int64_t hi);
int bigclam_set_owned_nodes(bigclam_ctx *ctx, const int32_t *nodes, int64_t count);   /* arbitrary owned set */
int bigclam_set_uset(bigclam_ctx *ctx, const uint8_t *node_mask);   /* uset of the following bigclam_step_local calls (NULL = all) */
int bigclam_step_local(bigclam_ctx *ctx, void **partials_dev /* 2*ld+2 doubles */);
int bigclam_finish_local(bigclam_ctx *ctx, double *llh_pre_out, int64_t *n_updated_out);  /* both NULL: asynchronous, no host sync */
int bigclam_collect_timing(bigclam_ctx *ctx);   /* sync + sum the kernel timings recorded since the last collection */
int bigclam_llh_local(bigclam_ctx *ctx, void **partials_dev /* llh at [2*ld] */);
/* Undo the most recent bigclam_finish_local (the previous F and sumF are still intact in the other
 * halves of the double buffers): used to drop the speculative step of a pipelined convergence loop. */
int bigclam_rollback(bigclam_ctx *ctx);

/*
 * Peer replicas over NVLink (one process per GPU on one box).  bigclam_ipc_export writes the two CUDA IPC
 * handles (2 x 64 bytes) of this context's F double buffer; the caller all-gathers them over its own
 * plumbing and hands all of them (world x 2 x 64 bytes, rank order) to bigclam_ipc_open_peers.  From then
 * on bigclam_step_local pushes every owned row that this step or the previous one changed straight into
 * the peers' replicas (plain stores to peer memory inside the step kernel): the row exchange that
 * replaces the reference's re-broadcast of F (bigclam4-7.scala:154) is fused into the compute kernel and
 * only the all-reduce of the partials remains.  bigclam_mark_all_changed forces a full publish (after
 * bigclam_set_F).
 */
int bigclam_ipc_export(bigclam_ctx *ctx, void *handles_out);
int bigclam_ipc_open_peers(bigclam_ctx *ctx, int32_t world, int32_t rank, const void *all_handles);
int bigclam_mark_all_changed(bigclam_ctx *ctx);
/*
 * With BIGCLAM_F_SPARSE_ROWS the replicas are (header, pool) pairs: bigclam_ipc_handle_count() handles per rank
 * (4 instead of 2) travel through bigclam_ipc_export / bigclam_ipc_open_peers, every rank allocates its owned
 * rows inside its own part of the output pool (bigclam_set_pool_region: disjoint parts, 8-byte words) and the
 * step kernel writes each owned row to the same offset of every replica — all owned rows, every step (the
 * output pool is rebuilt per step, so there is no changed-row bookkeeping).
 */
int bigclam_ipc_handle_count(const bigclam_ctx *ctx);
/*
 * Fused collective of the node-partitioned path (sparse rows): instead of an all-reduce by the host framework, the
 * reduction kernel behind every step kernel stores this rank's sums [sum(old-new) | llh | n_updated] into its slot
 * of every rank's exchange buffer (peer memory over NVLink) and raises a flag there; bigclam_finish_local /
 * bigclam_llh_finish_local then wait for all flags on the device and add the slots up in rank order (every rank
 * gets the same bits).  bigclam_xchg_export allocates the buffers and writes their 2 CUDA IPC handles (2 x 64
 * bytes); the caller all-gathers them and passes all of them (world x 2 x 64 bytes, rank order) to
 * bigclam_xchg_open_peers.  Replaces the driver-side reduce of bigclam4-7.scala:191-192 and :219.
 */
int bigclam_xchg_export(bigclam_ctx *ctx, int32_t world, int32_t rank, void *handles_out);
int bigclam_xchg_open_peers(bigclam_ctx *ctx, const void *all_handles);
int bigclam_llh_finish_local(bigclam_ctx *ctx, double *llh_out);

/*
 * All the GPUs of one box behind ONE handle, driven by one host thread — what a JVM/JNI caller uses (INTEGRATION.md):
 * one context per device (sparse rows), nodes dealt over the ranks by degree, each rank's new rows stored straight
 * into every replica by the step kernel, sums combined by the fused collective above.  No NCCL, no Python.
 * devices: `world` CUDA ordinals, NULL = 0 .. world-1.  The entry points mirror the single-GPU ones
 * (same reference lines); rank selects the replica a getter reads (they are identical).
 */
typedef struct bigclam_multi bigclam_multi;
int  bigclam_multi_create(bigclam_multi **out, int64_t n, const int64_t *rowptr, const int32_t *col,
                          const bigclam_params *params, int32_t world, const int32_t *devices);
void bigclam_multi_destroy(bigclam_multi *m);
const char *bigclam_multi_last_error(const bigclam_multi *m);     /* m may be NULL: last create error */
int  bigclam_multi_world(const bigclam_multi *m);
int  bigclam_multi_set_F(bigclam_multi *m, const double *F);
int  bigclam_multi_set_F_csr(bigclam_multi *m, const int64_t *indptr, const int32_t *indices, const double *values);
int  bigclam_multi_set_sumF(bigclam_multi *m, const double *sumF);
int  bigclam_multi_get_F(bigclam_multi *m, int32_t rank, double *F_out);
int  bigclam_multi_get_sumF(bigclam_multi *m, int32_t rank, double *sumF_out);
int  bigclam_multi_get_F_nnz(bigclam_multi *m, int64_t *nnz_out);
int  bigclam_multi_get_F_csr(bigclam_multi *m, int64_t *indptr_out, int32_t *indices_out, double *values_out);
int  bigclam_multi_step(bigclam_multi *m, const uint8_t *node_mask, double *llh_out, int64_t *n_updated_out);
int  bigclam_multi_loglikelihood(bigclam_multi *m, double *llh_out);
int  bigclam_multi_run(bigclam_multi *m, int32_t variant, double rel_tol, int64_t max_outer, double *llh_out,
                       int64_t *calls_out, double *llh_trace, int64_t trace_cap);
int  bigclam_multi_get_kernel_time(bigclam_multi *m, double *max_rank_ms_sum, int64_t *step_kernel_launches);
int  bigclam_multi_get_ls_stats(bigclam_multi *m, int64_t *nodes_asked, int64_t *nodes_searched);   /* bigclam_get_ls_stats summed over the ranks */

/*
 * F as CSR rows, the shape of the reference's RDD[(Long, BSV[Double])] (bigclam4-7.scala:97-104): indptr[n + 1],
 * indices (component of each entry, any order inside a row), values.  sumF becomes the column sums (:105-106).
 * With BIGCLAM_F_SPARSE_ROWS no dense n x K image is ever built.  bigclam_get_F_nnz sizes the output of
 * bigclam_get_F_csr (ascending indices inside a row, explicit zeros never stored).
 */
int bigclam_set_F_csr(bigclam_ctx *ctx, const int64_t *indptr, const int32_t *indices, const double *values);
int bigclam_get_F_nnz(bigclam_ctx *ctx, int64_t *nnz_out);
int bigclam_get_F_csr(bigclam_ctx *ctx, int64_t *indptr_out, int32_t *indices_out, double *values_out);
int bigclam_set_pool_region(bigclam_ctx *ctx, int64_t base_words, int64_t cap_words);
int bigclam_get_pool_capacity(bigclam_ctx *ctx, int64_t *words_out);   /* words of each row pool (what the regions partition) */

/*
 * Edge-list reader with GraphX semantics (GraphLoader.edgeListFile, bigclam4-7.scala:45;
 * collectNeighborIds(EdgeDirection.Either), :50): '#' and blank lines skipped, whitespace split,
 * CRLF safe; each edge line adds dst to src's list and src to dst's list.  Vertex ids are relabelled
 * to 0..n-1 in ascending id order (ids_out gives the original id of each dense index).
 * multiplicity: 0 = keep (literal GraphX), 1 = dedup (simple undirected graph, self loops dropped).
 * Neighbour lists are sorted ascending.  Buffers are malloc'ed by the library; release with
 * bigclam_graph_free.
 */
typedef struct {
    int64_t  n;
    int64_t  nnz;
    int64_t *rowptr;   /* n+1 */
    int32_t *col;      /* nnz */
    int64_t *ids;      /* n: original vertex id of dense index i */
    int64_t  n_edge_lines;
} bigclam_graph;

int  bigclam_graph_read_edgelist(const char *path, int32_t multiplicity, bigclam_graph *out,
                                 char *errbuf, int64_t errbuf_len);
void bigclam_graph_free(bigclam_graph *g);

/*
 * The caller behind the hot path: community extraction, Bigclamv2.scala:223-230 (SURVEY.md §8f-3).
 * member_out[u*k + c] = 1 iff F_uc >= delta, or, when the row maximum is below delta, iff F_uc equals the
 * row maximum (ties included, as coded at :227).  delta is computed by the caller:
 * sqrt(-log(1 - e)) with e = 2*count/(N*(N-1)) (:223-224; `count` there is the number of vertices that
 * have edges, not |E|).
 */
int bigclam_extract(bigclam_ctx *ctx, double delta, uint8_t *member_out, double *fmax_out);

/*
 * Callers in front of the hot path (host side, one-off integer graph work; SURVEY.md §8f-2).
 * bigclam_conductance_seeds = conductanceLocalMin() (bigclam4-7.scala:58-73): ego-net conductance of every
 * node, candidates = the min-id neighbour of each node (tuple .min at :70), ranked by conductance ascending
 * (ties by id).  seeds_out has room for n ids; *n_seeds_out receives the number of candidates.
 * bigclam_init_neighbor_com_F = initNeighborComF(K) (bigclam4-7.scala:81-108): column c of F is the
 * indicator of the neighbours of the c-th (in id order) of the first K ranked seeds; include_self adds the
 * seed (Bigclamv2.scala:70); missing columns are random 0/1 from a seeded xorshift64* (the reference's
 * Random is unseeded).  The result goes to bigclam_set_F.
 */
int bigclam_conductance_seeds(int64_t n, const int64_t *rowptr, const int32_t *col, double *conductance_out,
                              int32_t *seeds_out, int64_t *n_seeds_out);
/* The same ranking with the ego-net conductances computed on the GPU (one warp per node, csrc/initf_gpu.cu); device:
 * CUDA ordinal, -1 = current.  Fails without a CUDA device (BIGCLAM_ECUDA): bigclam_conductance_seeds is the host path. */
int bigclam_conductance_seeds_gpu(int64_t n, const int64_t *rowptr, const int32_t *col, int32_t device,
                                  double *conductance_out, int32_t *seeds_out, int64_t *n_seeds_out);
int bigclam_init_neighbor_com_F(int64_t n, const int64_t *rowptr, const int32_t *col, int32_t k,
                                const int32_t *ranked_seeds, int64_t n_ranked, int32_t include_self,
                                uint64_t pad_seed, double *F_out);

/* Library / device probe (no compute): returns the number of visible CUDA devices or <0. */
int bigclam_device_count(void);
const char *bigclam_version(void);

#ifdef __cplusplus
}
#endif
#endif /* BIGCLAM_B200_H */
