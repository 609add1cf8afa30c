/*
 * hammock_b200.h -- C ABI of the B200-native greedy-clustering stage of Hammock.
 *
 * Drop-in boundary.  The reference has no FFI layer; its narrowest seam for this path is
 * the Java interface
 *     SequenceClusterer { List<Cluster> cluster(List<UniqueSequence>) }
 *         (reference src/cz/krejciadam/hammock/SequenceClusterer.java:15-26)
 * instantiated for greedy in exactly one place
 *         new ShiftedScorer(scoringMatrix, shiftPenalty, maxShift)           Hammock.java:402
 *         new LimitedGreedySequenceClusterer(scorer, threshold, limit)       Hammock.java:403
 *         clusterer.cluster(sequences)                                       Hammock.java:409
 * hmk_greedy_cluster() replaces that call: the host hands over the (already ordered,
 * UniqueSequence.sortSequences, UniqueSequence.java:176-203) sequences as residue codes plus
 * the scorer/clusterer constructor arguments and rebuilds List<Cluster> from cluster_id /
 * member_rank / result_order.  INTEGRATION.md shows the JNI / FFM stub.
 *
 * Everything runs on the GPU (CUDA, sm_100a).  There is NO CPU fallback: without a usable
 * device every entry point returns HMK_ERR_CUDA.
 *
 * All pointers are host memory owned by the caller and only read/written during the call.
 */
#ifndef HAMMOCK_B200_H
#define HAMMOCK_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMK_ABI_VERSION 2

/* status codes: the reference's failure modes on this path */
#define HMK_STATUS_OK 0
#define HMK_STATUS_SHIFT_TOO_BIG 1 /* DataException "Shift too big"      ShiftedScorer.java:59-62 */
#define HMK_STATUS_NULL_CLUSTER 2  /* NullPointerException               LimitedGreedySequenceClusterer.java:104,108 */
#define HMK_STATUS_BAD_RESIDUE 3   /* residue code >= 24                  UniqueSequence.java:51-54 */
#define HMK_STATUS_CUDA 4          /* CUDA / NCCL failure (no CPU fallback) */
#define HMK_STATUS_BAD_ARG 5
#define HMK_STATUS_UNSUPPORTED 6   /* hmk_clinkage_cluster / hmk_clinkage_run only, see there */

typedef struct {
    int32_t n;                /* sequences, ALREADY in clustering order                              */
    const uint8_t* residues;  /* concatenated codes 0..23, alphabet "ARNDCQEGHILKMFPSTWYVBZX*"        */
                              /*   (UniqueSequence.java:23-26)                                        */
    const int32_t* offsets;   /* n+1 prefix offsets into residues                                    */
    const int32_t* abundance; /* UniqueSequence.size() (UniqueSequence.java:81-88), Java int          */
    const int32_t* matrix;    /* 24*24 row-major, as FileIOManager.loadScoringMatrix returns it       */
                              /*   (FileIOManager.java:46-81)                                         */
    int32_t threshold;        /* LimitedGreedySequenceClusterer ctor  (...Clusterer.java:22-26)       */
    int32_t max_shift;        /* ShiftedScorer ctor                   (ShiftedScorer.java:28-32)      */
    int32_t shift_penalty;    /* ShiftedScorer ctor                                                   */
    int32_t max_clusters;     /* LimitedGreedySequenceClusterer ctor                                  */
} hmk_greedy_in;

typedef struct {
    int32_t* cluster_id;      /* [n] Cluster.getId() of the sequence's cluster = founder's index      */
    int32_t* member_rank;     /* [n] position in Cluster.getSequences() (0 founder, 1 partner, ...)   */
    int32_t* result_order;    /* [n] ids of the returned List<Cluster>, in list order                 */
    int32_t n_result;         /* length of that list                                                  */
    int32_t n_multi;          /* multi-member clusters (they form the list's prefix)                  */
    int32_t error_step;       /* phase-1 step index for HMK_STATUS_NULL_CLUSTER, else -1              */
} hmk_greedy_out;

/* executed-work and timing report of the last run */
typedef struct {
    int64_t bulk_pairs;       /* pair scores executed by the bulk kernels                             */
    int64_t scalar_pairs;     /* pair scores executed one at a time (member checks, resolvers)        */
    int64_t bulk_cells;       /* matrix cells summed by the bulk kernels                              */
    int64_t bulk_ops;         /* algorithmic int ops = cells + shifts (SURVEY.md 8d)                  */
    double bulk_kernel_ms;    /* sum of CUDA-event durations of the bulk scoring launches             */
    double total_ms;          /* whole hmk_run, device timed                                          */
    double phase1_ms, phase2_ms;
    int32_t bulk_launches;    /* bulk scoring kernel launches                                         */
    int32_t total_launches;   /* all kernel launches                                                  */
    int32_t p1_steps, p1_joins, p1_new_clusters, p1_orphans, p1_batches, p1_restarts;
    int32_t p2_queries, p2_assigned, p2_rounds;
    int64_t p2_hits, p2_candidates;
    int32_t fast_path;        /* 0: generic scalar kernel, 1: packed SWAR kernel (one length), 2: packed per length bucket */
    int32_t lane_bits;        /* 8 or 16 on the fast path                                             */
    int32_t error_step;       /* phase-1 step of HMK_STATUS_NULL_CLUSTER in the last run, else -1     */
    int32_t flags;            /* HMK_FLAG_* of the last run                                           */
    int64_t xhits_kept;       /* phase-1 partner-search hits the run wanted to keep for phase 2       */
    int64_t xhits_capacity;   /* entries the kept-hit buffer had; kept > capacity == overflow         */
} hmk_stats;
/* hmk_stats.flags */
#define HMK_FLAG_P2_REUSED 1      /* phase 2 took its founder hits from the phase-1 partner searches   */
#define HMK_FLAG_XHIT_OVERFLOW 2  /* the kept-hit buffer overflowed: this run paid the separate founder  */
                                  /* pass (about 1.4x slower); the next run on this context sizes it right */
#define HMK_FLAG_ASYMMETRIC 4     /* substitution matrix not symmetric: hit reuse not applicable        */

typedef struct hmk_ctx hmk_ctx;

int hmk_abi_version(void);

/* One blocking call == SequenceClusterer.cluster(sequences).  Uses CUDA device `device`.  The library
 * keeps one context per device between calls (device buffers stay allocated, so repeated calls do not
 * pay allocation again); hmk_release_cached frees them. */
int hmk_greedy_cluster(const hmk_greedy_in* in, hmk_greedy_out* out, int device, char* errbuf, size_t errlen);
/* The same blocking call on n_gpus devices of THIS process (SURVEY.md 8b's `n_gpus`): the reference's host is
 * one JVM that calls cluster() once, synchronously (Hammock.java:409), so the library itself runs one worker
 * thread per device and builds the NCCL communicator (one unique id, ncclCommInitRank per thread).
 * devices == NULL means devices 0 .. n_gpus-1.  Contexts and the communicator are kept for the next call
 * with the same device list.  The result is identical to the one-GPU result. */
int hmk_greedy_cluster_multi(const hmk_greedy_in* in, hmk_greedy_out* out, const int32_t* devices, int32_t n_gpus,
                             char* errbuf, size_t errlen);
/* SURVEY.md 8(f) N1 -- the EXACT complete-linkage initial clustering, Hammock's default initial stage for up to 10 000
 * unique sequences (Hammock.java:371-373):  new ClinkageSequenceClusterer(scorer, threshold).cluster(sequences)
 * (Hammock.java:457-462, ClinkageSequenceClusterer.java:43-124; nearest-neighbour chain over complete-linkage scores with
 * CachedClusterScorer.java:38-125).  Same input struct (max_clusters is ignored; the sequences come in the caller's order --
 * runClinkageClustering does not sort).  Outputs: cluster_id[i] = Cluster.getId() of sequence i's cluster (i + 1 for
 * singletons, n + 2, n + 3, ... for merged clusters, in merge order), member_rank[i] = position in getSequences(),
 * result_order[0 .. n_result) = the ids of the returned list IN ITS ORDER, n_multi = clusters with more than one member.
 * The chain start and the order of the returned list come from java.util.HashSet iteration; they are reproduced for the
 * OpenJDK 8+ HashMap.  Any n: up to 32768 sequences (option clinkage_dense_max) the scores are kept as a dense n x n
 * matrix, above that only the pairs scoring >= threshold are kept, as sparse rows in device memory (12 bytes per pair and
 * direction); both give the same result.  HMK_STATUS_UNSUPPORTED: asymmetric matrix (the reference's cached scores then
 * depend on the thread schedule), sparse rows that do not fit in the free device memory (errbuf then names the number of
 * valid pairs and the bytes needed), or a hash bin that the JDK would turn into a tree.  An empty input (the reference
 * throws NoSuchElementException) returns HMK_STATUS_BAD_ARG. */
int hmk_clinkage_cluster(const hmk_greedy_in* in, hmk_greedy_out* out, int device, char* errbuf, size_t errlen);
/* hmk_clinkage_cluster on the caller's context: its options apply, and hmk_get_stats / hmk_get_section_ms report the call.
 * Fields hmk_stats holds afterwards: bulk_pairs (pair scores executed; the sparse path scores the upper triangle twice,
 * once to count and once to fill the rows), p1_steps (nearest-neighbour searches), total_ms = phase1_ms (device time of
 * the call), bulk_kernel_ms (with option profile), bulk_launches, total_launches, fast_path, lane_bits; sparse path only:
 * xhits_kept (directed valid pairs = entries of the rows) and xhits_capacity (entries the row storage holds).  The other
 * fields are 0.  The context's uploaded sequences are replaced by `in`. */
int hmk_clinkage_run(hmk_ctx* ctx, const hmk_greedy_in* in, hmk_greedy_out* out, char* errbuf, size_t errlen);
/* Frees the contexts the two calls above keep.  Call it before the process unloads CUDA if the memory
 * matters; the library never tears them down from a static destructor. */
void hmk_release_cached(void);

/* Handle API: the same work split into upload / device-resident run / download, so that a
 * host can keep the sequences resident and time the stages separately. */
int hmk_create(hmk_ctx** ctx, int device, char* errbuf, size_t errlen);
void hmk_destroy(hmk_ctx* ctx);
int hmk_upload(hmk_ctx* ctx, const hmk_greedy_in* in, char* errbuf, size_t errlen);
int hmk_run(hmk_ctx* ctx, char* errbuf, size_t errlen);
int hmk_download(hmk_ctx* ctx, hmk_greedy_out* out, char* errbuf, size_t errlen);
int hmk_get_stats(hmk_ctx* ctx, hmk_stats* stats);
/* Multi-GPU: one process per GPU.  Rank 0 obtains a 128-byte NCCL unique id, the host distributes
 * it (any channel), every rank calls hmk_init_distributed on its own context and then makes the
 * SAME upload / run / download calls with the SAME input.  Phase 1 stripes the later singletons
 * across ranks and all-gathers the per-rank best-hit lists; phase 2 shards the queries and
 * all-gathers the candidate lists; decisions are replicated, so every rank returns the full,
 * identical result. */
int hmk_nccl_unique_id(void* id128, char* errbuf, size_t errlen);
int hmk_init_distributed(hmk_ctx* ctx, int rank, int world, const void* id128, char* errbuf, size_t errlen);

/* CUDA-event stopwatch on the library's stream (brackets upload + run + download for end-to-end
 * timing); hmk_timer_end synchronises and returns milliseconds. */
int hmk_timer_begin(hmk_ctx* ctx);
int hmk_timer_end(hmk_ctx* ctx, double* ms);
/* roofline denominators measured on this device: out4[0] IADD3 lane-instructions/s (the INT32 ALU
 * peak), out4[1] lane-instructions/s of an IADD3 + IMAD mix (both integer pipes), out4[2]
 * conflict-free shared-memory load bytes/s, out4[3] SM count */
int hmk_measure_peaks(hmk_ctx* ctx, double* out4, char* errbuf, size_t errlen);
/* device time per section of the last run (only filled when option "profile" is 1):
 * p1_select, p1_partner, p1_cluster, p1_intra, p1_resolve, p2_setup, p2_filter, p2_check, p2_sort,
 * p2_base, p2_iterate, p2_commit, final
 * After hmk_clinkage_run the first three slots hold the stages of the complete-linkage call instead: [0] scoring (dense:
 * the n x n matrix; sparse: the counting pass), [1] sparse row build (the filling pass, row sort and twin index; 0 on the
 * dense path), [2] nearest-neighbour chain; the others are 0.
 * hmk_score_graph adds to slots [0] (scoring passes) and [1] (shift, sort and edge passes) the device time of the batches
 * it computes; a call at cursor {0, 0} sets both to 0 first.
 * hmk_nearest sets slots [0] (scoring pass: profiles and the top-k launch) and [1] (list merge, score and shift) to the
 * device time of the row batches of the call. */
#define HMK_NSECTIONS 13
int hmk_get_section_ms(hmk_ctx* ctx, double* out, int n);
/* tuning knobs; unknown names and out-of-range values return HMK_STATUS_BAD_ARG.  None of them changes the result.
 *   batch      phase-1 queries per batch (0 = automatic: 8 profile tiles, at most 512 and what the resolver's
 *              shared memory holds)
 *   kb         partner candidates kept per query (1..32, default 8)
 *   capq       initial capacity of the per-query cluster-candidate arrays (grown on demand)
 *   lookahead  batches prepared ahead on a side stream while batch i is resolved: 0, 1 or 2 (default 2)
 *   filter     1 = upper-bound filter + exact verify kernel where it applies (default), 0 = exact kernel only
 *   reuse      1 = phase 2 takes its founder hits from the phase-1 partner searches when the matrix is
 *              symmetric (default), 0 = always run the separate founder pass
 *   qt, waves  profiles per shared-memory tile (0 = as many as fit), grid waves per launch
 *   reserve    SMs the look-ahead bulk launches leave free for the main stream (resolver + small kernels; default 4)
 *   min_iters, bucket_aux   static grids: block iterations per stripe at least; mixed lengths: per-length launches on separate streams
 *   persistent  1 = the filter kernel runs as one CTA per SM taking database chunks dynamically (default), 0 = static grid
 *   p2_chunk, p2_window, hit_cap   phase-2 chunking / window size / initial hit-buffer size
 *   p2_first   queries in the first phase-2 window (0 = automatic; later windows grow towards p2_window)
 *   xhit_cap   entries of the buffer that keeps the phase-1 hits for phase 2 (0 = automatic: what the last run on this
 *              context needed, else 96 per sequence); an overflow is reported in hmk_stats.flags
 *   force_generic  1 = scalar kernel for everything (correctness path)
 *   clinkage_dense_max  complete linkage: largest n that keeps the dense n x n score matrix (0..32768, default 32768);
 *              larger inputs take the sparse path
 *   clinkage_threads  complete linkage, sparse path: threads of the chain kernel (0 = automatic from the mean row length,
 *              else a multiple of 32 up to 1024)
 *   graph_cap  hmk_score_graph: pairs scoring >= threshold one batch of query rows may hold on the device (0 = automatic,
 *              4 194 304; never fewer than n); a batch with more is split
 *   profile    1 = time every bulk launch with CUDA events (hmk_stats.bulk_kernel_ms) */
int hmk_set_option(hmk_ctx* ctx, const char* name, int64_t value);

/* SequenceScorer.sequenceScore over a block of pairs (SequenceScorer.java:12-15,
 * ShiftedScorer.java:97-100): scores[a * n_second + b] = sequenceScore(seq1 = first_ids[a],
 * seq2 = second_ids[b]) for the uploaded sequences.  Used by the parity tests of the kernel. */
int hmk_score_block(hmk_ctx* ctx, const int32_t* first_ids, int32_t n_first, const int32_t* second_ids,
                    int32_t n_second, int32_t* scores, char* errbuf, size_t errlen);

/* One edge of the score graph: scoreWithShift(seq1 = partner, seq2 = seq) = (score, shift), seq < partner. */
typedef struct {
    int32_t seq, partner, score, shift;
} hmk_graph_edge;

/* The score graph of the uploaded sequences: every pair seq < partner (ids in upload order) whose
 * AligningSequenceScorer.scoreWithShift(seq1 = partner, seq2 = seq) (ShiftedScorer.java:48-95) reaches the threshold,
 * with that score and shift (the lowest winning diagonal, negated when seq1 is the shorter sequence), ordered by seq,
 * then partner.  For a symmetric matrix these are the pairs complete linkage keeps; an asymmetric matrix is accepted.
 * Paged pull: cursor = {i, r} continues at row i (the edges with seq == i) after its first r edges; {0, 0} starts.  The call
 * writes min(cap, remaining) edges to out, *n_out = their number, and advances the cursor; {n, 0} means done.  Every valid
 * cursor gives the same suffix, so a host may restart from a saved one.  A cursor that continues the previous call reuses
 * the batch of rows kept on the device; any other cursor scores the rows from its row on again.  Device memory stays
 * bounded by one batch (option graph_cap).  Status: HMK_STATUS_SHIFT_TOO_BIG when n >= 2 and max_shift >= the shortest
 * length, HMK_STATUS_BAD_RESIDUE, HMK_STATUS_BAD_ARG for a call before hmk_upload, a negative cap, a negative cursor,
 * i > n, or r beyond row i's length.  n of 0 or 1: an empty graph. */
int hmk_score_graph(hmk_ctx* ctx, int64_t cursor[2], hmk_graph_edge* out, int64_t cap, int64_t* n_out, char* errbuf,
                    size_t errlen);
/* AligningSequenceScorer.scoreWithShift for arbitrary pairs of the uploaded sequences, on the GPU:
 * (scores[e], shifts[e]) = scoreWithShift(seq1 = seq1_ids[e], seq2 = seq2_ids[e]).  Status: HMK_STATUS_SHIFT_TOO_BIG when
 * max_shift >= the shorter length of some pair, HMK_STATUS_BAD_RESIDUE, HMK_STATUS_BAD_ARG for ids out of range or a
 * call before hmk_upload. */
int hmk_score_pairs(hmk_ctx* ctx, const int32_t* seq1_ids, const int32_t* seq2_ids, int32_t n_pairs, int32_t* scores,
                    int32_t* shifts, char* errbuf, size_t errlen);

/* Nearest partners: for each row i in [row_begin, row_begin + n_rows) of the uploaded sequences (ids in upload order), the
 * k best-scoring other sequences j with s = scoreWithShift(seq1 = j, seq2 = i).score >= threshold (the partner search's
 * argument order), ordered by (s desc, abundance[j] desc, j asc) -- the partner search's candidate order, for any order
 * of the abundances.  partner, score and shift are [n_rows][k], row-major: entry r of row i is its (r + 1)-th partner
 * with that score and its shift (the lowest winning diagonal, negated when seq1 is the shorter sequence); slots past
 * count[i - row_begin] hold partner -1, score 0, shift 0.  more[i - row_begin] = 1 when more than k sequences qualify.
 * For j > i an entry is the score graph's edge (i, j); with a symmetric matrix every score equals the graph's.  An
 * asymmetric matrix is accepted.  Rows are independent and the call keeps no state, so a host may bound its memory by
 * pulling row ranges, or split the rows over contexts.  Option kb does not apply.  Status: HMK_STATUS_SHIFT_TOO_BIG when
 * n >= 2 and max_shift >= the shortest length, HMK_STATUS_BAD_RESIDUE, HMK_STATUS_BAD_ARG for a call before hmk_upload,
 * k outside 1 .. HMK_NEAREST_MAX_K, a row range outside [0, n], or a null output with n_rows > 0.  n of 0 or 1: empty
 * lists. */
#define HMK_NEAREST_MAX_K 31
int hmk_nearest(hmk_ctx* ctx, int32_t k, int32_t row_begin, int32_t n_rows, int32_t* partner, int32_t* score,
                int32_t* shift, int32_t* count, int32_t* more, char* errbuf, size_t errlen);

/* One bulk scoring launch over the uploaded sequences with the context's scheme and options.  Used by the kernel tests.
 * Profile side: query_ids[0 .. n_query), as seq2.  Thread side (seq1): db_ids[0 .. n_db), or with db_ids NULL the ids
 * db_begin .. db_begin + n_db - 1.  clustered (optional, one byte per uploaded sequence): non-zero items are skipped.
 *   mode 0, partner search: a thread-side id qualifies for query t when it is > query_ids[t] and scores >= threshold.
 *     keys[t * kb ..] (kb = option kb) = the merged best-hit list in descending key order (score, then the tie-break rank
 *     (abundance desc, id asc)), counts[t] = its length, overflow[t] = 1 when more than kb ids qualified.  hits receives
 *     every qualifying hit as (query id, thread-side id, score).
 *   mode 1, hits: hits receives every pair scoring >= threshold as (query index, thread-side id, score).
 * hits holds hit_cap triples; *hit_count = the hits the kernel found (may exceed hit_cap; then hit_cap are stored).
 * kernel[5] = the kernel that ran: kind (0 hmk_bulk_generic, 1 hmk_bulk_fast, 2 hmk_bulk_filter, 3 hmk_bulk_long; -1 when
 * n_query or n_db is 0 and nothing was launched), hmk_bulk_filter's compile-time length (12 or 0; else -1), 32-bit words
 * per profile entry, lane bits (32: generic; 0: nothing launched), persistent grid (1) or static grid (0). */
int hmk_bulk_probe(hmk_ctx* ctx, int32_t mode, const int32_t* query_ids, int32_t n_query, const int32_t* db_ids,
                   int32_t db_begin, int32_t n_db, const uint8_t* clustered, uint64_t* keys, int32_t* counts,
                   int32_t* overflow, int32_t* hits, int64_t hit_cap, int64_t* hit_count, int32_t* kernel, char* errbuf,
                   size_t errlen);

/* What hmk_batch_probe returns.  Host arrays owned by the caller, sized for the nq it asks for (kb = option kb,
 * nw = (nq + 31) / 32, capq as passed or option capq); the first nq_out rows are filled, rows packed without padding. */
typedef struct {
    int32_t nq_out;      /* queries of the batch: the first nq singletons with id >= cur, fewer when fewer remain          */
    int32_t* qid;        /* [nq] their ids, ascending                                                                    */
    uint64_t* bk_key;    /* [nq][kb] merged partner lists over the later singletons, hmk_bulk_probe's key order          */
    int32_t* bk_cnt;     /* [nq] list lengths                                                                            */
    int32_t* bk_ovf;     /* [nq] 1 = more later singletons scored >= threshold than the list holds                      */
    int32_t* ib;         /* [nq][nq] ib[b][b2] = score(member = qid[b2], query = qid[b])                                 */
    uint32_t* ibm;       /* [nq][nw] bit b2 (word b2 / 32, bit b2 % 32): b2 < b and ib[b][b2] >= threshold              */
    uint32_t* ibm2;      /* [nq][nw] bits of ibm whose ib also reaches the lowest score of b's list (none: empty list)   */
    int32_t* pcand;      /* [nq][kb] ids of the partner lists, padded with the query's own id                           */
    int32_t* pd;         /* [nq][nq * kb] pd[b][e] = score(member = pcand[e], query = qid[b])                             */
    int32_t* fhits;      /* [fhit_cap][3] founder hits: (query index, founder id, score >= threshold)                    */
    int64_t fhit_cap;
    int64_t fhit_count;  /* founder hits found (may exceed fhit_cap; then fhit_cap are stored)                           */
    int32_t* ac_cnt;     /* [nq] clusters whose founder hit and every other member score >= threshold (may exceed capq) */
    int32_t* ac_slot;    /* [nq][capq] the first min(ac_cnt, capq) of them, in no particular order                       */
    int32_t* ac_score;   /* [nq][capq] their complete-linkage score: the minimum over all members                        */
    int32_t* ac_best;    /* [nq][4] the best of them as (score, abundance-weighted size, founder id, cluster); -1: none  */
    /* kernels that ran: [0..4] the partner search as hmk_bulk_probe's kernel[5], [5] partner-search launches (one per
     * length bucket with later singletons on mixed lengths), [6] kind of the bulk kernel that made ib and pd (-1: the
     * one-thread-per-pair hmk_dense_packed), [7] its launches, [8] kind of the founder filter (-1: none ran), [9] its
     * launches, [10] scorer of the member check: 0 hmk_state_score, 1 hmk_packed_pair_score, 2 hmk_score12x3, -1 none */
    int32_t kernel[11];
} hmk_batch_probe_out;

/* Phase 1's per-batch work on a given clustering state, for the kernel tests.  Writes the state into the context --
 * members[member_off[c] .. member_off[c + 1]) are cluster c's members in chain order, founder first, for ncl <=
 * max_clusters clusters; every other sequence is a singleton -- with cur as the first unvisited id.  Then runs what a
 * run runs for one batch: the partner search with its tail (merged lists, score tables and masks) and the founder filter
 * on one stream (tail_stream 0) or the tail on a second stream (tail_stream 1), then the member check and the candidate
 * records.  capq: rows of the candidate arrays per query (0 = option capq).  A later hmk_run starts from a clean state.
 * Unlike a run, the bulk launches are planned for every SM (a run's look-ahead leaves some to the resolver), and
 * tail_stream 1 always puts the tail on the tail stream (a run's look-ahead does so on the packed paths; on the generic
 * path it stages a whole batch on one side stream). */
int hmk_batch_probe(hmk_ctx* ctx, const int32_t* member_off, const int32_t* members, int32_t ncl, int32_t cur, int32_t nq,
                    int32_t capq, int32_t tail_stream, hmk_batch_probe_out* out, char* errbuf, size_t errlen);

#ifdef __cplusplus
}
#endif
#endif
