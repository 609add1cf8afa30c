// hmk_common.h -- shared host/device primitives of the B200 greedy-clustering engine.
//
// Compiles under nvcc (device + host) and under plain g++.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HMK_HD __host__ __device__ __forceinline__
#else
#define HMK_HD inline
#endif

// -DHMK_CHECKED (hammock_b200.build.build(defines=["HMK_CHECKED"], out=...)): in-kernel bounds assertions at every write
// whose index comes from an atomic counter, a scheduler or decoded data.  A failing device assert prints file:line and
// makes the launch fail (cudaErrorAssert -> HMK_STATUS_CUDA).  Compiled out otherwise: the default build's SASS is
// identical with and without these lines.  (compute-sanitizer is not available on the target pool.)
#if defined(HMK_CHECKED) && defined(__CUDACC__)
#include <assert.h>
#define HMK_CHECK(cond) assert(cond)
#else
#define HMK_CHECK(cond) ((void)0)
#endif

#define HMK_NRES 24
#define HMK_JMIN ((int32_t)0x80000000)
#define HMK_JMAX ((int32_t)0x7fffffff)

// Java int arithmetic wraps
HMK_HD int32_t hmk_wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
HMK_HD int32_t hmk_wmul(int32_t a, int32_t b) { return (int32_t)((uint32_t)a * (uint32_t)b); }

// Scalar gapless all-offset score S(seq1, seq2) == ShiftedScorer.sequenceScore(seq1, seq2)
// (reference ShiftedScorer.java:48-100).  seq1 = member of the database cluster, seq2 = the
// compared (query) sequence at every call site of the greedy path
// (ClinkageClusterScorer.java:38).  Formulated per diagonal k = (position in longer) -
// (position in shorter); equal lengths make the SECOND argument the "shorter" one.
// Requires max_shift < shorter length (checked by the caller -> status 1).
// `st1` / `st2`: element strides of the two residue arrays (1 = contiguous; the generic bulk kernel keeps the thread-side
// sequences position-major in shared memory, stride = block size).
// `shift` (may be NULL; the callers that only want the score pass NULL and compile to the score-only loop) receives
// what ShiftedScorer.scoreWithShift reports (:86-93): the lowest diagonal reaching the best score, negated when seq1 is
// the shorter sequence.
HMK_HD int32_t hmk_pair_score_strided(const uint8_t* seq1, int st1, int len1, const uint8_t* seq2, int st2, int len2,
                                      const int32_t* M, int X, int P, int* shift = nullptr) {
    const uint8_t* s;
    const uint8_t* l;
    int ls, ll, ss, sl;
    if (len1 >= len2) { s = seq2; ls = len2; ss = st2; l = seq1; ll = len1; sl = st1; }
    else              { s = seq1; ls = len1; ss = st1; l = seq2; ll = len2; sl = st2; }
    const int d = ll - ls;
    int32_t best = HMK_JMIN;
    int best_k = 0;
    for (int k = -X; k <= X + d; k++) {
        // longer index j pairs with shorter index j-k
        int j0 = k > 0 ? k : 0;
        int j1 = ls + k < ll ? ls + k : ll;
        int32_t sc = 0;
        for (int j = j0; j < j1; j++) sc = hmk_wadd(sc, M[s[(j - k) * ss] * HMK_NRES + l[j * sl]]);
        sc = hmk_wadd(sc, hmk_wmul(d, P));
        if (k < 0) sc = hmk_wadd(sc, hmk_wmul(-2 * k, P));
        if (k > d) sc = hmk_wadd(sc, hmk_wmul(2 * (k - d), P));
        if (sc > best) { best = sc; best_k = k; }
    }
    if (shift) *shift = len1 >= len2 ? best_k : -best_k;
    return best;
}
HMK_HD int32_t hmk_pair_score(const uint8_t* seq1, int len1, const uint8_t* seq2, int len2,
                              const int32_t* M, int X, int P) {
    return hmk_pair_score_strided(seq1, 1, len1, seq2, 1, len2, M, X, P);
}
// ShiftedScorer.scoreWithShift(seq1, seq2) (ShiftedScorer.java:48-95, AligningScorerResult = score + shift)
HMK_HD int32_t hmk_score_with_shift(const uint8_t* seq1, int len1, const uint8_t* seq2, int len2,
                                    const int32_t* M, int X, int P, int* shift) {
    return hmk_pair_score_strided(seq1, 1, len1, seq2, 1, len2, M, X, P, shift);
}

// cells / shifts summed by one pair score (SURVEY.md 3.2) -- work accounting only
HMK_HD int64_t hmk_pair_cells(int len1, int len2, int X) {
    int ls = len1 < len2 ? len1 : len2, ll = len1 < len2 ? len2 : len1;
    int d = ll - ls;
    int64_t cells = 0;
    for (int k = -X; k <= X + d; k++) {
        int j0 = k > 0 ? k : 0;
        int j1 = ls + k < ll ? ls + k : ll;
        if (j1 > j0) cells += j1 - j0;
    }
    return cells;
}

// Best-hit key for the singleton (partner) search: bigger key == preferred candidate under
// NearestClusterRunner's order (score desc, size desc, id asc;
// ClinkageSequenceClusterer.java:258-293).  `tierank` is the candidate's rank under
// (abundance desc, id asc); it equals the id when the input is abundance-sorted.
HMK_HD uint64_t hmk_key_make(int32_t score, uint32_t tierank) {
    return ((uint64_t)((uint32_t)score ^ 0x80000000u) << 32) | (uint64_t)(uint32_t)(~tierank);
}
HMK_HD int32_t hmk_key_score(uint64_t key) { return (int32_t)((uint32_t)(key >> 32) ^ 0x80000000u); }
HMK_HD uint32_t hmk_key_rank(uint64_t key) { return ~(uint32_t)key; }

// ---------------------------------------------------------------- packed sequences (<= 12 residues per 64-bit word)
// 5 bits per residue, position j in bits 5j..5j+4; one-word sequences carry their length in bits 60..63.
// Host + device so that the CPU tests can run them against the oracle (tests/cpp/common_shim.cpp).
#define HMK_MAXL1 12           // residues per 64-bit packed word
#if defined(__CUDACC__)
#define HMK_UNROLL _Pragma("unroll")
#else
#define HMK_UNROLL
#endif

// S(seq1 = member, seq2 = query) from two packed words that carry their lengths (<= 12 residues each): the reference's
// roles (ShiftedScorer.java:51-57: the shorter sequence slides, equal lengths make seq2 the shorter one) and orientation
// M[shorter][longer] (:71,75,110), Java-int arithmetic.
HMK_HD int32_t hmk_packed_pair_score(uint64_t w1, uint64_t w2, const int32_t* sM, int X, int P) {
    const int len1 = (int)(w1 >> 60), len2 = (int)(w2 >> 60);
    uint64_t ws, wl;
    int ls, ll;
    if (len1 >= len2) { ws = w2; ls = len2; wl = w1; ll = len1; }
    else              { ws = w1; ls = len1; wl = w2; ll = len2; }
    const int d = ll - ls;
    int32_t best = HMK_JMIN;
    for (int k = -X; k <= X + d; k++) {
        const int j0 = k > 0 ? k : 0, j1 = ls + k < ll ? ls + k : ll;      // longer index j pairs with shorter index j - k
        int32_t v = 0;
        for (int j = j0; j < j1; j++) {
            const uint32_t rs = (uint32_t)(ws >> (5 * (j - k))) & 31u, rl = (uint32_t)(wl >> (5 * j)) & 31u;
            v = hmk_wadd(v, sM[rs * HMK_NRES + rl]);
        }
        v = hmk_wadd(v, hmk_wmul(d, P));
        if (k < 0) v = hmk_wadd(v, hmk_wmul(-2 * k, P));
        if (k > d) v = hmk_wadd(v, hmk_wmul(2 * (k - d), P));
        if (v > best) best = v;
    }
    return best;
}

// S(member, query) with both sequences given as packed words: uniform length 12, max shift 3, matrix in shared memory.
// qrow[j] = 24 * (query residue j).  77 x (address add + LDS + accumulate); when a warp scores 32 members against ONE
// query, the loads of a step hit one matrix row (conflict free).
HMK_HD int32_t hmk_score12x3(const int32_t (&qrow)[HMK_MAXL1], uint64_t wm, const int32_t* sM, int32_t P) {
    int32_t rm[HMK_MAXL1];
HMK_UNROLL
    for (int j = 0; j < HMK_MAXL1; j++) rm[j] = (int32_t)((uint32_t)(wm >> (5 * j)) & 31u);
    int32_t best = HMK_JMIN;
HMK_UNROLL
    for (int k = -3; k <= 3; k++) {       // equal lengths: shorter = query (second argument), ShiftedScorer.java:51-57
        int32_t v = 2 * (k < 0 ? -k : k) * P;
HMK_UNROLL
        for (int j = 0; j < HMK_MAXL1; j++)
            if (j - k >= 0 && j - k < HMK_MAXL1) v += sM[qrow[j - k] + rm[j]];
        best = v > best ? v : best;
    }
    return best;
}
HMK_HD void hmk_qrow12(uint64_t wq, int32_t (&qrow)[HMK_MAXL1]) {
HMK_UNROLL
    for (int j = 0; j < HMK_MAXL1; j++) qrow[j] = (int32_t)((uint32_t)(wq >> (5 * j)) & 31u) * HMK_NRES;
}

// Residue prefix shared by a warp's items (hmk_bulk_filter).  The filter bound is a u32 sum over positions, so where
// every scored lane of a warp holds the same residues 0 .. HMK_PREFIX_RES - 1, their rows are summed once per query for
// the warp instead of once per lane.  The warp reduces the lanes' prefix keys to their least (hmk_prefix_lo) and
// greatest (hmk_prefix_hi) value; a lane whose item is not scored adds the neutral value of each reduction, so the two
// agree exactly when the scored lanes share the prefix, and never for a warp without a scored lane.
#define HMK_PREFIX_RES 3
HMK_HD uint32_t hmk_prefix_key(uint64_t w) { return (uint32_t)w & ((1u << (5 * HMK_PREFIX_RES)) - 1u); }
HMK_HD uint32_t hmk_prefix_lo(uint64_t w, bool scored) { return scored ? hmk_prefix_key(w) : 0xffffffffu; }
HMK_HD uint32_t hmk_prefix_hi(uint64_t w, bool scored) { return scored ? hmk_prefix_key(w) : 0u; }
// residues shared (HMK_PREFIX_RES or 0) given kmin = min over the warp of hmk_prefix_lo, kmax = max of hmk_prefix_hi
HMK_HD int hmk_prefix_shared(uint32_t kmin, uint32_t kmax) { return kmin == kmax ? HMK_PREFIX_RES : 0; }

// status codes of the engine / C ABI (include/hammock_b200.h)
enum {
    HMK_OK = 0,
    HMK_ERR_SHIFT_TOO_BIG = 1,  // DataException "Shift too big" (ShiftedScorer.java:59-62)
    HMK_ERR_NULL_CLUSTER = 2,   // NullPointerException (LimitedGreedySequenceClusterer.java:104,108)
    HMK_ERR_BAD_RESIDUE = 3,    // residue code >= 24 (UniqueSequence.java:51-54)
    HMK_ERR_CUDA = 4,           // CUDA / NCCL failure; there is no CPU fallback
    HMK_ERR_BAD_ARG = 5
};

// phase-1 resolver exit reasons (device -> host, per batch)
enum {
    HMK_P1_CONTINUE = 0,  // batch fully consumed, more work
    HMK_P1_DONE = 1,      // K clusters reached or list exhausted
    HMK_P1_NPE = 2,       // reference would throw NullPointerException at this step
    HMK_P1_RESTART = 3,   // partner list exhausted but truncated: rescore from ctl.cur
    HMK_P1_GROW = 4,      // per-query cluster-candidate arrays too small: grow and rescore from ctl.cur
    HMK_P1_GROWHITS = 5   // the founder-hit buffer of the cluster search was too small (needed size in ctl.pad0): redo it
};

struct HmkCtl {
    int32_t cur;           // first id not yet visited by phase 1
    int32_t ncl;           // multi-member clusters so far (actualClusters.size())
    int32_t unproc_alive;  // initialList.size() - index
    int32_t status;        // HMK_P1_*
    int32_t npe_step;
    int32_t steps, joins, creates, orphans;
    int32_t restarts;
    int32_t pad0, pad1;
    int32_t discards;      // resolver exits that threw the prepared batches away (any status but CONTINUE / GROWHITS)
    int32_t pad2;
    int64_t scalar_pairs;  // pair scores computed one at a time (resolvers, member checks)
    int64_t scalar_cells;
    int64_t dbg[8];        // resolver cycle counters (only filled when built with -DHMK_RESOLVE_TIMING)
    int64_t cnt[4];        // resolver statistics: windows tried, steps they applied, sequential steps
};
