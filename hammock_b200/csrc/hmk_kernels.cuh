// hmk_kernels.cuh -- sm_100a kernels of the greedy-clustering engine.
//
// Hot kernel: hmk_bulk_filter<MODE, LT>, the partner search and founder filter on sequences of
// <= 12 residues; it screens pairs with an upper-bound table and re-scores the survivors with
// the exact scheme of hmk_bulk_fast<NW, MODE>.  There one thread owns one database peptide
// (5-bit packed, one 64-bit word, <= 12 residues) and scores it against a tile of "profile"
// sequences held in shared memory.  A profile is the substitution matrix pre-arranged per diagonal:
// entry[h][j][r] (32 bit) holds, for database position j carrying residue r, the
// contributions to 4 (u8 lanes) or 2 (s16 lanes) of the 2X+1 shift diagonals.  One pair score
// = L x NW conflict-free LDS.32 + 3-input adds on packed lanes; lanes are biased so that
// "score >= threshold" is the lane's top bit, i.e. the common path ends in a single
// LOP3/branch and only hits (rare) are decoded.  This replaces the reference's scalar
// triple loop (ShiftedScorer.java:67-90) and the per-candidate ClinkageClusterScorer call
// (ClinkageClusterScorer.java:30-49) for all candidates of a batch at once.
//
// Profile tiles are staged global->shared with the TMA bulk-copy engine
// (cp.async.bulk + mbarrier; SASS UBLKCP).
#pragma once
#include <cooperative_groups.h>
#include <type_traits>
#include <cuda_runtime.h>
#include <stdint.h>

#include "hmk_common.h"
#include "hmk_resolve.h"

#define HMK_MAXLEN 36          // longest sequence the packed kernels take (three words)
#define HMK_NWMAX 10           // most 32-bit words per profile entry (long kernel)
#define HMK_LONG_THREADS 512
#define HMK_FPW 868            // words per profile with the filter sub-table: 3 x 288 + 4 (the +16 B skews the tables over the banks)
#define HMK_FILTER_QT 56       // filter kernel: most profiles per tile (Engine::qt_max)
#define HMK_FGROUP 32          // filter kernel: queries whose filter results one lane keeps as bits before they are handed out
                               // (four octets of one 32-bit mask per exact word; the kernel relies on 32)
#ifndef HMK_BULK_THREADS
#define HMK_BULK_THREADS 768
#endif

enum { HMK_MODE_TOPK = 0, HMK_MODE_EMIT = 1, HMK_MODE_DENSE = 2 };
enum { HMK_PROF_QUERY = 0, HMK_PROF_MEMBER = 1 };

// ---------------------------------------------------------------- scoring scheme
struct HmkScheme {
    int32_t L;        // uniform sequence length of the fast path
    int32_t X, P, T;
    int32_t nw;       // 32-bit words per profile entry
    int32_t lane16;   // 0: four u8 lanes per word, 1: two s16 lanes per word
    int32_t bias;     // added to every valid cell so entries are >= 0
    int32_t half;     // 128 or 32768: lane value >= half  <=>  score >= T
    int32_t prof_words;  // one word: nw * HMK_MAXL1 * 24 (fixed row stride so LDS offsets are immediates); long: nw * L * 24
    int32_t words;       // 64-bit words per packed sequence (1..3)
    int32_t long_layout; // 0: prof[t][h][j][r] for hmk_bulk_fast, 1: prof[t][j][h][r] for hmk_bulk_long
    int32_t filter;      // 1: u8 lanes, nw == 2, and a third sub-table with pair-of-diagonals upper bounds (HMK_FPW words per profile)
};

// ---------------------------------------------------------------- profile builder
// prof[t][h][j][r] with j < HMK_MAXL1 (rows j >= n are zero), for THREAD-side sequences of length
// n = sc.L and a profile sequence p of length m (read per profile, so batches may mix lengths).
// Reference roles (ShiftedScorer.java:51-57): the shorter sequence is "s", the longer "l", equal
// lengths make seq2 the shorter one; d = |n - m|; shifts k = -X .. X+d; matrix index
// M[shorter][longer] (:71,75,110).
//   mode QUERY : profile = seq2 (compared sequence), threads carry seq1 (member / candidate)
//   mode MEMBER: profile = seq1 (member),            threads carry seq2 (query)
// profile is the shorter one ("ps") iff m <= n (QUERY) resp. m < n (MEMBER):
//   ps : thread position j is l[j]   -> lane k gets M[p[j-k]][r], valid 0 <= j-k < m
//   !ps: thread position i is s[i]   -> lane k gets M[r][p[i+k]], valid 0 <= i+k < m
// Lane k's constant (added at position 0): penalties + (half - T) - cells_k * bias, so that
// lane value >= half  <=>  score_k >= T.
__global__ void hmk_build_profiles(HmkScheme sc, int mode, const int32_t* __restrict__ ids, int nq,
                                   const uint8_t* __restrict__ res, const int32_t* __restrict__ off,
                                   const int32_t* __restrict__ M, uint32_t* __restrict__ prof,
                                   uint32_t* __restrict__ prof_cells, uint32_t* __restrict__ prof_ops) {
    __shared__ int32_t sM[HMK_NRES * HMK_NRES];
    __shared__ uint8_t sp[HMK_MAXLEN];
    const int t = blockIdx.x;
    if (t >= nq) return;
    for (int i = threadIdx.x; i < HMK_NRES * HMK_NRES; i += blockDim.x) sM[i] = M[i];
    const int32_t id = ids[t];
    const int m = off[id + 1] - off[id], n = sc.L;
    if (threadIdx.x < m && threadIdx.x < HMK_MAXLEN) sp[threadIdx.x] = res[off[id] + threadIdx.x];
    __syncthreads();
    const bool ps = mode == HMK_PROF_QUERY ? (m <= n) : (m < n);
    const int ls = m < n ? m : n, ll = m < n ? n : m, d = ll - ls;
    const int lanes_per_word = sc.lane16 ? 2 : 4, lane_bits = sc.lane16 ? 16 : 8;
    uint32_t* out = prof + (size_t)t * sc.prof_words;
    for (int e = threadIdx.x; e < sc.prof_words; e += blockDim.x) {
        const int r = e % HMK_NRES;
        const int j = sc.long_layout ? e / (HMK_NRES * sc.nw) : (e / HMK_NRES) % HMK_MAXL1;
        const int h = sc.long_layout ? (e / HMK_NRES) % sc.nw : e / (HMK_NRES * HMK_MAXL1);
        uint32_t word = 0;
        if (j >= n || h > sc.nw || (h == sc.nw && !sc.filter)) { out[e] = 0; continue; }
        // value of lane `lam` at (j, r): biased cell + (at position 0) the lane constant
        auto lane_val = [&](int lam) -> int32_t {
            if (lam > 2 * sc.X + d) return 0;
            const int k = lam - sc.X;
            int32_t val = 0;
            const int pi = ps ? j - k : j + k;
            if (pi >= 0 && pi < m) val = (ps ? sM[sp[pi] * HMK_NRES + r] : sM[r * HMK_NRES + sp[pi]]) + sc.bias;
            if (j == 0) {
                const int cells = (ls + k < ll ? ls + k : ll) - (k > 0 ? k : 0);
                const int pen = d * sc.P + (k < 0 ? -2 * k * sc.P : 0) + (k > d ? 2 * (k - d) * sc.P : 0);
                val += pen + sc.half - sc.T - cells * sc.bias;
            }
            return val;
        };
        if (h < sc.nw) {
            for (int b = 0; b < lanes_per_word; b++)
                word |= ((uint32_t)lane_val(h * lanes_per_word + b) & ((1u << lane_bits) - 1u)) << (b * lane_bits);
        } else {
            // filter sub-table (u8): byte g bounds the lanes of group g from above (max per position, so the
            // sum bounds every lane's sum): "no filter byte reaches 128" proves "no diagonal reaches T".
            // Positions outside a diagonal count as score 0 here (value `bias`, the lane constant is
            // reduced to match) -- with 0 there, the maximum would pick up the neighbour's real cell.
            // One length only (d == 0).  Group g = lanes 2g, 2g+1: bytes 0,1 bound exact word 0, bytes 2,3 word 1.
            const int nl = 2 * sc.X + 1;
            for (int g = 0; g < 4; g++) {
                const int l0 = 2 * g, l1 = l0 + 1 < nl ? l0 + 1 : nl - 1;
                int32_t best = 0;
                for (int lam = l0; lam <= l1; lam++) {
                    const int k = lam - sc.X;
                    const int pi = ps ? j - k : j + k;
                    int32_t val = sc.bias;
                    if (pi >= 0 && pi < m) val += ps ? sM[sp[pi] * HMK_NRES + r] : sM[r * HMK_NRES + sp[pi]];
                    if (j == 0) val += 2 * sc.P * (k < 0 ? -k : k) + sc.half - sc.T - n * sc.bias;
                    best = val > best ? val : best;
                }
                word |= ((uint32_t)best & 0xffu) << (8 * g);
            }
        }
        out[e] = word;
    }
    if (threadIdx.x == 0 && prof_cells) {   // work accounting (SURVEY.md 8d): cells and cells + shifts of one pair
        prof_cells[t] = (uint32_t)hmk_pair_cells(m, n, sc.X);
        prof_ops[t] = prof_cells[t] + (uint32_t)(2 * sc.X + d + 1);
    }
}

// ---------------------------------------------------------------- TMA bulk copy helpers
__device__ __forceinline__ uint32_t hmk_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void hmk_mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(hmk_smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void hmk_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(hmk_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void hmk_bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     hmk_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(hmk_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void hmk_mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(ok)
            : "r"(hmk_smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!ok);
    // lanes leave the spin loop (and may have been suspended in try_wait) at different times; everything that
    // follows uses warp-wide primitives, so re-converge here.  Always called by whole warps.  Without this the
    // resolver dead-locked at a later __syncwarp on some inputs.
    __syncwarp();
}

// every warp adds its pair-score count once; one address for all of them serialises in L2, so the counter is sharded
#define HMK_PAIR_SHARDS 64
__device__ __forceinline__ void hmk_count_pairs(unsigned long long* parts, long long n) {
    if (n) atomicAdd(parts + (size_t)((blockIdx.x * 8 + (threadIdx.x >> 5)) % HMK_PAIR_SHARDS) * 16, (unsigned long long)n);
}

// ---------------------------------------------------------------- bulk arguments
struct HmkBulkArgs {
    HmkScheme sc;
    // profile side
    const uint32_t* prof;      // [nq][prof_words]
    int32_t nq, qt, nqt;       // profiles, profiles per tile, tiles
    // thread side ("database")
    const uint64_t* packed;    // by sequence id
    const int32_t* db_ids;     // NULL: id = db_begin + i
    int32_t db_begin, ndb;
    int32_t nstripes, chunk;   // items per stripe
    int32_t stripe_base;       // first slot of this launch in tk_* (several launches, e.g. one per length, share a merge)
    const int32_t* slot;       // non-NULL: skip items whose slot >= 0 (no longer singletons)
    const int32_t* q_minid;    // non-NULL: only ids > q_minid[t] qualify (initialList[index+1..])
    const int32_t* tierank;    // NULL: tierank == id
    // MODE_TOPK
    int32_t kb;
    uint64_t* tk_key;          // [nstripes][nq][kb] descending
    int32_t* tk_cnt;           // [nstripes][nq]
    int32_t* tk_ovf;           // [nstripes][nq]
    unsigned long long* tk_gmin;   // optional [nq], zeroed: lower bound of the kb-th best key over ALL stripes (published by
                                   // every CTA whose list is full) -- hits below it cannot reach the merged list
    // MODE_TOPK, optional: every qualifying hit is also appended here for phase 2 (see Engine::phase2)
    int4* xhits;               // (profile-side sequence id, thread-side sequence id, score, xbatch)
    unsigned long long* xhit_count;
    unsigned long long xhit_cap;
    int32_t xbatch;
    // MODE_EMIT
    int4* hits;                // (profile index, thread-side sequence id, score, 0)
    unsigned int* hit_count;
    unsigned int hit_cap;
    // MODE_DENSE
    int32_t* dense;            // dense[t * dense_stride + i]
    int32_t dense_stride;
    unsigned long long* pair_counter;   // [0] pairs, [1] cells, [2] int ops (the last two only with prof_cells)
    const uint32_t* prof_cells;         // per profile: cells of one pair against this launch's thread-side length
    const uint32_t* prof_ops;
    // persistent mode (hmk_bulk_filter): one CTA per SM, the database is cut into nchunks chunks of `chunk` items per
    // profile tile and CTAs take chunks dynamically -- sched[t] = next chunk of tile t, sched[nqt + t] = output slots
    // (CTA x tile engagements) handed out for tile t; nstripes = slots per query in tk_* (>= CTAs)
    int32_t* sched;
    int32_t nchunks;
    // optional, persistent mode: a phase-1 batch prepared ahead stops taking chunks once the resolver's discard counter
    // (HmkCtl::discards) differs from the value the host knew when it staged the batch -- its results are thrown away
    const int32_t* discards;
    int32_t discards_seen;
    const int32_t* ndb_dev;   // optional: the real number of thread-side items (<= ndb, which then only sizes the grid)
    int32_t db_min_id;        // generic kernel with a length-sorted id list: ids below this are not scored at all
};

// ---------------------------------------------------------------- hit handling
// The scoring loops are kept free of divergence: a hit (score >= T, rare) is only APPENDED to
// a per-warp queue in shared memory (slot = ballot rank, no atomics, no branches that split
// the warp for long); queues are drained by the whole warp at warp-uniform points.
#define HMK_QCAP 64   // entries per warp queue; drained when fewer than 32 slots remain

struct HmkTopkSmem {
    uint64_t* key;    // [qt][kb]
    uint64_t* minkey; // [qt]
    int* cnt;         // [qt]
    int* lock;        // [qt]
    int* ovf;         // [qt]
};

// A packed-path hit has T <= score <= T + (top - half) of its lanes, at most T + 32767 with 16-bit lanes, so the queue
// stores score - T as an unsigned 16-bit number (a signed 16-bit score would wrap above 32767).
struct HmkHitQueue {
    uint64_t* q;      // this warp's HMK_QCAP entries: (tile-local query << 48) | ((score - T) as u16 << 32) | item
    int32_t* s32;     // generic kernel only: full int32 scores (NULL on the packed path)
    int cnt;          // warp-uniform
};

__device__ __forceinline__ uint64_t hmk_hit_pack(int tl, uint32_t over, int32_t i) {
    return ((uint64_t)(uint32_t)tl << 48) | ((uint64_t)(uint16_t)over << 32) | (uint32_t)i;
}

// executed by ONE lane of a warp at a time (the others wait at a ballot), so the spin only
// ever contends with other warps
__device__ __forceinline__ void hmk_topk_insert_locked(const HmkTopkSmem& s, int t, int kb, uint64_t key, unsigned long long* gmin) {
    volatile uint64_t* keys = s.key + (size_t)t * kb;
    volatile uint64_t* mink = s.minkey + t;
    volatile int* cnt = s.cnt + t;
    while (atomicCAS(s.lock + t, 0, 1) != 0) {}
    __threadfence_block();
    int c = *cnt;
    HMK_CHECK(t >= 0 && c >= 0 && c <= kb);
    if (c < kb) {
        keys[c] = key;
        c++;
        if (c == kb) {
            uint64_t m = keys[0];
            for (int i = 1; i < kb; i++) { uint64_t v = keys[i]; m = v < m ? v : m; }
            *mink = m;
            if (gmin) atomicMax(gmin, (unsigned long long)m);
        }
        *cnt = c;
    } else {
        s.ovf[t] = 1;
        if (key > *mink) {
            int mi = 0;
            uint64_t m = keys[0];
            for (int i = 1; i < kb; i++) { uint64_t v = keys[i]; if (v < m) { m = v; mi = i; } }
            keys[mi] = key;
            m = keys[0];
            for (int i = 1; i < kb; i++) { uint64_t v = keys[i]; m = v < m ? v : m; }
            *mink = m;
            if (gmin) atomicMax(gmin, (unsigned long long)m);
        }
    }
    __threadfence_block();
    atomicExch(s.lock + t, 0);
}

// whole warp, converged
template <int MODE>
__device__ __noinline__ void hmk_queue_drain(const HmkBulkArgs& a, const HmkTopkSmem& tk, int q0, HmkHitQueue& hq) {
    const int lane = threadIdx.x & 31;
    const int n = hq.cnt;
    HMK_CHECK(n >= 0 && n <= HMK_QCAP);
    __syncwarp();
    if (MODE == HMK_MODE_EMIT) {
        unsigned int base = 0;
        if (lane == 0) base = atomicAdd(a.hit_count, (unsigned int)n);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int e = lane; e < n; e += 32) {
            const uint64_t v = hq.q[e];
            const unsigned int pos = base + e;
            const int32_t sc = hq.s32 ? hq.s32[e] : a.sc.T + (int32_t)(uint16_t)(v >> 32);
            const int32_t i = (int32_t)(uint32_t)v;
            HMK_CHECK(i >= 0 && i < a.ndb && (int)(v >> 48) < a.qt);
            const int32_t id = a.db_ids ? a.db_ids[i] : a.db_begin + i;
            if (pos < a.hit_cap) a.hits[pos] = make_int4(q0 + (int)(v >> 48), id, sc, 0);
        }
    } else if (MODE == HMK_MODE_TOPK) {
        for (int e0 = 0; e0 < n; e0 += 32) {
            const int e = e0 + lane;
            bool pending = false;
            int tl = 0;
            int32_t id = 0, sc = 0;
            uint64_t key = 0;
            if (e < n) {
                const uint64_t v = hq.q[e];
                tl = (int)(v >> 48);
                const int32_t i = (int32_t)(uint32_t)v;
                HMK_CHECK(i >= 0 && i < a.ndb && tl < a.qt && q0 + tl < a.nq);
                id = a.db_ids ? a.db_ids[i] : a.db_begin + i;
                sc = hq.s32 ? hq.s32[e] : a.sc.T + (int32_t)(uint16_t)(v >> 32);
                pending = !(a.q_minid && id <= a.q_minid[q0 + tl]);   // initialList[index+1 ..] only
            }
            if (a.xhits) {   // keep every qualifying hit for phase 2
                const unsigned xm = __ballot_sync(0xffffffffu, pending);
                if (xm) {
                    unsigned long long xb = 0;
                    const int leader = __ffs(xm) - 1;
                    if (lane == leader) xb = atomicAdd(a.xhit_count, (unsigned long long)__popc(xm));
                    xb = __shfl_sync(0xffffffffu, xb, leader);
                    if (pending) {
                        const unsigned long long pos = xb + __popc(xm & ((1u << lane) - 1u));
                        if (pos < a.xhit_cap) a.xhits[pos] = make_int4(a.q_minid[q0 + tl], id, sc, a.xbatch);
                    }
                }
            }
            if (pending) {
                const uint32_t rk = a.tierank ? (uint32_t)a.tierank[id] : (uint32_t)id;
                key = hmk_key_make(sc, rk);
                // cheap reject without the lock (minkey only grows once the list is full; tk_gmin is some
                // stripe's kb-th best key, so at least kb better hits exist)
                if ((a.tk_gmin && key < __ldcg(a.tk_gmin + q0 + tl)) ||
                    (*(volatile int*)(tk.cnt + tl) >= a.kb && key <= *(volatile uint64_t*)(tk.minkey + tl))) {
                    tk.ovf[tl] = 1;
                    pending = false;
                }
            }
            unsigned m;
            while ((m = __ballot_sync(0xffffffffu, pending)) != 0) {
                if (lane == __ffs(m) - 1) {
                    hmk_topk_insert_locked(tk, tl, a.kb, key, a.tk_gmin ? a.tk_gmin + q0 + tl : nullptr);
                    pending = false;
                }
            }
        }
    }
    __syncwarp();
    hq.cnt = 0;
}

// append this lane's hit (if any); must be called by the whole, converged warp
template <int MODE>
__device__ __forceinline__ void hmk_queue_push(const HmkBulkArgs& a, const HmkTopkSmem& tk, int q0, HmkHitQueue& hq,
                                               bool hit, int tl, int32_t score, int32_t i) {
    const unsigned m = __ballot_sync(0xffffffffu, hit);
    if (m) {
        const int lane = threadIdx.x & 31;
        if (hit) {
            const int pos = hq.cnt + __popc(m & ((1u << lane) - 1u));
            const uint32_t over = (uint32_t)score - (uint32_t)a.sc.T;   // 0 .. 0xffff on the packed path
            HMK_CHECK(pos >= 0 && pos < HMK_QCAP && (hq.s32 || over <= 0xffffu));
            hq.q[pos] = hmk_hit_pack(tl, over, i);
            if (hq.s32) hq.s32[pos] = score;
        }
        hq.cnt += __popc(m);
        if (hq.cnt > HMK_QCAP - 32) hmk_queue_drain<MODE>(a, tk, q0, hq);
    }
}

__device__ __forceinline__ int32_t hmk_lane_max(const uint32_t* acc, int nw, int lane16) {
    if (lane16) {
        uint32_t m = acc[0];
        for (int w = 1; w < nw; w++) m = __vmaxu2(m, acc[w]);
        uint32_t lo = m & 0xffffu, hi = m >> 16;
        return (int32_t)(lo > hi ? lo : hi);
    }
    uint32_t m = acc[0];
    for (int w = 1; w < nw; w++) m = __vmaxu4(m, acc[w]);
    uint32_t a = m & 0xffu, b = (m >> 8) & 0xffu, c = (m >> 16) & 0xffu, d = m >> 24;
    a = a > b ? a : b;
    c = c > d ? c : d;
    return (int32_t)(a > c ? a : c);
}

// common CTA prologue/epilogue for the top-k buffers
__device__ __forceinline__ void hmk_topk_init(const HmkTopkSmem& tk, int qn, int kb) {
    for (int i = threadIdx.x; i < qn; i += blockDim.x) { tk.cnt[i] = 0; tk.lock[i] = 0; tk.ovf[i] = 0; tk.minkey[i] = 0; }
}
__device__ __forceinline__ void hmk_topk_flush(const HmkBulkArgs& a, const HmkTopkSmem& tk, int q0, int qn, int stripe) {   // stripe = output slot
    HMK_CHECK(stripe >= 0 && stripe < a.nstripes && q0 >= 0 && q0 + qn <= a.nq);
    for (int t = threadIdx.x; t < qn; t += blockDim.x) {
        uint64_t* k = tk.key + (size_t)t * a.kb;
        int c = tk.cnt[t];
        for (int i = 1; i < c; i++) {   // insertion sort, descending
            uint64_t v = k[i];
            int j = i - 1;
            while (j >= 0 && k[j] < v) { k[j + 1] = k[j]; j--; }
            k[j + 1] = v;
        }
        size_t o = (size_t)(a.stripe_base + stripe) * a.nq + q0 + t;
        for (int i = 0; i < c; i++) a.tk_key[o * a.kb + i] = k[i];
        a.tk_cnt[o] = c;
        a.tk_ovf[o] = tk.ovf[t];
    }
}

// shared-memory carve-up behind the per-kernel payload (profiles / residues)
__device__ __forceinline__ void hmk_carve(unsigned char* p, int qt, int kb, bool wide, HmkTopkSmem& tk, HmkHitQueue& hq) {
    tk.key = reinterpret_cast<uint64_t*>(p);    p += (size_t)qt * kb * 8;
    tk.minkey = reinterpret_cast<uint64_t*>(p); p += (size_t)qt * 8;
    hq.q = reinterpret_cast<uint64_t*>(p) + (size_t)(threadIdx.x >> 5) * HMK_QCAP;
    p += (size_t)(blockDim.x >> 5) * HMK_QCAP * 8;
    hq.s32 = nullptr;
    if (wide) {
        hq.s32 = reinterpret_cast<int32_t*>(p) + (size_t)(threadIdx.x >> 5) * HMK_QCAP;
        p += (size_t)(blockDim.x >> 5) * HMK_QCAP * 4;
    }
    tk.cnt = reinterpret_cast<int*>(p);  p += (size_t)qt * 4;
    tk.lock = reinterpret_cast<int*>(p); p += (size_t)qt * 4;
    tk.ovf = reinterpret_cast<int*>(p);
    hq.cnt = 0;
}
__host__ __device__ inline size_t hmk_carve_bytes(int qt, int kb, int threads, bool wide) {
    return (size_t)qt * kb * 8 + (size_t)qt * 8 + (size_t)(threads / 32) * HMK_QCAP * (wide ? 12 : 8) + (size_t)qt * 12;
}

// ---------------------------------------------------------------- pieces shared by the bulk kernels
// Packed kernels' shared memory: the profile tile (qt profiles of pwb bytes) from offset 0, the TMA barrier at `bar`,
// the carve-up for `threads` threads at `carve`, and for the filter kernel the warps' prefix sums at `pfx`
// (hmk_pfx_words(qt) u32 per warp, 16-byte aligned); `total` is a launch's dynamic size.
struct HmkPackedSmem { size_t bar, carve, pfx, total; };
__host__ __device__ inline int hmk_pfx_words(int qt) { return (qt + 3) & ~3; }
__host__ __device__ inline HmkPackedSmem hmk_packed_smem(int qt, uint32_t pwb, int kb, int threads, bool filter) {
    const size_t bar = ((size_t)qt * pwb + 15) & ~(size_t)15;
    const size_t end = bar + 16 + hmk_carve_bytes(qt, kb, threads, false);
    const size_t pfx = (end + 15) & ~(size_t)15;
    return {bar, bar + 16, pfx, filter ? pfx + (size_t)(threads / 32) * hmk_pfx_words(qt) * 4 : end};
}

// carves a packed kernel's shared memory and initialises the tile barrier (visible after the next __syncthreads)
__device__ __forceinline__ uint64_t* hmk_packed_carve(unsigned char* smem, const HmkBulkArgs& a, uint32_t pwb, HmkTopkSmem& tk,
                                                      HmkHitQueue& hq) {
    const HmkPackedSmem ly = hmk_packed_smem(a.qt, pwb, a.kb, blockDim.x, false);
    hmk_carve(smem + ly.carve, a.qt, a.kb, false, tk, hq);
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + ly.bar);
    if (threadIdx.x == 0) hmk_mbar_init(bar, 1);
    return bar;
}

// stages profiles q0 .. q0 + qn - 1 (pwb bytes each) at the start of shared memory with the TMA bulk-copy engine and
// waits for them (barrier parity `phase`); TOPK first clears the tile's lists
template <int MODE>
__device__ __forceinline__ void hmk_stage_tile(unsigned char* smem, uint64_t* bar, uint32_t phase, const HmkBulkArgs& a,
                                               const HmkTopkSmem& tk, int q0, int qn, uint32_t pwb) {
    if (MODE == HMK_MODE_TOPK) hmk_topk_init(tk, qn, a.kb);
    __syncthreads();
    if (threadIdx.x == 0) {
        const uint32_t total = (uint32_t)qn * pwb;
        hmk_mbar_expect_tx(bar, total);
        const unsigned char* src = reinterpret_cast<const unsigned char*>(a.prof) + (size_t)q0 * pwb;
        uint32_t done = 0;
        while (done < total) {
            uint32_t n = min(total - done, 32768u);
            hmk_bulk_g2s(smem + done, src + done, n, bar);
            done += n;
        }
    }
    hmk_mbar_wait(bar, phase);
}

// end of the thread-side items of the chunk that starts at i_begin: ndb, or *ndb_dev when given
__device__ __forceinline__ int hmk_items_end(const HmkBulkArgs& a, int i_begin) {
    return min(a.ndb_dev ? min(a.ndb, __ldg(a.ndb_dev)) : a.ndb, i_begin + a.chunk);
}

// thread-side item i: its sequence id (0 past the end) and whether it is scored -- before i_end, not below min_id and
// still a singleton.  The packed kernels pass min_id = 0: ids are >= 0, so the unsigned test folds away (a runtime
// a.db_min_id there costs registers); the generic kernel passes a.db_min_id, tested before the slot load.
__device__ __forceinline__ bool hmk_item(const HmkBulkArgs& a, int i, int i_end, int32_t min_id, int32_t& id) {
    bool valid = i < i_end;
    id = valid ? (a.db_ids ? a.db_ids[i] : a.db_begin + i) : 0;
    if (valid && ((uint32_t)id < (uint32_t)min_id || (a.slot && a.slot[id] >= 0))) valid = false;
    return valid;
}

// end of a tile: the warp's last queued hits, then (TOPK) the tile's lists into output slot `slot`
template <int MODE>
__device__ __forceinline__ void hmk_tile_end(const HmkBulkArgs& a, const HmkTopkSmem& tk, int q0, int qn, HmkHitQueue& hq,
                                             int slot) {
    if (MODE != HMK_MODE_DENSE && hq.cnt) hmk_queue_drain<MODE>(a, tk, q0, hq);
    if (MODE == HMK_MODE_TOPK) {
        __syncthreads();
        hmk_topk_flush(a, tk, q0, qn, slot);
    }
}

// pair accounting: the pairs this warp scored; with prof_cells (mixed lengths: the items of a launch share one length,
// cells differ per profile of the tile q0 .. q0 + qn - 1, qn > 0) also their cells and int ops.  prof_cells needs a
// CTA that scores one tile: hmk_bulk_filter, which may move between tiles, never gets it
__device__ __forceinline__ void hmk_count_scored(const HmkBulkArgs& a, unsigned long long scored, int q0, int qn) {
    if (!a.pair_counter) return;
    for (int s = 16; s > 0; s >>= 1) scored += __shfl_xor_sync(0xffffffffu, scored, s);
    if ((threadIdx.x & 31) == 0 && scored) {
        atomicAdd(a.pair_counter, scored);
        if (a.prof_cells) {
            unsigned long long tc = 0, to = 0;
            for (int t = 0; t < qn; t++) { tc += a.prof_cells[q0 + t]; to += a.prof_ops[q0 + t]; }
            atomicAdd(a.pair_counter + 1, scored / qn * tc);
            atomicAdd(a.pair_counter + 2, scored / qn * to);
        }
    }
}

// ---------------------------------------------------------------- fast bulk kernel
#define HMK_ROWB (HMK_NRES * 4)                    // bytes of one (h, j) row: 24 residues x u32

template <int NW, int MODE, bool FSTRIDE = false>
__global__ void __launch_bounds__(HMK_BULK_THREADS, 1) hmk_bulk_fast(const __grid_constant__ HmkBulkArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr uint32_t PWB = FSTRIDE ? HMK_FPW * 4 : NW * HMK_MAXL1 * HMK_ROWB;   // bytes per profile (compile time)
    const int qtile = blockIdx.x % a.nqt, stripe = blockIdx.x / a.nqt;
    const int q0 = qtile * a.qt;
    const int qn = min(a.qt, a.nq - q0);
    if (qn <= 0) return;
    const int L = a.sc.L;
    HmkTopkSmem tk;
    HmkHitQueue hq;
    uint64_t* bar = hmk_packed_carve(smem_raw, a, PWB, tk, hq);
    hmk_stage_tile<MODE>(smem_raw, bar, 0, a, tk, q0, qn, PWB);

    const int i_begin = stripe * a.chunk;
    const int i_end = hmk_items_end(a, i_begin);
    unsigned long long scored = 0;
    const uint32_t topmask = a.sc.lane16 ? 0x80008000u : 0x80808080u;
    const int32_t dec = a.sc.T - a.sc.half;
    const unsigned char* sbase = smem_raw;

    // warp-uniform trip count; lanes past the end (or whose item is no longer a singleton)
    // compute on a dummy item and are masked out of the hit test
    for (int ib = i_begin + (threadIdx.x & ~31); ib < i_end; ib += blockDim.x) {
        const int i = ib + (threadIdx.x & 31);
        int32_t id;
        const bool valid = hmk_item(a, i, i_end, 0, id);
        if (!__any_sync(0xffffffffu, valid)) continue;
        const uint64_t w = valid ? a.packed[id] : 0ull;
        // rowp[j] = &profile[0][h=0][j][residue_j]; later profiles/halves are immediates away
        const unsigned char* rowp[HMK_MAXL1];
#pragma unroll
        for (int j = 0; j < HMK_MAXL1; j++)
            rowp[j] = sbase + j * HMK_ROWB + (uint32_t)((w >> (5 * j)) & 31u) * 4u;
        if (valid) scored += qn;

        auto score = [&](const int tu, uint32_t (&acc)[NW]) {
#pragma unroll
            for (int h = 0; h < NW; h++) acc[h] = 0;
#pragma unroll
            for (int j = 0; j < HMK_MAXL1; j++) {
                if (j < L) {
#pragma unroll
                    for (int h = 0; h < NW; h++)
                        acc[h] += *reinterpret_cast<const uint32_t*>(rowp[j] + tu * PWB + h * (HMK_MAXL1 * HMK_ROWB));
                }
            }
        };
        auto finish = [&](const int t, const uint32_t (&acc)[NW]) {
            uint32_t any = acc[0];
#pragma unroll
            for (int h = 1; h < NW; h++) any |= acc[h];
            if (MODE == HMK_MODE_DENSE) {
                if (valid) a.dense[(size_t)(q0 + t) * a.dense_stride + i] = hmk_lane_max(acc, NW, a.sc.lane16) + dec;
            } else {
                const bool hit = valid && (any & topmask) != 0;
                hmk_queue_push<MODE>(a, tk, q0, hq, hit, t, hit ? hmk_lane_max(acc, NW, a.sc.lane16) + dec : 0, i);
            }
        };

        int t = 0;
        for (; t + 4 <= qn; t += 4) {
            uint32_t a0[NW], a1[NW], a2[NW], a3[NW];
            score(0, a0); score(1, a1); score(2, a2); score(3, a3);
            finish(t, a0); finish(t + 1, a1); finish(t + 2, a2); finish(t + 3, a3);
#pragma unroll
            for (int j = 0; j < HMK_MAXL1; j++) rowp[j] += 4 * PWB;
        }
        for (; t < qn; t++) {
            uint32_t a0[NW];
            score(0, a0);
            finish(t, a0);
#pragma unroll
            for (int j = 0; j < HMK_MAXL1; j++) rowp[j] += PWB;
        }
    }
    hmk_count_scored(a, scored, q0, qn);
    hmk_tile_end<MODE>(a, tk, q0, qn, hq, stripe);
}

// ---------------------------------------------------------------- filter candidates
// whole warp: lane l holds row l of a 32 x 32 bit matrix (bit c = element (l, c)); returns column `lane`
// (bit l = element (l, lane)).  Recursive block transpose, one exchange per halving of the block size.
__device__ __forceinline__ uint32_t hmk_transpose32(uint32_t x, int lane) {
    const uint32_t keep[5] = {0x0000ffffu, 0x00ff00ffu, 0x0f0f0f0fu, 0x33333333u, 0x55555555u};
#pragma unroll
    for (int i = 0, s = 16; i < 5; i++, s >>= 1) {
        const uint32_t y = __shfl_xor_sync(0xffffffffu, x, s);
        x = (lane & s) ? ((x & ~keep[i]) | ((y & ~keep[i]) >> s)) : ((x & keep[i]) | ((y & keep[i]) << s));
    }
    return x;
}

// position of the n-th (from 0) set bit of m; n < popc(m)
__device__ __forceinline__ int hmk_nth_bit(uint32_t m, int n) {
    int pos = 0;
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) {
        const int c = __popc(m & ((1u << s) - 1u));
        if (n >= c) { n -= c; m >>= s; pos += s; }
    }
    return pos;
}

// ---------------------------------------------------------------- filter + verify bulk kernel
// The exact kernel needs 24 shared-memory look-ups per pair and is bound by that pipe.  Here every pair
// first takes 12 look-ups in a FILTER table whose four u8 lanes bound PAIRS of neighbouring diagonals from
// above (max of the two exact entries per position); only pairs where some bound reaches the threshold
// (about 4 % for the synthetic 12-mers at T = 20, against 0.3 % real hits) are re-scored exactly, 32
// candidates at a time, one per lane.  No false negatives (sum of maxima >= each sum), exact scores for
// everything that is reported.  u8 lanes, two exact words, lengths <= 12.
// Candidates never go through shared memory: a lane keeps, for HMK_FGROUP queries, one bit per (query, half)
// that passed for its own item.  At the end of the group the warp lists them query-major (lane minor) and
// hands them out into a round of 32 held in registers, one candidate per lane, fetching the item's packed
// word from the owning lane by shuffle; a part-filled round is carried into the next group and is verified
// when it is full or when the chunk ends.
// At the fixed length, an item block whose scored lanes share residues 0..2 (three warps in four on the clustering-order
// walk) takes the sum of those three filter rows per query from a per-warp array instead: 9 look-ups plus a quarter of
// a broadcast LDS.128 per query, against 12.
// LT: compile-time length (0 = use sc.L; then the twelve look-ups are predicated, which costs issue slots)
template <int MODE, int LT>
__global__ void __launch_bounds__(HMK_BULK_THREADS, 1) hmk_bulk_filter(const __grid_constant__ HmkBulkArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr uint32_t PWB = HMK_FPW * 4;
    constexpr uint32_t SUB = HMK_MAXL1 * HMK_ROWB;   // bytes of one sub-table
    constexpr int OCT_UNROLL = LT ? 2 : 1;
    // shared residue prefixes (below) in the partner search (TOPK) at a fixed length only: with them the general-length
    // TOPK build spills at 80 registers, and the founder filter's launches (EMIT, a few profiles per tile) got slower
    constexpr bool PREFIX = MODE == HMK_MODE_TOPK && LT >= HMK_PREFIX_RES;
    __shared__ int s_next[3];                         // persistent mode: (tile, chunk, output slot) of the next piece of work
    const int L = LT ? LT : a.sc.L;
    HMK_CHECK(!a.prof_cells);                         // a CTA may score several tiles (hmk_count_scored)
    HmkTopkSmem tk;
    HmkHitQueue hq;
    uint64_t* bar = hmk_packed_carve(smem_raw, a, PWB, tk, hq);
    __syncthreads();

    unsigned long long scored = 0;
    const int32_t dec = a.sc.T - a.sc.half;
    const unsigned char* sbase = smem_raw;
    const int lane = threadIdx.x & 31;
    // this warp's prefix sums: pfx[t] = the filter rows 0 .. HMK_PREFIX_RES - 1 of query t at the residues its items share
    uint32_t* pfx = reinterpret_cast<uint32_t*>(smem_raw + hmk_packed_smem(a.qt, PWB, a.kb, blockDim.x, true).pfx) +
                    (threadIdx.x >> 5) * hmk_pfx_words(a.qt);
    const bool persistent = a.sched != nullptr;
    int cur_tile = -1, slot = 0, q0 = 0, qn = 0, home = blockIdx.x % a.nqt;
    uint32_t bar_phase = 0;
    int i_begin = 0, i_end = 0;

    // the round: lanes below rfill hold a candidate -- the item's packed word rw and the entry re: bits 24..31 =
    // tile-local query, bit 22 / bit 23 = "a filter byte of exact word 0 / word 1 passed", the low 22 bits = the
    // item's offset in the chunk.  Free lanes keep rw = 0 and re = bit 22, so their look-ups hit the row everybody
    // else reads in profile 0.
    int rfill = 0;   // warp-uniform
    uint32_t re = 1u << 22;
    uint64_t rw = 0ull;

    // exact re-scoring of the round.  Only the exact word(s) whose filter bytes passed are summed (both: rare,
    // handled in a divergent tail)
    auto verify = [&]() {
        const bool have = lane < rfill;
        const int t = (int)(re >> 24);
        const uint32_t halves = (re >> 22) & 3u;
        const int32_t i = i_begin + (int32_t)(re & 0x3fffffu);
        HMK_CHECK(!have || (t < qn && i >= i_begin && i < i_end && halves != 0u));
        const uint64_t w = rw;
        const unsigned char* pb = sbase + (uint32_t)t * PWB + ((halves & 1u) ? 0u : SUB);
        uint32_t acc0 = 0, acc1 = 0;
#pragma unroll
        for (int j = 0; j < HMK_MAXL1; j++)
            if (j < L) acc0 += *reinterpret_cast<const uint32_t*>(pb + j * HMK_ROWB + (uint32_t)((w >> (5 * j)) & 31u) * 4u);
        if (halves == 3u) {
#pragma unroll
            for (int j = 0; j < HMK_MAXL1; j++)
                if (j < L) acc1 += *reinterpret_cast<const uint32_t*>(pb + SUB + j * HMK_ROWB + (uint32_t)((w >> (5 * j)) & 31u) * 4u);
        }
        __syncwarp();
        const bool hit = have && ((acc0 | acc1) & 0x80808080u) != 0;
        rfill = 0; re = 1u << 22; rw = 0ull;
        const uint32_t mx = __vmaxu4(acc0, acc1);
        const uint32_t m2 = __vmaxu4(mx, mx >> 16);
        const uint32_t m1 = (m2 & 0xffu) > ((m2 >> 8) & 0xffu) ? (m2 & 0xffu) : ((m2 >> 8) & 0xffu);
        hmk_queue_push<MODE>(a, tk, q0, hq, hit, t, hit ? (int32_t)m1 + dec : 0, i);
    };

    for (;;) {
        // ---- next piece of work: (tile, chunk).  Static mode: exactly one, named by the block index.  Persistent mode:
        // chunks of the home tile first; when it runs dry, the CTA moves on to the next tile that still has chunks left
        int tile, chunk_idx;
        if (!persistent) {
            if (cur_tile >= 0) break;
            tile = blockIdx.x % a.nqt; chunk_idx = blockIdx.x / a.nqt;
            slot = chunk_idx;
        } else {
            __syncthreads();            // everybody is done with s_next (and with the previous chunk)
            if (threadIdx.x == 0) {
                int t = home, ch = a.nchunks;
                if (!a.discards || __ldcg(a.discards) == a.discards_seen) {   // else the batch was thrown away: stop
                    ch = atomicAdd(a.sched + t, 1);
                    for (int k = 1; ch >= a.nchunks && k < a.nqt; k++) {
                        t = (home + k) % a.nqt;
                        ch = __ldcg(a.sched + t) < a.nchunks ? atomicAdd(a.sched + t, 1) : a.nchunks;
                    }
                }
                if (ch >= a.nchunks) t = -1;
                else if (t != cur_tile) s_next[2] = atomicAdd(a.sched + a.nqt + t, 1);
                s_next[0] = t; s_next[1] = ch;
            }
            __syncthreads();
            tile = s_next[0]; chunk_idx = s_next[1];
            if (tile < 0) break;
            HMK_CHECK(tile < a.nqt && chunk_idx >= 0 && chunk_idx < a.nchunks);
        }
        if (tile != cur_tile) {
            if (cur_tile >= 0) {        // leave the previous tile: the round was verified at the end of the chunk
                HMK_CHECK(rfill == 0);
                hmk_tile_end<MODE>(a, tk, q0, qn, hq, slot);
                __syncthreads();
            }
            if (persistent) { slot = s_next[2]; home = tile; }
            cur_tile = tile;
            q0 = tile * a.qt;
            qn = min(a.qt, a.nq - q0);
            if (qn <= 0) { if (persistent) continue; else return; }
            hmk_stage_tile<MODE>(smem_raw, bar, bar_phase, a, tk, q0, qn, PWB);
            bar_phase ^= 1u;
        }
        i_begin = chunk_idx * a.chunk;
        i_end = hmk_items_end(a, i_begin);

        for (int ib = i_begin + (threadIdx.x & ~31); ib < i_end; ib += blockDim.x) {
            const int i = ib + lane;
            int32_t id;
            const bool valid = hmk_item(a, i, i_end, 0, id);
            if (!__any_sync(0xffffffffu, valid)) continue;
            const uint64_t w = valid ? a.packed[id] : 0ull;
            if (valid) scored += qn;
            // Items are walked in id order, the clustering order (abundance, then sequence, descending), so the scored
            // lanes of most warps share their first residues.  Then the filter rows of those positions are summed once
            // per query into pfx (lane l: queries l, l + 32, ...) and the query loop below looks up the other rows only.
            // u32 addition is associative: every bound is bit for bit the full twelve-row sum.
            bool shared = false;
            if (PREFIX) {
                const uint32_t kmin = __reduce_min_sync(0xffffffffu, hmk_prefix_lo(w, valid));
                const uint32_t kmax = __reduce_max_sync(0xffffffffu, hmk_prefix_hi(w, valid));
                shared = hmk_prefix_shared(kmin, kmax) == HMK_PREFIX_RES;
                if (shared) {
                    for (int t = lane; t < qn; t += 32) {
                        const unsigned char* pt = sbase + (uint32_t)t * PWB + 2 * SUB;
                        uint32_t f = 0;
#pragma unroll
                        for (int j = 0; j < HMK_PREFIX_RES; j++)
                            f += *reinterpret_cast<const uint32_t*>(pt + j * HMK_ROWB + ((kmin >> (5 * j)) & 31u) * 4u);
                        pfx[t] = f;
                    }
                    __syncwarp();
                }
            }
            // bit k of m0 / m1: a filter byte of exact word 0 / word 1 passed against query g0 + k.  They are built an
            // octet of queries at a time: x = (x >> 1) | (f & 0x80808080) over c <= 8 queries leaves query q's top bit
            // of filter byte b at bit 8b + q + 8 - c (two instructions per query; no bit crosses into the byte below
            // before the eighth shift), and `octet` moves the bytes of the two exact words into the top of m0 / m1
            uint32_t m0 = 0, m1 = 0;
            auto octet = [&](uint32_t x, const int c) {
                x >>= 8 - c;
                const uint32_t y = x | (x >> 8);            // byte 0: exact word 0, byte 2: exact word 1
                m0 = __funnelshift_r(m0, y, 8);
                m1 = __funnelshift_r(m1, y >> 16, 8);
            };
            // hand the group's candidates out into the round, query-major with the lane as the minor key
            auto resolve = [&](const int g0) {
                // lanes without an item looked up residue 0 (same row as everybody else: no bank conflict); drop them here
                const uint32_t pm = valid ? (m0 | m1) : 0u;
                if (!__any_sync(0xffffffffu, pm != 0u)) return;
                const uint32_t col = hmk_transpose32(pm, lane);   // lanes with a candidate against query g0 + lane
                const int cnt = __popc(col);
                int incl = cnt;                                    // candidates of queries g0 .. g0 + lane
#pragma unroll
                for (int s = 1; s < 32; s <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, s);
                    if (lane >= s) incl += v;
                }
                const int n = __shfl_sync(0xffffffffu, incl, 31);
                for (int base = 0; base < n;) {
                    const int take = min(32 - rfill, n - base);
                    const int g = base + lane - rfill;            // this lane's candidate in the group's list
                    const int gq = min(max(g, 0), n - 1);
                    int k = 0;                                     // its query: the first k with incl[k] > gq
#pragma unroll
                    for (int s = 16; s > 0; s >>= 1)
                        if (__shfl_sync(0xffffffffu, incl, k + s - 1) <= gq) k += s;
                    const uint32_t ck = __shfl_sync(0xffffffffu, col, k);
                    const int first = __shfl_sync(0xffffffffu, incl - cnt, k);
                    const int src = hmk_nth_bit(ck, gq - first); // the lane that owns the item
                    const uint64_t ws = __shfl_sync(0xffffffffu, w, src);
                    const uint32_t h = (__shfl_sync(0xffffffffu, m0, src) >> k & 1u) |
                                       (__shfl_sync(0xffffffffu, m1, src) >> k & 1u) << 1;
                    if (lane >= rfill && g < base + take) {
                        HMK_CHECK(k < HMK_FGROUP && g0 + k < qn && src >= 0 && src < 32 && (ck >> src & 1u) && h != 0u &&
                                  ib + src - i_begin < (1 << 22));
                        re = (uint32_t)(g0 + k) << 24 | h << 22 | (uint32_t)(ib + src - i_begin);
                        rw = ws;
                    }
                    rfill += take;
                    base += take;
                    if (rfill == 32) verify();
                }
            };

            // the queries of the tile; U = residues whose rows come from pfx (a compile-time 0 or HMK_PREFIX_RES: a row
            // predicated off at run time would still take an issue slot)
            auto scan = [&](auto prefix) {
                constexpr int U = decltype(prefix)::value;
                const unsigned char* rowp[HMK_MAXL1];   // &filter[t][j][residue_j], j >= U
                // f = pfx[t + tu] (p, when U > 0) + the rows j >= U of query t + tu
                auto bound = [&](const int tu, const uint32_t p) -> uint32_t {
                    uint32_t f = U ? p : 0u;
#pragma unroll
                    for (int j = U; j < HMK_MAXL1; j++)
                        if (j < L) f += *reinterpret_cast<const uint32_t*>(rowp[j] + tu * PWB);
                    return f;
                };
                int t = 0;
                for (int g0 = 0; g0 < qn; g0 += HMK_FGROUP) {
                    const int gend = min(qn, g0 + HMK_FGROUP);
                    // set up per group, so that the pointers are not live while the group's candidates are handed out
#pragma unroll
                    for (int j = U; j < HMK_MAXL1; j++)
                        rowp[j] = sbase + (uint32_t)g0 * PWB + 2 * SUB + j * HMK_ROWB + (uint32_t)((w >> (5 * j)) & 31u) * 4u;
                    for (; t + 8 <= gend; t += 8) {
                        uint32_t x = 0;
                        // two blocks of four queries; unrolled only at a fixed length, where the predicate-free look-ups
                        // leave the registers for it (the general-length build would spill)
#pragma unroll OCT_UNROLL
                        for (int u = 0; u < 2; u++) {
                            // t + 4u is a multiple of 4: one broadcast LDS.128 for the four queries' prefix sums
                            const uint4 p = U ? *reinterpret_cast<const uint4*>(pfx + t + 4 * u) : make_uint4(0u, 0u, 0u, 0u);
                            const uint32_t f0 = bound(0, p.x), f1 = bound(1, p.y), f2 = bound(2, p.z), f3 = bound(3, p.w);
                            x = (x >> 1) | (f0 & 0x80808080u); x = (x >> 1) | (f1 & 0x80808080u);
                            x = (x >> 1) | (f2 & 0x80808080u); x = (x >> 1) | (f3 & 0x80808080u);
#pragma unroll
                            for (int j = U; j < HMK_MAXL1; j++) rowp[j] += 4 * PWB;
                        }
                        octet(x, 8);
                    }
                    if (t < gend) {                             // last, part-filled octet of the group
                        const int c = gend - t;
                        uint32_t x = 0;
                        for (; t < gend; t++) {
                            x = (x >> 1) | (bound(0, U ? pfx[t] : 0u) & 0x80808080u);
#pragma unroll
                            for (int j = U; j < HMK_MAXL1; j++) rowp[j] += PWB;
                        }
                        octet(x, c);
                    }
                    const int octets = (gend - g0 + 7) >> 3;     // the first octet sits in the lowest byte
                    m0 >>= 8 * (4 - octets);
                    m1 >>= 8 * (4 - octets);
                    resolve(g0);
                    m0 = 0; m1 = 0;
                }
            };
            if (PREFIX && shared) scan(std::integral_constant<int, PREFIX ? HMK_PREFIX_RES : 0>());
            else scan(std::integral_constant<int, 0>());
        }
        if (rfill) verify();      // the round must be empty before the tile (and with it q0) can change
    }
    if (cur_tile >= 0 && qn > 0) hmk_tile_end<MODE>(a, tk, q0, qn, hq, slot);
    hmk_count_scored(a, scored, q0, qn);
}

// ---------------------------------------------------------------- long bulk kernel
// Same scheme for sequences of 13..36 residues (two or three packed words) and up to HMK_NWMAX words
// per profile entry (s16 lanes: up to 20 shift diagonals).  Layout prof[t][j][h][r]: all words of one
// position are 96 B apart, so they are immediates off one per-position pointer; L and nw are runtime
// (fully unrolled, predicated).  One query at a time (the NW independent accumulators give the ILP).
template <int MODE>
__global__ void __launch_bounds__(HMK_LONG_THREADS, 1) hmk_bulk_long(const __grid_constant__ HmkBulkArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int qtile = blockIdx.x % a.nqt, stripe = blockIdx.x / a.nqt;
    const int q0 = qtile * a.qt;
    const int qn = min(a.qt, a.nq - q0);
    if (qn <= 0) return;
    const int L = a.sc.L, nw = a.sc.nw, W = a.sc.words;
    const uint32_t PWB = (uint32_t)a.sc.prof_words * 4u;
    HmkTopkSmem tk;
    HmkHitQueue hq;
    uint64_t* bar = hmk_packed_carve(smem_raw, a, PWB, tk, hq);
    hmk_stage_tile<MODE>(smem_raw, bar, 0, a, tk, q0, qn, PWB);

    const int i_begin = stripe * a.chunk;
    const int i_end = hmk_items_end(a, i_begin);
    unsigned long long scored = 0;
    const uint32_t topmask = a.sc.lane16 ? 0x80008000u : 0x80808080u;
    const int32_t dec = a.sc.T - a.sc.half;
    const uint32_t jstride = (uint32_t)nw * HMK_ROWB;

    for (int ib = i_begin + (threadIdx.x & ~31); ib < i_end; ib += blockDim.x) {
        const int i = ib + (threadIdx.x & 31);
        int32_t id;
        const bool valid = hmk_item(a, i, i_end, 0, id);
        if (!__any_sync(0xffffffffu, valid)) continue;
        uint64_t w[3] = {0ull, 0ull, 0ull};
#pragma unroll
        for (int k = 0; k < 3; k++)
            if (valid && k < W) w[k] = a.packed[(size_t)id * W + k];
        const unsigned char* rowp[HMK_MAXLEN];
#pragma unroll
        for (int j = 0; j < HMK_MAXLEN; j++)
            rowp[j] = smem_raw + j * jstride + (uint32_t)((w[j / HMK_MAXL1] >> (5 * (j % HMK_MAXL1))) & 31u) * 4u;
        if (valid) scored += qn;
        for (int t = 0; t < qn; t++) {
            uint32_t acc[HMK_NWMAX];
#pragma unroll
            for (int h = 0; h < HMK_NWMAX; h++) acc[h] = 0;
#pragma unroll
            for (int j = 0; j < HMK_MAXLEN; j++) {
                if (j < L) {
#pragma unroll
                    for (int h = 0; h < HMK_NWMAX; h++)
                        if (h < nw) acc[h] += *reinterpret_cast<const uint32_t*>(rowp[j] + h * HMK_ROWB);
                    rowp[j] += PWB;
                }
            }
            // both lane widths, then a select: hmk_lane_max's branch on lane16 would let the compiler duplicate this loop
            uint32_t any = 0, m2 = 0, m4 = 0;
#pragma unroll
            for (int h = 0; h < HMK_NWMAX; h++)
                if (h < nw) { any |= acc[h]; m2 = __vmaxu2(m2, acc[h]); m4 = __vmaxu4(m4, acc[h]); }
            int32_t best;
            if (a.sc.lane16) { const uint32_t lo = m2 & 0xffffu, hi = m2 >> 16; best = (int32_t)(lo > hi ? lo : hi); }
            else {
                uint32_t x = m4 & 0xffu, y = (m4 >> 8) & 0xffu, z = (m4 >> 16) & 0xffu, v = m4 >> 24;
                x = x > y ? x : y; z = z > v ? z : v;
                best = (int32_t)(x > z ? x : z);
            }
            if (MODE == HMK_MODE_DENSE) {
                if (valid) a.dense[(size_t)(q0 + t) * a.dense_stride + i] = best + dec;
            } else {
                const bool hit = valid && (any & topmask) != 0;
                hmk_queue_push<MODE>(a, tk, q0, hq, hit, t, hit ? best + dec : 0, i);
            }
        }
    }
    hmk_count_scored(a, scored, q0, qn);
    hmk_tile_end<MODE>(a, tk, q0, qn, hq, stripe);
}

// ---------------------------------------------------------------- generic bulk kernel
// Any lengths, any int32 matrix, any penalty: scalar Java-int arithmetic per pair.  Same
// outputs as the fast kernel.  prof_ids[t] are the profile-side sequence ids; `prof_is_query`
// says whether they are the reference's seq2 (query) or seq1 (member).
struct HmkGenericArgs {
    HmkBulkArgs b;
    const int32_t* prof_ids;
    int32_t prof_is_query;
    const uint8_t* res;
    const int32_t* off;
    const int32_t* M;
    int32_t maxlen;
    int32_t db_smem;      // 1: the thread-side residues are staged in shared memory ([maxlen][threads] fits)
};

#define HMK_GENERIC_THREADS 256

// generic kernel's shared memory: the matrix from offset 0, the carve-up at `carve`, the profile lengths at `slen`, the
// profile residues ([qt][maxlen]) at `sres`, with db_smem the thread-side residues at `sdb`; `total` is a launch's size
struct HmkGenericSmem { size_t carve, slen, sres, sdb, total; };
__host__ __device__ inline HmkGenericSmem hmk_generic_smem(int qt, int kb, int maxlen, bool db_smem) {
    HmkGenericSmem l;
    l.carve = HMK_NRES * HMK_NRES * 4;
    l.slen = l.carve + hmk_carve_bytes(qt, kb, HMK_GENERIC_THREADS, true);
    l.sres = l.slen + (size_t)qt * 4;
    l.sdb = l.sres + (((size_t)qt * maxlen + 15) & ~(size_t)15);
    l.total = l.sdb + (db_smem ? (size_t)maxlen * HMK_GENERIC_THREADS : 0) + 16;
    return l;
}

// EMIT and DENSE: five CTAs per SM (48 registers); left free, the compiler takes 64 there, which allows only four.
// TOPK needs its 64.
template <int MODE>
__global__ void __launch_bounds__(HMK_GENERIC_THREADS, MODE == HMK_MODE_TOPK ? 4 : 5) hmk_bulk_generic(const __grid_constant__ HmkGenericArgs g) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const HmkBulkArgs& a = g.b;
    const int qtile = blockIdx.x % a.nqt, stripe = blockIdx.x / a.nqt;
    const int q0 = qtile * a.qt;
    const int qn = min(a.qt, a.nq - q0);
    if (qn <= 0) return;
    const HmkGenericSmem ly = hmk_generic_smem(a.qt, a.kb, g.maxlen, g.db_smem);
    int32_t* sM = reinterpret_cast<int32_t*>(smem_raw);
    HmkTopkSmem tk;
    HmkHitQueue hq;
    hmk_carve(smem_raw + ly.carve, a.qt, a.kb, true, tk, hq);
    int32_t* slen = reinterpret_cast<int32_t*>(smem_raw + ly.slen);
    uint8_t* sres = smem_raw + ly.sres;
    // the thread-side sequences of the current iteration, position-major ([j][thread]): the inner loops then read shared
    // memory only, conflict free, instead of one global byte per cell and lane
    uint8_t* sdb = smem_raw + ly.sdb;
    for (int i = threadIdx.x; i < HMK_NRES * HMK_NRES; i += blockDim.x) sM[i] = g.M[i];
    for (int t = threadIdx.x; t < qn; t += blockDim.x) {
        int32_t id = g.prof_ids[q0 + t];
        int len = g.off[id + 1] - g.off[id];
        slen[t] = len;
        for (int j = 0; j < len; j++) sres[(size_t)t * g.maxlen + j] = g.res[g.off[id] + j];
    }
    if (MODE == HMK_MODE_TOPK) hmk_topk_init(tk, qn, a.kb);
    __syncthreads();
    const int i_begin = stripe * a.chunk;
    const int i_end = hmk_items_end(a, i_begin);
    unsigned long long scored = 0;
    for (int ib = i_begin + (threadIdx.x & ~31); ib < i_end; ib += blockDim.x) {
        const int i = ib + (threadIdx.x & 31);
        int32_t id;
        const bool valid = hmk_item(a, i, i_end, a.db_min_id, id);
        if (!__any_sync(0xffffffffu, valid)) continue;
        const uint8_t* dres = g.res + g.off[id];
        const int dlen = valid ? g.off[id + 1] - g.off[id] : 0;
        uint8_t* mine = sdb + threadIdx.x;
        if (g.db_smem) {
            for (int j = 0; j < dlen; j++) mine[(size_t)j * HMK_GENERIC_THREADS] = dres[j];
            __syncwarp();
        }
        const uint8_t* dseq = g.db_smem ? mine : dres;
        const int dst = g.db_smem ? HMK_GENERIC_THREADS : 1;
        if (valid) scored += qn;
        for (int t = 0; t < qn; t++) {
            const uint8_t* pres = sres + (size_t)t * g.maxlen;
            int32_t s = 0;
            if (valid)
                s = g.prof_is_query ? hmk_pair_score_strided(dseq, dst, dlen, pres, 1, slen[t], sM, a.sc.X, a.sc.P)
                                    : hmk_pair_score_strided(pres, 1, slen[t], dseq, dst, dlen, sM, a.sc.X, a.sc.P);
            __syncwarp();
            if (MODE == HMK_MODE_DENSE) { if (valid) a.dense[(size_t)(q0 + t) * a.dense_stride + i] = s; }
            else hmk_queue_push<MODE>(a, tk, q0, hq, valid && s >= a.sc.T, t, s, i);
        }
    }
    hmk_count_scored(a, scored, q0, qn);
    hmk_tile_end<MODE>(a, tk, q0, qn, hq, stripe);
}

// ---------------------------------------------------------------- top-k merge across stripes
// one warp per query: kb rounds of "largest key below the previous pick" (keys are distinct)
// `slots_of_tile` (persistent launches): the number of lists tile t / qt really got, instead of nstripes
__global__ void hmk_topk_merge(int nq, int nstripes, int kb, const uint64_t* __restrict__ tk_key,
                               const int32_t* __restrict__ tk_cnt, const int32_t* __restrict__ tk_ovf,
                               uint64_t* __restrict__ out_key, int32_t* __restrict__ out_cnt,
                               int32_t* __restrict__ out_ovf, const int32_t* __restrict__ slots_of_tile = nullptr, int qt = 1) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= nq) return;
    if (slots_of_tile) { HMK_CHECK(slots_of_tile[t / qt] >= 0 && slots_of_tile[t / qt] <= nstripes); nstripes = min(nstripes, slots_of_tile[t / qt]); }
    int total = 0, ovf = 0;
    for (int s = lane; s < nstripes; s += 32) {
        HMK_CHECK(tk_cnt[(size_t)s * nq + t] >= 0 && tk_cnt[(size_t)s * nq + t] <= kb);
        total += tk_cnt[(size_t)s * nq + t];
        ovf |= tk_ovf[(size_t)s * nq + t];
    }
    for (int s = 16; s > 0; s >>= 1) { total += __shfl_xor_sync(0xffffffffu, total, s); ovf |= __shfl_xor_sync(0xffffffffu, ovf, s); }
    uint64_t prev = ~0ull;
    const int take = total < kb ? total : kb;
    for (int r = 0; r < take; r++) {
        uint64_t best = 0;
        for (int e = lane; e < nstripes * kb; e += 32) {
            const int s = e / kb, i = e % kb;
            if (i < tk_cnt[(size_t)s * nq + t]) {
                uint64_t v = tk_key[((size_t)s * nq + t) * kb + i];
                if (v < prev && v > best) best = v;
            }
        }
        for (int s = 16; s > 0; s >>= 1) { uint64_t v = __shfl_xor_sync(0xffffffffu, best, s); best = v > best ? v : best; }
        if (lane == 0) out_key[(size_t)t * kb + r] = best;
        prev = best;
    }
    if (lane == 0) { out_cnt[t] = take; out_ovf[t] = (ovf || total > kb) ? 1 : 0; }
}

// ---------------------------------------------------------------- batch selection (phase 1)
// single CTA: the next `want` ids >= cur that are still singletons, ascending
// `start_after` (optional): start right behind that id (the last query of the previous batch) instead
// of at ctl->cur -- used when the next batch is prepared while the current one is still resolving
__global__ void hmk_select_queries(const int32_t* __restrict__ slot, int n, const HmkCtl* ctl, const int32_t* start_after,
                                   int want, int32_t* __restrict__ qid, int32_t* __restrict__ nq_out) {
    __shared__ int warp_cnt[32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    const int first = start_after ? *start_after + 1 : ctl->cur;
    for (int start = first; start < n; start += blockDim.x) {
        const int i = start + threadIdx.x;
        const bool f = i < n && __ldcg(slot + i) < 0;
        const unsigned m = __ballot_sync(0xffffffffu, f);
        if (lane == 0) warp_cnt[wid] = __popc(m);
        __syncthreads();
        int pre = 0, tot = 0;
        for (int w2 = 0; w2 < nwarps; w2++) { int c = warp_cnt[w2]; if (w2 < wid) pre += c; tot += c; }
        const int pos = base + pre + __popc(m & ((1u << lane) - 1u));
        if (f && pos < want) qid[pos] = i;
        __syncthreads();
        if (threadIdx.x == 0) base += tot;
        __syncthreads();
        if (base >= want) break;
    }
    // a speculative batch near the end of the list may find fewer ids: pad with the last one found (the
    // resolver skips duplicates because the first occurrence is processed or consumed by then)
    if (threadIdx.x == 0) *nq_out = base < want ? base : want;
}

// ---------------------------------------------------------------- one-at-a-time pair scores
// S(member, query) for the irregular parts of the path (member checks, phase-2 resolution).
// Uniform length <= 12: residues come from the two packed words and the matrix from shared
// memory; otherwise the generic byte path.  Java-int arithmetic either way.
struct HmkScalar {
    const uint64_t* packed;   // NULL -> generic path
    const int32_t* sM;        // 24x24 in shared memory
    int32_t L;
};

__device__ __forceinline__ void hmk_load_matrix_smem(int32_t* sM, const int32_t* M) {
    for (int i = threadIdx.x; i < HMK_NRES * HMK_NRES; i += blockDim.x) sM[i] = M[i];
    __syncthreads();
}

__device__ __forceinline__ int32_t hmk_scalar_score(const HmkState& S, const HmkScalar& sc, int32_t member, int32_t query) {
    if (!sc.packed) return hmk_state_score(S, member, query);
    return hmk_packed_pair_score(sc.packed[member], sc.packed[query], sc.sM, S.X, S.P);
}

// Dense table of pair scores for sequences of mixed lengths <= 12 straight from the packed words (which carry their
// lengths): dense[t * stride + i] = S(seq1 = db item i, seq2 = profile-side sequence t).  One thread per pair; used for
// the small intra-batch tables of mixed-length inputs, where the per-length packed kernel would need one launch per
// (length, table) and the generic byte kernel is several times slower.
__global__ void __launch_bounds__(256) hmk_dense_packed(const uint64_t* __restrict__ packed, const int32_t* __restrict__ prof_ids, int nq,
                                                        const int32_t* __restrict__ db_ids, int ndb, const int32_t* __restrict__ M,
                                                        int X, int P, int32_t* __restrict__ dense, int stride,
                                                        unsigned long long* pair_counter) {
    __shared__ int32_t sM[HMK_NRES * HMK_NRES];
    hmk_load_matrix_smem(sM, M);
    const size_t total = (size_t)nq * ndb;
    for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < total; e += (size_t)gridDim.x * blockDim.x) {
        const int t = (int)(e / ndb), i = (int)(e % ndb);
        dense[(size_t)t * stride + i] = hmk_packed_pair_score(packed[db_ids[i]], packed[prof_ids[t]], sM, X, P);
    }
    if (pair_counter && blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(pair_counter, (unsigned long long)total);
}

// ---------------------------------------------------------------- member check (complete linkage)
// One thread per founder hit: does the query also score >= T against every other current
// member of that cluster?  (ClinkageClusterScorer.java:30-49; early exit keeps it cheap.)
struct HmkCheckArgs {
    HmkState S;
    const int4* hits;
    const unsigned int* hit_count;
    unsigned int hit_cap;
    int32_t hit_t_is_query;      // 1: hit.x = query index, hit.y = founder's id; 0: hit.x = cluster slot, hit.y = query's id
                                 // 2: phase-1 partner-search hits (xhits): (profile-side id, thread-side id, score, batch)
    const unsigned long long* xhit_count;   // mode 2: number of entries in hits
    unsigned long long* hit_valid;          // mode 2: counts the hits that are (founder, single) pairs of valid batches
    const int32_t* qids;         // phase 1: query index -> sequence id
    const int32_t* sidx;         // phase 2: sequence id -> index in the singles list
    // phase 1 output: per-query arrays ac_slot/ac_score[qi * capq + k], k < ac_cnt[qi]
    int32_t* ac_cnt; int32_t* ac_slot; int32_t* ac_score; int32_t capq;
    // phase 2 output: flat candidate arrays
    unsigned long long* cand_key_q;   // (query index << cbits) | slot      -- fields packed tight: the radix sort only
    int32_t cbits;                    //                                       touches cbits + qbits bits
    int32_t* cand_score;
    unsigned int* cand_count;
    unsigned int cand_cap;
    int32_t linked;
    const uint64_t* packed;      // non-NULL: uniform length <= 12, use the packed scalar scorer
    int32_t L;
    unsigned long long* pair_parts;   // sharded pair-score counter
};

// FAST: uniform length 12, max shift 3 -- the unrolled scorer (hmk_score12x3) on the packed words
template <bool FAST>
__global__ void hmk_member_check(const HmkCheckArgs a) {
    __shared__ int32_t sM[HMK_NRES * HMK_NRES];
    hmk_load_matrix_smem(sM, a.S.M);
    HmkScalar sc;
    sc.packed = a.packed; sc.sM = sM; sc.L = a.L;
    const size_t nh = a.hit_t_is_query == 2 ? (size_t)*a.xhit_count : (size_t)min(*a.hit_count, a.hit_cap);
    long long npairs = 0, nvalid = 0;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < nh; e += (size_t)gridDim.x * blockDim.x) {
        const int4 h = a.hits[e];
        int qi, c;
        int32_t q;
        if (a.hit_t_is_query == 2) {
            // S is symmetric here (checked by the host), so the partner-search score of (x, y) is the founder
            // score of either role assignment; the batch tag drops scans of batches that were re-done
            if (a.S.qbatch[h.x] != h.w) continue;
            const int32_t sx = a.S.slot[h.x], sy = a.S.slot[h.y];
            if (sx >= 0 && sy < 0 && a.S.c_founder[sx] == h.x) { c = sx; q = h.y; }
            else if (sy >= 0 && sx < 0 && a.S.c_founder[sy] == h.y) { c = sy; q = h.x; }
            else continue;
            qi = a.sidx[q];
            nvalid++;
        } else {
            // phase 1: (query index, founder's sequence id); phase 2: (founder = cluster slot, query's sequence id)
            qi = a.hit_t_is_query ? h.x : a.sidx[h.y];
            c = a.hit_t_is_query ? a.S.slot[h.y] : h.x;
            q = a.hit_t_is_query ? a.qids[qi] : h.y;
        }
        int32_t cl = h.z;
        bool ok = true;
        int32_t qrow[HMK_MAXL1];
        HMK_CHECK(c >= 0 && c < a.S.K && q >= 0 && q < a.S.n && qi >= 0);
        if (FAST) hmk_qrow12(a.packed[q], qrow);
        for (int32_t m = a.S.next[a.S.c_founder[c]]; m >= 0; m = a.S.next[m]) {
            const int32_t s = FAST ? hmk_score12x3(qrow, a.packed[m], sM, a.S.P) : hmk_scalar_score(a.S, sc, m, q);
            npairs++;
            if (s < cl) cl = s;
            if (s < a.S.T) { ok = false; break; }
        }
        if (!ok) continue;
        if (a.linked) {
            const int k = atomicAdd(a.ac_cnt + qi, 1);     // the resolver checks ac_cnt against capq
            if (k < a.capq) {
                a.ac_slot[(size_t)qi * a.capq + k] = c;
                a.ac_score[(size_t)qi * a.capq + k] = cl;
            }
            continue;
        }
        unsigned int pos = atomicAdd(a.cand_count, 1u);
        if (pos >= a.cand_cap) continue;
        {
            const uint32_t gq = (uint32_t)qi;
            a.cand_key_q[pos] = ((unsigned long long)gq << a.cbits) | (uint32_t)c;
            a.cand_score[pos] = cl;
        }
    }
    for (int s = 16; s > 0; s >>= 1) npairs += __shfl_xor_sync(0xffffffffu, npairs, s);
    if ((threadIdx.x & 31) == 0) hmk_count_pairs(a.pair_parts, npairs);
    if (a.hit_t_is_query == 2) {
        for (int s = 16; s > 0; s >>= 1) nvalid += __shfl_xor_sync(0xffffffffu, nvalid, s);
        if ((threadIdx.x & 31) == 0 && nvalid) atomicAdd(a.hit_valid, (unsigned long long)nvalid);
    }
}

// ---------------------------------------------------------------- phase-1 resolver
// Replays firstPhase (LimitedGreedySequenceClusterer.java:90-116) for one batch in reference
// order.  One warp; every per-query step is lane-parallel (partner list, static cluster
// candidates, bitmask tests) so a step costs a few dependent memory round trips.
// Bookkeeping of what changed inside the batch lives in shared memory:
//   touched table: clusters that received members in this batch -> bitmask of the batch
//   queries that joined/founded them (+ the partner's sequence id for clusters born here)
//   founder mask : batch queries that founded a cluster in this batch
// ibm[b] is the bitmask of earlier batch queries b2 with S(q_b2, q_b) >= T, so "every added
// member scores >= T" is (member mask & ~ibm[b]) == 0.
#define HMK_MAXBATCH 512
#define HMK_MAXW (HMK_MAXBATCH / 32)

struct HmkP1Batch {
    int32_t nq, batch_id;
    const int32_t* qid;       // [nq] ascending ids, all singletons at batch start
    int32_t kb;               // <= 32
    const uint64_t* bk_key;   // [nq][kb] best later singletons at batch start, descending
    const int32_t* bk_cnt;    // [nq]
    const int32_t* bk_ovf;    // [nq] 1 = more hits existed than the list holds
    int32_t capq;
    const int32_t* ac_cnt;    // [nq] pre-batch clusters whose every pre-batch member scores >= T
    const int32_t* ac_slot;   // [nq][capq]
    const int32_t* ac_score;  // min over the pre-batch members
    const int4* ac_full;      // [nq][capq] the same candidates as (slot, score, Cluster.size(), founder id) -- hmk_p1_prepare_candidates
    const int4* best;         // [nq] the best of them under the reference's key as (score, size, founder id, slot); slot -1 = none
    const unsigned int* hit_count;   // founder hits the cluster search produced / room it had: the resolver refuses to run on
    unsigned int hit_cap;            //   a truncated hit list (HMK_P1_GROWHITS, state untouched)
    const int32_t* ib;        // ib[b*ib_stride + b2] = S(member = qid[b2], query = qid[b])
    int32_t ib_stride;
    const uint32_t* ibm;      // [nq][nw]
    const uint32_t* ibm2;     // [nq][nw] subset of ibm: founders that could beat query b's own pair (see hmk_ib_mask)
    int32_t nw;
    const int32_t* pcand;     // [nq][kb] sequence ids of the partner candidates (bk_key decoded)
    const int32_t* pd;        // pd[b*pd_stride + b2*kb + j] = S(member = j-th partner candidate of b2, query = qid[b])
    int32_t pd_stride;
};

// ids of every query's partner candidates (padding: the query itself)
__global__ void hmk_partner_ids(int nq, int kb, const uint64_t* __restrict__ bk_key, const int32_t* __restrict__ bk_cnt,
                                const int32_t* __restrict__ id_of_rank, const int32_t* __restrict__ qid,
                                int32_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nq * kb) return;
    const int b = i / kb, j = i % kb;
    int32_t id = qid[b];
    if (j < bk_cnt[b]) {
        const uint32_t r = hmk_key_rank(bk_key[i]);
        id = id_of_rank ? id_of_rank[r] : (int32_t)r;
    }
    out[i] = id;
}

// ibm [b][w]: earlier batch queries b2 with S(q_b2, q_b) >= T;
// ibm2[b][w]: those with S(q_b2, q_b) >= the LOWEST score in query b's partner list -- whichever partner b ends up
// with scores at least that, so a cluster founded by a b2 outside ibm2 can never beat b's own pair (its
// complete-linkage score is at most the founder's score)
__global__ void hmk_ib_mask(int nq, int nw, int32_t T, const int32_t* __restrict__ ib, int stride, uint32_t* __restrict__ ibm,
                            int kb, const uint64_t* __restrict__ bk_key, const int32_t* __restrict__ bk_cnt, uint32_t* __restrict__ ibm2) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= nq * nw) return;
    const int b = idx / nw, w = idx % nw;
    const int cnt = bk_cnt[b];
    const int32_t thr = cnt > 0 ? hmk_key_score(bk_key[(size_t)b * kb + cnt - 1]) : HMK_JMAX;
    uint32_t m = 0, m2 = 0;
    for (int k = 0; k < 32; k++) {
        const int b2 = w * 32 + k;
        if (b2 < b) {
            const int32_t s = ib[(size_t)b * stride + b2];
            if (s >= T) m |= 1u << k;
            if (s >= T && s >= thr) m2 |= 1u << k;
        }
    }
    ibm[idx] = m;
    ibm2[idx] = m2;
}

// warp arg-max under the reference's key (score desc, size desc, id asc) with three hardware
// reductions (REDUX) instead of a 5-round shuffle butterfly over four fields
__device__ __forceinline__ void hmk_best_reduce(HmkBestCluster& b) {
    const unsigned FULL = 0xffffffffu;
    const bool has = b.slot >= 0;
    const int32_t mx = __reduce_max_sync(FULL, has ? b.score : HMK_JMIN);
    const bool in1 = has && b.score == mx;
    if (__ballot_sync(FULL, in1) == 0) { b.slot = -1; return; }
    const int32_t ms = __reduce_max_sync(FULL, in1 ? b.size : HMK_JMIN);
    const bool in2 = in1 && b.size == ms;
    const int32_t mf = __reduce_min_sync(FULL, in2 ? b.fid : HMK_JMAX);
    const unsigned win = __ballot_sync(FULL, in2 && b.fid == mf);
    b.slot = __shfl_sync(FULL, b.slot, __ffs(win) - 1);
    b.score = mx; b.size = ms; b.fid = mf;
}

// One warp per batch query, right behind the member check: the query's valid pre-batch clusters with everything a
// resolver step needs in one 16-byte record, and the best of them under the reference's key.  The best stays an
// upper bound of what a pre-batch cluster can offer for the whole batch (complete-linkage scores only fall when
// members are added), which is what the resolver's windows test against.
__global__ void hmk_p1_prepare_candidates(const HmkState S, int nq, int capq, const int32_t* __restrict__ ac_cnt,
                                          const int32_t* __restrict__ ac_slot, const int32_t* __restrict__ ac_score,
                                          int4* __restrict__ ac_full, int4* __restrict__ best) {
    const int b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (b >= nq) return;
    HmkBestCluster bb;
    bb.score = HMK_JMIN; bb.size = 0; bb.fid = 0; bb.slot = -1;
    const int cnt = min(ac_cnt[b], capq);
    for (int e = lane; e < cnt; e += 32) {
        const size_t g = (size_t)b * capq + e;
        const int32_t c = ac_slot[g], sc = ac_score[g], sz = S.c_size[c], fd = S.c_founder[c];
        ac_full[g] = make_int4(c, sc, sz, fd);
        hmk_consider(bb, sc, sz, fd, c);
    }
    hmk_best_reduce(bb);
    if (lane == 0) best[b] = make_int4(bb.score, bb.size, bb.fid, bb.slot);
}

#define HMK_RESOLVE_THREADS 256
#ifdef HMK_RESOLVE_TIMING
#define HMK_TICK(i) do { long long t_ = clock64(); dbg[i] += t_ - tlast; tlast = t_; } while (0)
#else
#define HMK_TICK(i) do {} while (0)
#endif
#ifdef HMK_RESOLVE_TRACE
#define HMK_TRACE(slot, v) do { if (lane == 0) *(volatile long long*)&ctl->dbg[slot] = (long long)(v); } while (0)
#define HMK_TRACE_LANES(slot) atomicOr((unsigned long long*)&ctl->dbg[slot], 1ull << lane)
#define HMK_TRACE_CLEAR() do { if (lane == 0) { ctl->dbg[4] = 0; ctl->dbg[5] = 0; ctl->dbg[6] = 0; ctl->dbg[7] = 0; } __syncwarp(); } while (0)
#else
#define HMK_TRACE(slot, v) do {} while (0)
#define HMK_TRACE_LANES(slot) do {} while (0)
#define HMK_TRACE_CLEAR() do {} while (0)
#endif
#define HMK_HASH_SIZE 2048          // >= 2 * HMK_MAXBATCH, power of two

// shared-memory bytes of the resolver for a batch of nq queries, before the candidate cache
__host__ __device__ inline size_t hmk_resolve_fixed_bytes(int nq, int nw, int kb) {
    size_t o = (size_t)nq * 4 * 5;           // qid, qab, bk_cnt, bk_ovf, ac_raw
    o += (size_t)(nq + 1) * 4;               // ac_off
    o += (size_t)nq * nw * 4 * 3;            // ibm, ibm2, t_mask
    o += (size_t)nq * 4 * 10;                // t_fb, t_size, t_fid, t_count, t_tail, t_nmem, t_first, f_slot, f_pick, f_tidx
    o += (size_t)nq * kb * 4 * 3;            // bk_id, bk_score, bk_ab
    o += (size_t)nq * 4 * 3;                 // per-step list of touched candidates (tc_c, tc_cl, tc_row)
    o += (size_t)nq * 16 + ((size_t)nw * 4 + 16) * 2;   // best untouched static candidate per query, dirty mask, founder mask
    return o;
}
#define HMK_RESOLVE_CAND_BYTES 16            // cached candidate: slot, score, size, founder id

__device__ __forceinline__ uint32_t hmk_hash(uint32_t x) { return (x * 2654435761u) >> (32 - 11); }   // log2(HMK_HASH_SIZE) = 11

// The CTA first stages every per-batch input in shared memory (all warps, parallel gathers),
// then warp 0 replays the steps in reference order.  What changes inside the batch is tracked
// in shared memory too -- a hash set of the partners consumed so far, a hash map cluster ->
// row for the clusters that received members, and each such cluster's running size / count /
// tail (written through to global memory) -- so a typical step issues NO global loads.
__global__ void __launch_bounds__(HMK_RESOLVE_THREADS) hmk_p1_resolve_kernel(const HmkState S, const HmkP1Batch B, int cache_entries) {
#ifdef HMK_RESOLVE_TIMING
    long long dbg[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64();
#endif
    extern __shared__ __align__(128) unsigned char rs_raw[];
    const int nq = B.nq, nw = B.nw, kb = B.kb;
    unsigned char* p = rs_raw;
    int32_t* s_qid = reinterpret_cast<int32_t*>(p);     p += (size_t)nq * 4;
    int32_t* s_qab = reinterpret_cast<int32_t*>(p);     p += (size_t)nq * 4;
    int32_t* s_bkcnt = reinterpret_cast<int32_t*>(p);   p += (size_t)nq * 4;
    int32_t* s_bkovf = reinterpret_cast<int32_t*>(p);   p += (size_t)nq * 4;
    int32_t* s_acraw = reinterpret_cast<int32_t*>(p);   p += (size_t)nq * 4;
    int32_t* s_acoff = reinterpret_cast<int32_t*>(p);   p += (size_t)(nq + 1) * 4;
    uint32_t* s_ibm = reinterpret_cast<uint32_t*>(p);   p += (size_t)nq * nw * 4;
    uint32_t* s_ibm2 = reinterpret_cast<uint32_t*>(p);  p += (size_t)nq * nw * 4;
    uint32_t* t_mask = reinterpret_cast<uint32_t*>(p);  p += (size_t)nq * nw * 4;   // [row][nw] batch queries added to the cluster
    int32_t* t_fb = reinterpret_cast<int32_t*>(p);      p += (size_t)nq * 4;   // founder's batch index, -1 = pre-batch cluster
    int32_t* t_size = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;   // running Cluster.size()
    int32_t* t_fid = reinterpret_cast<int32_t*>(p);     p += (size_t)nq * 4;   // Cluster.getId()
    int32_t* t_count = reinterpret_cast<int32_t*>(p);   p += (size_t)nq * 4;   // running getUniqueSize()
    int32_t* t_tail = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;
    int32_t* t_nmem = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;   // batch queries the cluster received
    int32_t* t_first = reinterpret_cast<int32_t*>(p);   p += (size_t)nq * 4;   // the first of them
    int32_t* f_slot = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;   // cluster founded by batch query b
    int32_t* f_pick = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;   // which of its candidates the founder took
    int32_t* f_tidx = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;   // its row
    int32_t* s_bkid = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * kb * 4;
    int32_t* s_bksc = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * kb * 4;
    int32_t* s_bkab = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * kb * 4;
    int32_t* tc_c = reinterpret_cast<int32_t*>(p);      p += (size_t)nq * 4;
    int32_t* tc_cl = reinterpret_cast<int32_t*>(p);     p += (size_t)nq * 4;
    int32_t* tc_row = reinterpret_cast<int32_t*>(p);    p += (size_t)nq * 4;
    p = rs_raw + ((size_t)(p - rs_raw + 15) & ~(size_t)15);
    int4* s_best = reinterpret_cast<int4*>(p);           p += (size_t)nq * 16;   // per query: best static candidate (score, size, fid, slot)
    uint32_t* s_dirty = reinterpret_cast<uint32_t*>(p);  p += (((size_t)nw * 4 + 15) & ~(size_t)15);   // queries whose static list saw a change
    uint32_t* s_fmask = reinterpret_cast<uint32_t*>(p);  p += (((size_t)nw * 4 + 15) & ~(size_t)15);   // batch queries that founded a cluster in this batch
    int4* s_cand = reinterpret_cast<int4*>(p);           // cache: (slot, score, size, fid)
    __shared__ int32_t h_cons[HMK_HASH_SIZE];            // set: sequence ids consumed as partners in this batch
    __shared__ int32_t h_tkey[HMK_HASH_SIZE], h_trow[HMK_HASH_SIZE];   // map: cluster slot -> row
    __shared__ int32_t s_wb[32];                         // window scratch: partner taken by each lane
    __shared__ int32_t s_wpick[32];                      //   ... and which entry of its list that is
    __shared__ int s_ncached;                            // queries [0, s_ncached) have their candidates cached

    // the cluster search must have seen every founder hit (nothing below has touched the state yet)
    if (*B.hit_count > B.hit_cap) {
        if (threadIdx.x == 0) { S.ctl->status = HMK_P1_GROWHITS; S.ctl->pad0 = (int32_t)min(*B.hit_count, 0x7fffffffu); }
        return;
    }
    for (int i = threadIdx.x; i < HMK_HASH_SIZE; i += blockDim.x) { h_cons[i] = -1; h_tkey[i] = -1; }
    for (int i = threadIdx.x; i < nq; i += blockDim.x) {
        const int32_t q = B.qid[i];
        s_qid[i] = q; s_qab[i] = S.ab[q]; s_bkcnt[i] = B.bk_cnt[i]; s_bkovf[i] = B.bk_ovf[i]; s_acraw[i] = B.ac_cnt[i];
    }
    for (int i = threadIdx.x; i < nq * nw; i += blockDim.x) { s_ibm[i] = B.ibm[i]; s_ibm2[i] = B.ibm2[i]; }
    for (int i = threadIdx.x; i < nq * kb; i += blockDim.x) {
        const int32_t id = B.pcand[i];
        s_bkid[i] = id; s_bksc[i] = hmk_key_score(B.bk_key[i]); s_bkab[i] = S.ab[id];
    }
    __syncthreads();
    // The partner lists may have been computed while the previous batch was still resolving: whatever
    // stopped being a singleton since (queries or candidates) enters the consumed set up front.
    for (int i = threadIdx.x; i < nq * (kb + 1); i += blockDim.x) {
        const int b = i / (kb + 1), j = i % (kb + 1);
        if (j > 0 && j - 1 >= s_bkcnt[b]) continue;
        const int32_t id = j == 0 ? s_qid[b] : s_bkid[b * kb + j - 1];
        if (__ldcg(S.slot + id) < 0) continue;
        uint32_t h = hmk_hash((uint32_t)id);
        for (;;) {
            const int32_t v = atomicCAS(&h_cons[h], -1, id);
            if (v == -1 || v == id) break;
            h = (h + 1) & (HMK_HASH_SIZE - 1);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int run = 0, nc = 0;
        for (int i = 0; i < nq; i++) {
            s_acoff[i] = run;
            const int c = min(s_acraw[i], B.capq);
            if (nc == i && run + c <= cache_entries) { run += c; nc = i + 1; }
        }
        s_acoff[nq] = run;
        s_ncached = nc;
    }
    __syncthreads();
    const int ncached = s_ncached;
    {
        const int total = ncached ? s_acoff[ncached - 1] + min(s_acraw[ncached - 1], B.capq) : 0;
        for (int e = threadIdx.x; e < total; e += blockDim.x) {
            int lo = 0, hi = ncached - 1;          // query of entry e
            while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (s_acoff[mid] <= e) lo = mid; else hi = mid - 1; }
            s_cand[e] = B.ac_full[(size_t)lo * B.capq + (e - s_acoff[lo])];
        }
    }
    // each query's best pre-batch candidate (hmk_p1_prepare_candidates).  For cached queries it stays THE best as long
    // as none of their candidates changes (dirty bits); for every query its score stays an upper bound of what a
    // pre-batch cluster can offer, because complete-linkage scores only fall when members are added.
    for (int i = threadIdx.x; i < nw; i += blockDim.x) { s_dirty[i] = 0; s_fmask[i] = 0; }
    for (int i = threadIdx.x; i < nq; i += blockDim.x) s_best[i] = B.best[i];
    __syncthreads();
    if (threadIdx.x >= 32) return;
    HMK_TICK(0);   // staging

    const int lane = threadIdx.x;
    const unsigned FULL = 0xffffffffu;
    int fresh_joins = 0;            // pre-batch clusters changed in this batch (each costs a scan of the cache)
    bool all_dirty = false;
    HmkCtl* ctl = S.ctl;
    int32_t ncl = ctl->ncl, unproc = ctl->unproc_alive;
    int32_t steps = ctl->steps, joins = ctl->joins, creates = ctl->creates, orphans = ctl->orphans;
    int32_t status = HMK_P1_CONTINUE, npe_step = -1, cur = ctl->cur;
    int32_t tn = 0;                 // rows of the touched table

    auto consumed = [&](int32_t id) -> bool {
        uint32_t h = hmk_hash((uint32_t)id);
        for (;;) {
            const int32_t v = h_cons[h];
            if (v == id) return true;
            if (v < 0) return false;
            h = (h + 1) & (HMK_HASH_SIZE - 1);
        }
    };
    auto touched_row = [&](int32_t c) -> int {
        uint32_t h = hmk_hash((uint32_t)c);
        for (;;) {
            const int32_t v = h_tkey[h];
            if (v == c) return h_trow[h];
            if (v < 0) return -1;
            h = (h + 1) & (HMK_HASH_SIZE - 1);
        }
    };
    // complete linkage over the members cluster row `row` received in this batch, evaluated by ONE
    // lane (lanes work on different candidate clusters in parallel): every batch query that joined
    // must be in the hit mask of query b, a partner must score >= T (table pd), then the minimum
    auto eval_touched = [&](int row, int b, int32_t& cl) -> bool {
        const uint32_t* tm = t_mask + row * nw;
        const uint32_t* hm = s_ibm + b * nw;
        const int32_t* ibr = B.ib + (size_t)b * B.ib_stride;     // S(member = batch query b2, query b): the few entries
        const int32_t* pdr = B.pd + (size_t)b * B.pd_stride;     // a step needs are read straight from L2
        const int32_t fb = t_fb[row];
        if (t_nmem[row] == 1) {     // the usual case: one batch query (+ its partner if the cluster was born here)
            const int b2 = t_first[row];
            if (((hm[b2 >> 5] >> (b2 & 31)) & 1u) == 0) return false;
            int32_t mn1 = __ldcg(ibr + b2);
            if (fb >= 0) {
                const int32_t s = __ldcg(pdr + fb * kb + f_pick[fb]);
                if (s < S.T) return false;
                mn1 = s < mn1 ? s : mn1;
            }
            cl = mn1 < cl ? mn1 : cl;
            return true;
        }
        for (int w = 0; w < nw; w++)
            if (tm[w] & ~hm[w]) return false;
        int32_t mn = cl;
        if (fb >= 0) {     // cluster born in this batch: its partner was one of the founder's candidates
            const int32_t s = __ldcg(pdr + fb * kb + f_pick[fb]);
            if (s < S.T) return false;
            mn = s < mn ? s : mn;
        }
        for (int w = 0; w < nw; w++) {
            uint32_t m = tm[w];
            while (m) {
                const int b2 = w * 32 + __ffs(m) - 1;
                m &= m - 1;
                const int32_t s = __ldcg(ibr + b2);
                mn = s < mn ? s : mn;
            }
        }
        cl = mn;
        return true;
    };
    // ------------------------------------------------------------------------------------------------
    // Most steps are "q founds a new cluster with its best still-alive partner" and do not interact with
    // their neighbours.  A WINDOW of up to 32 consecutive batch queries is therefore evaluated with one
    // query per lane against the state at the window start; a lane is only trusted if
    //   * it is a plain case: consumed query (skipped), new pair, or orphan -- joins, truncated lists, ... take
    //     the sequential path below,
    //   * no cluster it could join can reach its partner's score: the best pre-batch cluster's score at batch
    //     start (later members only lower it) and the FOUNDER score S(founder, q) of every cluster born in
    //     this batch (complete linkage <= founder score) are all below the partner score -- this includes
    //     the pairs created by earlier lanes of the window,
    //   * no earlier lane of the window takes its partner or the query itself, and K is not reached.
    // The longest prefix of trusted lanes is applied in parallel (cluster ids = creation order), the first
    // untrusted step runs sequentially, and the next window starts behind it.  Same decisions, same order.
    // ------------------------------------------------------------------------------------------------
    int b = 0, penalty = 0;
    int n_win = 0, n_win_steps = 0, n_seq = 0;      // statistics: windows tried, lanes they applied, sequential steps
    while (b < nq) {
        HMK_TRACE(0, b); HMK_TRACE(1, 1);
#ifdef HMK_NO_WINDOW
        penalty = 1;
#endif
        if (penalty == 0 && ncl > 0 && ncl < S.K && unproc > 96) {
            const int W = min(32, nq - b);
            const int bi = b + lane;
            const bool in = lane < W;
            const int32_t q = in ? s_qid[bi] : -1;
            // 0 = skip (already consumed), 1 = new pair, 2 = orphan, 3 = sequential path
            int kind = 3;
            int32_t bid = -1, bscore = HMK_JMIN;
            int bpick = 0;
            if (in) {
                if (consumed(q)) kind = 0;
                else if (s_acraw[bi] <= B.capq) {
                    const int bcnt = s_bkcnt[bi];
                    int pick = -1;
                    for (int j = 0; j < bcnt; j++)
                        if (pick < 0 && !consumed(s_bkid[bi * kb + j])) pick = j;
                    if (!(pick < 0 && s_bkovf[bi])) {
                        // best pre-batch candidate at batch start: its score bounds every pre-batch cluster's
                        // current score from above (members only lower a complete-linkage score)
                        const int4 sb = s_best[bi];      // (score, size, fid, slot)
                        if (pick >= 0) {
                            bpick = pick; bid = s_bkid[bi * kb + pick]; bscore = s_bksc[bi * kb + pick];
                            if (!(sb.w >= 0 && sb.x >= bscore)) kind = 1;
                        } else if (sb.w < 0) kind = 2;
                    }
                }
            }
            __syncwarp();
            HMK_TICK(7);   // window: partner pick
            HMK_TRACE(1, 2);
            // Clusters born in this batch (before the window, or by earlier lanes of it): such a cluster is {founder b2,
            // the partner b2 picked, ...}, so min(S(founder, q), S(partner, q)) bounds its complete-linkage score from
            // above (further members only lower it).  A lane stays trusted if no such cluster can reach what the lane
            // is about to do: for a new pair, a bound >= T that also reaches the partner's score would make the reference
            // join instead; an orphan joins any valid cluster.  The bit masks pre-select the founders worth a look
            // (ibm2: founder score >= T and >= the lowest listed partner score; ibm: founder score >= T); the two
            // scores themselves come from the dense tables ib / pd.
            const unsigned cm0 = __ballot_sync(FULL, kind == 1);
            const unsigned lt = (1u << lane) - 1u;
            s_wpick[lane] = bpick;
            __syncwarp();
            {
                const int w0 = b >> 5, sh = b & 31;
                const unsigned mine = cm0 & lt;
                const uint32_t* hmrow = kind == 1 ? s_ibm2 + bi * nw : s_ibm + bi * nw;
                const int32_t need = kind == 1 ? (bscore > S.T ? bscore : S.T) : S.T;
                bool threat = false;
                if (kind == 1 || kind == 2) {
                    for (int w = 0; w < nw && !threat; w++) {
                        uint32_t m = s_fmask[w];
                        m |= w == w0 ? mine << sh : 0u;
                        m |= (w == w0 + 1 && sh) ? mine >> (32 - sh) : 0u;
                        m &= hmrow[w];
                        while (m && !threat) {
                            const int b2 = w * 32 + __ffs(m) - 1;
                            m &= m - 1;
                            const int pk = b2 >= b ? s_wpick[b2 - b] : f_pick[b2];      // founded by an earlier lane of this window?
                            const int32_t sf = __ldcg(B.ib + (size_t)bi * B.ib_stride + b2);
                            const int32_t sp = __ldcg(B.pd + (size_t)bi * B.pd_stride + b2 * kb + pk);
                            threat = (sf < sp ? sf : sp) >= need;
                        }
                    }
                }
                if (threat) kind = 3;
            }
            __syncwarp();
            HMK_TICK(6);   // window: founder bounds
            HMK_TRACE(1, 3);
            // partners / queries taken by earlier lanes of the window
            bool bad = in && kind == 3;
            {
                s_wb[lane] = kind == 1 ? bid : -1;
                __syncwarp();
                bool taken = false;
#pragma unroll
                for (int j = 0; j < 32; j++) taken |= (j < lane) & (s_wb[j] == q);
                const unsigned same = __match_any_sync(FULL, kind == 1 ? bid : -2 - lane);
                bad |= in && kind != 0 && (taken || (same & lt) != 0);
                __syncwarp();
            }
            if (in && ncl + __popc(cm0 & lt) >= S.K) bad = true;          // :90, checked before anything else of a step
            const unsigned badm = __ballot_sync(FULL, bad || !in);
            const int Pn = badm ? __ffs(badm) - 1 : 32;      // lanes [0, Pn) are applied
            HMK_TRACE(1, 4); HMK_TRACE(2, Pn);
            n_win++; n_win_steps += Pn;
            HMK_TICK(2);
            if (Pn > 0) {
                const bool act = lane < Pn;
                const unsigned cm = __ballot_sync(FULL, act && kind == 1);
                const unsigned om = __ballot_sync(FULL, act && kind == 2);
                if (act && kind == 1) {
                    const int r = __popc(cm & lt);
                    const int32_t c = ncl + r;
                    const int row = tn + r;
                    HMK_CHECK(c < S.K && row < HMK_MAXBATCH && q >= 0 && q < S.n && bid > q && bid < S.n && S.slot[q] < 0);
                    for (int w = 0; w < nw; w++) t_mask[row * nw + w] = 0;
                    t_mask[row * nw + (bi >> 5)] = 1u << (bi & 31);
                    uint32_t h = hmk_hash((uint32_t)c);
                    while (atomicCAS(&h_tkey[h], -1, c) != -1) h = (h + 1) & (HMK_HASH_SIZE - 1);
                    h_trow[h] = row;
                    const int32_t sz = hmk_wadd(s_qab[bi], s_bkab[bi * kb + bpick]);
                    t_nmem[row] = 1; t_first[row] = bi; t_fb[row] = bi; t_fid[row] = q;
                    t_count[row] = 2; t_tail[row] = bid; t_size[row] = sz;
                    f_slot[bi] = c; f_pick[bi] = bpick; f_tidx[bi] = row;
                    S.c_founder[c] = q; S.c_tail[c] = bid; S.c_count[c] = 2; S.c_size[c] = sz;
                    S.next[q] = bid; S.next[bid] = -1;
                    S.slot[q] = c; S.rank[q] = 0; S.slot[bid] = c; S.rank[bid] = 1;
                    h = hmk_hash((uint32_t)bid);
                    while (atomicCAS(&h_cons[h], -1, bid) != -1) h = (h + 1) & (HMK_HASH_SIZE - 1);
                }
                if (act && kind != 0 && S.qbatch) S.qbatch[q] = B.batch_id;
                {   // founder mask: window bit i is batch query b + i
                    const int w0 = b >> 5, sh = b & 31;
                    if (lane == w0) s_fmask[lane] |= cm << sh;
                    else if (lane == w0 + 1 && sh) s_fmask[lane] |= cm >> (32 - sh);
                }
                const int nC = __popc(cm), nO = __popc(om);
                ncl += nC; tn += nC; creates += nC; orphans += nO;
                steps += nC + nO; unproc -= 2 * nC + nO;
                const unsigned done = cm | om;
                if (done) cur = __shfl_sync(FULL, q, 31 - __clz(done)) + 1;
                __syncwarp();
                b += Pn;
            }
            penalty = Pn >= 4 ? 0 : 4;      // crowded stretch: a few sequential steps before the next attempt
            HMK_TICK(1);   // window
            if (Pn == W) continue;
        } else if (penalty > 0) penalty--;

        // ---- one step in reference order
        HMK_TRACE(1, 5);
        n_seq++;
        const int32_t q = s_qid[b];
        if (ncl >= S.K) { status = HMK_P1_DONE; cur = q; break; }                   // :90
        if (consumed(q)) { b++; continue; }   // taken as a partner earlier in this batch (:101,110)
        const int32_t acnt = s_acraw[b];
        if (acnt > B.capq) { status = HMK_P1_GROW; cur = q; break; }   // candidate arrays too small: host grows them
        const int32_t bcnt = s_bkcnt[b];
        uint32_t fmask = lane < nw ? s_fmask[lane] : 0u;   // this lane's word of the founder mask

        // ---- B: nearest among initialList[index+1 ..]                               (:93)
        int bkind = 0;   // 0 = Java null, 1 = found, 2 = (null cluster, MIN_VALUE) object
        int32_t bscore = HMK_JMIN, bid = -1, bpick = 0;
        if (unproc - 1 == 0) bkind = 2;            // empty sub-list (ClinkageSequenceClusterer.java:138-140)
        else {
            const bool alive = lane < bcnt && !consumed(s_bkid[b * kb + lane]);
            const unsigned am = __ballot_sync(FULL, alive);
            if (am) {
                bpick = __ffs(am) - 1;              // list is sorted: first alive entry wins
                bid = s_bkid[b * kb + bpick];
                bscore = s_bksc[b * kb + bpick];
                bkind = 1;
            } else if (s_bkovf[b]) {
                status = HMK_P1_RESTART; cur = q; break;    // list truncated: rescore from q
            }
        }
        HMK_TRACE(1, 6);
        HMK_TRACE(1, 7);
        HMK_TRACE_CLEAR();
        HMK_TRACE_LANES(4);

        HMK_TICK(2);   // consumed check + B part
        // ---- A: nearest among actualClusters (complete linkage)                      (:92)
        int akind = 0;
        HmkBestCluster best;
        best.score = HMK_JMIN; best.size = 0; best.fid = 0; best.slot = -1;
        if (ncl == 0) akind = 2;
        else {
            const uint32_t hm = lane < nw ? s_ibm[b * nw + lane] : 0u;
            int nt = 0;   // touched candidates collected for this step (warp-uniform)
            const bool clean = b < ncached && !all_dirty && ((s_dirty[b >> 5] >> (b & 31)) & 1u) == 0;
            if (clean) {   // none of this query's pre-batch candidates changed: the staged best is final
                const int4 v = s_best[b];
                if (lane == 0 && v.w >= 0) { best.score = v.x; best.size = v.y; best.fid = v.z; best.slot = v.w; }
            }
            // pre-batch clusters: untouched ones are final, touched ones need the batch members too
            for (int e0 = 0; !clean && e0 < acnt; e0 += 32) {
                const int e = e0 + lane;
                int32_t c = -1, cl = 0;
                int row = -1;
                if (e < acnt) {
                    int32_t sz, fd;
                    if (b < ncached) { const int4 v = s_cand[s_acoff[b] + e]; c = v.x; cl = v.y; sz = v.z; fd = v.w; }
                    else { const int4 v = B.ac_full[(size_t)b * B.capq + e]; c = v.x; cl = v.y; sz = v.z; fd = v.w; }
                    row = tn ? touched_row(c) : -1;
                    if (row < 0) hmk_consider(best, cl, sz, fd, c);
                }
                const unsigned tmk = __ballot_sync(FULL, row >= 0);
                if (row >= 0) {
                    const int pos = nt + __popc(tmk & ((1u << lane) - 1u));
                    tc_c[pos] = c; tc_cl[pos] = cl; tc_row[pos] = row;
                }
                nt += __popc(tmk);
            }
            HMK_TRACE_LANES(5);
            HMK_TRACE(1, 71); HMK_TRACE(3, nt);
            HMK_TICK(3);   // static candidates
            // clusters born in this batch whose founder scores >= T
            {
                const uint32_t bits = fmask & hm;
                const unsigned anyb = __ballot_sync(FULL, bits != 0);
                if (anyb) {
                    int mine = __popc(bits), pre = mine;
#pragma unroll
                    for (int d2 = 1; d2 < 32; d2 <<= 1) { const int v = __shfl_up_sync(FULL, pre, d2); if (lane >= d2) pre += v; }
                    const int total = __shfl_sync(FULL, pre, 31);
                    int pos = nt + pre - mine;
                    uint32_t m = bits;
                    while (m) {
                        const int b2 = lane * 32 + __ffs(m) - 1;
                        m &= m - 1;
                        tc_c[pos] = f_slot[b2]; tc_cl[pos] = HMK_JMAX; tc_row[pos] = f_tidx[b2];
                        pos++;
                    }
                    nt += total;
                }
            }
            HMK_TRACE_LANES(6);
            HMK_TRACE(1, 72); HMK_TRACE(3, nt);
            if (nt) {
                __syncwarp();
                HMK_TRACE(1, 721);
                for (int i0 = 0; i0 < nt; i0 += 32) {
                    const int i = i0 + lane;
                    if (i < nt) {
                        const int row = tc_row[i];
                        int32_t cl2 = tc_cl[i];
                        if (eval_touched(row, b, cl2)) hmk_consider(best, cl2, t_size[row], t_fid[row], tc_c[i]);
                    }
                }
                HMK_TRACE(1, 722);
                __syncwarp();
            }
            HMK_TRACE_LANES(7);
            HMK_TRACE(1, 73);
            if (clean && nt == 0) {      // only lane 0 holds a candidate: broadcast instead of reducing
                best.score = __shfl_sync(FULL, best.score, 0); best.size = __shfl_sync(FULL, best.size, 0);
                best.fid = __shfl_sync(FULL, best.fid, 0); best.slot = __shfl_sync(FULL, best.slot, 0);
            } else hmk_best_reduce(best);
            if (best.slot >= 0) akind = 1;
        }

        HMK_TRACE(1, 8);
        HMK_TICK(4);   // founders + touched evaluation + reduce
        // ---- decision                                                               (:94-114)
        const int32_t ascore = akind == 1 ? best.score : HMK_JMIN;
        bool join = false, create = false;
        if (akind != 0) {
            if (bkind != 0) { if (ascore >= bscore) join = true; else create = true; }
            else join = true;
        } else if (bkind != 0) create = true;
        if ((join && akind == 2) || (create && bkind == 2)) {    // null.insertAll / null.getSequences
            status = HMK_P1_NPE; npe_step = steps; cur = q; break;
        }
        if (join || create) {
            const int32_t c = join ? best.slot : ncl;
            int row = create ? -1 : (tn ? touched_row(c) : -1);
            const bool fresh = row < 0;
            if (fresh) {
                row = tn++;
                if (lane < nw) t_mask[row * nw + lane] = 0;
                if (lane == 0) {
                    uint32_t h = hmk_hash((uint32_t)c);
                    while (h_tkey[h] >= 0) h = (h + 1) & (HMK_HASH_SIZE - 1);
                    h_tkey[h] = c; h_trow[h] = row;
                    t_nmem[row] = 0; t_first[row] = b;
                    if (create) { t_fb[row] = b; t_size[row] = 0; t_fid[row] = q; t_count[row] = 0; t_tail[row] = -1; }
                    else {       // first change of a pre-batch cluster in this batch: fetch its running state
                        t_fb[row] = -1; t_size[row] = __ldcg(S.c_size + c); t_fid[row] = __ldcg(S.c_founder + c);
                        t_count[row] = __ldcg(S.c_count + c); t_tail[row] = __ldcg(S.c_tail + c);
                    }
                }
                if (!create && !all_dirty) {
                    // later queries that list this cluster can no longer use their staged best
                    if (++fresh_joins > 32) all_dirty = true;
                    else if (b + 1 < ncached) {
                        const int e_lo = s_acoff[b + 1], e_hi = s_acoff[ncached - 1] + min(s_acraw[ncached - 1], B.capq);
                        for (int e = e_lo + lane; e < e_hi; e += 32) {
                            if (s_cand[e].x == c) {
                                int lo = b + 1, hi = ncached - 1;
                                while (lo < hi) { int mid = (lo + hi + 1) >> 1; if (s_acoff[mid] <= e) lo = mid; else hi = mid - 1; }
                                atomicOr(&s_dirty[lo >> 5], 1u << (lo & 31));
                            }
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == (b >> 5)) t_mask[row * nw + lane] |= 1u << (b & 31);
            if (create && lane == (b >> 5)) s_fmask[lane] |= 1u << (b & 31);
            if (lane == 0) {
                HMK_CHECK(row >= 0 && row < HMK_MAXBATCH && c >= 0 && c < S.K && q >= 0 && q < S.n && S.slot[q] < 0);
                HMK_CHECK(join || (bid > q && bid < S.n));
                t_nmem[row] += 1;
                if (join) {                                               // insertAll({q})   (:97,104)
                    S.next[t_tail[row]] = q; S.next[q] = -1;
                    S.rank[q] = t_count[row]; S.slot[q] = c;
                    t_tail[row] = q; t_count[row] += 1; t_size[row] = hmk_wadd(t_size[row], s_qab[b]);
                } else {                                                  // new cluster {q, partner}   (:99-101,108-110)
                    f_slot[b] = c; f_pick[b] = bpick; f_tidx[b] = row;
                    S.c_founder[c] = q;
                    S.next[q] = bid; S.next[bid] = -1;
                    S.slot[q] = c; S.rank[q] = 0; S.slot[bid] = c; S.rank[bid] = 1;
                    t_tail[row] = bid; t_count[row] = 2; t_size[row] = hmk_wadd(s_qab[b], s_bkab[b * kb + bpick]);
                    uint32_t h = hmk_hash((uint32_t)bid);
                    while (h_cons[h] >= 0) h = (h + 1) & (HMK_HASH_SIZE - 1);
                    h_cons[h] = bid;
                }
                S.c_tail[c] = t_tail[row]; S.c_count[c] = t_count[row]; S.c_size[c] = t_size[row];   // write through
            }
        }
        if (join) joins++;
        else if (create) { ncl++; unproc--; creates++; }
        else orphans++;
        steps++;
        unproc--;
        cur = q + 1;
        if (lane == 0 && S.qbatch) S.qbatch[q] = B.batch_id;
        __syncwarp();
        HMK_TICK(5);   // decision + apply
        b++;
    }
    if (status == HMK_P1_CONTINUE && (ncl >= S.K || unproc <= 0)) status = HMK_P1_DONE;
#ifdef HMK_RESOLVE_TIMING
    if (lane == 0) for (int i = 0; i < 8; i++) ctl->dbg[i] += dbg[i];
#endif
    if (lane == 0) {
        ctl->cnt[0] += n_win; ctl->cnt[1] += n_win_steps; ctl->cnt[2] += n_seq;
        ctl->cur = cur; ctl->ncl = ncl; ctl->unproc_alive = unproc; ctl->status = status;
        if (npe_step >= 0) ctl->npe_step = npe_step;
        ctl->steps = steps; ctl->joins = joins; ctl->creates = creates; ctl->orphans = orphans;
        if (status == HMK_P1_RESTART) ctl->restarts += 1;
        if (status != HMK_P1_CONTINUE) ctl->discards += 1;     // cancels the partner searches prepared behind this batch
    }
}

// ---------------------------------------------------------------- phase 2: windowed resolution
// Candidate pairs (query q, cluster c) -- founder and every phase-1 member score >= T -- are
// held grouped by query (cq_*).  Queries are resolved in windows of consecutive queries.
// Inside a window the reference's sequential decisions
// (LimitedGreedySequenceClusterer.java:59-66) are the unique fixed point of
//     A[q] = best valid cluster of q given { q' < q : A[q'] = c } as extra members of c,
// reached by iterating that map from A = "nobody joins" (after t iterations the first t
// queries are final; in practice a handful of iterations suffice).  Members that joined in
// earlier windows are final.
//
// Per cluster the joiners live in one array dyn[cstart[c] ..]: first the dyn_n[c] FINAL phase-2 members
// (query indices, join order == query order), then the tent_n[c] tentative joiners of the current
// iteration, sorted.  Room: a cluster can never receive more joiners than it has candidate pairs.
//
// Iterations are enqueued in groups without a host round trip: iteration `it` leaves flags[it % R] != 0
// iff some assignment changed, and every kernel of iteration it > 0 returns at once when the previous
// iteration did not change anything (the fixed point has been reached; nothing may be touched any more).
// Buffers indexed by iteration parity: a[2][ns], dirty[2][ncl], tent_n[2][ncl].
#define HMK_P2_CLEAN 0x7f7f7f7f
#define HMK_P2_CHG 1024          // changed clusters listed per iteration; more: every query gathers dirty[] itself

// one joiner of a cluster: everything a later query needs to score against it comes with ONE 16-byte load
struct __align__(16) HmkDynEntry {
    uint64_t w;     // packed residues (uniform length <= 12), else unused
    int32_t qi;     // query index (into singles)
    int32_t ab;     // abundance
};
// per cluster, one 16-byte record: [0] offset into dyn, [1] final phase-2 members, [2] tentative joiners, [3] unused
#define HMK_CI 4
// control words of a window (P.ctl): per parity [0..1] work-list entries, [2..3] entries consumed, [4..5] clusters on the
// changed list, [6..7] "some assignment changed"; [8] iterations the window took (read by the host)
#define HMK_P2_CTL 16

struct HmkP2 {
    HmkState S;
    const uint64_t* packed;   // NULL -> generic scalar scorer
    int32_t L;
    int32_t ncl, ns;
    const int32_t* singles;   // [ns] ascending ids of the phase-2 queries
    const int32_t* qstart;    // [ns+1] into cq_*
    const int32_t* cq_c;      // candidate cluster slot (ascending inside a query)
    const int32_t* cq_q;      // query index of the pair
    const int32_t* cq_s;      // complete-linkage min over the phase-1 members ("static" score)
    const int32_t* cstart;    // [ncl+1] candidate pairs per cluster, prefix sums
    const int32_t* cc_q;      // the pairs grouped by cluster: query indices, ascending inside a cluster
    int32_t* base_cl;         // per pair: static score with the first FINAL phase-2 member folded in; HMK_JMIN = some final member scores < T
    int32_t* cinfo;           // [ncl][HMK_CI]
    HmkDynEntry* dyn;         // per cluster: final members (join order == query order), then the tentative joiners in query order
    int32_t* a;               // [ns] tentative assignment (-1 = none)
    int32_t* dirty;           // [ncl] smallest query whose tentative assignment to/from c changed in the last iteration
    int32_t* stamp;           // [ns] generation in which the query was last put on a work list
    int32_t* work;            // [2][wcap] queries to re-evaluate
    int32_t* chg;             // [2][HMK_P2_CHG] clusters whose tentative joiner list changed in the last iteration
    int32_t* ctl;             // [HMK_P2_CTL]
    int32_t wcap;
    unsigned long long* pair_parts;   // scalar pair-score counter, sharded over HMK_PAIR_SHARDS cache lines
    int32_t qa, qb;           // window = queries [qa, qb)
    int32_t gen0;             // generation of the window's first iteration (unique across windows)
    int32_t max_iters;
    unsigned long long* tim;  // optional [64] phase boundaries in ns (profiling builds): start, base, then R / D ends per iteration
};

// candidate pairs per cluster (cq_c is grouped by query, so neighbours rarely collide)
__global__ void hmk_p2_count_clusters(const int32_t* __restrict__ cq_c, int n, int32_t* __restrict__ cnt) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) atomicAdd(cnt + cq_c[i], 1);
}

// single block: out[0..n] = exclusive prefix sums of cnt[0..n)
__global__ void __launch_bounds__(1024) hmk_exclusive_scan(const int32_t* __restrict__ cnt, int n, int32_t* __restrict__ out) {
    __shared__ int32_t part[1024];
    const int per = (n + blockDim.x - 1) / blockDim.x;
    const int lo = min(n, (int)threadIdx.x * per), hi = min(n, lo + per);
    int32_t s = 0;
    for (int i = lo; i < hi; i++) s += cnt[i];
    part[threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t run = 0;
        for (int i = 0; i < (int)blockDim.x; i++) { const int32_t v = part[i]; part[i] = run; run += v; }
        out[n] = run;
    }
    __syncthreads();
    int32_t run = part[threadIdx.x];
    for (int i = lo; i < hi; i++) { out[i] = run; run += cnt[i]; }
}

__global__ void hmk_p2_init_cinfo(int ncl, const int32_t* __restrict__ cstart, int32_t* __restrict__ cinfo) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ncl) return;
    reinterpret_cast<int4*>(cinfo)[c] = make_int4(cstart[c], 0, 0, 0);
}

// S(member entry, query) -- FAST: hmk_score12x3 on the entry's packed word; else the general scalar scorer
template <bool FAST>
struct HmkQueryScorer {
    const HmkP2& P;
    HmkScalar sc;
    int32_t q;
    int32_t qrow[HMK_MAXL1];
    __device__ __forceinline__ HmkQueryScorer(const HmkP2& P_, const int32_t* sM, int32_t q_) : P(P_), q(q_) {
        sc.packed = P.packed; sc.sM = sM; sc.L = P.L;
        if (FAST) hmk_qrow12(P.packed[q], qrow);
    }
    __device__ __forceinline__ int32_t score(const HmkDynEntry& m) const {
        if (FAST) return hmk_score12x3(qrow, m.w, sc.sM, P.S.P);
        return hmk_scalar_score(P.S, sc, P.singles[m.qi], q);
    }
};

// The decision of one query given the tentative joiners before it (one warp).
// Evaluation is lazy: the static score of a pair bounds its final score from above, so a candidate whose static score
// is below the best valid score found so far is never evaluated.  The base pass has already folded the first final member
// of every cluster into base_cl (and killed almost every unrelated candidate), so per chunk of 32 candidates the few
// survivors are evaluated one after the other, best static score first, with the 32 lanes striding over the member list.
// Every global load chain is short: pair -> cluster record (16 B) -> member entry (16 B, carries the packed word).
template <bool FAST>
__device__ __forceinline__ void hmk_p2_decide_query(const HmkP2& P, const int32_t* sM, int qi, int par, long long& npairs) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int32_t T = P.S.T;
    const int4* cinfo = reinterpret_cast<const int4*>(P.cinfo);
    const int e0 = P.qstart[qi], e1 = P.qstart[qi + 1];
    const int32_t old = P.a[qi];
    const int32_t q = P.singles[qi];
    const HmkQueryScorer<FAST> scorer(P, sM, q);
    HmkBestCluster best;        // warp-uniform
    best.score = HMK_JMIN; best.size = 0; best.fid = 0; best.slot = -1;
    for (int eb = e0; eb < e1; eb += 32) {
        const int e = eb + lane;
        int32_t c = -1, st = HMK_JMIN, cl = HMK_JMIN, off = 0, nd = 0, tn = 0;
        if (e < e1) { cl = P.base_cl[e]; st = P.cq_s[e]; c = P.cq_c[e]; }
        const bool alive = cl != HMK_JMIN && !(best.slot >= 0 && st < best.score);
        if (alive) { const int4 ci = cinfo[c]; off = ci.x; nd = ci.y; tn = ci.z; }
        const int start = nd > 0 ? 1 : 0;             // member 0 of the final members is in base_cl already
        const bool more = alive && nd + tn > start;
        {   // candidates without further members are decided: fold them into the warp's best (prunes the rest)
            HmkBestCluster mine;
            mine.score = HMK_JMIN; mine.size = 0; mine.fid = 0; mine.slot = -1;
            if (alive && !more) hmk_consider(mine, cl, P.S.c_size[c], P.S.c_founder[c], c);
            if (__any_sync(FULL, mine.slot >= 0)) {
                hmk_best_reduce(mine);
                if (mine.slot >= 0) hmk_consider(best, mine.score, mine.size, mine.fid, mine.slot);
            }
        }
        unsigned todo = __ballot_sync(FULL, more);
        while (todo) {                    // survivors with more members, best static score first
            const bool in_todo = (todo >> lane) & 1u;
            const int32_t mx = __reduce_max_sync(FULL, in_todo ? st : HMK_JMIN);
            if (best.slot >= 0 && mx < best.score) break;          // nothing left can reach the best any more
            const int pick = __ffs(__ballot_sync(FULL, in_todo && st == mx)) - 1;
            const int32_t poff = __shfl_sync(FULL, off, pick), pnd = __shfl_sync(FULL, nd, pick),
                          ptot = pnd + __shfl_sync(FULL, tn, pick);
            bool ok = true, final_fail = false;
            int32_t mn = HMK_JMAX;
            uint32_t sz = 0;
            for (int i0 = pnd > 0 ? 1 : 0; i0 < ptot; i0 += 32) {
                const int i = i0 + lane;
                bool act = i < ptot;
                HmkDynEntry m;
                m.w = 0; m.qi = 0; m.ab = 0;
                HMK_CHECK(!act || (poff >= 0 && poff + i < P.cstart[P.ncl]));
                if (act) m = P.dyn[poff + i];
                const bool behind = act && i >= pnd && m.qi >= qi;      // tentative joiners at or behind q do not count
                act = act && !behind;
                bool bad = false;
                if (act) {
                    const int32_t s = scorer.score(m);
                    npairs++;
                    bad = s < T;
                    mn = s < mn ? s : mn;
                    if (i >= pnd) sz += (uint32_t)m.ab;
                }
                const unsigned badm = __ballot_sync(FULL, bad);
                if (badm) { ok = false; final_fail = __any_sync(FULL, bad && i < pnd); break; }
                if (__any_sync(FULL, behind)) break;                  // in query order: everything further is behind q as well
            }
            mn = __reduce_min_sync(FULL, mn);
            sz = __reduce_add_sync(FULL, sz);
            int32_t k_cl = 0, k_size = 0, k_fid = 0, k_c = -1;
            if (lane == pick) {
                if (!ok && final_fail) P.base_cl[e] = HMK_JMIN;
                if (ok) { k_cl = mn < cl ? mn : cl; k_size = (int32_t)((uint32_t)P.S.c_size[c] + sz); k_fid = P.S.c_founder[c]; k_c = c; }
            }
            if (ok) {
                k_cl = __shfl_sync(FULL, k_cl, pick); k_size = __shfl_sync(FULL, k_size, pick);
                k_fid = __shfl_sync(FULL, k_fid, pick); k_c = __shfl_sync(FULL, k_c, pick);
                hmk_consider(best, k_cl, k_size, k_fid, k_c);
            }
            todo &= ~(1u << pick);
        }
    }
    if (lane == 0 && best.slot != old) {
        P.a[qi] = best.slot;
        P.ctl[6 + par] = 1;
        const int32_t two[2] = {old, best.slot};
        for (int k = 0; k < 2; k++) {
            const int32_t c = two[k];
            if (c < 0) continue;
            if (atomicMin(P.dirty + c, qi) == HMK_P2_CLEAN) {       // first change of this cluster in this iteration
                const int pos = atomicAdd(P.ctl + 4 + par, 1);
                HMK_CHECK(pos >= 0 && pos < P.ncl);
                if (pos < HMK_P2_CHG) P.chg[(size_t)par * HMK_P2_CHG + pos] = c;
            }
        }
    }
    __syncwarp();
}

// ONE cooperative launch resolves one window: setup, base pass, the fixed-point iterations and the commit are phases of
// the same grid separated by grid-wide barriers, so an iteration that re-evaluates a handful of queries costs a few
// microseconds instead of several launches and a host round trip.
//   setup   per cluster: nobody joins
//   base    one thread per candidate pair of the window: fold the FIRST final phase-2 member of the cluster into the
//           pair's score (HMK_JMIN if it scores < T).  Unrelated candidates -- nearly all of them -- die here.
//   iteration t:
//     R  (t > 0) one warp per cluster whose joiners changed in iteration t-1 walks the cluster's candidate queries of the
//        window (grouped by cluster, ascending): those currently assigned to it become its tentative joiner list, in
//        query order; those behind the first change are put on the work list (once: generation stamp)
//     D  warps take queries off the work list (iteration 0: the whole window) and decide them
//   until an iteration changes nothing; commit: the tentative joiners become final members.
template <bool FAST>
__global__ void __launch_bounds__(256) hmk_p2_window(const HmkP2 P) {
    namespace cg = cooperative_groups;
    cg::grid_group grid = cg::this_grid();
    __shared__ int32_t sM[HMK_NRES * HMK_NRES];
    hmk_load_matrix_smem(sM, P.S.M);
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
    const int gwarp = gtid >> 5, gwarps = gthreads >> 5;
    long long npairs = 0;
    // ---- setup + base
    for (int c = gtid; c < P.ncl; c += gthreads) { P.cinfo[c * HMK_CI + 2] = 0; P.dirty[c] = HMK_P2_CLEAN; }
    if (gtid < HMK_P2_CTL) P.ctl[gtid] = 0;
    {
        const int e0 = P.qstart[P.qa], e1 = P.qstart[P.qb];
        for (int e = e0 + gtid; e < e1; e += gthreads) {
            const int32_t c = P.cq_c[e];
            const int32_t nd = P.cinfo[c * HMK_CI + 1];
            int32_t cl = P.cq_s[e];
            if (nd > 0) {                                  // the cluster has final phase-2 members
                const HmkDynEntry m = P.dyn[P.cinfo[c * HMK_CI]];
                const HmkQueryScorer<FAST> scorer(P, sM, P.singles[P.cq_q[e]]);
                const int32_t s = scorer.score(m);
                npairs++;
                cl = s < P.S.T ? HMK_JMIN : (s < cl ? s : cl);
            }
            P.base_cl[e] = cl;
        }
    }
    grid.sync();
    int tslot = 0;
    auto mark_time = [&]() {
        if (P.tim && gtid == 0 && tslot < 64) { unsigned long long ns; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(ns)); P.tim[tslot] = ns; }
        tslot++;
    };
    mark_time();
    int t = 0;
    for (;; t++) {
        const int par = t & 1;
        if (t > 0) {
            // ---- R: rebuild the joiner lists of the clusters that changed, and collect the queries behind the changes
            const int nchg = P.ctl[4 + (par ^ 1)];
            const int32_t gen = P.gen0 + t;
            int32_t* work = P.work + (size_t)par * P.wcap;
            const bool listed = nchg <= HMK_P2_CHG;
            const int ncl_it = listed ? nchg : P.ncl;
            for (int k = gwarp; k < ncl_it; k += gwarps) {
                const int32_t c = listed ? P.chg[(size_t)(par ^ 1) * HMK_P2_CHG + k] : k;
                const int32_t dpos = P.dirty[c];
                if (dpos == HMK_P2_CLEAN) continue;
                int32_t* ci = P.cinfo + c * HMK_CI;
                HmkDynEntry* out = P.dyn + ci[0] + ci[1];
                int lo = P.cstart[c], hi = P.cstart[c + 1];
                const int end = hi;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (P.cc_q[mid] < P.qa) lo = mid + 1; else hi = mid; }
                int n = 0;
                for (int i0 = lo; i0 < end; i0 += 32) {
                    const int i = i0 + lane;
                    const int32_t qi = i < end ? P.cc_q[i] : 0x7fffffff;
                    const bool inw = qi < P.qb;
                    const bool joins = inw && P.a[qi] == c;
                    const unsigned jm = __ballot_sync(FULL, joins);
                    if (joins) {
                        const int32_t id = P.singles[qi];
                        HmkDynEntry en;
                        en.w = P.packed ? P.packed[id] : 0ull; en.qi = qi; en.ab = P.S.ab[id];
                        HMK_CHECK(ci[1] + n + __popc(jm) <= P.cstart[c + 1] - P.cstart[c]);     // final + tentative <= candidates
                        out[n + __popc(jm & ((1u << lane) - 1u))] = en;
                    }
                    n += __popc(jm);
                    if (inw && qi > dpos && atomicMax(P.stamp + qi, gen) < gen) {
                        const int wpos = atomicAdd(P.ctl + par, 1);
                        HMK_CHECK(wpos >= 0 && wpos < P.wcap);
                        work[wpos] = qi;
                    }
                    if (!__all_sync(FULL, inw)) break;
                }
                __syncwarp();
                if (lane == 0) { ci[2] = n; P.dirty[c] = HMK_P2_CLEAN; }
            }
            if (gtid == 0) { P.ctl[4 + par] = 0; P.ctl[6 + par] = 0; P.ctl[2 + par] = 0; P.ctl[par ^ 1] = 0; }
            grid.sync();
            mark_time();
        }
        // ---- D
        {
            const int nwork = t == 0 ? P.qb - P.qa : P.ctl[par];
            const int32_t* work = P.work + (size_t)par * P.wcap;
            for (;;) {
                int wi = 0;
                if (lane == 0) wi = atomicAdd(P.ctl + 2 + par, 1);
                wi = __shfl_sync(FULL, wi, 0);
                if (wi >= nwork) break;
                const int qi = t == 0 ? P.qa + wi : work[wi];
                HMK_CHECK(qi >= P.qa && qi < P.qb && nwork <= P.wcap);
                if (t == 0 && P.qstart[qi] == P.qstart[qi + 1]) continue;       // no candidate: stays unassigned
                hmk_p2_decide_query<FAST>(P, sM, qi, par, npairs);
            }
        }
        grid.sync();
        mark_time();
        if (gtid == 0 && P.tim && tslot < 62) { P.tim[62] = (unsigned long long)(t == 0 ? P.qb - P.qa : P.ctl[par]); }
        if (!P.ctl[6 + par] || t + 1 >= P.max_iters) break;
    }
    // ---- commit: the tentative lists (rebuilt in R of the last iteration, unchanged since) are the final joiners
    for (int c = gtid; c < P.ncl; c += gthreads) {
        int32_t* ci = P.cinfo + c * HMK_CI;
        const int n = ci[2];
        if (n == 0) continue;
        const int32_t nd = ci[1];
        int32_t cnt = P.S.c_count[c], size = P.S.c_size[c];
        const HmkDynEntry* tl = P.dyn + ci[0] + nd;
        HMK_CHECK(nd + n <= P.cstart[c + 1] - P.cstart[c]);
        for (int i = 0; i < n; i++) {
            const int32_t q = P.singles[tl[i].qi];
            P.S.rank[q] = cnt++;
            size = hmk_wadd(size, tl[i].ab);
            P.S.slot[q] = c;
        }
        ci[1] = nd + n; P.S.c_count[c] = cnt; P.S.c_size[c] = size;
    }
    if (gtid == 0) P.ctl[8] = t + 1;
    for (int s = 16; s > 0; s >>= 1) npairs += __shfl_xor_sync(FULL, npairs, s);
    if (lane == 0) hmk_count_pairs(P.pair_parts, npairs);
}

// ---------------------------------------------------------------- small utilities
__global__ void hmk_fill_i32(int32_t* p, int32_t v, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

// 5 bits per residue, 12 residues per 64-bit word, `words` words per sequence (residue j lives in word
// j / 12 at bits [5 (j % 12), +5)); also validates the residue codes
__global__ void hmk_pack_sequences(int n, int words, const uint8_t* __restrict__ res, const int32_t* __restrict__ off,
                                   uint64_t* __restrict__ packed, int32_t* __restrict__ bad) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int len = off[i + 1] - off[i];
    uint64_t w[3] = {0, 0, 0};
    for (int j = 0; j < len; j++) {
        uint32_t r = res[off[i] + j];
        if (r >= HMK_NRES) { atomicExch(bad, 1); r = 0; }
        if (j < HMK_MAXL1 * words) w[j / HMK_MAXL1] |= (uint64_t)r << (5 * (j % HMK_MAXL1));
    }
    // one-word sequences (<= 12 residues use bits 0..59) carry their length in bits 60..63: the one-at-a-time scorer
    // then needs nothing but the two words (the bulk kernels only ever look at the residue fields)
    if (words == 1) w[0] |= (uint64_t)(len <= HMK_MAXL1 ? len : 0) << 60;
    for (int k = 0; k < words; k++) packed[(size_t)i * words + k] = w[k];
}

// flags -> exclusive positions, three-step scan (per-block counts, single-block scan, scatter)
__global__ void hmk_count_unassigned(const int32_t* __restrict__ slot, int n, int32_t* __restrict__ block_cnt) {
    __shared__ int wsum[32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool f = i < n && slot[i] < 0;
    const unsigned m = __ballot_sync(0xffffffffu, f);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = __popc(m);
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += wsum[w];
        block_cnt[blockIdx.x] = t;
    }
}
__global__ void hmk_scan_blocks(int32_t* block_cnt, int nblocks, int32_t* total) {
    // single thread block, sequential chunks (nblocks is n/1024: tiny)
    if (threadIdx.x == 0) {
        int run = 0;
        for (int b = 0; b < nblocks; b++) { int c = block_cnt[b]; block_cnt[b] = run; run += c; }
        *total = run;
    }
}
__global__ void hmk_scatter_unassigned(const int32_t* __restrict__ slot, int n, const int32_t* __restrict__ block_off,
                                       int32_t* __restrict__ out) {
    __shared__ int wsum[32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool f = i < n && slot[i] < 0;
    const unsigned m = __ballot_sync(0xffffffffu, f);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) wsum[wid] = __popc(m);
    __syncthreads();
    int pre = 0;
    for (int w = 0; w < wid; w++) pre += wsum[w];
    if (f) out[block_off[blockIdx.x] + pre + __popc(m & ((1u << lane) - 1u))] = i;
}

__global__ void hmk_index_of(const int32_t* __restrict__ list, int n, int32_t* __restrict__ index_of) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) index_of[list[i]] = i;
}

// split an id list by sequence length: out[len * stride + k], k < count[len] (order inside a bucket is arbitrary)
__global__ void hmk_bucket_by_length(const int32_t* __restrict__ ids, int n, const int32_t* __restrict__ off, int stride,
                                     int32_t* __restrict__ out, int32_t* __restrict__ count) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int32_t id = ids[i];
    const int len = off[id + 1] - off[id];
    if (len > HMK_MAXLEN) return;
    const int k = atomicAdd(count + len, 1);
    HMK_CHECK(len >= 0 && k >= 0 && k < stride);
    out[(size_t)len * stride + k] = id;
}

// first index whose key's high field (bits >= shift) is >= s, for s = 0..nseg (start[nseg] = n)
__global__ void hmk_segment_starts(const unsigned long long* __restrict__ keys, int n, int nseg, int shift, int32_t* __restrict__ start) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > nseg) return;
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if ((int64_t)(keys[mid] >> shift) < (int64_t)s) lo = mid + 1; else hi = mid;
    }
    start[s] = lo;
}
__global__ void hmk_segment_starts_i32(const int32_t* __restrict__ keys, int n, int nseg, int32_t* __restrict__ start) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s > nseg) return;
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (keys[mid] < s) lo = mid + 1; else hi = mid;
    }
    start[s] = lo;
}
__global__ void hmk_split_keys_lo(const unsigned long long* __restrict__ keys, int n, int shift, int32_t* __restrict__ lo,
                                  int32_t* __restrict__ hi) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    lo[i] = (int32_t)(uint32_t)(keys[i] & ((1ull << shift) - 1ull));
    if (hi) hi[i] = (int32_t)(uint32_t)(keys[i] >> shift);
}

__global__ void hmk_finalize(int n, const int32_t* __restrict__ slot, const int32_t* __restrict__ rank,
                             const int32_t* __restrict__ c_founder, int32_t* __restrict__ cluster_id,
                             int32_t* __restrict__ member_rank) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int s = slot[i];
    cluster_id[i] = s >= 0 ? c_founder[s] : i;
    member_rank[i] = s >= 0 ? rank[i] : 0;
}

// ---------------------------------------------------------------- roofline microbenchmarks
// Measured denominators for the roofline report (SURVEY.md 8d: "PEAK_INT32 must be measured on
// the box").  (a) dependent-free integer adds, 8 independent chains per thread -- ptxas fuses
// each pair of adds into one IADD3 (checked with cuobjdump), so instructions = adds / 2;
// (a') the same with every other chain on mad.lo (IMAD, the FMA pipe): the dual-pipe ceiling;
// (b) conflict-free 32-bit shared-memory loads (the pipe that actually bounds hmk_bulk_fast).
__global__ void __launch_bounds__(1024) hmk_peak_iadd(int iters, int32_t* out) {
    int32_t a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const int32_t b = blockIdx.x + 1;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a0) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a1) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a2) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a3) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a4) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a5) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a6) : "r"(b));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a7) : "r"(b));
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

// half of the chains as add (ALU pipe), half as mad.lo (FMA pipe): the dual-pipe integer ceiling
__global__ void __launch_bounds__(1024) hmk_peak_imix(int iters, int32_t one, int32_t* out) {
    int32_t a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const int32_t b = blockIdx.x + 1;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a0) : "r"(b));
            asm volatile("mad.lo.s32 %0, %1, %2, %0;" : "+r"(a1) : "r"(b), "r"(one));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a2) : "r"(b));
            asm volatile("mad.lo.s32 %0, %1, %2, %0;" : "+r"(a3) : "r"(b), "r"(one));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a4) : "r"(b));
            asm volatile("mad.lo.s32 %0, %1, %2, %0;" : "+r"(a5) : "r"(b), "r"(one));
            asm volatile("add.s32 %0, %0, %1;" : "+r"(a6) : "r"(b));
            asm volatile("mad.lo.s32 %0, %1, %2, %0;" : "+r"(a7) : "r"(b), "r"(one));
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}

__global__ void __launch_bounds__(1024) hmk_peak_lds(int iters, int32_t* out) {
    __shared__ uint32_t tab[4096];
    for (int i = threadIdx.x; i < 4096; i += blockDim.x) tab[i] = i * 2654435761u;
    __syncthreads();
    uint32_t acc0 = 0, acc1 = 0, acc2 = 0, acc3 = 0;
    uint32_t idx = threadIdx.x & 31;           // distinct banks inside a warp: conflict free
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            acc0 += tab[(idx + u * 128) & 4095];
            acc1 += tab[(idx + u * 128 + 32) & 4095];
            acc2 += tab[(idx + u * 128 + 64) & 4095];
            acc3 += tab[(idx + u * 128 + 96) & 4095];
        }
        idx = (idx + 1024) & 4095 & ~31u | (threadIdx.x & 31);
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = (int32_t)(acc0 ^ acc1 ^ acc2 ^ acc3);
}

// ---------------------------------------------------------------- exact complete-linkage clustering (NN chain)
// SURVEY.md 8(f) N1: ClinkageSequenceClusterer.cluster (reference ClinkageSequenceClusterer.java:43-124), Hammock's default
// initial stage for <= 10 000 unique sequences (Hammock.java:371-373), on the same pair scorer: the dense matrix of
// sequence-pair scores comes from the bulk kernel (MODE_DENSE), this kernel runs the nearest-neighbour chain on it.
//   D[a][b]   complete-linkage score of the clusters in slots a, b (ClinkageClusterScorer.java:30-49): min over the
//             member pairs, HMK_CL_BELOW as soon as one pair scores < T; merging two clusters takes the element-wise
//             minimum of their rows -- what CachedClusterScorer.join does (CachedClusterScorer.java:96-125)
//   nearest   arg-max over the other active clusters under NearestClusterRunner's order (score, Cluster.size(), smaller
//             id; ClinkageSequenceClusterer.java:258-293) -- a strict total order, so the scan order does not matter
//   HashSets  the chain restarts from activeClusters.iterator().next() (:70) and the result is new ArrayList(readyClusters)
//             (:119-123): both are java.util.HashSet<Cluster>, iterated in bucket order.  Emulated for OpenJDK 8+:
//             bucket = (h ^ h >>> 16) & (capacity - 1) with h = Cluster.hashCode() = 79 * 7 + id (Cluster.java:179-183),
//             chains in insertion order.  The table of activeClusters only grows while the n singletons are added, and a
//             resize keeps the relative order inside a bin, so inserting into the final table directly gives the same
//             chains; the same holds for readyClusters (insert only).  A bin that reaches 8 entries would be turned into
//             a tree by the JDK (different order): reported as unsupported -- it cannot happen with these consecutive
//             hash codes unless n is tiny.
// One CTA: a chain step is a row scan + a block reduction; steps are inherently sequential (about 3 n of them).
#define HMK_CL_BELOW (HMK_JMIN + 1)
#define HMK_CL_THREADS 1024

struct HmkClinkage {
    int32_t n, T;
    int32_t* D;            // dense path: [n][n]
    // sparse path (hmk_clinkage_chain_sparse): the entries with score >= T, both directions, each row sorted by slot.
    // Entry = (neighbour slot << 32) | (uint32) score; a killed entry has score HMK_JMIN.  twin[e] = position of the
    // mirror entry (in the row of e's neighbour, pointing back at e's row), relative to the start of that row.
    const int64_t* row_off;   // [n + 1]
    uint64_t* rows;
    const int32_t* twin;
    const int32_t* ab;
    int32_t acap;          // capacity of the activeClusters table
    int32_t* a_head;       // [acap] -1 = empty bin
    int32_t* a_tail;       // [acap]
    int32_t* a_next;       // [2n + 3] chain links by cluster id
    int32_t* a_prev;
    int32_t* slot_of;      // [2n + 3] cluster id -> slot
    int32_t* id_of;        // [n] slot -> cluster id, -1 = slot not active
    int32_t* size_of;      // [n] Cluster.size() (abundance weighted, Java int)
    int32_t* mhead;        // [n] member list of the slot's cluster
    int32_t* mtail;
    int32_t* mnext;
    int32_t* stack;        // [n + 1] cluster ids
    int32_t* ready;        // [n] ready clusters in insertion order
    int32_t* r_head;       // [4][rcap_max] scratch: two (head, tail) tables of the growing readyClusters set
    int32_t rcap_max;
    int32_t* r_next;       // [2n + 3]
    int32_t* cluster_id;   // outputs
    int32_t* member_rank;
    int32_t* result_order;
    int32_t* out_scalars;  // [0] n_result, [1] n_multi, [2] status (0 ok, 1 a bin reached the tree threshold), [3] nearest searches
};

__device__ __forceinline__ uint32_t hmk_cluster_hash(int32_t id) {
    const uint32_t h = (uint32_t)(79 * 7 + id);
    return h ^ (h >> 16);
}

__global__ void hmk_clinkage_threshold(int32_t* D, size_t total, int32_t T) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x)
        if (D[i] < T) D[i] = HMK_CL_BELOW;
}

// ---- helpers shared by the dense and the sparse chain kernel
// activeClusters.add(id): append at the tail of its bin; a bin that already holds 7 entries would become a tree in the
// JDK (different order) -> `treeified`.  One thread.  Returns the bin.
__device__ __forceinline__ int hmk_cl_set_add(const HmkClinkage& C, int32_t id, int32_t& treeified) {
    const int b = (int)(hmk_cluster_hash(id) & (uint32_t)(C.acap - 1));
    HMK_CHECK(id >= 1 && id < 2 * C.n + 3 && b >= 0 && b < C.acap);
    int len = 0;
    for (int k = C.a_head[b]; k >= 0; k = C.a_next[k]) len++;
    if (len >= 7) treeified = 1;
    C.a_next[id] = -1; C.a_prev[id] = C.a_tail[b];
    if (C.a_tail[b] >= 0) C.a_next[C.a_tail[b]] = id; else C.a_head[b] = id;
    C.a_tail[b] = id;
    return b;
}

// activeClusters.remove(id).  One thread.
__device__ __forceinline__ void hmk_cl_set_remove(const HmkClinkage& C, int32_t id) {
    const int b = (int)(hmk_cluster_hash(id) & (uint32_t)(C.acap - 1));
    HMK_CHECK(id >= 1 && id < 2 * C.n + 3 && b >= 0 && b < C.acap);
    const int32_t p = C.a_prev[id], nx = C.a_next[id];
    if (p >= 0) C.a_next[p] = nx; else C.a_head[b] = nx;
    if (nx >= 0) C.a_prev[nx] = p; else C.a_tail[b] = p;
}

// the n singleton clusters, ids 1..n (:48-54): slot tables by all threads, then the set in id order by thread 0.
// Returns (on thread 0) the lowest non-empty bin.  Ends with a barrier.
__device__ __forceinline__ int hmk_cl_init(const HmkClinkage& C, int32_t& treeified) {
    const int n = C.n;
    for (int b = threadIdx.x; b < C.acap; b += blockDim.x) { C.a_head[b] = -1; C.a_tail[b] = -1; }
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        C.id_of[i] = i + 1; C.slot_of[i + 1] = i; C.size_of[i] = C.ab[i];
        C.mhead[i] = i; C.mtail[i] = i; C.mnext[i] = -1;
    }
    __syncthreads();
    int lowest = C.acap;
    if (threadIdx.x == 0) {
        treeified = 0;
        for (int id = 1; id <= n; id++) lowest = min(lowest, hmk_cl_set_add(C, id, treeified));   // insertion order = id order
    }
    __syncthreads();
    return lowest;
}

// merge bookkeeping of thread 0 (:95-109): new Cluster(top.getSequences() ++ nearest.getSequences(), ++currentId) in slot
// ts, the nearest's slot bs dies.  Returns the bin of the new id.
__device__ __forceinline__ int hmk_cl_merge(const HmkClinkage& C, int32_t top, int32_t best, int ts, int bs, int32_t& cur_id,
                                            int32_t& treeified) {
    cur_id++;
    HMK_CHECK(cur_id < 2 * C.n + 3 && bs >= 0 && bs < C.n && ts >= 0 && ts < C.n && bs != ts);
    hmk_cl_set_remove(C, top);
    hmk_cl_set_remove(C, best);
    C.mnext[C.mtail[ts]] = C.mhead[bs];
    C.mtail[ts] = C.mtail[bs];
    C.size_of[ts] = hmk_wadd(C.size_of[ts], C.size_of[bs]);
    C.id_of[ts] = cur_id; C.id_of[bs] = -1;
    C.slot_of[cur_id] = ts;
    return hmk_cl_set_add(C, cur_id, treeified);
}

// the last cluster is ready too (:116); then new ArrayList(readyClusters): bucket order of a table that grew with the set
// (capacity 16, doubled whenever the size exceeded 0.75 x capacity).  Thread 0; `from_bin` <= the lowest non-empty bin;
// `nr` (ready clusters so far) counts the last one on return.
__device__ __forceinline__ void hmk_cl_finish(const HmkClinkage& C, int32_t& nr, int from_bin, int32_t treeified, int32_t searches) {
    for (int b = from_bin; b < C.acap; b++)
        if (C.a_head[b] >= 0) { C.ready[nr++] = C.a_head[b]; break; }
    HMK_CHECK(nr <= C.n);
    // the set as HashMap builds it: append at the bin's tail, double the table (bins split in order) whenever the size
    // exceeds 0.75 x capacity
    int rcap = 16, rsize = 0;
    int32_t* head = C.r_head;                     // two (head, tail) table pairs, used alternately across resizes
    int32_t* tail = C.r_head + C.rcap_max;
    int32_t* head2 = C.r_head + 2 * C.rcap_max;
    int32_t* tail2 = C.r_head + 3 * C.rcap_max;
    for (int b = 0; b < rcap; b++) { head[b] = -1; tail[b] = -1; }
    for (int i = 0; i < nr; i++) {
        const int32_t id = C.ready[i];
        const int b = (int)(hmk_cluster_hash(id) & (uint32_t)(rcap - 1));
        int len = 0;
        for (int32_t k = head[b]; k >= 0; k = C.r_next[k]) len++;
        if (len >= 7) treeified = 1;
        C.r_next[id] = -1;
        if (tail[b] >= 0) C.r_next[tail[b]] = id; else head[b] = id;
        tail[b] = id;
        if (++rsize > (int)(rcap * 0.75f)) {
            const int ncap = rcap * 2;
            HMK_CHECK(ncap <= C.rcap_max);
            for (int b2 = 0; b2 < ncap; b2++) { head2[b2] = -1; tail2[b2] = -1; }
            for (int b2 = 0; b2 < rcap; b2++)
                for (int32_t k = head[b2], nx; k >= 0; k = nx) {
                    nx = C.r_next[k];
                    const int nb = (int)(hmk_cluster_hash(k) & (uint32_t)(ncap - 1));
                    C.r_next[k] = -1;
                    if (tail2[nb] >= 0) C.r_next[tail2[nb]] = k; else head2[nb] = k;
                    tail2[nb] = k;
                }
            int32_t* t1 = head; head = head2; head2 = t1;
            t1 = tail; tail = tail2; tail2 = t1;
            rcap = ncap;
        }
    }
    int o = 0, multi = 0;
    for (int b = 0; b < rcap; b++)
        for (int32_t id = head[b]; id >= 0; id = C.r_next[id]) { HMK_CHECK(o < nr); C.result_order[o++] = id; }
    for (int i = 0; i < nr; i++) { const int s = C.slot_of[C.result_order[i]]; multi += C.mhead[s] != C.mtail[s]; }
    C.out_scalars[0] = nr; C.out_scalars[1] = multi; C.out_scalars[2] = treeified; C.out_scalars[3] = searches;
}

// cluster_id / member_rank of every member of the nr returned clusters.  All threads, after a barrier.
__device__ __forceinline__ void hmk_cl_members(const HmkClinkage& C, int nr) {
    for (int i = threadIdx.x; i < nr; i += blockDim.x) {
        const int32_t id = C.result_order[i];
        int32_t rank = 0;
        for (int32_t m = C.mhead[C.slot_of[id]]; m >= 0; m = C.mnext[m]) {
            HMK_CHECK(m >= 0 && m < C.n);
            C.cluster_id[m] = id; C.member_rank[m] = rank++;
        }
    }
}

// arg-max of the block's per-thread candidates under hmk_consider's order; the result is valid on thread 0 only.
// r_*: [32] shared scratch.  Ends without a barrier (the caller's next one separates the reuse of r_*).
__device__ __forceinline__ HmkBestCluster hmk_cl_block_best(HmkBestCluster bb, int32_t* r_score, int32_t* r_size, int32_t* r_id) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    hmk_best_reduce(bb);
    if (lane == 0) { r_score[wid] = bb.slot >= 0 ? bb.score : HMK_JMIN; r_size[wid] = bb.size; r_id[wid] = bb.slot >= 0 ? bb.fid : -1; }
    __syncthreads();
    HmkBestCluster g;
    g.score = HMK_JMIN; g.size = 0; g.fid = 0; g.slot = -1;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); w++)
            if (r_id[w] >= 0) hmk_consider(g, r_score[w], r_size[w], r_id[w], w);
    return g;
}

__global__ void __launch_bounds__(HMK_CL_THREADS, 1) hmk_clinkage_chain(const HmkClinkage C) {
    __shared__ int32_t r_score[32], r_size[32], r_id[32];
    __shared__ int32_t s_top, s_best, s_action, s_ts, s_bs;     // action: 0 ready, 1 merge, 2 push
    __shared__ int32_t s_first[32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = C.n;
    const unsigned FULL = 0xffffffffu;
    __shared__ int32_t sp, nr, nactive, cur_id, treeified, searches;
    hmk_cl_init(C, treeified);
    if (tid == 0) { sp = 0; nr = 0; nactive = n; cur_id = n + 1; searches = 0; }
    __syncthreads();
    for (;;) {
        // ---- empty stack: activeClusters.iterator().next() -- the head of the first non-empty bin (:62-70)
        if (sp == 0) {
            if (nactive <= 1) break;                  // (uniform: shared variables, read after a barrier)
            int first = 0x7fffffff;
            for (int b = tid; b < C.acap; b += blockDim.x)
                if (C.a_head[b] >= 0) { first = b; break; }
            first = __reduce_min_sync(FULL, first);
            if (lane == 0) s_first[wid] = first;
            __syncthreads();
            if (tid == 0) {
                int f = 0x7fffffff;
                for (int w = 0; w < (int)(blockDim.x >> 5); w++) f = min(f, s_first[w]);
                C.stack[0] = C.a_head[f];
                sp = 1;
            }
            __syncthreads();
        }
        if (tid == 0) { s_top = C.stack[sp - 1]; s_ts = C.slot_of[s_top]; searches++; }
        __syncthreads();
        const int32_t top = s_top, ts = s_ts;
        // ---- nearest neighbour of `top` (:75-82)
        HmkBestCluster bb;
        bb.score = HMK_JMIN; bb.size = 0; bb.fid = 0; bb.slot = -1;
        for (int k = tid; k < n; k += blockDim.x) {
            const int32_t id = C.id_of[k];
            if (id < 0 || k == ts) continue;
            hmk_consider(bb, C.D[(size_t)ts * n + k], C.size_of[k], id, k);
        }
        const HmkBestCluster g = hmk_cl_block_best(bb, r_score, r_size, r_id);
        if (tid == 0) {
            const int32_t best = g.slot >= 0 ? g.fid : -1, bscore = g.slot >= 0 ? g.score : HMK_JMIN;
            s_best = best;
            HMK_CHECK(sp >= 1 && sp <= n && nr < n && ts >= 0 && ts < n);
            if (bscore < C.T) {                                           // :85-91
                sp--;
                C.ready[nr++] = top;
                hmk_cl_set_remove(C, top);
                nactive--;
                C.id_of[ts] = -1;
                s_action = 0;
            } else if (sp > 1 && C.stack[sp - 2] == best) {               // :95-109
                s_bs = C.slot_of[best];
                s_action = 1;
            } else {
                C.stack[sp++] = best;                                     // :111
                s_action = 2;
            }
        }
        __syncthreads();
        if (s_action == 1) {
            const int32_t bs = s_bs;
            // CachedClusterScorer.join: the merged cluster's scores are the element-wise minimum of the two rows
            for (int k = tid; k < n; k += blockDim.x) {
                const int32_t a = C.D[(size_t)ts * n + k], b2 = C.D[(size_t)bs * n + k], m = a < b2 ? a : b2;
                C.D[(size_t)ts * n + k] = m;
                C.D[(size_t)k * n + ts] = m;
            }
            if (tid == 0) {
                sp -= 2;
                hmk_cl_merge(C, top, s_best, ts, bs, cur_id, treeified);
                nactive--;
            }
        }
        __syncthreads();
    }
    if (tid == 0) hmk_cl_finish(C, nr, 0, treeified, searches);
    __syncthreads();
    hmk_cl_members(C, nr);
}

// ---- sparse chain: the same state machine on rows of valid entries only (sizes beyond the dense n x n matrix).
// Exactness: a step either takes a neighbour scoring >= T or declares the top ready, so the arg-max over the valid entries
// of active clusters is the dense scan's choice whenever it is used.  join's element-wise minimum with
// min(x, BELOW) == BELOW makes the merged cluster's valid set the INTERSECTION of its parts' sets (scored by the minimum):
// rows only shrink.  Entries of inactive slots are skipped lazily (a slot never becomes active again); entries that leave
// an intersection are killed in place (score HMK_JMIN), so rows keep their layout and the twin positions stay valid.
// Restarts take the head of the lowest non-empty bin from a cursor instead of scanning the acap bins: an add into a lower
// bin moves it back, and it moves forward over emptied bins when a restart needs it.
// Block shape: a step costs a few dependent global loads per row pass plus the barriers, so the block is sized from the
// row lengths by the host (see Engine::clinkage).
__device__ __forceinline__ int32_t hmk_cl_entry_score(uint64_t v) { return (int32_t)(uint32_t)v; }
__device__ __forceinline__ int32_t hmk_cl_entry_slot(uint64_t v) { return (int32_t)(v >> 32); }

__global__ void __launch_bounds__(HMK_CL_THREADS, 1) hmk_clinkage_chain_sparse(const HmkClinkage C) {
    __shared__ int32_t r_score[32], r_size[32], r_id[32];
    __shared__ int32_t s_top, s_best, s_action, s_ts, s_bs;     // action: 0 ready, 1 merge, 2 push
    __shared__ int32_t sp, nr, nactive, cur_id, treeified, searches, cursor;
    const int tid = threadIdx.x;
    const int n = C.n;
    const int lowest = hmk_cl_init(C, treeified);
    if (tid == 0) { sp = 0; nr = 0; nactive = n; cur_id = n + 1; searches = 0; cursor = lowest; }
    __syncthreads();
    for (;;) {
        if (sp == 0 && nactive <= 1) break;           // (uniform: shared variables, read after a barrier)
        if (tid == 0) {
            if (sp == 0) {                            // activeClusters.iterator().next() (:62-70)
                while (C.a_head[cursor] < 0) { cursor++; HMK_CHECK(cursor < C.acap); }
                C.stack[0] = C.a_head[cursor];
                sp = 1;
            }
            s_top = C.stack[sp - 1]; s_ts = C.slot_of[s_top]; searches++;
        }
        __syncthreads();
        const int32_t top = s_top, ts = s_ts;
        HMK_CHECK(ts >= 0 && ts < n);
        const int64_t e0 = C.row_off[ts], e1 = C.row_off[ts + 1];
        // ---- nearest neighbour of `top` over its valid entries (:75-82)
        HmkBestCluster bb;
        bb.score = HMK_JMIN; bb.size = 0; bb.fid = 0; bb.slot = -1;
        for (int64_t e = e0 + tid; e < e1; e += blockDim.x) {
            const uint64_t v = C.rows[e];
            const int32_t sc = hmk_cl_entry_score(v), k = hmk_cl_entry_slot(v);
            if (sc < C.T) continue;
            HMK_CHECK(k >= 0 && k < n && k != ts);
            const int32_t id = C.id_of[k];
            if (id < 0) continue;
            hmk_consider(bb, sc, C.size_of[k], id, k);
        }
        const HmkBestCluster g = hmk_cl_block_best(bb, r_score, r_size, r_id);
        if (tid == 0) {
            const int32_t best = g.slot >= 0 ? g.fid : -1, bscore = g.slot >= 0 ? g.score : HMK_JMIN;
            s_best = best;
            HMK_CHECK(sp >= 1 && sp <= n && nr < n);
            if (bscore < C.T) {                                           // :85-91
                sp--;
                C.ready[nr++] = top;
                hmk_cl_set_remove(C, top);
                nactive--;
                C.id_of[ts] = -1;
                s_action = 0;
            } else if (sp > 1 && C.stack[sp - 2] == best) {               // :95-109
                s_bs = C.slot_of[best];
                s_action = 1;
            } else {
                C.stack[sp++] = best;                                     // :111
                s_action = 2;
            }
        }
        __syncthreads();
        if (s_action == 1) {
            const int32_t bs = s_bs;
            HMK_CHECK(bs >= 0 && bs < n && bs != ts);
            const int64_t b0 = C.row_off[bs], b1 = C.row_off[bs + 1];
            // row(ts) := row(ts) & row(bs), minimum score; the mirror entry in the neighbour's row follows.  Only row(bs)
            // is searched, and no thread writes it (its entry for ts is not in row(ts) -- no self entries)
            for (int64_t e = e0 + tid; e < e1; e += blockDim.x) {
                const uint64_t v = C.rows[e];
                const int32_t sc = hmk_cl_entry_score(v), k = hmk_cl_entry_slot(v);
                if (sc < C.T) continue;
                int32_t m = HMK_JMIN;
                const bool live = k != bs && C.id_of[k] >= 0;
                if (live) {
                    int64_t lo = b0, hi = b1;                             // first entry of row(bs) with slot >= k
                    while (lo < hi) {
                        const int64_t mid = (lo + hi) >> 1;
                        if (hmk_cl_entry_slot(C.rows[mid]) < k) lo = mid + 1; else hi = mid;
                    }
                    if (lo < b1) {
                        const uint64_t w = C.rows[lo];
                        const int32_t sb = hmk_cl_entry_score(w);
                        if (hmk_cl_entry_slot(w) == k && sb >= C.T) m = sc < sb ? sc : sb;
                    }
                }
                C.rows[e] = (v & 0xffffffff00000000ull) | (uint32_t)m;
                if (live) {
                    const int64_t t = C.row_off[k] + C.twin[e];
                    HMK_CHECK(t >= C.row_off[k] && t < C.row_off[k + 1] && hmk_cl_entry_slot(C.rows[t]) == ts);
                    C.rows[t] = ((uint64_t)(uint32_t)ts << 32) | (uint32_t)m;
                }
            }
            if (tid == 0) {
                sp -= 2;
                const int b = hmk_cl_merge(C, top, s_best, ts, bs, cur_id, treeified);
                nactive--;
                if (b < cursor) cursor = b;
            }
        }
        __syncthreads();
    }
    if (tid == 0) hmk_cl_finish(C, nr, cursor, treeified, searches);
    __syncthreads();
    hmk_cl_members(C, nr);
}

// ---- sparse row build (Engine::clinkage): the bulk kernel's EMIT hits of one query batch, upper triangle only
// (profile index p = query q0 + p, thread-side id > query).  Pass 1 counts the entries per row, pass 2 scatters both
// directions behind per-row cursors (row order is fixed afterwards by a segmented sort).
__global__ void hmk_cl_count_hits(const int4* __restrict__ hits, const unsigned int* __restrict__ count, unsigned int cap,
                                  int32_t q0, int32_t n, unsigned long long* deg) {
    const unsigned int m = min(*count, cap);
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        const int4 h = hits[i];
        const int32_t q = q0 + h.x;
        HMK_CHECK(q >= 0 && q < n && h.y >= 0 && h.y < n);
        if (h.y <= q) continue;
        atomicAdd(deg + q, 1ull);
        atomicAdd(deg + h.y, 1ull);
    }
}

__global__ void hmk_cl_scatter_hits(const int4* __restrict__ hits, const unsigned int* __restrict__ count, unsigned int cap,
                                    int32_t q0, int32_t n, const int64_t* __restrict__ row_off, unsigned long long* cur,
                                    uint64_t* rows) {
    const unsigned int m = min(*count, cap);
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        const int4 h = hits[i];
        const int32_t q = q0 + h.x;
        if (h.y <= q) continue;
        const int64_t pa = row_off[q] + (int64_t)atomicAdd(cur + q, 1ull);
        const int64_t pb = row_off[h.y] + (int64_t)atomicAdd(cur + h.y, 1ull);
        HMK_CHECK(pa < row_off[q + 1] && pb < row_off[h.y + 1]);
        rows[pa] = ((uint64_t)(uint32_t)h.y << 32) | (uint32_t)h.z;
        rows[pb] = ((uint64_t)(uint32_t)q << 32) | (uint32_t)h.z;
    }
}

// rel[i] = row_off[r0 + i] - row_off[r0], i = 0..nr: int32 segment offsets of one sort group
__global__ void hmk_cl_rel_offsets(const int64_t* __restrict__ row_off, int32_t r0, int32_t nr, int32_t* rel) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i <= nr; i += gridDim.x * blockDim.x)
        rel[i] = (int32_t)(row_off[r0 + i] - row_off[r0]);
}

// twin[e] = position of e's mirror entry in the neighbour's row (relative to its start): binary search for the row's slot
// in the neighbour's sorted row.  One warp per row.
__global__ void hmk_cl_twins(const int64_t* __restrict__ row_off, const uint64_t* __restrict__ rows, int32_t n, int32_t* twin) {
    const int lane = threadIdx.x & 31;
    for (int64_t a = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; a < n; a += ((int64_t)gridDim.x * blockDim.x) >> 5) {
        for (int64_t e = row_off[a] + lane; e < row_off[a + 1]; e += 32) {
            const int32_t b = (int32_t)(rows[e] >> 32);
            HMK_CHECK(b >= 0 && b < n && b != a);
            int64_t lo = row_off[b], hi = row_off[b + 1];
            while (lo < hi) {
                const int64_t mid = (lo + hi) >> 1;
                if ((int32_t)(rows[mid] >> 32) < (int32_t)a) lo = mid + 1; else hi = mid;
            }
            HMK_CHECK(lo < row_off[b + 1] && (int32_t)(rows[lo] >> 32) == (int32_t)a);
            twin[e] = (int32_t)(lo - row_off[b]);
        }
    }
}

// ---- score graph (Engine::graph_batch) and hmk_score_pairs: ShiftedScorer.scoreWithShift, one thread per pair, with the
// one-at-a-time scorer of the generic kernel.  pairs[i] = (seq2 = q0 + x, seq1 = y, score z).
//   graph (keys != NULL): the EMIT hits of one query batch (count = the kernel's hit counter, at most cap stored).  A
//     pair with seq1 <= seq2 is dropped; a kept one gets the sort key (x << jbits) | y, the value (score, shift) and a
//     count in its query's row.  The recomputed score equals the emitted one.
//   pairs (keys == NULL): the first cap pairs, none dropped; score[i] / shift[i] in input order.
struct HmkShiftArgs {
    const int4* pairs;
    const unsigned int* count;
    unsigned int cap;
    int32_t q0, jbits;
    const uint8_t* res;
    const int32_t* off;
    const int32_t* M;
    int32_t X, P, n;
    unsigned long long* keys;
    unsigned long long* vals;
    unsigned int* kept;     // [0] kept pairs, [1 + x] pairs kept in query row x
    int32_t* score;
    int32_t* shift;
};

__global__ void hmk_score_shift(HmkShiftArgs a) {
    const unsigned int m = a.count ? min(*a.count, a.cap) : a.cap;
    const int lane = threadIdx.x & 31;
    const unsigned int stride = gridDim.x * blockDim.x;
    // every lane of a warp takes the same number of turns: the kept pairs are counted with one atomic per warp
    for (unsigned int base = blockIdx.x * blockDim.x + (threadIdx.x & ~31u); base < m; base += stride) {
        const unsigned int i = base + lane;
        bool keep = false;
        int4 h = make_int4(0, 0, 0, 0);
        int32_t s = 0;
        int k = 0;
        if (i < m) {
            h = a.pairs[i];
            const int32_t q = a.q0 + h.x;
            HMK_CHECK(q >= 0 && q < a.n && h.y >= 0 && h.y < a.n);
            if (!a.keys || h.y > q) {
                s = hmk_score_with_shift(a.res + a.off[h.y], a.off[h.y + 1] - a.off[h.y], a.res + a.off[q], a.off[q + 1] - a.off[q],
                                         a.M, a.X, a.P, &k);
                if (!a.keys) { a.score[i] = s; a.shift[i] = k; }
                else { HMK_CHECK(s == h.z); keep = true; }
            }
        }
        if (!a.keys) continue;
        const unsigned int km = __ballot_sync(0xffffffffu, keep);
        if (!km) continue;
        unsigned int pos = 0;
        const int leader = __ffs(km) - 1;
        if (lane == leader) pos = atomicAdd(a.kept, (unsigned int)__popc(km));
        pos = __shfl_sync(0xffffffffu, pos, leader) + __popc(km & ((1u << lane) - 1u));
        if (keep) {
            HMK_CHECK(pos < a.cap);
            a.keys[pos] = ((unsigned long long)(uint32_t)h.x << a.jbits) | (uint32_t)h.y;
            a.vals[pos] = ((unsigned long long)(uint32_t)s << 32) | (uint32_t)k;
            atomicAdd(a.kept + 1 + h.x, 1u);
        }
    }
}

// the sorted (key, value) pairs of a graph batch as edges (seq, partner, score, shift) == hmk_graph_edge
__global__ void hmk_graph_edges(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ vals,
                                unsigned int m, int32_t q0, int32_t jbits, int4* __restrict__ edges) {
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        const unsigned long long k = keys[i], v = vals[i];
        edges[i] = make_int4(q0 + (int32_t)(k >> jbits), (int32_t)(k & ((1ull << jbits) - 1)), (int32_t)(v >> 32), (int32_t)(uint32_t)v);
    }
}

// ---- nearest partners (Engine::nearest): one warp per row t of a query batch (row id r0 + t) over its merged list of
// the k + 1 best keys among the thread-side ids [0, n).  The row's own id is dropped and the list cut to k: lane o fills
// output slot o with the partner id, scoreWithShift(seq1 = partner, seq2 = row) and its shift, or partner -1, score 0,
// shift 0 past the row's count.  The recomputed score equals the key's.  more[t] = 1 when more than k other ids qualify:
// with the row's own id in the list that is the merged overflow flag (more than k + 1 keys), without it a full list of
// k + 1 keys (the row's own key, if it qualifies, ranks behind all of them).
struct HmkNearestArgs {
    int32_t nq, k, r0, n;
    const uint64_t* key;        // [nq][k + 1] merged lists (hmk_topk_merge)
    const int32_t* cnt;
    const int32_t* ovf;
    const int32_t* id_of_rank;  // NULL: rank == id
    const uint8_t* res;
    const int32_t* off;
    const int32_t* M;
    int32_t X, P;
    int32_t* partner;           // [nq][k]
    int32_t* score;
    int32_t* shift;
    int32_t* count;             // [nq]
    int32_t* more;
};

__global__ void hmk_nearest_rows(HmkNearestArgs a) {
    const int t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (t >= a.nq) return;      // warp-uniform
    const int kb = a.k + 1, row = a.r0 + t;
    const int c = a.cnt[t];
    HMK_CHECK(kb <= 32 && c >= 0 && c <= kb && row < a.n);
    const uint64_t* key = a.key + (size_t)t * kb;
    int32_t id = -1;
    if (lane < c) {
        const uint32_t r = hmk_key_rank(key[lane]);
        id = a.id_of_rank ? a.id_of_rank[r] : (int32_t)r;
    }
    const unsigned self = __ballot_sync(0xffffffffu, lane < c && id == row);
    const int s = self ? __ffs(self) - 1 : kb;                  // list position of the row's own id
    const int src = lane < s ? lane : lane + 1;                 // the list entry output slot `lane` takes
    const int m = min(c - (self ? 1 : 0), a.k);
    const int32_t p = __shfl_sync(0xffffffffu, id, src & 31);
    if (lane < a.k) {
        int32_t sc = 0, sh = 0;
        if (lane < m) {
            HMK_CHECK(p >= 0 && p < a.n && p != row);
            sc = hmk_score_with_shift(a.res + a.off[p], a.off[p + 1] - a.off[p], a.res + a.off[row], a.off[row + 1] - a.off[row],
                                      a.M, a.X, a.P, &sh);
            HMK_CHECK(sc == hmk_key_score(key[src]));
        }
        const size_t o = (size_t)t * a.k + lane;
        a.partner[o] = lane < m ? p : -1;
        a.score[o] = sc;
        a.shift[o] = sh;
    }
    if (lane == 0) {
        a.count[t] = m;
        a.more[t] = self ? (a.ovf[t] ? 1 : 0) : (c == kb ? 1 : 0);
    }
}
