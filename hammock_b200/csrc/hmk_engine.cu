// hmk_engine.cu -- host driver of the B200 greedy-clustering engine + the C ABI
// (include/hammock_b200.h).  Replaces LimitedGreedySequenceClusterer.cluster()
// (reference LimitedGreedySequenceClusterer.java:39-69) and everything below it.
//
// Structure of one run (all state device-resident, one CUDA stream):
//   phase 1  batches of B abundance-ordered queries:
//              select -> profiles -> bulk partner search (top-k per query over all later
//              singletons) -> founder filter + member check (cluster search) -> intra-batch
//              scores -> in-order resolver (one warp, reference order)
//   phase 2  founder profiles -> bulk founder filter over all remaining singletons ->
//              member check -> candidate lists sorted by query and by cluster ->
//              wavefront rounds that resolve queries in reference order
// There is no CPU fallback: every scoring and every decision happens in CUDA kernels.
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <cub/cub.cuh>
#include <numeric>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include <dlfcn.h>
#include <unistd.h>

#include "../../include/hammock_b200.h"
#include "hmk_kernels.cuh"

namespace {

// ---------------------------------------------------------------- NCCL, loaded on demand
// The single-GPU path has no NCCL dependency; hmk_init_distributed dlopen()s libnccl.so.2 (the
// copy the host process already loaded, e.g. torch's, or the system one).
struct NcclApi {
    typedef struct { char internal[128]; } UniqueId;
    typedef void* Comm;
    int (*GetUniqueId)(UniqueId*) = nullptr;
    int (*CommInitRank)(Comm*, int, UniqueId, int) = nullptr;
    int (*CommDestroy)(Comm) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, Comm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
    bool ok = false;
    std::string error;
    static NcclApi& get() {
        static NcclApi api;
        static bool tried = false;
        if (!tried) {
            tried = true;
            void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
            if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
            if (!h) { api.error = std::string("cannot load libnccl: ") + dlerror(); return api; }
            auto sym = [&](const char* n) { void* p = dlsym(h, n); if (!p) api.error = std::string("libnccl lacks ") + n; return p; };
            api.GetUniqueId = (int (*)(UniqueId*))sym("ncclGetUniqueId");
            api.CommInitRank = (int (*)(Comm*, int, UniqueId, int))sym("ncclCommInitRank");
            api.CommDestroy = (int (*)(Comm))sym("ncclCommDestroy");
            api.AllGather = (int (*)(const void*, void*, size_t, int, Comm, cudaStream_t))sym("ncclAllGather");
            api.GroupStart = (int (*)())sym("ncclGroupStart");
            api.GroupEnd = (int (*)())sym("ncclGroupEnd");
            api.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
            api.ok = api.error.empty();
        }
        return api;
    }
};
enum { HMK_NCCL_CHAR = 0 };   // ncclInt8 / ncclChar

struct CudaError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

#define NK(call)                                                                                   \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0)                                                                               \
            throw CudaError(std::string(#call) + " failed: " + NcclApi::get().GetErrorString(r_)); \
    } while (0)

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            throw CudaError(std::string(#call) + " failed: " + cudaGetErrorString(e_) + " (" + __FILE__ + \
                            ":" + std::to_string(__LINE__) + ")");                                \
    } while (0)

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    void reserve(size_t n) {   // contents are NOT preserved
        if (n <= cap) return;
        if (p) CK(cudaFree(p));
        p = nullptr;
        CK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
        cap = n;
    }
    void release() {
        if (p) CK(cudaFree(p));
        p = nullptr;
        cap = 0;
    }
    void grow_keep(size_t n, size_t used, cudaStream_t st) {
        if (n <= cap) return;
        T* q = nullptr;
        CK(cudaMalloc(&q, n * sizeof(T)));
        if (p && used) CK(cudaMemcpyAsync(q, p, used * sizeof(T), cudaMemcpyDeviceToDevice, st));
        CK(cudaStreamSynchronize(st));
        if (p) CK(cudaFree(p));
        p = q;
        cap = n;
    }
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-DEVICE attribute of a kernel, and setting it REPLACES the value:
// the largest size configured so far is tracked per (device, kernel) for the whole process, under a mutex -- not in
// per-kernel statics (a second device would never be configured) and not per context (a context that needs less would
// lower the limit under another context of the same device).
struct SmemConfig {
    int device = 0;
    template <class K>
    void ensure(K kernel, size_t smem) {
        static std::mutex mu;
        static std::map<std::pair<int, const void*>, size_t> done;
        const void* f = reinterpret_cast<const void*>(kernel);
        std::lock_guard<std::mutex> lock(mu);
        size_t& have = done[{device, f}];
        if (smem > have) {
            CK(cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            have = smem;
        }
    }
};

// the bulk kernel a launch runs (Engine::launch_planned); `kind` numbers as in hmk_bulk_probe's kernel array
struct BulkKernel {
    enum Kind { GENERIC = 0, FAST = 1, FILTER = 2, LONG = 3 };
    int kind;
    int lt;            // hmk_bulk_filter's compile-time length (12 or 0); -1 for the other kernels
    int threads;
    const void* fn;    // takes HmkGenericArgs (GENERIC) or HmkBulkArgs
};

enum { HMK_MAXTILES_PERSISTENT = 1024 };   // profile tiles a persistent bulk launch schedules (more: static grid)
enum { HMK_FB_STRIDE = 1 << 16 };   // founders per slice of the per-length split of the cluster search
enum { HMK_NAUX = 6 };         // auxiliary streams for launches that are independent of each other (length buckets)
enum { HMK_NBATCHBUF = 3 };   // the batch being resolved + up to two prepared ahead
enum { SEC_P1_SELECT = 0, SEC_P1_PARTNER, SEC_P1_CLUSTER, SEC_P1_INTRA, SEC_P1_RESOLVE, SEC_P2_SETUP, SEC_P2_FILTER,
       SEC_P2_CHECK, SEC_P2_SORT, SEC_P2_BASE, SEC_P2_ITERATE, SEC_P2_COMMIT, SEC_FINAL };

struct Options {
    int64_t batch = 0;          // phase-1 queries per batch (0 = three profile tiles)
    int64_t capq = 256;         // initial per-query capacity of the cluster-candidate arrays
    int64_t reuse = 1;          // 1: phase 2 takes its founder hits from the phase-1 partner searches (symmetric matrices)
    int64_t filter = 1;         // 1: filter + verify kernel where it applies (u8 lanes, two words, one length <= 12)
    int64_t lookahead = 2;      // batches whose partner search is prepared on the side stream while the current batch resolves (0..2)
    int64_t qt = 0;             // profiles per CTA tile (0 = as many as shared memory holds)
    int64_t kb = 8;             // partner candidates kept per query
    int64_t waves = 2;          // CTAs per SM targeted by the stripe split
    int64_t p2_chunk = 1 << 18; // phase-2 queries per founder-filter launch
    int64_t hit_cap = 1 << 22;  // initial founder-hit capacity
    int64_t force_generic = 0;  // 1: never use the packed SWAR kernel
    int64_t profile = 0;        // 1: time every bulk launch with CUDA events
    int64_t p2_window = 1 << 16;  // phase-2 queries resolved per window
    int64_t min_iters = 1;        // static grids: block iterations a stripe must at least have
    int64_t bucket_aux = 1;       // mixed lengths: run the per-length launches of a batch on separate streams
    int64_t reserve = 4;          // SMs the look-ahead bulk launches leave to the main stream (resolver + small kernels)
    int64_t persistent = 1;       // 1: filter kernel as one CTA per SM taking database chunks dynamically; 0: static grid
    int64_t p2_first = 0;         // queries in the first phase-2 window (0 = automatic)
    int64_t xhit_cap = 0;         // capacity of the kept-hit buffer (0 = automatic: the last run's need, else 96 per sequence)
    int64_t clinkage_dense_max = 32768;   // exact complete linkage: largest n that takes the dense n x n path
    int64_t clinkage_threads = 0;         // threads of the sparse chain kernel (0 = automatic, from the row lengths)
    int64_t graph_cap = 0;                // score graph: hits one query batch may hold (0 = automatic, 1 << 22; at least n)
};

class Engine {
public:
    explicit Engine(int device) : device_(device) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count <= 0)
            throw CudaError(std::string("no CUDA device available (") + cudaGetErrorString(e) +
                            "); libhammock_b200 has no CPU fallback");
        if (device < 0 || device >= count) throw CudaError("invalid CUDA device index");
        CK(cudaSetDevice(device_));
        smem_cfg_.device = device_;
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device_));
        sm_count_ = prop.multiProcessorCount;
        smem_optin_ = prop.sharedMemPerBlockOptin;
        int prio_lo = 0, prio_hi = 0;
        CK(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
        CK(cudaStreamCreateWithPriority(&st_, cudaStreamNonBlocking, prio_hi));    // resolvers, small kernels
        CK(cudaStreamCreateWithPriority(&st2_, cudaStreamNonBlocking, prio_lo));   // look-ahead partner search
        CK(cudaStreamCreateWithPriority(&st3_, cudaStreamNonBlocking, prio_hi));   // look-ahead tails (small kernels)
        for (auto& b : bb_) CK(cudaEventCreateWithFlags(&b.ready, cudaEventDisableTiming));
        for (auto& b : bb_) CK(cudaEventCreateWithFlags(&b.searched, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&part1_ev_, cudaEventDisableTiming));
        for (auto& a : aux_) CK(cudaStreamCreateWithPriority(&a, cudaStreamNonBlocking, prio_lo));
        CK(cudaEventCreateWithFlags(&fork_ev_, cudaEventDisableTiming));
        for (auto& e : join_ev_) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaMallocHost(&h_ctl_, sizeof(HmkCtl)));
        CK(cudaMallocHost(&h_scalars_, 16 * sizeof(int32_t)));
        CK(cudaMallocHost(&h_p2flags_, HMK_P2_CTL * sizeof(int32_t)));
        CK(cudaEventCreate(&ev_a_));
        CK(cudaEventCreate(&ev_b_));
        CK(cudaEventCreate(&ev_c_));
        CK(cudaEventCreate(&ev_t0_));
        CK(cudaEventCreate(&ev_t1_));
    }
    ~Engine() {
        cudaSetDevice(device_);
        for (auto& e : ev_pool_) cudaEventDestroy(e);
        if (ev_a_) cudaEventDestroy(ev_a_);
        if (ev_b_) cudaEventDestroy(ev_b_);
        if (ev_c_) cudaEventDestroy(ev_c_);
        if (ev_t0_) cudaEventDestroy(ev_t0_);
        if (ev_t1_) cudaEventDestroy(ev_t1_);
        if (h_ctl_) cudaFreeHost(h_ctl_);
        if (h_scalars_) cudaFreeHost(h_scalars_);
        if (h_p2flags_) cudaFreeHost(h_p2flags_);
        if (comm_) NcclApi::get().CommDestroy(comm_);
        for (auto& b : bb_) if (b.ready) cudaEventDestroy(b.ready);
        for (auto& b : bb_) if (b.searched) cudaEventDestroy(b.searched);
        if (part1_ev_) cudaEventDestroy(part1_ev_);
        for (auto& e : join_ev_) if (e) cudaEventDestroy(e);
        if (fork_ev_) cudaEventDestroy(fork_ev_);
        for (auto& a : aux_) if (a) cudaStreamDestroy(a);
        if (st3_) cudaStreamDestroy(st3_);
        if (st2_) cudaStreamDestroy(st2_);
        if (st_) cudaStreamDestroy(st_);
    }

    Options opt;

    void upload(const hmk_greedy_in* in);
    int run();
    void download(hmk_greedy_out* out);
    void score_block(const int32_t* first, int32_t nf, const int32_t* second, int32_t ns, int32_t* scores);
    void bulk_probe(int mode, const int32_t* qids, int32_t nq, const int32_t* db_ids, int32_t db_begin, int32_t ndb,
                    const uint8_t* clustered, uint64_t* keys, int32_t* cnt, int32_t* ovf, int32_t* hits, int64_t hit_cap,
                    int64_t* hit_count, int32_t* kernel);
    void batch_probe(const int32_t* member_off, const int32_t* members, int32_t ncl, int32_t cur, int32_t nq, int32_t capq,
                     int32_t tail_stream, hmk_batch_probe_out* out);
    int clinkage(const hmk_greedy_in* in, hmk_greedy_out* out);
    int score_graph(int64_t* cursor, hmk_graph_edge* out, int64_t cap, int64_t* n_out);
    int score_pairs(const int32_t* seq1, const int32_t* seq2, int32_t np, int32_t* scores, int32_t* shifts);
    int nearest(int32_t k, int32_t row_begin, int32_t n_rows, int32_t* partner, int32_t* score, int32_t* shift,
                int32_t* count, int32_t* more);
    std::string status_msg;      // details of the last non-zero status, when there are any
    hmk_stats stats{};
    int error_step = -1;
    void timer_begin() { CK(cudaSetDevice(device_)); CK(cudaEventRecord(ev_t0_, st_)); }
    double timer_end() {
        CK(cudaSetDevice(device_));
        CK(cudaEventRecord(ev_t1_, st_));
        CK(cudaEventSynchronize(ev_t1_));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ev_t0_, ev_t1_));
        return ms;
    }
    void measure_peaks(double* out);
    void init_distributed(int rank, int world, const void* id128);
    void release_comm() {
        if (comm_) { cudaSetDevice(device_); NcclApi::get().CommDestroy(comm_); comm_ = nullptr; }
        rank_ = 0; world_ = 1;
    }

private:
    // ---- problem
    int device_;
    int rank_ = 0, world_ = 1;
    NcclApi::Comm comm_ = nullptr;
    DevBuf<int32_t> d_gcount_, d_gs_;
    DevBuf<unsigned long long> d_gq_;
    void allgather(const void* send, void* recv, size_t bytes, cudaStream_t s) {
        NK(NcclApi::get().AllGather(send, recv, bytes, HMK_NCCL_CHAR, comm_, s));
    }
    int sm_count_ = 148;
    size_t smem_optin_ = 0;
    SmemConfig smem_cfg_;
    cudaStream_t st_ = nullptr;
    int32_t n_ = 0, T_ = 0, X_ = 0, P_ = 0, K_ = 0;
    int32_t min_len_ = 0, max_len_ = 0;
    bool uploaded_ = false, ran_ = false, bad_residue_ = false;
    bool fast_ = false;
    bool mixed_ = false;         // lengths differ but every (m, n) pair fits the packed lanes
    int words_ = 1;              // 64-bit words per packed sequence
    int nw_len_[HMK_MAXLEN + 1] = {0};
    std::vector<int32_t> h_bucket_[HMK_MAXLEN + 1];   // ids per length, ascending
    DevBuf<int32_t> d_bucket_[HMK_MAXLEN + 1];
    DevBuf<int32_t> d_sidx_, d_sb_ids_, d_sb_cnt_;
    DevBuf<int32_t> d_ids_;      // 0 .. n - 1: the profile ids of the whole-input calls (identity_ids)
    bool ids_filled_ = false;
    DevBuf<uint32_t> d_pcells_, d_pops_;
    bool fast_scalar_ = false;   // every length <= 12: the one-at-a-time scorer works on the packed words (which carry the lengths)
    HmkScheme sc_{};
    std::vector<int32_t> h_off_;
    DevBuf<uint8_t> d_res_;
    DevBuf<int32_t> d_off_, d_ab_, d_M_, d_tierank_, d_id_of_rank_;
    DevBuf<uint64_t> d_packed_;
    bool identity_rank_ = true;
    // ---- clustering state
    DevBuf<int32_t> d_slot_, d_rank_, d_next_, d_cf_, d_cs_, d_cc_, d_ct_;
    DevBuf<HmkCtl> d_ctl_;
    HmkCtl* h_ctl_ = nullptr;
    int32_t* h_scalars_ = nullptr;
    int32_t* h_p2flags_ = nullptr;
    // ---- phase-1 per-batch buffers, a ring: while batch i is resolved on the main stream the partner searches of
    // batches i+1 and i+2 already run on the side stream, and their tails (merge, dense tables, masks) on the tail stream
    struct BatchBuf {
        DevBuf<int32_t> qid, gqid, nq_dev, tk_cnt, tk_ovf, bk_cnt, bk_ovf, gk_cnt, gk_ovf;
        DevBuf<uint64_t> tk_key, bk_key, gk_key;
        DevBuf<unsigned long long> gmin;   // per query: published lower bound of the kb-th best key (prunes top-k insertions)
        DevBuf<uint32_t> prof;
        int prof_len_batch[HMK_MAXLEN + 1] = {0};   // batch for which prof_len[L] was built
        DevBuf<int32_t> fb_ids, fb_cnt;             // founders of the cluster search split by length (mixed lengths)
        DevBuf<int32_t> sched, sched2;   // chunk / slot counters of the persistent partner-search / cluster-search launches
        // cluster search, part 1: founder hits of the clusters that existed when the batch was prepared
        DevBuf<int4> hits;
        DevBuf<unsigned int> hcount;     // [0] founder hits (may exceed hit_cap: the resolver then asks for a bigger buffer)
        size_t hit_cap = 0;
        int ncl_ahead = 0;               // clusters [0, ncl_ahead) are covered by part 1
        DevBuf<uint32_t> prof_len[HMK_MAXLEN + 1], pcells[HMK_MAXLEN + 1], pops[HMK_MAXLEN + 1];   // mixed lengths: per thread-side length
        // state-independent inputs of the resolver: intra-batch scores (+ bit mask), partner candidate ids and
        // their scores against every batch query
        DevBuf<int32_t> ib, pcand, pd;
        DevBuf<uint32_t> ibm, ibm2;
        cudaEvent_t ready = nullptr;     // everything above is complete
        cudaEvent_t searched = nullptr;  // the partner search is issued (qid final; the tail starts behind it)
        bool valid = false;      // partner search for the batch starting behind `after` has been issued
        int nq = 0;
        int batch_id = 0;
    };
    BatchBuf bb_[HMK_NBATCHBUF];
    cudaStream_t st2_ = nullptr, st3_ = nullptr;
    cudaEvent_t part1_ev_ = nullptr;
    cudaStream_t aux_[HMK_NAUX] = {nullptr};
    cudaEvent_t fork_ev_ = nullptr, join_ev_[HMK_NAUX] = {nullptr};
    void stage_partner_search(BatchBuf& bb, int nq, int db_from, const int32_t* start_after, int ncl_known, cudaStream_t s,
                              cudaStream_t t);
    void drain_lookahead() {
        CK(cudaStreamSynchronize(st2_));
        CK(cudaStreamSynchronize(st3_));
        for (auto& b : bb_) b.valid = false;
    }
    void founder_hits(BatchBuf& bb, int from, int to, cudaStream_t s, DevBuf<int32_t>& sched);
    void check_members(const BatchBuf& cb, int ncl, int capq);
    // bulk launches per mode (HMK_MODE_*) while a batch probe runs: the last kernel launched and how many launches
    struct LaunchLog {
        BulkKernel last[3] = {{-1, -1, 0, nullptr}, {-1, -1, 0, nullptr}, {-1, -1, 0, nullptr}};
        int count[3] = {0, 0, 0};
        bool persistent = false;
        int member_check = -1;   // scorer of the member check: 0 hmk_state_score, 1 hmk_packed_pair_score, 2 hmk_score12x3
    };
    LaunchLog* launch_log_ = nullptr;
    size_t hit_cap_ = 0;
    // ---- phase-1 scratch
    DevBuf<int32_t> d_qid_, d_nq_,
        d_ac_cnt_, d_ac_slot_, d_ac_score_, d_dirty_a_;
    DevBuf<int4> d_ac_full_, d_ac_best_;
    DevBuf<int32_t> d_sched_, d_clD_, d_cli_, d_lsort_;
    // sparse complete-linkage rows (see clinkage_rows)
    DevBuf<int64_t> d_cloff_;
    DevBuf<unsigned long long> d_cldeg_;
    DevBuf<uint64_t> d_clrows_, d_clalt_;
    DevBuf<int32_t> d_cltwin_, d_clrel_;
    int clinkage_rows(int* threads);
    size_t emit_hits(int q0, int sn, size_t cap, bool count = true);
    // score graph: the batch of query rows [q0, q1) kept on the device as edges in graph order, row r's edges at
    // row_off[r - q0] .. row_off[r - q0 + 1]; (next_i, next_r) = the cursor the last hmk_score_graph call returned
    struct GraphBatch {
        bool valid = false;
        int q0 = 0, q1 = 0, sn = HMK_MAXBATCH;   // sn: queries the next batch tries (cut while a batch overflows)
        std::vector<int64_t> row_off;
        int64_t next_i = -1, next_r = -1;
        DevBuf<unsigned long long> key[2], val[2];
        DevBuf<unsigned int> kept;
        DevBuf<int4> edges;
    } graph_;
    void graph_batch(int q0);
    void shift_pass(const int4* pairs, const unsigned int* count, unsigned int cap, int q0, int jbits,
                    unsigned long long* keys, unsigned long long* vals, unsigned int* kept, int32_t* score, int32_t* shift);
    // nearest partners (hmk_nearest): the query batch's profiles, top-k lists and gmin bounds, and its output rows --
    // the nearest search's own, so that nothing of it reaches a clustering run's batch buffers
    BatchBuf near_bb_;
    DevBuf<int32_t> d_near_out_;
    bool lsort_ = false;
    // phase-1 partner-search hits kept for phase 2 (opt.reuse): buffer, 64-bit counters [0] appended, [1] valid
    DevBuf<int4> d_xhits_;
    DevBuf<unsigned long long> d_xcount_;
    DevBuf<int32_t> d_qbatch_;
    size_t xhit_want_ = 0;            // entries the last run would have needed
    bool sym_ = false, reuse_ = false;
    int plan_sms_ = 0;                // SMs a bulk launch may count on (one less while the resolver holds an SM)
    int batch_id_ = 0;
    DevBuf<uint32_t> d_prof_;
    DevBuf<int4> d_hits_;
    DevBuf<unsigned int> d_counts_;   // [0] hit_count, [1] cand_count
    DevBuf<unsigned long long> d_pairctr_;
    // ---- phase-2 scratch
    DevBuf<int32_t> d_singles_, d_blockcnt_, d_cand_score_, d_cand_score2_, d_cq_c_, d_cq_q_, d_qstart_, d_cstart_, d_ccount_,
        d_a0_, d_flags_, d_base_cl_, d_cinfo_, d_work_, d_stamp_, d_cc_q_, d_cc_c_;
    DevBuf<unsigned long long> d_pairparts_, d_p2tim_;
    DevBuf<HmkDynEntry> d_dyn_;
    DevBuf<unsigned long long> d_key_q_, d_key_tmp_;
    DevBuf<unsigned char> d_cub_;
    DevBuf<uint32_t> d_fprof_;
    // ---- outputs
    DevBuf<int32_t> d_cluster_id_, d_member_rank_;
    int32_t n_unassigned_ = 0;
    size_t ncand_padded_ = 0;
    // ---- timing
    cudaEvent_t ev_a_ = nullptr, ev_b_ = nullptr, ev_c_ = nullptr, ev_t0_ = nullptr, ev_t1_ = nullptr;
    std::vector<cudaEvent_t> ev_pool_;
    size_t ev_used_ = 0;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> bulk_events_;
    int launches_ = 0, bulk_launches_ = 0;
    int64_t bulk_pairs_host_ = 0;

    HmkState state() {
        HmkState S;
        S.n = n_; S.res = d_res_.p; S.off = d_off_.p; S.ab = d_ab_.p; S.M = d_M_.p;
        S.T = T_; S.X = X_; S.P = P_; S.K = K_;
        S.id_of_rank = identity_rank_ ? nullptr : d_id_of_rank_.p;
        S.slot = d_slot_.p; S.rank = d_rank_.p; S.next = d_next_.p;
        S.c_founder = d_cf_.p; S.c_size = d_cs_.p; S.c_count = d_cc_.p; S.c_tail = d_ct_.p;
        S.qbatch = reuse_ ? d_qbatch_.p : nullptr;
        S.ctl = d_ctl_.p;
        return S;
    }
    void choose_scheme(const int32_t* M);
    int qt_max(const HmkScheme& sc, int kb) const;
    HmkScheme scheme_for(int n) const;
    void launch_profiles(int mode, const int32_t* ids, int nq, uint32_t* prof, const HmkScheme& sc, cudaStream_t s,
                         uint32_t* cells = nullptr, uint32_t* ops = nullptr);
    const int32_t* identity_ids();
    HmkBulkArgs query_batch(const int32_t* ids, int nq, uint32_t* prof, int kb);
    void merge_topk(int nq, int nstripes, int kb, const uint64_t* key, const int32_t* cnt, const int32_t* ovf, BatchBuf& out,
                    cudaStream_t s, const int32_t* slots = nullptr, int qt = 1);
    void report_kernel(const BulkKernel& k, bool persistent, int32_t* out) const;
    void plan_bulk(int mode, HmkBulkArgs& a, const HmkScheme* sch, int32_t* sched = nullptr) const;
    BulkKernel launch_planned(int mode, HmkBulkArgs a, const HmkScheme* sch, const int32_t* prof_ids, int prof_is_query,
                              cudaStream_t s);
    HmkBulkArgs launch_bulk(int mode, HmkBulkArgs a, const int32_t* prof_ids, int prof_is_query, cudaStream_t s = nullptr,
                            BatchBuf* bb = nullptr, DevBuf<int32_t>* sched_buf = nullptr, BulkKernel* ran = nullptr);
    cudaEvent_t next_event();
    // per-section device timers (only with opt.profile)
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> sections_;
    int sec_open_ = -1;
    cudaEvent_t sec_start_ = nullptr;
    void sec(int id) {   // close the open section and start section `id` (-1: just close)
        if (!opt.profile) return;
        cudaEvent_t e = next_event();
        CK(cudaEventRecord(e, st_));
        if (sec_open_ >= 0) sections_.push_back({sec_open_, {sec_start_, e}});
        sec_open_ = id;
        sec_start_ = e;
    }
    void reset_timing() {   // a call's timing starts empty: no recorded events, no open section
        ev_used_ = 0;
        bulk_events_.clear();
        sections_.clear();
        sec_open_ = -1;
    }
    double fold_timing();
public:
    double section_ms[HMK_NSECTIONS] = {0};
private:
    void fetch_ctl() {
        CK(cudaMemcpyAsync(h_ctl_, d_ctl_.p, sizeof(HmkCtl), cudaMemcpyDeviceToHost, st_));
#ifdef HMK_DEBUG
        if (getenv("HMK_DEBUG_HANG")) {      // debugging aid (debug builds only): report where the device is stuck
            for (int i = 0; i < 5000 && cudaStreamQuery(st_) == cudaErrorNotReady; i++) usleep(1000);
            if (cudaStreamQuery(st_) == cudaErrorNotReady) {
                cudaStream_t s3;
                cudaStreamCreateWithFlags(&s3, cudaStreamNonBlocking);
                cudaMemcpyAsync(h_ctl_, d_ctl_.p, sizeof(HmkCtl), cudaMemcpyDeviceToHost, s3);
                cudaStreamSynchronize(s3);
                fprintf(stderr, "HANG: side stream %s; ctl cur %d ncl %d unproc %d steps %d dbg %lld %lld %lld %lld lanes %llx %llx %llx %llx\n",
                        cudaStreamQuery(st2_) == cudaErrorNotReady ? "busy" : "idle", h_ctl_->cur, h_ctl_->ncl, h_ctl_->unproc_alive,
                        h_ctl_->steps, (long long)h_ctl_->dbg[0], (long long)h_ctl_->dbg[1], (long long)h_ctl_->dbg[2], (long long)h_ctl_->dbg[3],
                        (unsigned long long)h_ctl_->dbg[4], (unsigned long long)h_ctl_->dbg[5], (unsigned long long)h_ctl_->dbg[6], (unsigned long long)h_ctl_->dbg[7]);
                fflush(stderr);
                throw CudaError("device did not answer within 5 s (HMK_DEBUG_HANG)");
            }
        }
#endif
        CK(cudaStreamSynchronize(st_));
    }
    // the unrolled one-at-a-time pair scorer applies: uniform length 12, max shift 3, lane-sized matrix entries
    bool scalar12x3() const { return fast_scalar_ && fast_ && min_len_ == HMK_MAXL1 && max_len_ == HMK_MAXL1 && X_ == 3; }
    int phase1();
    void phase2();
    int compact_unassigned(int32_t* out);
    void sort_pairs(unsigned long long* keys, int32_t* vals, int n, int begin_bit, int end_bit);
};

// ---------------------------------------------------------------- upload
void Engine::choose_scheme(const int32_t* M) {
    fast_ = false;
    mixed_ = false;
    sc_ = HmkScheme{};
    sc_.L = max_len_; sc_.X = X_; sc_.P = P_; sc_.T = T_;
    if (opt.force_generic) return;
    if (n_ <= 0 || min_len_ < 1 || max_len_ > HMK_MAXLEN) return;
    const bool lng = max_len_ > HMK_MAXL1;       // more than one packed word: hmk_bulk_long
    const int nwcap = lng ? HMK_NWMAX : 4;
    if (X_ < 0 || X_ >= min_len_) return;
    int64_t mmin = M[0], mmax = M[0];
    for (int i = 0; i < HMK_NRES * HMK_NRES; i++) { mmin = std::min<int64_t>(mmin, M[i]); mmax = std::max<int64_t>(mmax, M[i]); }
    const int64_t bias = mmin < 0 ? -mmin : 0;
    bool present[HMK_MAXLEN + 1] = {false};
    for (int i = 0; i < n_; i++) present[h_off_[i + 1] - h_off_[i]] = true;
    // every pair of lengths (m, n) that occurs must fit the packed lanes: 2X+1+|n-m| lanes, and for each
    // shift k the lane value stays inside [0, top] with "score >= T" at the lane's top bit
    for (int lane16 = 0; lane16 <= 1; lane16++) {
        const int64_t half = lane16 ? 32768 : 128, top = lane16 ? 65535 : 255;
        const int lpw = lane16 ? 2 : 4;
        bool ok = true;
        int nw[HMK_MAXLEN + 1] = {0};
        for (int n = 1; n <= HMK_MAXLEN && ok; n++) {
            if (!present[n]) continue;
            for (int m = 1; m <= HMK_MAXLEN && ok; m++) {
                if (!present[m]) continue;
                const int ls = std::min(m, n), ll = std::max(m, n), d = ll - ls;
                const int lanes = 2 * X_ + 1 + d;
                nw[n] = std::max(nw[n], (lanes + lpw - 1) / lpw);
                if (nw[n] > nwcap) { ok = false; break; }
                for (int k = -X_; k <= X_ + d && ok; k++) {
                    const int64_t cells = std::min(ls + k, ll) - std::max(k, 0);
                    const int64_t pen = (int64_t)d * P_ + (k < 0 ? -2LL * k * P_ : 0) + (k > d ? 2LL * (k - d) * P_ : 0);
                    const int64_t init = pen + half - (int64_t)T_ - cells * bias;
                    const int64_t hi = init + cells * (mmax + bias);
                    if (init < 0 || hi > top || init > top) ok = false;
                }
            }
        }
        if (!ok) continue;
        sc_.lane16 = lane16; sc_.bias = (int32_t)bias; sc_.half = (int32_t)half;
        sc_.words = words_; sc_.long_layout = lng ? 1 : 0;
        sc_.filter = 0;
        if (min_len_ == max_len_) {
            fast_ = true;
            sc_.nw = nw[max_len_];
            if (opt.filter && !lane16 && !lng && sc_.nw == 2) {
                // the filter bytes (max of two neighbouring lanes, summed) must stay below 256
                int64_t worst = 0;
                for (int k = -X_; k <= X_; k++)   // filter lanes count every position (padding = score 0)
                    worst = std::max<int64_t>(worst, 2LL * P_ * (k < 0 ? -k : k) + half - (int64_t)T_ - max_len_ * bias);
                if (worst + (int64_t)max_len_ * (mmax + bias) <= 255) sc_.filter = 1;
            }
        } else {
            mixed_ = true;
            sc_.nw = 0;
            for (int n = 0; n <= HMK_MAXLEN; n++) { nw_len_[n] = nw[n]; sc_.nw = std::max(sc_.nw, nw[n]); }
        }
        sc_.prof_words = sc_.filter ? HMK_FPW : sc_.nw * (lng ? max_len_ : HMK_MAXL1) * HMK_NRES;
        return;
    }
}

void Engine::upload(const hmk_greedy_in* in) {
    CK(cudaSetDevice(device_));
    uploaded_ = false;      // a rejected upload leaves nothing to run
    ran_ = false;
    ids_filled_ = false;
    graph_.valid = false; graph_.next_i = graph_.next_r = -1; graph_.sn = HMK_MAXBATCH;
    if (!in || in->n < 0 || (in->n > 0 && (!in->residues || !in->offsets || !in->abundance)) || !in->matrix)
        throw std::invalid_argument("hmk_upload: null input");
    if (in->n > 0 && in->offsets[0] != 0) throw std::invalid_argument("hmk_upload: offsets[0] must be 0");
    for (int i = 0; i < in->n; i++)      // int32 prefix offsets: monotone also rules out a total length beyond int32
        if (in->offsets[i + 1] < in->offsets[i]) throw std::invalid_argument("hmk_upload: offsets not monotone");
    n_ = in->n; T_ = in->threshold; X_ = in->max_shift; P_ = in->shift_penalty; K_ = in->max_clusters;
    if (n_) h_off_.assign(in->offsets, in->offsets + n_ + 1);
    else h_off_.assign(1, 0);
    const size_t total = n_ ? (size_t)h_off_[n_] : 0;
    min_len_ = n_ ? INT32_MAX : 0; max_len_ = 0;
    for (int i = 0; i < n_; i++) {
        int l = h_off_[i + 1] - h_off_[i];
        min_len_ = std::min(min_len_, l); max_len_ = std::max(max_len_, l);
    }
    d_res_.reserve(total + 16); d_off_.reserve(n_ + 1); d_ab_.reserve(n_); d_M_.reserve(HMK_NRES * HMK_NRES);
    if (total) CK(cudaMemcpyAsync(d_res_.p, in->residues, total, cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(d_off_.p, h_off_.data(), sizeof(int32_t) * (n_ + 1), cudaMemcpyHostToDevice, st_));
    if (n_) CK(cudaMemcpyAsync(d_ab_.p, in->abundance, sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(d_M_.p, in->matrix, sizeof(int32_t) * HMK_NRES * HMK_NRES, cudaMemcpyHostToDevice, st_));
    sym_ = true;   // S(a, b) == S(b, a) for every pair iff the matrix is symmetric (equal lengths transpose it)
    for (int i = 0; i < HMK_NRES && sym_; i++)
        for (int j = 0; j < i; j++)
            if (in->matrix[i * HMK_NRES + j] != in->matrix[j * HMK_NRES + i]) { sym_ = false; break; }
    xhit_want_ = 0;
    // tie-break rank of the partner search: (abundance desc, id asc); identity when the
    // input is abundance-sorted (order "size", UniqueSequence.java:180)
    identity_rank_ = true;
    for (int i = 1; i < n_; i++)
        if (in->abundance[i] > in->abundance[i - 1]) { identity_rank_ = false; break; }
    if (!identity_rank_) {
        std::vector<int32_t> ids(n_), rk(n_);
        std::iota(ids.begin(), ids.end(), 0);
        const int32_t* ab = in->abundance;
        std::stable_sort(ids.begin(), ids.end(), [ab](int32_t a, int32_t b) { return ab[a] > ab[b]; });
        for (int i = 0; i < n_; i++) rk[ids[i]] = i;
        d_tierank_.reserve(n_); d_id_of_rank_.reserve(n_);
        CK(cudaMemcpyAsync(d_tierank_.p, rk.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
        CK(cudaMemcpyAsync(d_id_of_rank_.p, ids.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
        CK(cudaStreamSynchronize(st_));
    }
    words_ = max_len_ <= HMK_MAXLEN ? std::max(1, (max_len_ + HMK_MAXL1 - 1) / HMK_MAXL1) : 1;
    choose_scheme(in->matrix);
    for (auto& v : h_bucket_) v.clear();
    if (mixed_) {
        for (int i = 0; i < n_; i++) h_bucket_[h_off_[i + 1] - h_off_[i]].push_back(i);
        for (int L = 1; L <= HMK_MAXLEN; L++) {
            if (h_bucket_[L].empty()) continue;
            d_bucket_[L].reserve(h_bucket_[L].size());
            CK(cudaMemcpyAsync(d_bucket_[L].p, h_bucket_[L].data(), sizeof(int32_t) * h_bucket_[L].size(), cudaMemcpyHostToDevice, st_));
        }
        CK(cudaStreamSynchronize(st_));
    }
    // generic kernel on lengths that differ: the thread side is walked in (length, id) order, so that the lanes of a warp
    // run the same loop bounds
    lsort_ = !fast_ && !mixed_ && n_ > 0 && min_len_ != max_len_;
    if (lsort_) {
        std::vector<int32_t> ids(n_);
        std::iota(ids.begin(), ids.end(), 0);
        const int32_t* o = h_off_.data();
        std::stable_sort(ids.begin(), ids.end(), [o](int32_t a, int32_t b) { return o[a + 1] - o[a] < o[b + 1] - o[b]; });
        d_lsort_.reserve(n_);
        CK(cudaMemcpyAsync(d_lsort_.p, ids.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
        CK(cudaStreamSynchronize(st_));
    }
    fast_scalar_ = n_ > 0 && min_len_ >= 1 && max_len_ <= HMK_MAXL1 && X_ >= 0 && X_ < min_len_;
    // validate residues + pack 5 bits/residue on the device
    d_packed_.reserve((size_t)std::max(n_, 1) * words_);
    d_flags_.reserve(8);
    CK(cudaMemsetAsync(d_flags_.p, 0, 8 * sizeof(int32_t), st_));
    if (n_) {
        hmk_pack_sequences<<<(n_ + 255) / 256, 256, 0, st_>>>(n_, words_, d_res_.p, d_off_.p, d_packed_.p, d_flags_.p);
        CK(cudaGetLastError());
    }
    CK(cudaMemcpyAsync(h_scalars_, d_flags_.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    bad_residue_ = h_scalars_[0] != 0;
    const int kc = std::max(K_, 1);
    d_slot_.reserve(std::max(n_, 1)); d_rank_.reserve(std::max(n_, 1)); d_next_.reserve(std::max(n_, 1));
    d_cf_.reserve(kc); d_cs_.reserve(kc); d_cc_.reserve(kc); d_ct_.reserve(kc);
    d_ctl_.reserve(1); d_counts_.reserve(4); d_pairctr_.reserve(4);
    d_sidx_.reserve(std::max(n_, 1)); d_pcells_.reserve(std::max(K_, HMK_MAXBATCH)); d_pops_.reserve(std::max(K_, HMK_MAXBATCH));
    d_cluster_id_.reserve(std::max(n_, 1)); d_member_rank_.reserve(std::max(n_, 1));
    d_singles_.reserve(std::max(n_, 1)); d_blockcnt_.reserve((n_ + 1023) / 1024 + 1);
    uploaded_ = true;
    ran_ = false;
}

// ---------------------------------------------------------------- launch helpers
cudaEvent_t Engine::next_event() {
    if (ev_used_ == ev_pool_.size()) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        ev_pool_.push_back(e);
    }
    return ev_pool_[ev_used_++];
}

// adds each closed section's device time to its slot of section_ms and returns the summed time of the recorded bulk
// launches, then recycles the event pool; the events on other streams than st_ must be complete
double Engine::fold_timing() {
    if (opt.profile) CK(cudaStreamSynchronize(st_));
    double bulk_ms = 0;
    for (auto& pr : bulk_events_) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, pr.first, pr.second));
        bulk_ms += ms;
    }
    for (auto& sct : sections_) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, sct.second.first, sct.second.second));
        section_ms[sct.first] += ms;
    }
    reset_timing();
    return bulk_ms;
}

// kb: the per-query list length of the launch (HmkBulkArgs::kb); EMIT and DENSE launches are sized with it too
int Engine::qt_max(const HmkScheme& sc, int kb) const {
    if (opt.qt > 0) return (int)opt.qt;
    // a profile with its share of the carve-up, beside the hit queues of a 768-thread block and 128 bytes for the barrier
    // and alignment.  The 512-thread long kernel is sized the same way: its tiles are the ones it was measured with.
    // The filter kernel adds a prefix sum per profile and warp (hmk_packed_smem), with up to 12 bytes of alignment per warp.
    const size_t warps = HMK_BULK_THREADS / 32;
    const size_t per = (size_t)sc.prof_words * 4 + hmk_carve_bytes(1, kb, 0, false) + (sc.filter ? warps * 4 : 0);
    const size_t fixed = 128 + hmk_carve_bytes(0, kb, HMK_BULK_THREADS, false) + (sc.filter ? 16 + warps * 12 : 0);
    // the filter kernel's tile stays at the 56 profiles the batch size and chunking were measured with (more would fit)
    const size_t cap = sc.filter ? HMK_FILTER_QT : 255;
    return (int)std::min<size_t>(cap, std::max<size_t>(1, (smem_optin_ - fixed) / per));
}

// scheme of a launch whose thread-side sequences all have length n
HmkScheme Engine::scheme_for(int n) const {
    HmkScheme sc = sc_;
    sc.L = n;
    if (mixed_) sc.nw = nw_len_[n];
    sc.prof_words = sc.filter ? HMK_FPW : sc.nw * (sc.long_layout ? n : HMK_MAXL1) * HMK_NRES;
    return sc;
}

void Engine::launch_profiles(int mode, const int32_t* ids, int nq, uint32_t* prof, const HmkScheme& sc, cudaStream_t s,
                             uint32_t* cells, uint32_t* ops) {
    if (nq <= 0) return;
    hmk_build_profiles<<<nq, 128, 0, s>>>(sc, mode, ids, nq, d_res_.p, d_off_.p, d_M_.p, prof, cells, ops);
    CK(cudaGetLastError());
    launches_++;
}

// the ids 0 .. n - 1 on the device, copied once per upload when a call first needs them
const int32_t* Engine::identity_ids() {
    if (!ids_filled_) {
        std::vector<int32_t> ids(n_);
        std::iota(ids.begin(), ids.end(), 0);
        d_ids_.reserve(std::max(n_, 1));
        CK(cudaMemcpyAsync(d_ids_.p, ids.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
        ids_filled_ = true;
    }
    return d_ids_.p;
}

// the profile side of a bulk launch on st_ over the query ids[0 .. nq): their profiles in `prof` (packed kernels) and
// the list length kb; the caller sets the thread side and the mode's fields
HmkBulkArgs Engine::query_batch(const int32_t* ids, int nq, uint32_t* prof, int kb) {
    if (fast_) launch_profiles(HMK_PROF_QUERY, ids, nq, prof, sc_, st_);
    HmkBulkArgs a{};
    a.prof = prof; a.nq = nq; a.kb = kb;
    a.packed = d_packed_.p;
    return a;
}

// merges nstripes lists of kb keys per query ([nstripes][nq][kb]) into out.bk_*; slots / qt: the slot counters of a
// persistent launch (HmkBulkArgs::sched + nqt) and its profiles per tile
void Engine::merge_topk(int nq, int nstripes, int kb, const uint64_t* key, const int32_t* cnt, const int32_t* ovf, BatchBuf& out,
                        cudaStream_t s, const int32_t* slots, int qt) {
    hmk_topk_merge<<<(nq * 32 + 255) / 256, 256, 0, s>>>(nq, nstripes, kb, key, cnt, ovf, out.bk_key.p, out.bk_cnt.p, out.bk_ovf.p,
                                                         slots, qt);
    CK(cudaGetLastError());
    launches_++;
}

// which kernel a probe's launch ran (kind -1: none, the launch was empty): kind, the filter kernel's compile-time length,
// words per profile entry, lane bits, persistent grid
void Engine::report_kernel(const BulkKernel& k, bool persistent, int32_t* out) const {
    const bool packed = k.kind > BulkKernel::GENERIC;
    out[0] = k.kind;
    out[1] = k.lt;
    out[2] = packed ? sc_.nw : 0;
    out[3] = packed ? (sc_.lane16 ? 16 : 8) : k.fn ? 32 : 0;
    out[4] = persistent ? 1 : 0;
}

// (x, y, z) of the first `stored` hits of a device buffer, as int32 triples
static void copy_hit_triples(const int4* d_hits, size_t stored, int32_t* out) {
    if (!stored) return;
    std::vector<int4> h(stored);
    CK(cudaMemcpy(h.data(), d_hits, sizeof(int4) * stored, cudaMemcpyDeviceToHost));
    for (size_t e = 0; e < stored; e++) { out[3 * e] = h[e].x; out[3 * e + 1] = h[e].y; out[3 * e + 2] = h[e].z; }
}

// the bulk kernel of a (MODE, scheme) pair; `sch` NULL: the generic kernel
template <int MODE>
static BulkKernel pick_bulk_kernel(const HmkScheme* sch) {
    constexpr int FM = MODE == HMK_MODE_DENSE ? HMK_MODE_EMIT : MODE;   // hmk_bulk_filter has no DENSE form
    if (!sch) return {BulkKernel::GENERIC, -1, HMK_GENERIC_THREADS, (const void*)hmk_bulk_generic<MODE>};
    if (sch->long_layout) return {BulkKernel::LONG, -1, HMK_LONG_THREADS, (const void*)hmk_bulk_long<MODE>};
    if (sch->filter) {
        if (MODE == HMK_MODE_DENSE)    // every score is wanted: exact kernel on the filter-layout profiles
            return {BulkKernel::FAST, -1, HMK_BULK_THREADS, (const void*)hmk_bulk_fast<2, HMK_MODE_DENSE, true>};
        if (sch->L == 12) return {BulkKernel::FILTER, 12, HMK_BULK_THREADS, (const void*)hmk_bulk_filter<FM, 12>};
        return {BulkKernel::FILTER, 0, HMK_BULK_THREADS, (const void*)hmk_bulk_filter<FM, 0>};
    }
    switch (sch->nw) {
        case 1: return {BulkKernel::FAST, -1, HMK_BULK_THREADS, (const void*)hmk_bulk_fast<1, MODE>};
        case 2: return {BulkKernel::FAST, -1, HMK_BULK_THREADS, (const void*)hmk_bulk_fast<2, MODE>};
        case 3: return {BulkKernel::FAST, -1, HMK_BULK_THREADS, (const void*)hmk_bulk_fast<3, MODE>};
        default: return {BulkKernel::FAST, -1, HMK_BULK_THREADS, (const void*)hmk_bulk_fast<4, MODE>};
    }
}
static BulkKernel bulk_kernel(int mode, const HmkScheme* sch) {
    return mode == HMK_MODE_TOPK ? pick_bulk_kernel<HMK_MODE_TOPK>(sch)
         : mode == HMK_MODE_EMIT ? pick_bulk_kernel<HMK_MODE_EMIT>(sch) : pick_bulk_kernel<HMK_MODE_DENSE>(sch);
}

// tiling of a bulk launch: nqt profile tiles x nstripes database stripes; the grid is an exact
// multiple of the SM count whenever the database is large enough (one CTA per SM is resident:
// the profile tile fills shared memory)
void Engine::plan_bulk(int mode, HmkBulkArgs& a, const HmkScheme* sch, int32_t* sched) const {
    const int threads = bulk_kernel(mode, sch).threads;
    const int sms = plan_sms_ > 0 ? plan_sms_ : sm_count_;
    int qmax = sch ? qt_max(*sch, a.kb) : 128;
    if (!sch) {     // generic kernel: a thread scores its item against the whole tile, one pair after the other -- small
                    // databases get small tiles, so that there are about two CTAs per SM instead of a few long threads
        const int64_t blocks = (a.ndb + threads - 1) / threads;
        qmax = (int)std::max<int64_t>(8, std::min<int64_t>(128, (int64_t)a.nq * blocks / (2 * sms)));
    }
    a.nqt = (a.nq + qmax - 1) / qmax;
    a.qt = (a.nq + a.nqt - 1) / a.nqt;
    a.sched = nullptr; a.nchunks = 0;
    if (sched && opt.persistent && sch && sch->filter && a.nqt <= HMK_MAXTILES_PERSISTENT) {
        // filter kernel, persistent form: one CTA per SM, dynamic chunks (about 8 per CTA and tile, a multiple of the
        // block size) -- no tail wave, and a CTA loads a profile tile once instead of once per stripe
        const int64_t units = (int64_t)a.nqt * ((a.ndb + threads - 1) / threads);
        const int G = (int)std::max<int64_t>(1, std::min<int64_t>(sms, units));
        const int per_tile = std::max(1, G / a.nqt);
        int chunk = (a.ndb / (per_tile * 8) + threads - 1) / threads * threads;
        chunk = std::max(threads, std::min(chunk, 8 * threads));
        a.chunk = chunk;
        a.nchunks = (a.ndb + chunk - 1) / chunk;
        a.nstripes = G;           // output slots per query: a CTA engages a tile at most once
        a.sched = sched;
        return;
    }
    int want = (int)((sms * opt.waves + a.nqt - 1) / a.nqt);
    if (a.nqt <= sms * opt.waves && (sms * opt.waves) % a.nqt != 0) {
        // nqt does not divide waves*SMs: round the total up to the next multiple of the SM count
        int total = (int)((((int64_t)want * a.nqt + sms - 1) / sms) * sms);
        want = std::max(1, total / a.nqt);
    }
    // a CTA stages a whole profile tile (up to 190 KB) before it scores anything: at least 8 block iterations per stripe
    int max_stripes = std::max<int64_t>(1, a.ndb / (std::max<int64_t>(1, opt.min_iters) * threads));
    if (a.nqt > sms * opt.waves) {
        // more profile tiles than resident CTAs: take the stripe count (<= 8, stripes of >= 16 K items) that
        // fills the last wave best
        double best = 0;
        for (int s = 1; s <= 8 && (s == 1 || a.ndb / s >= 16384); s++) {
            const int64_t total = (int64_t)a.nqt * s;
            const double eff = (double)total / (double)(((total + sms - 1) / sms) * sms);
            if (eff > best + 0.01) { best = eff; want = s; }
        }
    }
    a.nstripes = std::max(1, std::min(want, max_stripes));
    a.chunk = (a.ndb + a.nstripes - 1) / a.nstripes;
    if (sch && sch->filter) a.chunk = std::min(a.chunk, (1 << 22) - 1);   // candidate entries hold 22 bits of stripe offset
    a.nstripes = (a.ndb + a.chunk - 1) / a.chunk;
}

// launches a planned bulk pass.  `sch` non-NULL: packed SWAR kernel with that scheme (a.prof holds
// matching profiles); NULL: generic scalar kernel (prof_ids / prof_is_query name the profile side).
BulkKernel Engine::launch_planned(int mode, HmkBulkArgs a, const HmkScheme* sch, const int32_t* prof_ids, int prof_is_query,
                                  cudaStream_t s) {
    a.sc = sch ? *sch : sc_;
    a.pair_counter = d_pairctr_.p;
    const int grid = a.sched ? a.nstripes : a.nqt * a.nstripes;
    if (a.sched) CK(cudaMemsetAsync(a.sched, 0, sizeof(int32_t) * 2 * a.nqt, s));
    const BulkKernel k = bulk_kernel(mode, sch);
    HmkGenericArgs g;
    size_t smem;
    void* args[1];
    if (sch) {
        smem = hmk_packed_smem(a.qt, (uint32_t)sch->prof_words * 4, a.kb, k.threads, k.kind == BulkKernel::FILTER).total;
        args[0] = &a;
    } else {
        g.b = a; g.prof_ids = prof_ids; g.prof_is_query = prof_is_query;
        g.res = d_res_.p; g.off = d_off_.p; g.M = d_M_.p; g.maxlen = std::max(max_len_, 1);
        g.db_smem = g.maxlen <= 128 ? 1 : 0;
        smem = hmk_generic_smem(a.qt, a.kb, g.maxlen, g.db_smem).total;
        args[0] = &g;
    }
    smem_cfg_.ensure(k.fn, smem);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (opt.profile) { e0 = next_event(); e1 = next_event(); CK(cudaEventRecord(e0, s)); }
    CK(cudaLaunchKernel(k.fn, dim3(grid), dim3(k.threads), args, smem, s));
    if (opt.profile) { CK(cudaEventRecord(e1, s)); bulk_events_.push_back({e0, e1}); }
    launches_++;
    bulk_launches_++;
    if (launch_log_) {
        launch_log_->last[mode] = k;
        launch_log_->count[mode]++;
        if (mode == HMK_MODE_TOPK && a.sched) launch_log_->persistent = true;
    }
    return k;
}

// one-launch convenience: the uniform packed kernel when the whole input has one length <= 12, else the generic kernel.
// Returns the planned arguments (a TOPK launch's per-stripe lists are merged by the caller, with hmk_topk_merge).
HmkBulkArgs Engine::launch_bulk(int mode, HmkBulkArgs a, const int32_t* prof_ids, int prof_is_query, cudaStream_t s, BatchBuf* bb,
                                DevBuf<int32_t>* sched_buf, BulkKernel* ran) {
    if (a.nq <= 0 || a.ndb <= 0) return a;
    if (!s) s = st_;
    const HmkScheme* sch = fast_ ? &sc_ : nullptr;
    DevBuf<int32_t>& sched = sched_buf ? *sched_buf : (bb ? bb->sched : d_sched_);      // launches on different streams overlap: one each
    sched.reserve(2 * HMK_MAXTILES_PERSISTENT);
    plan_bulk(mode, a, sch, mode == HMK_MODE_DENSE ? nullptr : sched.p);
    if (mode == HMK_MODE_TOPK) {
        const size_t slots = (size_t)a.nstripes * a.nq;
        bb->tk_key.reserve(slots * a.kb); bb->tk_cnt.reserve(slots); bb->tk_ovf.reserve(slots);
        a.tk_key = bb->tk_key.p; a.tk_cnt = bb->tk_cnt.p; a.tk_ovf = bb->tk_ovf.p;
        a.stripe_base = 0;
    }
    const BulkKernel k = launch_planned(mode, a, sch, prof_ids, prof_is_query, s);
    if (ran) *ran = k;
    return a;
}

int Engine::compact_unassigned(int32_t* out) {
    if (n_ == 0) return 0;
    const int nb = (n_ + 1023) / 1024;
    hmk_count_unassigned<<<nb, 1024, 0, st_>>>(d_slot_.p, n_, d_blockcnt_.p);
    hmk_scan_blocks<<<1, 32, 0, st_>>>(d_blockcnt_.p, nb, d_flags_.p + 4);
    hmk_scatter_unassigned<<<nb, 1024, 0, st_>>>(d_slot_.p, n_, d_blockcnt_.p, out);
    CK(cudaGetLastError());
    launches_ += 3;
    CK(cudaMemcpyAsync(h_scalars_ + 4, d_flags_.p + 4, sizeof(int32_t), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    return h_scalars_[4];
}

void Engine::sort_pairs(unsigned long long* keys, int32_t* vals, int n, int begin_bit, int end_bit) {
    // ancillary plumbing (grouping the sparse candidate list); CUB radix sort, in place via temporaries
    d_key_tmp_.reserve(n);
    d_cand_score2_.reserve(n);
    size_t bytes = 0;
    CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, keys, d_key_tmp_.p, vals, d_cand_score2_.p, n, begin_bit, end_bit, st_));
    d_cub_.reserve(bytes);
    CK(cub::DeviceRadixSort::SortPairs(d_cub_.p, bytes, keys, d_key_tmp_.p, vals, d_cand_score2_.p, n, begin_bit, end_bit, st_));
    CK(cudaMemcpyAsync(keys, d_key_tmp_.p, sizeof(unsigned long long) * n, cudaMemcpyDeviceToDevice, st_));
    CK(cudaMemcpyAsync(vals, d_cand_score2_.p, sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, st_));
    launches_ += 8;
}

// ---------------------------------------------------------------- phase 1
// founder filter of the cluster search for the clusters [from, to): appends (query index, founder id, score) to bb.hits
void Engine::founder_hits(BatchBuf& bb, int from, int to, cudaStream_t s, DevBuf<int32_t>& sched) {
    if (to <= from) return;
    HmkBulkArgs a{};
    a.prof = bb.prof.p; a.nq = bb.nq; a.kb = (int)opt.kb;
    a.packed = d_packed_.p; a.db_ids = d_cf_.p + from; a.db_begin = 0; a.ndb = to - from;
    a.hits = bb.hits.p; a.hit_count = bb.hcount.p; a.hit_cap = (unsigned int)bb.hit_cap;
    a.discards = &d_ctl_.p->discards; a.discards_seen = h_ctl_->discards;
    if (!mixed_ || max_len_ > HMK_MAXL1) { launch_bulk(HMK_MODE_EMIT, a, bb.qid.p, 1, s, nullptr, &sched); return; }
    // mixed lengths <= 12: the founders are split by length on the device (no host round trip: every bucket is launched
    // for the upper bound `to - from` and reads its real size on the device) and each bucket runs the packed kernel on
    // the profiles of that thread-side length -- built by the partner search of this batch, or here
    const int cnt = to - from;
    bb.fb_ids.reserve((size_t)(HMK_MAXL1 + 1) * HMK_FB_STRIDE); bb.fb_cnt.reserve(HMK_MAXLEN + 1);
    for (int f0 = 0; f0 < cnt; f0 += HMK_FB_STRIDE) {       // (more founders than the bucket arrays hold: in slices)
        const int fn = std::min<int>(HMK_FB_STRIDE, cnt - f0);
        CK(cudaMemsetAsync(bb.fb_cnt.p, 0, sizeof(int32_t) * (HMK_MAXLEN + 1), s));
        hmk_bucket_by_length<<<(fn + 255) / 256, 256, 0, s>>>(d_cf_.p + from + f0, fn, d_off_.p, HMK_FB_STRIDE, bb.fb_ids.p, bb.fb_cnt.p);
        launches_++;
        for (int L = min_len_; L <= max_len_; L++) {
            if (h_bucket_[L].empty()) continue;
            const HmkScheme sch = scheme_for(L);
            auto& pf = bb.prof_len[L];
            if (bb.prof_len_batch[L] != bb.batch_id) {      // no later singleton of this length: the partner search skipped it
                pf.reserve((size_t)HMK_MAXBATCH * sch.prof_words);
                bb.pcells[L].reserve(HMK_MAXBATCH); bb.pops[L].reserve(HMK_MAXBATCH);
                launch_profiles(HMK_PROF_QUERY, bb.qid.p, bb.nq, pf.p, sch, s, bb.pcells[L].p, bb.pops[L].p);
                bb.prof_len_batch[L] = bb.batch_id;
            }
            HmkBulkArgs b = a;
            b.prof = pf.p; b.prof_cells = bb.pcells[L].p; b.prof_ops = bb.pops[L].p;
            b.db_ids = bb.fb_ids.p + (size_t)L * HMK_FB_STRIDE; b.ndb = fn; b.ndb_dev = bb.fb_cnt.p + L;
            plan_bulk(HMK_MODE_EMIT, b, &sch);
            launch_planned(HMK_MODE_EMIT, b, &sch, bb.qid.p, 1, s);
        }
    }
}

// Selects the next batch, builds its query profiles and runs the partner search (+ the multi-GPU best-hit exchange) and
// part 1 of the cluster search on stream `s`.  The rest of the batch's state-independent work -- merging the per-stripe
// top-k lists, the intra-batch and partner-candidate score tables and their masks -- runs on stream `t` behind the
// partner search, so that the next batch's partner search follows this one directly on `s`.  bb.ready fires when both
// are complete; bb.searched when the query ids are final (the next batch starts behind the last of them).
void Engine::stage_partner_search(BatchBuf& bb, int nq, int db_from, const int32_t* start_after, int ncl_known, cudaStream_t s,
                                  cudaStream_t t) {
    const int kb = (int)opt.kb;
    bb.qid.reserve(HMK_MAXBATCH); bb.nq_dev.reserve(1);
    bb.bk_key.reserve((size_t)HMK_MAXBATCH * kb); bb.bk_cnt.reserve(HMK_MAXBATCH); bb.bk_ovf.reserve(HMK_MAXBATCH);
    if (fast_) bb.prof.reserve((size_t)HMK_MAXBATCH * sc_.prof_words);
    hmk_select_queries<<<1, 1024, 0, s>>>(d_slot_.p, n_, d_ctl_.p, start_after, nq, bb.qid.p, bb.nq_dev.p);
    CK(cudaGetLastError());
    launches_++;
    if (world_ > 1) {
        // A batch prepared ahead is selected while the resolver of an earlier batch is still turning singletons into
        // members, so WHICH ids it picks depends on timing.  On one GPU that is harmless (the resolver skips what has
        // been consumed in the meantime); across ranks every rank must score the SAME queries, or the best-hit exchange
        // below would merge lists of different queries position by position.  Rank 0's selection wins.
        bb.gqid.reserve((size_t)world_ * HMK_MAXBATCH);
        allgather(bb.qid.p, bb.gqid.p, sizeof(int32_t) * nq, s);
        CK(cudaMemcpyAsync(bb.qid.p, bb.gqid.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToDevice, s));
    }
    HmkBulkArgs a{};
    a.nq = nq; a.kb = kb;
    a.packed = d_packed_.p; a.slot = d_slot_.p; a.q_minid = bb.qid.p;
    a.tierank = identity_rank_ ? nullptr : d_tierank_.p;
    a.discards = &d_ctl_.p->discards; a.discards_seen = h_ctl_->discards;
    bb.batch_id = ++batch_id_;
    bb.gmin.reserve(HMK_MAXBATCH);
    CK(cudaMemsetAsync(bb.gmin.p, 0, sizeof(unsigned long long) * nq, s));
    a.tk_gmin = bb.gmin.p;
    if (reuse_) {
        a.xhits = d_xhits_.p; a.xhit_count = d_xcount_.p; a.xhit_cap = d_xhits_.cap; a.xbatch = bb.batch_id;
    }
    // the per-stripe top-k lists of the partner search, merged into bb.bk_* (at world > 1 on `s`: the all-gather below
    // needs this rank's merged lists, and every NCCL call stays on one stream, in the same order on every rank)
    int merge_stripes = 0;
    const int32_t* merge_slots = nullptr;
    int merge_qt = 1;
    if (!mixed_) {
        if (fast_) launch_profiles(HMK_PROF_QUERY, bb.qid.p, nq, bb.prof.p, sc_, s);
        a.prof = bb.prof.p;
        // this rank's stripe of the later singletons (the whole range on one GPU)
        const int64_t span = (int64_t)n_ - db_from;
        int lo = db_from + (int)(span * rank_ / world_), hi = db_from + (int)(span * (rank_ + 1) / world_);
        a.db_ids = nullptr; a.db_begin = lo; a.ndb = hi - lo;
        if (lsort_) {       // the whole (length, id)-ordered list, striped across the ranks; ids before db_from are skipped
            lo = (int)((int64_t)n_ * rank_ / world_); hi = (int)((int64_t)n_ * (rank_ + 1) / world_);
            a.db_ids = d_lsort_.p + lo; a.db_begin = 0; a.ndb = hi - lo; a.db_min_id = db_from;
        }
        if (a.ndb > 0) {
            const HmkBulkArgs p = launch_bulk(HMK_MODE_TOPK, a, bb.qid.p, 1, s, &bb);
            merge_stripes = p.nstripes; merge_qt = p.qt;
            merge_slots = p.sched ? p.sched + p.nqt : nullptr;
        }
    } else {
        // mixed lengths: one packed-kernel launch per length bucket of the later singletons (profiles are
        // built per thread-side length), all writing into one set of per-stripe lists merged once
        struct Plan { int L; HmkBulkArgs a; HmkScheme sc; };
        std::vector<Plan> plans;
        int total_stripes = 0;
        for (int L = 1; L <= HMK_MAXLEN; L++) {
            const auto& ids = h_bucket_[L];
            if (ids.empty()) continue;
            const int first = (int)(std::lower_bound(ids.begin(), ids.end(), db_from) - ids.begin());
            const int64_t span = (int64_t)ids.size() - first;
            const int lo = first + (int)(span * rank_ / world_), hi = first + (int)(span * (rank_ + 1) / world_);
            if (hi <= lo) continue;
            Plan p;
            p.L = L; p.sc = scheme_for(L); p.a = a;
            p.a.db_ids = d_bucket_[L].p + lo; p.a.db_begin = 0; p.a.ndb = hi - lo;
            plan_bulk(HMK_MODE_TOPK, p.a, &p.sc);
            p.a.stripe_base = total_stripes;
            total_stripes += p.a.nstripes;
            plans.push_back(p);
        }
        if (!plans.empty()) {
            const size_t slots = (size_t)total_stripes * nq;
            bb.tk_key.reserve(slots * kb); bb.tk_cnt.reserve(slots); bb.tk_ovf.reserve(slots);
            // the buckets are independent (own profiles, own output slots): fork them over the auxiliary streams so
            // that the small launches of a 100 k-sequence input fill the GPU together, then join
            CK(cudaEventRecord(fork_ev_, s));
            int k = 0;
            for (auto& p : plans) {
                cudaStream_t as = opt.bucket_aux ? aux_[k % HMK_NAUX] : s;
                if (opt.bucket_aux && k < HMK_NAUX) CK(cudaStreamWaitEvent(as, fork_ev_, 0));
                auto& pf = bb.prof_len[p.L];
                pf.reserve((size_t)HMK_MAXBATCH * p.sc.prof_words);
                bb.pcells[p.L].reserve(HMK_MAXBATCH); bb.pops[p.L].reserve(HMK_MAXBATCH);
                launch_profiles(HMK_PROF_QUERY, bb.qid.p, nq, pf.p, p.sc, as, bb.pcells[p.L].p, bb.pops[p.L].p);
                bb.prof_len_batch[p.L] = bb.batch_id;
                p.a.prof = pf.p; p.a.prof_cells = bb.pcells[p.L].p; p.a.prof_ops = bb.pops[p.L].p;
                p.a.tk_key = bb.tk_key.p; p.a.tk_cnt = bb.tk_cnt.p; p.a.tk_ovf = bb.tk_ovf.p;
                launch_planned(HMK_MODE_TOPK, p.a, &p.sc, bb.qid.p, 1, as);
                k++;
            }
            for (int j = 0; opt.bucket_aux && j < std::min(k, (int)HMK_NAUX); j++) {
                CK(cudaEventRecord(join_ev_[j], aux_[j]));
                CK(cudaStreamWaitEvent(s, join_ev_[j], 0));
            }
            merge_stripes = total_stripes;
        }
    }
    if (merge_stripes == 0) {
        CK(cudaMemsetAsync(bb.bk_cnt.p, 0, sizeof(int32_t) * nq, s));
        CK(cudaMemsetAsync(bb.bk_ovf.p, 0, sizeof(int32_t) * nq, s));
    }
    auto merge_stripe_lists = [&](cudaStream_t ms) {
        if (merge_stripes) merge_topk(nq, merge_stripes, kb, bb.tk_key.p, bb.tk_cnt.p, bb.tk_ovf.p, bb, ms, merge_slots, merge_qt);
    };
    if (world_ > 1) {
        merge_stripe_lists(s);
        // best-hit exchange: every rank contributes its stripe's top-k per query (a few KB),
        // then every rank merges the same lists -> identical, replicated decisions
        bb.gk_key.reserve((size_t)world_ * nq * kb); bb.gk_cnt.reserve((size_t)world_ * nq); bb.gk_ovf.reserve((size_t)world_ * nq);
        NK(NcclApi::get().GroupStart());
        allgather(bb.bk_key.p, bb.gk_key.p, sizeof(uint64_t) * nq * kb, s);
        allgather(bb.bk_cnt.p, bb.gk_cnt.p, sizeof(int32_t) * nq, s);
        allgather(bb.bk_ovf.p, bb.gk_ovf.p, sizeof(int32_t) * nq, s);
        NK(NcclApi::get().GroupEnd());
    }
    // ---- tail, on `t`
    CK(cudaEventRecord(bb.searched, s));
    if (t != s) CK(cudaStreamWaitEvent(t, bb.searched, 0));
    if (world_ > 1) merge_topk(nq, world_, kb, bb.gk_key.p, bb.gk_cnt.p, bb.gk_ovf.p, bb, t);
    else merge_stripe_lists(t);
    // intra-batch scores S(member = q_b2, query = q_b); row strides padded to 16 bytes for the TMA row prefetch
    const int ib_stride = (nq + 3) & ~3, pd_stride = (nq * kb + 3) & ~3, nw = (nq + 31) / 32;
    bb.ib.reserve((size_t)HMK_MAXBATCH * (HMK_MAXBATCH + 4)); bb.ibm.reserve((size_t)HMK_MAXBATCH * (HMK_MAXBATCH / 32)); bb.ibm2.reserve((size_t)HMK_MAXBATCH * (HMK_MAXBATCH / 32));
    bb.pcand.reserve((size_t)nq * kb); bb.pd.reserve((size_t)nq * (pd_stride + 4));
    const bool dense_packed = mixed_ && fast_scalar_;      // mixed lengths <= 12: one thread per pair on the packed words
    if (dense_packed) {
        hmk_dense_packed<<<std::min(sm_count_ * 8, (nq * nq + 255) / 256), 256, 0, t>>>(d_packed_.p, bb.qid.p, nq, bb.qid.p, nq, d_M_.p, X_, P_,
                                                                                       bb.ib.p, ib_stride, d_pairctr_.p);
        launches_++;
    } else {
        HmkBulkArgs d{};
        d.prof = bb.prof.p; d.nq = nq; d.kb = kb;
        d.packed = d_packed_.p; d.db_ids = bb.qid.p; d.db_begin = 0; d.ndb = nq;
        d.dense = bb.ib.p; d.dense_stride = ib_stride;
        launch_bulk(HMK_MODE_DENSE, d, bb.qid.p, 1, t);
    }
    hmk_ib_mask<<<(nq * nw + 127) / 128, 128, 0, t>>>(nq, nw, T_, bb.ib.p, ib_stride, bb.ibm.p, kb, bb.bk_key.p, bb.bk_cnt.p, bb.ibm2.p);
    launches_++;
    // S(partner candidate, query) for every candidate of the batch: clusters born inside the
    // batch have one of these as their second member
    {
        const int npc = nq * kb;
        hmk_partner_ids<<<(npc + 127) / 128, 128, 0, t>>>(nq, kb, bb.bk_key.p, bb.bk_cnt.p,
                                                          identity_rank_ ? nullptr : d_id_of_rank_.p, bb.qid.p, bb.pcand.p);
        launches_++;
        if (dense_packed) {
            hmk_dense_packed<<<std::min(sm_count_ * 8, (nq * npc + 255) / 256), 256, 0, t>>>(d_packed_.p, bb.qid.p, nq, bb.pcand.p, npc, d_M_.p, X_,
                                                                                            P_, bb.pd.p, pd_stride, d_pairctr_.p);
            launches_++;
        } else {
            HmkBulkArgs d{};
            d.prof = bb.prof.p; d.nq = nq; d.kb = kb;
            d.packed = d_packed_.p; d.db_ids = bb.pcand.p; d.db_begin = 0; d.ndb = npc;
            d.dense = bb.pd.p; d.dense_stride = pd_stride;
            launch_bulk(HMK_MODE_DENSE, d, bb.qid.p, 1, t);
        }
    }
    CK(cudaGetLastError());
    // cluster search, part 1 (state independent as well: founders never change), on `s`: the clusters that exist now.  The
    // ones created until the batch is resolved are added on the main stream (phase1)
    bb.nq = nq;
    bb.hit_cap = hit_cap_;
    bb.hits.reserve(bb.hit_cap); bb.hcount.reserve(4);
    bb.sched2.reserve(2 * HMK_MAXTILES_PERSISTENT);
    CK(cudaMemsetAsync(bb.hcount.p, 0, 4 * sizeof(unsigned int), s));
    bb.ncl_ahead = ncl_known;
    founder_hits(bb, 0, ncl_known, s, bb.sched2);
    if (t != s) {
        CK(cudaEventRecord(part1_ev_, s));
        CK(cudaStreamWaitEvent(t, part1_ev_, 0));
    }
    CK(cudaEventRecord(bb.ready, t));
    bb.valid = true;
}

// Cluster search, part 2, on the main stream: the linked member check of batch cb's founder hits against the clusters
// [0, ncl) (ac_cnt / ac_slot / ac_score, capq rows per query), then each query's candidate records and best candidate
void Engine::check_members(const BatchBuf& cb, int ncl, int capq) {
    const int nq = cb.nq;
    CK(cudaMemsetAsync(d_ac_cnt_.p, 0, sizeof(int32_t) * nq, st_));
    if (ncl > 0) {
        HmkCheckArgs c{};
        c.S = state(); c.hits = cb.hits.p; c.hit_count = cb.hcount.p; c.hit_cap = (unsigned int)cb.hit_cap;
        c.hit_t_is_query = 1; c.qids = cb.qid.p; c.sidx = nullptr;
        c.ac_cnt = d_ac_cnt_.p; c.ac_slot = d_ac_slot_.p; c.ac_score = d_ac_score_.p; c.capq = capq;
        c.cand_count = cb.hcount.p + 1; c.cand_cap = 0; c.linked = 1;
        c.packed = fast_scalar_ ? d_packed_.p : nullptr; c.L = max_len_; c.pair_parts = d_pairparts_.p;
        const bool fast = scalar12x3();
        if (fast) hmk_member_check<true><<<sm_count_ * 2, 256, 0, st_>>>(c);
        else hmk_member_check<false><<<sm_count_ * 2, 256, 0, st_>>>(c);
        CK(cudaGetLastError());
        launches_++;
        if (launch_log_) launch_log_->member_check = fast ? 2 : c.packed ? 1 : 0;
    }
    hmk_p1_prepare_candidates<<<(nq * 32 + 255) / 256, 256, 0, st_>>>(state(), nq, capq, d_ac_cnt_.p, d_ac_slot_.p, d_ac_score_.p,
                                                                     d_ac_full_.p, d_ac_best_.p);
    CK(cudaGetLastError());
    launches_++;
}

int Engine::phase1() {
    int B = (int)opt.batch;
    if (B <= 0) B = fast_ ? (sc_.filter ? 8 : 3) * qt_max(sc_, (int)opt.kb) : 192;   // measured optimum on the 1 M workload
    B = std::max(1, std::min(B, HMK_MAXBATCH));
    const size_t resolve_avail = smem_optin_ - 3 * HMK_HASH_SIZE * 4 - 1024;   // minus the kernel's static shared memory
    {   // the resolver keeps the whole batch's bookkeeping in shared memory
        auto need = [&](int b) { return hmk_resolve_fixed_bytes(b, (b + 31) / 32, (int)opt.kb) + 64; };
        while (B > 32 && need(B) > resolve_avail) B -= 32;
    }
    size_t capq = (size_t)std::max<int64_t>(1, opt.capq);
    d_ac_cnt_.reserve(B); d_ac_slot_.reserve((size_t)B * capq); d_ac_score_.reserve((size_t)B * capq);
    d_ac_full_.reserve((size_t)B * capq); d_ac_best_.reserve(B);
    batch_id_ = 0;
    reuse_ = opt.reuse && sym_ && K_ > 0 && n_ > 1;
    if (reuse_) {
        // room for every partner-search hit: the last run's need if known, else ~96 per sequence; a run that
        // overflows falls back to the separate founder pass in phase 2 (HMK_FLAG_XHIT_OVERFLOW) and remembers the
        // size it needed
        size_t want = opt.xhit_cap > 0 ? (size_t)opt.xhit_cap
                      : xhit_want_   ? xhit_want_ + xhit_want_ / 8
                                     : std::max<size_t>((size_t)1 << 20, (size_t)n_ * 96);
        want = std::min<size_t>(want, (size_t)1 << 30);
        d_xhits_.reserve(want); d_xcount_.reserve(2); d_qbatch_.reserve(n_);
        CK(cudaMemsetAsync(d_xcount_.p, 0, 2 * sizeof(unsigned long long), st_));
        CK(cudaMemsetAsync(d_qbatch_.p, 0xff, sizeof(int32_t) * n_, st_));
    }
    hit_cap_ = (size_t)opt.hit_cap;
    // batch ids restart at 1, so per-length profiles that an earlier run or a batch probe built must not be taken for
    // this run's batches of the same id
    for (auto& b : bb_) {
        b.valid = false;
        std::fill(std::begin(b.prof_len_batch), std::end(b.prof_len_batch), 0);
    }
    const int depth = (int)std::max<int64_t>(0, std::min<int64_t>(opt.lookahead, HMK_NBATCHBUF - 1));
    // SMs the side stream's bulk launches leave alone while the main stream works on a batch: one for the resolver,
    // the others for the small kernels around it (new founders, member check), which then never wait for a CTA of a
    // millisecond-long partner search to finish
    const int reserve = depth > 0 ? (int)std::max<int64_t>(1, std::min<int64_t>(opt.reserve, sm_count_ / 2)) : 0;
    int head = 0;
    fetch_ctl();
    while (h_ctl_->ncl < K_ && h_ctl_->unproc_alive > 0) {
        BatchBuf& cb = bb_[head];
        const int cur = h_ctl_->cur, ncl = h_ctl_->ncl;
        sec(SEC_P1_PARTNER);
        if (!cb.valid) stage_partner_search(cb, std::min(B, h_ctl_->unproc_alive), cur, nullptr, ncl, st_, st_);   // not prepared ahead
        else CK(cudaStreamWaitEvent(st_, cb.ready, 0));
        const int nq = cb.nq;
        const int32_t* d_qid = cb.qid.p;
        // A: clusters whose founder scores >= T (part 1 came with the batch; part 2 = the clusters created since), then
        // complete linkage over their members
        sec(SEC_P1_CLUSTER);
        if (ncl > cb.ncl_ahead) {
            plan_sms_ = (fast_ && reserve > 1) ? reserve - 1 : 0;      // while a prepared partner search holds the other SMs
            founder_hits(cb, cb.ncl_ahead, ncl, st_, d_sched_);
            plan_sms_ = 0;
        }
        check_members(cb, ncl, (int)capq);
        const int ib_stride = (nq + 3) & ~3, pd_stride = (nq * (int)opt.kb + 3) & ~3;
        const int nw = (nq + 31) / 32;
        HmkP1Batch pb{};
        pb.nq = nq; pb.batch_id = cb.batch_id; pb.qid = d_qid; pb.kb = (int)opt.kb;
        pb.bk_key = cb.bk_key.p; pb.bk_cnt = cb.bk_cnt.p; pb.bk_ovf = cb.bk_ovf.p;
        pb.capq = (int32_t)capq; pb.ac_cnt = d_ac_cnt_.p; pb.ac_slot = d_ac_slot_.p; pb.ac_score = d_ac_score_.p;
        pb.ac_full = d_ac_full_.p; pb.best = d_ac_best_.p;
        pb.hit_count = cb.hcount.p; pb.hit_cap = (unsigned int)cb.hit_cap;   // truncated hit lists: the resolver returns HMK_P1_GROWHITS
        pb.ib = cb.ib.p; pb.ib_stride = ib_stride; pb.ibm = cb.ibm.p; pb.ibm2 = cb.ibm2.p; pb.nw = nw;
        pb.pcand = cb.pcand.p;
        pb.pd = cb.pd.p; pb.pd_stride = pd_stride;
        sec(SEC_P1_RESOLVE);
        {
            const size_t fixed = hmk_resolve_fixed_bytes(nq, nw, (int)opt.kb) + 64;
            const size_t room = resolve_avail > fixed ? resolve_avail - fixed : 0;
            const int cache_entries = (int)std::min<size_t>(room / HMK_RESOLVE_CAND_BYTES, (size_t)nq * capq);
            const size_t smem = fixed + (size_t)cache_entries * HMK_RESOLVE_CAND_BYTES;
            smem_cfg_.ensure(hmk_p1_resolve_kernel, resolve_avail);
            hmk_p1_resolve_kernel<<<1, HMK_RESOLVE_THREADS, smem, st_>>>(state(), pb, cache_entries);
        }
        CK(cudaGetLastError());
        launches_++;
        // look ahead: the partner searches of the next `depth` batches (and everything else that does not depend on
        // the clustering state) run on the side streams while this batch is resolved; they are issued right behind
        // the resolver so that the resolver's CTA is placed first.  A batch only needs its predecessor's last query
        // id; whatever the batches before it consume in the meantime is filtered by the resolver's consumed set.
        // A resolver that throws the prepared batches away bumps ctl.discards, and their persistent launches stop.
        sec(SEC_P1_INTRA);   // host time of issuing the look-ahead
        for (int d = 1; d <= depth; d++) {
            BatchBuf& prev = bb_[(head + d - 1) % HMK_NBATCHBUF];
            BatchBuf& nb = bb_[(head + d) % HMK_NBATCHBUF];
            if (nb.valid) continue;
            if (!prev.valid || prev.nq != B || h_ctl_->unproc_alive < nq + (2 + d) * B) break;
            plan_sms_ = sm_count_ - reserve;
            // the tail stream takes the tails of the packed kernels' batches; the generic scalar kernel's dense tables are
            // long launches that slowed the main stream down at the tail stream's priority (7-30 mixed: 32.1 -> 33.6 ms),
            // so on that path a batch is staged behind the whole previous one, as on a single side stream
            const bool tail = fast_ || mixed_;
            CK(cudaStreamWaitEvent(st2_, tail ? prev.searched : prev.ready, 0));   // prev.qid is written on the stream that staged prev
            stage_partner_search(nb, B, cur, prev.qid.p + (prev.nq - 1), ncl, st2_, tail ? st3_ : st2_);
            plan_sms_ = 0;
        }
        sec(-1);
        fetch_ctl();
        const int st = h_ctl_->status;
#ifdef HMK_DEBUG
        if (getenv("HMK_DEBUG_BATCH"))
            fprintf(stderr, "batch %d nq %d: cur %d ncl %d unproc %d status %d steps %d\n", cb.batch_id, nq, h_ctl_->cur, h_ctl_->ncl,
                    h_ctl_->unproc_alive, st, h_ctl_->steps);
#endif
        if (st == HMK_P1_GROWHITS) {   // the state is untouched: redo the cluster search of this batch with a bigger buffer
            hit_cap_ = std::max(hit_cap_, (size_t)(uint32_t)h_ctl_->pad0 * 5 / 4 + 1024);
            cb.hit_cap = hit_cap_;
            cb.hits.reserve(cb.hit_cap);
            CK(cudaMemsetAsync(cb.hcount.p, 0, 4 * sizeof(unsigned int), st_));
            cb.ncl_ahead = 0;           // every founder again, on the main stream
            h_ctl_->status = HMK_P1_CONTINUE;
            continue;       // cb (and the batches prepared behind it) stay valid
        }
        stats.p1_batches++;
        cb.valid = false;
        if (st != HMK_P1_CONTINUE) drain_lookahead();    // the prepared batches do not follow this one after all
        if (st == HMK_P1_NPE) { error_step = h_ctl_->npe_step; stats.error_step = error_step; return HMK_ERR_NULL_CLUSTER; }
        if (st == HMK_P1_DONE) break;
        if (st == HMK_P1_GROW) {   // a query had more valid clusters than its arrays hold
            capq *= 2;
            d_ac_slot_.reserve((size_t)B * capq); d_ac_score_.reserve((size_t)B * capq); d_ac_full_.reserve((size_t)B * capq);
        }
        head = (head + 1) % HMK_NBATCHBUF;
    }
    drain_lookahead();      // phase 2 reads d_xcount_, which the look-ahead searches append to
    return HMK_OK;
}

// ---------------------------------------------------------------- phase 2
void Engine::phase2() {
    const int ncl = h_ctl_->ncl;
    sec(SEC_P2_SETUP);
    const int ns = compact_unassigned(d_singles_.p);
    stats.p2_queries = ns;
    if (ncl == 0 || ns == 0) { sec(-1); return; }
    hmk_index_of<<<(ns + 255) / 256, 256, 0, st_>>>(d_singles_.p, ns, d_sidx_.p);   // sequence id -> query index
    launches_++;
    size_t hit_cap = d_hits_.cap ? d_hits_.cap : (size_t)opt.hit_cap;
    d_hits_.reserve(hit_cap);
    size_t cand_cap = std::max<size_t>(1 << 20, (size_t)ns / 2);
    d_key_q_.reserve(cand_cap); d_cand_score_.reserve(cand_cap);
    cand_cap = std::min(d_key_q_.cap, d_cand_score_.cap);
    size_t ncand = 0;
    // candidate keys: two tight fields; 2^bits > count, so the all-ones padding keys of the multi-GPU exchange
    // stay above every real key
    auto bits_for = [](int x) { int b = 1; while ((1ll << b) <= (long long)x) b++; return b; };
    const int cbits = bits_for(ncl), qbits = bits_for(ns);
    CK(cudaMemsetAsync(d_counts_.p, 0, 4 * sizeof(unsigned int), st_));
    const int chunk = (int)std::max<int64_t>(1024, opt.p2_chunk);
    // this rank's share of the phase-2 queries (all of them on one GPU)
    const int my_lo = (int)((int64_t)ns * rank_ / world_), my_hi = (int)((int64_t)ns * (rank_ + 1) / world_);

    // founder filter + member check for one list of queries (`sch` NULL: generic kernel)
    auto run_list = [&](const int32_t* ids, int count, const HmkScheme* sch) {
        for (int c0 = 0; c0 < count;) {
            const int cn = std::min(chunk, count - c0);
            sec(SEC_P2_FILTER);
            CK(cudaMemsetAsync(d_counts_.p, 0, sizeof(unsigned int), st_));
            HmkBulkArgs a{};
            a.prof = d_fprof_.p; a.nq = ncl; a.kb = (int)opt.kb;
            a.packed = d_packed_.p; a.db_ids = ids + c0; a.db_begin = 0; a.ndb = cn;
            a.hits = d_hits_.p; a.hit_count = d_counts_.p; a.hit_cap = (unsigned int)hit_cap;
            if (sch && mixed_) { a.prof_cells = d_pcells_.p; a.prof_ops = d_pops_.p; }
            plan_bulk(HMK_MODE_EMIT, a, sch);
            launch_planned(HMK_MODE_EMIT, a, sch, d_cf_.p, 0, st_);
            sec(SEC_P2_CHECK);
            CK(cudaMemcpyAsync(h_scalars_, d_counts_.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st_));
            CK(cudaStreamSynchronize(st_));
            const size_t nh = (uint32_t)h_scalars_[0];
            if (nh > hit_cap) {   // redo this chunk with a bigger buffer
                hit_cap = nh * 5 / 4 + 1024;
                d_hits_.reserve(hit_cap);
                continue;
            }
            stats.p2_hits += (int64_t)nh;
            if (nh) {
                if (ncand + nh > cand_cap) {
                    size_t nc = std::max(cand_cap * 2, ncand + nh);
                    d_key_q_.grow_keep(nc, ncand, st_); d_cand_score_.grow_keep(nc, ncand, st_);
                    cand_cap = nc;
                }
                HmkCheckArgs c{};
                c.S = state(); c.hits = d_hits_.p; c.hit_count = d_counts_.p; c.hit_cap = (unsigned int)hit_cap;
                c.hit_t_is_query = 0; c.qids = nullptr; c.sidx = d_sidx_.p;
                c.cand_key_q = d_key_q_.p; c.cand_score = d_cand_score_.p;
                c.cand_count = d_counts_.p + 1; c.cand_cap = (unsigned int)cand_cap; c.linked = 0; c.cbits = cbits;
                c.packed = fast_scalar_ ? d_packed_.p : nullptr; c.L = max_len_; c.pair_parts = d_pairparts_.p;
                if (scalar12x3()) hmk_member_check<true><<<sm_count_ * 4, 256, 0, st_>>>(c);
                else hmk_member_check<false><<<sm_count_ * 4, 256, 0, st_>>>(c);
                CK(cudaGetLastError());
                launches_++;
                CK(cudaMemcpyAsync(h_scalars_ + 1, d_counts_.p + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, st_));
                CK(cudaStreamSynchronize(st_));
                ncand = (uint32_t)h_scalars_[1];
            }
            c0 += cn;
        }
    };

    // opt.reuse: every (founder, single) pair scoring >= T was already seen by a phase-1 partner search --
    // the founder was a query of some batch and the single a later singleton of that scan (or the other way
    // round for a phase-1 orphan), and S is symmetric.  The member check filters the kept hits down to those
    // pairs (and to scans of batches that were not re-done) instead of scoring founders x singles again.
    bool reused = false;
    if (reuse_) {
        CK(cudaMemcpyAsync(h_scalars_ + 10, d_xcount_.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        unsigned long long nx;
        memcpy(&nx, h_scalars_ + 10, sizeof(nx));
        xhit_want_ = (size_t)nx;
        reused = nx <= d_xhits_.cap;      // else: some hits were dropped -> separate founder pass below
        stats.xhits_kept = (int64_t)nx; stats.xhits_capacity = (int64_t)d_xhits_.cap;
        if (!reused) stats.flags |= HMK_FLAG_XHIT_OVERFLOW;
        if (world_ > 1) {                 // every rank must take the same path
            d_gcount_.reserve(world_ + 1);
            int32_t mine = reused ? 1 : 0;
            CK(cudaMemcpyAsync(d_gcount_.p + world_, &mine, sizeof(int32_t), cudaMemcpyHostToDevice, st_));
            allgather(d_gcount_.p + world_, d_gcount_.p, sizeof(int32_t), st_);
            std::vector<int32_t> all(world_);
            CK(cudaMemcpyAsync(all.data(), d_gcount_.p, sizeof(int32_t) * world_, cudaMemcpyDeviceToHost, st_));
            CK(cudaStreamSynchronize(st_));
            for (int r = 0; r < world_; r++) reused = reused && all[r] != 0;
        }
    }
    if (reused) stats.flags |= HMK_FLAG_P2_REUSED;
    if (reused) {
        sec(SEC_P2_CHECK);
        for (;;) {
            CK(cudaMemsetAsync(d_counts_.p + 1, 0, sizeof(unsigned int), st_));
            CK(cudaMemsetAsync(d_xcount_.p + 1, 0, sizeof(unsigned long long), st_));
            HmkCheckArgs c{};
            c.S = state(); c.hits = d_xhits_.p; c.hit_t_is_query = 2; c.xhit_count = d_xcount_.p; c.hit_valid = d_xcount_.p + 1;
            c.qids = nullptr; c.sidx = d_sidx_.p;
            c.cand_key_q = d_key_q_.p; c.cand_score = d_cand_score_.p;
            c.cand_count = d_counts_.p + 1; c.cand_cap = (unsigned int)cand_cap; c.linked = 0; c.cbits = cbits;
            c.packed = fast_scalar_ ? d_packed_.p : nullptr; c.L = max_len_; c.pair_parts = d_pairparts_.p;
            if (scalar12x3()) hmk_member_check<true><<<sm_count_ * 8, 256, 0, st_>>>(c);
            else hmk_member_check<false><<<sm_count_ * 8, 256, 0, st_>>>(c);
            CK(cudaGetLastError());
            launches_++;
            CK(cudaMemcpyAsync(h_scalars_ + 1, d_counts_.p + 1, sizeof(unsigned int), cudaMemcpyDeviceToHost, st_));
            CK(cudaMemcpyAsync(h_scalars_ + 10, d_xcount_.p + 1, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
            CK(cudaStreamSynchronize(st_));
            ncand = (uint32_t)h_scalars_[1];
            if (ncand <= cand_cap) break;
            const size_t nc = ncand + ncand / 16;      // candidates beyond the capacity were only counted: redo
            d_key_q_.reserve(nc); d_cand_score_.reserve(nc);
            cand_cap = std::min(d_key_q_.cap, d_cand_score_.cap);
        }
        unsigned long long nv;
        memcpy(&nv, h_scalars_ + 10, sizeof(nv));
        stats.p2_hits = (int64_t)nv;
    } else if (!mixed_) {
        // founder profiles (member side), built once: founders are fixed during phase 2
        if (fast_) {
            d_fprof_.reserve((size_t)ncl * sc_.prof_words);
            launch_profiles(HMK_PROF_MEMBER, d_cf_.p, ncl, d_fprof_.p, sc_, st_);
        }
        run_list(d_singles_.p + my_lo, my_hi - my_lo, fast_ ? &sc_ : nullptr);
    } else if (my_hi > my_lo) {
        // mixed lengths: split this rank's queries by length; per length, founder profiles for that
        // thread-side length and one packed-kernel pass
        const int my_n = my_hi - my_lo;
        d_sb_ids_.reserve((size_t)(HMK_MAXLEN + 1) * my_n); d_sb_cnt_.reserve(HMK_MAXLEN + 1);
        CK(cudaMemsetAsync(d_sb_cnt_.p, 0, sizeof(int32_t) * (HMK_MAXLEN + 1), st_));
        hmk_bucket_by_length<<<(my_n + 255) / 256, 256, 0, st_>>>(d_singles_.p + my_lo, my_n, d_off_.p, my_n, d_sb_ids_.p, d_sb_cnt_.p);
        launches_++;
        int32_t cnt[HMK_MAXLEN + 1];
        CK(cudaMemcpyAsync(cnt, d_sb_cnt_.p, sizeof(cnt), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        for (int L = 1; L <= HMK_MAXLEN; L++) {
            if (cnt[L] <= 0) continue;
            const HmkScheme sch = scheme_for(L);
            d_fprof_.reserve((size_t)ncl * sch.prof_words);
            launch_profiles(HMK_PROF_MEMBER, d_cf_.p, ncl, d_fprof_.p, sch, st_, d_pcells_.p, d_pops_.p);
            run_list(d_sb_ids_.p + (size_t)L * my_n, cnt[L], &sch);
        }
    }
    if (world_ > 1) {
        // candidate exchange: all-gather the per-rank candidate lists (padded to the longest; the
        // padding keys are ~0 and sort to the end)
        d_gcount_.reserve(world_ + 1);
        int32_t mine = (int32_t)ncand;
        CK(cudaMemcpyAsync(d_gcount_.p + world_, &mine, sizeof(int32_t), cudaMemcpyHostToDevice, st_));
        allgather(d_gcount_.p + world_, d_gcount_.p, sizeof(int32_t), st_);
        std::vector<int32_t> counts(world_);
        CK(cudaMemcpyAsync(counts.data(), d_gcount_.p, sizeof(int32_t) * world_, cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        size_t maxc = 0, total = 0;
        for (int r = 0; r < world_; r++) { maxc = std::max<size_t>(maxc, counts[r]); total += counts[r]; }
        if (maxc > 0) {
            if (maxc > cand_cap) {
                d_key_q_.grow_keep(maxc, ncand, st_); d_cand_score_.grow_keep(maxc, ncand, st_);
                cand_cap = maxc;
            }
            if (maxc > ncand) {
                CK(cudaMemsetAsync(d_key_q_.p + ncand, 0xff, sizeof(unsigned long long) * (maxc - ncand), st_));
                CK(cudaMemsetAsync(d_cand_score_.p + ncand, 0, sizeof(int32_t) * (maxc - ncand), st_));
            }
            DevBuf<unsigned long long>& gq = d_gq_;   // persistent: swapped with the local lists below
            DevBuf<int32_t>& gs = d_gs_;
            gq.reserve(maxc * world_); gs.reserve(maxc * world_);
            NK(NcclApi::get().GroupStart());
            allgather(d_key_q_.p, gq.p, sizeof(unsigned long long) * maxc, st_);
            allgather(d_cand_score_.p, gs.p, sizeof(int32_t) * maxc, st_);
            NK(NcclApi::get().GroupEnd());
            std::swap(d_key_q_.p, gq.p); std::swap(d_key_q_.cap, gq.cap);
            std::swap(d_cand_score_.p, gs.p); std::swap(d_cand_score_.cap, gs.cap);
        }
        ncand = total;
        ncand_padded_ = maxc * world_;
        cand_cap = std::min(d_key_q_.cap, d_cand_score_.cap);
    } else ncand_padded_ = ncand;
    stats.p2_candidates = (int64_t)ncand;
    sec(SEC_P2_SORT);
    if (ncand == 0) { sec(-1); return; }
    const int nc = (int)ncand;
    const int ncp = (int)ncand_padded_;   // >= nc: padded entries carry key ~0 and sort to the end
    // group by query: a stable radix sort over the query field only (the order of the candidates inside a query does not
    // matter: every decision is an arg-max under a strict total order)
    sort_pairs(d_key_q_.p, d_cand_score_.p, ncp, cbits, cbits + qbits);
    d_cq_c_.reserve(nc); d_cq_q_.reserve(nc); d_qstart_.reserve(ns + 2); d_cstart_.reserve(ncl + 2); d_ccount_.reserve(ncl + 1);
    hmk_split_keys_lo<<<(nc + 255) / 256, 256, 0, st_>>>(d_key_q_.p, nc, cbits, d_cq_c_.p, d_cq_q_.p);
    hmk_segment_starts<<<(ns + 1 + 255) / 256, 256, 0, st_>>>(d_key_q_.p, nc, ns, cbits, d_qstart_.p);
    CK(cudaGetLastError());
    launches_ += 2;
    // the pairs once more, grouped by cluster with ascending queries inside a cluster: a STABLE sort of the query-ordered
    // list by the cluster field alone (cbits bits, two radix passes); the clusters' offsets are cstart
    d_cc_q_.reserve(nc); d_cc_c_.reserve(nc);
    {
        size_t bytes = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, d_cq_c_.p, d_cc_c_.p, d_cq_q_.p, d_cc_q_.p, nc, 0, cbits, st_));
        d_cub_.reserve(bytes);
        CK(cub::DeviceRadixSort::SortPairs(d_cub_.p, bytes, d_cq_c_.p, d_cc_c_.p, d_cq_q_.p, d_cc_q_.p, nc, 0, cbits, st_));
        launches_ += 4;
    }
    d_cinfo_.reserve((size_t)ncl * HMK_CI);
    hmk_segment_starts_i32<<<(ncl + 1 + 255) / 256, 256, 0, st_>>>(d_cc_c_.p, nc, ncl, d_cstart_.p);
    hmk_p2_init_cinfo<<<(ncl + 255) / 256, 256, 0, st_>>>(ncl, d_cstart_.p, d_cinfo_.p);
    CK(cudaGetLastError());
    launches_ += 2;
    const int Wmax = (int)std::max<int64_t>(1, opt.p2_window);
    d_dyn_.reserve(nc); d_base_cl_.reserve(nc);
    d_a0_.reserve(ns); d_dirty_a_.reserve(ncl); d_stamp_.reserve(ns);
    d_work_.reserve(2 * (size_t)Wmax + HMK_P2_CTL + 2 * HMK_P2_CHG);
    CK(cudaMemsetAsync(d_a0_.p, 0xff, sizeof(int32_t) * (size_t)ns, st_));
    CK(cudaMemsetAsync(d_stamp_.p, 0xff, sizeof(int32_t) * (size_t)ns, st_));
    HmkP2 P{};
    P.S = state(); P.packed = fast_scalar_ ? d_packed_.p : nullptr; P.L = max_len_;
    P.ncl = ncl; P.ns = ns; P.singles = d_singles_.p; P.qstart = d_qstart_.p; P.cq_c = d_cq_c_.p; P.cq_q = d_cq_q_.p; P.cq_s = d_cand_score_.p;
    P.cstart = d_cstart_.p; P.cc_q = d_cc_q_.p;
    P.base_cl = d_base_cl_.p; P.cinfo = d_cinfo_.p; P.dyn = d_dyn_.p;
    P.a = d_a0_.p; P.dirty = d_dirty_a_.p; P.stamp = d_stamp_.p;
    P.wcap = Wmax; P.work = d_work_.p; P.ctl = d_work_.p + 2 * (size_t)Wmax; P.chg = P.ctl + HMK_P2_CTL;
    P.pair_parts = d_pairparts_.p;
#ifdef HMK_DEBUG
    d_p2tim_.reserve(64);
    P.tim = d_p2tim_.p;
#endif
    // the unrolled pair scorer: uniform length 12, max shift 3, lane-sized matrix entries
    const bool p2_fast = scalar12x3();
    const void* kernel = p2_fast ? (const void*)hmk_p2_window<true> : (const void*)hmk_p2_window<false>;
    int per_sm = 0;      // the cooperative grid must be resident as a whole
    if (p2_fast) CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hmk_p2_window<true>, 256, 0));
    else CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, hmk_p2_window<false>, 256, 0));
    if (per_sm < 1) throw CudaError("hmk_p2_window does not fit on an SM");
    // window size adapts to how hard the fixed point is: dense inputs (everything joins) need many
    // iterations per window unless few queries per cluster are in flight at a time.  The first windows are small: the
    // members they make final let the base pass reject most candidate pairs of every later window up front
    int W = std::min<int64_t>(Wmax, opt.p2_first > 0 ? opt.p2_first : std::max(1024, ncl / 4));
    int gen = 0;
    sec(SEC_P2_ITERATE);
    for (int qa = 0; qa < ns;) {
        const int qb = std::min(ns, qa + W);
        P.qa = qa; P.qb = qb; P.gen0 = gen; P.max_iters = qb - qa + 2;
        const int grid = std::max(1, std::min(per_sm * sm_count_, std::max((qb - qa + 7) / 8, (ncl + 255) / 256)));
        void* args[] = {(void*)&P};
        CK(cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(256), args, 0, st_));
        launches_++;
        CK(cudaMemcpyAsync(h_p2flags_, P.ctl, sizeof(int32_t) * HMK_P2_CTL, cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        const int iters = h_p2flags_[8];
        stats.p2_rounds += iters;
        gen += iters + 1;
#ifdef HMK_DEBUG
        if (getenv("HMK_DEBUG_P2")) {
            unsigned long long tm[64];
            CK(cudaMemcpy(tm, P.tim, sizeof(tm), cudaMemcpyDeviceToHost));
            fprintf(stderr, "p2 window [%d, %d) W %d grid %d: %d iterations; us: D0 %.0f", qa, qb, W, grid, iters, (tm[1] - tm[0]) * 1e-3);
            for (int k = 1; k < iters && 2 * k + 1 < 62; k++) fprintf(stderr, " | R %.0f D %.0f", (tm[2 * k] - tm[2 * k - 1]) * 1e-3, (tm[2 * k + 1] - tm[2 * k]) * 1e-3);
            fprintf(stderr, "\n");
        }
#endif
        qa = qb;
        if (iters > 8) W = std::min(Wmax, std::max(256, W / 2));
        else if (iters <= 5) W = std::min(Wmax, W * 2);
    }
    sec(-1);
}

// ---------------------------------------------------------------- run / download
int Engine::run() {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_run before hmk_upload");
    stats = hmk_stats{};
    stats.error_step = -1;
    error_step = -1;
    launches_ = bulk_launches_ = 0;
    reset_timing();
    for (double& v : section_ms) v = 0;
    ran_ = false;
    if (bad_residue_) return HMK_ERR_BAD_RESIDUE;
    stats.fast_path = fast_ ? 1 : (mixed_ ? 2 : 0);     // 2: packed kernel per length bucket (mixed lengths)
    stats.lane_bits = (fast_ || mixed_) ? (sc_.lane16 ? 16 : 8) : 32;
    if (!sym_) stats.flags |= HMK_FLAG_ASYMMETRIC;
    CK(cudaEventRecord(ev_a_, st_));
    if (n_) {
        hmk_fill_i32<<<sm_count_ * 2, 256, 0, st_>>>(d_slot_.p, -1, (size_t)n_);
        hmk_fill_i32<<<sm_count_ * 2, 256, 0, st_>>>(d_next_.p, -1, (size_t)n_);
        CK(cudaMemsetAsync(d_rank_.p, 0, sizeof(int32_t) * n_, st_));
        launches_ += 2;
    }
    HmkCtl c0{};
    c0.cur = 0; c0.ncl = 0; c0.unproc_alive = n_; c0.status = HMK_P1_CONTINUE; c0.npe_step = -1;
    *h_ctl_ = c0;
    CK(cudaMemcpyAsync(d_ctl_.p, h_ctl_, sizeof(HmkCtl), cudaMemcpyHostToDevice, st_));
    CK(cudaMemsetAsync(d_pairctr_.p, 0, 4 * sizeof(unsigned long long), st_));
    d_pairparts_.reserve(HMK_PAIR_SHARDS * 16);
    CK(cudaMemsetAsync(d_pairparts_.p, 0, HMK_PAIR_SHARDS * 16 * sizeof(unsigned long long), st_));
    // DataException "Shift too big" (ShiftedScorer.java:59-62): thrown by the first pair score
    // touching a sequence not longer than maxShift; step 0 of phase 1 scores every sequence.
    if (K_ > 0 && n_ >= 2 && X_ >= min_len_) return HMK_ERR_SHIFT_TOO_BIG;
    int rc = phase1();
    CK(cudaEventRecord(ev_b_, st_));
    if (rc == HMK_OK) phase2();
    if (rc == HMK_OK && n_) {
        sec(SEC_FINAL);
        hmk_finalize<<<(n_ + 255) / 256, 256, 0, st_>>>(n_, d_slot_.p, d_rank_.p, d_cf_.p, d_cluster_id_.p, d_member_rank_.p);
        CK(cudaGetLastError());
        launches_++;
        n_unassigned_ = compact_unassigned(d_singles_.p);
        sec(-1);
    }
    CK(cudaEventRecord(ev_c_, st_));
    fetch_ctl();
    unsigned long long pc[4] = {0, 0, 0, 0};
    std::vector<unsigned long long> parts(HMK_PAIR_SHARDS * 16);
    CK(cudaMemcpyAsync(pc, d_pairctr_.p, sizeof(pc), cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(parts.data(), d_pairparts_.p, parts.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    unsigned long long scalar_sharded = 0;
    for (int i = 0; i < HMK_PAIR_SHARDS; i++) scalar_sharded += parts[(size_t)i * 16];
    float ms1 = 0, ms2 = 0;
    CK(cudaEventElapsedTime(&ms1, ev_a_, ev_b_));
    CK(cudaEventElapsedTime(&ms2, ev_b_, ev_c_));
    stats.phase1_ms = ms1; stats.phase2_ms = ms2; stats.total_ms = ms1 + ms2;
    stats.bulk_kernel_ms = fold_timing();
    stats.bulk_pairs = (int64_t)pc[0];
    stats.scalar_pairs = h_ctl_->scalar_pairs + (int64_t)scalar_sharded;
#ifdef HMK_DEBUG
    if (getenv("HMK_DEBUG_TIMING"))
        fprintf(stderr, "resolver: %lld windows applied %lld lanes, %lld sequential steps\n", (long long)h_ctl_->cnt[0], (long long)h_ctl_->cnt[1],
                (long long)h_ctl_->cnt[2]);
    if (getenv("HMK_DEBUG_TIMING"))
        fprintf(stderr, "resolver cycles: staging %lld window(rest) %lld bpart %lld static %lld eval %lld apply %lld window(pick) %lld window(bounds) %lld\n", (long long)h_ctl_->dbg[0],
                (long long)h_ctl_->dbg[1], (long long)h_ctl_->dbg[2], (long long)h_ctl_->dbg[3], (long long)h_ctl_->dbg[4], (long long)h_ctl_->dbg[5], (long long)h_ctl_->dbg[7], (long long)h_ctl_->dbg[6]);
#endif
    if (min_len_ == max_len_) {
        stats.bulk_cells = stats.bulk_pairs * hmk_pair_cells(max_len_, max_len_, X_);
        stats.bulk_ops = stats.bulk_cells + stats.bulk_pairs * (2 * (int64_t)X_ + 1);
    } else if (mixed_) {   // counted by the packed-kernel launches (the small generic launches are not included)
        stats.bulk_cells = (int64_t)pc[1];
        stats.bulk_ops = (int64_t)pc[2];
    }
    stats.bulk_launches = bulk_launches_; stats.total_launches = launches_;
    stats.p1_steps = h_ctl_->steps; stats.p1_joins = h_ctl_->joins; stats.p1_new_clusters = h_ctl_->creates;
    stats.p1_orphans = h_ctl_->orphans; stats.p1_restarts = h_ctl_->restarts;
    if (rc == HMK_OK) {
        stats.p2_assigned = stats.p2_queries - n_unassigned_;
        ran_ = true;
    }
    return rc;
}

void Engine::download(hmk_greedy_out* out) {
    CK(cudaSetDevice(device_));
    if (!ran_) throw std::invalid_argument("hmk_download without a successful hmk_run");
    if (!out || (n_ > 0 && (!out->cluster_id || !out->member_rank || !out->result_order)))
        throw std::invalid_argument("hmk_download: null output array");
    const int ncl = h_ctl_->ncl;
    if (n_) {
        CK(cudaMemcpyAsync(out->cluster_id, d_cluster_id_.p, sizeof(int32_t) * n_, cudaMemcpyDeviceToHost, st_));
        CK(cudaMemcpyAsync(out->member_rank, d_member_rank_.p, sizeof(int32_t) * n_, cudaMemcpyDeviceToHost, st_));
        if (ncl) CK(cudaMemcpyAsync(out->result_order, d_cf_.p, sizeof(int32_t) * ncl, cudaMemcpyDeviceToHost, st_));
        if (n_unassigned_)
            CK(cudaMemcpyAsync(out->result_order + ncl, d_singles_.p, sizeof(int32_t) * n_unassigned_, cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
    }
    out->n_result = ncl + n_unassigned_;
    out->n_multi = ncl;
    out->error_step = -1;
}

void Engine::score_block(const int32_t* first, int32_t nf, const int32_t* second, int32_t ns, int32_t* scores) {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_score_block before hmk_upload");
    if (nf <= 0 || ns <= 0) return;
    DevBuf<int32_t> d_first, d_second, d_out;
    DevBuf<uint32_t> d_prof;
    const int chunk = 256;
    d_first.reserve(nf); d_second.reserve(chunk); d_out.reserve((size_t)chunk * nf);
    if (fast_) d_prof.reserve((size_t)chunk * sc_.prof_words);
    CK(cudaMemcpyAsync(d_first.p, first, sizeof(int32_t) * nf, cudaMemcpyHostToDevice, st_));
    std::vector<int32_t> tmp((size_t)chunk * nf);
    for (int s0 = 0; s0 < ns; s0 += chunk) {
        const int sn = std::min(chunk, ns - s0);
        CK(cudaMemcpyAsync(d_second.p, second + s0, sizeof(int32_t) * sn, cudaMemcpyHostToDevice, st_));
        HmkBulkArgs a = query_batch(d_second.p, sn, d_prof.p, (int)opt.kb);
        a.db_ids = d_first.p; a.db_begin = 0; a.ndb = nf;
        a.dense = d_out.p; a.dense_stride = nf;
        launch_bulk(HMK_MODE_DENSE, a, d_second.p, 1);
        CK(cudaMemcpyAsync(tmp.data(), d_out.p, sizeof(int32_t) * (size_t)sn * nf, cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        for (int b = 0; b < sn; b++)
            for (int a2 = 0; a2 < nf; a2++) scores[(size_t)a2 * ns + s0 + b] = tmp[(size_t)b * nf + a2];
    }
}

// One bulk launch with the context's scheme and options, for the kernel tests (hmk_bulk_probe).  Mode 0 is the partner
// search of stage_partner_search's uniform-length branch: only ids > qids[t] qualify, the per-stripe lists are merged
// with hmk_topk_merge and every qualifying hit is kept.  Mode 1 emits every hit.
void Engine::bulk_probe(int mode, const int32_t* qids, int32_t nq, const int32_t* db_ids, int32_t db_begin, int32_t ndb,
                        const uint8_t* clustered, uint64_t* keys, int32_t* cnt, int32_t* ovf, int32_t* hits, int64_t hit_cap,
                        int64_t* hit_count, int32_t* kernel) {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_bulk_probe before hmk_upload");
    if ((mode != 0 && mode != 1) || nq < 0 || ndb < 0 || hit_cap < 0 || (nq && !qids) || (nq && mode == 0 && (!keys || !cnt || !ovf)) ||
        (hit_cap && !hits) || !hit_count || !kernel)
        throw std::invalid_argument("hmk_bulk_probe: bad argument");
    for (int32_t t = 0; t < nq; t++)
        if (qids[t] < 0 || qids[t] >= n_) throw std::invalid_argument("hmk_bulk_probe: query id out of range");
    for (int32_t i = 0; i < ndb; i++) {
        const int64_t id = db_ids ? db_ids[i] : (int64_t)db_begin + i;
        if (id < 0 || id >= n_) throw std::invalid_argument("hmk_bulk_probe: thread-side id out of range");
    }
    const int kb = (int)opt.kb;
    DevBuf<int32_t> d_q, d_db, d_slot;
    BatchBuf bb;
    d_q.reserve(std::max(nq, 1));
    if (nq) CK(cudaMemcpyAsync(d_q.p, qids, sizeof(int32_t) * nq, cudaMemcpyHostToDevice, st_));
    if (fast_) bb.prof.reserve((size_t)std::max(nq, 1) * sc_.prof_words);
    HmkBulkArgs a = query_batch(d_q.p, nq, bb.prof.p, kb);
    a.db_begin = db_begin; a.ndb = ndb;
    if (db_ids) {
        d_db.reserve(std::max(ndb, 1));
        if (ndb) CK(cudaMemcpyAsync(d_db.p, db_ids, sizeof(int32_t) * ndb, cudaMemcpyHostToDevice, st_));
        a.db_ids = d_db.p; a.db_begin = 0;
    }
    std::vector<int32_t> h_slot;
    if (clustered) {
        h_slot.resize(std::max(n_, 1));
        for (int i = 0; i < n_; i++) h_slot[i] = clustered[i] ? 0 : -1;
        d_slot.reserve(h_slot.size());
        CK(cudaMemcpyAsync(d_slot.p, h_slot.data(), sizeof(int32_t) * h_slot.size(), cudaMemcpyHostToDevice, st_));
        a.slot = d_slot.p;
    }
    DevBuf<int4> d_hits;
    DevBuf<unsigned long long> d_count;
    d_hits.reserve(std::max<int64_t>(hit_cap, 1));
    d_count.reserve(2);
    CK(cudaMemsetAsync(d_count.p, 0, 2 * sizeof(unsigned long long), st_));
    HmkBulkArgs p = a;
    BulkKernel k{-1, -1, 0, nullptr};
    if (mode == 0) {
        a.q_minid = d_q.p;
        a.tierank = identity_rank_ ? nullptr : d_tierank_.p;
        bb.gmin.reserve(std::max(nq, 1));
        CK(cudaMemsetAsync(bb.gmin.p, 0, sizeof(unsigned long long) * std::max(nq, 1), st_));
        a.tk_gmin = bb.gmin.p;
        a.xhits = d_hits.p; a.xhit_count = d_count.p; a.xhit_cap = (unsigned long long)hit_cap;
        p = launch_bulk(HMK_MODE_TOPK, a, d_q.p, 1, st_, &bb, nullptr, &k);
        bb.bk_key.reserve((size_t)std::max(nq, 1) * kb); bb.bk_cnt.reserve(std::max(nq, 1)); bb.bk_ovf.reserve(std::max(nq, 1));
        if (nq && ndb) {
            merge_topk(nq, p.nstripes, kb, bb.tk_key.p, bb.tk_cnt.p, bb.tk_ovf.p, bb, st_, p.sched ? p.sched + p.nqt : nullptr, p.qt);
            CK(cudaMemcpyAsync(keys, bb.bk_key.p, sizeof(uint64_t) * nq * kb, cudaMemcpyDeviceToHost, st_));
            CK(cudaMemcpyAsync(cnt, bb.bk_cnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
            CK(cudaMemcpyAsync(ovf, bb.bk_ovf.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
        } else {
            for (int t = 0; t < nq; t++) { cnt[t] = 0; ovf[t] = 0; }
        }
    } else {
        a.hits = d_hits.p; a.hit_count = reinterpret_cast<unsigned int*>(d_count.p);
        a.hit_cap = (unsigned int)std::min<int64_t>(hit_cap, UINT32_MAX);
        p = launch_bulk(HMK_MODE_EMIT, a, d_q.p, 1, st_, nullptr, nullptr, &k);
    }
    CK(cudaMemcpyAsync(h_scalars_, d_count.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    unsigned long long total;
    if (mode == 0) total = *reinterpret_cast<unsigned long long*>(h_scalars_);
    else total = *reinterpret_cast<unsigned int*>(h_scalars_);
    *hit_count = (int64_t)total;
    copy_hit_triples(d_hits.p, (size_t)std::min<unsigned long long>(total, (unsigned long long)hit_cap), hits);
    report_kernel(k, k.fn && p.sched, kernel);
}

// Phase 1's per-batch work on a clustering state given by the caller (hmk_batch_probe): the state goes into the
// context's own buffers, then stage_partner_search and check_members run as phase1 calls them, on the first batch
// buffer.  Whatever of this a run reads, run() and phase1() set again: the clustering state, the control block, the
// batch buffers' validity and profile ids, the batch counter, the hit capacity and the pair counters.
void Engine::batch_probe(const int32_t* member_off, const int32_t* members, int32_t ncl, int32_t cur, int32_t nq, int32_t capq,
                         int32_t tail_stream, hmk_batch_probe_out* out) {
    CK(cudaSetDevice(device_));
    if (!uploaded_ || n_ <= 0 || bad_residue_) throw std::invalid_argument("hmk_batch_probe needs an uploaded, valid input");
    if (!out || ncl < 0 || ncl > K_ || (ncl && (!member_off || !members)) || cur < 0 || cur > n_ || nq < 1 ||
        nq > HMK_MAXBATCH || capq < 0 || (out->fhit_cap && !out->fhits) || out->fhit_cap < 0 || !out->qid || !out->bk_key ||
        !out->bk_cnt || !out->bk_ovf || !out->ib || !out->ibm || !out->ibm2 || !out->pcand || !out->pd || !out->ac_cnt ||
        !out->ac_slot || !out->ac_score || !out->ac_best)
        throw std::invalid_argument("hmk_batch_probe: bad argument");
    if (X_ >= min_len_) throw std::invalid_argument("hmk_batch_probe: max shift not below the shortest length");
    // ---- the clustering state
    std::vector<int32_t> ab(n_), slot(n_, -1), rank(n_, 0), next(n_, -1), cf(ncl), cs(ncl), cc(ncl), ct(ncl);
    CK(cudaMemcpy(ab.data(), d_ab_.p, sizeof(int32_t) * n_, cudaMemcpyDeviceToHost));
    for (int c = 0; c < ncl; c++) {
        const int32_t b = member_off[c], e = member_off[c + 1];
        if (b < 0 || e <= b) throw std::invalid_argument("hmk_batch_probe: member_off must rise, every cluster non-empty");
        uint32_t size = 0;      // Cluster.size(): Java int sum of the abundances
        for (int32_t i = b; i < e; i++) {
            const int32_t m = members[i];
            if (m < 0 || m >= n_ || slot[m] >= 0) throw std::invalid_argument("hmk_batch_probe: member id out of range or repeated");
            slot[m] = c; rank[m] = i - b;
            if (i + 1 < e) next[m] = members[i + 1];
            size += (uint32_t)ab[m];
        }
        cf[c] = members[b]; cs[c] = (int32_t)size; cc[c] = e - b; ct[c] = members[e - 1];
    }
    int32_t unproc = 0;
    for (int i = cur; i < n_; i++) unproc += slot[i] < 0;
    if (unproc == 0) throw std::invalid_argument("hmk_batch_probe: no singleton at or after cur");
    CK(cudaMemcpyAsync(d_slot_.p, slot.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(d_rank_.p, rank.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
    CK(cudaMemcpyAsync(d_next_.p, next.data(), sizeof(int32_t) * n_, cudaMemcpyHostToDevice, st_));
    if (ncl) {
        CK(cudaMemcpyAsync(d_cf_.p, cf.data(), sizeof(int32_t) * ncl, cudaMemcpyHostToDevice, st_));
        CK(cudaMemcpyAsync(d_cs_.p, cs.data(), sizeof(int32_t) * ncl, cudaMemcpyHostToDevice, st_));
        CK(cudaMemcpyAsync(d_cc_.p, cc.data(), sizeof(int32_t) * ncl, cudaMemcpyHostToDevice, st_));
        CK(cudaMemcpyAsync(d_ct_.p, ct.data(), sizeof(int32_t) * ncl, cudaMemcpyHostToDevice, st_));
    }
    HmkCtl c0{};
    c0.cur = cur; c0.ncl = ncl; c0.unproc_alive = unproc; c0.status = HMK_P1_CONTINUE; c0.npe_step = -1;
    *h_ctl_ = c0;
    CK(cudaMemcpyAsync(d_ctl_.p, h_ctl_, sizeof(HmkCtl), cudaMemcpyHostToDevice, st_));
    d_pairparts_.reserve(HMK_PAIR_SHARDS * 16);
    CK(cudaStreamSynchronize(st_));      // the side streams start from here
    // ---- one batch, as phase1 runs it (no kept hits for phase 2, every SM for the bulk launches)
    const int kb = (int)opt.kb;
    const int cq = capq > 0 ? capq : (int)std::max<int64_t>(1, opt.capq);
    nq = std::min(nq, unproc);
    reuse_ = false;
    plan_sms_ = 0;
    hit_cap_ = (size_t)opt.hit_cap;
    d_ac_cnt_.reserve(nq); d_ac_slot_.reserve((size_t)nq * cq); d_ac_score_.reserve((size_t)nq * cq);
    d_ac_full_.reserve((size_t)nq * cq); d_ac_best_.reserve(nq);
    LaunchLog log;
    struct Unset { LaunchLog*& p; ~Unset() { p = nullptr; } } unset{launch_log_};
    launch_log_ = &log;
    BatchBuf& bb = bb_[0];
    if (tail_stream) stage_partner_search(bb, nq, cur, nullptr, ncl, st2_, st3_);
    else stage_partner_search(bb, nq, cur, nullptr, ncl, st_, st_);
    bb.valid = false;
    CK(cudaStreamWaitEvent(st_, bb.ready, 0));
    check_members(bb, ncl, cq);
    // ---- results
    const int nw = (nq + 31) / 32, ib_stride = (nq + 3) & ~3, pd_stride = (nq * kb + 3) & ~3;
    std::vector<int32_t> ib((size_t)nq * ib_stride), pd((size_t)nq * pd_stride);
    std::vector<int4> best(nq);
    unsigned int hcount = 0;
    CK(cudaMemcpyAsync(out->qid, bb.qid.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->bk_key, bb.bk_key.p, sizeof(uint64_t) * nq * kb, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->bk_cnt, bb.bk_cnt.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->bk_ovf, bb.bk_ovf.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(ib.data(), bb.ib.p, sizeof(int32_t) * ib.size(), cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->ibm, bb.ibm.p, sizeof(uint32_t) * nq * nw, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->ibm2, bb.ibm2.p, sizeof(uint32_t) * nq * nw, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->pcand, bb.pcand.p, sizeof(int32_t) * nq * kb, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(pd.data(), bb.pd.p, sizeof(int32_t) * pd.size(), cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(&hcount, bb.hcount.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->ac_cnt, d_ac_cnt_.p, sizeof(int32_t) * nq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->ac_slot, d_ac_slot_.p, sizeof(int32_t) * nq * cq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->ac_score, d_ac_score_.p, sizeof(int32_t) * nq * cq, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(best.data(), d_ac_best_.p, sizeof(int4) * nq, cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    out->nq_out = nq;
    for (int b = 0; b < nq; b++) {
        std::copy_n(&ib[(size_t)b * ib_stride], nq, out->ib + (size_t)b * nq);
        std::copy_n(&pd[(size_t)b * pd_stride], nq * kb, out->pd + (size_t)b * nq * kb);
        const int4 r = best[b];
        out->ac_best[4 * b] = r.x; out->ac_best[4 * b + 1] = r.y; out->ac_best[4 * b + 2] = r.z; out->ac_best[4 * b + 3] = r.w;
    }
    out->fhit_count = hcount;
    copy_hit_triples(bb.hits.p, std::min<size_t>({(size_t)hcount, bb.hit_cap, (size_t)out->fhit_cap}), out->fhits);
    int32_t* kr = out->kernel;
    report_kernel(log.last[HMK_MODE_TOPK], log.persistent, kr);
    kr[5] = log.count[HMK_MODE_TOPK];
    kr[6] = log.last[HMK_MODE_DENSE].kind;
    kr[7] = log.count[HMK_MODE_DENSE];
    kr[8] = log.last[HMK_MODE_EMIT].kind;
    kr[9] = log.count[HMK_MODE_EMIT];
    kr[10] = log.member_check;
}

// ---------------------------------------------------------------- exact complete-linkage clustering (SURVEY.md 8f N1)
// ClinkageSequenceClusterer.cluster (ClinkageSequenceClusterer.java:43-124).  n <= opt.clinkage_dense_max: dense pair
// scores from the bulk kernel, nearest-neighbour chain in hmk_clinkage_chain.  Larger n: the entries scoring >= T only
// (clinkage_rows), chain in hmk_clinkage_chain_sparse -- the same result.  Returns the status; fills `out` on success.
int Engine::clinkage(const hmk_greedy_in* in, hmk_greedy_out* out) {
    upload(in);
    stats = hmk_stats{};
    stats.error_step = -1;
    status_msg.clear();
    launches_ = bulk_launches_ = 0;
    reset_timing();
    for (double& v : section_ms) v = 0;
    if (!out || (n_ > 0 && (!out->cluster_id || !out->member_rank || !out->result_order)))
        throw std::invalid_argument("hmk_clinkage_cluster: null output array");
    out->n_result = 0; out->n_multi = 0; out->error_step = -1;
    if (n_ == 0)      // activeClusters.iterator().next() on an empty set (ClinkageSequenceClusterer.java:116)
        throw std::invalid_argument("hmk_clinkage_cluster: no sequences (the reference throws NoSuchElementException)");
    if (bad_residue_) return HMK_ERR_BAD_RESIDUE;
    if (!sym_) return HMK_STATUS_UNSUPPORTED;          // CachedClusterScorer keeps one value per unordered pair of clusters
    if (n_ >= 2 && X_ >= min_len_) return HMK_ERR_SHIFT_TOO_BIG;
    const bool sparse = n_ > opt.clinkage_dense_max;
    const size_t n = (size_t)n_;
    CK(cudaEventRecord(ev_a_, st_));
    sec(0);
    int threads = HMK_CL_THREADS;
    if (!sparse) {   // D[q][i] = sequenceScore(seq i, seq q) (symmetric), one batch of profiles at a time
        d_clD_.reserve(n * n);
        const int32_t* ids = identity_ids();
        const int chunk = HMK_MAXBATCH;
        if (fast_) d_prof_.reserve((size_t)chunk * sc_.prof_words);
        for (int q0 = 0; q0 < n_; q0 += chunk) {
            const int sn = std::min(chunk, n_ - q0);
            HmkBulkArgs a = query_batch(ids + q0, sn, d_prof_.p, (int)opt.kb);
            a.db_ids = nullptr; a.db_begin = 0; a.ndb = n_;
            a.dense = d_clD_.p + (size_t)q0 * n; a.dense_stride = n_;
            launch_bulk(HMK_MODE_DENSE, a, ids + q0, 1);
        }
        hmk_clinkage_threshold<<<sm_count_ * 8, 256, 0, st_>>>(d_clD_.p, n * n, T_);
        stats.bulk_pairs = (int64_t)n * (int64_t)n;
    } else {
        const int rc = clinkage_rows(&threads);
        if (rc) { sec(-1); return rc; }
    }
    sec(2);
    int acap = 16;
    while (n_ > (int)(acap * 0.75f)) acap *= 2;          // java.util.HashMap: doubled whenever size > 0.75 x capacity
    int rcap = 16;
    while ((int)(rcap * 0.75f) < n_) rcap *= 2;
    const size_t maxid = 2 * n + 3;
    d_cli_.reserve((size_t)acap * 2 + maxid * 4 + n * 8 + 1 + (size_t)rcap * 4 + 8);
    HmkClinkage C{};
    int32_t* p = d_cli_.p;
    C.n = n_; C.T = T_; C.ab = d_ab_.p; C.acap = acap;
    if (sparse) { C.row_off = d_cloff_.p; C.rows = d_clrows_.p; C.twin = d_cltwin_.p; }
    else C.D = d_clD_.p;
    C.a_head = p; p += acap; C.a_tail = p; p += acap;
    C.a_next = p; p += maxid; C.a_prev = p; p += maxid; C.slot_of = p; p += maxid; C.r_next = p; p += maxid;
    C.id_of = p; p += n; C.size_of = p; p += n; C.mhead = p; p += n; C.mtail = p; p += n; C.mnext = p; p += n;
    C.stack = p; p += n + 1; C.ready = p; p += n; C.result_order = p; p += n;
    C.r_head = p; p += (size_t)rcap * 4; C.rcap_max = rcap;
    C.out_scalars = p; p += 8;
    C.cluster_id = d_cluster_id_.p; C.member_rank = d_member_rank_.p;
    if (sparse) hmk_clinkage_chain_sparse<<<1, threads, 0, st_>>>(C);
    else hmk_clinkage_chain<<<1, HMK_CL_THREADS, 0, st_>>>(C);
    CK(cudaGetLastError());
    launches_ += 2;
    sec(-1);
    CK(cudaEventRecord(ev_c_, st_));
    int32_t sc[8];
    CK(cudaMemcpyAsync(sc, C.out_scalars, sizeof(sc), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, ev_a_, ev_c_));
    stats.total_ms = ms; stats.phase1_ms = ms;
    stats.bulk_kernel_ms = fold_timing();
    stats.bulk_launches = bulk_launches_; stats.total_launches = launches_;
    stats.p1_steps = sc[3];                          // nearest-neighbour searches
    stats.fast_path = fast_ ? 1 : 0;
    stats.lane_bits = fast_ ? (sc_.lane16 ? 16 : 8) : 32;
    if (sc[2]) return HMK_STATUS_UNSUPPORTED;         // a HashMap bin reached the tree threshold
    CK(cudaMemcpyAsync(out->cluster_id, d_cluster_id_.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->member_rank, d_member_rank_.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(out->result_order, C.result_order, sizeof(int32_t) * sc[0], cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    out->n_result = sc[0];
    out->n_multi = sc[1];
    return HMK_OK;
}

// Sparse complete-linkage scores: every pair of the upper triangle scoring >= T, found by the bulk kernel's EMIT mode one
// query batch at a time (queries [q0, q0 + B) against the thread-side ids [q0, n); pairs with id <= query are dropped),
// stored as rows of BOTH directions with int64 offsets, each row sorted by neighbour slot, plus the twin index of every
// entry.  Two scoring passes: the first counts the entries per row (a batch whose hits overflow the buffer is re-run with
// a bigger one), the second scatters them -- the pair scores are cheap next to the chain, device memory is not.  Before
// the rows are allocated their bytes are compared with the free device memory: HMK_STATUS_UNSUPPORTED with the count of
// valid pairs in status_msg when they do not fit.  *threads = block size of the chain kernel.
int Engine::clinkage_rows(int* threads) {
    const int n = n_;
    d_clD_.release();     // the dense matrix of an earlier call on this context
    const int chunk = HMK_MAXBATCH;
    if (fast_) d_prof_.reserve((size_t)chunk * sc_.prof_words);
    d_cldeg_.reserve((size_t)n + 1); d_cloff_.reserve((size_t)n + 1);
    CK(cudaMemsetAsync(d_cldeg_.p, 0, sizeof(unsigned long long) * ((size_t)n + 1), st_));
    d_hits_.reserve(std::max<size_t>(d_hits_.cap, (size_t)1 << 20));
    const int grid = sm_count_ * 4;
    for (int q0 = 0; q0 < n; q0 += chunk) {          // pass 1: entries per row
        emit_hits(q0, std::min(chunk, n - q0), 0);
        hmk_cl_count_hits<<<grid, 256, 0, st_>>>(d_hits_.p, d_counts_.p, (unsigned int)d_hits_.cap, q0, n, d_cldeg_.p);
        CK(cudaGetLastError());
        launches_++;
    }
    size_t bytes = 0;
    unsigned long long* off = reinterpret_cast<unsigned long long*>(d_cloff_.p);
    CK(cub::DeviceScan::ExclusiveSum(nullptr, bytes, d_cldeg_.p, off, n + 1, st_));
    d_cub_.reserve(bytes);
    CK(cub::DeviceScan::ExclusiveSum(d_cub_.p, bytes, d_cldeg_.p, off, n + 1, st_));
    std::vector<int64_t> h_off((size_t)n + 1);
    CK(cudaMemcpyAsync(h_off.data(), d_cloff_.p, sizeof(int64_t) * ((size_t)n + 1), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    const size_t E = (size_t)h_off[n];
    size_t maxrow = 0;
    for (int i = 0; i < n; i++) maxrow = std::max<size_t>(maxrow, (size_t)(h_off[i + 1] - h_off[i]));
    // the rows are sorted in groups of consecutive rows (cub's segmented sort counts items in int)
    const size_t group_cap = std::max<size_t>(maxrow, std::min<size_t>(E, (size_t)1 << 28));
    size_t sort_bytes = 0;
    {
        cub::DoubleBuffer<uint64_t> db(nullptr, nullptr);
        CK(cub::DeviceSegmentedSort::SortKeys(nullptr, sort_bytes, db, (int)std::max<size_t>(group_cap, 1), n, d_clrel_.p,
                                              d_clrel_.p + 1, st_));
    }
    const size_t need = E * (sizeof(uint64_t) + sizeof(int32_t)) + group_cap * sizeof(uint64_t) + sort_bytes +
                        ((size_t)n + 1) * sizeof(int32_t);
    size_t free_b = 0, total_b = 0;
    CK(cudaMemGetInfo(&free_b, &total_b));
    const size_t have = free_b + d_clrows_.cap * sizeof(uint64_t) + d_cltwin_.cap * sizeof(int32_t) +
                        d_clalt_.cap * sizeof(uint64_t) + d_cub_.cap + d_clrel_.cap * sizeof(int32_t);
    stats.xhits_kept = (int64_t)E;
    if (need > have) {
        status_msg = "exact complete-linkage clustering of " + std::to_string(n) + " sequences: " + std::to_string(E / 2) +
                     " valid pairs (" + std::to_string(E) + " directed entries) need " + std::to_string(need) +
                     " bytes of device memory, " + std::to_string(have) + " are available";
        return HMK_STATUS_UNSUPPORTED;
    }
    sec(1);
    d_clrows_.reserve(E); d_cltwin_.reserve(E); d_clalt_.reserve(group_cap); d_cub_.reserve(sort_bytes);
    d_clrel_.reserve((size_t)n + 1);
    stats.xhits_capacity = (int64_t)d_clrows_.cap;
    CK(cudaMemsetAsync(d_cldeg_.p, 0, sizeof(unsigned long long) * ((size_t)n + 1), st_));
    for (int q0 = 0; q0 < n; q0 += chunk) {          // pass 2: the same hits (the buffer already fits every batch), scattered
        emit_hits(q0, std::min(chunk, n - q0), d_hits_.cap, false);
        hmk_cl_scatter_hits<<<grid, 256, 0, st_>>>(d_hits_.p, d_counts_.p, (unsigned int)d_hits_.cap, q0, n, d_cloff_.p,
                                                   d_cldeg_.p, d_clrows_.p);
        CK(cudaGetLastError());
        launches_++;
    }
    for (int r0 = 0; r0 < n;) {                      // rows sorted by neighbour slot (slots are unique in a row)
        int r1 = r0 + 1;
        while (r1 < n && (size_t)(h_off[r1 + 1] - h_off[r0]) <= group_cap) r1++;
        const size_t items = (size_t)(h_off[r1] - h_off[r0]);
        if (items > 1) {
            hmk_cl_rel_offsets<<<(r1 - r0 + 256) / 256, 256, 0, st_>>>(d_cloff_.p, r0, r1 - r0, d_clrel_.p);
            CK(cudaGetLastError());
            uint64_t* base = d_clrows_.p + h_off[r0];
            cub::DoubleBuffer<uint64_t> db(base, d_clalt_.p);
            size_t b2 = d_cub_.cap;
            CK(cub::DeviceSegmentedSort::SortKeys(d_cub_.p, b2, db, (int)items, r1 - r0, d_clrel_.p, d_clrel_.p + 1, st_));
            if (db.Current() != base)
                CK(cudaMemcpyAsync(base, db.Current(), sizeof(uint64_t) * items, cudaMemcpyDeviceToDevice, st_));
            launches_ += 2;
        }
        r0 = r1;
    }
    if (E) {
        hmk_cl_twins<<<sm_count_ * 8, 256, 0, st_>>>(d_cloff_.p, d_clrows_.p, n, d_cltwin_.p);
        CK(cudaGetLastError());
        launches_++;
    }
    // a step passes over one row a few times and ends with barriers: a block about as wide as the mean row (rows only
    // shrink), at least 128 threads
    int t = 128;
    while (t < HMK_CL_THREADS && (size_t)t * n < E) t *= 2;
    *threads = opt.clinkage_threads > 0 ? (int)opt.clinkage_threads : t;
    return HMK_OK;
}

// One query batch of the upper-triangle pair search (clinkage_rows, the score graph): the bulk kernel's EMIT mode scores
// the queries [q0, q0 + sn) (profiles, seq2) against the thread-side ids [q0, n) (seq1)
// and writes every pair scoring >= T to d_hits_ as (query - q0, thread-side id, score); pairs with id <= query are among
// them and are the caller's to drop.  Returns the hit count (count = false: returns 0 without waiting for the batch).
// cap == 0: a batch whose hits overflow d_hits_ is re-run with a bigger buffer; else at most cap (<= d_hits_.cap) hits
// are stored, and a count above cap tells the caller to split the batch.
size_t Engine::emit_hits(int q0, int sn, size_t cap, bool count) {
    const int32_t* ids = identity_ids() + q0;
    for (;;) {
        const size_t c = cap ? cap : d_hits_.cap;
        CK(cudaMemsetAsync(d_counts_.p, 0, sizeof(unsigned int), st_));
        HmkBulkArgs a = query_batch(ids, sn, d_prof_.p, (int)opt.kb);
        a.db_ids = nullptr; a.db_begin = q0; a.ndb = n_ - q0;
        a.hits = d_hits_.p; a.hit_count = d_counts_.p; a.hit_cap = (unsigned int)std::min<size_t>(c, UINT32_MAX);
        launch_bulk(HMK_MODE_EMIT, a, ids, 1);
        stats.bulk_pairs += (int64_t)sn * (n_ - q0);
        if (!count) return 0;
        CK(cudaMemcpyAsync(h_scalars_, d_counts_.p, sizeof(unsigned int), cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        const size_t cnt = *reinterpret_cast<unsigned int*>(h_scalars_);
        if (cap || cnt <= d_hits_.cap) return cnt;
        d_hits_.reserve(cnt + cnt / 4);          // the hit counter kept counting past the capacity: re-run the batch
    }
}

// hmk_score_shift over `cap` pairs (graph: the first min(*count, cap) EMIT hits of the batch at q0)
void Engine::shift_pass(const int4* pairs, const unsigned int* count, unsigned int cap, int q0, int jbits,
                        unsigned long long* keys, unsigned long long* vals, unsigned int* kept, int32_t* score, int32_t* shift) {
    HmkShiftArgs s{};
    s.pairs = pairs; s.count = count; s.cap = cap; s.q0 = q0; s.jbits = jbits;
    s.res = d_res_.p; s.off = d_off_.p; s.M = d_M_.p; s.X = X_; s.P = P_; s.n = n_;
    s.keys = keys; s.vals = vals; s.kept = kept; s.score = score; s.shift = shift;
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(sm_count_ * 8, ((int64_t)cap + 255) / 256));
    hmk_score_shift<<<grid, 256, 0, st_>>>(s);
    CK(cudaGetLastError());
    launches_++;
}

// ---------------------------------------------------------------- score graph (hmk_score_graph)
static_assert(sizeof(hmk_graph_edge) == sizeof(int4), "hmk_graph_edge is copied from the int4 edges of hmk_graph_edges");
// Every pair i < j with scoreWithShift(seq1 = j, seq2 = i) >= T, as (i, j, score, shift) ordered by i, then j: the
// upper-triangle pairs emit_hits finds (the same pairs clinkage_rows keeps), the shift of each from hmk_score_shift, and
// a radix sort of the batch on (i, j).  Device memory is bounded by one batch: a batch whose hits overflow the buffer
// (at least n entries, so that one query always fits) is re-run with fewer queries.
void Engine::graph_batch(int q0) {
    GraphBatch& g = graph_;
    g.valid = false;
    const int n = n_;
    const size_t H = std::min<size_t>(UINT32_MAX, std::max<size_t>(opt.graph_cap > 0 ? (size_t)opt.graph_cap : (size_t)1 << 22, (size_t)n));
    // every buffer at its bound before the timed passes: no allocation inside a batch
    d_hits_.reserve(H);
    if (fast_) d_prof_.reserve((size_t)HMK_MAXBATCH * sc_.prof_words);
    for (auto& b : g.key) b.reserve(H);
    for (auto& b : g.val) b.reserve(H);
    g.kept.reserve(HMK_MAXBATCH + 1);
    g.edges.reserve(H);
    {
        cub::DoubleBuffer<unsigned long long> dk(g.key[0].p, g.key[1].p), dv(g.val[0].p, g.val[1].p);
        size_t bytes = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, (int)H, 0, 64, st_));
        d_cub_.reserve(bytes);
    }
    int sn = std::min(g.sn, n - q0);
    sec(0);
    for (size_t cnt; (cnt = emit_hits(q0, sn, H)) > H;) {
        if (sn == 1) throw std::logic_error("score graph: one query row exceeds the hit buffer");
        sn = std::max(1, std::min(sn / 2, (int)((double)sn * H / cnt)));
    }
    sec(1);
    int jbits = 1, tbits = 1;
    while (((int64_t)1 << jbits) < n) jbits++;
    while ((1 << tbits) < sn) tbits++;
    CK(cudaMemsetAsync(g.kept.p, 0, sizeof(unsigned int) * (sn + 1), st_));
    shift_pass(d_hits_.p, d_counts_.p, (unsigned int)H, q0, jbits, g.key[0].p, g.val[0].p, g.kept.p, nullptr, nullptr);
    std::vector<unsigned int> kept(sn + 1);
    CK(cudaMemcpyAsync(kept.data(), g.kept.p, sizeof(unsigned int) * (sn + 1), cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    const unsigned int m = kept[0];
    if (m > 1) {
        cub::DoubleBuffer<unsigned long long> dk(g.key[0].p, g.key[1].p), dv(g.val[0].p, g.val[1].p);
        size_t bytes = 0;
        CK(cub::DeviceRadixSort::SortPairs(nullptr, bytes, dk, dv, (int)m, 0, jbits + tbits, st_));
        d_cub_.reserve(bytes);      // within the bound reserved above
        CK(cub::DeviceRadixSort::SortPairs(d_cub_.p, bytes, dk, dv, (int)m, 0, jbits + tbits, st_));
        launches_ += 4;
        hmk_graph_edges<<<std::min<int64_t>(sm_count_ * 8, (m + 255) / 256), 256, 0, st_>>>(dk.Current(), dv.Current(), m, q0, jbits, g.edges.p);
    } else if (m == 1) {
        hmk_graph_edges<<<1, 32, 0, st_>>>(g.key[0].p, g.val[0].p, m, q0, jbits, g.edges.p);
    }
    CK(cudaGetLastError());
    sec(-1);
    fold_timing();
    g.row_off.assign(sn + 1, 0);
    for (int t = 0; t < sn; t++) g.row_off[t + 1] = g.row_off[t] + kept[t + 1];
    g.q0 = q0; g.q1 = q0 + sn;
    g.sn = std::min(HMK_MAXBATCH, 2 * sn);      // rows only get shorter: the next batch may take more queries again
    g.valid = true;
}

int Engine::score_graph(int64_t* cursor, hmk_graph_edge* out, int64_t cap, int64_t* n_out) {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_score_graph before hmk_upload");
    if (!cursor || !n_out || cap < 0 || (cap > 0 && !out)) throw std::invalid_argument("hmk_score_graph: bad argument");
    *n_out = 0;
    if (bad_residue_) return HMK_ERR_BAD_RESIDUE;
    if (n_ >= 2 && X_ >= min_len_) return HMK_ERR_SHIFT_TOO_BIG;
    int64_t i = cursor[0], r = cursor[1];
    if (i < 0 || r < 0 || i > n_ || (i == n_ && r != 0) || (n_ < 2 && r != 0))
        throw std::invalid_argument("hmk_score_graph: cursor outside the graph");
    GraphBatch& g = graph_;
    if (i == 0 && r == 0 && opt.profile) section_ms[0] = section_ms[1] = 0;
    reset_timing();
    if (!(g.valid && i == g.next_i && r == g.next_r)) g.valid = false;   // only a continuing cursor reuses the kept batch
    if (n_ < 2) i = n_;
    int64_t got = 0;
    for (bool first = true; i < n_; first = false) {
        if (!g.valid || i < g.q0 || i >= g.q1) graph_batch((int)i);
        const int64_t* ro = g.row_off.data();
        const int64_t t = i - g.q0, end = ro[g.q1 - g.q0];
        if (first && r > ro[t + 1] - ro[t]) throw std::invalid_argument("hmk_score_graph: cursor beyond the row's edges");
        const int64_t p = ro[t] + r, take = std::min(cap - got, end - p);
        if (take > 0) {
            CK(cudaMemcpyAsync(out + got, g.edges.p + p, sizeof(hmk_graph_edge) * take, cudaMemcpyDeviceToHost, st_));
            CK(cudaStreamSynchronize(st_));
            got += take;
        }
        const int64_t e = p + take;
        if (e == end) {          // batch done
            i = g.q1; r = 0;
            if (got == cap) break;
            continue;
        }
        const int64_t row = std::upper_bound(ro, ro + (g.q1 - g.q0) + 1, e) - ro - 1;   // ro[row] <= e < ro[row + 1]
        i = g.q0 + row; r = e - ro[row];
        break;
    }
    cursor[0] = i; cursor[1] = r;
    g.next_i = i; g.next_r = r;
    *n_out = got;
    return HMK_OK;
}

int Engine::score_pairs(const int32_t* seq1, const int32_t* seq2, int32_t np, int32_t* scores, int32_t* shifts) {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_score_pairs before hmk_upload");
    if (np < 0 || (np > 0 && (!seq1 || !seq2 || !scores || !shifts))) throw std::invalid_argument("hmk_score_pairs: bad argument");
    std::vector<int4> pairs(np);
    bool too_big = false;
    for (int32_t e = 0; e < np; e++) {
        if (seq1[e] < 0 || seq1[e] >= n_ || seq2[e] < 0 || seq2[e] >= n_) throw std::invalid_argument("hmk_score_pairs: id out of range");
        const int l1 = h_off_[seq1[e] + 1] - h_off_[seq1[e]], l2 = h_off_[seq2[e] + 1] - h_off_[seq2[e]];
        too_big |= X_ >= std::min(l1, l2);
        pairs[e] = make_int4(seq2[e], seq1[e], 0, 0);
    }
    if (bad_residue_) return HMK_ERR_BAD_RESIDUE;
    if (too_big) return HMK_ERR_SHIFT_TOO_BIG;
    if (np == 0) return HMK_OK;
    DevBuf<int4> d_pairs;
    DevBuf<int32_t> d_out;
    d_pairs.reserve(np); d_out.reserve(2 * (size_t)np);
    CK(cudaMemcpyAsync(d_pairs.p, pairs.data(), sizeof(int4) * np, cudaMemcpyHostToDevice, st_));
    shift_pass(d_pairs.p, nullptr, (unsigned int)np, 0, 0, nullptr, nullptr, nullptr, d_out.p, d_out.p + np);
    CK(cudaMemcpyAsync(scores, d_out.p, sizeof(int32_t) * np, cudaMemcpyDeviceToHost, st_));
    CK(cudaMemcpyAsync(shifts, d_out.p + np, sizeof(int32_t) * np, cudaMemcpyDeviceToHost, st_));
    CK(cudaStreamSynchronize(st_));
    return HMK_OK;
}

// ---------------------------------------------------------------- nearest partners (hmk_nearest)
// Row i's list: the k best ids j != i with scoreWithShift(seq1 = j, seq2 = i) >= T under the partner search's key
// (score desc, then tie-break rank: abundance desc, id asc).  Per batch of rows: the partner search's TOPK launch with
// kb = k + 1 over every thread-side id [0, n) (no q_minid: the row's own id competes too), the stripe merge, and
// hmk_nearest_rows, which drops the row's own id, cuts the list to k and adds each entry's score and shift.  The top
// k + 1 keys of all ids contain the top k of the others, so the lists are exact, and so is `more` (see the kernel).
int Engine::nearest(int32_t k, int32_t row_begin, int32_t n_rows, int32_t* partner, int32_t* score, int32_t* shift,
                    int32_t* count, int32_t* more) {
    CK(cudaSetDevice(device_));
    if (!uploaded_) throw std::invalid_argument("hmk_nearest before hmk_upload");
    if (k < 1 || k > HMK_NEAREST_MAX_K) throw std::invalid_argument("hmk_nearest: k outside 1 .. 31");
    if (row_begin < 0 || n_rows < 0 || (int64_t)row_begin + n_rows > n_)
        throw std::invalid_argument("hmk_nearest: row range outside [0, n]");
    if (n_rows > 0 && (!partner || !score || !shift || !count || !more)) throw std::invalid_argument("hmk_nearest: null output");
    if (bad_residue_) return HMK_ERR_BAD_RESIDUE;
    if (n_ >= 2 && X_ >= min_len_) return HMK_ERR_SHIFT_TOO_BIG;
    if (opt.profile) section_ms[0] = section_ms[1] = 0;
    if (n_ < 2) {        // no partner exists
        for (int64_t e = 0; e < (int64_t)n_rows * k; e++) { partner[e] = -1; score[e] = 0; shift[e] = 0; }
        for (int32_t t = 0; t < n_rows; t++) { count[t] = 0; more[t] = 0; }
        return HMK_OK;
    }
    const int kb = k + 1;
    BatchBuf& bb = near_bb_;
    bb.gmin.reserve(HMK_MAXBATCH);
    bb.bk_key.reserve((size_t)HMK_MAXBATCH * kb); bb.bk_cnt.reserve(HMK_MAXBATCH); bb.bk_ovf.reserve(HMK_MAXBATCH);
    if (fast_) bb.prof.reserve((size_t)HMK_MAXBATCH * sc_.prof_words);
    d_near_out_.reserve((size_t)HMK_MAXBATCH * (3 * k + 2));
    int32_t* const o_partner = d_near_out_.p;
    int32_t* const o_score = o_partner + (size_t)HMK_MAXBATCH * k;
    int32_t* const o_shift = o_score + (size_t)HMK_MAXBATCH * k;
    int32_t* const o_count = o_shift + (size_t)HMK_MAXBATCH * k;
    int32_t* const o_more = o_count + HMK_MAXBATCH;
    const int32_t* ids = identity_ids();
    reset_timing();
    for (int32_t r0 = row_begin; r0 < row_begin + n_rows; r0 += HMK_MAXBATCH) {
        const int sn = std::min<int32_t>(HMK_MAXBATCH, row_begin + n_rows - r0);
        sec(0);
        CK(cudaMemsetAsync(bb.gmin.p, 0, sizeof(unsigned long long) * sn, st_));
        HmkBulkArgs a = query_batch(ids + r0, sn, bb.prof.p, kb);
        a.db_ids = nullptr; a.db_begin = 0; a.ndb = n_;
        a.tierank = identity_rank_ ? nullptr : d_tierank_.p;
        a.tk_gmin = bb.gmin.p;
        const HmkBulkArgs p = launch_bulk(HMK_MODE_TOPK, a, ids + r0, 1, st_, &bb);
        stats.bulk_pairs += (int64_t)sn * n_;
        sec(1);
        merge_topk(sn, p.nstripes, kb, bb.tk_key.p, bb.tk_cnt.p, bb.tk_ovf.p, bb, st_, p.sched ? p.sched + p.nqt : nullptr, p.qt);
        HmkNearestArgs na{};
        na.nq = sn; na.k = k; na.r0 = r0; na.n = n_;
        na.key = bb.bk_key.p; na.cnt = bb.bk_cnt.p; na.ovf = bb.bk_ovf.p;
        na.id_of_rank = identity_rank_ ? nullptr : d_id_of_rank_.p;
        na.res = d_res_.p; na.off = d_off_.p; na.M = d_M_.p; na.X = X_; na.P = P_;
        na.partner = o_partner; na.score = o_score; na.shift = o_shift; na.count = o_count; na.more = o_more;
        hmk_nearest_rows<<<(sn * 32 + 255) / 256, 256, 0, st_>>>(na);
        CK(cudaGetLastError());
        launches_++;
        sec(-1);
        const size_t e0 = (size_t)(r0 - row_begin) * k, t0 = (size_t)(r0 - row_begin), ne = (size_t)sn * k;
        CK(cudaMemcpyAsync(partner + e0, o_partner, sizeof(int32_t) * ne, cudaMemcpyDeviceToHost, st_));
        CK(cudaMemcpyAsync(score + e0, o_score, sizeof(int32_t) * ne, cudaMemcpyDeviceToHost, st_));
        CK(cudaMemcpyAsync(shift + e0, o_shift, sizeof(int32_t) * ne, cudaMemcpyDeviceToHost, st_));
        CK(cudaMemcpyAsync(count + t0, o_count, sizeof(int32_t) * sn, cudaMemcpyDeviceToHost, st_));
        CK(cudaMemcpyAsync(more + t0, o_more, sizeof(int32_t) * sn, cudaMemcpyDeviceToHost, st_));
        CK(cudaStreamSynchronize(st_));
        fold_timing();
    }
    return HMK_OK;
}

void Engine::init_distributed(int rank, int world, const void* id128) {
    CK(cudaSetDevice(device_));
    if (world < 1 || rank < 0 || rank >= world || !id128) throw std::invalid_argument("hmk_init_distributed: bad rank/world/id");
    NcclApi& api = NcclApi::get();
    if (!api.ok) throw CudaError("NCCL unavailable: " + api.error);
    if (comm_) { api.CommDestroy(comm_); comm_ = nullptr; }
    NcclApi::UniqueId id;
    std::memcpy(id.internal, id128, 128);
    NK(api.CommInitRank(&comm_, world, id, rank));
    rank_ = rank;
    world_ = world;
}

// out[0] = IADD3 lane-instructions/s, out[1] = lane-instructions/s of an IADD3 + IMAD mix,
// out[2] = shared-memory LDS.32 bytes/s (conflict free), out[3] = SM count
void Engine::measure_peaks(double* out) {
    CK(cudaSetDevice(device_));
    DevBuf<int32_t> sink;
    const int blocks = sm_count_ * 2, threads = 1024, iters = 2000;
    sink.reserve((size_t)blocks * threads);
    auto time_it = [&](int which) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {
            CK(cudaEventRecord(ev_t0_, st_));
            if (which == 0) hmk_peak_iadd<<<blocks, threads, 0, st_>>>(iters, sink.p);
            else if (which == 1) hmk_peak_imix<<<blocks, threads, 0, st_>>>(iters, 1, sink.p);
            else hmk_peak_lds<<<blocks, threads, 0, st_>>>(iters, sink.p);
            CK(cudaGetLastError());
            CK(cudaEventRecord(ev_t1_, st_));
            CK(cudaEventSynchronize(ev_t1_));
            float ms = 0;
            CK(cudaEventElapsedTime(&ms, ev_t0_, ev_t1_));
            if (rep > 0) best = std::min(best, ms);
        }
        return (double)best * 1e-3;
    };
    const double lanes = (double)blocks * threads;
    // lane-instructions per second: 128 adds -> 64 IADD3 per unrolled body; the mixed kernel
    // issues 32 IADD3 (4 add chains, fused in pairs) + 64 IMAD (4 mad chains)
    out[0] = lanes * iters * 64 / time_it(0);
    out[1] = lanes * iters * 96 / time_it(1);
    out[2] = lanes * iters * 32 * 4.0 / time_it(2);
    out[3] = sm_count_;
}

}  // namespace

// ---------------------------------------------------------------- C ABI
struct hmk_ctx {
    Engine engine;
    explicit hmk_ctx(int device) : engine(device) {}
};

// Contexts kept between one-shot calls, keyed by device.  Every access holds cache_mutex().  The map is
// deliberately leaked at process exit: destroying it from a static destructor would call cudaFree /
// cudaStreamDestroy / ncclCommDestroy after the CUDA runtime has been torn down.  A host that wants the
// memory back calls hmk_release_cached().
static std::mutex& cache_mutex() {
    static std::mutex* mu = new std::mutex();
    return *mu;
}
static std::map<int, std::unique_ptr<hmk_ctx>>& cached_ctx() {
    static auto* m = new std::map<int, std::unique_ptr<hmk_ctx>>();
    return *m;
}
// the device set of the last hmk_greedy_cluster_multi call (its contexts live in cached_ctx())
static std::vector<int>& cached_group() {
    static auto* g = new std::vector<int>();
    return *g;
}
// caller holds cache_mutex().  The communicators of a group are destroyed inside one NCCL group call: one
// thread destroying them one after the other could wait for its own later calls.
static void clear_cached() {
    if (!cached_group().empty() && NcclApi::get().ok) {
        NcclApi::get().GroupStart();
        for (auto& kv : cached_ctx()) if (kv.second) kv.second->engine.release_comm();
        NcclApi::get().GroupEnd();
    }
    cached_group().clear();
    cached_ctx().clear();
}

static void set_err(char* errbuf, size_t errlen, const char* msg) {
    if (errbuf && errlen) {
        std::strncpy(errbuf, msg, errlen - 1);
        errbuf[errlen - 1] = 0;
    }
}

template <class F>
static int guarded(char* errbuf, size_t errlen, F&& f) {
    try {
        return f();
    } catch (const CudaError& e) {
        set_err(errbuf, errlen, e.what());
        return HMK_STATUS_CUDA;
    } catch (const std::invalid_argument& e) {
        set_err(errbuf, errlen, e.what());
        return HMK_STATUS_BAD_ARG;
    } catch (const std::exception& e) {
        set_err(errbuf, errlen, e.what());
        return HMK_STATUS_CUDA;
    }
}

static const char* status_text(int rc) {
    switch (rc) {
        case HMK_STATUS_SHIFT_TOO_BIG: return "DataException: Shift too big (max_shift >= length of the shortest sequence)";
        case HMK_STATUS_NULL_CLUSTER: return "NullPointerException: nearest cluster object without a cluster (see error_step)";
        case HMK_STATUS_BAD_RESIDUE: return "FileFormatException: residue code outside 0..23";
        case HMK_STATUS_UNSUPPORTED: return "unsupported input for the exact complete-linkage clusterer: asymmetric substitution matrix, "
                                            "valid pairs beyond the free device memory, or a java.util.HashMap bin that would be treeified";
        default: return "";
    }
}

extern "C" {

int hmk_abi_version(void) { return HMK_ABI_VERSION; }

void hmk_release_cached(void) {
    std::lock_guard<std::mutex> lock(cache_mutex());
    clear_cached();
}

int hmk_create(hmk_ctx** ctx, int device, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    *ctx = nullptr;
    return guarded(errbuf, errlen, [&] {
        *ctx = new hmk_ctx(device);
        return HMK_STATUS_OK;
    });
}

void hmk_destroy(hmk_ctx* ctx) { delete ctx; }

int hmk_upload(hmk_ctx* ctx, const hmk_greedy_in* in, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.upload(in);
        return HMK_STATUS_OK;
    });
}

int hmk_run(hmk_ctx* ctx, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        int rc = ctx->engine.run();
        if (rc) set_err(errbuf, errlen, status_text(rc));
        return rc;
    });
}

int hmk_download(hmk_ctx* ctx, hmk_greedy_out* out, char* errbuf, size_t errlen) {
    if (!ctx || !out) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.download(out);
        return HMK_STATUS_OK;
    });
}

int hmk_get_stats(hmk_ctx* ctx, hmk_stats* stats) {
    if (!ctx || !stats) return HMK_STATUS_BAD_ARG;
    *stats = ctx->engine.stats;
    return HMK_STATUS_OK;
}

int hmk_nccl_unique_id(void* id128, char* errbuf, size_t errlen) {
    if (!id128) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        NcclApi& api = NcclApi::get();
        if (!api.ok) throw CudaError("NCCL unavailable: " + api.error);
        NcclApi::UniqueId id;
        NK(api.GetUniqueId(&id));
        std::memcpy(id128, id.internal, 128);
        return HMK_STATUS_OK;
    });
}

int hmk_init_distributed(hmk_ctx* ctx, int rank, int world, const void* id128, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.init_distributed(rank, world, id128);
        return HMK_STATUS_OK;
    });
}

int hmk_timer_begin(hmk_ctx* ctx) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(nullptr, 0, [&] { ctx->engine.timer_begin(); return HMK_STATUS_OK; });
}

int hmk_timer_end(hmk_ctx* ctx, double* ms) {
    if (!ctx || !ms) return HMK_STATUS_BAD_ARG;
    return guarded(nullptr, 0, [&] { *ms = ctx->engine.timer_end(); return HMK_STATUS_OK; });
}

int hmk_measure_peaks(hmk_ctx* ctx, double* out4, char* errbuf, size_t errlen) {
    if (!ctx || !out4) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] { ctx->engine.measure_peaks(out4); return HMK_STATUS_OK; });
}

int hmk_get_section_ms(hmk_ctx* ctx, double* out, int n) {
    if (!ctx || !out) return HMK_STATUS_BAD_ARG;
    for (int i = 0; i < n && i < HMK_NSECTIONS; i++) out[i] = ctx->engine.section_ms[i];
    return HMK_STATUS_OK;
}

int hmk_set_option(hmk_ctx* ctx, const char* name, int64_t value) {
    if (!ctx || !name) return HMK_STATUS_BAD_ARG;
    Options& o = ctx->engine.opt;
    std::string s(name);
    // every knob has a range; values outside it are rejected instead of reaching a launch configuration
    struct Knob { const char* name; int64_t* slot; int64_t lo, hi; };
    const Knob knobs[] = {
        {"batch", &o.batch, 0, HMK_MAXBATCH},       {"qt", &o.qt, 0, 255},
        {"capq", &o.capq, 1, 1 << 20},              {"lookahead", &o.lookahead, 0, 2},
        {"filter", &o.filter, 0, 1},                {"reuse", &o.reuse, 0, 1},
        {"kb", &o.kb, 1, 32},                       {"waves", &o.waves, 1, 16},
        {"p2_chunk", &o.p2_chunk, 1024, 1 << 24},   {"hit_cap", &o.hit_cap, 1024, (int64_t)1 << 30},
        {"force_generic", &o.force_generic, 0, 1},  {"profile", &o.profile, 0, 1},
        {"p2_window", &o.p2_window, 1, 1 << 24},
        {"xhit_cap", &o.xhit_cap, 0, (int64_t)1 << 30}, {"p2_first", &o.p2_first, 0, 1 << 24},
        {"persistent", &o.persistent, 0, 1},        {"reserve", &o.reserve, 1, 64},
        {"min_iters", &o.min_iters, 1, 64},         {"bucket_aux", &o.bucket_aux, 0, 1},
        {"clinkage_dense_max", &o.clinkage_dense_max, 0, 32768},
        {"clinkage_threads", &o.clinkage_threads, 0, HMK_CL_THREADS},
        {"graph_cap", &o.graph_cap, 0, (int64_t)1 << 30},
    };
    for (const Knob& k : knobs) {
        if (s != k.name) continue;
        if (value < k.lo || value > k.hi) return HMK_STATUS_BAD_ARG;
        if (k.slot == &o.clinkage_threads && value % 32) return HMK_STATUS_BAD_ARG;   // whole warps
        *k.slot = value;
        return HMK_STATUS_OK;
    }
    return HMK_STATUS_BAD_ARG;
}

int hmk_score_block(hmk_ctx* ctx, const int32_t* first_ids, int32_t n_first, const int32_t* second_ids,
                    int32_t n_second, int32_t* scores, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.score_block(first_ids, n_first, second_ids, n_second, scores);
        return HMK_STATUS_OK;
    });
}

int hmk_score_graph(hmk_ctx* ctx, int64_t cursor[2], hmk_graph_edge* out, int64_t cap, int64_t* n_out, char* errbuf,
                    size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        int rc = ctx->engine.score_graph(cursor, out, cap, n_out);
        if (rc) set_err(errbuf, errlen, status_text(rc));
        return rc;
    });
}

int hmk_score_pairs(hmk_ctx* ctx, const int32_t* seq1_ids, const int32_t* seq2_ids, int32_t n_pairs, int32_t* scores,
                    int32_t* shifts, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        int rc = ctx->engine.score_pairs(seq1_ids, seq2_ids, n_pairs, scores, shifts);
        if (rc) set_err(errbuf, errlen, status_text(rc));
        return rc;
    });
}

int hmk_nearest(hmk_ctx* ctx, int32_t k, int32_t row_begin, int32_t n_rows, int32_t* partner, int32_t* score,
                int32_t* shift, int32_t* count, int32_t* more, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        int rc = ctx->engine.nearest(k, row_begin, n_rows, partner, score, shift, count, more);
        if (rc) set_err(errbuf, errlen, status_text(rc));
        return rc;
    });
}

int hmk_bulk_probe(hmk_ctx* ctx, int32_t mode, const int32_t* query_ids, int32_t n_query, const int32_t* db_ids,
                   int32_t db_begin, int32_t n_db, const uint8_t* clustered, uint64_t* keys, int32_t* counts,
                   int32_t* overflow, int32_t* hits, int64_t hit_cap, int64_t* hit_count, int32_t* kernel, char* errbuf,
                   size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.bulk_probe(mode, query_ids, n_query, db_ids, db_begin, n_db, clustered, keys, counts, overflow, hits,
                               hit_cap, hit_count, kernel);
        return HMK_STATUS_OK;
    });
}

int hmk_batch_probe(hmk_ctx* ctx, const int32_t* member_off, const int32_t* members, int32_t ncl, int32_t cur, int32_t nq,
                    int32_t capq, int32_t tail_stream, hmk_batch_probe_out* out, char* errbuf, size_t errlen) {
    if (!ctx) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        ctx->engine.batch_probe(member_off, members, ncl, cur, nq, capq, tail_stream, out);
        return HMK_STATUS_OK;
    });
}

int hmk_greedy_cluster(const hmk_greedy_in* in, hmk_greedy_out* out, int device, char* errbuf, size_t errlen) {
    if (!in || !out) return HMK_STATUS_BAD_ARG;
    // one cached context per device: repeated calls reuse its device buffers (released by
    // hmk_release_cached or at process exit); calls are serialised
    std::lock_guard<std::mutex> lock(cache_mutex());
    return guarded(errbuf, errlen, [&] {
        if (!cached_group().empty()) clear_cached();      // contexts of a multi-GPU group carry a communicator: start afresh
        auto& slot = cached_ctx()[device];
        if (!slot) slot.reset(new hmk_ctx(device));
        hmk_ctx& ctx = *slot;
        ctx.engine.upload(in);
        int rc = ctx.engine.run();
        out->n_result = 0; out->n_multi = 0; out->error_step = ctx.engine.error_step;
        if (rc) { set_err(errbuf, errlen, status_text(rc)); return rc; }
        ctx.engine.download(out);
        return HMK_STATUS_OK;
    });
}


int hmk_clinkage_cluster(const hmk_greedy_in* in, hmk_greedy_out* out, int device, char* errbuf, size_t errlen) {
    if (!in || !out) return HMK_STATUS_BAD_ARG;
    std::lock_guard<std::mutex> lock(cache_mutex());
    return guarded(errbuf, errlen, [&] {
        if (!cached_group().empty()) clear_cached();
        auto& slot = cached_ctx()[device];
        if (!slot) slot.reset(new hmk_ctx(device));
        int rc = slot->engine.clinkage(in, out);
        if (rc) set_err(errbuf, errlen, slot->engine.status_msg.empty() ? status_text(rc) : slot->engine.status_msg.c_str());
        return rc;
    });
}

int hmk_clinkage_run(hmk_ctx* ctx, const hmk_greedy_in* in, hmk_greedy_out* out, char* errbuf, size_t errlen) {
    if (!ctx || !in || !out) return HMK_STATUS_BAD_ARG;
    return guarded(errbuf, errlen, [&] {
        int rc = ctx->engine.clinkage(in, out);
        if (rc) set_err(errbuf, errlen, ctx->engine.status_msg.empty() ? status_text(rc) : ctx->engine.status_msg.c_str());
        return rc;
    });
}

int hmk_greedy_cluster_multi(const hmk_greedy_in* in, hmk_greedy_out* out, const int32_t* devices, int32_t n_gpus,
                             char* errbuf, size_t errlen) {
    if (!in || !out || n_gpus < 1 || n_gpus > 64) return HMK_STATUS_BAD_ARG;
    std::vector<int> devs(n_gpus);
    for (int r = 0; r < n_gpus; r++) devs[r] = devices ? devices[r] : r;
    for (int r = 0; r < n_gpus; r++)
        for (int q = 0; q < r; q++)
            if (devs[q] == devs[r]) { set_err(errbuf, errlen, "hmk_greedy_cluster_multi: duplicate device"); return HMK_STATUS_BAD_ARG; }
    if (n_gpus == 1) return hmk_greedy_cluster(in, out, devs[0], errbuf, errlen);
    std::lock_guard<std::mutex> lock(cache_mutex());
    // one worker thread per device for every stage; a stage ends when all its threads have joined, so a
    // failure before the first collective (allocation, bad input) is reported without leaving ranks waiting
    std::vector<int> rcs(n_gpus, HMK_STATUS_OK);
    std::vector<std::string> errs(n_gpus);
    auto stage = [&](auto&& body) {
        std::vector<std::thread> th;
        for (int r = 0; r < n_gpus; r++)
            th.emplace_back([&, r] {
                char eb[512] = {0};
                rcs[r] = guarded(eb, sizeof eb, [&] { return body(r); });
                errs[r] = eb;
            });
        for (auto& t : th) t.join();
        for (int r = 0; r < n_gpus; r++)
            if (rcs[r] != HMK_STATUS_OK) return r;
        return -1;
    };
    auto fail = [&](int r) {
        set_err(errbuf, errlen, errs[r].c_str());
        return rcs[r];
    };
    out->n_result = 0; out->n_multi = 0; out->error_step = -1;
    if (cached_group() != devs) {       // (re)build the group: contexts + one NCCL communicator over them
        clear_cached();
        NcclApi::UniqueId id;
        int rc0 = guarded(errbuf, errlen, [&] {
            NcclApi& api = NcclApi::get();
            if (!api.ok) throw CudaError("NCCL unavailable: " + api.error);
            NK(api.GetUniqueId(&id));
            return HMK_STATUS_OK;
        });
        if (rc0) return rc0;
        std::vector<std::unique_ptr<hmk_ctx>> fresh(n_gpus);
        int bad = stage([&](int r) {
            fresh[r].reset(new hmk_ctx(devs[r]));
            fresh[r]->engine.init_distributed(r, n_gpus, id.internal);
            return HMK_STATUS_OK;
        });
        if (bad >= 0) return fail(bad);
        for (int r = 0; r < n_gpus; r++) cached_ctx()[devs[r]] = std::move(fresh[r]);
        cached_group() = devs;
    }
    std::vector<hmk_ctx*> ctx(n_gpus);
    for (int r = 0; r < n_gpus; r++) ctx[r] = cached_ctx()[devs[r]].get();
    int bad = stage([&](int r) { ctx[r]->engine.upload(in); return HMK_STATUS_OK; });
    if (bad >= 0) return fail(bad);
    bad = stage([&](int r) { return ctx[r]->engine.run(); });     // replicated decisions: every rank returns the same status
    out->error_step = ctx[0]->engine.error_step;
    if (bad >= 0) {
        if (errs[bad].empty()) set_err(errbuf, errlen, status_text(rcs[bad]));
        else set_err(errbuf, errlen, errs[bad].c_str());
        if (rcs[bad] == HMK_STATUS_CUDA) clear_cached();      // a rank died mid-run: the group is not reusable
        return rcs[bad];
    }
    return guarded(errbuf, errlen, [&] { ctx[0]->engine.download(out); return HMK_STATUS_OK; });
}

}  // extern "C"
