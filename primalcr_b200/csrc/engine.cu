// engine.cu -- host orchestration of the Primal-CR / Primal-CR++ alternating Newton-CG loop on one GPU,
// and the C ABI declared in include/primalcr.h.
//
// Control flow mirrors the reference exactly (SURVEY.md 3.2 / 3.3):
//   update_V  : pcrpp.cpp:415-444 (pcr.cpp:279-330) with solve_delta_new :335-358
//   update_U  : pcrpp.cpp:818-838 / update_u_new :779-815 (pcr.cpp:587-611 / :523-585), batched over users
//   driver    : pcrpp.cpp:841-901 / pcr.cpp:616-704
// Arithmetic runs in the kernels of k_core.cu / k_pairs.cu.  There is no CPU implementation of any stage.
#include "kernels.h"
#include "../../include/primalcr.h"
#include "../host/loader.hpp"
#include "../host/rankmetrics.hpp"
#include "../host/textio.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstring>
#include <dlfcn.h>
#include <random>
#include <mutex>

// ---- NCCL, bound at run time (only needed when world > 1) -----------------------------------------
typedef struct { char internal[128]; } pcr_ncclUniqueId;
typedef void *pcr_ncclComm_t;
enum { PCR_NCCL_FLOAT64 = 8, PCR_NCCL_SUM = 0 };

namespace pcr {

struct NcclApi {
    void *h = nullptr;
    int (*GetUniqueId)(pcr_ncclUniqueId *) = nullptr;
    int (*CommInitRank)(pcr_ncclComm_t *, int, pcr_ncclUniqueId, int) = nullptr;
    int (*AllReduce)(const void *, void *, size_t, int, int, pcr_ncclComm_t, cudaStream_t) = nullptr;
    int (*ReduceScatter)(const void *, void *, size_t, int, int, pcr_ncclComm_t, cudaStream_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, pcr_ncclComm_t, cudaStream_t) = nullptr;
    int (*CommDestroy)(pcr_ncclComm_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    bool load() {
        if (h) return true;
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) { h = dlopen(n, RTLD_NOW | RTLD_GLOBAL); if (h) break; }
        if (!h) return false;
        GetUniqueId = (decltype(GetUniqueId))dlsym(h, "ncclGetUniqueId");
        CommInitRank = (decltype(CommInitRank))dlsym(h, "ncclCommInitRank");
        AllReduce = (decltype(AllReduce))dlsym(h, "ncclAllReduce");
        ReduceScatter = (decltype(ReduceScatter))dlsym(h, "ncclReduceScatter");
        AllGather = (decltype(AllGather))dlsym(h, "ncclAllGather");
        CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
        GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
        return GetUniqueId && CommInitRank && AllReduce && ReduceScatter && AllGather && CommDestroy;
    }
};
static NcclApi g_nccl;

// Communicators are per-process state: the first engine of a (device, rank, world) creates one from a ncclUniqueId,
// later engines of the same process may re-attach to it (primalcr_comm_init with a NULL id) instead of paying
// ncclCommInitRank (~1-2 s) again.  Cached communicators live until the process exits.
struct CommKey { int device, rank, world; bool operator<(const CommKey &o) const {
    return device != o.device ? device < o.device : (rank != o.rank ? rank < o.rank : world < o.world); } };
static std::map<CommKey, pcr_ncclComm_t> g_comm_cache;
static std::mutex g_comm_mutex;

static thread_local std::string g_last_error;

// leading dimension of every factor-shaped array: rows start on 128-byte lines (a 128-byte row chunk never straddles two)
static int ceil16(int k) { return (k + 15) & ~15; }

struct Engine {
    primalcr_config cfg;
    cudaStream_t stream = nullptr;
    // side stream: the chunk-parallel heavy-user kernels (few, small grids) run beside the tile kernels of the same stage
    cudaStream_t aux = nullptr; cudaEvent_t ev_fork = nullptr, ev_join = nullptr; Ctx ctx_aux;
    Profiler prof;
    DevPool pool;
    Ctx ctx;
    int sms = 148;
    int k = 0, ld = 0, T = 0;
    i64 d1 = 0, d2 = 0;
    std::vector<i64> levels;
    bool levels_user_set = false;
    DevCsr X, XT;
    bool has_train = false, has_test = false, has_factors = false, use_tiles = true;
    bool ratings_integer = false;     // every training rating equals its lround: levels order ratings like the exact doubles
    double *level_vals = nullptr;     // [8] the level table as doubles (NDCG gains from the sorted state)
    i64 *ev_err_user = nullptr;
    // CSC of the training set (by item)
    i64 *col_ptr = nullptr; int32_t *csc_user = nullptr, *csc2csr = nullptr;
    int32_t *cu_seg = nullptr; i64 *cu_start = nullptr, *cu_end = nullptr; i64 n_cunits = 0; i64 *col_unit_ptr = nullptr;
    int32_t *col_unit_idx = nullptr; int n_user_blocks = 1;
    // multi-GPU, large item sets: V-side vectors are reduce-scattered by item rows, the CG algebra runs on this rank's row
    // slice and the search direction is all-gathered (see update_V); d2p = d2 rounded up to a multiple of the world size
    bool sharded_cg = false; i64 d2p = 0, vs_row0 = 0, vs_rows = 0;
    // factors (padded leading dimension ld)
    double *U = nullptr, *V = nullptr;
    // per-rating work buffers
    double *m = nullptr, *b = nullptr, *cbuf = nullptr;
    SortedMeta meta;
    bool scores_valid = false, meta_valid = false;
    // heavy-user scratch of the one-CTA-per-user kernels (allocated on demand: T > 8, or the score-order outputs for tests)
    double *h_v = nullptr, *h_p1 = nullptr, *h_p2 = nullptr, *h_acc = nullptr; int32_t *h_cnt = nullptr;
    HeavyLM hv;                       // chunk-parallel heavy-user path (k_heavy.cu)
    bool heavy_chunked = false, heavy_windows_valid = false;
    HeavySortPlan hsort;              // hand-written segmented sort of the heavy users (k_hsort.cu)
    // V-side vectors [d2 x ld]
    double *g = nullptr, *delta = nullptr, *rr = nullptr, *p = nullptr, *Hp = nullptr, *Vnew = nullptr;
    double *partial = nullptr;
    double *red_partials = nullptr, *slots = nullptr; double *h_slots = nullptr;
    int *h_counters = nullptr;
    UState us;
    uint8_t *has_pairs = nullptr;
    double *obj_item = nullptr;
    i64 *stats_dev = nullptr; i64 *h_stats = nullptr;
    // evaluation buffers (sized for max(train, test))
    double *ev_score_t = nullptr; i64 *ev_err_item = nullptr;
    double *ev_a = nullptr, *ev_b = nullptr, *ev_c = nullptr, *ev_d = nullptr;
    // comm
    int rank = 0, world = 1; pcr_ncclComm_t comm = nullptr;
    primalcr_counters counters;
    int v_accepted = 1;

    explicit Engine(const primalcr_config &c) : cfg(c) {
        memset(&counters, 0, sizeof(counters));
        memset(&us, 0, sizeof(us));
        PCR_REQUIRE(cfg.solver == 1 || cfg.solver == 2, "solver must be 1 (Primal-CR) or 2 (Primal-CR++)");
        PCR_REQUIRE(cfg.k >= 1 && cfg.k <= 256, "rank k out of range [1, 256]");
        // NDCG@k keeps the top-k of a user in a 64-entry shared-memory table (k_pairs.cu eval_users_kernel); the reference's
        // min(ndcg_k, len) with ndcg_k <= 0 divides 0 by 0 (util.cpp:513-531)
        PCR_REQUIRE(cfg.ndcg_k >= 1 && cfg.ndcg_k <= 64, "ndcg_k out of range [1, 64]");
        int ndev = 0;
        cudaError_t e = cudaGetDeviceCount(&ndev);
        if (e != cudaSuccess || ndev == 0)
            throw Error(PRIMALCR_ECUDA, "no CUDA device available: libprimalcr_b200 has no CPU fallback");
        PCR_REQUIRE(cfg.device >= 0 && cfg.device < ndev, "bad device ordinal");
        PCR_CUDA(cudaSetDevice(cfg.device));
        cudaDeviceProp prop;
        PCR_CUDA(cudaGetDeviceProperties(&prop, cfg.device));
        sms = prop.multiProcessorCount;
        PCR_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
        pool.init(stream);
        ctx.stream = stream; ctx.prof = &prof; ctx.sms = sms;
        {   // highest priority: the few CTAs of the heavy-user kernels are placed first whenever SM slots free up, so they finish
            // inside the tile kernel that runs beside them instead of after it
            int prio_lo = 0, prio_hi = 0;
            PCR_CUDA(cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi));
            PCR_CUDA(cudaStreamCreateWithPriority(&aux, cudaStreamNonBlocking, prio_hi));
        }
        PCR_CUDA(cudaEventCreateWithFlags(&ev_fork, cudaEventDisableTiming));
        PCR_CUDA(cudaEventCreateWithFlags(&ev_join, cudaEventDisableTiming));
        k = cfg.k; ld = ceil16(k);
        PCR_CUDA(cudaMallocHost(&h_slots, sizeof(double) * 32));
        PCR_CUDA(cudaMallocHost(&h_counters, sizeof(int) * 4));
        PCR_CUDA(cudaMallocHost(&h_stats, sizeof(i64) * 8));
        slots = pool.alloc<double>(32);
        red_partials = pool.alloc<double>(2048);     // >= 2 x RED_BLOCKS (k_cg_dots2 / k_cg_update)
        us.counters = pool.alloc<int>(4);
        ctx.ticket = pool.alloc<unsigned long long>(1);
        ctx_aux = ctx; ctx_aux.stream = aux;          // (the heavy-user kernels do not use the ticket counter)
        stats_dev = pool.alloc<i64>(8);
    }
    ~Engine() {
        cudaSetDevice(cfg.device);      // the communicator stays in the process-wide cache
        if (aux) cudaStreamSynchronize(aux);
        if (stream) cudaStreamSynchronize(stream);
        prof.resolve();
        if (ev_fork) cudaEventDestroy(ev_fork);
        if (ev_join) cudaEventDestroy(ev_join);
        if (aux) cudaStreamDestroy(aux);
        pool.release();
        if (h_slots) cudaFreeHost(h_slots);
        if (h_counters) cudaFreeHost(h_counters);
        if (h_stats) cudaFreeHost(h_stats);
        if (stream) cudaStreamDestroy(stream);
    }
    void bind() { PCR_CUDA(cudaSetDevice(cfg.device)); }
    // heavy-user work of a stage goes to the side stream between fork and join (disjoint users => disjoint outputs)
    void fork_aux() { PCR_CUDA(cudaEventRecord(ev_fork, stream)); PCR_CUDA(cudaStreamWaitEvent(aux, ev_fork, 0)); }
    void join_aux() { PCR_CUDA(cudaEventRecord(ev_join, aux)); PCR_CUDA(cudaStreamWaitEvent(stream, ev_join, 0)); }
    void sync() { PCR_CUDA(cudaStreamSynchronize(stream)); prof.resolve(); }

    template <typename Tp> Tp *upload(const Tp *h, size_t n) {
        Tp *d = pool.alloc<Tp>(n);
        if (n) PCR_CUDA(cudaMemcpyAsync(d, h, sizeof(Tp) * n, cudaMemcpyHostToDevice, stream));
        return d;
    }
    template <typename Tp> Tp *upload_vec(const std::vector<Tp> &v) { return upload(v.data(), v.size()); }

    // ------------------------------------------------------------------ data
    void build_csr_common(DevCsr &C, i64 d1_, i64 nnz, const i64 *row_ptr, const int32_t *item, const double *rating) {
        C.d1 = d1_; C.nnz = nnz;
        C.h_row_ptr.assign(row_ptr, row_ptr + d1_ + 1);
        PCR_REQUIRE(C.h_row_ptr[0] == 0 && C.h_row_ptr[d1_] == nnz, "row_ptr must start at 0 and end at nnz");
        PCR_REQUIRE(nnz < ((i64)1 << 31) - 64, "nnz per engine must be < 2^31 (shard the users)");
        C.row_ptr = upload(row_ptr, (size_t)d1_ + 1);
        C.item = upload(item, (size_t)nnz);
        C.rating = upload(rating, (size_t)nnz);
        C.user = pool.alloc<int32_t>((size_t)nnz);
        {   // item ids are used as array indices by every kernel: validate them first
            int *bad = pool.alloc<int>(1);
            PCR_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), stream));
            k_check_range(ctx, C.item, nnz, d2, bad);
            PCR_CUDA(cudaMemcpyAsync(h_counters, bad, sizeof(int), cudaMemcpyDeviceToHost, stream));
            PCR_CUDA(cudaStreamSynchronize(stream));
            PCR_REQUIRE(h_counters[0] == 0, "item id out of range [0, d2)");
        }
        for (i64 u = 0; u < d1_; ++u) PCR_REQUIRE(C.h_row_ptr[u + 1] >= C.h_row_ptr[u], "row_ptr must be non-decreasing");
        k_expand_users(ctx, C.row_ptr, d1_, nnz, C.user);
        // pair-tile work items
        std::vector<int32_t> ptu, ptj; std::vector<i64> ptp((size_t)d1_ + 1, 0);
        C.max_len = 0;
        for (i64 u = 0; u < d1_; ++u) {
            const i64 len = C.h_row_ptr[u + 1] - C.h_row_ptr[u];
            PCR_REQUIRE(len >= 0, "row_ptr must be non-decreasing");
            C.max_len = std::max(C.max_len, len);
            ptp[u] = (i64)ptu.size();
            for (i64 j0 = 0; j0 < len; j0 += PAIR_TJ) { ptu.push_back((int32_t)u); ptj.push_back((int32_t)j0); }
        }
        ptp[d1_] = (i64)ptu.size();
        C.n_pt = (i64)ptu.size();
        C.pt_user = upload_vec(ptu); C.pt_j0 = upload_vec(ptj); C.pt_ptr = upload_vec(ptp);
        sync();   // host vectors above go out of scope
    }

    static void make_units(const std::vector<i64> &ptr, std::vector<int32_t> &seg, std::vector<i64> &start,
                           std::vector<i64> &seg_unit_ptr) {
        const i64 nseg = (i64)ptr.size() - 1;
        seg.clear(); start.clear(); seg_unit_ptr.assign((size_t)nseg + 1, 0);
        for (i64 s = 0; s < nseg; ++s) {
            seg_unit_ptr[s] = (i64)seg.size();
            for (i64 b = ptr[s]; b < ptr[s + 1]; b += ROWSUM_CHUNK) { seg.push_back((int32_t)s); start.push_back(b); }
        }
        seg_unit_ptr[nseg] = (i64)seg.size();
        start.push_back(ptr[nseg]);
    }

    void set_levels(const i64 *vals, int n) {
        PCR_REQUIRE(n >= 1 && n <= MAX_LEVELS, "number of rating levels must be in [1, 256]");
        levels.assign(vals, vals + n);
        for (int i = 1; i < n; ++i) PCR_REQUIRE(levels[i] > levels[i - 1], "level table must be strictly ascending");
        levels_user_set = true;
    }

    struct Lap {
        bool on; std::chrono::steady_clock::time_point t;
        Lap() : on(getenv("PRIMALCR_VERBOSE_SETUP") != nullptr), t(std::chrono::steady_clock::now()) {}
        void operator()(const char *what) {
            if (!on) return;
            auto n = std::chrono::steady_clock::now();
            fprintf(stderr, "[primalcr setup] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(n - t).count());
            t = n;
        }
    };
    void set_train(i64 d1_, i64 d2_, i64 nnz, const i64 *row_ptr, const int32_t *item, const double *rating) {
        bind();
        Lap lap;
        PCR_REQUIRE(!has_train, "training set already loaded (one data set per engine)");
        PCR_REQUIRE(d1_ >= 0 && d2_ >= 1 && nnz >= 0, "bad sizes");
        d1 = d1_; d2 = d2_;
        build_csr_common(X, d1_, nnz, row_ptr, item, rating);
        lap("upload CSR + pair tiles");
        // ---- rating levels (find_levels pcrpp.cpp:38-49, as one global order-preserving table).  Primal-CR (-s 1) never
        // looks at levels (pcr.cpp compares the exact ratings), so any rating scale is accepted there.
        X.level = pool.alloc<uint8_t>((size_t)nnz);
        if (cfg.solver == 1) {
            levels.assign(1, 0); T = 1;
            PCR_CUDA(cudaMemsetAsync(X.level, 0, (size_t)(nnz > 0 ? nnz : 1), stream));
        } else {
            if (!levels_user_set) {
                i64 lo = 0, hi = 0; bool any = false;
                for (i64 e = 0; e < nnz; ++e) {
                    const i64 v = llround(rating[e]);
                    if (!any) { lo = hi = v; any = true; }
                    if (v < lo) lo = v; if (v > hi) hi = v;
                    if (hi - lo >= 65536) break;
                }
                if (!any) { lo = hi = 0; }
                std::vector<i64> distinct;
                if (hi - lo + 1 <= 8) {
                    // a superset of the levels present is harmless: an empty level contributes 0*x - 0 (SURVEY App. A)
                    for (i64 v = lo; v <= hi; ++v) distinct.push_back(v);
                } else if (hi - lo < 65536) {
                    std::vector<uint8_t> seen((size_t)(hi - lo + 1), 0);
                    for (i64 e = 0; e < nnz; ++e) seen[(size_t)(llround(rating[e]) - lo)] = 1;
                    for (i64 v = lo; v <= hi; ++v) if (seen[(size_t)(v - lo)]) distinct.push_back(v);
                } else {
                    for (i64 e = 0; e < nnz; ++e) {
                        const i64 v = llround(rating[e]);
                        auto it = std::lower_bound(distinct.begin(), distinct.end(), v);
                        if (it == distinct.end() || *it != v) distinct.insert(it, v);
                        if ((int)distinct.size() > MAX_LEVELS) break;
                    }
                }
                // more than 8 levels: the per-user T-vector kernels take over from the tile kernels (any T up to 256, the
                // range of the uint8 level index); the reference itself has no cap (find_levels is a per-user set)
                PCR_REQUIRE((int)distinct.size() <= MAX_LEVELS, "more than 256 distinct lround(rating) levels (Primal-CR++ level index is 8 bits; -s 1 has no limit)");
                levels = distinct;
            }
            T = (int)levels.size();
            {
                std::vector<double> lv(std::max<size_t>(levels.size(), 8), 0.0);
                for (size_t q = 0; q < levels.size(); ++q) lv[q] = (double)levels[q];
                level_vals = upload_vec(lv);
            }
            i64 *tab = upload_vec(levels);
            int *bad = pool.alloc<int>(1);
            PCR_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), stream));
            k_levels(ctx, X.rating, nnz, tab, T, X.level, bad);
            PCR_CUDA(cudaMemcpyAsync(h_counters, bad, sizeof(int), cudaMemcpyDeviceToHost, stream));
            sync();
            PCR_REQUIRE((h_counters[0] & 1) == 0, "a rating rounds to a level that is not in the level table");
            ratings_integer = (h_counters[0] & 2) == 0;
        }
        lap("levels");
        // ---- size classes, heavy scratch
        std::vector<int32_t> cls[3];
        std::vector<i64> hoff((size_t)d1, -1), hb, he;
        i64 htot = 0;
        use_tiles = T <= 8;
        // tiles: runs of consecutive users; geometry 0 takes users with len <= TILE_CAP, geometry 1 users with
        // TILE_CAP < len <= TILE_CAP_M, geometry 2 users with TILE_CAP_M < len <= TILE_CAP_L; anything longer is heavy
        struct Builder { std::vector<int32_t> first, num; i64 cur_first = -1, cur_nnz = 0, cur_users = 0, nnz = 0; i64 cap;
            void close() { if (cur_first >= 0 && cur_nnz > 0) { first.push_back((int32_t)cur_first); num.push_back((int32_t)cur_users); nnz += cur_nnz; }
                           cur_first = -1; cur_nnz = 0; cur_users = 0; }
            void add(i64 u, i64 len) { if (cur_first >= 0 && (cur_nnz + len > cap || cur_users + 1 > TILE_MAX_USERS)) close();
                                       if (cur_first < 0) cur_first = u; cur_nnz += len; cur_users += 1; } };
        Builder tb[3]; tb[0].cap = TILE_CAP; tb[1].cap = TILE_CAP_M; tb[2].cap = TILE_CAP_L;
        for (i64 u = 0; u < d1; ++u) {
            const i64 len = X.h_row_ptr[u + 1] - X.h_row_ptr[u];
            if (use_tiles && len <= TILE_CAP) { tb[1].close(); tb[2].close(); tb[0].add(u, len); continue; }
            if (use_tiles && T <= 5 && len <= TILE_CAP_M) { tb[0].close(); tb[2].close(); tb[1].add(u, len); continue; }   // T>5: smem
            if (use_tiles && T <= 5 && len <= TILE_CAP_L) { tb[0].close(); tb[1].close(); tb[2].add(u, len); continue; }
            tb[0].close(); tb[1].close(); tb[2].close();
            if (len == 0) continue;
            if (len <= S_CAP) cls[0].push_back((int32_t)u);
            else if (len <= L_CAP) cls[1].push_back((int32_t)u);
            else { cls[2].push_back((int32_t)u); hoff[u] = htot; htot += len + 1; hb.push_back(X.h_row_ptr[u]); he.push_back(X.h_row_ptr[u + 1]); }
        }
        for (int gq = 0; gq < 3; ++gq) {
            tb[gq].close();
            X.tiles[gq].n = (i64)tb[gq].first.size(); X.tiles[gq].nnz = tb[gq].nnz;
            X.tiles[gq].first = upload_vec(tb[gq].first); X.tiles[gq].nusers = upload_vec(tb[gq].num);
            std::vector<i64> te0(tb[gq].first.size()); std::vector<int32_t> tne(tb[gq].first.size());
            for (size_t q = 0; q < te0.size(); ++q) {
                te0[q] = X.h_row_ptr[tb[gq].first[q]];
                tne[q] = (int32_t)(X.h_row_ptr[(size_t)tb[gq].first[q] + tb[gq].num[q]] - te0[q]);
            }
            X.tiles[gq].e0 = upload_vec(te0); X.tiles[gq].ne = upload_vec(tne);
            sync();
        }
        for (int q = 0; q < 3; ++q) { X.n_cls[q] = (int)cls[q].size(); X.cls_users[q] = upload_vec(cls[q]); }
        X.heavy_off = upload_vec(hoff); X.heavy_total = htot;
        X.heavy_begin = upload_vec(hb); X.heavy_end = upload_vec(he);
        if (!cls[2].empty()) {            // work list of the heavy-user sort: the same chunks of 2048 ratings, any T
            std::vector<i64> soff; std::vector<int32_t> scu, sclo;
            i64 run = 0, maxlen = 0;
            for (size_t q = 0; q < cls[2].size(); ++q) {
                const i64 len = he[q] - hb[q];
                soff.push_back(run); run += len; maxlen = std::max(maxlen, len);
                for (i64 lo = 0; lo < len; lo += HEAVY_CHUNK) { scu.push_back((int32_t)q); sclo.push_back((int32_t)lo); }
            }
            hsort.n_users = (int)cls[2].size(); hsort.n_chunks = (int)scu.size();
            hsort.max_passes = 0;
            while (((i64)HEAVY_CHUNK << hsort.max_passes) < maxlen) ++hsort.max_passes;
            hsort.begin = X.heavy_begin; hsort.end = X.heavy_end;
            hsort.off = upload_vec(soff); hsort.chunk_user = upload_vec(scu); hsort.chunk_lo = upload_vec(sclo);
            hsort.tmp_s = pool.alloc<double>((size_t)run); hsort.tmp_pos = pool.alloc<int32_t>((size_t)run);
            sync();
        }
        heavy_chunked = use_tiles && !cls[2].empty();
        if (heavy_chunked) {
            std::vector<i64> hoff_h; std::vector<int32_t> cu, clo, c0;
            for (size_t q = 0; q < cls[2].size(); ++q) {
                hoff_h.push_back(hoff[cls[2][q]]);
                c0.push_back((int32_t)cu.size());
                for (i64 lo = 0; lo < he[q] - hb[q]; lo += HEAVY_CHUNK) { cu.push_back((int32_t)q); clo.push_back((int32_t)lo); }
            }
            c0.push_back((int32_t)cu.size());
            hv.n_users = (int)cls[2].size(); hv.n_chunks = (int)cu.size(); hv.htot = htot;
            hv.users = X.cls_users[2]; hv.begin = X.heavy_begin; hv.end = X.heavy_end;
            hv.off = upload_vec(hoff_h); hv.chunk_user = upload_vec(cu); hv.chunk_lo = upload_vec(clo); hv.chunk0 = upload_vec(c0);
            hv.ccnt = pool.alloc<int32_t>((size_t)hv.n_chunks * 8); hv.B = pool.alloc<int32_t>((size_t)hv.n_users * 9);
            hv.idx = pool.alloc<int32_t>((size_t)std::max(T - 1, 1) * (size_t)htot);
            hv.G = pool.alloc<double>((size_t)htot); hv.G2 = pool.alloc<double>((size_t)htot);
            hv.pos = pool.alloc<int32_t>((size_t)htot); hv.lo = pool.alloc<int32_t>((size_t)htot); hv.hi = pool.alloc<int32_t>((size_t)htot);
            hv.lev = pool.alloc<uint8_t>((size_t)htot);
            hv.csum = pool.alloc<double>((size_t)hv.n_chunks * 2);
            sync();
        } else {
            alloc_heavy_cta_scratch();
        }
        // ---- row-sum work units over the CSR
        {
            std::vector<int32_t> useg; std::vector<i64> ustart, supt;
            make_units(X.h_row_ptr, useg, ustart, supt);
            X.n_units = (i64)useg.size();
            X.un_seg = upload_vec(useg); X.un_start = upload_vec(ustart); X.seg_unit_ptr = upload_vec(supt);
            sync();
        }
        lap("classes, tiles, user units");
        // ---- CSC by item + its work units
        col_ptr = pool.alloc<i64>((size_t)d2 + 1);
        csc2csr = pool.alloc<int32_t>((size_t)nnz); csc_user = pool.alloc<int32_t>((size_t)nnz);
        k_build_csc(ctx, pool, X.item, X.user, nnz, d2, col_ptr, csc2csr, csc_user);
        std::vector<i64> h_col((size_t)d2 + 1);
        PCR_CUDA(cudaMemcpyAsync(h_col.data(), col_ptr, sizeof(i64) * ((size_t)d2 + 1), cudaMemcpyDeviceToHost, stream));
        sync();
        PCR_REQUIRE(h_col[d2] == nnz, "item id out of range [0, d2)");
        lap("CSC build (device)");
        // Work units of the item-major row sum, ordered USER-BLOCK-major: every unit only touches U rows of one block
        // of <= ~40 MB, so while the persistent grid walks the unit list the gathered rows stay L2-resident
        // (users ascend inside a column, so a column's entries of one block are contiguous).
        {
            const double blk_bytes = getenv("PRIMALCR_UBLOCK_MB") ? atof(getenv("PRIMALCR_UBLOCK_MB")) * 1e6 : 24e6;
            const double u_bytes = (double)d1 * ld * 8.0;
            int nb = (int)std::ceil(u_bytes / blk_bytes);
            // ... but never so many blocks that an (item, user block) unit averages fewer than ~32 ratings: with many
            // items (Yahoo / power-law shapes, d2 >= 500 k) the tiny units and their partial rows cost more than the L2
            // misses of a larger block (measured: 24 MB -> ~100 MB blocks, -8 % per iteration on both shapes)
            if (getenv("PRIMALCR_UBLOCK_MB") == nullptr) {
                const i64 nb_max = std::max<i64>(1, nnz / (32 * std::max<i64>(d2, 1)));
                if (nb > nb_max) nb = (int)nb_max;
            }
            if (nb < 1) nb = 1;
            if (nb > 64) nb = 64;
            const i64 bu = (d1 + nb - 1) / nb > 0 ? (d1 + nb - 1) / nb : 1;
            n_user_blocks = nb;
            std::vector<i64> bpos((size_t)d2 * (nb + 1));
            i64 *bpos_d = nullptr;
            bpos_d = (i64 *)pool.raw_alloc(sizeof(i64) * bpos.size());
            k_csc_block_bounds(ctx, col_ptr, csc_user, d2, nb, bu, bpos_d);
            PCR_CUDA(cudaMemcpyAsync(bpos.data(), bpos_d, sizeof(i64) * bpos.size(), cudaMemcpyDeviceToHost, stream));
            sync();
            pool.raw_free(bpos_d);
            std::vector<int32_t> cseg, cidx; std::vector<i64> cstart, cend, csup((size_t)d2 + 1, 0);
            for (int blk = 0; blk < nb; ++blk)
                for (i64 pcol = 0; pcol < d2; ++pcol) {
                    const i64 lo = bpos[(size_t)pcol * (nb + 1) + blk], hi = blk + 1 == nb ? h_col[pcol + 1] : bpos[(size_t)pcol * (nb + 1) + blk + 1];
                    // popular items get longer units so that no item has more than ~48 + nb partial sums to add up
                    const i64 collen = h_col[pcol + 1] - h_col[pcol];
                    const i64 chunk = std::max<i64>(ROWSUM_CHUNK, (collen + 47) / 48);
                    for (i64 bb = lo; bb < hi; bb += chunk) {
                        cseg.push_back((int32_t)pcol); cstart.push_back(bb); cend.push_back(std::min(bb + chunk, hi));
                        csup[pcol + 1] += 1;
                    }
                }
            n_cunits = (i64)cseg.size();
            for (i64 pcol = 0; pcol < d2; ++pcol) csup[pcol + 1] += csup[pcol];
            cidx.resize(cseg.size());
            std::vector<i64> fill(csup.begin(), csup.end() - 1);
            for (size_t uu = 0; uu < cseg.size(); ++uu) cidx[fill[cseg[uu]]++] = (int32_t)uu;
            cu_seg = upload_vec(cseg); cu_start = upload_vec(cstart); cu_end = upload_vec(cend);
            col_unit_ptr = upload_vec(csup); col_unit_idx = upload_vec(cidx);
            sync();
        }
        lap("item units (user blocks)");
        // ---- work buffers
        m = pool.alloc<double>((size_t)nnz); b = pool.alloc<double>((size_t)nnz); cbuf = pool.alloc<double>((size_t)nnz);
        meta.s = pool.alloc<double>((size_t)nnz); meta.pos = pool.alloc<int32_t>((size_t)nnz);
        meta.lev = pool.alloc<uint8_t>((size_t)nnz);
        meta.ub = pool.alloc<int32_t>((size_t)nnz); meta.lb = pool.alloc<int32_t>((size_t)nnz);
        meta.cnt_lo = pool.alloc<int32_t>((size_t)nnz); meta.cnt_hi = pool.alloc<int32_t>((size_t)nnz);
        meta.nnz = nnz;
        if (use_tiles) {     // level-major copy for the tile users
            meta.lm_s = pool.alloc<double>((size_t)nnz);
            meta.lm_w0 = pool.alloc<unsigned long long>((size_t)nnz); meta.lm_w1 = pool.alloc<unsigned long long>((size_t)nnz);
            if (T > 5) meta.lm_w2 = pool.alloc<unsigned long long>((size_t)nnz);
            meta.ulev = pool.alloc<uint16_t>((size_t)d1 * 8);
            PCR_CUDA(cudaMemsetAsync(meta.ulev, 0, sizeof(uint16_t) * (size_t)d1 * 8, stream));
        }
        const size_t vn = (size_t)d2 * ld, un = (size_t)d1 * ld;
        U = pool.alloc<double>(un);
        // V-side CG vectors: d2 rows padded to a multiple of the world size (equal row slices for reduce-scatter / all-gather;
        // the padding rows stay zero).  Sharded CG algebra pays off once a vector is large: 64 MB by default
        // (Netflix-shape 15.9 MB: one all-reduce is cheaper than reduce-scatter + 2 scalar all-reduces + all-gather).
        d2p = world > 1 ? (d2 + world - 1) / world * world : d2;
        vs_rows = d2p / std::max(world, 1); vs_row0 = (i64)rank * vs_rows;
        sharded_cg = world > 1 && (double)vn * 8.0 >= 64e6;
        if (const char *sc_env = getenv("PRIMALCR_SHARDED_CG")) sharded_cg = world > 1 && atoi(sc_env) != 0;
        const size_t vnp = (size_t)d2p * ld;
        g = pool.alloc<double>(vnp); delta = pool.alloc<double>(vnp); rr = pool.alloc<double>(vnp);
        p = pool.alloc<double>(vnp); Hp = pool.alloc<double>(vnp); V = pool.alloc<double>(vnp); Vnew = pool.alloc<double>(vnp);
        for (double *vec : {g, delta, rr, p, Hp, V, Vnew}) PCR_CUDA(cudaMemsetAsync(vec, 0, sizeof(double) * vnp, stream));
        partial = pool.alloc<double>((size_t)std::max(X.n_units, n_cunits) * ld);
        us.g = pool.alloc<double>(un); us.delta = pool.alloc<double>(un); us.rr = pool.alloc<double>(un);
        us.p = pool.alloc<double>(un); us.Hp = pool.alloc<double>(un); us.Unew = pool.alloc<double>(un);
        us.err = pool.alloc<double>((size_t)d1); us.step = pool.alloc<double>((size_t)d1);
        us.prev_obj = pool.alloc<double>((size_t)d1); us.obj_new = pool.alloc<double>((size_t)d1);
        us.loss = pool.alloc<double>((size_t)d1);
        us.cg_active = pool.alloc<uint8_t>((size_t)d1); us.ls_active = pool.alloc<uint8_t>((size_t)d1);
        us.skipped = pool.alloc<uint8_t>((size_t)d1);
        us.cg_its = pool.alloc<int32_t>((size_t)d1); us.ls_trials = pool.alloc<int32_t>((size_t)d1);
        k_fill(ctx, us.loss, d1, 0.0);
        has_pairs = pool.alloc<uint8_t>((size_t)d1);
        k_has_pairs(ctx, X, has_pairs);
        obj_item = pool.alloc<double>((size_t)X.n_pt);
        ensure_eval_buffers(X);
        sync();
        lap("work buffers");
        has_train = true;
    }

    void alloc_heavy_cta_scratch() {
        if (h_v != nullptr || X.heavy_total <= 0) return;
        const size_t htot = (size_t)X.heavy_total;
        h_v = pool.alloc<double>(htot); h_p1 = pool.alloc<double>(htot);
        h_p2 = pool.alloc<double>(htot); h_acc = pool.alloc<double>(htot);
        h_cnt = pool.alloc<int32_t>(htot);
    }
    // score-order window pointers / counters of the heavy users: only the stage entry points read them when the
    // chunk-parallel path is on (the sweeps use the level-major ranks)
    void ensure_heavy_windows() {
        if (!heavy_chunked || heavy_windows_valid || X.n_cls[2] == 0) return;
        alloc_heavy_cta_scratch();
        k_windows(ctx, 2, X.cls_users[2], X.n_cls[2], nullptr, X.row_ptr, meta, T, X.heavy_off, h_cnt);
        heavy_windows_valid = true;
    }
    i64 ev_cap_pt = 0, ev_cap_d1 = 0, ev_cap_nnz = 0;
    void ensure_eval_buffers(const DevCsr &C) {
        if (C.n_pt > ev_cap_pt) { ev_err_item = pool.alloc<i64>((size_t)C.n_pt); ev_cap_pt = C.n_pt; }
        if (C.d1 > ev_cap_d1 || ev_a == nullptr) {
            ev_err_user = pool.alloc<i64>((size_t)C.d1);
            ev_a = pool.alloc<double>((size_t)C.d1); ev_b = pool.alloc<double>((size_t)C.d1);
            ev_c = pool.alloc<double>((size_t)C.d1); ev_d = pool.alloc<double>((size_t)C.d1); ev_cap_d1 = C.d1;
        }
    }

    void set_test(i64 nnz, const i64 *row_ptr, const int32_t *item, const double *rating) {
        bind();
        PCR_REQUIRE(has_train, "load the training set first");
        PCR_REQUIRE(!has_test, "test set already loaded");
        build_csr_common(XT, d1, nnz, row_ptr, item, rating);
        ev_score_t = pool.alloc<double>((size_t)nnz);
        ensure_eval_buffers(XT);
        has_test = nnz > 0;
    }

    // host [rows x k] (compact) <-> device [rows x ld] (rows padded to 128-byte lines).  Download: one pitched copy, no
    // staging buffer (a temporary of a size the pool has not seen makes it grow, which is slow once NCCL enabled peer access)
    void put_matrix(const double *h, i64 rows, double *dst) {
        if (rows == 0) return;
        if (ld == k) {
            PCR_CUDA(cudaMemcpyAsync(dst, h, sizeof(double) * (size_t)rows * k, cudaMemcpyHostToDevice, stream));
        } else {
            // upload compact, pad on the device (measured: a pitched H2D copy of 480 k rows of 800 bytes runs at 7.7 GB/s,
            // 7x slower than one flat copy + the padding kernel; the download direction below is the opposite)
            double *tmp = (double *)pool.raw_alloc(sizeof(double) * (size_t)rows * k);
            PCR_CUDA(cudaMemcpyAsync(tmp, h, sizeof(double) * (size_t)rows * k, cudaMemcpyHostToDevice, stream));
            k_pad_copy(ctx, tmp, rows, k, ld, dst);
            PCR_CUDA(cudaStreamSynchronize(stream));
            pool.raw_free(tmp);
        }
    }
    void get_matrix(const double *src, i64 rows, double *h) {
        if (rows == 0) return;
        if (ld == k) {
            PCR_CUDA(cudaMemcpyAsync(h, src, sizeof(double) * (size_t)rows * k, cudaMemcpyDeviceToHost, stream));
        } else {
            PCR_CUDA(cudaMemcpy2DAsync(h, sizeof(double) * k, src, sizeof(double) * ld, sizeof(double) * k, (size_t)rows,
                                       cudaMemcpyDeviceToHost, stream));
        }
        PCR_CUDA(cudaStreamSynchronize(stream));
    }
    void set_factors(const double *Uh, const double *Vh) {
        bind();
        PCR_REQUIRE(has_train, "load the training set first");
        put_matrix(Uh, d1, U); put_matrix(Vh, d2, V);
        sync();
        has_factors = true; scores_valid = false; meta_valid = false; loss_matches_m = false; last_m_is_stale = false; v_trial_pending = false;
    }
    void get_factors(double *Uh, double *Vh) {
        bind();
        PCR_REQUIRE(has_factors, "no factors set");
        if (Uh) get_matrix(U, d1, Uh);
        if (Vh) get_matrix(V, d2, Vh);
        sync();
    }

    // ------------------------------------------------------------------ small helpers
    void read_slots(int n) {
        PCR_CUDA(cudaMemcpyAsync(h_slots, slots, sizeof(double) * n, cudaMemcpyDeviceToHost, stream));
        PCR_CUDA(cudaStreamSynchronize(stream));
    }
    int read_counter(int which) {
        PCR_CUDA(cudaMemcpyAsync(h_counters, us.counters, sizeof(int) * 2, cudaMemcpyDeviceToHost, stream));
        PCR_CUDA(cudaStreamSynchronize(stream));
        return h_counters[which];
    }
    void zero_counters() { PCR_CUDA(cudaMemsetAsync(us.counters, 0, sizeof(int) * 4, stream)); }
    void allreduce(double *buf, size_t n) {
        if (world <= 1) return;
        prof.begin("nccl_allreduce", stream, 0.0);
        int r = g_nccl.AllReduce(buf, buf, n, PCR_NCCL_FLOAT64, PCR_NCCL_SUM, comm, stream);
        prof.end(stream);
        if (r != 0) throw Error(PRIMALCR_ENCCL, std::string("ncclAllReduce failed: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "?"));
    }
    double pass_bytes(i64 n, i64 prows) const { return (double)n * (8.0 * k + 12.0) + 8.0 * k * (double)prows; }

    // scores of all training ratings under (Um, Vm): comp_m_new pcrpp.cpp:17-35
    void scores(const double *Um, const double *Vm, double *out, const uint8_t *active) {
        train_dots(Um, Vm, out, active);
    }
    // out[e] = P[user(e)] . Q[item(e)] over the training set
    void train_dots(const double *P, const double *Q, double *out, const uint8_t *active) {
        const double bytes = active ? 0.0 : pass_bytes(X.nnz, d1);
        k_dots_units(ctx, X.un_seg, X.un_start, nullptr, X.n_units, P, Q, X.item, ld, k, active, out, bytes);
    }
    // get_sorted_mm + window pointers for every (active) user
    void prepare(const double *sc, const uint8_t *active) {
        Ctx &hc = heavy_chunked ? ctx_aux : ctx;
        if (heavy_chunked) fork_aux();
        if (X.n_cls[2] > 0) {
            k_heavy_sort(hc, hsort, sc, meta.s, meta.pos);
            k_gather_level(hc, X.cls_users[2], X.n_cls[2], nullptr, X.row_ptr, X.level, meta);
            if (heavy_chunked) k_heavy_prepare(hc, hv, meta, T);
        }
        for (int gq = 0; gq < 3; ++gq) k_tile_prepare(ctx, X, gq, active, sc, meta, T);
        k_sort_users(ctx, 0, X.cls_users[0], X.n_cls[0], active, X.row_ptr, sc, X.level, meta);
        k_sort_users(ctx, 1, X.cls_users[1], X.n_cls[1], active, X.row_ptr, sc, X.level, meta);
        for (int q = 0; q < 3; ++q) {
            if (q == 2 && heavy_chunked) continue;
            k_windows(ctx, q, X.cls_users[q], X.n_cls[q], q == 2 ? nullptr : active, X.row_ptr, meta, T, X.heavy_off, h_cnt);
        }
        if (heavy_chunked) join_aux();
        heavy_windows_valid = false;
        meta_valid = true;
    }
    void sweep_coeff(int mode, const uint8_t *active, const double *bsrc) {
        if (heavy_chunked) { fork_aux(); k_heavy_sweep(ctx_aux, mode, hv, active, meta, bsrc, cbuf, nullptr, T); }
        for (int gq = 0; gq < 3; ++gq) k_tile_sweep(ctx, mode, X, gq, active, meta, bsrc, cbuf, nullptr, T);
        if (heavy_chunked) join_aux();
        for (int q = 0; q < 3; ++q) {
            if (q == 2 && heavy_chunked) continue;
            k_sweep_coeff(ctx, q, mode, X.cls_users[q], X.n_cls[q], active, X.row_ptr, meta, bsrc, cbuf, T, X.heavy_off, h_v, h_p1, h_acc);
        }
    }
    void sweep_obj(const uint8_t *active) {
        if (heavy_chunked) { fork_aux(); k_heavy_sweep(ctx_aux, 2, hv, active, meta, nullptr, nullptr, us.loss, T); }
        for (int gq = 0; gq < 3; ++gq) k_tile_sweep(ctx, 2, X, gq, active, meta, nullptr, nullptr, us.loss, T);
        if (heavy_chunked) join_aux();
        for (int q = 0; q < 3; ++q) {
            if (q == 2 && heavy_chunked) continue;
            k_sweep_obj(ctx, q, X.cls_users[q], X.n_cls[q], active, X.row_ptr, meta, us.loss, T, X.heavy_off, h_p1, h_p2, h_acc);
        }
    }
    // per-user losses of the current scores `sc` into us.loss (both solvers)
    void user_losses(const double *sc, const uint8_t *active) {
        if (cfg.solver == 2) sweep_obj(active);
        else { k_pairs(ctx, 2, X, active, sc, nullptr, nullptr, obj_item); k_pair_obj_users(ctx, X, active, obj_item, us.loss); }
    }
    // coefficient c_e (CSR order) into cbuf: mode 0 gradient, mode 1 Hv with b
    void coeffs(int mode, const uint8_t *active) {
        if (cfg.solver == 2) sweep_coeff(mode, active, b);
        else k_pairs(ctx, mode, X, active, m, b, cbuf, nullptr);
    }
    // full objective of (Um, Vm) given that us.loss holds the per-user losses:
    //   sum loss + lambda (||U||^2 + ||V||^2) / 2        pcrpp.cpp:410, pcr.cpp:41
    double total_objective(const double *Um, const double *Vm) {
        k_sum(ctx, us.loss, d1, red_partials, slots + 0);
        k_dot(ctx, Um, Um, d1 * ld, red_partials, slots + 1);
        k_dot(ctx, Vm, Vm, d2 * ld, red_partials, slots + 2);
        allreduce(slots, 2);
        read_slots(3);
        return h_slots[0] + cfg.lambda * (h_slots[1] + h_slots[2]) / 2.0;
    }
    // out = lambda*x + sum over the CSC of cbuf[e] * U[user(e)]    (V-side gradient / Hessian-vector product)
    void rowsum_items(const double *x, double *out) {
        const double bytes = pass_bytes(X.nnz, d2);
        if (world <= 1) {
            k_rowsum(ctx, cu_seg, cu_start, cu_end, n_cunits, col_unit_ptr, col_unit_idx, d2, csc_user, csc2csr, cbuf, U, ld, nullptr, partial,
                     cfg.lambda, x, out, 0, bytes, k);
        } else {
            k_rowsum(ctx, cu_seg, cu_start, cu_end, n_cunits, col_unit_ptr, col_unit_idx, d2, csc_user, csc2csr, cbuf, U, ld, nullptr, partial,
                     0.0, nullptr, out, 0, bytes, k);
            allreduce(out, (size_t)d2 * ld);
            k_axpby(ctx, out, 1.0, out, cfg.lambda, x, d2 * ld);
        }
    }
    // Sharded form (multi-GPU, large d2): this rank's partial sums over ALL items, then a reduce-scatter by item rows -- only
    // the rows [vs_row0, vs_row0 + vs_rows) of `out` hold the global sum (+ lambda x) afterwards
    void rowsum_items_rs(const double *x, double *out) {
        const double bytes = pass_bytes(X.nnz, d2);
        k_rowsum(ctx, cu_seg, cu_start, cu_end, n_cunits, col_unit_ptr, col_unit_idx, d2, csc_user, csc2csr, cbuf, U, ld, nullptr, partial,
                 0.0, nullptr, out, 0, bytes, k);
        const size_t off = (size_t)vs_row0 * ld, n = (size_t)vs_rows * ld;
        prof.begin("nccl_reduce_scatter", stream, 0.0);
        int r = g_nccl.ReduceScatter(out, out + off, n, PCR_NCCL_FLOAT64, PCR_NCCL_SUM, comm, stream);     // in place
        prof.end(stream);
        if (r != 0) throw Error(PRIMALCR_ENCCL, "ncclReduceScatter failed");
        k_axpby(ctx, out + off, 1.0, out + off, cfg.lambda, x + off, (i64)n);
    }
    void allgather_rows(double *vec) {      // every rank contributes its row slice of a d2p x ld vector
        prof.begin("nccl_all_gather", stream, 0.0);
        int r = g_nccl.AllGather(vec + (size_t)vs_row0 * ld, vec, (size_t)vs_rows * ld, PCR_NCCL_FLOAT64, comm, stream);   // in place
        prof.end(stream);
        if (r != 0) throw Error(PRIMALCR_ENCCL, "ncclAllGather failed");
    }
    // out[i] = lambda*x[i] + sum over user i of cbuf[e] * V[item(e)]   (U-side gradient / Hessian-vector product)
    void rowsum_users(const double *x, double *out, const uint8_t *active, int zero_if_empty) {
        k_rowsum(ctx, X.un_seg, X.un_start, nullptr, X.n_units, X.seg_unit_ptr, nullptr, d1, X.item, nullptr, cbuf, V, ld,
                 active, partial, cfg.lambda, x, out, zero_if_empty, active ? 0.0 : pass_bytes(X.nnz, d1), k);
    }

    void require_ready() {
        PCR_REQUIRE(has_train && has_factors, "engine needs a training set and factors");
        bind();
    }
    void ensure_scores() {
        if (scores_valid) return;
        scores(U, V, m, nullptr);
        scores_valid = true; meta_valid = false; loss_matches_m = false;
        last_m_is_stale = false;      // m is comp_m(U, V) again, no longer the scores of a rejected V trial
    }
    void ensure_meta() { ensure_scores(); if (cfg.solver == 2 && !meta_valid) prepare(m, nullptr); }

    // ------------------------------------------------------------------ stage entry points
    double objective_current() {   // objective_new(m, U, V) / objective(m, U, V)
        require_ready(); ensure_meta();
        user_losses(m, nullptr);
        return total_objective(U, V);
    }
    void grad_V(double *out_dev) { // obtain_g_new / obtain_g
        require_ready(); ensure_meta();
        coeffs(0, nullptr);
        rowsum_items(V, out_dev);
    }
    void hv_V(const double *a_dev, double *out_dev) {   // compute_Ha_new / compute_Ha
        require_ready(); ensure_meta();
        train_dots(U, a_dev, b, nullptr);
        coeffs(1, nullptr);
        rowsum_items(a_dev, out_dev);
    }

    // ------------------------------------------------------------------ update_V(_new)
    double update_V() {
        require_ready();
        const i64 vn = d2 * ld;
        // comp_m_new + get_sorted_mm (:417-418).  After an update_U the scores, the sorted state and the per-user losses of
        // every user's LAST line-search trial are exactly those of the committed (U, V) -- same kernels, same inputs --
        // so they are reused instead of being recomputed (update_U sets the three flags only when that holds).
        if (!(scores_valid && (cfg.solver != 2 || meta_valid))) {
            scores(U, V, m, nullptr); scores_valid = true; meta_valid = false; loss_matches_m = false;
            if (cfg.solver == 2) prepare(m, nullptr);
        }
        coeffs(0, nullptr);
        if (sharded_cg) rowsum_items_rs(V, g); else rowsum_items(V, g);
        // prev_obj = objective(m, U, V): m and the sorted state do not change during CG, so evaluate it now
        if (!loss_matches_m) user_losses(m, nullptr);
        const double prev_obj = total_objective(U, V);
        // ---- solve_delta(_new): pcrpp.cpp:335-358
        int its = 0;
        if (!sharded_cg) {
            k_fill(ctx, delta, vn, 0.0);
            k_axpby(ctx, rr, -1.0, g, 0.0, g, vn);
            k_axpby(ctx, p, 1.0, g, 0.0, g, vn);
            k_dot(ctx, rr, rr, vn, red_partials, slots + 0);
            read_slots(1);
            const double err = std::sqrt(h_slots[0]) * 0.01;
            for (int it = 1; it <= 10; ++it) {
                train_dots(U, p, b, nullptr);
                coeffs(1, nullptr);
                rowsum_items(p, Hp);
                ++its;
                // p.Hp, rr.p -> alpha (on the device) -> delta, rr updated -> rr.rr, rr.Hp: two fused passes, ONE host read
                k_cg_dots2(ctx, p, Hp, rr, vn, red_partials, slots + 0);
                k_cg_update(ctx, delta, rr, p, Hp, vn, slots + 0, red_partials, slots + 2);
                read_slots(4);
                const double prod_p_Hp = h_slots[0];
                if (std::sqrt(h_slots[2]) < err) break;
                const double beta = h_slots[3] / prod_p_Hp;
                k_axpby(ctx, p, -1.0, rr, beta, p, vn);
            }
        } else {
            // Same recurrences on this rank's ROW SLICE of the V-side vectors (g was reduce-scattered above): the dot
            // products are summed over ranks (2 x 2 scalars per iteration), the search direction p -- the only vector the
            // next N*k pass needs in full -- is all-gathered, delta once at the end.  The replicated CG algebra (15 passes
            // over d2 x k doubles per iteration, 1.4 ms at Yahoo-shape) shrinks by the world size.
            const i64 sn = vs_rows * ld; const size_t so = (size_t)vs_row0 * ld;
            double *g_s = g + so, *d_s = delta + so, *rr_s = rr + so, *p_s = p + so, *Hp_s = Hp + so;
            k_fill(ctx, d_s, sn, 0.0);
            k_axpby(ctx, rr_s, -1.0, g_s, 0.0, g_s, sn);
            k_axpby(ctx, p_s, 1.0, g_s, 0.0, g_s, sn);
            allgather_rows(p);
            k_dot(ctx, rr_s, rr_s, sn, red_partials, slots + 0);
            allreduce(slots, 1);
            read_slots(1);
            const double err = std::sqrt(h_slots[0]) * 0.01;
            for (int it = 1; it <= 10; ++it) {
                train_dots(U, p, b, nullptr);
                coeffs(1, nullptr);
                rowsum_items_rs(p, Hp);
                ++its;
                k_cg_dots2(ctx, p_s, Hp_s, rr_s, sn, red_partials, slots + 0);
                allreduce(slots, 2);
                k_cg_update(ctx, d_s, rr_s, p_s, Hp_s, sn, slots + 0, red_partials, slots + 2);
                allreduce(slots + 2, 2);
                read_slots(4);
                const double prod_p_Hp = h_slots[0];
                if (std::sqrt(h_slots[2]) < err) break;
                const double beta = h_slots[3] / prod_p_Hp;
                k_axpby(ctx, p_s, -1.0, rr_s, beta, p_s, sn);
                allgather_rows(p);
            }
            allgather_rows(delta);
        }
        // ---- line search: pcrpp.cpp:427-441
        double stepsize = cfg.stepsize, now_obj = prev_obj;
        int trials = 0, accepted = 0;
        for (int iter = 0; iter < 20; ++iter) {
            k_axpby(ctx, Vnew, 1.0, V, -stepsize, delta, vn);
            scores(U, Vnew, m, nullptr);
            if (cfg.solver == 2) prepare(m, nullptr);
            user_losses(m, nullptr);
            now_obj = total_objective(U, Vnew);
            ++trials;
            if (now_obj < prev_obj) { std::swap(V, Vnew); accepted = 1; break; }
            stepsize /= 2.0;
        }
        // m (and the sorted state) are those of the LAST trial, accepted or not -- as in the reference (:443)
        scores_valid = accepted != 0;   // if rejected, m belongs to a V that was thrown away
        loss_matches_m = true;
        counters.v_cg_iters = its; counters.v_ls_trials = trials; counters.v_ls_accepted = accepted;
        v_accepted = accepted;
        last_m_is_stale = !accepted;
        v_trial_pending = !accepted;
        return now_obj;
    }
    bool last_m_is_stale = false;
    // update_V rejected every trial and no update_U or write has run since: Vnew still holds the last trial's V.  A read-only
    // call may replace m (ensure_scores, primalcr_scores) in the meantime; update_U then rebuilds that trial's state from
    // (U, Vnew) -- the same kernels on the same inputs, so the same bits -- and consumes it as if nothing had been read.
    bool v_trial_pending = false;
    bool loss_matches_m = false;   // us.loss == per-user losses of the scores in m (set by update_V's last trial)

    // ------------------------------------------------------------------ update_U(_new), batched over users
    double update_U() {
        require_ready();
        if (v_trial_pending && !last_m_is_stale) {      // what update_V's last trial left behind, see there
            scores(U, Vnew, m, nullptr);
            if (cfg.solver == 2) prepare(m, nullptr);
            user_losses(m, nullptr);
            scores_valid = false; loss_matches_m = true; last_m_is_stale = true;
        }
        v_trial_pending = false;
        if (!scores_valid && !last_m_is_stale) { scores(U, V, m, nullptr); scores_valid = true; meta_valid = false; loss_matches_m = false; }
        if (cfg.solver == 2 && !meta_valid) prepare(m, nullptr);
        // m holds scores(U, V) for every user (not the scores of a rejected V trial): then what the line search leaves
        // behind is valid for the next update_V (see there)
        const bool m_covers_all_users = scores_valid && cfg.solver == 2;
        // gradient coefficients from m (stale m included, as precompute_ui / obtain_g_u do)
        coeffs(0, nullptr);
        // prev_obj: Primal-CR++ takes it from the same sorted state (objective_u_new :785); Primal-CR recomputes
        // the scores with the current (u_i, V) (compute_mm pcr.cpp:549), which differs only if V's search failed
        if (cfg.solver == 1 && last_m_is_stale) {
            train_dots(U, V, b, nullptr);
            user_losses(b, nullptr);
        } else if (!loss_matches_m) {
            user_losses(m, nullptr);      // else: us.loss still holds the losses of these very scores (last V trial)
        }
        loss_matches_m = false;
        rowsum_users(U, us.g, nullptr, 1);
        zero_counters();
        k_u_init(ctx, us, U, X.row_ptr, cfg.solver == 1 ? has_pairs : nullptr, d1, ld, cfg.lambda);
        int n_active = read_counter(0);
        // ---- solve_delta_u(_new): <= 10 CG iterations, each user leaves when its residual test fires
        for (int it = 1; it <= 10 && n_active > 0; ++it) {
            train_dots(us.p, V, b, us.cg_active);
            coeffs(1, us.cg_active);
            zero_counters();
            // unit partials of V_i^T c, then finalize (Hs = lambda s + sum) fused with the user's CG recurrences
            k_rowsum(ctx, X.un_seg, X.un_start, nullptr, X.n_units, X.seg_unit_ptr, nullptr, /*n_seg=*/0, X.item, nullptr, cbuf, V, ld,
                     us.cg_active, partial, cfg.lambda, us.p, us.Hp, 0, 0.0, k);
            k_u_finalize_cg(ctx, X.seg_unit_ptr, partial, us, d1, ld, k, cfg.lambda);
            n_active = read_counter(0);
        }
        // ---- line search: <= 20 halvings per user; the last trial is kept even if it never decreased (:814)
        zero_counters();
        int n_ls = -1;
        for (int trial = 0; trial < 20; ++trial) {
            k_u_ls_trial(ctx, us, U, d1, ld, cfg.stepsize, trial == 0);
            if (trial == 0) { n_ls = read_counter(1); if (n_ls == 0) break; }
            double *dst = cfg.solver == 2 ? m : b;
            train_dots(us.Unew, V, dst, us.ls_active);
            if (cfg.solver == 2) prepare(dst, us.ls_active);
            user_losses(dst, us.ls_active);
            zero_counters();
            k_u_ls_check(ctx, us, d1, ld, cfg.lambda, 0);
            n_ls = read_counter(1);
            if (n_ls == 0) break;
        }
        k_u_commit(ctx, us, U, d1, ld);
        // Primal-CR++: every user that moved went through trial 0 at least, so m / the sorted state / us.loss are those
        // of its last trial = its committed row; users that were skipped kept their row and their entries.
        scores_valid = m_covers_all_users; meta_valid = m_covers_all_users; loss_matches_m = m_covers_all_users;
        last_m_is_stale = false;
        // now_obj = sum_i obj_u + lambda/2 ||V||^2   (pcrpp.cpp:832-836)
        k_sum(ctx, us.obj_new, d1, red_partials, slots + 0);
        k_dot(ctx, V, V, d2 * ld, red_partials, slots + 1);
        allreduce(slots, 1);
        PCR_CUDA(cudaMemsetAsync(stats_dev, 0, sizeof(i64) * 8, stream));
        k_u_stats(ctx, us, X.row_ptr, d1, stats_dev);
        PCR_CUDA(cudaMemcpyAsync(h_stats, stats_dev, sizeof(i64) * 8, cudaMemcpyDeviceToHost, stream));
        read_slots(2);
        counters.u_cg_len_sum = h_stats[3]; counters.u_ls_len_sum = h_stats[4]; counters.u_skipped = h_stats[5];
        counters.u_cg_iters = h_stats[6]; counters.u_ls_trials = h_stats[7];
        return h_slots[0] + cfg.lambda / 2.0 * h_slots[1];
    }

    // U-side stage outputs for tests: g_u (d1 x ld) and obj_u from the current scores
    void grad_U_stage() {
        require_ready(); ensure_meta();
        coeffs(0, nullptr);
        user_losses(m, nullptr);
        rowsum_users(U, us.g, nullptr, 1);
        zero_counters();
        k_u_init(ctx, us, U, X.row_ptr, cfg.solver == 1 ? has_pairs : nullptr, d1, ld, cfg.lambda);
    }
    void hv_U_stage(const double *S_dev, double *out_dev) {
        require_ready(); ensure_meta();
        train_dots(S_dev, V, b, nullptr);
        coeffs(1, nullptr);
        rowsum_users(S_dev, out_dev, nullptr, 0);
    }

    // ------------------------------------------------------------------ compute_pairwise_error_ndcg util.cpp:434-542
    // pair errors from the sorted state (O(len * T)) are possible for the training set of Primal-CR++ whenever the
    // sorted state of the CURRENT scores exists and the ratings are integers (levels == exact ratings), T <= 8
    bool eval_sorted_ok(int which) const {
        return which == 0 && cfg.solver == 2 && scores_valid && meta_valid && ratings_integer && T <= 8;
    }
    // method: -1 automatic, 0 all-pairs kernel (the reference's O(len^2) loop util.cpp:467-479), 1 sorted-state count
    void eval(int which, double *err, double *ndcg, int method = -1, i64 *err_user_host = nullptr, double *ndcg_user_host = nullptr) {
        require_ready();
        DevCsr &C = which == 0 ? X : XT;
        PCR_REQUIRE(which == 0 || has_test, "no test set loaded");
        if (method == 1 && which == 0 && cfg.solver == 2 && ratings_integer && T <= 8) ensure_meta();
        PCR_REQUIRE(method != 1 || eval_sorted_ok(which), "sorted-state evaluation needs the Primal-CR++ training set with integer ratings and <= 8 levels");
        const bool sorted = method == 1 || (method < 0 && eval_sorted_ok(which));
        double *sc = which == 0 ? b : ev_score_t;
        if (which == 0 && scores_valid) sc = m;                      // m already holds U_i . V_j of the current factors
        else if (which == 0) train_dots(U, V, sc, nullptr);           // user-major units kernel (2x the generic one)
        else k_dots(ctx, U, C.user, V, C.item, C.nnz, ld, k, nullptr, sc, 0.0);
        if (sorted) {       // pair errors AND NDCG@k of every user from the sorted state, one kernel
            k_eval_sorted(ctx, C, meta, T, ev_err_user, level_vals, cfg.ndcg_k, ev_a, ev_b, ev_c, ev_d);
        } else {
            k_eval_pairs(ctx, C, sc, ev_err_item);
            k_eval_users(ctx, C, sc, ev_err_item, 0, cfg.ndcg_k, ev_a, ev_b, ev_c, ev_d);
        }
        if (err_user_host) {
            if (!sorted) k_eval_item_to_user(ctx, C, ev_err_item, ev_err_user);
            if (C.d1) PCR_CUDA(cudaMemcpyAsync(err_user_host, ev_err_user, sizeof(i64) * (size_t)C.d1, cudaMemcpyDeviceToHost, stream));
        }
        if (ndcg_user_host && C.d1) PCR_CUDA(cudaMemcpyAsync(ndcg_user_host, ev_b, sizeof(double) * (size_t)C.d1, cudaMemcpyDeviceToHost, stream));
        k_sum(ctx, ev_a, C.d1, red_partials, slots + 0);
        k_sum(ctx, ev_b, C.d1, red_partials, slots + 1);
        k_sum(ctx, ev_c, C.d1, red_partials, slots + 2);
        k_sum(ctx, ev_d, C.d1, red_partials, slots + 3);
        allreduce(slots, 4);
        read_slots(4);
        *err = h_slots[0] / h_slots[2];
        *ndcg = h_slots[1] / h_slots[3];
    }

    // ------------------------------------------------------------------ pcrpp() / pcr() driver with the reference's log lines
    static std::string fmt_g(double v) { char buf[64]; snprintf(buf, sizeof(buf), "%g", v); return buf; }
    void run(primalcr_log_fn log, void *lctx) {
        require_ready();
        auto say = [&](const std::string &s) { if (log && rank == 0) log(s.c_str(), lctx); };
        say(std::string(cfg.solver == 2 ? "running PrimalCR++ ndcg_k is " : "running PrimalCR ndcg_k is ") + std::to_string(cfg.ndcg_k));
        say("using " + std::to_string(cfg.threads) + " threads. ");          // verbatim, pcrpp.cpp:855 / pcr.cpp:631
        if (rank == 0) fprintf(stderr, "primalcr_b200: users sharded over %d GPU(s)\n", world);   // not part of the stdout contract
        double now_obj = objective_current();
        say("Iter 0 time 0 obj " + fmt_g(now_obj));
        auto do_eval = [&]() {
            if (!cfg.do_predict) return;
            double e = 0, n = 0;
            eval(0, &e, &n);
            say("(Training) pairwise error is " + fmt_g(e) + " and ndcg is " + fmt_g(n));
            if (has_test) { eval(1, &e, &n); say("(Testing) pairwise error is " + fmt_g(e) + " and ndcg is " + fmt_g(n)); }
        };
        do_eval();
        double total_time = 0.0;
        for (int iter = 1; iter <= cfg.maxiter; ++iter) {
            sync();
            auto t0 = std::chrono::steady_clock::now();
            update_V();
            now_obj = update_U();
            sync();
            total_time += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
            say("Iter " + std::to_string(iter) + " time " + fmt_g(total_time) + " obj " + fmt_g(now_obj));
            do_eval();
        }
    }
};

}  // namespace pcr

// ======================================================================================================
// C ABI
// ======================================================================================================
using pcr::Engine;

struct primalcr_engine { Engine *impl; };

#define API_BEGIN try {
#define API_END                                                                  \
    } catch (const pcr::Error &e) { pcr::g_last_error = e.what(); return e.code; } \
    catch (const std::exception &e) { pcr::g_last_error = e.what(); return PRIMALCR_EINTERNAL; } \
    return PRIMALCR_OK;
#define CHECK_E(e) if (!(e) || !(e)->impl) { pcr::g_last_error = "null engine"; return PRIMALCR_EARG; }

extern "C" {

const char *primalcr_last_error(void) { return pcr::g_last_error.c_str(); }
const char *primalcr_version(void) { return "primalcr_b200 0.2.0 (sm_100a)"; }

void primalcr_default_config(primalcr_config *cfg) {
    if (!cfg) return;
    cfg->solver = PRIMALCR_SOLVER_PCRPP; cfg->k = 10; cfg->lambda = 5000; cfg->stepsize = 1.0;
    cfg->maxiter = 10; cfg->ndcg_k = 10; cfg->do_predict = 1; cfg->device = 0; cfg->threads = 4;
}

int primalcr_create(primalcr_engine **out, const primalcr_config *cfg) {
    if (!out || !cfg) { pcr::g_last_error = "null argument"; return PRIMALCR_EARG; }
    *out = nullptr;
    API_BEGIN
    Engine *e = new Engine(*cfg);
    primalcr_engine *h = new primalcr_engine; h->impl = e; *out = h;
    API_END
}

void primalcr_destroy(primalcr_engine *e) {
    if (!e) return;
    try { delete e->impl; } catch (...) {}
    delete e;
}

int primalcr_set_levels(primalcr_engine *e, const int64_t *vals, int n) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(vals != nullptr, "null level table");
    std::vector<pcr::i64> v(vals, vals + (n > 0 ? n : 0));
    e->impl->set_levels(v.data(), n);
    API_END
}

int primalcr_set_train_csr(primalcr_engine *e, int64_t d1, int64_t d2, int64_t nnz, const int64_t *row_ptr,
                           const int32_t *item, const double *rating) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(row_ptr && (nnz == 0 || (item && rating)), "null CSR array");
    e->impl->set_train(d1, d2, nnz, (const pcr::i64 *)row_ptr, item, rating);
    API_END
}

int primalcr_set_test_csr(primalcr_engine *e, int64_t nnz, const int64_t *row_ptr, const int32_t *item, const double *rating) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(row_ptr && (nnz == 0 || (item && rating)), "null CSR array");
    e->impl->set_test(nnz, (const pcr::i64 *)row_ptr, item, rating);
    API_END
}

int primalcr_set_factors(primalcr_engine *e, const double *U, const double *V) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(U && V, "null factor matrix");
    e->impl->set_factors(U, V);
    API_END
}

int primalcr_get_factors(primalcr_engine *e, double *U, double *V) {
    CHECK_E(e) API_BEGIN
    e->impl->get_factors(U, V);
    API_END
}

int primalcr_nccl_unique_id(void *id128) {
    API_BEGIN
    PCR_REQUIRE(id128 != nullptr, "null id buffer");
    if (!pcr::g_nccl.load()) throw pcr::Error(PRIMALCR_ENCCL, "cannot load libnccl.so.2");
    pcr_ncclUniqueId id;
    int r = pcr::g_nccl.GetUniqueId(&id);
    if (r != 0) throw pcr::Error(PRIMALCR_ENCCL, "ncclGetUniqueId failed");
    memcpy(id128, &id, sizeof(id));
    API_END
}

int primalcr_comm_init(primalcr_engine *e, int rank, int world, const void *id128) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
    Engine *E = e->impl;
    E->bind();
    E->rank = rank; E->world = world;
    if (world > 1) {
        const pcr::CommKey key{E->cfg.device, rank, world};
        if (id128 == nullptr) {          // re-attach to this process's communicator
            std::lock_guard<std::mutex> lock(pcr::g_comm_mutex);
            auto it = pcr::g_comm_cache.find(key);
            PCR_REQUIRE(it != pcr::g_comm_cache.end(), "no cached communicator for this (device, rank, world): pass a ncclUniqueId");
            E->comm = it->second;
        } else {
            if (!pcr::g_nccl.load()) throw pcr::Error(PRIMALCR_ENCCL, "cannot load libnccl.so.2");
            pcr_ncclUniqueId id; memcpy(&id, id128, sizeof(id));
            int r = pcr::g_nccl.CommInitRank(&E->comm, world, id, rank);
            if (r != 0) throw pcr::Error(PRIMALCR_ENCCL, std::string("ncclCommInitRank failed: ") +
                                         (pcr::g_nccl.GetErrorString ? pcr::g_nccl.GetErrorString(r) : "?"));
            std::lock_guard<std::mutex> lock(pcr::g_comm_mutex);
            pcr::g_comm_cache[key] = E->comm;
        }
    }
    API_END
}

int primalcr_initial_objective(primalcr_engine *e, double *obj) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    E->scores_valid = false; E->meta_valid = false; E->v_trial_pending = false;
    const double o = E->objective_current();
    E->sync();
    if (obj) *obj = o;
    API_END
}

int primalcr_objective(primalcr_engine *e, double *obj) {
    CHECK_E(e) API_BEGIN
    const double o = e->impl->objective_current();
    e->impl->sync();
    if (obj) *obj = o;
    API_END
}

int primalcr_update_V(primalcr_engine *e, double *now_obj) {
    CHECK_E(e) API_BEGIN
    const double o = e->impl->update_V();
    e->impl->sync();
    if (now_obj) *now_obj = o;
    API_END
}

int primalcr_update_U(primalcr_engine *e, double *now_obj) {
    CHECK_E(e) API_BEGIN
    const double o = e->impl->update_U();
    e->impl->sync();
    if (now_obj) *now_obj = o;
    API_END
}

int primalcr_outer_iteration(primalcr_engine *e, double *now_obj) {
    CHECK_E(e) API_BEGIN
    e->impl->update_V();
    const double o = e->impl->update_U();
    e->impl->sync();
    if (now_obj) *now_obj = o;
    API_END
}

int primalcr_eval(primalcr_engine *e, int which, double *pairwise_error, double *ndcg) {
    CHECK_E(e) API_BEGIN
    double a = 0, b = 0;
    e->impl->eval(which, &a, &b);
    e->impl->sync();
    if (pairwise_error) *pairwise_error = a;
    if (ndcg) *ndcg = b;
    API_END
}

int primalcr_eval_error_counts(primalcr_engine *e, int which, int method, int64_t *err_per_user, double *ndcg_per_user,
                               double *pairwise_error, double *ndcg) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(method == 0 || method == 1, "method must be 0 (all pairs) or 1 (sorted state)");
    double a = 0, b = 0;
    e->impl->eval(which, &a, &b, method, (pcr::i64 *)err_per_user, ndcg_per_user);
    e->impl->sync();
    if (pairwise_error) *pairwise_error = a;
    if (ndcg) *ndcg = b;
    API_END
}

int primalcr_run(primalcr_engine *e, primalcr_log_fn log, void *ctx) {
    CHECK_E(e) API_BEGIN
    e->impl->run(log, ctx);
    e->impl->sync();
    API_END
}

int primalcr_get_counters(primalcr_engine *e, primalcr_counters *out) {
    CHECK_E(e) API_BEGIN
    PCR_REQUIRE(out != nullptr, "null output");
    *out = e->impl->counters;
    API_END
}

// ---- stage entry points ---------------------------------------------------------------------------
int primalcr_scores(primalcr_engine *e, double *m_out) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    E->scores(E->U, E->V, E->m, nullptr); E->scores_valid = true; E->meta_valid = false; E->last_m_is_stale = false; E->loss_matches_m = false;
    if (m_out && E->X.nnz) PCR_CUDA(cudaMemcpyAsync(m_out, E->m, sizeof(double) * (size_t)E->X.nnz, cudaMemcpyDeviceToHost, E->stream));
    E->sync();
    API_END
}

int primalcr_set_scores(primalcr_engine *e, const double *m) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    PCR_REQUIRE(m != nullptr || E->X.nnz == 0, "null scores");
    if (E->X.nnz) PCR_CUDA(cudaMemcpyAsync(E->m, m, sizeof(double) * (size_t)E->X.nnz, cudaMemcpyHostToDevice, E->stream));
    E->sync();
    E->scores_valid = true; E->meta_valid = false; E->last_m_is_stale = false; E->loss_matches_m = false; E->v_trial_pending = false;
    API_END
}

int primalcr_num_levels(primalcr_engine *e) {
    if (!e || !e->impl) return PRIMALCR_EARG;
    return e->impl->T;
}

int primalcr_sort_segments(primalcr_engine *e, double *sorted, int32_t *perm, int32_t *level, int32_t *ub, int32_t *lb,
                           int32_t *cnt_lo, int32_t *cnt_hi) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    PCR_REQUIRE(E->cfg.solver == 2, "sorted state exists only for Primal-CR++");
    E->ensure_scores();
    E->prepare(E->m, nullptr);
    E->ensure_heavy_windows();
    E->sync();
    const size_t n = (size_t)E->X.nnz;
    if (n) {
        if (sorted) PCR_CUDA(cudaMemcpy(sorted, E->meta.s, sizeof(double) * n, cudaMemcpyDeviceToHost));
        if (ub) PCR_CUDA(cudaMemcpy(ub, E->meta.ub, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
        if (lb) PCR_CUDA(cudaMemcpy(lb, E->meta.lb, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
        if (cnt_lo) PCR_CUDA(cudaMemcpy(cnt_lo, E->meta.cnt_lo, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
        if (cnt_hi) PCR_CUDA(cudaMemcpy(cnt_hi, E->meta.cnt_hi, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
        if (perm) {
            std::vector<int32_t> pos(n);
            PCR_CUDA(cudaMemcpy(pos.data(), E->meta.pos, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
            for (pcr::i64 u = 0; u < E->d1; ++u)
                for (pcr::i64 q = E->X.h_row_ptr[u]; q < E->X.h_row_ptr[u + 1]; ++q) perm[q] = pos[q] - (int32_t)E->X.h_row_ptr[u];
        }
        if (level) {
            std::vector<uint8_t> lv(n);
            PCR_CUDA(cudaMemcpy(lv.data(), E->meta.lev, n, cudaMemcpyDeviceToHost));
            for (size_t q = 0; q < n; ++q) level[q] = lv[q];
        }
    }
    API_END
}

int primalcr_level_counts(primalcr_engine *e, int32_t *cnt_left, int32_t *cnt_right) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    PCR_REQUIRE(E->cfg.solver == 2, "sorted state exists only for Primal-CR++");
    E->ensure_meta();
    E->ensure_heavy_windows();
    const size_t n = (size_t)E->X.nnz * E->T;
    int32_t *dl = nullptr, *dr = nullptr;
    dl = (int32_t *)E->pool.raw_alloc(sizeof(int32_t) * (n ? n : 1));
    dr = (int32_t *)E->pool.raw_alloc(sizeof(int32_t) * (n ? n : 1));
    pcr::k_level_counts(E->ctx, E->X.row_ptr, E->d1, E->meta, E->T, dl, dr);
    E->sync();
    if (n && cnt_left) PCR_CUDA(cudaMemcpy(cnt_left, dl, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    if (n && cnt_right) PCR_CUDA(cudaMemcpy(cnt_right, dr, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
    E->pool.raw_free(dl); E->pool.raw_free(dr);
    API_END
}

int primalcr_grad_V(primalcr_engine *e, double *g_out) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->grad_V(E->g);
    if (g_out) E->get_matrix(E->g, E->d2, g_out);
    E->sync();
    API_END
}

int primalcr_hv_V(primalcr_engine *e, const double *a, double *Ha_out) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    PCR_REQUIRE(a != nullptr, "null direction");
    E->put_matrix(a, E->d2, E->p);
    E->hv_V(E->p, E->Hp);
    if (Ha_out) E->get_matrix(E->Hp, E->d2, Ha_out);
    E->sync();
    API_END
}

int primalcr_grad_U(primalcr_engine *e, double *g_out, double *obj_u_out) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->grad_U_stage();
    if (g_out) E->get_matrix(E->us.g, E->d1, g_out);
    if (obj_u_out && E->d1) PCR_CUDA(cudaMemcpyAsync(obj_u_out, E->us.prev_obj, sizeof(double) * (size_t)E->d1, cudaMemcpyDeviceToHost, E->stream));
    E->sync();
    API_END
}

int primalcr_hv_U(primalcr_engine *e, const double *S, double *HS_out) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->require_ready();
    PCR_REQUIRE(S != nullptr, "null direction");
    E->put_matrix(S, E->d1, E->us.p);
    E->hv_U_stage(E->us.p, E->us.Hp);
    if (HS_out) E->get_matrix(E->us.Hp, E->d1, HS_out);
    E->sync();
    API_END
}

// ---- measurement ------------------------------------------------------------------------------------
void *primalcr_stream(primalcr_engine *e) { return (e && e->impl) ? (void *)e->impl->stream : nullptr; }
int64_t primalcr_launch_count(primalcr_engine *e) { return (e && e->impl) ? e->impl->prof.launches : -1; }
int primalcr_profile_enable(primalcr_engine *e, int on) {
    CHECK_E(e) API_BEGIN
    e->impl->bind(); e->impl->sync();
    e->impl->prof.enabled = on != 0;
    API_END
}
int primalcr_profile_reset(primalcr_engine *e) {
    CHECK_E(e) API_BEGIN
    e->impl->bind(); e->impl->sync();
    e->impl->prof.reset();
    API_END
}
int primalcr_profile_count(primalcr_engine *e) { return (e && e->impl) ? (int)e->impl->prof.acc.size() : -1; }
int primalcr_profile_get(primalcr_engine *e, int idx, const char **name, double *total_ms, int64_t *launches, double *bytes) {
    CHECK_E(e) API_BEGIN
    Engine *E = e->impl;
    E->bind(); E->sync();
    PCR_REQUIRE(idx >= 0 && idx < (int)E->prof.acc.size(), "profile index out of range");
    const auto &a = E->prof.acc[idx];
    if (name) *name = a.name.c_str();
    if (total_ms) *total_ms = a.ms;
    if (launches) *launches = a.launches;
    if (bytes) *bytes = a.bytes;
    API_END
}
int64_t primalcr_device_bytes(primalcr_engine *e) { return (e && e->impl) ? e->impl->pool.bytes : -1; }

// ---- prediction (pmf-predict.cpp:57-64) ---------------------------------------------------------------
int primalcr_predict(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int32_t *user,
                     const int32_t *item, int64_t n, double *out, int device) {
    API_BEGIN
    PCR_REQUIRE(U && V && (n == 0 || (user && item && out)) && k >= 1 && d1 >= 0 && d2 >= 0, "bad argument");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw pcr::Error(PRIMALCR_ECUDA, "no CUDA device available: libprimalcr_b200 has no CPU fallback");
    for (int64_t t = 0; t < n; ++t)
        PCR_REQUIRE(user[t] >= 0 && user[t] < d1 && item[t] >= 0 && item[t] < d2, "user/item id out of range");
    PCR_CUDA(cudaSetDevice(device));
    const int ld = pcr::ceil16(k);
    pcr::DevPool pool; pcr::Profiler prof; pcr::Ctx ctx;
    cudaDeviceProp prop; PCR_CUDA(cudaGetDeviceProperties(&prop, device));
    cudaStream_t st; PCR_CUDA(cudaStreamCreate(&st));
    ctx.stream = st; ctx.prof = &prof; ctx.sms = prop.multiProcessorCount; ctx.ticket = pool.alloc<unsigned long long>(1);
    double *Uc = pool.alloc<double>((size_t)d1 * k), *Vc = pool.alloc<double>((size_t)d2 * k);
    double *Ud = pool.alloc<double>((size_t)d1 * ld), *Vd = pool.alloc<double>((size_t)d2 * ld), *od = pool.alloc<double>((size_t)n);
    int32_t *ud = pool.alloc<int32_t>((size_t)n), *id = pool.alloc<int32_t>((size_t)n);
    PCR_CUDA(cudaMemcpyAsync(Uc, U, sizeof(double) * (size_t)d1 * k, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(Vc, V, sizeof(double) * (size_t)d2 * k, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(ud, user, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(id, item, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    pcr::k_pad_copy(ctx, Uc, d1, k, ld, Ud); pcr::k_pad_copy(ctx, Vc, d2, k, ld, Vd);
    pcr::k_dots(ctx, Ud, ud, Vd, id, n, ld, k, nullptr, od, 0.0);
    if (n) PCR_CUDA(cudaMemcpyAsync(out, od, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    PCR_CUDA(cudaStreamSynchronize(st));
    cudaStreamDestroy(st);
    API_END
}

// ---- top-N recommendation ---------------------------------------------------------------------------------------
// the exclusion CSR of primalcr_recommend / primalcr_rank_heldout: both pointers or neither, ascending rows -> its nnz
static int64_t check_exclusion(int64_t d1, int64_t d2, const int64_t *excl_row_ptr, const int32_t *excl_item) {
    if (!excl_row_ptr) return 0;
    const std::string err = pcrhost::csr_error("exclusion", d1, d2, excl_row_ptr, excl_item, true);
    PCR_REQUIRE(err.empty(), err);
    return excl_row_ptr[d1];
}

// exclusion CSR to the device (both nullptr when there is none)
static void upload_exclusion(pcr::DevPool &pool, cudaStream_t st, int64_t d1, const int64_t *excl_row_ptr,
                             const int32_t *excl_item, int64_t ex_nnz, int64_t *&exp_d, int32_t *&exi_d) {
    exp_d = nullptr; exi_d = nullptr;
    if (!excl_row_ptr) return;
    exp_d = pool.alloc<int64_t>((size_t)d1 + 1); exi_d = pool.alloc<int32_t>((size_t)ex_nnz);
    PCR_CUDA(cudaMemcpyAsync(exp_d, excl_row_ptr, sizeof(int64_t) * ((size_t)d1 + 1), cudaMemcpyHostToDevice, st));
    if (ex_nnz) PCR_CUDA(cudaMemcpyAsync(exi_d, excl_item, sizeof(int32_t) * (size_t)ex_nnz, cudaMemcpyHostToDevice, st));
}

int primalcr_recommend(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int64_t *excl_row_ptr,
                       const int32_t *excl_item, const int32_t *users, int64_t n_users, int topn, int32_t *items_out,
                       double *scores_out, int device) {
    API_BEGIN
    PCR_REQUIRE(k >= 1 && k <= 256, "rank k out of range [1, 256]");
    PCR_REQUIRE(topn >= 1 && topn <= 256, "topn out of range [1, 256]");
    PCR_REQUIRE(d1 >= 0 && d2 >= 0 && d1 <= INT32_MAX && d2 <= INT32_MAX, "d1 / d2 out of range");
    PCR_REQUIRE((U || d1 == 0) && (V || d2 == 0), "null factor matrix");
    PCR_REQUIRE(n_users >= 0 && (users || n_users == d1), "users == NULL requires n_users == d1");
    PCR_REQUIRE(n_users == 0 || items_out, "null items_out");
    PCR_REQUIRE((excl_row_ptr == nullptr) == (excl_item == nullptr), "excl_row_ptr and excl_item must both be given or both be NULL");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw pcr::Error(PRIMALCR_ECUDA, "no CUDA device available: libprimalcr_b200 has no CPU fallback");
    PCR_REQUIRE(device >= 0 && device < ndev, "bad device ordinal");
    // every id the kernel reads through is checked here, before anything runs
    bool bad_user = false;
    if (users) {
#pragma omp parallel for reduction(|| : bad_user) schedule(static)
        for (int64_t t = 0; t < n_users; ++t) bad_user = bad_user || users[t] < 0 || users[t] >= d1;
    }
    PCR_REQUIRE(!bad_user, "user id out of range");
    const int64_t ex_nnz = check_exclusion(d1, d2, excl_row_ptr, excl_item);
    if (n_users == 0) return PRIMALCR_OK;
    PCR_CUDA(cudaSetDevice(device));
    pcr::DevPool pool; pcr::Profiler prof; pcr::Ctx ctx;
    // declared after the pool, so on every exit the stream is drained and destroyed before the buffers are freed
    struct StreamGuard { cudaStream_t s = nullptr; ~StreamGuard() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } } sg;
    PCR_CUDA(cudaStreamCreateWithFlags(&sg.s, cudaStreamNonBlocking));
    cudaStream_t st = sg.s;
    cudaDeviceProp prop; PCR_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx.stream = st; ctx.prof = &prof; ctx.sms = prop.multiProcessorCount; ctx.ticket = nullptr;
    double *Ud = pool.alloc<double>((size_t)d1 * k), *Vd = pool.alloc<double>((size_t)d2 * k);
    int32_t *ud = pool.alloc<int32_t>((size_t)n_users), *itd = pool.alloc<int32_t>((size_t)n_users * topn);
    double *scd = scores_out ? pool.alloc<double>((size_t)n_users * topn) : nullptr;
    int64_t *exp_d; int32_t *exi_d;
    if (d1) PCR_CUDA(cudaMemcpyAsync(Ud, U, sizeof(double) * (size_t)d1 * k, cudaMemcpyHostToDevice, st));
    if (d2) PCR_CUDA(cudaMemcpyAsync(Vd, V, sizeof(double) * (size_t)d2 * k, cudaMemcpyHostToDevice, st));
    if (users) PCR_CUDA(cudaMemcpyAsync(ud, users, sizeof(int32_t) * (size_t)n_users, cudaMemcpyHostToDevice, st));
    else pcr::k_iota32(ctx, ud, n_users);
    upload_exclusion(pool, st, d1, excl_row_ptr, excl_item, ex_nnz, exp_d, exi_d);
    pcr::k_topn(ctx, Ud, Vd, d2, k, (const pcr::i64 *)exp_d, exi_d, ud, n_users, topn, itd, scd);
    PCR_CUDA(cudaMemcpyAsync(items_out, itd, sizeof(int32_t) * (size_t)n_users * topn, cudaMemcpyDeviceToHost, st));
    if (scores_out) PCR_CUDA(cudaMemcpyAsync(scores_out, scd, sizeof(double) * (size_t)n_users * topn, cudaMemcpyDeviceToHost, st));
    PCR_CUDA(cudaStreamSynchronize(st));
    API_END
}

// ---- held-out ranking evaluation --------------------------------------------------------------------------------
int primalcr_rank_heldout(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int64_t *excl_row_ptr,
                          const int32_t *excl_item, const int64_t *ho_row_ptr, const int32_t *ho_item, int32_t *rank_out,
                          double *score_out, int device) {
    API_BEGIN
    PCR_REQUIRE(k >= 1 && k <= 256, "rank k out of range [1, 256]");
    PCR_REQUIRE(d1 >= 0 && d2 >= 0 && d1 <= INT32_MAX && d2 <= INT32_MAX, "d1 / d2 out of range");
    PCR_REQUIRE((U || d1 == 0) && (V || d2 == 0), "null factor matrix");
    PCR_REQUIRE(ho_row_ptr, "null ho_row_ptr");
    PCR_REQUIRE((excl_row_ptr == nullptr) == (excl_item == nullptr), "excl_row_ptr and excl_item must both be given or both be NULL");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw pcr::Error(PRIMALCR_ECUDA, "no CUDA device available: libprimalcr_b200 has no CPU fallback");
    PCR_REQUIRE(device >= 0 && device < ndev, "bad device ordinal");
    // every id the kernel reads through is checked here, before anything runs
    const int64_t nnz = ho_row_ptr[d1];
    PCR_REQUIRE(nnz == 0 || (ho_item && rank_out), "null ho_item or rank_out");
    const std::string err = pcrhost::csr_error("held-out", d1, d2, ho_row_ptr, ho_item, false);
    PCR_REQUIRE(err.empty(), err);
    const int64_t ex_nnz = check_exclusion(d1, d2, excl_row_ptr, excl_item);
    if (nnz == 0) return PRIMALCR_OK;
    // units: a user and at most RANK_UNIT consecutive entries of its row; they tile [0, nnz) in order
    std::vector<int32_t> unit_user;
    std::vector<int64_t> unit_beg;
    for (int64_t u = 0; u < d1; ++u)
        for (int64_t e = ho_row_ptr[u]; e < ho_row_ptr[u + 1]; e += pcr::RANK_UNIT) { unit_user.push_back((int32_t)u); unit_beg.push_back(e); }
    unit_beg.push_back(nnz);
    const int64_t n_units = (int64_t)unit_user.size();
    PCR_CUDA(cudaSetDevice(device));
    pcr::DevPool pool; pcr::Profiler prof; pcr::Ctx ctx;
    // declared after the pool, so on every exit the stream is drained and destroyed before the buffers are freed
    struct StreamGuard { cudaStream_t s = nullptr; ~StreamGuard() { if (s) { cudaStreamSynchronize(s); cudaStreamDestroy(s); } } } sg;
    PCR_CUDA(cudaStreamCreateWithFlags(&sg.s, cudaStreamNonBlocking));
    cudaStream_t st = sg.s;
    cudaDeviceProp prop; PCR_CUDA(cudaGetDeviceProperties(&prop, device));
    ctx.stream = st; ctx.prof = &prof; ctx.sms = prop.multiProcessorCount; ctx.ticket = nullptr;
    double *Ud = pool.alloc<double>((size_t)d1 * k), *Vd = pool.alloc<double>((size_t)d2 * k);
    int32_t *hid = pool.alloc<int32_t>((size_t)nnz), *rkd = pool.alloc<int32_t>((size_t)nnz);
    int32_t *uud = pool.alloc<int32_t>((size_t)n_units);
    int64_t *ubd = pool.alloc<int64_t>((size_t)n_units + 1);
    double *scd = score_out ? pool.alloc<double>((size_t)nnz) : nullptr;
    int64_t *exp_d; int32_t *exi_d;
    if (d1) PCR_CUDA(cudaMemcpyAsync(Ud, U, sizeof(double) * (size_t)d1 * k, cudaMemcpyHostToDevice, st));
    if (d2) PCR_CUDA(cudaMemcpyAsync(Vd, V, sizeof(double) * (size_t)d2 * k, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(hid, ho_item, sizeof(int32_t) * (size_t)nnz, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(uud, unit_user.data(), sizeof(int32_t) * (size_t)n_units, cudaMemcpyHostToDevice, st));
    PCR_CUDA(cudaMemcpyAsync(ubd, unit_beg.data(), sizeof(int64_t) * ((size_t)n_units + 1), cudaMemcpyHostToDevice, st));
    upload_exclusion(pool, st, d1, excl_row_ptr, excl_item, ex_nnz, exp_d, exi_d);
    pcr::k_rank_heldout(ctx, Ud, Vd, d2, k, (const pcr::i64 *)exp_d, exi_d, hid, uud, (const pcr::i64 *)ubd, n_units, rkd, scd);
    PCR_CUDA(cudaMemcpyAsync(rank_out, rkd, sizeof(int32_t) * (size_t)nnz, cudaMemcpyDeviceToHost, st));
    if (score_out) PCR_CUDA(cudaMemcpyAsync(score_out, scd, sizeof(double) * (size_t)nnz, cudaMemcpyDeviceToHost, st));
    PCR_CUDA(cudaStreamSynchronize(st));
    API_END
}

int primalcr_rank_metrics(int64_t d1, int64_t d2, const int64_t *excl_row_ptr, const int32_t *excl_item,
                          const int64_t *ho_row_ptr, const int32_t *ho_item, const double *ho_rating, const int32_t *rank,
                          double min_rating, const int32_t *cutoffs, int n_cutoffs, double *recall, double *precision,
                          double *ndcg, double *mrr, double *auc, int64_t *n_users) {
    API_BEGIN
    pcrhost::RankMetrics m;
    const std::string err = pcrhost::rank_metrics(d1, d2, excl_row_ptr, excl_item, ho_row_ptr, ho_item, ho_rating, rank,
                                                  min_rating, cutoffs, n_cutoffs, m);
    PCR_REQUIRE(err.empty(), err);
    for (int c = 0; c < n_cutoffs; ++c) {
        if (recall) recall[c] = m.recall[(size_t)c];
        if (precision) precision[c] = m.precision[(size_t)c];
        if (ndcg) ndcg[c] = m.ndcg[(size_t)c];
    }
    if (mrr) *mrr = m.mrr;
    if (auc) *auc = m.auc;
    if (n_users) *n_users = m.n_users;
    API_END
}

// ---- host loader ------------------------------------------------------------------------------------------
struct primalcr_dataset { pcrhost::DataDir d; };

int primalcr_load_dir(const char *data_dir, int threads, primalcr_dataset **out) {
    API_BEGIN
    PCR_REQUIRE(data_dir && out, "null argument");
#ifdef _OPENMP
    if (threads > 0) omp_set_num_threads(threads);
#endif
    primalcr_dataset *ds = new primalcr_dataset;
    try { ds->d = pcrhost::load_dir(data_dir); }
    catch (const std::exception &ex) { delete ds; throw pcr::Error(PRIMALCR_EARG, ex.what()); }
    *out = ds;
    API_END
}
int primalcr_dataset_info(const primalcr_dataset *ds, int64_t *d1, int64_t *d2, int64_t *nnz_train, int64_t *nnz_test) {
    API_BEGIN
    PCR_REQUIRE(ds != nullptr, "null dataset");
    if (d1) *d1 = ds->d.train.d1;
    if (d2) *d2 = ds->d.train.d2;
    if (nnz_train) *nnz_train = ds->d.train.nnz;
    if (nnz_test) *nnz_test = ds->d.test.nnz;
    API_END
}
int primalcr_dataset_csr(const primalcr_dataset *ds, int which, const int64_t **row_ptr, const int32_t **item, const double **rating) {
    API_BEGIN
    PCR_REQUIRE(ds != nullptr && (which == 0 || which == 1), "bad argument");
    const pcrhost::Csr &c = which == 0 ? ds->d.train : ds->d.test;
    if (row_ptr) *row_ptr = c.row_ptr.data();
    if (item) *item = c.item.data();
    if (rating) *rating = c.rating.data();
    API_END
}
void primalcr_dataset_free(primalcr_dataset *ds) { delete ds; }

// ---- host utilities -----------------------------------------------------------------------------------
int primalcr_write_text_matrix(const char *path, const double *M, int64_t rows, int k) {
    API_BEGIN
    PCR_REQUIRE(path && (M || rows == 0) && rows >= 0 && k >= 1, "bad argument");
    if (!pcrhost::write_text_matrix(path, M, (long)rows, k)) throw pcr::Error(PRIMALCR_EARG, std::string("cannot open ") + path);
    API_END
}

void primalcr_reference_init(double *out, int64_t n, int64_t k) {
    // initial() util.cpp:80-93: a default-constructed std::default_random_engine per call
    std::default_random_engine generator;
    std::normal_distribution<double> distribution(0.0, 1.0);
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j < k; ++j) out[i * k + j] = distribution(generator);
}

}  // extern "C"
