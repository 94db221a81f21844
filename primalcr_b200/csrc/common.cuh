// common.cuh -- shared declarations of libprimalcr_b200 (sm_100a only; no CPU fallback).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <map>
#include <stdexcept>

namespace pcr {

typedef long long i64;

// leading dimension of every factor-shaped array: rows start on 128-byte lines (a 128-byte row chunk never straddles two)
inline int ceil16(int k) { return (k + 15) & ~15; }

// ------------------------------------------------------------------ errors
struct Error : public std::runtime_error {
    int code;
    Error(int c, const std::string &w) : std::runtime_error(w), code(c) {}
};

#define PCR_CUDA(call)                                                                         \
    do {                                                                                       \
        cudaError_t _e = (call);                                                               \
        if (_e != cudaSuccess) {                                                               \
            char _b[512];                                                                      \
            snprintf(_b, sizeof(_b), "CUDA error %s at %s:%d: %s", cudaGetErrorName(_e),       \
                     __FILE__, __LINE__, cudaGetErrorString(_e));                              \
            throw pcr::Error(-2, _b);                                                          \
        }                                                                                      \
    } while (0)

#define PCR_REQUIRE(cond, msg)                                                                 \
    do { if (!(cond)) throw pcr::Error(-1, std::string(msg)); } while (0)

// ------------------------------------------------------------------ profiler: CUDA events around every launch
struct Profiler {
    struct Rec { int id; cudaEvent_t a, b; double bytes; };
    struct Acc { std::string name; double ms = 0; i64 launches = 0; double bytes = 0; };
    bool enabled = false;
    i64 launches = 0;                 // counted whether or not event timing is on
    std::vector<Rec> pending;
    std::vector<Acc> acc;
    std::map<std::string, int> ids;
    std::vector<cudaEvent_t> pool;

    int id_of(const char *name) {
        auto it = ids.find(name);
        if (it != ids.end()) return it->second;
        int id = (int)acc.size();
        ids[name] = id;
        Acc a; a.name = name; acc.push_back(a);
        return id;
    }
    cudaEvent_t get_event() {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e; PCR_CUDA(cudaEventCreate(&e)); return e;
    }
    void begin(const char *name, cudaStream_t s, double bytes) {
        ++launches;
        if (!enabled) return;
        Rec r; r.id = id_of(name); r.a = get_event(); r.b = get_event(); r.bytes = bytes;
        PCR_CUDA(cudaEventRecord(r.a, s));
        pending.push_back(r);
    }
    void end(cudaStream_t s) {
        if (!enabled) return;
        PCR_CUDA(cudaEventRecord(pending.back().b, s));
    }
    void resolve() {   // caller has synchronised the stream
        // PRIMALCR_TRACE=<file>: one line per launch, "start_ms duration_ms name" (start relative to the first launch of the batch)
        static const char *trace_path = getenv("PRIMALCR_TRACE");
        FILE *tf = (trace_path && !pending.empty()) ? fopen(trace_path, "a") : nullptr;
        for (auto &r : pending) {
            float ms = 0;
            if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
                acc[r.id].ms += ms; acc[r.id].launches += 1; acc[r.id].bytes += r.bytes;
                if (tf) {
                    float t0 = 0;
                    cudaEventElapsedTime(&t0, pending.front().a, r.a);
                    fprintf(tf, "%.4f %.4f %s\n", t0, ms, acc[r.id].name.c_str());
                }
            }
            pool.push_back(r.a); pool.push_back(r.b);
        }
        pending.clear();
        if (tf) { fprintf(tf, "# batch end\n"); fclose(tf); }
    }
    void reset() { resolve(); for (auto &a : acc) { a.ms = 0; a.launches = 0; a.bytes = 0; } }
    ~Profiler() { for (auto &r : pending) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); } for (auto e : pool) cudaEventDestroy(e); }
};

// RAII device buffer bookkeeping.  Stream-ordered allocation (cudaMallocAsync from the device's default memory pool,
// release threshold raised so that freed blocks are kept for the next engine of the process): a plain cudaMalloc gets
// ~10x slower once NCCL has enabled peer access, because every allocation is then mapped into all peers
// (measured at 2 GPUs: 0.74 s for the ~100 buffers of a 50 M-rating shard vs 0.08 s).  Falls back to cudaMalloc / cudaFree
// when the default memory pool cannot be obtained.
struct DevPool {
    std::vector<void *> ptrs;
    i64 bytes = 0;
    cudaStream_t stream = nullptr;
    bool async = false;
    void init(cudaStream_t s) {
        stream = s;
        int dev = 0; cudaMemPool_t mp;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetDefaultMemPool(&mp, dev) != cudaSuccess) { cudaGetLastError(); return; }
        async = true;
        unsigned long long keep = ~0ull;
        cudaMemPoolSetAttribute(mp, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    void *raw_alloc(size_t b) {
        void *p = nullptr;
        if (b == 0) b = 1;
        if (async) PCR_CUDA(cudaMallocAsync(&p, b, stream)); else PCR_CUDA(cudaMalloc(&p, b));
        return p;
    }
    void raw_free(void *p) {            // temporaries: stream-ordered, so earlier work on `stream` that uses p is safe
        if (!p) return;
        if (async) cudaFreeAsync(p, stream); else cudaFree(p);
    }
    template <typename T> T *alloc(size_t n) {
        const size_t b = (n > 0 ? n : 1) * sizeof(T);
        void *p = raw_alloc(b);
        ptrs.push_back(p); bytes += (i64)b;
        return (T *)p;
    }
    void release() {
        for (void *p : ptrs) raw_free(p);
        if (async && stream && !ptrs.empty()) cudaStreamSynchronize(stream);
        ptrs.clear(); bytes = 0;
    }
    ~DevPool() { release(); }
};

struct TileList { int32_t *first = nullptr, *nusers = nullptr, *ne = nullptr; i64 *e0 = nullptr; i64 n = 0, nnz = 0; };

// ------------------------------------------------------------------ a ratings set on the device (CSR by user)
struct DevCsr {
    i64 d1 = 0, nnz = 0;
    i64 *row_ptr = nullptr;      // [d1+1]
    int32_t *item = nullptr;     // [nnz] item id
    int32_t *user = nullptr;     // [nnz] owning user (local id)
    double *rating = nullptr;    // [nnz] exact rating (eval, Primal-CR)
    uint8_t *level = nullptr;    // [nnz] global level index of lround(rating) (Primal-CR++)
    std::vector<i64> h_row_ptr;  // host copy
    // size classes: users with 0 < len <= S_CAP, S_CAP < len <= L_CAP, len > L_CAP
    int32_t *cls_users[3] = {nullptr, nullptr, nullptr};
    int n_cls[3] = {0, 0, 0};
    i64 *heavy_off = nullptr;    // [d1] offset into the heavy scratch arrays, -1 if not heavy
    i64 heavy_total = 0;         // sum over heavy users of (len + 1)
    i64 *heavy_begin = nullptr, *heavy_end = nullptr;  // [n_cls[2]] absolute segment bounds (heavy-user sort, k_hsort.cu)
    i64 max_len = 0;
    // tiles of consecutive users: [0] small (<= TILE_CAP ratings in total), [1] medium (users with TILE_CAP < len <= TILE_CAP_M),
    // [2] large (TILE_CAP_M < len <= TILE_CAP_L)
    TileList tiles[3];
    // pair-tile work items (Primal-CR pair kernels and pairwise-error evaluation)
    int32_t *pt_user = nullptr; int32_t *pt_j0 = nullptr; i64 n_pt = 0;
    i64 *pt_ptr = nullptr;       // [d1+1] first work item of each user
    // row-sum work units over this CSR (segments = users)
    int32_t *un_seg = nullptr; i64 *un_start = nullptr; i64 n_units = 0;   // un_start[n_units+1]
    i64 *seg_unit_ptr = nullptr; // [d1+1]
};

struct SortedMeta {          // per rating, in (user, ascending score) order
    double *s = nullptr;     // sorted scores
    int32_t *pos = nullptr;  // CSR position of the rating that sits at this sorted slot
    uint8_t *lev = nullptr;  // its level
    int32_t *ub = nullptr, *lb = nullptr;      // window pointers (local to the user)
    int32_t *cnt_lo = nullptr, *cnt_hi = nullptr;
    // level-major copy for the users served by tiles: per rating in (user, level, ascending score) order
    // (heavy users keep their own 32-bit arrays, HeavyLM; only lm_s is shared with them)
    double *lm_s = nullptr;
    // packed record of a tile user's rating, 13-bit fields (a tile holds <= 4096 ratings):
    //   lm_w0 = pos - tile_e0 | cnt_lo << 13 | cnt_hi << 26 | level << 39 | user index inside the tile << 42
    //   lm_w1 = rank (inside the user, level-major) of the window end in the 1st..4th OTHER level, 13 bits each
    //   lm_w2 = the same for the 5th..7th other level (only allocated when T > 5)
    unsigned long long *lm_w0 = nullptr, *lm_w1 = nullptr, *lm_w2 = nullptr;
    uint16_t *ulev = nullptr;     // [d1][8] ratings per level of every user
    i64 nnz = 0;
};

// heavy users (more ratings than the largest tile) cut into chunks, all stages are grids over chunks (k_heavy.cu)
static const int HEAVY_CHUNK = 2048;
struct HeavyLM {
    int n_users = 0, n_chunks = 0;
    const int32_t *users = nullptr;        // [n_users] user id
    const i64 *begin = nullptr, *end = nullptr;   // [n_users] absolute rating range of the user
    const i64 *off = nullptr;              // [n_users] offset into the scratch arrays below (users are spaced len + 1 apart)
    const int32_t *chunk_user = nullptr;   // [n_chunks] index into users[]
    const int32_t *chunk_lo = nullptr;     // [n_chunks] first element of the chunk inside its user
    const int32_t *chunk0 = nullptr;       // [n_users + 1] first chunk of every heavy user
    int32_t *ccnt = nullptr;               // [n_chunks x 8] ratings per level of a chunk -> exclusive bases inside the user
    int32_t *B = nullptr;                  // [n_users x 9] first level-major rank of every level (B[8] = len)
    int32_t *idx = nullptr;                // [(T - 1) planes][htot] rank of the window end in every OTHER level
    int32_t *pos = nullptr, *lo = nullptr, *hi = nullptr;   // [htot] level-major order: CSR position, aggregated counters
    uint8_t *lev = nullptr;                // [htot] level-major order: level
    double *G = nullptr, *G2 = nullptr;    // [htot] running prefixes of the stream in level-major order
    double *csum = nullptr;                // [n_chunks x 2] chunk sums
    i64 htot = 0;
};

// work list of the heavy-user segmented sort (k_hsort.cu): chunks of HEAVY_CHUNK ratings, one scratch (score, position) pair
struct HeavySortPlan {
    int n_users = 0, n_chunks = 0, max_passes = 0;
    const i64 *begin = nullptr, *end = nullptr;   // [n_users] absolute rating range of the user
    const i64 *off = nullptr;                     // [n_users] offset of the user inside the scratch pair
    const int32_t *chunk_user = nullptr;          // [n_chunks] index into begin/end/off
    const int32_t *chunk_lo = nullptr;            // [n_chunks] first rating of the chunk inside its user
    double *tmp_s = nullptr; int32_t *tmp_pos = nullptr;   // [sum of heavy lens] ping-pong partner of SortedMeta::s / pos
};

static const int TILE_CAP = 1024;        // ratings per tile of consecutive users (k_tiles.cu)
static const int TILE_MAX_USERS = 128;   // users per tile
static const int TILE_CAP_M = 2048;      // medium tiles: 512 threads, two CTAs per SM (most users above TILE_CAP are below 2048:
                                         // in 4096-rating tiles they left 60 % of the threads idle)
static const int TILE_CAP_L = 4096;      // large tiles: 1024 threads
static const int S_CAP = 1024;   // block class  (256 threads, shared memory)
static const int L_CAP = 4096;   // large class  (1024 threads, shared memory)
#ifndef PCR_ROWSUM_CHUNK
#define PCR_ROWSUM_CHUNK 256
#endif
static const int ROWSUM_CHUNK = PCR_ROWSUM_CHUNK;
static const int PAIR_TJ = 256;  // j elements per pair work item
static const int MAX_LEVELS = 256;  // levels are uint8 indices; more than 8 levels -> per-user T-vector kernels (k_core.cu)

}  // namespace pcr
