// k_heavy.cu -- heavy users (more ratings than a tile holds) as CHUNK-parallel kernels.
//
// A user with 5 000 .. 100 000+ ratings cannot live in one CTA's shared memory.  The first version gave each such user
// ONE 1024-thread CTA that scanned through global scratch once per rating level: its run time is set by the single
// longest user, it does not shrink when the users are sharded over more GPUs, and it makes the rank that owns the
// longest users arrive late at every all-reduce.  Here every heavy user is cut into chunks of HCH ratings and all
// stages are grids over CHUNKS, so the critical path no longer depends on how long the longest user is.
//
// Same restatement as tile_lm_sweep (k_tiles.cu): the ratings of a user are kept in (level, score) order, each level is
// a block [B_t, B_t+1), and every per-level prefix sum of the sweep (pcrpp.cpp:214-236, :294-318, :396-406) is a
// difference of ONE running prefix G over that order, looked up at ranks that only depend on the scores:
//   idx_t(j) = B_t + #{q in level t : s_q <= fl(s_j + 1.0)}   for t > l_j     (left window, pcrpp.cpp:218)
//   idx_t(j) = B_t + #{q in level t : s_q <  fl(s_j - 1.0)}   for t < l_j     (right window, pcrpp.cpp:224)
//
//   prepare:  segmented sort by score (k_hsort.cu) -> level histogram per chunk -> bases -> stable scatter into
//             (level, score) order -> per-level binary searches for idx_t / cnt_lo / cnt_hi
//   sweep:    chunk sums of the stream -> per-chunk exclusive scan + base = G -> look-ups -> c_j / objective
// All sums have a fixed association order (deterministic, independent of the grid schedule).
#include "kernels.h"
#include "block_prims.cuh"
#include <math_constants.h>

namespace pcr {

#define LAUNCH(ctx, name, bytes, kernel, grid, block, smem, ...)                         \
    do {                                                                                 \
        (ctx).prof->begin(name, (ctx).stream, (double)(bytes));                          \
        kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);                  \
        (ctx).prof->end((ctx).stream);                                                   \
        PCR_CUDA(cudaGetLastError());                                                    \
    } while (0)

static const int HTH = 256;                 // threads per chunk CTA
static const int HTE = HEAVY_CHUNK / HTH;   // elements per thread

struct ChunkInfo { int hu, u, lo, cnt, n; i64 start, off; };

__device__ __forceinline__ ChunkInfo chunk_info(const HeavyLM &h, int c) {
    ChunkInfo ci;
    ci.hu = h.chunk_user[c];
    ci.u = h.users[ci.hu];
    ci.lo = h.chunk_lo[c];
    ci.start = h.begin[ci.hu];
    ci.n = (int)(h.end[ci.hu] - ci.start);
    ci.cnt = ci.n - ci.lo < HEAVY_CHUNK ? ci.n - ci.lo : HEAVY_CHUNK;
    ci.off = h.off[ci.hu];
    return ci;
}

// ---------------------------------------------------------------- prepare 1: per-chunk level histogram (score order)
__global__ void __launch_bounds__(HTH) hv_level_hist_kernel(HeavyLM h, const uint8_t *__restrict__ lev_sorted) {
    __shared__ int hist[8];
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    const int tid = threadIdx.x;
    if (tid < 8) hist[tid] = 0;
    __syncthreads();
    int lc[8];
#pragma unroll
    for (int t = 0; t < 8; ++t) lc[t] = 0;
    for (int i = tid; i < ci.cnt; i += HTH) {
        const int l = lev_sorted[ci.start + ci.lo + i];
#pragma unroll
        for (int t = 0; t < 8; ++t) lc[t] += (t == l) ? 1 : 0;
    }
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int w = __reduce_add_sync(FULL, lc[t]);
        if ((tid & 31) == 0 && w) atomicAdd(&hist[t], w);      // integer adds: order does not matter
    }
    __syncthreads();
    if (tid < 8) h.ccnt[(size_t)blockIdx.x * 8 + tid] = hist[tid];
}

// ---------------------------------------------------------------- prepare 2: chunk bases per level + level block starts
__global__ void __launch_bounds__(32) hv_level_base_kernel(HeavyLM h) {
    const int hu = blockIdx.x, t = threadIdx.x;
    __shared__ int tot[8];
    if (t < 8) {
        int run = 0;
        for (int c = h.chunk0[hu]; c < h.chunk0[hu + 1]; ++c) {
            const int v = h.ccnt[(size_t)c * 8 + t];
            h.ccnt[(size_t)c * 8 + t] = run;
            run += v;
        }
        tot[t] = run;
    }
    __syncwarp();
    if (t == 0) {
        int run = 0;
        for (int q = 0; q < 8; ++q) { h.B[hu * 9 + q] = run; run += tot[q]; }
        h.B[hu * 9 + 8] = run;
    }
}

// ---------------------------------------------------------------- prepare 3: stable scatter into (level, score) order
__global__ void __launch_bounds__(HTH) hv_scatter_lm_kernel(HeavyLM h, const double *__restrict__ s_sorted,
                                                            const int32_t *__restrict__ pos_sorted,
                                                            const uint8_t *__restrict__ lev_sorted, SortedMeta lm) {
    __shared__ uint8_t slev[HEAVY_CHUNK];
    __shared__ int srank[HEAVY_CHUNK];
    __shared__ unsigned long long wa[HTH / 32], wb[HTH / 32];
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < ci.cnt; i += HTH) slev[i] = lev_sorted[ci.start + ci.lo + i];
    __syncthreads();
    // per-level counts of this thread's HTE consecutive elements, packed 4 x 16 bits per word (counts <= HEAVY_CHUNK)
    unsigned long long pa = 0ull, pb = 0ull;
    const int lo = tid * HTE;
#pragma unroll
    for (int q = 0; q < HTE; ++q) {
        const int i = lo + q;
        if (i < ci.cnt) { const int l = slev[i]; if (l < 4) pa += 1ull << (16 * l); else pb += 1ull << (16 * (l - 4)); }
    }
    unsigned long long ia = pa, ib = pb;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long ta = __shfl_up_sync(FULL, ia, o), tb = __shfl_up_sync(FULL, ib, o);
        if (lane >= o) { ia += ta; ib += tb; }
    }
    if (lane == 31) { wa[warp] = ia; wb[warp] = ib; }
    __syncthreads();
    unsigned long long ea = ia - pa, eb = ib - pb;          // exclusive inside the warp
    for (int w = 0; w < warp; ++w) { ea += wa[w]; eb += wb[w]; }
    const int *cb = h.ccnt + (size_t)blockIdx.x * 8;        // ranks of this chunk's first element of every level
    const int *B = h.B + ci.hu * 9;
#pragma unroll
    for (int q = 0; q < HTE; ++q) {
        const int i = lo + q;
        if (i < ci.cnt) {
            const int l = slev[i];
            int r;
            if (l < 4) { r = (int)((ea >> (16 * l)) & 0xFFFFull); ea += 1ull << (16 * l); }
            else       { r = (int)((eb >> (16 * (l - 4))) & 0xFFFFull); eb += 1ull << (16 * (l - 4)); }
            srank[i] = B[l] + cb[l] + r;
        }
    }
    __syncthreads();
    for (int i = tid; i < ci.cnt; i += HTH) {
        const i64 src = ci.start + ci.lo + i, dst = ci.start + srank[i];
        const i64 hd = ci.off + srank[i];
        lm.lm_s[dst] = s_sorted[src]; h.pos[hd] = pos_sorted[src]; h.lev[hd] = slev[i];
    }
}

// ---------------------------------------------------------------- prepare 4: window ranks in every other level
// (chunks of the level-major order; binary searches over the level blocks with exactly fl(s + 1.0) / fl(s - 1.0))
__global__ void __launch_bounds__(HTH) hv_windows_lm_kernel(HeavyLM h, SortedMeta lm, int T) {
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    const int *B = h.B + ci.hu * 9;
    const double *ss = lm.lm_s + ci.start;
    for (int i = threadIdx.x; i < ci.cnt; i += HTH) {
        const int x = ci.lo + i;
        const double sj = ss[x];
        const int l = h.lev[ci.off + x];
        const double hi = __dadd_rn(sj, 1.0), lo = __dadd_rn(sj, -1.0);
        int chi = 0, clo = 0;
        for (int t = 0; t < T; ++t) {
            if (t == l) continue;
            int a = B[t], b = B[t + 1];
            if (t > l) { while (a < b) { const int mid = (a + b) >> 1; if (ss[mid] <= hi) a = mid + 1; else b = mid; } chi += a - B[t]; }
            else       { while (a < b) { const int mid = (a + b) >> 1; if (ss[mid] < lo) a = mid + 1; else b = mid; } clo += B[t + 1] - a; }
            h.idx[(size_t)(t < l ? t : t - 1) * h.htot + ci.off + x] = a;
        }
        h.lo[ci.off + x] = clo; h.hi[ci.off + x] = chi;
    }
}

// ---------------------------------------------------------------- sweep 1: chunk sums of the stream (level-major order)
// MODE 0: v = s, MODE 1: v = b[pos], MODE 2: v = s - 1 and (s - 1)^2
template <int MODE>
__device__ __forceinline__ double hv_stream(const HeavyLM &h, const SortedMeta &lm, const double *__restrict__ b_g, const ChunkInfo &ci, int x) {
    if (MODE == 1) return b_g[h.pos[ci.off + x]];
    if (MODE == 2) return lm.lm_s[ci.start + x] - 1.0;
    return lm.lm_s[ci.start + x];
}

template <int MODE>
__global__ void __launch_bounds__(HTH) hv_chunk_sums_kernel(HeavyLM h, const uint8_t *__restrict__ active, SortedMeta lm,
                                                            const double *__restrict__ b_g) {
    __shared__ double wsum[HTH / 32];
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    if (active && !active[ci.u]) return;
    double a = 0.0, a2 = 0.0;
    for (int i = threadIdx.x; i < ci.cnt; i += HTH) {
        const double v = hv_stream<MODE>(h, lm, b_g, ci, ci.lo + i);
        a += v;
        if (MODE == 2) a2 += v * v;
    }
    const double s1 = block_sum<HTH>(a, wsum);
    if (threadIdx.x == 0) h.csum[(size_t)blockIdx.x * 2] = s1;
    if (MODE == 2) {
        const double s2 = block_sum<HTH>(a2, wsum);
        if (threadIdx.x == 0) h.csum[(size_t)blockIdx.x * 2 + 1] = s2;
    }
}

// ---------------------------------------------------------------- sweep 2: G = exclusive prefix over the user
template <int MODE>
__global__ void __launch_bounds__(HTH) hv_chunk_scan_kernel(HeavyLM h, const uint8_t *__restrict__ active, SortedMeta lm,
                                                            const double *__restrict__ b_g) {
    __shared__ double a[HEAVY_CHUNK + 1];
    __shared__ double wsum[HTH / 32 + 1];
    __shared__ double s_base[2];
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    if (active && !active[ci.u]) return;
    const int tid = threadIdx.x;
    if (tid < (MODE == 2 ? 2 : 1)) {          // sum of the previous chunks of this user, in chunk order
        double run = 0.0;
        for (int c = h.chunk0[ci.hu]; c < (int)blockIdx.x; ++c) run += h.csum[(size_t)c * 2 + tid];
        s_base[tid] = run;
    }
    const bool last = ci.lo + ci.cnt == ci.n;
    for (int pass = 0; pass < (MODE == 2 ? 2 : 1); ++pass) {
        for (int i = tid; i < ci.cnt; i += HTH) {
            const double v = hv_stream<MODE>(h, lm, b_g, ci, ci.lo + i);
            a[i] = pass == 0 ? v : v * v;
        }
        __syncthreads();
        block_excl_scan<double, HTH>(a, ci.cnt, wsum);
        double *G = pass == 0 ? h.G : h.G2;
        const double base = s_base[pass];
        for (int i = tid; i < ci.cnt; i += HTH) G[ci.off + ci.lo + i] = base + a[i];
        if (last && tid == 0) G[ci.off + ci.n] = base + a[ci.cnt];
        __syncthreads();
    }
}

// ---------------------------------------------------------------- sweep 3: look-ups -> coefficient / objective terms
template <int MODE>
__global__ void __launch_bounds__(HTH) hv_lookup_kernel(HeavyLM h, const uint8_t *__restrict__ active, SortedMeta lm,
                                                        const double *__restrict__ b_g, double *__restrict__ c_out, int T) {
    __shared__ double wsum[HTH / 32];
    __shared__ double Kt[8], Kt2[8];
    const ChunkInfo ci = chunk_info(h, blockIdx.x);
    if (active && !active[ci.u]) return;
    const int *B = h.B + ci.hu * 9;
    const double *G = h.G + ci.off, *G2 = h.G2 + ci.off;
    if (threadIdx.x < T) {                    // per-user constants K_u[l] (see tile_lm_sweep_kernel)
        const int l = threadIdx.x;
        double k1 = 0.0, k2 = 0.0;
        for (int t = 0; t < T; ++t) {
            if (t > l) { k1 -= G[B[t]]; if (MODE == 2) k2 -= G2[B[t]]; }
            else if (t < l && MODE != 2) k1 += G[B[t + 1]];
        }
        Kt[l] = k1; Kt2[l] = k2;
    }
    __syncthreads();
    double part = 0.0;
    for (int i = threadIdx.x; i < ci.cnt; i += HTH) {
        const int x = ci.lo + i;
        const i64 at = ci.start + x;
        const i64 ha = ci.off + x;
        const int l = h.lev[ha];
        double acc = Kt[l], acc2 = MODE == 2 ? Kt2[l] : 0.0;
        for (int t = 0; t < T; ++t) {
            if (t == l) continue;
            if (MODE == 2 && t < l) continue;
            const int r = h.idx[(size_t)(t < l ? t : t - 1) * h.htot + ci.off + x];
            if (t > l) { acc += G[r]; if (MODE == 2) acc2 += G2[r]; }
            else acc -= G[r];
        }
        if (MODE == 2) {
            const double v = lm.lm_s[at];
            part += (double)h.hi[ha] * (v * v) - 2.0 * v * acc + acc2;
        } else {
            const int pos = h.pos[ha];
            const double v = MODE == 0 ? lm.lm_s[at] : b_g[pos];
            const double lo = (double)h.lo[ha], hi = (double)h.hi[ha];
            const double cc = MODE == 0 ? lo * (v - 1.0) + hi * (v + 1.0) - acc : (lo + hi) * v - acc;
            c_out[pos] = 2.0 * cc;
        }
    }
    if (MODE == 2) {
        const double s = block_sum<HTH>(part, wsum);
        if (threadIdx.x == 0) h.csum[(size_t)blockIdx.x * 2] = s;
    }
}

// ---------------------------------------------------------------- sweep 4 (objective): per-user sum of the chunk terms
__global__ void __launch_bounds__(128) hv_obj_users_kernel(HeavyLM h, const uint8_t *__restrict__ active, double *__restrict__ obj_user) {
    const int hu = blockIdx.x * 128 + threadIdx.x;
    if (hu >= h.n_users) return;
    const int u = h.users[hu];
    if (active && !active[u]) return;
    double run = 0.0;
    for (int c = h.chunk0[hu]; c < h.chunk0[hu + 1]; ++c) run += h.csum[(size_t)c * 2];
    obj_user[u] = run;
}

// ---------------------------------------------------------------- launchers
void k_heavy_prepare(Ctx &c, const HeavyLM &h, SortedMeta &meta, int T) {
    if (h.n_chunks <= 0) return;
    PCR_REQUIRE(T <= 8 && meta.lm_s != nullptr, "chunked heavy-user path needs T <= 8 and the level-major arrays");
    LAUNCH(c, "hv_level_hist", 0.0, hv_level_hist_kernel, h.n_chunks, HTH, 0, h, meta.lev);
    LAUNCH(c, "hv_level_base", 0.0, hv_level_base_kernel, h.n_users, 32, 0, h);
    LAUNCH(c, "hv_scatter_lm", 0.0, hv_scatter_lm_kernel, h.n_chunks, HTH, 0, h, meta.s, meta.pos, meta.lev, meta);
    LAUNCH(c, "hv_windows_lm", 0.0, hv_windows_lm_kernel, h.n_chunks, HTH, 0, h, meta, T);
}

void k_heavy_sweep(Ctx &c, int mode, const HeavyLM &h, const uint8_t *active, const SortedMeta &meta, const double *b,
                   double *c_out, double *obj_user, int T) {
    if (h.n_chunks <= 0) return;
#define HV(MODE, NAME)                                                                                                      \
    LAUNCH(c, NAME "_sums", 0.0, hv_chunk_sums_kernel<MODE>, h.n_chunks, HTH, 0, h, active, meta, b);                         \
    LAUNCH(c, NAME "_scan", 0.0, hv_chunk_scan_kernel<MODE>, h.n_chunks, HTH, 0, h, active, meta, b);                         \
    LAUNCH(c, NAME "_look", 0.0, hv_lookup_kernel<MODE>, h.n_chunks, HTH, 0, h, active, meta, b, c_out, T);
    if (mode == 0) { HV(0, "hv_grad") }
    else if (mode == 1) { HV(1, "hv_hv") }
    else {
        HV(2, "hv_obj")
        LAUNCH(c, "hv_obj_users", 0.0, hv_obj_users_kernel, (h.n_users + 127) / 128, 128, 0, h, active, obj_user);
    }
#undef HV
}

}  // namespace pcr
