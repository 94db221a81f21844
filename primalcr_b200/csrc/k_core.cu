// k_core.cu -- the Primal-CR++ hot path as hand-written sm_100a kernels.
//
//   dots        K1  comp_m_new pcrpp.cpp:17-35, b = U_i . a[p] pcrpp.cpp:266-271, b = s . V[p] :592-594,
//                   compute_mm_old :728-744          (score gather, 16-byte vector loads, shuffle reduce)
//   sort        K2  get_sorted_mm pcrpp.cpp:52-83    (per-user bitonic sort in shared memory)
//   windows     K3  the two sweep pointers + integer level counters pcrpp.cpp:214-229
//   sweep_*     K3  c_j of obtain_g_new :230-238 / compute_Ha_new :310-318 / obtain_g_u_new :527-535 /
//                   obtain_Hs_new :613-621 and the objective :392-407, :556-571 as per-level prefix scans
//   rowsum      K4  G[p,:] += c * U_i  pcrpp.cpp:240-243, :323-327 (item-major over the CSC, no atomics) and
//                   g += c * V[p] :536, :622 (user-major over the CSR)
//   u_*         K6  per-user truncated Newton-CG bookkeeping update_u_new :779-815, solve_delta_u_new :628-647
//   vec         K5  CG vector algebra of solve_delta_new :335-358
#include "kernels.h"
#include "block_prims.cuh"
#include <math_constants.h>
#include <algorithm>
#include <cstdlib>

namespace pcr {

#ifndef FULL
#define FULL 0xffffffffu
#endif

// which rating levels a user holds: a 256-bit map in shared memory (levels are uint8 indices into the global table)
__device__ __forceinline__ void lvl_mark(unsigned *m, int l) {
    const unsigned bit = 1u << (l & 31);
    if (!(reinterpret_cast<volatile unsigned *>(m)[l >> 5] & bit)) atomicOr(&m[l >> 5], bit);
}
__device__ __forceinline__ bool lvl_has(const unsigned *m, int t) { return (m[t >> 5] >> (t & 31)) & 1u; }
__device__ __forceinline__ bool lvl_any_below(const unsigned *m, int t) {
    for (int w = 0; w < (t >> 5); ++w) if (m[w]) return true;
    return (m[t >> 5] & ((1u << (t & 31)) - 1u)) != 0u;
}
__device__ __forceinline__ int lvl_count(const unsigned *m) {
    int c = 0;
#pragma unroll
    for (int w = 0; w < MAX_LEVELS / 32; ++w) c += __popc(m[w]);
    return c;
}

// minimum resident CTAs per SM requested from ptxas for the two N*k kernels (register budget = 65536 / (256 * MINB))
#ifndef PCR_ROWSUM_MINB
#define PCR_ROWSUM_MINB 4
#endif
#ifndef PCR_DOTS_MINB
#define PCR_DOTS_MINB 3
#endif

#define LAUNCH(ctx, name, bytes, kernel, grid, block, smem, ...)                         \
    do {                                                                                 \
        (ctx).prof->begin(name, (ctx).stream, (double)(bytes));                          \
        kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);                  \
        (ctx).prof->end((ctx).stream);                                                   \
        PCR_CUDA(cudaGetLastError());                                                    \
    } while (0)

static inline unsigned grid_for(i64 work_items, int per_block, int max_blocks) {
    i64 b = (work_items + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > max_blocks) b = max_blocks;
    return (unsigned)b;
}

// grid of a persistent (grid-stride) kernel: exactly what fits at once, so there is a single full wave
template <typename K>
static unsigned resident_grid(K kernel, int block, size_t smem, int sms, i64 max_useful) {
    int per_sm = 0;
    PCR_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
    if (per_sm < 1) per_sm = 1;
    i64 g = (i64)per_sm * sms;
    if (g > max_useful) g = max_useful;
    if (g < 1) g = 1;
    return (unsigned)g;
}

// ------------------------------------------------------------------ K1: dots

template <int G>
__global__ void __launch_bounds__(256) dots_kernel(const double *__restrict__ P, const int32_t *__restrict__ prow,
                                                   const double *__restrict__ Q, const int32_t *__restrict__ qrow,
                                                   i64 n, int nch, int ld, const uint8_t *__restrict__ active,
                                                   double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int lg = lane % G;
    const int per_warp = 32 / G;
    const i64 warp_global = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    const i64 nwarps = ((i64)gridDim.x * 256) >> 5;
    for (i64 base = warp_global * per_warp; base < n; base += nwarps * per_warp) {
        const i64 e = base + lane / G;
        bool doit = e < n;
        int pr = 0, qr = 0;
        if (doit) { pr = prow[e]; qr = qrow[e]; if (active && !active[pr]) doit = false; }
        double ax = 0.0, ay = 0.0;
        if (doit) {
            const double2 *p2 = reinterpret_cast<const double2 *>(P + (size_t)pr * ld);
            const double2 *q2 = reinterpret_cast<const double2 *>(Q + (size_t)qr * ld);
#pragma unroll 4
            for (int c = lg; c < nch; c += G) {
                const double2 a = __ldg(p2 + c);
                const double2 b = __ldg(q2 + c);
                ax = fma(a.x, b.x, ax);
                ay = fma(a.y, b.y, ay);
            }
        }
        double s = ax + ay;
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(FULL, s, o);
        if (doit && lg == 0) out[e] = s;
    }
}

void k_dots(Ctx &c, const double *P, const int32_t *prow, const double *Q, const int32_t *qrow, i64 n, int ld, int kk,
            const uint8_t *active, double *out, double bytes) {
    if (n <= 0) return;
    const int nch = (kk + 1) / 2;      // 16-byte chunks that carry payload (rows are padded to ld for 128-byte alignment)
    if (nch <= 4) {
        LAUNCH(c, active ? "dots_active" : "dots", bytes, dots_kernel<4>, resident_grid(dots_kernel<4>, 256, 0, c.sms, (n + 63) / 64), 256, 0, P, prow, Q, qrow, n, nch, ld, active, out);
    } else {
        LAUNCH(c, active ? "dots_active" : "dots", bytes, dots_kernel<8>, resident_grid(dots_kernel<8>, 256, 0, c.sms, (n + 31) / 32), 256, 0, P, prow, Q, qrow, n, nch, ld, active, out);
    }
}

// user-major variant for the training set: one warp per (user, <=ROWSUM_CHUNK ratings) unit; the user's row P[seg]
// stays in registers, the 32 item indices of a batch are fetched with one coalesced load, and the NC 16-byte loads of
// a rating's Q row are issued back to back before the first FMA (NC is a template parameter => fully unrolled).
template <int G, int NC>
__global__ void __launch_bounds__(256, PCR_DOTS_MINB) dots_units_kernel(const int32_t *__restrict__ un_seg, const i64 *__restrict__ un_start,
                                                         const i64 *__restrict__ un_end,
                                                         i64 n_units, unsigned long long *__restrict__ ticket,
                                                         const double *__restrict__ P,
                                                         const double *__restrict__ Q, const int32_t *__restrict__ qrow,
                                                         int nch, int ld, const uint8_t *__restrict__ active,
                                                         double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int lg = lane % G, grp = lane / G;
    constexpr int PW = 32 / G;
    for (;;) {
        // dynamic (work-stealing) unit scheduling: units differ in length, a ticket counter keeps every warp busy
        unsigned long long tk = 0;
        if (lane == 0) tk = atomicAdd(ticket, 1ull);
        const i64 u = (i64)__shfl_sync(FULL, tk, 0);
        if (u >= n_units) break;
        const int seg = un_seg[u];
        if (active && !active[seg]) continue;           // warp-uniform
        const i64 b = un_start[u], e = un_end ? un_end[u] : un_start[u + 1];
        double2 pr[NC];
        const double2 *p2 = reinterpret_cast<const double2 *>(P + (size_t)seg * ld);
#pragma unroll
        for (int i = 0; i < NC; ++i) { const int c = lg + G * i; pr[i] = c < nch ? __ldg(p2 + c) : make_double2(0.0, 0.0); }
        for (i64 base = b; base < e; base += 32) {
            const i64 me = base + lane;
            const int qi = me < e ? qrow[me] : 0;
            const int cnt = (e - base) < 32 ? (int)(e - base) : 32;
#pragma unroll 2
            for (int t = 0; t < cnt; t += PW) {
                const int j = t + grp;
                const bool valid = j < cnt;
                const int r = __shfl_sync(FULL, qi, j & 31);
                const double2 *q2 = reinterpret_cast<const double2 *>(Q + (size_t)r * ld);
                double2 qv[NC];
#pragma unroll
                for (int i = 0; i < NC; ++i) {
                    const int c = lg + G * i;
                    qv[i] = (valid && c < nch) ? __ldg(q2 + c) : make_double2(0.0, 0.0);
                }
                double ax = 0.0, ay = 0.0;
#pragma unroll
                for (int i = 0; i < NC; ++i) { ax = fma(pr[i].x, qv[i].x, ax); ay = fma(pr[i].y, qv[i].y, ay); }
                double sres = ax + ay;
#pragma unroll
                for (int o = G / 2; o > 0; o >>= 1) sres += __shfl_xor_sync(FULL, sres, o);
                if (valid && lg == 0) out[base + j] = sres;
            }
        }
    }
}

template <int G, int NC>
static void launch_dots_units(Ctx &c, const int32_t *un_seg, const i64 *un_start, const i64 *un_end, i64 n_units, const double *P, const double *Q,
                              const int32_t *qrow, int nch, int ld, const uint8_t *active, double *out, double bytes) {
    const unsigned grid = resident_grid(dots_units_kernel<G, NC>, 256, 0, c.sms, (n_units + 7) / 8);
    PCR_CUDA(cudaMemsetAsync(c.ticket, 0, sizeof(unsigned long long), c.stream));
    LAUNCH(c, active ? "dots_active" : "dots", bytes, (dots_units_kernel<G, NC>), grid, 256, 0, un_seg, un_start, un_end, n_units, c.ticket, P, Q, qrow,
           nch, ld, active, out);
}

void k_dots_units(Ctx &c, const int32_t *un_seg, const i64 *un_start, const i64 *un_end, i64 n_units, const double *P, const double *Q,
                  const int32_t *qrow, int ld, int kk, const uint8_t *active, double *out, double bytes) {
    if (n_units <= 0) return;
    const int nch = (kk + 1) / 2;
    PCR_REQUIRE(nch <= 128, "rank too large for dots kernel (k <= 256)");
#define DU(G, NC) launch_dots_units<G, NC>(c, un_seg, un_start, un_end, n_units, P, Q, qrow, nch, ld, active, out, bytes); return;
    if (nch <= 56) {
        switch ((nch + 7) / 8) { case 1: DU(8, 1) case 2: DU(8, 2) case 3: DU(8, 3) case 4: DU(8, 4) case 5: DU(8, 5) case 6: DU(8, 6) default: DU(8, 7) }
    } else if (nch <= 112) {
        switch ((nch + 15) / 16) { case 4: DU(16, 4) case 5: DU(16, 5) case 6: DU(16, 6) default: DU(16, 7) }
    } else {
        DU(32, 4)
    }
#undef DU
}

// ------------------------------------------------------------------ K4: segmented weighted row sums

// L2 cache-policy loads of the item-major pass: the gathered U rows of the current user block are asked to stay
// (evict_last), the ids / coefficients that stream through once are asked to leave first
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long p; asm("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long p; asm("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p)); return p;
}
__device__ __forceinline__ double2 ldg_hint_d2(const double2 *p, unsigned long long pol) {
    double2 v; asm volatile("ld.global.nc.L2::cache_hint.v2.f64 {%0, %1}, [%2], %3;" : "=d"(v.x), "=d"(v.y) : "l"(p), "l"(pol)); return v;
}
__device__ __forceinline__ int ldg_hint_i32(const int32_t *p, unsigned long long pol) {
    int v; asm volatile("ld.global.nc.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol)); return v;
}

// HINT: gathered rows evict_last, the two id streams evict_first; the coefficient gather keeps the default policy (its
// 32-byte sectors hold 4 coefficients that other items' units read soon: evict_first there cost +3 GB of DRAM reads per launch)
template <int NCH, bool HINT = false>
__global__ void __launch_bounds__(256, PCR_ROWSUM_MINB) rowsum_kernel(const int32_t *__restrict__ un_seg, const i64 *__restrict__ un_start,
                                                     const i64 *__restrict__ un_end,
                                                     i64 n_units, unsigned long long *__restrict__ ticket,
                                                     const int32_t *__restrict__ ridx,
                                                     const int32_t *__restrict__ widx, const double *__restrict__ w,
                                                     const double *__restrict__ M, int ld, int nch,
                                                     const uint8_t *__restrict__ active, double *__restrict__ partial) {
    const int lane = threadIdx.x & 31;
    unsigned long long pol_keep = 0, pol_stream = 0;
    if (HINT) { pol_keep = l2_policy_evict_last(); pol_stream = l2_policy_evict_first(); }
    for (;;) {
        unsigned long long tk = 0;
        if (lane == 0) tk = atomicAdd(ticket, 1ull);     // units are consumed in list order (user-block-major for the CSC)
        const i64 u = (i64)__shfl_sync(FULL, tk, 0);
        if (u >= n_units) break;
        const int seg = un_seg[u];
        if (active && !active[seg]) continue;           // warp-uniform
        const i64 b = un_start[u], e = un_end ? un_end[u] : un_start[u + 1];
        double2 acc[NCH];
#pragma unroll
        for (int q = 0; q < NCH; ++q) acc[q] = make_double2(0.0, 0.0);
        for (i64 base = b; base < e; base += 32) {
            const i64 me = base + lane;
            int ri = 0; double wi = 0.0;
            if (me < e) {
                if (HINT) { ri = ldg_hint_i32(ridx + me, pol_stream); wi = w[ldg_hint_i32(widx + me, pol_stream)]; }
                else { ri = ridx[me]; wi = widx ? w[widx[me]] : w[me]; }
            }
            const int cnt = (e - base) < 32 ? (int)(e - base) : 32;
            // (measured: requesting the NEXT batch's ids / weights one batch ahead costs 8 registers and is slower: item-major
            //  pass 5.8 -> 6.3 ms, dots 4.23 -> 4.29 ms)
            // (measured: forcing 8 or 16 loads per lane in flight with an explicit load-then-FMA batch costs more in
            //  occupancy than it gains -- 89 ms and 206 ms vs 73 ms per step for the item-major pass; the compiler's own
            //  interleaving of this 4x unrolled loop at 56 registers is the fastest variant)
#pragma unroll 4
            for (int j = 0; j < cnt; ++j) {
                const int r = __shfl_sync(FULL, ri, j);
                const double ww = __shfl_sync(FULL, wi, j);
                const double2 *row = reinterpret_cast<const double2 *>(M + (size_t)r * ld);
#pragma unroll
                for (int q = 0; q < NCH; ++q) {
                    const int ci = lane + 32 * q;
                    if (ci < nch) {
                        const double2 x = HINT ? ldg_hint_d2(row + ci, pol_keep) : __ldg(row + ci);
                        acc[q].x = fma(ww, x.x, acc[q].x);
                        acc[q].y = fma(ww, x.y, acc[q].y);
                    }
                }
            }
        }
        double2 *o = reinterpret_cast<double2 *>(partial + (size_t)u * ld);
#pragma unroll
        for (int q = 0; q < NCH; ++q) { const int ci = lane + 32 * q; if (ci < nch) o[ci] = acc[q]; }
    }
}

// out[seg] = lambda*x[seg] + partial[first unit] + partial[second unit] + ...   (fixed order => deterministic)
// One warp per segment; a lane owns up to 4 double2 chunks of the row and walks the unit list once with all of them in
// flight (16-byte loads).  kp = payload columns (even), the padding up to ld is kept exactly zero.
__global__ void __launch_bounds__(256) rowsum_finalize_kernel(const i64 *__restrict__ seg_unit_ptr,
                                                              const int32_t *__restrict__ seg_unit_idx, i64 n_seg,
                                                              const double *__restrict__ partial, int ld,
                                                              const uint8_t *__restrict__ active, double lambda,
                                                              const double *__restrict__ x, double *__restrict__ out,
                                                              int zero_if_empty, int kp) {
    const int lane = threadIdx.x & 31;
    const i64 warp_global = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    const i64 nwarps = ((i64)gridDim.x * 256) >> 5;
    const int nch = kp >> 1, nch_ld = ld >> 1;
    for (i64 seg = warp_global; seg < n_seg; seg += nwarps) {
        if (active && !active[seg]) continue;
        const i64 u0 = seg_unit_ptr[seg], u1 = seg_unit_ptr[seg + 1];
        const bool use_x = x != nullptr && !(zero_if_empty && u0 == u1);
        double2 v[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int ci = lane + 32 * q;
            v[q] = make_double2(0.0, 0.0);
            if (use_x && ci < nch) {
                const double2 xv = reinterpret_cast<const double2 *>(x + (size_t)seg * ld)[ci];
                v[q] = make_double2(lambda * xv.x, lambda * xv.y);
            }
        }
        for (i64 u = u0; u < u1; ++u) {
            const double2 *prow = reinterpret_cast<const double2 *>(partial + (size_t)(seg_unit_idx ? seg_unit_idx[u] : u) * ld);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int ci = lane + 32 * q;
                if (ci < nch) { const double2 t = prow[ci]; v[q].x += t.x; v[q].y += t.y; }
            }
        }
        double2 *orow = reinterpret_cast<double2 *>(out + (size_t)seg * ld);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int ci = lane + 32 * q;
            if (ci < nch) orow[ci] = v[q];
            else if (ci < nch_ld) orow[ci] = make_double2(0.0, 0.0);
        }
    }
}

void k_rowsum(Ctx &c, const int32_t *un_seg, const i64 *un_start, const i64 *un_end, i64 n_units, const i64 *seg_unit_ptr,
              const int32_t *seg_unit_idx, i64 n_seg, const int32_t *ridx, const int32_t *widx, const double *w, const double *M, int ld,
              const uint8_t *active, double *partial, double lambda, const double *x, double *out,
              int zero_if_empty, double bytes, int kk) {
    const int nch = (kk + 1) / 2;
    const int NCH = (nch + 31) / 32;
    PCR_REQUIRE(NCH <= 4, "rank too large for rowsum kernel (k <= 256)");
    const char *rs_name = widx ? "rowsum_items" : (active ? "rowsum_users_active" : "rowsum_users");
    if (n_units > 0) {
        PCR_CUDA(cudaMemsetAsync(c.ticket, 0, sizeof(unsigned long long), c.stream));
        // L2 hints on the item-major pass only: measured -2.3 % per launch (profiles/experiments/README.md r02_rowsum_l2hint)
#define RSL(N, H) { const unsigned grid = resident_grid(rowsum_kernel<N, H>, 256, 0, c.sms, (n_units + 7) / 8); \
                  LAUNCH(c, rs_name, bytes, (rowsum_kernel<N, H>), grid, 256, 0, un_seg, un_start, un_end, n_units, c.ticket, ridx, widx, w, M, ld, nch, active, partial); }
#define RS(N) { if (widx) RSL(N, true) else RSL(N, false) }
        switch (NCH) { case 1: RS(1) break; case 2: RS(2) break; case 3: RS(3) break; default: RS(4) break; }
#undef RS
#undef RSL
    }
    if (n_seg > 0)
        LAUNCH(c, "rowsum_finalize", 0.0, rowsum_finalize_kernel, grid_for(n_seg, 8, c.sms * 8), 256, 0, seg_unit_ptr, seg_unit_idx, n_seg,
               partial, ld, active, lambda, x, out, zero_if_empty, 2 * nch);
}

// ------------------------------------------------------------------ K2: per-user bitonic sort (classes S and L)

template <int THREADS, int CAP>
__global__ void __launch_bounds__(THREADS) sort_users_kernel(const int32_t *__restrict__ users, int n_users,
                                                             const uint8_t *__restrict__ active,
                                                             const i64 *__restrict__ row_ptr,
                                                             const double *__restrict__ m,
                                                             const uint8_t *__restrict__ level,
                                                             double *__restrict__ s_out, int32_t *__restrict__ pos_out,
                                                             uint8_t *__restrict__ lev_out) {
    __shared__ double keys[CAP];
    __shared__ uint16_t idx[CAP];
    const int u = users[blockIdx.x];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    int np2 = 1;
    while (np2 < n) np2 <<= 1;
    const int tid = threadIdx.x;
    for (int j = tid; j < np2; j += THREADS) {
        keys[j] = j < n ? m[start + j] : CUDART_INF;
        idx[j] = (uint16_t)j;
    }
    __syncthreads();
    for (int k = 2; k <= np2; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int t = tid; t < (np2 >> 1); t += THREADS) {
                const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                const int p = i | j;
                const bool asc = (i & k) == 0;
                const double ki = keys[i], kp = keys[p];
                const uint16_t ii = idx[i], ip = idx[p];
                const bool gt = (ki > kp) || (ki == kp && ii > ip);
                if (gt == asc) { keys[i] = kp; keys[p] = ki; idx[i] = ip; idx[p] = ii; }
            }
            __syncthreads();
        }
    }
    for (int j = tid; j < n; j += THREADS) {
        const int src = idx[j];
        s_out[start + j] = keys[j];
        pos_out[start + j] = (int32_t)(start + src);
        lev_out[start + j] = level[start + src];
    }
}

void k_sort_users(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                  const double *m, const uint8_t *level, SortedMeta &meta) {
    if (n_users <= 0) return;
    if (cls == 0)
        LAUNCH(c, "sort_users_S", 0.0, (sort_users_kernel<256, S_CAP>), n_users, 256, 0, users, n_users, active, row_ptr, m, level, meta.s, meta.pos, meta.lev);
    else
        LAUNCH(c, "sort_users_L", 0.0, (sort_users_kernel<1024, L_CAP>), n_users, 1024, 0, users, n_users, active, row_ptr, m, level, meta.s, meta.pos, meta.lev);
}

// heavy users: k_hsort.cu wrote s and pos; fetch the levels
__global__ void __launch_bounds__(256) gather_level_kernel(const int32_t *__restrict__ users, int n_users,
                                                           const uint8_t *__restrict__ active,
                                                           const i64 *__restrict__ row_ptr,
                                                           const uint8_t *__restrict__ level,
                                                           const int32_t *__restrict__ pos, uint8_t *__restrict__ lev_out) {
    const int u = users[blockIdx.x];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u], end = row_ptr[u + 1];
    for (i64 j = start + threadIdx.x; j < end; j += 256) lev_out[j] = level[pos[j]];
}

void k_gather_level(Ctx &c, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                    const uint8_t *level, SortedMeta &meta) {
    if (n_users <= 0) return;
    LAUNCH(c, "gather_level", 0.0, gather_level_kernel, n_users, 256, 0, users, n_users, active, row_ptr, level, meta.pos, meta.lev);
}

// ------------------------------------------------------------------ K3: window pointers + integer level counters
//
// ub_j = #{q : s_q <= fl(s_j + 1.0)}  (now_left  after the first  while loop, pcrpp.cpp:218-223)
// lb_j = #{q : s_q <  fl(s_j - 1.0)}  (now_right after the second while loop, pcrpp.cpp:224-229)
// cnt_hi_j = sum_{t > l_j} count_left[t]  = #{q < ub_j : l_q > l_j}
// cnt_lo_j = sum_{t < l_j} count_right[t] = #{q >= lb_j : l_q < l_j}
// computed with one exclusive scan per level threshold t: C(x) = #{q < x : l_q >= t}.

template <int THREADS>
__global__ void __launch_bounds__(THREADS) windows_kernel(const int32_t *__restrict__ users, int n_users,
                                                          const uint8_t *__restrict__ active,
                                                          const i64 *__restrict__ row_ptr,
                                                          const double *__restrict__ s_g, const uint8_t *__restrict__ lev_g,
                                                          int32_t *__restrict__ ub_g, int32_t *__restrict__ lb_g,
                                                          int32_t *__restrict__ lo_g, int32_t *__restrict__ hi_g,
                                                          int T, int smem_cap, const i64 *__restrict__ heavy_off,
                                                          int32_t *__restrict__ g_cnt) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ int wsum[THREADS / 32 + 1];
    __shared__ unsigned s_mask[MAX_LEVELS / 32];
    const int u = users[blockIdx.x];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const int tid = threadIdx.x;
    const double *keys;
    int *cnt;
    if (tid < MAX_LEVELS / 32) s_mask[tid] = 0u;
    if (n <= smem_cap) {
        double *k = reinterpret_cast<double *>(smraw);
        for (int j = tid; j < n; j += THREADS) k[j] = s_g[start + j];
        keys = k;
        cnt = reinterpret_cast<int *>(k + smem_cap);
    } else {
        keys = s_g + start;
        cnt = g_cnt + heavy_off[u];
    }
    __syncthreads();
    for (int j = tid; j < n; j += THREADS) {
        const double sj = keys[j];
        const double hi = __dadd_rn(sj, 1.0), lo = __dadd_rn(sj, -1.0);
        int a = j + 1, b = n;            // first q in [j+1, n] with keys[q] > hi
        while (a < b) { const int mid = (a + b) >> 1; if (keys[mid] <= hi) a = mid + 1; else b = mid; }
        const int ub = a;
        a = 0; b = j;                    // first q in [0, j] with keys[q] >= lo
        while (a < b) { const int mid = (a + b) >> 1; if (keys[mid] < lo) a = mid + 1; else b = mid; }
        const int lb = a;
        ub_g[start + j] = ub; lb_g[start + j] = lb;
        lo_g[start + j] = 0;  hi_g[start + j] = 0;
        lvl_mark(s_mask, lev_g[start + j]);
    }
    __syncthreads();
    for (int t = 1; t < T; ++t) {
        if (!lvl_has(s_mask, t) && !lvl_has(s_mask, t - 1)) continue;     // block-uniform
        for (int j = tid; j < n; j += THREADS) cnt[j] = lev_g[start + j] >= t ? 1 : 0;
        __syncthreads();
        block_excl_scan<int, THREADS>(cnt, n, wsum);
        const int total = cnt[n];
        for (int j = tid; j < n; j += THREADS) {
            const int l = lev_g[start + j];
            if (l + 1 == t) hi_g[start + j] = cnt[ub_g[start + j]];
            if (l == t) { const int lb = lb_g[start + j]; lo_g[start + j] = (n - lb) - (total - cnt[lb]); }
        }
        __syncthreads();
    }
}

void k_windows(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
               SortedMeta &meta, int T, const i64 *heavy_off, int32_t *g_cnt) {
    if (n_users <= 0) return;
    if (cls == 0) {
        const size_t sm = (size_t)S_CAP * 8 + ((size_t)S_CAP + 1) * 4;
        LAUNCH(c, "windows_S", 0.0, windows_kernel<256>, n_users, 256, sm, users, n_users, active, row_ptr, meta.s, meta.lev,
               meta.ub, meta.lb, meta.cnt_lo, meta.cnt_hi, T, S_CAP, heavy_off, g_cnt);
    } else if (cls == 1) {
        const size_t sm = (size_t)L_CAP * 8 + ((size_t)L_CAP + 1) * 4;
        PCR_CUDA(cudaFuncSetAttribute(windows_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        LAUNCH(c, "windows_L", 0.0, windows_kernel<1024>, n_users, 1024, sm, users, n_users, active, row_ptr, meta.s, meta.lev,
               meta.ub, meta.lb, meta.cnt_lo, meta.cnt_hi, T, L_CAP, heavy_off, g_cnt);
    } else {
        LAUNCH(c, "windows_H", 0.0, windows_kernel<1024>, n_users, 1024, 0, users, n_users, active, row_ptr, meta.s, meta.lev,
               meta.ub, meta.lb, meta.cnt_lo, meta.cnt_hi, T, 0, heavy_off, g_cnt);
    }
}

// test entry point: the per-level counters themselves, by direct counting from ub / lb
__global__ void __launch_bounds__(128) level_counts_kernel(const i64 *__restrict__ row_ptr, i64 d1,
                                                           const uint8_t *__restrict__ lev, const int32_t *__restrict__ ub,
                                                           const int32_t *__restrict__ lb, int T,
                                                           int32_t *__restrict__ cntL, int32_t *__restrict__ cntR) {
    const i64 u = blockIdx.x;
    if (u >= d1) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    for (int j = threadIdx.x; j < n; j += 128) {
        int cl[MAX_LEVELS], cr[MAX_LEVELS];
        for (int t = 0; t < T; ++t) { cl[t] = 0; cr[t] = 0; }
        const int ubj = ub[start + j], lbj = lb[start + j];
        for (int q = 0; q < n; ++q) {
            const int l = lev[start + q];
            if (q < ubj) cl[l]++;
            if (q >= lbj) cr[l]++;
        }
        for (int t = 0; t < T; ++t) { cntL[(start + j) * T + t] = cl[t]; cntR[(start + j) * T + t] = cr[t]; }
    }
}

void k_level_counts(Ctx &c, const i64 *row_ptr, i64 d1, const SortedMeta &meta, int T, int32_t *cntL, int32_t *cntR) {
    if (d1 <= 0) return;
    LAUNCH(c, "level_counts", 0.0, level_counts_kernel, (unsigned)d1, 128, 0, row_ptr, d1, meta.lev, meta.ub, meta.lb, T, cntL, cntR);
}

// ------------------------------------------------------------------ K3: sweep coefficients
//
// gradient (MODE 0, stream v = s):  c_j = 2 [ cnt_lo (s_j - 1) + cnt_hi (s_j + 1) - acc_j ]
// Hv       (MODE 1, stream v = b):  c_j = 2 [ (cnt_lo + cnt_hi) b_j - acc_j ]
// acc_j = sum_{t < l_j} (S_t(n) - S_t(lb_j)) + sum_{t > l_j} S_t(ub_j),  S_t(x) = sum_{q < x, l_q = t} v_q

template <int THREADS, int MODE>
__global__ void __launch_bounds__(THREADS) sweep_coeff_kernel(const int32_t *__restrict__ users, int n_users,
                                                              const uint8_t *__restrict__ active,
                                                              const i64 *__restrict__ row_ptr,
                                                              const double *__restrict__ s_g, const int32_t *__restrict__ pos_g,
                                                              const uint8_t *__restrict__ lev_g,
                                                              const int32_t *__restrict__ ub_g, const int32_t *__restrict__ lb_g,
                                                              const int32_t *__restrict__ lo_g, const int32_t *__restrict__ hi_g,
                                                              const double *__restrict__ b_g, double *__restrict__ c_out,
                                                              int T, int smem_cap, const i64 *__restrict__ heavy_off,
                                                              double *__restrict__ g_v, double *__restrict__ g_p,
                                                              double *__restrict__ g_acc) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double wsum[THREADS / 32 + 1];
    __shared__ unsigned s_mask[MAX_LEVELS / 32];
    const int u = users[blockIdx.x];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const int tid = threadIdx.x;
    double *v, *P, *acc;
    if (n <= smem_cap) {
        v = reinterpret_cast<double *>(smraw); P = v + smem_cap; acc = P + smem_cap + 1;
    } else {
        const i64 off = heavy_off[u];
        v = g_v + off; P = g_p + off; acc = g_acc + off;
    }
    if (tid < MAX_LEVELS / 32) s_mask[tid] = 0u;
    __syncthreads();
    for (int j = tid; j < n; j += THREADS) {
        v[j] = MODE == 0 ? s_g[start + j] : b_g[pos_g[start + j]];
        acc[j] = 0.0;
        lvl_mark(s_mask, lev_g[start + j]);
    }
    __syncthreads();
    if (lvl_count(s_mask) >= 2) {          // at least two levels present, otherwise every c_j is 0
        for (int t = 0; t < T; ++t) {
            if (!lvl_has(s_mask, t)) continue;
            for (int j = tid; j < n; j += THREADS) P[j] = lev_g[start + j] == t ? v[j] : 0.0;
            __syncthreads();
            block_excl_scan<double, THREADS>(P, n, wsum);
            const double total = P[n];
            for (int j = tid; j < n; j += THREADS) {
                const int l = lev_g[start + j];
                if (l < t) acc[j] += P[ub_g[start + j]];
                else if (l > t) acc[j] += total - P[lb_g[start + j]];
            }
            __syncthreads();
        }
    }
    for (int j = tid; j < n; j += THREADS) {
        const double lo = (double)lo_g[start + j], hi = (double)hi_g[start + j];
        double cc;
        if (MODE == 0) {
            const double sj = v[j];
            cc = lo * (sj - 1.0) + hi * (sj + 1.0) - acc[j];
        } else {
            cc = (lo + hi) * v[j] - acc[j];
        }
        c_out[pos_g[start + j]] = 2.0 * cc;
    }
}

void k_sweep_coeff(Ctx &c, int cls, int mode, const int32_t *users, int n_users, const uint8_t *active,
                   const i64 *row_ptr, const SortedMeta &meta, const double *b, double *c_out, int T,
                   const i64 *heavy_off, double *g_v, double *g_p, double *g_acc) {
    if (n_users <= 0) return;
#define SWEEP_ARGS users, n_users, active, row_ptr, meta.s, meta.pos, meta.lev, meta.ub, meta.lb, meta.cnt_lo, meta.cnt_hi, b, c_out, T
    if (cls == 0) {
        const size_t sm = ((size_t)3 * S_CAP + 1) * 8;
        if (mode == 0) LAUNCH(c, "sweep_grad_S", 0.0, (sweep_coeff_kernel<256, 0>), n_users, 256, sm, SWEEP_ARGS, S_CAP, heavy_off, g_v, g_p, g_acc);
        else           LAUNCH(c, "sweep_hv_S",   0.0, (sweep_coeff_kernel<256, 1>), n_users, 256, sm, SWEEP_ARGS, S_CAP, heavy_off, g_v, g_p, g_acc);
    } else if (cls == 1) {
        const size_t sm = ((size_t)3 * L_CAP + 1) * 8;
        PCR_CUDA(cudaFuncSetAttribute(sweep_coeff_kernel<1024, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        PCR_CUDA(cudaFuncSetAttribute(sweep_coeff_kernel<1024, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        if (mode == 0) LAUNCH(c, "sweep_grad_L", 0.0, (sweep_coeff_kernel<1024, 0>), n_users, 1024, sm, SWEEP_ARGS, L_CAP, heavy_off, g_v, g_p, g_acc);
        else           LAUNCH(c, "sweep_hv_L",   0.0, (sweep_coeff_kernel<1024, 1>), n_users, 1024, sm, SWEEP_ARGS, L_CAP, heavy_off, g_v, g_p, g_acc);
    } else {
        if (mode == 0) LAUNCH(c, "sweep_grad_H", 0.0, (sweep_coeff_kernel<1024, 0>), n_users, 1024, 0, SWEEP_ARGS, 0, heavy_off, g_v, g_p, g_acc);
        else           LAUNCH(c, "sweep_hv_H",   0.0, (sweep_coeff_kernel<1024, 1>), n_users, 1024, 0, SWEEP_ARGS, 0, heavy_off, g_v, g_p, g_acc);
    }
#undef SWEEP_ARGS
}

// ------------------------------------------------------------------ K3: objective sweep
// loss_u = sum_j [ cnt_hi_j s_j^2 - 2 s_j sum_{t>l_j} S1_t(ub_j) + sum_{t>l_j} S2_t(ub_j) ],
// S1 = prefix of (s-1), S2 = prefix of (s-1)^2 per level   (objective_new pcrpp.cpp:392-407)

template <int THREADS>
__global__ void __launch_bounds__(THREADS) sweep_obj_kernel(const int32_t *__restrict__ users, int n_users,
                                                            const uint8_t *__restrict__ active,
                                                            const i64 *__restrict__ row_ptr,
                                                            const double *__restrict__ s_g, const uint8_t *__restrict__ lev_g,
                                                            const int32_t *__restrict__ ub_g, const int32_t *__restrict__ hi_g,
                                                            double *__restrict__ obj_user, int T, int smem_cap,
                                                            const i64 *__restrict__ heavy_off, double *__restrict__ g_p1,
                                                            double *__restrict__ g_p2, double *__restrict__ g_acc) {
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ double wsum[THREADS / 32 + 1];
    __shared__ unsigned s_mask[MAX_LEVELS / 32];
    const int u = users[blockIdx.x];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const int tid = threadIdx.x;
    double *P1, *P2, *acc;
    if (n <= smem_cap) {
        P1 = reinterpret_cast<double *>(smraw); P2 = P1 + smem_cap + 1; acc = P2 + smem_cap + 1;
    } else {
        const i64 off = heavy_off[u];
        P1 = g_p1 + off; P2 = g_p2 + off; acc = g_acc + off;
    }
    if (tid < MAX_LEVELS / 32) s_mask[tid] = 0u;
    __syncthreads();
    for (int j = tid; j < n; j += THREADS) { acc[j] = 0.0; lvl_mark(s_mask, lev_g[start + j]); }
    __syncthreads();
    if (lvl_count(s_mask) >= 2) {
        for (int t = 1; t < T; ++t) {
            if (!lvl_has(s_mask, t)) continue;
            if (!lvl_any_below(s_mask, t)) continue;      // nothing below level t
            for (int j = tid; j < n; j += THREADS) {
                const double d = s_g[start + j] - 1.0;
                const bool on = lev_g[start + j] == t;
                P1[j] = on ? d : 0.0;
                P2[j] = on ? d * d : 0.0;
            }
            __syncthreads();
            block_excl_scan<double, THREADS>(P1, n, wsum);
            block_excl_scan<double, THREADS>(P2, n, wsum);
            for (int j = tid; j < n; j += THREADS) {
                if (lev_g[start + j] < t) {
                    const int ub = ub_g[start + j];
                    const double sj = s_g[start + j];
                    acc[j] += P2[ub] - 2.0 * sj * P1[ub];
                }
            }
            __syncthreads();
        }
    }
    double part = 0.0;
    for (int j = tid; j < n; j += THREADS) {
        const double sj = s_g[start + j];
        part += (double)hi_g[start + j] * (sj * sj) + acc[j];
    }
    const double tot = block_sum<THREADS>(part, wsum);
    if (tid == 0) obj_user[u] = tot;
}

void k_sweep_obj(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                 const SortedMeta &meta, double *obj_user, int T, const i64 *heavy_off, double *g_p1, double *g_p2,
                 double *g_acc) {
    if (n_users <= 0) return;
#define OBJ_ARGS users, n_users, active, row_ptr, meta.s, meta.lev, meta.ub, meta.cnt_hi, obj_user, T
    if (cls == 0) {
        const size_t sm = ((size_t)3 * S_CAP + 2) * 8;
        LAUNCH(c, "sweep_obj_S", 0.0, sweep_obj_kernel<256>, n_users, 256, sm, OBJ_ARGS, S_CAP, heavy_off, g_p1, g_p2, g_acc);
    } else if (cls == 1) {
        const size_t sm = ((size_t)3 * L_CAP + 2) * 8;
        PCR_CUDA(cudaFuncSetAttribute(sweep_obj_kernel<1024>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        LAUNCH(c, "sweep_obj_L", 0.0, sweep_obj_kernel<1024>, n_users, 1024, sm, OBJ_ARGS, L_CAP, heavy_off, g_p1, g_p2, g_acc);
    } else {
        LAUNCH(c, "sweep_obj_H", 0.0, sweep_obj_kernel<1024>, n_users, 1024, 0, OBJ_ARGS, 0, heavy_off, g_p1, g_p2, g_acc);
    }
#undef OBJ_ARGS
}

// ------------------------------------------------------------------ K5: dense vector helpers

__global__ void fill_kernel(double *x, i64 n, double v) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) x[i] = v;
}
// out may alias x or y (in-place CG updates): no __restrict__ here
__global__ void axpby_kernel(double *out, double a, const double *x, double b, const double *y, i64 n) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x)
        out[i] = a * x[i] + b * y[i];
}

static const int RED_BLOCKS = 592;   // 4 x 148

// MODE 0: x.y   1: sum x
template <int MODE>
__global__ void __launch_bounds__(256) reduce_kernel(const double *__restrict__ x, const double *__restrict__ y, i64 n,
                                                     double *__restrict__ partials) {
    __shared__ double wsum[8];
    double acc = 0.0;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n; i += (i64)gridDim.x * 256) {
        if (MODE == 0) acc = fma(x[i], y[i], acc);
        else acc += x[i];
    }
    const double t = block_sum<256>(acc, wsum);
    if (threadIdx.x == 0) partials[blockIdx.x] = t;
}
__global__ void __launch_bounds__(256) reduce_final_kernel(const double *__restrict__ partials, int nb, double *__restrict__ slot) {
    __shared__ double wsum[8];
    double acc = 0.0;
    for (int i = threadIdx.x; i < nb; i += 256) acc += partials[i];
    const double t = block_sum<256>(acc, wsum);
    if (threadIdx.x == 0) *slot = t;
}

// ---- fused vector algebra of one V-side CG iteration (solve_delta_new pcrpp.cpp:344-352).  Same per-thread
// accumulation order, block tree and final reduction as reduce_kernel<0>, so the scalars equal those of separate k_dot calls.
// partials[0..RED_BLOCKS) <- p.Hp, partials[RED_BLOCKS..2 RED_BLOCKS) <- rr.p
__global__ void __launch_bounds__(256) cg_dots2_kernel(const double *__restrict__ p, const double *__restrict__ Hp,
                                                       const double *__restrict__ rr, i64 n, double *__restrict__ partials) {
    __shared__ double wsum[8];
    double a0 = 0.0, a1 = 0.0;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n; i += (i64)gridDim.x * 256) {
        const double pi = p[i];
        a0 = fma(pi, Hp[i], a0);
        a1 = fma(rr[i], pi, a1);
    }
    const double t0 = block_sum<256>(a0, wsum);
    if (threadIdx.x == 0) partials[blockIdx.x] = t0;
    const double t1 = block_sum<256>(a1, wsum);
    if (threadIdx.x == 0) partials[gridDim.x + blockIdx.x] = t1;
}
// alpha = -(rr.p) / (p.Hp) from slot[1], slot[0]; delta += alpha p; rr += alpha Hp; partials of rr.rr and rr.Hp
__global__ void __launch_bounds__(256) cg_update_kernel(double *__restrict__ delta, double *__restrict__ rr,
                                                        const double *__restrict__ p, const double *__restrict__ Hp, i64 n,
                                                        const double *__restrict__ slot, double *__restrict__ partials) {
    __shared__ double wsum[8];
    const double alpha = -1.0 * slot[1] / slot[0];
    double a0 = 0.0, a1 = 0.0;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < n; i += (i64)gridDim.x * 256) {
        const double hp = Hp[i];
        delta[i] = delta[i] + alpha * p[i];
        const double r = rr[i] + alpha * hp;
        rr[i] = r;
        a0 = fma(r, r, a0);
        a1 = fma(r, hp, a1);
    }
    const double t0 = block_sum<256>(a0, wsum);
    if (threadIdx.x == 0) partials[blockIdx.x] = t0;
    const double t1 = block_sum<256>(a1, wsum);
    if (threadIdx.x == 0) partials[gridDim.x + blockIdx.x] = t1;
}
// slot[b] = sum of partials[b * nb .. (b + 1) * nb)   (one block per slot)
__global__ void __launch_bounds__(256) reduce_final_multi_kernel(const double *__restrict__ partials, int nb, double *__restrict__ slot) {
    __shared__ double wsum[8];
    double acc = 0.0;
    for (int i = threadIdx.x; i < nb; i += 256) acc += partials[(size_t)blockIdx.x * nb + i];
    const double t = block_sum<256>(acc, wsum);
    if (threadIdx.x == 0) slot[blockIdx.x] = t;
}
void k_cg_dots2(Ctx &c, const double *p, const double *Hp, const double *rr, i64 n, double *partials, double *slot2) {
    LAUNCH(c, "cg_dots2", 24.0 * n, cg_dots2_kernel, RED_BLOCKS, 256, 0, p, Hp, rr, n, partials);
    LAUNCH(c, "reduce_final", 0.0, reduce_final_multi_kernel, 2, 256, 0, partials, RED_BLOCKS, slot2);
}
void k_cg_update(Ctx &c, double *delta, double *rr, const double *p, const double *Hp, i64 n, const double *slot_in, double *partials,
                 double *slot2_out) {
    LAUNCH(c, "cg_update", 48.0 * n, cg_update_kernel, RED_BLOCKS, 256, 0, delta, rr, p, Hp, n, slot_in, partials);
    LAUNCH(c, "reduce_final", 0.0, reduce_final_multi_kernel, 2, 256, 0, partials, RED_BLOCKS, slot2_out);
}

void k_fill(Ctx &c, double *x, i64 n, double v) {
    if (n <= 0) return;
    LAUNCH(c, "fill", 0.0, fill_kernel, grid_for(n, 1024, c.sms * 8), 256, 0, x, n, v);
}
void k_axpby(Ctx &c, double *out, double a, const double *x, double b, const double *y, i64 n) {
    if (n <= 0) return;
    LAUNCH(c, "axpby", 24.0 * n, axpby_kernel, grid_for(n, 1024, c.sms * 8), 256, 0, out, a, x, b, y, n);
}
void k_dot(Ctx &c, const double *x, const double *y, i64 n, double *partials, double *slot) {
    LAUNCH(c, "dot", 16.0 * n, reduce_kernel<0>, RED_BLOCKS, 256, 0, x, y, n, partials);
    LAUNCH(c, "reduce_final", 0.0, reduce_final_kernel, 1, 256, 0, partials, RED_BLOCKS, slot);
}
void k_sum(Ctx &c, const double *x, i64 n, double *partials, double *slot) {
    LAUNCH(c, "sum", 8.0 * n, reduce_kernel<1>, RED_BLOCKS, 256, 0, x, (const double *)nullptr, n, partials);
    LAUNCH(c, "reduce_final", 0.0, reduce_final_kernel, 1, 256, 0, partials, RED_BLOCKS, slot);
}

__global__ void pad_copy_kernel(const double *__restrict__ src, i64 rows, int k, int ld, double *__restrict__ dst) {
    const i64 total = rows * ld;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (i64)gridDim.x * blockDim.x) {
        const i64 r = i / ld; const int cidx = (int)(i - r * ld);
        dst[i] = cidx < k ? src[r * k + cidx] : 0.0;
    }
}
void k_pad_copy(Ctx &c, const double *src, i64 rows, int k, int ld, double *dst) {
    if (rows <= 0) return;
    LAUNCH(c, "pad_copy", 0.0, pad_copy_kernel, grid_for(rows * ld, 1024, c.sms * 8), 256, 0, src, rows, k, ld, dst);
}

// ------------------------------------------------------------------ K6: batched per-user Newton-CG bookkeeping
// One warp per user; the k-vectors live in [d1 x ld] arrays.  Follows update_u_new pcrpp.cpp:779-815 /
// update_u pcr.cpp:523-585 and solve_delta_u(_new) pcrpp.cpp:628-647 / pcr.cpp:498-520.

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    return v;
}

// after g (d1 x ld) and loss (d1) are known: prev_obj, skip test, CG initial state.  Register-resident for ld <= 64 * NV
// doubles: every lane owns NV 16-byte chunks of the user's k-vectors, each array is read once (all loads issued up front)
// and written once.
template <int NV>
__global__ void __launch_bounds__(256) u_init_vec_kernel(UState s, const double *__restrict__ U, const i64 *__restrict__ row_ptr,
                                                         const uint8_t *__restrict__ has_pairs, i64 d1, int ld, double lambda) {
    const int lane = threadIdx.x & 31;
    const i64 i = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (i >= d1) return;
    const size_t o = (size_t)i * ld;
    const int n2 = ld >> 1;
    const double2 *g2 = reinterpret_cast<const double2 *>(s.g + o), *u2 = reinterpret_cast<const double2 *>(U + o);
    double2 g[NV], u[NV];
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int c = lane + 32 * q;
        g[q] = c < n2 ? g2[c] : make_double2(0.0, 0.0);
        u[q] = c < n2 ? u2[c] : make_double2(0.0, 0.0);
    }
    double gg = 0.0, uu = 0.0;
#pragma unroll
    for (int q = 0; q < NV; ++q) { gg = fma(g[q].x, g[q].x, gg); gg = fma(g[q].y, g[q].y, gg); uu = fma(u[q].x, u[q].x, uu); uu = fma(u[q].y, u[q].y, uu); }
    gg = warp_sum(gg); uu = warp_sum(uu);
    const double prev = lambda / 2.0 * uu + s.loss[i];
    const bool skip = (gg < 0.0001) || (has_pairs != nullptr && !has_pairs[i]);
    double2 *d2p = reinterpret_cast<double2 *>(s.delta + o), *r2 = reinterpret_cast<double2 *>(s.rr + o);
    double2 *p2 = reinterpret_cast<double2 *>(s.p + o), *n2p = reinterpret_cast<double2 *>(s.Unew + o);
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int c = lane + 32 * q;
        if (c < n2) { d2p[c] = make_double2(0.0, 0.0); r2[c] = make_double2(-g[q].x, -g[q].y); p2[c] = g[q]; n2p[c] = u[q]; }
    }
    if (lane == 0) {
        s.prev_obj[i] = prev; s.obj_new[i] = prev;
        s.err[i] = sqrt(gg) * 0.01;
        s.skipped[i] = skip ? 1 : 0; s.cg_active[i] = skip ? 0 : 1; s.ls_active[i] = 0;
        s.cg_its[i] = 0; s.ls_trials[i] = 0;
        if (!skip) atomicAdd(&s.counters[0], 1);
    }
}

// rowsum_finalize (user side) + one CG iteration's updates in one pass: the warp that adds up a user's partial rows into
// Hp = lambda p + V_i^T c keeps the row in registers and runs the user's CG recurrences on it right away -- Hp is never
// written or re-read.  Same additions in the same order as rowsum_finalize_kernel.
template <int NV>
__global__ void __launch_bounds__(256) u_finalize_cg_kernel(const i64 *__restrict__ seg_unit_ptr,
                                                            const double *__restrict__ partial, UState s, i64 d1, int ld, int kp,
                                                            double lambda) {
    const int lane = threadIdx.x & 31;
    const i64 i = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (i >= d1) return;
    if (!s.cg_active[i]) return;
    const size_t o = (size_t)i * ld;
    const int n2 = ld >> 1, nch = kp >> 1;
    double2 *p2 = reinterpret_cast<double2 *>(s.p + o), *r2 = reinterpret_cast<double2 *>(s.rr + o);
    double2 *d2p = reinterpret_cast<double2 *>(s.delta + o);
    double2 p[NV], hp[NV], rr[NV], dl[NV];
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int c = lane + 32 * q;
        const double2 z = make_double2(0.0, 0.0);
        p[q] = c < n2 ? p2[c] : z; rr[q] = c < n2 ? r2[c] : z; dl[q] = c < n2 ? d2p[c] : z;
        hp[q] = c < nch ? make_double2(lambda * p[q].x, lambda * p[q].y) : z;        // rowsum_finalize: v = lambda * x ...
    }
    for (i64 u = seg_unit_ptr[i]; u < seg_unit_ptr[i + 1]; ++u) {                    // ... + the unit partials, in list order
        const double2 *prow = reinterpret_cast<const double2 *>(partial + (size_t)u * ld);
#pragma unroll
        for (int q = 0; q < NV; ++q) {
            const int c = lane + 32 * q;
            if (c < nch) { const double2 t = prow[c]; hp[q].x += t.x; hp[q].y += t.y; }
        }
    }
    double pHp = 0.0, rp = 0.0;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        pHp = fma(p[q].x, hp[q].x, pHp); pHp = fma(p[q].y, hp[q].y, pHp);
        rp = fma(rr[q].x, p[q].x, rp); rp = fma(rr[q].y, p[q].y, rp);
    }
    pHp = warp_sum(pHp); rp = warp_sum(rp);
    const double alpha = -1.0 * rp / pHp;
    double nr = 0.0, rHp = 0.0;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        dl[q].x = dl[q].x + p[q].x * alpha; dl[q].y = dl[q].y + p[q].y * alpha;
        rr[q].x = rr[q].x + hp[q].x * alpha; rr[q].y = rr[q].y + hp[q].y * alpha;
        nr = fma(rr[q].x, rr[q].x, nr); nr = fma(rr[q].y, rr[q].y, nr);
        rHp = fma(rr[q].x, hp[q].x, rHp); rHp = fma(rr[q].y, hp[q].y, rHp);
    }
    nr = warp_sum(nr); rHp = warp_sum(rHp);
    const int its = s.cg_its[i] + 1;
    const bool done = (sqrt(nr) < s.err[i]) || (its >= 10);
    const double beta = rHp / pHp;
#pragma unroll
    for (int q = 0; q < NV; ++q) {
        const int c = lane + 32 * q;
        if (c < n2) {
            d2p[c] = dl[q]; r2[c] = rr[q];
            if (!done) p2[c] = make_double2(-rr[q].x + p[q].x * beta, -rr[q].y + p[q].y * beta);
        }
    }
    if (lane == 0) {
        s.cg_its[i] = its;
        if (done) s.cg_active[i] = 0; else atomicAdd(&s.counters[0], 1);
    }
}

void k_u_finalize_cg(Ctx &c, const i64 *seg_unit_ptr, const double *partial, UState &s, i64 d1, int ld, int kk, double lambda) {
    if (d1 <= 0) return;
    PCR_REQUIRE(ld <= 256, "rank too large for the per-user CG kernels (k <= 256)");
    const unsigned grid = (unsigned)((d1 + 7) / 8);
    const int kp = 2 * ((kk + 1) / 2);
    if (ld <= 64) LAUNCH(c, "u_finalize_cg", 0.0, u_finalize_cg_kernel<1>, grid, 256, 0, seg_unit_ptr, partial, s, d1, ld, kp, lambda);
    else if (ld <= 128) LAUNCH(c, "u_finalize_cg", 0.0, u_finalize_cg_kernel<2>, grid, 256, 0, seg_unit_ptr, partial, s, d1, ld, kp, lambda);
    else LAUNCH(c, "u_finalize_cg", 0.0, u_finalize_cg_kernel<4>, grid, 256, 0, seg_unit_ptr, partial, s, d1, ld, kp, lambda);
}

__global__ void __launch_bounds__(256) u_ls_begin_kernel(UState s, i64 d1, double stepsize0) {
    const i64 i = (i64)blockIdx.x * 256 + threadIdx.x;
    if (i >= d1) return;
    const bool on = !s.skipped[i];
    s.ls_active[i] = on ? 1 : 0;
    s.step[i] = stepsize0;
    if (on) atomicAdd(&s.counters[1], 1);
}

// ui_new = ui - step * delta for users still searching
__global__ void __launch_bounds__(256) u_ls_trial_kernel(UState s, const double *__restrict__ U, i64 d1, int ld) {
    const int lane = threadIdx.x & 31;
    const i64 i = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (i >= d1) return;
    if (!s.ls_active[i]) return;
    const size_t o = (size_t)i * ld;
    const double st = s.step[i];
    for (int cidx = lane; cidx < ld; cidx += 32) s.Unew[o + cidx] = U[o + cidx] + s.delta[o + cidx] * (-st);
}

// loss[i] now holds the trial's loss: accept / halve (pcrpp.cpp:802-812)
__global__ void __launch_bounds__(256) u_ls_check_kernel(UState s, i64 d1, int ld, double lambda) {
    const int lane = threadIdx.x & 31;
    const i64 i = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (i >= d1) return;
    if (!s.ls_active[i]) return;
    const size_t o = (size_t)i * ld;
    double uu = 0.0;
    for (int cidx = lane; cidx < ld; cidx += 32) { const double u = s.Unew[o + cidx]; uu = fma(u, u, uu); }
    uu = warp_sum(uu);
    if (lane == 0) {
        const double obj = lambda / 2.0 * uu + s.loss[i];
        s.obj_new[i] = obj;
        const int tr = s.ls_trials[i] + 1;
        s.ls_trials[i] = tr;
        if (obj < s.prev_obj[i] || tr >= 20) s.ls_active[i] = 0;
        else { s.step[i] = s.step[i] / 2.0; atomicAdd(&s.counters[1], 1); }
    }
}

__global__ void u_commit_kernel(UState s, double *__restrict__ U, i64 d1, int ld) {
    const i64 total = d1 * ld;
    for (i64 t = (i64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (i64)gridDim.x * blockDim.x) {
        const i64 i = t / ld;
        if (!s.skipped[i]) U[t] = s.Unew[t];
    }
}

__global__ void __launch_bounds__(256) u_stats_kernel(UState s, const i64 *__restrict__ row_ptr, i64 d1, i64 *__restrict__ out8) {
    i64 a = 0, b = 0, sk = 0, ci = 0, li = 0;
    for (i64 i = (i64)blockIdx.x * 256 + threadIdx.x; i < d1; i += (i64)gridDim.x * 256) {
        const i64 len = row_ptr[i + 1] - row_ptr[i];
        a += len * s.cg_its[i]; b += len * s.ls_trials[i]; sk += s.skipped[i]; ci += s.cg_its[i]; li += s.ls_trials[i];
    }
    // warp-level sums first: one atomic per warp and counter instead of one per thread (0.5 ms -> a few microseconds)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        a += __shfl_xor_sync(FULL, a, o); b += __shfl_xor_sync(FULL, b, o); sk += __shfl_xor_sync(FULL, sk, o);
        ci += __shfl_xor_sync(FULL, ci, o); li += __shfl_xor_sync(FULL, li, o);
    }
    if ((threadIdx.x & 31) == 0) {
        atomicAdd((unsigned long long *)&out8[3], (unsigned long long)a);
        atomicAdd((unsigned long long *)&out8[4], (unsigned long long)b);
        atomicAdd((unsigned long long *)&out8[5], (unsigned long long)sk);
        atomicAdd((unsigned long long *)&out8[6], (unsigned long long)ci);
        atomicAdd((unsigned long long *)&out8[7], (unsigned long long)li);
    }
}

void k_u_init(Ctx &c, UState &s, const double *U, const i64 *row_ptr, const uint8_t *has_pairs, i64 d1, int ld, double lambda) {
    if (d1 <= 0) return;
    PCR_REQUIRE(ld <= 256, "rank too large for the per-user CG kernels (k <= 256)");
    const unsigned grid = (unsigned)((d1 + 7) / 8);
    if (ld <= 64) LAUNCH(c, "u_init", 0.0, u_init_vec_kernel<1>, grid, 256, 0, s, U, row_ptr, has_pairs, d1, ld, lambda);
    else if (ld <= 128) LAUNCH(c, "u_init", 0.0, u_init_vec_kernel<2>, grid, 256, 0, s, U, row_ptr, has_pairs, d1, ld, lambda);
    else LAUNCH(c, "u_init", 0.0, u_init_vec_kernel<4>, grid, 256, 0, s, U, row_ptr, has_pairs, d1, ld, lambda);
}
void k_u_ls_trial(Ctx &c, UState &s, const double *U, i64 d1, int ld, double stepsize0, int first) {
    if (d1 <= 0) return;
    if (first) LAUNCH(c, "u_ls_begin", 0.0, u_ls_begin_kernel, (unsigned)((d1 + 255) / 256), 256, 0, s, d1, stepsize0);
    LAUNCH(c, "u_ls_trial", 0.0, u_ls_trial_kernel, (unsigned)((d1 + 7) / 8), 256, 0, s, U, d1, ld);
}
void k_u_ls_check(Ctx &c, UState &s, i64 d1, int ld, double lambda, int last) {
    (void)last;
    if (d1 <= 0) return;
    LAUNCH(c, "u_ls_check", 0.0, u_ls_check_kernel, (unsigned)((d1 + 7) / 8), 256, 0, s, d1, ld, lambda);
}
void k_u_commit(Ctx &c, UState &s, double *U, i64 d1, int ld) {
    if (d1 <= 0) return;
    LAUNCH(c, "u_commit", 0.0, u_commit_kernel, grid_for(d1 * ld, 1024, c.sms * 8), 256, 0, s, U, d1, ld);
}
void k_u_stats(Ctx &c, UState &s, const i64 *row_ptr, i64 d1, i64 *out8) {
    if (d1 <= 0) return;
    LAUNCH(c, "u_stats", 0.0, u_stats_kernel, grid_for(d1, 256, c.sms * 4), 256, 0, s, row_ptr, d1, out8);
}

}  // namespace pcr
