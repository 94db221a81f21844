// k_tiles.cu -- "tile of users" kernels for the N-sized stages of Primal-CR++ (sort, windows, level sweeps).
//
// A tile is a run of consecutive users whose ratings (<= TILE_CAP in total) are handled by ONE 256-thread CTA as a
// single array with segment boundaries, so thread utilisation does not depend on how short the users are (the
// per-user kernels of k_core.cu keep serving users with more than TILE_CAP ratings).
//
//   tile_prepare  K2+K3  get_sorted_mm pcrpp.cpp:52-83 as one bitonic sort over (user, score, index) keys, then the
//                        window pointers and integer level counters of the sweep pcrpp.cpp:214-229
//   tile_lm_sweep K3     c_j of obtain_g_new :230-238 / compute_Ha_new :310-318 / obtain_g_u_new :527-535 /
//                        obtain_Hs_new :613-621 and the objective :392-407 / :556-571
//
// Per-level exclusive prefix sums S_t(x) = sum_{q<x, l_q=t} v_q of one user are produced by a SEGMENTED blocked scan
// (each thread owns TILE_E consecutive elements; a segment starts at a user's first element) and stored in shared
// memory at slot (x + user_start + user_index): every user gets one extra slot for its totals S_t(n).
#include "kernels.h"
#include <math_constants.h>

namespace pcr {

#define FULL 0xffffffffu
#define LAUNCH(ctx, name, bytes, kernel, grid, block, smem, ...)                         \
    do {                                                                                 \
        (ctx).prof->begin(name, (ctx).stream, (double)(bytes));                          \
        kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);                  \
        (ctx).prof->end((ctx).stream);                                                   \
        PCR_CUDA(cudaGetLastError());                                                    \
    } while (0)

static const int TE = 4;                       // elements per thread (blocked); a tile holds TH * TE ratings
// two geometries: small tiles (256 threads, 1024 ratings) and large tiles (1024 threads, 4096 ratings)

template <int CAP>
struct TileShared {
    int ustart[TILE_MAX_USERS + 1];            // tile-local start of every user; ustart[n_users] = ne
    uint8_t uact[TILE_MAX_USERS];              // user participates (active mask)
    uint8_t ul[CAP];                           // user index (inside the tile) of every element, position order
};

// ---------------------------------------------------------------- segmented blocked scan of per-level streams
// val(i) / lev(i): stream value and level of element i (i in sorted-position order, 0 <= i < ne).
// Writes S[t * SLOTS + slot] for t < T, slot = i + ul[i] (exclusive prefix) and the per-user totals.
template <typename VT, int TT, int TH, typename ValF, typename LevF>
__device__ __forceinline__ void tile_level_scan(const TileShared<TH * TE> &ts, int ne, int T, VT *S, VT *wagg /* [TH/32*TT] */,
                                                int *wflag /* [TH/32] */, ValF val, LevF lev) {
    constexpr int SLOTS = TH * TE + TILE_MAX_USERS;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int lo = tid * TE;
    VT agg[TT];
#pragma unroll
    for (int t = 0; t < TT; ++t) agg[t] = (VT)0;
    int flag = 0;
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = lo + q;
        if (i < ne) {
            const int u = ts.ul[i];
            if (i == ts.ustart[u]) {
#pragma unroll
                for (int t = 0; t < TT; ++t) agg[t] = (VT)0;
                flag = 1;
            }
            const int l = lev(i);
            const VT v = val(i);
#pragma unroll
            for (int t = 0; t < TT; ++t) agg[t] += (t == l) ? v : (VT)0;
        }
    }
    // inclusive segmented warp scan of (agg, flag)
    VT inc[TT];
#pragma unroll
    for (int t = 0; t < TT; ++t) inc[t] = agg[t];
    int finc = flag;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int of = __shfl_up_sync(FULL, finc, o);
#pragma unroll
        for (int t = 0; t < TT; ++t) {
            const VT ov = __shfl_up_sync(FULL, inc[t], o);
            if (lane >= o && !finc) inc[t] += ov;
        }
        if (lane >= o) finc |= of;
    }
    if (lane == 31) {
#pragma unroll
        for (int t = 0; t < TT; ++t) wagg[warp * TT + t] = inc[t];
        wflag[warp] = finc;
    }
    // exclusive within the warp
    VT exc[TT];
    int fexc = __shfl_up_sync(FULL, finc, 1);
#pragma unroll
    for (int t = 0; t < TT; ++t) { exc[t] = __shfl_up_sync(FULL, inc[t], 1); if (lane == 0) exc[t] = (VT)0; }
    if (lane == 0) fexc = 0;
    __syncthreads();
    // carry from the previous warps (sequential over <= 8 entries, same order in every thread => deterministic)
    VT carry[TT];
#pragma unroll
    for (int t = 0; t < TT; ++t) carry[t] = (VT)0;
    for (int w = 0; w < warp; ++w) {
        const int wf = wflag[w];
#pragma unroll
        for (int t = 0; t < TT; ++t) carry[t] = wf ? wagg[w * TT + t] : carry[t] + wagg[w * TT + t];
    }
#pragma unroll
    for (int t = 0; t < TT; ++t) carry[t] = fexc ? exc[t] : carry[t] + exc[t];
    // replay the chunk, emitting exclusive prefixes and the per-user totals
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = lo + q;
        if (i < ne) {
            const int u = ts.ul[i];
            if (i == ts.ustart[u]) {
#pragma unroll
                for (int t = 0; t < TT; ++t) carry[t] = (VT)0;
            }
            const int slot = i + u;
#pragma unroll
            for (int t = 0; t < TT; ++t) if (t < T) S[t * SLOTS + slot] = carry[t];
            const int l = lev(i);
            const VT v = val(i);
#pragma unroll
            for (int t = 0; t < TT; ++t) carry[t] += (t == l) ? v : (VT)0;
            if (i + 1 == ts.ustart[u + 1]) {
#pragma unroll
                for (int t = 0; t < TT; ++t) if (t < T) S[t * SLOTS + slot + 1] = carry[t];
            }
        }
    }
    __syncthreads();
}

// user starts + active flags of a tile.  Returns false (block-uniform) when no user of the tile takes part.
template <int TH>
__device__ __forceinline__ bool tile_users(TileShared<TH * TE> &ts, int first_user, int n_users, i64 e0,
                                           const i64 *__restrict__ row_ptr, const uint8_t *__restrict__ active) {
    const int tid = threadIdx.x;
    int any = 0;
    for (int u = tid; u <= n_users; u += TH) {
        const i64 rp = row_ptr[first_user + u];
        ts.ustart[u] = (int)(rp - e0);
        if (u < n_users) {
            const uint8_t a = active ? active[first_user + u] : (uint8_t)1;
            ts.uact[u] = a;
            if (a && row_ptr[first_user + u + 1] > rp) any = 1;
        }
    }
    return __syncthreads_or(any) != 0;
}

// ---------------------------------------------------------------- tile_prepare: sort + windows + counts
#ifndef PCR_PREP_MINB
#define PCR_PREP_MINB 4
#endif
template <int TT, int TH>
__global__ void __launch_bounds__(TH, TH == 256 ? PCR_PREP_MINB : (TH == 512 ? 2 : 1)) tile_prepare_kernel(const int32_t *__restrict__ tile_first,
                                                          const int32_t *__restrict__ tile_nusers,
                                                          const i64 *__restrict__ tile_e0, const int32_t *__restrict__ tile_ne,
                                                          const uint8_t *__restrict__ active,
                                                          const i64 *__restrict__ row_ptr, const int32_t *__restrict__ user_of,
                                                          const double *__restrict__ m, const uint8_t *__restrict__ level,
                                                          double *__restrict__ s_out, int32_t *__restrict__ pos_out,
                                                          uint8_t *__restrict__ lev_out, int32_t *__restrict__ ub_out,
                                                          int32_t *__restrict__ lb_out, int32_t *__restrict__ lo_out,
                                                          int32_t *__restrict__ hi_out, int T, SortedMeta lm) {
    constexpr int CAP = TH * TE, SLOTS = CAP + TILE_MAX_USERS;
    extern __shared__ __align__(16) unsigned char smraw[];
    __shared__ TileShared<CAP> ts;
    __shared__ int wagg[TH / 32 * TT];
    __shared__ int wflag[TH / 32];
    // dynamic layout: keys[CAP] f64 | pk[CAP] u64 | C[T][SLOTS] i32 | tag[CAP] u32 | lev[CAP] u8 | lev0[CAP] u8
    double *keys = reinterpret_cast<double *>(smraw);
    unsigned long long *pk = reinterpret_cast<unsigned long long *>(keys + CAP);
    int *C = reinterpret_cast<int *>(pk + CAP);
    uint32_t *tag = reinterpret_cast<uint32_t *>(C + T * SLOTS);
    uint8_t *slev = reinterpret_cast<uint8_t *>(tag + CAP);
    uint8_t *lev0 = slev + CAP;
    __shared__ int s_fallback;
    const int tid = threadIdx.x;
    const int first_user = tile_first[blockIdx.x], n_users = tile_nusers[blockIdx.x];
    const i64 e0 = tile_e0[blockIdx.x];
    const int ne = tile_ne[blockIdx.x];
    bool users_done = false;
    if (active) {                      // masked launch: find out first whether this tile has anything to do
        if (!tile_users<TH>(ts, first_user, n_users, e0, row_ptr, active)) return;
        users_done = true;
    }
    int np2 = 1;
    while (np2 < ne) np2 <<= 1;
    // all global reads of the tile are issued here, back to back
    double r_m[TE]; int r_u[TE]; uint8_t r_l[TE];
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        r_m[q] = CUDART_INF; r_u[q] = 0xFFFF; r_l[q] = 0;
        if (i < ne) { r_m[q] = m[e0 + i]; r_u[q] = user_of[e0 + i] - first_user; r_l[q] = level[e0 + i]; }
    }
    if (!users_done) tile_users<TH>(ts, first_user, n_users, e0, row_ptr, active);
    // ---- sort, fast path: ONE 64-bit integer per rating, [user:7 | order-preserving float32 image of the score:32 |
    // index:13], so a compare-exchange is a single 64-bit comparison; float32 rounding is monotone, hence the result can
    // differ from the exact (user, fp64 score, index) order only inside runs of equal float images, which the odd-even
    // fix-up below repairs with exact fp64 comparisons (zero or one sweep in practice).  keys[] keeps the fp64 scores in
    // input order for that purpose.  If the fix-up does not settle (pathological clusters) the exact network is used.
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        if (i < np2) {
            keys[i] = r_m[q];
            if (i < ne) {
                const float f = (float)r_m[q] + 0.0f;                       // -0.0f -> +0.0f
                const uint32_t b = __float_as_uint(f);
                const uint32_t fk = b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
                pk[i] = ((unsigned long long)r_u[q] << 45) | ((unsigned long long)fk << 13) | (unsigned long long)i;
                ts.ul[i] = (uint8_t)r_u[q]; lev0[i] = r_l[q];
            } else {
                pk[i] = ~0ull;
            }
        }
    }
    if (tid == 0) s_fallback = 0;
    __syncthreads();
    // Bitonic network with BLOCKED ownership (thread t holds positions 4t..4t+3 in registers): the j = 1, 2 stages are
    // register compare-exchanges, j = 4..64 are warp shuffles with lane ^ (j/4), and only j >= 128 (partner in another
    // warp) goes through shared memory -- 6 of the 55 stages of a 1024-key tile.  (ncu on the all-shared-memory version:
    // l1tex data-pipe wavefronts 87 % of peak, 137 M bank conflicts: the LDS/STS traffic of the network was the limit.)
    {
        const int p0 = tid * TE;
        const bool live = ((tid & ~31) * TE) < np2;            // warp-uniform: this warp owns positions below np2
        unsigned long long ek[TE];
#pragma unroll
        for (int q = 0; q < TE; ++q) ek[q] = pk[p0 + q];       // p0 + q < CAP always; entries >= np2 are never paired with < np2
        for (int k = 2; k <= np2; k <<= 1) {
            for (int j = k >> 1; j >= 32 * TE; j >>= 1) {      // partner thread lives in another warp
                __syncthreads();
#pragma unroll
                for (int q = 0; q < TE; ++q) pk[p0 + q] = ek[q];
                __syncthreads();
                const int m = j / TE;
                const int pp = (tid ^ m) * TE;
                const bool keep_min = (((tid & m) == 0) == ((p0 & k) == 0));
#pragma unroll
                for (int q = 0; q < TE; ++q) {
                    const unsigned long long o = pk[pp + q];
                    ek[q] = ((o < ek[q]) == keep_min) ? o : ek[q];      // one 64-bit compare (equal keys only among the padding)
                }
            }
            if (live) {
                const int jtop = (k >> 1) < 16 * TE ? (k >> 1) : 16 * TE;
                for (int j = jtop; j >= TE; j >>= 1) {          // partner lane = lane ^ (j / TE)
                    const int m = j / TE;
                    const bool keep_min = (((tid & m) == 0) == ((p0 & k) == 0));
#pragma unroll
                    for (int q = 0; q < TE; ++q) {
                        const unsigned long long o = __shfl_xor_sync(FULL, ek[q], m);
                        ek[q] = ((o < ek[q]) == keep_min) ? o : ek[q];      // one 64-bit compare (equal keys only among the padding)
                    }
                }
                if (k >= 4) {                                   // j = 2: pairs (0,2), (1,3); direction is per thread for k >= 4
                    const bool asc = ((p0 & k) == 0);
#pragma unroll
                    for (int q = 0; q < 2; ++q) {
                        const unsigned long long a = ek[q], b = ek[q + 2];
                        if ((a > b) == asc) { ek[q] = b; ek[q + 2] = a; }
                    }
                }
#pragma unroll
                for (int q = 0; q < TE; q += 2) {               // j = 1: pairs (0,1), (2,3)
                    const bool asc = (((p0 + q) & k) == 0);
                    const unsigned long long a = ek[q], b = ek[q + 1];
                    if ((a > b) == asc) { ek[q] = b; ek[q + 1] = a; }
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int q = 0; q < TE; ++q) pk[p0 + q] = ek[q];
        __syncthreads();
    }
    // exact fix-up inside runs of equal (user, float image): odd-even transposition with fp64 (score, index) order
    {
        int round = 0;
        for (;;) {
            int swapped = 0;
            for (int phase = 0; phase < 2; ++phase) {
                for (int i = 2 * tid + phase; i + 1 < ne; i += 2 * TH) {
                    const unsigned long long a = pk[i], b = pk[i + 1];
                    if ((a >> 13) == (b >> 13)) {
                        const int ia = (int)(a & 0x1FFFu), ib = (int)(b & 0x1FFFu);
                        const double ka = keys[ia], kb = keys[ib];
                        if (ka > kb || (ka == kb && ia > ib)) { pk[i] = b; pk[i + 1] = a; swapped = 1; }
                    }
                }
                __syncthreads();
            }
            if (!__syncthreads_or(swapped)) break;
            if (++round >= 48) { if (tid == 0) s_fallback = 1; break; }
        }
        __syncthreads();
    }
    const bool fallback = s_fallback != 0;
    // tag[] = (user, source index) of every sorted slot; keys[] <- fp64 scores in sorted order
    double srt[TE];
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        srt[q] = CUDART_INF;
        if (i < ne && !fallback) srt[q] = keys[(int)(pk[i] & 0x1FFFu)];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        if (i < np2) {
            if (!fallback) {
                if (i < ne) { keys[i] = srt[q]; tag[i] = ((uint32_t)ts.ul[i] << 16) | (uint32_t)(pk[i] & 0x1FFFu); }
            } else {
                keys[i] = r_m[q];
                tag[i] = i < ne ? (((uint32_t)r_u[q] << 16) | (uint32_t)i) : 0xFFFFFFFFu;
            }
        }
    }
    __syncthreads();
    if (fallback) {
        // exact bitonic network on the composite key (user, fp64 score, index)
        for (int k = 2; k <= np2; k <<= 1) {
            for (int j = k >> 1; j > 0; j >>= 1) {
                for (int t = tid; t < (np2 >> 1); t += TH) {
                    const int i = ((t & ~(j - 1)) << 1) | (t & (j - 1));
                    const int p = i | j;
                    const bool asc = (i & k) == 0;
                    const uint32_t ti = tag[i], tp = tag[p];
                    const double ki = keys[i], kp = keys[p];
                    const bool gt = ((ti >> 16) != (tp >> 16)) ? (ti > tp) : ((ki > kp) || (ki == kp && ti > tp));
                    if (gt == asc) { keys[i] = kp; keys[p] = ki; tag[i] = tp; tag[p] = ti; }
                }
                __syncthreads();
            }
        }
    }
    // sorted outputs: users stay in place (the user is the major key), scores ascending inside each user
    for (int i = tid; i < ne; i += TH) {
        const int src = (int)(tag[i] & 0xFFFFu);
        const uint8_t l = lev0[src];
        slev[i] = l;
        if (ts.uact[ts.ul[i]]) { s_out[e0 + i] = keys[i]; pos_out[e0 + i] = (int32_t)(e0 + src); lev_out[e0 + i] = l; }
    }
    __syncthreads();
    // per-level exclusive prefix COUNTS
    tile_level_scan<int, TT, TH>(ts, ne, T, C, wagg, wflag, [](int) { return 1; }, [&](int i) { return (int)slev[i]; });
    // window pointers by binary search inside the user's segment, then the aggregated counters
    for (int i = tid; i < ne; i += TH) {
        const int u = ts.ul[i];
        if (!ts.uact[u]) continue;
        const int u0 = ts.ustart[u], n = ts.ustart[u + 1] - u0, x = i - u0;
        const double *kk = keys + u0;
        const double sj = kk[x];
        const double hi = __dadd_rn(sj, 1.0), lo = __dadd_rn(sj, -1.0);
        int a = x + 1, b = n;
        while (a < b) { const int mid = (a + b) >> 1; if (kk[mid] <= hi) a = mid + 1; else b = mid; }
        const int ub = a;
        a = 0; b = x;
        while (a < b) { const int mid = (a + b) >> 1; if (kk[mid] < lo) a = mid + 1; else b = mid; }
        const int lb = a;
        const int base = u0 + u, l = slev[i];
        int chi = 0, clo = 0;
        for (int t = 0; t < T; ++t) {
            const int *Ct = C + t * SLOTS + base;
            if (t > l) chi += Ct[ub];
            else if (t < l) clo += Ct[n] - Ct[lb];
        }
        ub_out[e0 + i] = ub; lb_out[e0 + i] = lb; lo_out[e0 + i] = clo; hi_out[e0 + i] = chi;
        // level-major copy: rank of this rating in (level, score) order inside its user, and for every OTHER level t the
        // rank where its window ends: B_t + C_t(ub) above, B_t + C_t(lb) below  (B_t = first rank of level t)
        int run = 0, r = 0;
        uint16_t other[TT];
#pragma unroll
        for (int t = 0; t < TT; ++t) {
            other[t] = 0;
            if (t < T) {
                const int *Ct = C + t * SLOTS + base;
                if (t == l) r = run + Ct[x];
                else other[t] = (uint16_t)(run + (t > l ? Ct[ub] : Ct[lb]));
                run += Ct[n];
            }
        }
        const i64 gi = e0 + u0 + r;
        unsigned long long w1 = 0ull, w2 = 0ull;
#pragma unroll
        for (int t = 0; t < TT; ++t) {
            if (t < T && t != l) {
                const int slot = t < l ? t : t - 1;
                if (slot < 4) w1 |= (unsigned long long)other[t] << (13 * slot);
                else          w2 |= (unsigned long long)other[t] << (13 * (slot - 4));
            }
        }
        lm.lm_s[gi] = sj;
        lm.lm_w0[gi] = (unsigned long long)(tag[i] & 0xFFFFu) | ((unsigned long long)clo << 13) | ((unsigned long long)chi << 26) |
                       ((unsigned long long)l << 39) | ((unsigned long long)u << 42);
        lm.lm_w1[gi] = w1;
        if (TT > 5) lm.lm_w2[gi] = w2;
    }
    for (int w = tid; w < n_users * T; w += TH) {
        const int u = w / T, t = w - u * T;
        const int n = ts.ustart[u + 1] - ts.ustart[u];
        if (ts.uact[u]) lm.ulev[(i64)(first_user + u) * 8 + t] = (uint16_t)(n > 0 ? C[t * SLOTS + ts.ustart[u] + u + n] : 0);
    }
}

// ---------------------------------------------------------------- tile_lm_sweep: the sweeps on the level-major copy
// In (user, level, score) order the ratings of one level form a block, so every per-level prefix S_t(x) is a difference
// of ONE running prefix G over the user: S_t(x) = G[B_t + C_t(x)] - G[B_t].  A scalar segmented scan replaces the
// T-vector scan, and the look-up positions B_t + C_t(ub|lb) were stored by tile_prepare:
//   acc_j = sum_{t>l} (G[idx_t] - G[B_t]) + sum_{t<l} (G[B_{t+1}] - G[idx_t]) = K_u[l] + sum_{t>l} G[idx_t] - sum_{t<l} G[idx_t]
#ifndef PCR_LM_MINB
#define PCR_LM_MINB 5      // measured with the packed records: 4 -> 21.2, 5 -> 18.5, 6 -> 19.8 ms per iteration (Hv sweeps)
#endif
template <int MODE, int TT, int TH>
__global__ void __launch_bounds__(TH, TH == 256 ? PCR_LM_MINB : (TH == 512 ? 2 : 1)) tile_lm_sweep_kernel(const int32_t *__restrict__ tile_first,
                                                           const int32_t *__restrict__ tile_nusers,
                                                           const i64 *__restrict__ tile_e0, const int32_t *__restrict__ tile_ne,
                                                           const uint8_t *__restrict__ active,
                                                           const i64 *__restrict__ row_ptr, const int32_t *__restrict__ user_of,
                                                           SortedMeta lm, const double *__restrict__ b_g,
                                                           double *__restrict__ c_out, double *__restrict__ obj_user, int T) {
    constexpr int CAP = TH * TE, SLOTS = CAP + TILE_MAX_USERS;
    __shared__ TileShared<CAP> ts;
    __shared__ double wagg[TH / 32];
    __shared__ int wflag[TH / 32];
    extern __shared__ __align__(16) unsigned char smraw[];
    // dynamic layout: G[SLOTS] | sval[CAP] | G2[SLOTS] (objective) or stg[CAP] (coefficients: CSR-order staging of b / c)
    double *G = reinterpret_cast<double *>(smraw);
    double *sval = G + SLOTS;
    double *G2 = sval + CAP;
    double *stg = sval + CAP;
    __shared__ double Kt[TILE_MAX_USERS * TT], Kt2[MODE == 2 ? TILE_MAX_USERS * TT : 1];
    __shared__ uint16_t Bt[TILE_MAX_USERS * (TT + 1)];
    const int tid = threadIdx.x;
    const int first_user = tile_first[blockIdx.x], n_users = tile_nusers[blockIdx.x];
    const i64 e0 = tile_e0[blockIdx.x];
    const int ne = tile_ne[blockIdx.x];
    bool users_done = false;
    if (active) {
        if (!tile_users<TH>(ts, first_user, n_users, e0, row_ptr, active)) return;
        users_done = true;
    }
    // one packed record per rating (see SortedMeta): two (T <= 5) or three 8-byte loads instead of nine scalar ones
    unsigned long long r_w0[TE], r_w1[TE], r_w2[TT > 5 ? TE : 1];
    double r_v[TE];
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        r_w0[q] = 0ull; r_w1[q] = 0ull; r_v[q] = 0.0;
        if (TT > 5) r_w2[q] = 0ull;
        if (i < ne) {
            r_w0[q] = lm.lm_w0[e0 + i];
            r_w1[q] = lm.lm_w1[e0 + i];
            if (TT > 5) r_w2[q] = lm.lm_w2[e0 + i];
            if (MODE != 1) r_v[q] = lm.lm_s[e0 + i];
        }
    }
    if (MODE == 1) {
        // b arrives in CSR order: read the tile's slice COALESCED and independently of the records (no dependent global
        // gather), park it in shared memory and pick b[pos] from there
#pragma unroll
        for (int q = 0; q < TE; ++q) { const int i = tid + q * TH; if (i < ne) stg[i] = b_g[e0 + i]; }
    }
    if (!users_done) tile_users<TH>(ts, first_user, n_users, e0, row_ptr, active);
    // block starts of every user's levels (ranks inside the user)
    for (int u = tid; u < n_users; u += TH) {
        int run = 0;
        for (int t = 0; t < T; ++t) { Bt[u * (TT + 1) + t] = (uint16_t)run; run += lm.ulev[(i64)(first_user + u) * 8 + t]; }
        Bt[u * (TT + 1) + T] = (uint16_t)run;
    }
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        if (i < ne) { ts.ul[i] = (uint8_t)((r_w0[q] >> 42) & 0x7Full); if (MODE != 1) sval[i] = MODE == 2 ? r_v[q] - 1.0 : r_v[q]; }
    }
    __syncthreads();
    if (MODE == 1) {
#pragma unroll
        for (int q = 0; q < TE; ++q) {
            const int i = tid + q * TH;
            if (i < ne) { r_v[q] = stg[(int)(r_w0[q] & 0x1FFFull)]; sval[i] = r_v[q]; }
        }
        __syncthreads();
    }
    tile_level_scan<double, 1, TH>(ts, ne, 1, G, wagg, wflag, [&](int i) { return sval[i]; }, [](int) { return 0; });
    if (MODE == 2)
        tile_level_scan<double, 1, TH>(ts, ne, 1, G2, wagg, wflag, [&](int i) { const double d = sval[i]; return d * d; }, [](int) { return 0; });
    // per-user constants K_u[l]
    for (int w = tid; w < n_users * T; w += TH) {
        const int u = w / T, l = w - u * T;
        const int base = ts.ustart[u] + u;
        const uint16_t *B = Bt + u * (TT + 1);
        double k1 = 0.0, k2 = 0.0;
        for (int t = 0; t < T; ++t) {
            if (t > l) { k1 -= G[base + B[t]]; if (MODE == 2) k2 -= G2[base + B[t]]; }
            else if (t < l && MODE != 2) k1 += G[base + B[t + 1]];
        }
        Kt[u * TT + l] = k1;
        if (MODE == 2) Kt2[u * TT + l] = k2;
    }
    __syncthreads();
    double objj[TE];
#pragma unroll
    for (int q = 0; q < TE; ++q) {
        const int i = tid + q * TH;
        objj[q] = 0.0;
        if (i >= ne) continue;
        const unsigned long long w0 = r_w0[q];
        const int u = (int)((w0 >> 42) & 0x7Full);
        if (!ts.uact[u]) continue;
        const int base = ts.ustart[u] + u, l = (int)((w0 >> 39) & 7ull);
        double acc = Kt[u * TT + l], acc2 = MODE == 2 ? Kt2[u * TT + l] : 0.0;
#pragma unroll
        for (int t = 0; t < TT - 1; ++t) {
            if (t < T - 1) {
                const unsigned long long wi = (TT > 5 && t >= 4) ? r_w2[TT > 5 ? q : 0] >> (13 * (t - 4)) : r_w1[q] >> (13 * t);
                const int at = base + (int)(wi & 0x1FFFull);
                if (t >= l) { acc += G[at]; if (MODE == 2) acc2 += G2[at]; }      // other level t+1 > l
                else if (MODE != 2) acc -= G[at];                                    // other level t < l
            }
        }
        const double v = r_v[q];
        const double hi = (double)(int)((w0 >> 26) & 0x1FFFull);
        if (MODE == 2) {
            objj[q] = hi * (v * v) - 2.0 * v * acc + acc2;
        } else {
            const double lo = (double)(int)((w0 >> 13) & 0x1FFFull);
            const double cc = MODE == 0 ? lo * (v - 1.0) + hi * (v + 1.0) - acc : (lo + hi) * v - acc;
            // unmasked launch: every position of the tile gets a value, so c goes back through shared memory and leaves
            // as coalesced stores; masked launch (some users inactive): scattered stores of the active users only
            if (active == nullptr) stg[(int)(w0 & 0x1FFFull)] = 2.0 * cc;
            else c_out[e0 + (i64)(w0 & 0x1FFFull)] = 2.0 * cc;
        }
    }
    if (MODE != 2 && active == nullptr) {
        __syncthreads();
        for (int i = tid; i < ne; i += TH) c_out[e0 + i] = stg[i];
    }
    if (MODE == 2) {
        __syncthreads();
#pragma unroll
        for (int q = 0; q < TE; ++q) { const int i = tid + q * TH; if (i < ne) sval[i] = objj[q]; }
        __syncthreads();
        tile_level_scan<double, 1, TH>(ts, ne, 1, G, wagg, wflag, [&](int i) { return sval[i]; }, [](int) { return 0; });
        for (int u = tid; u < n_users; u += TH) {
            const int n = ts.ustart[u + 1] - ts.ustart[u];
            if (n > 0 && ts.uact[u]) obj_user[first_user + u] = G[ts.ustart[u] + u + n];
        }
    }
}

static size_t prepare_smem(int T, int cap) { return (size_t)cap * 16 + (size_t)T * (cap + TILE_MAX_USERS) * 4 + (size_t)cap * 4 + 2 * (size_t)cap; }

template <typename K>
static void set_smem(K kernel, size_t bytes) {
    PCR_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
}

// geo 0: small tiles (256 threads x 4 = TILE_CAP ratings), geo 1: medium (512 threads, TILE_CAP_M), geo 2: large (1024 threads, TILE_CAP_L)
void k_tile_prepare(Ctx &c, const DevCsr &X, int geo, const uint8_t *active, const double *m, SortedMeta &meta, int T) {
    const TileList &L = X.tiles[geo];
    if (L.n <= 0) return;
    PCR_REQUIRE(T <= 8, "tile kernels support at most 8 rating levels");
    // in: score 8 + user 4 + level 1; out: sorted score 8, position 4, level 1, ub/lb/cnt_lo/cnt_hi 16, level-major score 8 + records 16
    const double bytes = (double)L.nnz * (13 + 29 + 24);
#define PREP_ARGS L.first, L.nusers, L.e0, L.ne, active, X.row_ptr, X.user, m, X.level, meta.s, meta.pos, meta.lev, meta.ub, meta.lb, meta.cnt_lo, meta.cnt_hi, T, meta
#define PREP_LAUNCH(TT, TH, NAME) { const size_t sm = prepare_smem(T, TH * TE); set_smem(tile_prepare_kernel<TT, TH>, sm); \
        LAUNCH(c, NAME, bytes, (tile_prepare_kernel<TT, TH>), (unsigned)L.n, TH, sm, PREP_ARGS); }
    if (geo == 0)      { if (T <= 5) PREP_LAUNCH(5, 256, "tile_prepare") else PREP_LAUNCH(8, 256, "tile_prepare") }
    else if (geo == 1) { PCR_REQUIRE(T <= 5, "medium tiles need T <= 5"); PREP_LAUNCH(5, 512, "tile_prepare_M") }
    else               { PCR_REQUIRE(T <= 5, "large tiles need T <= 5"); PREP_LAUNCH(5, 1024, "tile_prepare_L") }
#undef PREP_LAUNCH
#undef PREP_ARGS
}

void k_tile_sweep(Ctx &c, int mode, const DevCsr &X, int geo, const uint8_t *active, const SortedMeta &meta, const double *b,
                  double *c_out, double *obj_user, int T) {
    const TileList &L = X.tiles[geo];
    if (L.n <= 0) return;
    PCR_REQUIRE(T <= 8, "tile kernels support at most 8 rating levels");
    // packed records 16 B + stream (score or b) 8 B + coefficient out 8 B (not for the objective)
    const double per = mode == 2 ? (16 + 8) : (16 + 8 + 8);
    const double bytes = (double)L.nnz * per;
    const unsigned grid = (unsigned)L.n;
#define LM_ARGS L.first, L.nusers, L.e0, L.ne, active, X.row_ptr, X.user, meta, b, c_out, obj_user, T
#define LM_LAUNCH(MODE, TT, TH, NAME) { const size_t sm = ((size_t)(TH * TE + TILE_MAX_USERS) * (MODE == 2 ? 2 : 1) + TH * TE * (MODE == 2 ? 1 : 2)) * 8; \
    set_smem(tile_lm_sweep_kernel<MODE, TT, TH>, sm); LAUNCH(c, NAME, bytes, (tile_lm_sweep_kernel<MODE, TT, TH>), grid, TH, sm, LM_ARGS); }
#define LM_MODE(MODE, NAME)                                                                                         \
    if (geo == 0)      { if (T <= 5) { LM_LAUNCH(MODE, 5, 256, NAME) } else { LM_LAUNCH(MODE, 8, 256, NAME) } }   \
    else if (geo == 1) { LM_LAUNCH(MODE, 5, 512, NAME "_M") }                                                    \
    else               { LM_LAUNCH(MODE, 5, 1024, NAME "_L") }
    if (mode == 0) { LM_MODE(0, "lm_sweep_grad") }
    else if (mode == 1) { LM_MODE(1, "lm_sweep_hv") }
    else { LM_MODE(2, "lm_sweep_obj") }
#undef LM_MODE
#undef LM_LAUNCH
#undef LM_ARGS
}

}  // namespace pcr
