// k_topn.cu -- top-N recommendation: every requested user scored against every item (fp64 DFMA register tiles) with the
// per-user selection fused in, so the d1 x d2 score matrix is never written anywhere.
//
// A CTA owns BU users and streams V through shared memory in tiles of BI consecutive items, ascending.  Each tile is
// computed as a small GEMM, k sliced in chunks of KC double-buffered with cp.async, 8 users x 8 items per thread.
// Scores stay in registers while they are filtered against each user's threshold (the current N-th best entry); the
// survivors go to a per-user candidate buffer in shared memory, and a buffer that fills (or the end of the item
// stream) merges the candidates into the user's sorted top-N and raises the threshold.  Excluded items (the user's
// ascending exclusion row) are masked per tile with a cursor per user, so the cost is O(nnz of the block + tiles).
//
// Order: (score descending, item ascending) on a 64-bit key of the score that equates +0.0 / -0.0 and ranks every NaN
// below -inf (NaNs tie, so the item decides).  Every score is the fma chain acc = fma(U[u][j], V[i][j], acc), j = 0..k-1,
// from +0.0 -- the same for every class and batch -- and the top-N under a total order is unique, so a user's row does not
// depend on the batch it is computed in.
//
// Similar rows (similar_kernel: topn_kernel with SELF, and COS for cosine) rank the rows of one matrix M against query rows
// of the same M: U = V = M.  SELF adds each query's own row to its tile exclusion mask; COS divides every register score
// by (|M[q]| * |M[i]|), norms from row_norms staged in shared memory, before it meets the filter, so the buffers and the
// merge only ever see final scores.
#include "kernels.h"

namespace pcr {

#ifndef FULL
#define FULL 0xffffffffu
#endif

typedef unsigned long long u64;

// 1 for NaN, order-preserving above it; 0 is below every key (the "no threshold yet" value)
__device__ __forceinline__ u64 score_key(double s) {
    if (s != s) return 1ull;
    if (s == 0.0) s = 0.0;                       // -0.0 -> +0.0: the two compare equal
    const u64 b = (u64)__double_as_longlong(s);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_score(u64 key) {
    if (key == 1ull) return __longlong_as_double(0x7ff8000000000000ll);
    return __longlong_as_double((long long)((key >> 63) ? (key & 0x7fffffffffffffffull) : ~key));
}
// a ranks before b
__device__ __forceinline__ bool better(u64 ka, int ia, u64 kb, int ib) { return ka > kb || (ka == kb && ia < ib); }

__device__ __forceinline__ void cp_async8(void *smem, const void *gmem, bool valid) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(s), "l"(gmem), "r"(valid ? 8 : 0));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N)); }

// The scoring tile shared by topn_kernel and rank_kernel.  UG: groups of 8 rows (BU = 8 UG rows, BI = 2048 / UG items per
// tile).  256 threads: thread (ug, ig) computes rows ug*8..+7 x items ig + IG*c, c = 0..7.
template <int UG>
struct TileCfg {
    static constexpr int THREADS = 256, WARPS = THREADS / 32;
    static constexpr int IG = THREADS / UG, BU = 8 * UG, BI = 8 * IG, KC = UG;   // KC * BI = 2048 doubles per V chunk
    static constexpr int PAD = 32 / KC;          // row padding: the transposing cp.async stores of a warp hit distinct banks
    static constexpr int VS = KC * (BI + PAD), US = KC * (BU + PAD), MW = BI / 32;
    static_assert(KC * BI == 2048 && BU * KC <= 2 * THREADS && IG >= 32, "tile shape");
};

// chunk kc of item tile t into buffer buf: V rows of the tile and U rows uid[0..nrows-1], k slice kc*KC..+KC-1
template <int UG>
__device__ __forceinline__ void tile_load(double *Vs, double *Us, const double *__restrict__ U, const double *__restrict__ V,
                                          i64 d2, int k, const int *uid, int nrows, int t, int kc, int buf) {
    typedef TileCfg<UG> C;
    constexpr int BU = C::BU, BI = C::BI, KC = C::KC, PAD = C::PAD;
    const int tid = threadIdx.x;
    const int k0 = kc * KC;
    const i64 base = (i64)t * BI;
    double *vs = Vs + buf * C::VS;
#pragma unroll
    for (int j = 0; j < 2048 / C::THREADS; ++j) {
        const int e = tid + j * C::THREADS, il = e / KC, kk = e % KC;
        const i64 item = base + il;
        const bool ok = item < d2 && k0 + kk < k;
        cp_async8(vs + kk * (BI + PAD) + il, ok ? V + item * k + k0 + kk : V, ok);
    }
    double *us = Us + buf * C::US;
    for (int e = tid; e < BU * KC; e += C::THREADS) {
        const int r = e / KC, kk = e % KC;
        const bool ok = r < nrows && k0 + kk < k;
        cp_async8(us + kk * (BU + PAD) + r, ok ? U + (i64)uid[r] * k + k0 + kk : U, ok);
    }
    cp_async_commit();
}

// Scores of item tile t into acc: acc[r][c] = U[uid[ug*8+r]] . V[t*BI + ig + IG*c], the fma chain over k from +0.0.  With
// `masked`, first the tile's rows x items exclusion bitmask, from each row's cursor cur[r] into its ascending exclusion row
// (ending at cend[r]); the cursors advance past the tile.  SELF (which needs `masked`): item uid[r] is masked in row r too.
// Chunk 0 of tile t must have been loaded into buffer buf; the first chunk of tile t+1 is prefetched.  Ends synchronised,
// with buf the buffer of that prefetch.
template <int UG, bool SELF = false>
__device__ __forceinline__ void score_tile(double (&acc)[8][8], double *Vs, double *Us, unsigned *mask, i64 *cur,
                                           const i64 *cend, const double *__restrict__ U, const double *__restrict__ V,
                                           i64 d2, int k, bool masked, const int32_t *__restrict__ ex_item, const int *uid,
                                           int nrows, int t, int ntiles, int nkc, int &buf) {
    typedef TileCfg<UG> C;
    constexpr int BU = C::BU, BI = C::BI, KC = C::KC, IG = C::IG, PAD = C::PAD, MW = C::MW;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ug = tid / IG, ig = tid % IG;
    const i64 base = (i64)t * BI;
    {
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) acc[r][c] = 0.0;
        if (masked) {                                   // exclusion bitmask of this tile
            for (int e = tid; e < BU * MW; e += C::THREADS) mask[e] = 0u;
            __syncthreads();
            const i64 lim = base + BI;
            for (int r = warp; r < nrows; r += C::WARPS) {
                i64 p = cur[r];
                const i64 pe = cend[r];
                while (true) {
                    const i64 q = p + lane;
                    const i64 it = q < pe ? (i64)ex_item[q] : lim;
                    const bool in = it < lim;
                    if (in) atomicOr(&mask[r * MW + (int)((it - base) >> 5)], 1u << ((it - base) & 31));
                    const int n = __popc(__ballot_sync(FULL, in));
                    p += n;
                    if (n < 32) break;
                }
                if (lane == 0) {
                    cur[r] = p;
                    if (SELF && uid[r] >= base && uid[r] < lim)
                        atomicOr(&mask[r * MW + (int)((uid[r] - base) >> 5)], 1u << ((uid[r] - base) & 31));
                }
            }
        }
    }
    for (int kc = 0; kc < nkc; ++kc, buf ^= 1) {
        // prefetch the next chunk (of this tile, or the first of the next) while this one is computed
        if (kc + 1 < nkc) { tile_load<UG>(Vs, Us, U, V, d2, k, uid, nrows, t, kc + 1, buf ^ 1); cp_async_wait<1>(); }
        else if (t + 1 < ntiles) { tile_load<UG>(Vs, Us, U, V, d2, k, uid, nrows, t + 1, 0, buf ^ 1); cp_async_wait<1>(); }
        else cp_async_wait<0>();
        __syncthreads();
        const double *vs = Vs + buf * C::VS + ig;
        const double *us = Us + buf * C::US + ug * 8;
#pragma unroll
        for (int kk = 0; kk < KC; ++kk) {
            double a[8], b[8];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const double2 v2 = *reinterpret_cast<const double2 *>(us + kk * (BU + PAD) + 2 * q);
                a[2 * q] = v2.x; a[2 * q + 1] = v2.y;
            }
#pragma unroll
            for (int c = 0; c < 8; ++c) b[c] = vs[kk * (BI + PAD) + IG * c];
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = fma(a[r], b[c], acc[r][c]);
        }
        __syncthreads();
    }
}

// NMAX: largest topn of the class; UG: the tile (BU = 8 UG users); CAP: candidates buffered per user between merges.
// COS: room for the norms of the BU query rows and of the BI rows of the current tile.
template <int NMAX, int UG, int CAP, bool COS = false>
struct TopnCfg : TileCfg<UG> {
    typedef TileCfg<UG> T;
    static constexpr int SCR = NMAX > CAP ? NMAX : CAP;
    static constexpr int BU = T::BU, WARPS = T::WARPS, MW = T::MW;
    // 8-byte arrays first, then 4-byte ones
    static constexpr size_t o_vs = 0, o_us = o_vs + 2 * T::VS, o_lkey = o_us + 2 * T::US, o_ckey = o_lkey + BU * NMAX,
                            o_skey = o_ckey + BU * CAP, o_thr = o_skey + WARPS * SCR, o_cur = o_thr + BU, o_end = o_cur + BU,
                            o_qn = o_end + BU, o_tn = o_qn + (COS ? BU : 0), n8 = o_tn + (COS ? T::BI : 0);
    static constexpr size_t o_litem = 0, o_citem = o_litem + BU * NMAX, o_sitem = o_citem + BU * CAP,
                            o_thri = o_sitem + WARPS * SCR, o_lcnt = o_thri + BU, o_ccnt = o_lcnt + BU, o_uid = o_ccnt + BU,
                            o_mask = o_uid + BU, n4 = o_mask + BU * MW;
    static constexpr size_t smem = n8 * 8 + n4 * 4;
    static_assert(smem <= 227 * 1024, "shared memory of one CTA");
};

// SELF: a row's own id (users[q], an index into V) is never its candidate.  COS: scores are divided by
// (norms[users[q]] * norms[item]); norms is unused otherwise.
template <int NMAX, int UG, int CAP, bool SELF = false, bool COS = false>
__global__ void __launch_bounds__(256, 1)
topn_kernel(const double *__restrict__ U, const double *__restrict__ V, i64 d2, int k, const i64 *__restrict__ ex_ptr,
            const int32_t *__restrict__ ex_item, const int32_t *__restrict__ users, i64 n_users, int topn,
            int32_t *__restrict__ items_out, double *__restrict__ scores_out, const double *__restrict__ norms) {
    typedef TopnCfg<NMAX, UG, CAP, COS> C;
    constexpr int BU = C::BU, BI = C::BI, KC = C::KC, IG = C::IG, MW = C::MW, SCR = C::SCR;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *Vs = reinterpret_cast<double *>(smem_raw) + C::o_vs;
    double *Us = reinterpret_cast<double *>(smem_raw) + C::o_us;
    u64 *lkey = reinterpret_cast<u64 *>(smem_raw) + C::o_lkey;
    u64 *ckey = reinterpret_cast<u64 *>(smem_raw) + C::o_ckey;
    u64 *skey_all = reinterpret_cast<u64 *>(smem_raw) + C::o_skey;
    u64 *thr_key = reinterpret_cast<u64 *>(smem_raw) + C::o_thr;
    i64 *cur = reinterpret_cast<i64 *>(smem_raw) + C::o_cur;
    i64 *cend = reinterpret_cast<i64 *>(smem_raw) + C::o_end;
    double *qnorm = reinterpret_cast<double *>(smem_raw) + C::o_qn;     // COS only
    double *tnorm = reinterpret_cast<double *>(smem_raw) + C::o_tn;
    int *i4 = reinterpret_cast<int *>(smem_raw + C::n8 * 8);
    int *litem = i4 + C::o_litem, *citem = i4 + C::o_citem, *sitem_all = i4 + C::o_sitem, *thr_item = i4 + C::o_thri;
    int *lcnt = i4 + C::o_lcnt, *ccnt = i4 + C::o_ccnt, *uid = i4 + C::o_uid;
    unsigned *mask = reinterpret_cast<unsigned *>(i4 + C::o_mask);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ug = tid / IG, ig = tid % IG;
    const i64 row0 = (i64)blockIdx.x * BU;
    const int nrows = (int)(n_users - row0 < BU ? n_users - row0 : BU);
    u64 *skey = skey_all + warp * SCR;
    int *sitem = sitem_all + warp * SCR;

    for (int r = tid; r < BU; r += C::THREADS) {
        const int u = r < nrows ? users[row0 + r] : 0;
        uid[r] = u; lcnt[r] = 0; ccnt[r] = 0; thr_key[r] = 0ull; thr_item[r] = 0;
        cur[r] = (ex_ptr && r < nrows) ? ex_ptr[u] : 0;
        cend[r] = (ex_ptr && r < nrows) ? ex_ptr[u + 1] : 0;
        if (COS) qnorm[r] = r < nrows ? norms[u] : 1.0;
    }
    __syncthreads();

    const int nkc = (k + KC - 1) / KC;
    const int ntiles = (int)((d2 + BI - 1) / BI);
    const bool masked = SELF || ex_ptr != nullptr;

    // merge every user's candidates into its sorted top-N (warp per user); caller synchronises before and after
    auto merge_all = [&]() {
        for (int r = warp; r < BU; r += C::WARPS) {
            const int m = min(ccnt[r], CAP);
            if (m == 0) continue;
            const u64 *ck = ckey + r * CAP; const int *ci = citem + r * CAP;
            u64 *lk = lkey + r * NMAX; int *li = litem + r * NMAX;
            const int nl = lcnt[r];
            for (int i = lane; i < m; i += 32) {          // candidates sorted by rank counting into the scratch
                const u64 ka = ck[i]; const int ia = ci[i];
                int rank = 0;
                for (int j = 0; j < m; ++j) rank += better(ck[j], ci[j], ka, ia);
                skey[rank] = ka; sitem[rank] = ia;
            }
            __syncwarp();
            for (int i = lane; i < m; i += 32) { ckey[r * CAP + i] = skey[i]; citem[r * CAP + i] = sitem[i]; }
            __syncwarp();
            // merge path: an element's place = its index + the number of entries of the other list that rank before it
            for (int i = lane; i < nl; i += 32) {
                const u64 ka = lk[i]; const int ia = li[i];
                int lo = 0, hi = m;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (better(ck[mid], ci[mid], ka, ia)) lo = mid + 1; else hi = mid; }
                if (i + lo < topn) { skey[i + lo] = ka; sitem[i + lo] = ia; }
            }
            for (int j = lane; j < m; j += 32) {
                const u64 ka = ck[j]; const int ia = ci[j];
                int lo = 0, hi = nl;
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (better(lk[mid], li[mid], ka, ia)) lo = mid + 1; else hi = mid; }
                if (j + lo < topn) { skey[j + lo] = ka; sitem[j + lo] = ia; }
            }
            __syncwarp();
            const int nn = min(nl + m, topn);
            for (int i = lane; i < nn; i += 32) { lk[i] = skey[i]; li[i] = sitem[i]; }
            if (lane == 0) {
                lcnt[r] = nn; ccnt[r] = 0;
                if (nn == topn) { thr_key[r] = skey[nn - 1]; thr_item[r] = sitem[nn - 1]; }
            }
            __syncwarp();
        }
    };

    double acc[8][8];
    int buf = 0;
    if (ntiles > 0) tile_load<UG>(Vs, Us, U, V, d2, k, uid, nrows, 0, 0, 0);
    for (int t = 0; t < ntiles; ++t) {
        const i64 base = (i64)t * BI;
        // the tile's norms, read after score_tile's barriers; the previous tile's reads all precede a barrier of its selection
        if (COS)
            for (int i = tid; i < BI; i += C::THREADS) tnorm[i] = base + i < d2 ? norms[base + i] : 1.0;
        score_tile<UG, SELF>(acc, Vs, Us, mask, cur, cend, U, V, d2, k, masked, ex_item, uid, nrows, t, ntiles, nkc, buf);
        if (COS) {
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const double qn = qnorm[ug * 8 + r];
#pragma unroll
                for (int c = 0; c < 8; ++c) acc[r][c] = acc[r][c] / (qn * tnorm[ig + IG * c]);
            }
        }

        // ---- selection of this tile's scores
        u64 pend = ~0ull;
        auto filter = [&]() {        // keeps the pending scores that are eligible and beat their user's threshold
            u64 keep = 0ull;
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const int row = ug * 8 + r;
                if (row >= nrows) continue;
                const u64 tk = thr_key[row]; const int ti = thr_item[row];
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const int il = ig + IG * c;
                    const u64 bit = 1ull << (r * 8 + c);
                    if (!(pend & bit) || base + il >= d2) continue;
                    if (masked && ((mask[row * MW + (il >> 5)] >> (il & 31)) & 1u)) continue;
                    if (better(score_key(acc[r][c]), (int)(base + il), tk, ti)) keep |= bit;
                }
            }
            pend = keep;
        };
        filter();
        while (true) {
#pragma unroll
            for (int r = 0; r < 8; ++r)
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    const u64 bit = 1ull << (r * 8 + c);
                    if (pend & bit) {
                        const int row = ug * 8 + r;
                        const int pos = atomicAdd(&ccnt[row], 1);
                        if (pos < CAP) {
                            ckey[row * CAP + pos] = score_key(acc[r][c]);
                            citem[row * CAP + pos] = (int)(base + ig + IG * c);
                            pend &= ~bit;
                        }
                    }
                }
            if (!__syncthreads_or(pend != 0ull)) break;
            merge_all();             // some buffer is full: merge, raise the thresholds, retry what did not fit
            __syncthreads();
            filter();
        }
    }
    __syncthreads();
    merge_all();
    __syncthreads();
    for (int r = warp; r < nrows; r += C::WARPS) {
        const i64 o = (row0 + r) * topn;
        const int n = lcnt[r];
        for (int j = lane; j < topn; j += 32) {
            const bool have = j < n;
            items_out[o + j] = have ? litem[r * NMAX + j] : -1;
            if (scores_out) scores_out[o + j] = have ? key_score(lkey[r * NMAX + j]) : key_score(1ull);
        }
    }
}

template <int NMAX, int UG, int CAP, bool SELF, bool COS>
static void launch_topn(Ctx &c, const char *name, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr,
                        const int32_t *ex_item, const int32_t *users, i64 n_users, int topn, int32_t *items_out,
                        double *scores_out, const double *norms) {
    typedef TopnCfg<NMAX, UG, CAP, COS> C;
    auto kern = topn_kernel<NMAX, UG, CAP, SELF, COS>;
    PCR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem));
    const i64 grid = (n_users + C::BU - 1) / C::BU;
    const double bytes = (double)grid * d2 * k * 8.0 + (double)n_users * (k * 8.0 + topn * 12.0);
    c.prof->begin(name, c.stream, bytes);
    kern<<<(unsigned)grid, C::THREADS, C::smem, c.stream>>>(U, V, d2, k, ex_ptr, ex_item, users, n_users, topn, items_out,
                                                             scores_out, norms);
    c.prof->end(c.stream);
    PCR_CUDA(cudaGetLastError());
}

// the class of topn: names[0] for topn <= 32, names[1] for <= 128, names[2] for <= 256
template <bool SELF, bool COS>
static void dispatch_topn(Ctx &c, const char *const (&names)[3], const double *U, const double *V, i64 d2, int k,
                          const i64 *ex_ptr, const int32_t *ex_item, const int32_t *users, i64 n_users, int topn,
                          int32_t *items_out, double *scores_out, const double *norms) {
    PCR_REQUIRE(topn >= 1 && topn <= 256 && k >= 1 && k <= 256, "topn / k out of range [1, 256]");
    if (n_users <= 0) return;
    if (topn <= 32)
        launch_topn<32, 8, 64, SELF, COS>(c, names[0], U, V, d2, k, ex_ptr, ex_item, users, n_users, topn, items_out, scores_out, norms);
    else if (topn <= 128)
        launch_topn<128, 8, 64, SELF, COS>(c, names[1], U, V, d2, k, ex_ptr, ex_item, users, n_users, topn, items_out, scores_out, norms);
    else
        launch_topn<256, 4, 128, SELF, COS>(c, names[2], U, V, d2, k, ex_ptr, ex_item, users, n_users, topn, items_out, scores_out, norms);
}

void k_topn(Ctx &c, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr, const int32_t *ex_item,
            const int32_t *users, i64 n_users, int topn, int32_t *items_out, double *scores_out) {
    static const char *const names[3] = {"pcr::topn_kernel<32,8,64>", "pcr::topn_kernel<128,8,64>", "pcr::topn_kernel<256,4,128>"};
    dispatch_topn<false, false>(c, names, U, V, d2, k, ex_ptr, ex_item, users, n_users, topn, items_out, scores_out, nullptr);
}

// |M[i]| = sqrt of the fma chain acc = fma(M[i][j], M[i][j], acc), j = 0..k-1, from +0.0
__global__ void row_norms_kernel(const double *__restrict__ M, i64 n, int k, double *__restrict__ out) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const double *m = M + i * k;
        double acc = 0.0;
        for (int j = 0; j < k; ++j) acc = fma(m[j], m[j], acc);
        out[i] = sqrt(acc);
    }
}

void k_similar(Ctx &c, const double *M, i64 n, int k, bool cosine, double *norms, const i64 *ex_ptr,
               const int32_t *ex_item, const int32_t *queries, i64 n_queries, int topn, int32_t *ids_out,
               double *scores_out) {
    PCR_REQUIRE(topn >= 1 && topn <= 256 && k >= 1 && k <= 256, "topn / k out of range [1, 256]");
    if (n_queries <= 0) return;
    if (cosine) {
        i64 blocks = (n + 255) / 256;
        if (blocks > (i64)c.sms * 16) blocks = (i64)c.sms * 16;
        c.prof->begin("pcr::row_norms", c.stream, (double)n * (k + 1) * 8.0);
        row_norms_kernel<<<(unsigned)(blocks > 0 ? blocks : 1), 256, 0, c.stream>>>(M, n, k, norms);
        c.prof->end(c.stream);
        PCR_CUDA(cudaGetLastError());
        static const char *const names[3] = {"pcr::similar_kernel<32,8,64,cos>", "pcr::similar_kernel<128,8,64,cos>",
                                              "pcr::similar_kernel<256,4,128,cos>"};
        dispatch_topn<true, true>(c, names, M, M, n, k, ex_ptr, ex_item, queries, n_queries, topn, ids_out, scores_out, norms);
    } else {
        static const char *const names[3] = {"pcr::similar_kernel<32,8,64,dot>", "pcr::similar_kernel<128,8,64,dot>",
                                              "pcr::similar_kernel<256,4,128,dot>"};
        dispatch_topn<true, false>(c, names, M, M, n, k, ex_ptr, ex_item, queries, n_queries, topn, ids_out, scores_out, nullptr);
    }
}

// ---- held-out ranks: the exact catalog rank of every held-out entry, under the same scores and order as topn_kernel
// A CTA owns BU units; a unit is one user and a run of at most H consecutive entries of its held-out row (rows longer
// than H become several units, each of which streams the whole catalog).  The prologue scores the unit's entries, drops
// the ones in the exclusion row (rank 0) and rank-sorts the rest best first.  Per tile, an eligible candidate that beats
// the unit's worst entry is binary-searched for the first sorted entry p it beats and counted in hist[p]; the rank of
// sorted entry q is then 1 + sum_{p <= q} hist[p].  An entry never beats itself (the order is strict and both scores are
// the same fma chain), so a held-out item is one of the candidates of its user's other entries and not of its own.
template <int UG, int H>
struct RankCfg : TileCfg<UG> {
    typedef TileCfg<UG> T;
    static constexpr int BU = T::BU, MW = T::MW;
    static constexpr size_t o_vs = 0, o_us = o_vs + 2 * T::VS, o_hkey = o_us + 2 * T::US, o_wkey = o_hkey + BU * H,
                            o_cur = o_wkey + BU, o_end = o_cur + BU, n8 = o_end + BU;
    static constexpr size_t o_hitem = 0, o_hoff = o_hitem + BU * H, o_hist = o_hoff + BU * H, o_witem = o_hist + BU * H,
                            o_nv = o_witem + BU, o_uid = o_nv + BU, o_mask = o_uid + BU, n4 = o_mask + BU * MW;
    static constexpr size_t smem = n8 * 8 + n4 * 4;
    static_assert(2 * T::VS >= BU * H, "the prologue's unsorted keys live in the V buffers");
    static_assert(H % 32 == 0, "H is a multiple of the warp");
};

template <int UG, int H>
__global__ void __launch_bounds__(256, 1)
rank_kernel(const double *__restrict__ U, const double *__restrict__ V, i64 d2, int k, const i64 *__restrict__ ex_ptr,
            const int32_t *__restrict__ ex_item, const int32_t *__restrict__ ho_item,
            const int32_t *__restrict__ unit_user, const i64 *__restrict__ unit_beg, i64 n_units,
            int32_t *__restrict__ rank_out, double *__restrict__ score_out) {
    typedef RankCfg<UG, H> C;
    constexpr int BU = C::BU, BI = C::BI, KC = C::KC, IG = C::IG, MW = C::MW;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *Vs = reinterpret_cast<double *>(smem_raw) + C::o_vs;
    double *Us = reinterpret_cast<double *>(smem_raw) + C::o_us;
    u64 *hkey = reinterpret_cast<u64 *>(smem_raw) + C::o_hkey;     // sorted entries of row r: [r*H, r*H + nv[r])
    u64 *wkey = reinterpret_cast<u64 *>(smem_raw) + C::o_wkey;     // the worst sorted entry of each row
    i64 *cur = reinterpret_cast<i64 *>(smem_raw) + C::o_cur;
    i64 *cend = reinterpret_cast<i64 *>(smem_raw) + C::o_end;
    int *i4 = reinterpret_cast<int *>(smem_raw + C::n8 * 8);
    int *hitem = i4 + C::o_hitem, *hoff = i4 + C::o_hoff, *hist = i4 + C::o_hist, *witem = i4 + C::o_witem;
    int *nv = i4 + C::o_nv, *uid = i4 + C::o_uid;
    unsigned *mask = reinterpret_cast<unsigned *>(i4 + C::o_mask);
    u64 *tkey = reinterpret_cast<u64 *>(Vs);       // prologue scratch: unsorted keys (V buffers) and items (hist)
    int *titem = hist;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int ug = tid / IG, ig = tid % IG;
    const i64 row0 = (i64)blockIdx.x * BU;
    const int nrows = (int)(n_units - row0 < BU ? n_units - row0 : BU);

    for (int r = tid; r < BU; r += C::THREADS) {
        const int u = r < nrows ? unit_user[row0 + r] : 0;
        uid[r] = u; nv[r] = 0;
        cur[r] = (ex_ptr && r < nrows) ? ex_ptr[u] : 0;
        cend[r] = (ex_ptr && r < nrows) ? ex_ptr[u + 1] : 0;
    }
    __syncthreads();

    // ---- prologue: score the entries (the tile's fma chain), look them up in the exclusion row, sort best first
    for (int e = tid; e < BU * H; e += C::THREADS) {
        const int r = e / H, j = e % H;
        titem[e] = -1;
        if (r >= nrows) continue;
        const i64 g = unit_beg[row0 + r] + j;
        if (g >= unit_beg[row0 + r + 1]) continue;
        const int item = ho_item[g];
        const double *ur = U + (i64)uid[r] * k, *vr = V + (i64)item * k;
        double acc = 0.0;
        for (int jj = 0; jj < k; ++jj) acc = fma(ur[jj], vr[jj], acc);
        const u64 key = score_key(acc);
        if (score_out) score_out[g] = key_score(key);       // as topn_kernel returns it: -0.0 as +0.0, one NaN
        i64 lo = cur[r], hi = cend[r];
        while (lo < hi) { const i64 mid = (lo + hi) >> 1; if (ex_item[mid] < item) lo = mid + 1; else hi = mid; }
        if (lo < cend[r] && ex_item[lo] == item) { rank_out[g] = 0; continue; }
        tkey[e] = key; titem[e] = item;
        atomicAdd(&nv[r], 1);
    }
    __syncthreads();
    for (int e = tid; e < BU * H; e += C::THREADS) {
        const int r = e / H, j = e % H;
        const u64 ka = tkey[e]; const int ia = titem[e];
        if (ia < 0) continue;
        int pos = 0;                  // entries before it: better ones, and equal ones (a repeated item) at smaller j
        for (int q = 0; q < H; ++q) {
            const int iq = titem[r * H + q];
            if (iq < 0) continue;
            const u64 kq = tkey[r * H + q];
            pos += better(kq, iq, ka, ia) || (kq == ka && iq == ia && q < j);
        }
        hkey[r * H + pos] = ka; hitem[r * H + pos] = ia; hoff[r * H + pos] = j;
    }
    __syncthreads();
    for (int e = tid; e < BU * H; e += C::THREADS) hist[e] = 0;
    for (int r = tid; r < BU; r += C::THREADS) {
        const int n = nv[r];
        wkey[r] = n ? hkey[r * H + n - 1] : ~0ull;          // ~0 / -1: nothing beats it
        witem[r] = n ? hitem[r * H + n - 1] : -1;
    }
    __syncthreads();

    // ---- main loop: every eligible candidate of every tile against the unit's sorted entries
    const int nkc = (k + KC - 1) / KC;
    const int ntiles = (int)((d2 + BI - 1) / BI);
    double acc[8][8];
    int buf = 0;
    if (ntiles > 0) tile_load<UG>(Vs, Us, U, V, d2, k, uid, nrows, 0, 0, 0);
    for (int t = 0; t < ntiles; ++t) {
        const i64 base = (i64)t * BI;
        score_tile<UG>(acc, Vs, Us, mask, cur, cend, U, V, d2, k, ex_ptr != nullptr, ex_item, uid, nrows, t, ntiles, nkc, buf);
#pragma unroll
        for (int r = 0; r < 8; ++r) {
            const int row = ug * 8 + r;
            if (row >= nrows) continue;
            const u64 wk = wkey[row]; const int wi = witem[row];
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const int il = ig + IG * c;
                const int item = (int)(base + il);
                if (base + il >= d2) continue;
                if (ex_ptr && ((mask[row * MW + (il >> 5)] >> (il & 31)) & 1u)) continue;
                const u64 ck = score_key(acc[r][c]);
                if (!better(ck, item, wk, wi)) continue;       // the common case: beats no entry of the unit
                const u64 *sk = hkey + row * H; const int *si = hitem + row * H;
                int lo = 0, hi = nv[row] - 1;                  // the worst entry is beaten: the answer is in [0, nv-1]
                while (lo < hi) { const int mid = (lo + hi) >> 1; if (better(ck, item, sk[mid], si[mid])) hi = mid; else lo = mid + 1; }
                atomicAdd(&hist[row * H + lo], 1);
            }
        }
        __syncthreads();                                      // the mask is rebuilt by the next tile
    }

    // ---- ranks: prefix sums of the histograms in sorted order, written to the entries' CSR positions
    constexpr int PER = H / 32;
    for (int r = warp; r < nrows; r += C::WARPS) {
        const int n = nv[r];
        const i64 g0 = unit_beg[row0 + r];
        int h[PER], s = 0;
#pragma unroll
        for (int q = 0; q < PER; ++q) { h[q] = hist[r * H + lane * PER + q]; s += h[q]; }
        int incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(FULL, incl, o); if (lane >= o) incl += v; }
        int run = incl - s;
#pragma unroll
        for (int q = 0; q < PER; ++q) {
            const int p = lane * PER + q;
            run += h[q];
            if (p < n) rank_out[g0 + hoff[r * H + p]] = 1 + run;
        }
    }
}

template <int UG, int H>
static void launch_rank(Ctx &c, const char *name, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr,
                        const int32_t *ex_item, const int32_t *ho_item, const int32_t *unit_user, const i64 *unit_beg,
                        i64 n_units, int32_t *rank_out, double *score_out) {
    typedef RankCfg<UG, H> C;
    auto kern = rank_kernel<UG, H>;
    PCR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::smem));
    const i64 grid = (n_units + C::BU - 1) / C::BU;
    const double bytes = (double)grid * d2 * k * 8.0 + (double)n_units * (k * 8.0 + H * 12.0);
    c.prof->begin(name, c.stream, bytes);
    kern<<<(unsigned)grid, C::THREADS, C::smem, c.stream>>>(U, V, d2, k, ex_ptr, ex_item, ho_item, unit_user, unit_beg,
                                                             n_units, rank_out, score_out);
    c.prof->end(c.stream);
    PCR_CUDA(cudaGetLastError());
}

void k_rank_heldout(Ctx &c, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr, const int32_t *ex_item,
                    const int32_t *ho_item, const int32_t *unit_user, const i64 *unit_beg, i64 n_units, int32_t *rank_out,
                    double *score_out) {
    PCR_REQUIRE(k >= 1 && k <= 256, "k out of range [1, 256]");
    if (n_units <= 0) return;
    launch_rank<8, RANK_UNIT>(c, "pcr::rank_kernel<8,64>", U, V, d2, k, ex_ptr, ex_item, ho_item, unit_user, unit_beg,
                              n_units, rank_out, score_out);
}

}  // namespace pcr
