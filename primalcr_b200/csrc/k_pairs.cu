// k_pairs.cu -- all-pairs kernels: Primal-CR (pcr.cpp) and the pairwise-error / NDCG evaluation (util.cpp:434-542).
//
// A work item is (user, tile of PAIR_TJ consecutive ratings j); each thread owns one j and walks over ALL
// ratings k of the user (staged through shared memory in tiles of 1024), so every output element has exactly
// one writer: no atomics, deterministic.  A pair (j,k) is visited from both ends, which restates the
// reference's `t[j] += x; t[k] -= x` updates (pcr.cpp:139-140, 220-221, 374-375, 480-481) as one sum per j.
#include "kernels.h"

namespace pcr {

#define FULL 0xffffffffu
#define LAUNCH(ctx, name, bytes, kernel, grid, block, smem, ...)                         \
    do {                                                                                 \
        (ctx).prof->begin(name, (ctx).stream, (double)(bytes));                          \
        kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);                  \
        (ctx).prof->end((ctx).stream);                                                   \
        PCR_CUDA(cudaGetLastError());                                                    \
    } while (0)

static const int KT = 1024;

template <typename T>
__device__ __forceinline__ T block_sum256(T v, T *wsum) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(FULL, v, o);
    __syncthreads();
    if (lane == 0) wsum[warp] = v;
    __syncthreads();
    T r = 0;
    if (warp == 0) {
        r = lane < 8 ? wsum[lane] : (T)0;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(FULL, r, o);
    }
    return r;
}

// MODE 0: gradient coefficient  t_j  (obtain_g pcr.cpp:125-143, obtain_g_u :352-382)
// MODE 1: Hv coefficient        cp_j (compute_Ha pcr.cpp:202-224, obtain_Hs :459-485; active set recomputed
//                                     from the same scores m that filled D[] in obtain_g_u)
// MODE 2: objective             sum over pairs (1-mask)^2 (objective pcr.cpp:18-38, objective_u :406-425)
template <int MODE>
__global__ void __launch_bounds__(256) pairs_kernel(const int32_t *__restrict__ pt_user, const int32_t *__restrict__ pt_j0,
                                                    const uint8_t *__restrict__ active, const i64 *__restrict__ row_ptr,
                                                    const double *__restrict__ rating, const double *__restrict__ m,
                                                    const double *__restrict__ b, double *__restrict__ c_out,
                                                    double *__restrict__ obj_item) {
    __shared__ double sm_m[KT], sm_v[KT], sm_b[MODE == 1 ? KT : 1];
    __shared__ double wsum[8];
    const int item = blockIdx.x;
    const int u = pt_user[item];
    if (active && !active[u]) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const int tid = threadIdx.x;
    const int j = pt_j0[item] + tid;
    const bool has = j < n;
    double mj = 0.0, vj = 0.0, bj = 0.0;
    if (has) { mj = m[start + j]; vj = rating[start + j]; if (MODE == 1) bj = b[start + j]; }
    double acc = 0.0;
    for (int k0 = 0; k0 < n; k0 += KT) {
        __syncthreads();
        const int kt = (n - k0) < KT ? (n - k0) : KT;
        for (int q = tid; q < kt; q += 256) {
            sm_m[q] = m[start + k0 + q]; sm_v[q] = rating[start + k0 + q];
            if (MODE == 1) sm_b[q] = b[start + k0 + q];
        }
        __syncthreads();
        if (has) {
            for (int q = 0; q < kt; ++q) {
                const double vk = sm_v[q];
                if (vk == vj) continue;
                double mask = mj - sm_m[q];
                const bool lt = vj < vk;
                if (lt) mask = -mask;
                if (mask < 1.0) {
                    if (MODE == 0) { const double sjk = 2.0 * (mask - 1.0); acc += lt ? -sjk : sjk; }
                    else if (MODE == 1) { acc += 2.0 * (bj - sm_b[q]); }
                    else { acc += (1.0 - mask) * (1.0 - mask); }
                }
            }
        }
    }
    if (MODE == 2) {
        const double tot = block_sum256<double>(acc, wsum);
        if (tid == 0) obj_item[item] = 0.5 * tot;      // every unordered pair was visited twice
    } else if (has) {
        c_out[start + j] = acc;
    }
}

void k_pairs(Ctx &c, int mode, const DevCsr &X, const uint8_t *active, const double *m, const double *b,
             double *c_out, double *obj_item) {
    if (X.n_pt <= 0) return;
    const unsigned grid = (unsigned)X.n_pt;
    if (mode == 0) LAUNCH(c, "pairs_grad", 0.0, pairs_kernel<0>, grid, 256, 0, X.pt_user, X.pt_j0, active, X.row_ptr, X.rating, m, b, c_out, obj_item);
    else if (mode == 1) LAUNCH(c, "pairs_hv", 0.0, pairs_kernel<1>, grid, 256, 0, X.pt_user, X.pt_j0, active, X.row_ptr, X.rating, m, b, c_out, obj_item);
    else LAUNCH(c, "pairs_obj", 0.0, pairs_kernel<2>, grid, 256, 0, X.pt_user, X.pt_j0, active, X.row_ptr, X.rating, m, b, c_out, obj_item);
}

__global__ void pair_obj_users_kernel(const i64 *__restrict__ pt_ptr, i64 d1, const uint8_t *__restrict__ active,
                                      const double *__restrict__ obj_item, double *__restrict__ obj_user) {
    const i64 u = (i64)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= d1) return;
    if (active && !active[u]) return;
    double s = 0.0;
    for (i64 it = pt_ptr[u]; it < pt_ptr[u + 1]; ++it) s += obj_item[it];
    obj_user[u] = s;
}

void k_pair_obj_users(Ctx &c, const DevCsr &X, const uint8_t *active, const double *obj_item, double *obj_user) {
    if (X.d1 <= 0) return;
    LAUNCH(c, "pair_obj_users", 0.0, pair_obj_users_kernel, (unsigned)((X.d1 + 255) / 256), 256, 0, X.pt_ptr, X.d1, active, obj_item, obj_user);
}

// cc != 0 of update_u pcr.cpp:552: the user has at least one pair with different (exact) ratings
__global__ void has_pairs_kernel(const i64 *__restrict__ row_ptr, i64 d1, const double *__restrict__ rating,
                                 uint8_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const i64 u = ((i64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (u >= d1) return;
    const i64 s = row_ptr[u], e = row_ptr[u + 1];
    int diff = 0;
    if (e > s) {
        const double v0 = rating[s];
        for (i64 q = s + lane; q < e; q += 32) if (rating[q] != v0) diff = 1;
    }
    diff = __any_sync(FULL, diff);
    if (lane == 0) out[u] = diff ? 1 : 0;
}

void k_has_pairs(Ctx &c, const DevCsr &X, uint8_t *has_pairs) {
    if (X.d1 <= 0) return;
    LAUNCH(c, "has_pairs", 0.0, has_pairs_kernel, (unsigned)((X.d1 + 7) / 8), 256, 0, X.row_ptr, X.d1, X.rating, has_pairs);
}

// ------------------------------------------------------------------ evaluation (util.cpp:434-542)
// error_comps_i = #{(j,k) : val_j < val_k and score_j >= score_k}: the two `if`s at util.cpp:471-476 are this
// one predicate seen from either end of the pair, so counting it over ORDERED (j,k) visits each pair once.
__global__ void __launch_bounds__(256) eval_pairs_kernel(const int32_t *__restrict__ pt_user, const int32_t *__restrict__ pt_j0,
                                                         const i64 *__restrict__ row_ptr, const double *__restrict__ rating,
                                                         const double *__restrict__ score, i64 *__restrict__ err_item) {
    __shared__ double sm_s[KT], sm_v[KT];
    __shared__ i64 wsum[8];
    const int item = blockIdx.x;
    const int u = pt_user[item];
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const int tid = threadIdx.x;
    const int j = pt_j0[item] + tid;
    const bool has = j < n;
    double sj = 0.0, vj = 0.0;
    if (has) { sj = score[start + j]; vj = rating[start + j]; }
    i64 acc = 0;
    for (int k0 = 0; k0 < n; k0 += KT) {
        __syncthreads();
        const int kt = (n - k0) < KT ? (n - k0) : KT;
        for (int q = tid; q < kt; q += 256) { sm_s[q] = score[start + k0 + q]; sm_v[q] = rating[start + k0 + q]; }
        __syncthreads();
        if (has) {
            int a = 0;
            for (int q = 0; q < kt; ++q) a += (vj < sm_v[q] && sj >= sm_s[q]) ? 1 : 0;
            acc += a;
        }
    }
    const i64 tot = block_sum256<i64>(acc, wsum);
    if (tid == 0) err_item[item] = tot;
}

void k_eval_pairs(Ctx &c, const DevCsr &X, const double *score, i64 *err_item) {
    if (X.n_pt <= 0) return;
    LAUNCH(c, "eval_pairs", 0.0, eval_pairs_kernel, (unsigned)X.n_pt, 256, 0, X.pt_user, X.pt_j0, X.row_ptr, X.rating, score, err_item);
}

// The same integer from the SORTED state of Primal-CR++ in O(len * T) instead of O(len^2) (SURVEY App. A):
//   errors_u = sum_b #{a : l_a < l_b and s_a >= s_b} = sum_b sum_{t < l_b} (C_t(n) - C_t(x_b)),
// x_b = first sorted position whose score is >= s_b (the start of b's run of equal scores), C_t(x) = #{q < x : l_q = t}.
// Valid when every rating is an integer (then the lround levels order the ratings exactly like the doubles the
// reference compares, util.cpp:468-474) -- the engine checks that and otherwise keeps the all-pairs kernel above.
// One warp per user walks the sorted positions 32 at a time: per-level ballots give the in-chunk prefix counts, two
// small carried tables hold the counts before the chunk and at the start of a run of ties that began in an earlier chunk.
// The same warp also produces the user's NDCG@k from the sorted state (util.cpp:494-531): the k best-scored ratings are the
// tail of the ascending order (runs of equal scores taken smallest position first, as the arg-max kernel below does), the
// ideal ordering follows from the per-level totals (integer ratings: rating == level value).
template <int T>
__global__ void __launch_bounds__(256) eval_sorted_kernel(const i64 *__restrict__ row_ptr, i64 d1, const double *__restrict__ s_sorted,
                                                          const uint8_t *__restrict__ lev_sorted, i64 *__restrict__ err_user,
                                                          const int32_t *__restrict__ pos_sorted, const double *__restrict__ rating,
                                                          const double *__restrict__ level_vals, int ndcg_k,
                                                          double *__restrict__ err_ratio, double *__restrict__ ndcg,
                                                          double *__restrict__ has_pair, double *__restrict__ has_any) {
    const int lane = threadIdx.x & 31;
    const i64 u = ((i64)blockIdx.x * 256 + threadIdx.x) >> 5;
    if (u >= d1) return;
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    const unsigned lt_mask = (1u << lane) - 1u, le_mask = lt_mask | (1u << lane);
    int total[T], carry[T], run_cnt[T];
#pragma unroll
    for (int t = 0; t < T; ++t) { total[t] = 0; carry[t] = 0; run_cnt[t] = 0; }
    for (int base = 0; base < n; base += 32) {
        const int j = base + lane;
        const int lj = j < n ? (int)lev_sorted[start + j] : -1;
#pragma unroll
        for (int t = 0; t < T; ++t) total[t] += __popc(__ballot_sync(FULL, lj == t));
    }
    i64 err = 0;
    double last_key = 0.0;
    for (int base = 0; base < n; base += 32) {
        const int j = base + lane;
        const bool valid = j < n;
        const double sj = valid ? s_sorted[start + j] : 0.0;
        const int lj = valid ? (int)lev_sorted[start + j] : -1;
        int excl[T];
        unsigned bal[T];
#pragma unroll
        for (int t = 0; t < T; ++t) { bal[t] = __ballot_sync(FULL, lj == t); excl[t] = __popc(bal[t] & lt_mask); }
        double sprev = __shfl_up_sync(FULL, sj, 1);
        if (lane == 0) sprev = last_key;
        const bool is_start = valid && (j == 0 || sprev != sj);        // double compare: -0.0 and +0.0 tie, as in `>=`
        const unsigned sm = __ballot_sync(FULL, is_start) & le_mask;
        const int sl = sm ? 31 - __clz(sm) : -1;                       // lane where my run of ties starts, -1: earlier chunk
        int cs[T];
#pragma unroll
        for (int t = 0; t < T; ++t) {
            const int at = __shfl_sync(FULL, excl[t], sl & 31);
            cs[t] = sl >= 0 ? carry[t] + at : run_cnt[t];
        }
        if (valid) {
#pragma unroll
            for (int t = 0; t < T; ++t) if (t < lj) err += (i64)(total[t] - cs[t]);
        }
        const int cnt = (n - base) < 32 ? (n - base) : 32;
#pragma unroll
        for (int t = 0; t < T; ++t) { run_cnt[t] = __shfl_sync(FULL, cs[t], cnt - 1); carry[t] += __popc(bal[t]); }
        last_key = __shfl_sync(FULL, sj, cnt - 1);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) err += __shfl_xor_sync(FULL, err, o);
    if (lane != 0) return;
    err_user[u] = err;
    if (ndcg == nullptr) return;
    if (n == 0) { err_ratio[u] = 0.0; ndcg[u] = 0.0; has_pair[u] = 0.0; has_any[u] = 0.0; return; }
    const i64 num = (i64)n * (n - 1) / 2;
    has_any[u] = 1.0;
    if (num != 0) { err_ratio[u] = (double)err / (double)num; has_pair[u] = 1.0; }
    else { err_ratio[u] = 0.0; has_pair[u] = 0.0; }
    const int nowk = ndcg_k < n ? ndcg_k : n;
    double dcg = 0.0, idcg = 0.0;
    int r = 0, j = n - 1;
    while (r < nowk) {                                   // runs of equal scores from the top, each in ascending position order
        int a = j;
        const double sj = s_sorted[start + j];
        while (a > 0 && s_sorted[start + a - 1] == sj) --a;
        for (int q = a; q <= j && r < nowk; ++q, ++r)
            dcg += (exp2(rating[pos_sorted[start + q]]) - 1.0) / log2((double)(r + 1) + 1.0);
        j = a - 1;
    }
    r = 0;
#pragma unroll
    for (int t = T - 1; t >= 0; --t) {
        const double gain = exp2(level_vals[t]) - 1.0;
        for (int q = 0; q < total[t] && r < nowk; ++q, ++r) idcg += gain / log2((double)(r + 1) + 1.0);
    }
    ndcg[u] = dcg / idcg;
}

void k_eval_sorted(Ctx &c, const DevCsr &X, const SortedMeta &meta, int T, i64 *err_user, const double *level_vals, int ndcg_k,
                   double *err_ratio_user, double *ndcg_user, double *has_pair_user, double *has_any_user) {
    if (X.d1 <= 0) return;
    const unsigned grid = (unsigned)((X.d1 + 7) / 8);
#define ES(TT) LAUNCH(c, "eval_sorted_T" #TT, 0.0, eval_sorted_kernel<TT>, grid, 256, 0, X.row_ptr, X.d1, meta.s, meta.lev, err_user, meta.pos, X.rating, \
                      level_vals, ndcg_k, err_ratio_user, ndcg_user, has_pair_user, has_any_user)
    if (T <= 5) ES(5); else ES(8);
#undef ES
}

// per user: error ratio, NDCG@k (top-k by repeated arg-max; ties -> smaller index).  One WARP per user: the arg-max is a
// shuffle reduction, no block barriers (the block-per-user version spent 60 __syncthreads per user: 11.5 ms for the
// 480 k users of the Netflix shape, 7.5 ms even for a 10-ratings-per-user test set).
__global__ void __launch_bounds__(256) eval_users_kernel(const i64 *__restrict__ row_ptr, const i64 *__restrict__ pt_ptr,
                                                         const double *__restrict__ rating, const double *__restrict__ score,
                                                         const i64 *__restrict__ err_item, int err_per_user, int ndcg_k, i64 d1,
                                                         double *__restrict__ err_ratio, double *__restrict__ ndcg,
                                                         double *__restrict__ has_pair, double *__restrict__ has_any) {
    __shared__ int sel_all[8][64];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const i64 u = (i64)blockIdx.x * 8 + warp;
    if (u >= d1) return;
    int *sel = sel_all[warp];
    const i64 start = row_ptr[u];
    const int n = (int)(row_ptr[u + 1] - start);
    if (n == 0) {
        if (lane == 0) { err_ratio[u] = 0.0; ndcg[u] = 0.0; has_pair[u] = 0.0; has_any[u] = 0.0; }
        return;
    }
    if (lane == 0) {
        i64 err = 0;
        if (err_per_user) err = err_item[u];
        else for (i64 it = pt_ptr[u]; it < pt_ptr[u + 1]; ++it) err += err_item[it];
        const i64 num = (i64)n * (n - 1) / 2;
        has_any[u] = 1.0;
        if (num != 0) { err_ratio[u] = (double)err / (double)num; has_pair[u] = 1.0; }
        else { err_ratio[u] = 0.0; has_pair[u] = 0.0; }
    }
    int nowk = ndcg_k < n ? ndcg_k : n;
    if (nowk > 64) nowk = 64;
    double dcg[2] = {0.0, 0.0};
    for (int which = 0; which < 2; ++which) {
        const double *key = which == 0 ? score + start : rating + start;
        for (int r = 0; r < nowk; ++r) {
            double best = 0.0; int besti = -1;
            for (int j = lane; j < n; j += 32) {
                bool taken = false;
                for (int q = 0; q < r; ++q) taken |= (sel[q] == j);
                if (taken) continue;
                const double kj = key[j];
                if (besti < 0 || kj > best) { best = kj; besti = j; }   // j ascending: first max wins ties
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ob = __shfl_xor_sync(FULL, best, o);
                const int oi = __shfl_xor_sync(FULL, besti, o);
                if (oi >= 0 && (besti < 0 || ob > best || (ob == best && oi < besti))) { best = ob; besti = oi; }
            }
            if (lane == 0) {
                sel[r] = besti;
                dcg[which] += (exp2(rating[start + besti]) - 1.0) / log2((double)(r + 1) + 1.0);
            }
            __syncwarp();
        }
        __syncwarp();
    }
    if (lane == 0) ndcg[u] = dcg[0] / dcg[1];
}

void k_eval_users(Ctx &c, const DevCsr &X, const double *score, const i64 *err_item, int err_per_user, int ndcg_k,
                  double *err_ratio_user, double *ndcg_user, double *has_pair_user, double *has_any_user) {
    if (X.d1 <= 0) return;
    LAUNCH(c, "eval_users", 0.0, eval_users_kernel, (unsigned)((X.d1 + 7) / 8), 256, 0, X.row_ptr, X.pt_ptr, X.rating, score, err_item,
           err_per_user, ndcg_k, X.d1, err_ratio_user, ndcg_user, has_pair_user, has_any_user);
}

// per-user sums of the all-pairs work items (test entry point: integer counts per user)
__global__ void __launch_bounds__(256) eval_item_to_user_kernel(const i64 *__restrict__ pt_ptr, i64 d1, const i64 *__restrict__ err_item,
                                                                i64 *__restrict__ err_user) {
    const i64 u = (i64)blockIdx.x * 256 + threadIdx.x;
    if (u >= d1) return;
    i64 err = 0;
    for (i64 it = pt_ptr[u]; it < pt_ptr[u + 1]; ++it) err += err_item[it];
    err_user[u] = err;
}
void k_eval_item_to_user(Ctx &c, const DevCsr &X, const i64 *err_item, i64 *err_user) {
    if (X.d1 <= 0) return;
    LAUNCH(c, "eval_item_to_user", 0.0, eval_item_to_user_kernel, (unsigned)((X.d1 + 255) / 256), 256, 0, X.pt_ptr, X.d1, err_item, err_user);
}

}  // namespace pcr
