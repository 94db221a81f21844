// kernels.h -- launchers of the hand-written sm_100a kernels (definitions in k_*.cu).
#pragma once
#include "common.cuh"

namespace pcr {

struct Ctx {               // what every launcher needs
    cudaStream_t stream;
    Profiler *prof;
    int sms;               // SM count of the device (grid sizing)
    unsigned long long *ticket;   // device counter for dynamically scheduled (work-stealing) kernels
};

// ---------------------------------------------------------------- k_setup.cu (one-time preprocessing)
void k_expand_users(Ctx &c, const i64 *row_ptr, i64 d1, i64 nnz, int32_t *user_out);
// *bad_flag |= 1: a rating rounds to a value outside the table; |= 2: some rating is not an integer
void k_levels(Ctx &c, const double *rating, i64 nnz, const i64 *table_dev, int T, uint8_t *level_out, int *bad_flag);
void k_iota32(Ctx &c, int32_t *out, i64 n);
void k_check_range(Ctx &c, const int32_t *idx, i64 n, i64 bound, int *bad_flag);   // *bad_flag |= 1 if any idx outside [0, bound)
// bpos[p*(nb+1)+j] = first CSC position of column p whose user id is >= j*block_users (users ascend inside a column)
void k_csc_block_bounds(Ctx &c, const i64 *col_ptr, const int32_t *csc_user, i64 d2, int nb, i64 block_users, i64 *bpos);
// CSC (by item) of a CSR: col_ptr[d2+1], csc2csr[nnz] (stable: users ascending inside an item), csc_user[nnz]
void k_build_csc(Ctx &c, DevPool &pool, const int32_t *item, const int32_t *user, i64 nnz, i64 d2,
                 i64 *col_ptr, int32_t *csc2csr, int32_t *csc_user);

// ---------------------------------------------------------------- k_hsort.cu
// heavy users: segmented sort of (score, position) pairs -- chunk sort in shared memory + merge-path passes over chunks
void k_heavy_sort(Ctx &c, const HeavySortPlan &h, const double *m, double *s_sorted, int32_t *pos_sorted);

// ---------------------------------------------------------------- k_core.cu
// out[e] = P[prow[e]] . Q[qrow[e]]  (rows are ld-strided, ld % 4 == 0); skipped when active[prow[e]] == 0
void k_dots(Ctx &c, const double *P, const int32_t *prow, const double *Q, const int32_t *qrow, i64 n, int ld, int kk,
            const uint8_t *active, double *out, double bytes);
// same as k_dots for the training set, user-major over row-sum units (P row in registers)
void k_dots_units(Ctx &c, const int32_t *un_seg, const i64 *un_start, const i64 *un_end, i64 n_units, const double *P, const double *Q,
                  const int32_t *qrow, int ld, int kk, const uint8_t *active, double *out, double bytes);
// out[seg] = lambda*x[seg] + sum_{e in seg} w[widx ? widx[e] : e] * M[ridx[e]]   (deterministic two-phase)
// un_end == nullptr: unit u covers [un_start[u], un_start[u+1]); seg_unit_idx == nullptr: a segment's units are contiguous
void k_rowsum(Ctx &c, const int32_t *un_seg, const i64 *un_start, const i64 *un_end, i64 n_units, const i64 *seg_unit_ptr,
              const int32_t *seg_unit_idx, i64 n_seg, const int32_t *ridx, const int32_t *widx, const double *w, const double *M, int ld,
              const uint8_t *active, double *partial, double lambda, const double *x, double *out,
              int zero_if_empty, double bytes, int kk);
// per-user sort of scores (classes S and L, bitonic in shared memory); writes s / pos / lev
void k_sort_users(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                  const double *m, const uint8_t *level, SortedMeta &meta);
void k_gather_level(Ctx &c, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                    const uint8_t *level, SortedMeta &meta);
// window pointers ub/lb and aggregated level counts cnt_lo/cnt_hi from the sorted scores
void k_windows(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
               SortedMeta &meta, int T, const i64 *heavy_off, int32_t *g_cnt);
// per-level counters of the sweep (test entry point): cntL/cntR [nnz x T] in sorted order
void k_level_counts(Ctx &c, const i64 *row_ptr, i64 d1, const SortedMeta &meta, int T, int32_t *cntL, int32_t *cntR);
// sweep coefficients: mode 0 gradient (stream = scores), 1 Hessian-vector (stream = b in CSR order); c_out CSR order
void k_sweep_coeff(Ctx &c, int cls, int mode, const int32_t *users, int n_users, const uint8_t *active,
                   const i64 *row_ptr, const SortedMeta &meta, const double *b, double *c_out, int T,
                   const i64 *heavy_off, double *g_v, double *g_p, double *g_acc);
// per-user objective (loss part only) -> obj_user[u]
void k_sweep_obj(Ctx &c, int cls, const int32_t *users, int n_users, const uint8_t *active, const i64 *row_ptr,
                 const SortedMeta &meta, double *obj_user, int T, const i64 *heavy_off, double *g_p1, double *g_p2,
                 double *g_acc);
// dense vector helpers (length n, deterministic reductions into slot[0..])
void k_fill(Ctx &c, double *x, i64 n, double v);
void k_axpby(Ctx &c, double *out, double a, const double *x, double b, const double *y, i64 n);  // out = a*x + b*y
void k_dot(Ctx &c, const double *x, const double *y, i64 n, double *partials, double *slot);      // slot = x.y
void k_sum(Ctx &c, const double *x, i64 n, double *partials, double *slot);
// one V-side CG iteration's vector algebra in two passes (partials: >= 2 x 592 doubles):
//   k_cg_dots2:  slot2[0] = p.Hp, slot2[1] = rr.p
//   k_cg_update: alpha = -slot_in[1] / slot_in[0] (on the device); delta += alpha p; rr += alpha Hp; slot2_out = {rr.rr, rr.Hp}
void k_cg_dots2(Ctx &c, const double *p, const double *Hp, const double *rr, i64 n, double *partials, double *slot2);
void k_cg_update(Ctx &c, double *delta, double *rr, const double *p, const double *Hp, i64 n, const double *slot_in, double *partials,
                 double *slot2_out);
void k_pad_copy(Ctx &c, const double *src, i64 rows, int k, int ld, double *dst);    // compact [rows x k] -> padded
// batched per-user Newton-CG state (one warp per user)
struct UState {
    double *g, *delta, *rr, *p, *Hp, *Unew;      // [d1 x ld]
    double *err, *step, *prev_obj, *obj_new, *loss;   // [d1]
    uint8_t *cg_active, *ls_active, *skipped;    // [d1]
    int32_t *cg_its, *ls_trials;                 // [d1]
    int *counters;                               // [0] active in CG, [1] active in LS
};
void k_u_init(Ctx &c, UState &s, const double *U, const i64 *row_ptr, const uint8_t *has_pairs, i64 d1, int ld,
              double lambda);
// the user-side rowsum_finalize (Hp = lambda p + unit partials, a user's units contiguous) and one CG iteration's
// scalar / vector updates of every user with cg_active, in one pass
void k_u_finalize_cg(Ctx &c, const i64 *seg_unit_ptr, const double *partial, UState &s, i64 d1, int ld, int kk, double lambda);
void k_u_ls_trial(Ctx &c, UState &s, const double *U, i64 d1, int ld, double stepsize0, int first);
void k_u_ls_check(Ctx &c, UState &s, i64 d1, int ld, double lambda, int last);
void k_u_commit(Ctx &c, UState &s, double *U, i64 d1, int ld);
void k_u_stats(Ctx &c, UState &s, const i64 *row_ptr, i64 d1, i64 *out8 /* device, 8 slots */);

// ---------------------------------------------------------------- k_tiles.cu (tiles of consecutive small users)
// geo 0: small tiles (users <= TILE_CAP ratings), geo 1: medium (TILE_CAP < len <= TILE_CAP_M), geo 2: large (<= TILE_CAP_L)
void k_tile_prepare(Ctx &c, const DevCsr &X, int geo, const uint8_t *active, const double *m, SortedMeta &meta, int T);
// mode 0 gradient coefficient, 1 Hv coefficient (stream b), 2 per-user loss
void k_tile_sweep(Ctx &c, int mode, const DevCsr &X, int geo, const uint8_t *active, const SortedMeta &meta, const double *b,
                  double *c_out, double *obj_user, int T);

// ---------------------------------------------------------------- k_heavy.cu (users longer than a tile, chunk-parallel)
// after k_heavy_sort + k_gather_level: level-major copy, window ranks and counters of every heavy user
void k_heavy_prepare(Ctx &c, const HeavyLM &h, SortedMeta &meta, int T);
// mode 0 gradient coefficient, 1 Hv coefficient (stream b), 2 per-user loss
void k_heavy_sweep(Ctx &c, int mode, const HeavyLM &h, const uint8_t *active, const SortedMeta &meta, const double *b,
                   double *c_out, double *obj_user, int T);

// ---------------------------------------------------------------- k_pairs.cu (Primal-CR pair kernels, evaluation)
// mode 0: gradient coefficient, 1: Hv coefficient (needs b), 2: objective partial per work item
void k_pairs(Ctx &c, int mode, const DevCsr &X, const uint8_t *active, const double *m, const double *b,
             double *c_out, double *obj_item);
void k_pair_obj_users(Ctx &c, const DevCsr &X, const uint8_t *active, const double *obj_item, double *obj_user);
void k_has_pairs(Ctx &c, const DevCsr &X, uint8_t *has_pairs);
// evaluation: pair errors per work item -> per user ratio; ndcg per user
void k_eval_pairs(Ctx &c, const DevCsr &X, const double *score, i64 *err_item);
// the same integer per USER from the sorted state (O(len * T), integer ratings only; T <= 8)
// ndcg_user != nullptr: also the per-user error ratio / NDCG@k / has-pair / has-any outputs of k_eval_users, from the same state
void k_eval_sorted(Ctx &c, const DevCsr &X, const SortedMeta &meta, int T, i64 *err_user, const double *level_vals, int ndcg_k,
                   double *err_ratio_user, double *ndcg_user, double *has_pair_user, double *has_any_user);
void k_eval_item_to_user(Ctx &c, const DevCsr &X, const i64 *err_item, i64 *err_user);
// err_per_user != 0: err_item holds one count per user (k_eval_sorted) instead of one per pair work item
void k_eval_users(Ctx &c, const DevCsr &X, const double *score, const i64 *err_item, int err_per_user, int ndcg_k,
                  double *err_ratio_user, double *ndcg_user, double *has_pair_user, double *has_any_user);

// ---------------------------------------------------------------- k_topn.cu (top-N recommendation)
// for each of n_users rows users[q]: the topn items of highest U[u] . V[i] (compact rows of k doubles), skipping the items
// of the user's ascending exclusion row (ex_ptr == nullptr: none); sorted best first, ties to the smaller item, NaN last;
// rows with fewer eligible items are padded with item -1 / score NaN.  scores_out may be nullptr.  1 <= topn, k <= 256.
void k_topn(Ctx &c, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr, const int32_t *ex_item,
            const int32_t *users, i64 n_users, int topn, int32_t *items_out, double *scores_out);
// similar rows: k_topn with U = V = M (n x k) and each query's own row never a candidate.  cosine: scores are
// dot / (|M[q]| * |M[i]|), the norms computed into norms[n] first (nullptr when !cosine).  1 <= topn, k <= 256.
void k_similar(Ctx &c, const double *M, i64 n, int k, bool cosine, double *norms, const i64 *ex_ptr,
               const int32_t *ex_item, const int32_t *queries, i64 n_queries, int topn, int32_t *ids_out,
               double *scores_out);
// held-out ranks: unit q is user unit_user[q] and held-out entries [unit_beg[q], unit_beg[q+1]) (at most RANK_UNIT of them,
// items ho_item[e]).  rank_out[e] = 1 + the number of the user's eligible items that rank before (score, item) of entry e in
// k_topn's order, or 0 when the item is in the user's exclusion row; score_out[e] (may be nullptr) is the score as k_topn
// returns it.  1 <= k <= 256.
constexpr int RANK_UNIT = 64;
void k_rank_heldout(Ctx &c, const double *U, const double *V, i64 d2, int k, const i64 *ex_ptr, const int32_t *ex_item,
                    const int32_t *ho_item, const int32_t *unit_user, const i64 *unit_beg, i64 n_units, int32_t *rank_out,
                    double *score_out);

}  // namespace pcr
