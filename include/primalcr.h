/*
 * primalcr.h -- C ABI of libprimalcr_b200.so: the B200-native Primal-CR / Primal-CR++ training path.
 *
 * This is the drop-in boundary for the reference's solver entry points
 *     extern "C" void pcr  (smat_t &X, mat_t &U, mat_t &V, testset_t &T, parameter &param);   pmf.h:54
 *     extern "C" void pcrpp(smat_t &X, mat_t &U, mat_t &V, testset_t &T, parameter &param);   pmf.h:55
 * (callers: run_pcr pmf-train.cpp:204, run_pcrpp pmf-train.cpp:273).  Those two symbols take C++
 * containers, so the replacement is a thin C++ shim (primalcr_b200/shim/pcr_shim.cpp, compiled against
 * the reference's own util.h/pmf.h) that flattens the containers and calls the plain-C functions below.
 * INTEGRATION.md shows the link line.  No torch / CUDA types appear in any signature.
 *
 * Conventions
 *   - every function returns 0 on success, a negative code on failure; primalcr_last_error() gives text;
 *   - host buffers are caller-owned, device buffers are library-owned;
 *   - one engine == one GPU == one host thread (or process).  Multi-GPU = one engine per GPU over a
 *     contiguous user shard, joined by primalcr_comm_init(); V-side sums go through NCCL allreduce;
 *   - users are 0-based rows of a CSR (row_ptr/item/rating) exactly as the reference's SparseMat
 *     (util.h:390-413): items ascending inside a user for the training set (util.h:240), file order for
 *     the test set (util.cpp:250-274);
 *   - U is d1 x k, V is d2 x k, row-major contiguous fp64, like the model file (util.cpp:30-51);
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with PRIMALCR_ECUDA.
 */
#ifndef PRIMALCR_H_
#define PRIMALCR_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRIMALCR_OK        0
#define PRIMALCR_EARG     -1   /* bad argument / call order            */
#define PRIMALCR_ECUDA    -2   /* CUDA runtime error (or no device)    */
#define PRIMALCR_ENCCL    -3   /* NCCL error / libnccl not loadable    */
#define PRIMALCR_EINTERNAL -4

#define PRIMALCR_SOLVER_PCR   1   /* pmf.h:6  enum {CCDR1, PCR, PCRPP}: -s 1 */
#define PRIMALCR_SOLVER_PCRPP 2   /*                                    -s 2 */

typedef struct primalcr_engine primalcr_engine;

/* mirrors the fields of `class parameter` (pmf.h:9-49) that pcr()/pcrpp() read */
typedef struct {
    int    solver;      /* param.solver_type : 1 Primal-CR, 2 Primal-CR++ (default 2)     */
    int    k;           /* param.k           : rank (default 10)                          */
    double lambda;      /* param.lambda      : default 5000                               */
    double stepsize;    /* param.stepsize    : default 1.0 (not settable from the CLI)    */
    int    maxiter;     /* param.maxiter     : outer iterations (default 10)              */
    int    ndcg_k;      /* param.ndcg_k      : default 10                                 */
    int    do_predict;  /* param.do_predict  : evaluate error/NDCG every iteration        */
    int    device;      /* CUDA device ordinal for this engine                            */
    int    threads;     /* param.threads     : only echoed in the "using N threads. " log line
                           (pcrpp.cpp:855, pcr.cpp:631); the GPU path has no use for it (default 4) */
} primalcr_config;

/* integer control-flow counters of the last outer iteration (they must match the oracle's) */
typedef struct {
    int64_t v_cg_iters;       /* CG iterations run by solve_delta(_new), <= 10                         */
    int64_t v_ls_trials;      /* line-search trials of update_V(_new), <= 20                           */
    int64_t v_ls_accepted;    /* 1 if a trial was accepted (V updated), 0 if V kept                    */
    int64_t u_cg_len_sum;     /* sum_i len_i * (CG iterations of user i)                               */
    int64_t u_ls_len_sum;     /* sum_i len_i * (line-search trials of user i)                          */
    int64_t u_skipped;        /* users returned unchanged (norm(g) < 1e-4, or cc == 0 for Primal-CR)   */
    int64_t u_cg_iters;       /* sum_i CG iterations                                                   */
    int64_t u_ls_trials;      /* sum_i line-search trials                                              */
} primalcr_counters;

typedef void (*primalcr_log_fn)(const char *line, void *ctx);

/* ---- lifecycle ------------------------------------------------------------------------------ */
void primalcr_default_config(primalcr_config *cfg);               /* pmf.h:26-47 defaults            */
int  primalcr_create(primalcr_engine **out, const primalcr_config *cfg);
void primalcr_destroy(primalcr_engine *e);
const char *primalcr_last_error(void);
const char *primalcr_version(void);

/* ---- data: replaces convert(smat_t&) util.cpp:219-247 and convert(testset_t&,..) util.cpp:250-274 -- */
/* Optional: the global table of distinct lround(rating) values, ascending (find_levels pcrpp.cpp:38-49
   computes it per user; a global order-preserving table gives identical results, SURVEY Appendix A).
   Needed when several engines shard one data set; otherwise derived from the training ratings. */
int primalcr_set_levels(primalcr_engine *e, const int64_t *level_values, int num_levels);
int primalcr_set_train_csr(primalcr_engine *e, int64_t d1, int64_t d2, int64_t nnz,
                           const int64_t *row_ptr, const int32_t *item, const double *rating);
int primalcr_set_test_csr(primalcr_engine *e, int64_t nnz,
                          const int64_t *row_ptr, const int32_t *item, const double *rating);
int primalcr_set_factors(primalcr_engine *e, const double *U, const double *V);
int primalcr_get_factors(primalcr_engine *e, double *U, double *V);

/* ---- multi-GPU: user shards + NCCL allreduce of the d2 x k V-side sums ------------------------- */
int primalcr_nccl_unique_id(void *id128);                         /* 128-byte ncclUniqueId, made on rank 0 */
/* id128 != NULL: create this (device, rank, world)'s communicator (collective: every rank calls it with the same id).
   id128 == NULL : re-attach to the communicator this PROCESS created earlier for the same (device, rank, world);
                   communicators are cached per process, so repeated solver calls pay ncclCommInitRank once. */
int primalcr_comm_init(primalcr_engine *e, int rank, int world, const void *id128);

/* ---- the solver: body of pcrpp() pcrpp.cpp:841-901 / pcr() pcr.cpp:616-704 ---------------------- */
int primalcr_initial_objective(primalcr_engine *e, double *obj);  /* comp_m + objective: "Iter 0 ... obj"      */
int primalcr_update_V(primalcr_engine *e, double *now_obj);       /* update_V_new pcrpp.cpp:415 / update_V pcr.cpp:279 */
int primalcr_update_U(primalcr_engine *e, double *now_obj);       /* update_U_new pcrpp.cpp:818 / update_U pcr.cpp:587 */
int primalcr_outer_iteration(primalcr_engine *e, double *now_obj);/* update_V then update_U                     */
/* compute_pairwise_error_ndcg util.cpp:434-542; which = 0 training set, 1 test set */
int primalcr_eval(primalcr_engine *e, int which, double *pairwise_error, double *ndcg);
/* the same evaluation with the integer pair-error count of every user written to err_per_user[d1] and every user's NDCG@k
   to ndcg_per_user[d1] (any pointer may be NULL).  A user's NDCG is 0 for an empty row, otherwise dcg / idcg of that user,
   which is NaN when idcg is 0 (every rating of the row is 0); the mean NDCG averages it over the non-empty rows.
   method 0: the reference's all-pairs count (util.cpp:467-479), O(len^2); method 1: the identical integer obtained from the
   Primal-CR++ sorted state in O(len * levels) (training set, integer ratings, <= 8 levels; PRIMALCR_EARG otherwise).
   primalcr_eval picks method 1 whenever it applies.  Both methods give bit-identical per-user NDCG. */
int primalcr_eval_error_counts(primalcr_engine *e, int which, int method, int64_t *err_per_user, double *ndcg_per_user,
                               double *pairwise_error, double *ndcg);
/* whole driver with the reference's stdout lines (one callback per line, without the newline) */
int primalcr_run(primalcr_engine *e, primalcr_log_fn log, void *ctx);
int primalcr_get_counters(primalcr_engine *e, primalcr_counters *out);

/* ---- per-stage entry points (parity tests call these through the same library) ----------------- */
/* comp_m_new pcrpp.cpp:17 : scores of every training rating, CSR order */
int primalcr_scores(primalcr_engine *e, double *m_out);
/* load externally supplied scores (so sort / counts can be compared bit-exactly on identical inputs); training-set
   evaluation (which = 0) then evaluates the loaded scores until the factors or the scores change */
int primalcr_set_scores(primalcr_engine *e, const double *m);
/* get_sorted_mm pcrpp.cpp:52 + the window pointers of the sweep pcrpp.cpp:214-229, for all users:
   per rating, in (user, ascending score) order: sorted score, local index of that score inside its user,
   global level index, ub = #{s <= s_j+1}, lb = #{s < s_j-1}, cnt_lo = sum_{t<l_j} count_right[t],
   cnt_hi = sum_{t>l_j} count_left[t].  Any output pointer may be NULL. */
int primalcr_sort_segments(primalcr_engine *e, double *sorted, int32_t *perm, int32_t *level,
                           int32_t *ub, int32_t *lb, int32_t *cnt_lo, int32_t *cnt_hi);
/* count_left[t] / count_right[t] of the sweep for every rating and level: [nnz x num_levels] each */
int primalcr_level_counts(primalcr_engine *e, int32_t *cnt_left, int32_t *cnt_right);
int primalcr_num_levels(primalcr_engine *e);
/* objective_new pcrpp.cpp:361 / objective pcr.cpp:5 on the current scores */
int primalcr_objective(primalcr_engine *e, double *obj);
/* obtain_g_new pcrpp.cpp:140 / obtain_g pcr.cpp:102 : d2 x k */
int primalcr_grad_V(primalcr_engine *e, double *g_out);
/* compute_Ha_new pcrpp.cpp:252 / compute_Ha pcr.cpp:167 : a and Ha are d2 x k */
int primalcr_hv_V(primalcr_engine *e, const double *a, double *Ha_out);
/* obtain_g_u_new pcrpp.cpp:493 + objective_u_new :542 for all users: g d1 x k, obj d1 */
int primalcr_grad_U(primalcr_engine *e, double *g_out, double *obj_u_out);
/* obtain_Hs_new pcrpp.cpp:576 / obtain_Hs pcr.cpp:430 for all users: S and HS are d1 x k */
int primalcr_hv_U(primalcr_engine *e, const double *S, double *HS_out);

/* ---- measurement -------------------------------------------------------------------------------- */
void   *primalcr_stream(primalcr_engine *e);                      /* cudaStream_t all kernels launch on  */
int64_t primalcr_launch_count(primalcr_engine *e);                /* kernels launched since create       */
int     primalcr_profile_enable(primalcr_engine *e, int on);      /* CUDA-event timing of every launch   */
int     primalcr_profile_reset(primalcr_engine *e);
int     primalcr_profile_count(primalcr_engine *e);               /* number of distinct kernel names     */
int     primalcr_profile_get(primalcr_engine *e, int idx, const char **name, double *total_ms,
                             int64_t *launches, double *bytes);   /* bytes = algorithmic bytes moved     */
int64_t primalcr_device_bytes(primalcr_engine *e);                /* device memory held by the engine    */

/* ---- prediction: the loop of omp-pmf-predict pmf-predict.cpp:57-64 as one batch on the GPU ------------------------
   out[t] = U[user[t]] . V[item[t]] for n (0-based) pairs; U is d1 x k, V is d2 x k row-major host arrays. */
int primalcr_predict(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int32_t *user,
                     const int32_t *item, int64_t n, double *out, int device);

/* ---- top-N recommendation: for each requested user, the topn items of highest U[u] . V[i] over all d2 items, skipping
   the items of that user's row in an optional exclusion CSR (normally the training set). U is d1 x k, V is d2 x k,
   row-major host arrays, as for primalcr_predict.
   - Order: sorted by score, highest first; ties go to the smaller item id.  Scores compare as doubles (+0.0 == -0.0);
     NaN ranks below -inf and NaN scores tie with each other, so the item id decides among them.
   - A returned item is never in the user's exclusion row and never repeats.  A user with fewer than topn eligible items
     gets the tail of its row padded with item -1 and score NaN.
   - A user's row is bit-identical from call to call and does not depend on which other users are in the batch or on
     n_users: each score is one fixed-order fp64 reduction over k.
   - 1 <= topn <= 256, 1 <= k <= 256.
   - Ids out of range, an exclusion row whose items do not ascend (repeats are allowed), excl_row_ptr without excl_item or
     any other bad argument returns PRIMALCR_EARG before any kernel runs; without a device the call returns PRIMALCR_ECUDA.
   - The library owns the stream and device memory of the call and releases them before returning. */
int primalcr_recommend(const double *U, int64_t d1, const double *V, int64_t d2, int k,
                       const int64_t *excl_row_ptr, const int32_t *excl_item,  /* d1+1 / row_ptr[d1]; both NULL: exclude nothing */
                       const int32_t *users, int64_t n_users,                  /* 0-based ids, any order, repeats allowed;
                                                                                  NULL: 0..d1-1, and n_users must be d1 */
                       int topn, int32_t *items_out, double *scores_out,       /* [n_users x topn] row-major; scores_out may be NULL */
                       int device);

/* ---- held-out ranking evaluation: the exact catalog rank of every held-out entry (normally the test set), scored and
   ordered as primalcr_recommend scores and orders, with every user's items of an optional exclusion CSR (normally the
   training set) removed from its candidates.  U, V, k and the exclusion CSR are as for primalcr_recommend.
   - Candidates of user u: the items not in u's exclusion row.  "Better" is primalcr_recommend's order: score descending,
     ties to the smaller item id, +0.0 == -0.0, NaN below -inf.
   - rank_out[e] for held-out entry e = (u, i): 1 + the number of u's candidates better than (score(u,i), i).  u's other
     held-out items are candidates too; an item never beats itself.  An entry whose item is in u's exclusion row gets 0
     (not a candidate, not ranked).
   - Held-out rows may be in any order and may repeat an item; every occurrence gets the same rank.
   - score_out[e] (may be NULL) is the score of entry e, the fma chain acc = fma(U[u][j], V[i][j], acc), j = 0..k-1, from
     +0.0, returned as primalcr_recommend returns scores (-0.0 as +0.0, every NaN as the default quiet NaN).  Hence, for
     every ranked entry with rank r <= N, primalcr_recommend(..., topn = N) returns item i at position r-1 of u's row with
     a bit-identical score, and for r > N item i is not in that row.
   - Ranks are bit-identical from call to call and do not depend on which other users have held-out entries.
   - 1 <= k <= 256, d1, d2 <= INT32_MAX.  The kernel scores the catalog once per user and run of 64 held-out entries.
   - Ids out of range, a decreasing ho_row_ptr or ho_row_ptr[0] != 0, the exclusion-row errors of primalcr_recommend, a
     NULL ho_row_ptr, or a NULL ho_item / rank_out when there are entries return PRIMALCR_EARG before any kernel runs;
     without a device the call returns PRIMALCR_ECUDA.
   - The library owns the stream and device memory of the call and releases them before returning.
   Several GPUs: split the users over devices (empty held-out rows cost nothing), one call per device. */
int primalcr_rank_heldout(const double *U, int64_t d1, const double *V, int64_t d2, int k,
                          const int64_t *excl_row_ptr, const int32_t *excl_item,  /* as primalcr_recommend; both NULL: none */
                          const int64_t *ho_row_ptr, const int32_t *ho_item,      /* held-out CSR: d1+1 / ho_row_ptr[d1] */
                          int32_t *rank_out, double *score_out,                   /* [ho_row_ptr[d1]], CSR order; score may be NULL */
                          int device);

/* ---- top-N metrics from held-out ranks (host only, no GPU).  rank[e] is primalcr_rank_heldout's rank of held-out entry e
   and ho_rating[e] its rating; the exclusion CSR is the one the ranks were computed with.  Per user u:
   - H_u: the distinct held-out items of u with rank > 0; an item's rating is the largest, its rank the smallest, among its
     entries with rank > 0.  R_u = {i in H_u : rating >= min_rating} are the relevant items (min_rating = -inf: all).
   - C_u = d2 - (number of distinct items in u's exclusion row); N_u = C_u - |R_u| non-relevant candidates.
   - Only users with |R_u| >= 1 are evaluated; *n_users is their number.
   - hits(N) = |{i in R_u : rank_i <= N}|;  recall@N = hits / |R_u|;  precision@N = hits / N.
   - NDCG@N with binary gains: DCG = sum_{i in R_u, rank_i <= N} 1 / log2(rank_i + 1), IDCG = sum_{p=1}^{min(N,|R_u|)}
     1 / log2(p + 1).  (2^r - 1 gains break on real-valued and negative ratings; min_rating carries the grading.)
   - MRR = 1 / min_{i in R_u} rank_i.
   - AUC_u = sum_{i in R_u} (N_u - (rank_i - 1 - pos_i)) / (|R_u| N_u), pos_i = the number of relevant items with a smaller
     rank; users with N_u = 0 are left out of the AUC mean.
   - Every metric is the plain mean over its users, summed in ascending user order in fp64 (deterministic); NaN when no
     user is evaluated.
   recall / precision / ndcg have n_cutoffs entries; any output may be NULL.  A rank outside [0, d2], a cutoff < 1, a
   malformed CSR (the exclusion rows must ascend as for primalcr_recommend) or a NULL array that is needed returns
   PRIMALCR_EARG. */
int primalcr_rank_metrics(int64_t d1, int64_t d2, const int64_t *excl_row_ptr, const int32_t *excl_item,
                          const int64_t *ho_row_ptr, const int32_t *ho_item, const double *ho_rating,
                          const int32_t *rank, double min_rating, const int32_t *cutoffs, int n_cutoffs,
                          double *recall, double *precision, double *ndcg,       /* [n_cutoffs] each; any may be NULL */
                          double *mrr, double *auc, int64_t *n_users);           /* any may be NULL */

/* ---- fast host loader for the reference's data directory (meta + ratings files): replaces load() util.cpp:6-25,
   smat_t::load_from_iterator util.h:201-271 and testset_t::load util.h:360-371 (no GPU needed) ------------------ */
typedef struct primalcr_dataset primalcr_dataset;
int  primalcr_load_dir(const char *data_dir, int threads, primalcr_dataset **out);
int  primalcr_dataset_info(const primalcr_dataset *ds, int64_t *d1, int64_t *d2, int64_t *nnz_train, int64_t *nnz_test);
/* which = 0 training CSR (sorted by user, item), 1 test CSR (file order inside a user); pointers stay owned by ds */
int  primalcr_dataset_csr(const primalcr_dataset *ds, int which, const int64_t **row_ptr, const int32_t **item,
                          const double **rating);
void primalcr_dataset_free(primalcr_dataset *ds);

/* ---- host utilities (no GPU needed) -------------------------------------------------------------- */
/* initial() util.cpp:80-93: default-seeded std::default_random_engine + normal_distribution<double>(0,1),
   row-major fill.  A fresh engine per call, so V equals the first d2 rows of U, as in the reference. */
void primalcr_reference_init(double *out, int64_t n, int64_t k);
/* The U.txt / V.txt side files of run_pcr / run_pcrpp (pmf-train.cpp:209-227, 276-295: `myfile << U[i][j]`, 6 significant
   digits, space separated, one row per line), formatted on all host threads; byte-identical to the reference's stream. */
int primalcr_write_text_matrix(const char *path, const double *M, int64_t rows, int k);

#ifdef __cplusplus
}
#endif
#endif /* PRIMALCR_H_ */
