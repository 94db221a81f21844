/*
 * pcr_oracle.c -- TEST INFRASTRUCTURE ONLY (parity oracle, not product code).
 *
 * A plain-C, single-threaded CPU restatement of the Primal-CR / Primal-CR++ training path of
 * wuliwei9278/primalCR.  Every function cites the reference file:line it follows.  Nothing in
 * primalcr_b200/ links, imports or executes this file; only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs may use it (as the checker / CPU baseline).
 *
 * Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4), so this
 * restatement is pinned against the reference ITSELF, compiled here from /root/reference into
 * oracle/_ref/ (see oracle/Makefile, oracle/ref_harness.cpp) -- tests/test_oracle_vs_ref.py -- and
 * against golden fixtures produced by that build (tests/golden/, generator tests/golden/make_golden.py).
 *
 * Conventions: CSR by user: index[d1+1], rows[nnz] = item id, vals[nnz] = rating (util.h:390-413,
 * util.cpp:219-247).  U is d1 x r, V is d2 x r, both row-major contiguous.  All arithmetic is fp64
 * and, inside one user's sweep, in exactly the reference's order (build with -ffp-contract=off).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>

typedef struct {
    long d1, d2, nnz;
    const long *index;   /* d1+1 */
    const long *rows;    /* item ids */
    const double *vals;  /* ratings */
} csr_t;

/* ---------------------------------------------------------------- dense helpers (util.cpp) */

/* util.cpp:103-109  dot(): iterates from the last element down */
static double dot_rev(const double *a, const double *b, long n) {
    double ret = 0;
    for (long i = n - 1; i >= 0; --i) ret += a[i] * b[i];
    return ret;
}
/* util.cpp:126-132  norm(vec) = SQUARED 2-norm, last element first */
static double norm_vec(const double *a, long n) {
    double ret = 0;
    for (long i = n - 1; i >= 0; --i) ret += a[i] * a[i];
    return ret;
}
/* util.cpp:133-138  norm(mat) = sum of row norms, last row first */
static double norm_mat(const double *M, long rows, long r) {
    double reg = 0;
    for (long i = rows - 1; i >= 0; --i) reg += norm_vec(M + i * r, r);
    return reg;
}
/* util.cpp:383-391 vec_prod_array: forward order */
static double dot_fwd(const double *a, const double *b, long n) {
    double res = 0.0;
    for (long i = 0; i < n; ++i) res += a[i] * b[i];
    return res;
}

/* ---------------------------------------------------------------- scores */

/* pcrpp.cpp:17-35 comp_m_new == pcr.cpp:47-66 comp_m : m[e] = sum_t U[u][t]*V[p][t], t ascending */
void orc_comp_m(long d1, long d2, long nnz, const long *index, const long *rows,
                const double *U, const double *V, int r, double *m) {
    (void)d2; (void)nnz;
    for (long u = 0; u < d1; ++u) {
        for (long e = index[u]; e < index[u + 1]; ++e) {
            const double *ui = U + u * r, *vj = V + rows[e] * r;
            double dot_res = 0;
            for (int j = 0; j < r; ++j) dot_res = dot_res + ui[j] * vj[j];
            m[e] = dot_res;
        }
    }
}

/* ---------------------------------------------------------------- per-user sorted state */

typedef struct { double key; long idx; } kv_t;

static int kv_cmp(const void *a, const void *b) {
    const kv_t *x = (const kv_t *)a, *y = (const kv_t *)b;
    if (x->key < y->key) return -1;
    if (x->key > y->key) return 1;
    /* std::sort is unstable (pcrpp.cpp:67-71); tie order never changes a result (every output is a
       function of the (score, level) multiset); we fix index order to make the oracle deterministic */
    return (x->idx > y->idx) - (x->idx < y->idx);
}

static int long_cmp(const void *a, const void *b) {
    long x = *(const long *)a, y = *(const long *)b;
    return (x > y) - (x < y);
}

/* struct infor_ui, pcrpp.cpp:5-14 */
typedef struct {
    long num_levels, len;
    double *mm_sorted;
    long *vals_sorted;   /* level index 0..num_levels-1 after the remap */
    long *d2bar_sorted;  /* item ids in sorted order */
    long *count_right;
    long *perm;          /* sorted position -> local index */
} infor_ui;

static void infor_free(infor_ui *p) {
    if (!p) return;
    free(p->mm_sorted); free(p->vals_sorted); free(p->d2bar_sorted); free(p->count_right); free(p->perm);
    free(p);
}

/* find_levels pcrpp.cpp:38-49 + get_sorted_mm :52-83 + get_sorted_vals :87-95 + get_sorted_d2bar
   :99-107 + the level remap loop :182-189 + get_count_right :129-137; this is precompute_ui :447-477
   (scores taken from mm[0..len), ratings/items from the user's CSR slice) */
static infor_ui *build_infor(const double *mm, const double *vals, const long *rows, long len) {
    infor_ui *p = (infor_ui *)calloc(1, sizeof(infor_ui));
    p->len = len;
    long nalloc = len > 0 ? len : 1;
    p->mm_sorted = (double *)malloc(sizeof(double) * nalloc);
    p->vals_sorted = (long *)malloc(sizeof(long) * nalloc);
    p->d2bar_sorted = (long *)malloc(sizeof(long) * nalloc);
    p->perm = (long *)malloc(sizeof(long) * nalloc);
    /* find_levels: distinct lround(vals), ascending */
    long *lv = (long *)malloc(sizeof(long) * nalloc);
    for (long i = 0; i < len; ++i) lv[i] = lround(vals[i]);
    qsort(lv, (size_t)len, sizeof(long), long_cmp);
    long nl = 0;
    for (long i = 0; i < len; ++i) if (i == 0 || lv[i] != lv[i - 1]) lv[nl++] = lv[i];
    p->num_levels = nl;
    /* argsort ascending */
    kv_t *kv = (kv_t *)malloc(sizeof(kv_t) * nalloc);
    for (long i = 0; i < len; ++i) { kv[i].key = mm[i]; kv[i].idx = i; }
    qsort(kv, (size_t)len, sizeof(kv_t), kv_cmp);
    for (long i = 0; i < len; ++i) {
        long j = kv[i].idx;
        p->perm[i] = j;
        p->mm_sorted[i] = kv[i].key;
        long v = lround(vals[j]);
        long k = 0;
        for (; k < nl; ++k) if (v == lv[k]) break;
        p->vals_sorted[i] = k;
        p->d2bar_sorted[i] = rows ? rows[j] : 0;
    }
    p->count_right = (long *)calloc((size_t)(nl > 0 ? nl : 1), sizeof(long));
    for (long i = 0; i < len; ++i) p->count_right[p->vals_sorted[i]] += 1;
    free(kv); free(lv);
    return p;
}

/* exported for the sort parity test: ascending argsort of one segment (get_sorted_mm pcrpp.cpp:52-83) */
void orc_sorted_mm(const double *mm, long len, double *mm_sorted, long *perm) {
    kv_t *kv = (kv_t *)malloc(sizeof(kv_t) * (size_t)(len > 0 ? len : 1));
    for (long i = 0; i < len; ++i) { kv[i].key = mm[i]; kv[i].idx = i; }
    qsort(kv, (size_t)len, sizeof(kv_t), kv_cmp);
    for (long i = 0; i < len; ++i) { mm_sorted[i] = kv[i].key; perm[i] = kv[i].idx; }
    free(kv);
}

/* The two-pointer sweep shared by obtain_g_new (pcrpp.cpp:194-236), compute_Ha_new (:287-318),
   obtain_g_u_new (:506-535) and obtain_Hs_new (:595-621).
   stream = mm_sorted for the gradient (add1 = 1: uses (mm-1)/(mm+1) factors), b_sorted for Hv (add1 = 0).
   Writes c[j] (already multiplied by 2.0) for every sorted position j.
   If cntL/cntR are non-NULL they receive, per j and level k, the integer counters count_left[k] /
   count_right[k] as they stand when c_j is formed (these are loop locals in the reference). */
static void sweep_coeff(const infor_ui *p, const double *stream, int add1, double *c,
                        long *cntL, long *cntR) {
    long len = p->len, nl = p->num_levels;
    const double *mm_sorted = p->mm_sorted;
    const long *vals_sorted = p->vals_sorted;
    long nlal = nl > 0 ? nl : 1;
    double *now_right_sum = (double *)calloc((size_t)nlal, sizeof(double));
    double *now_left_sum = (double *)calloc((size_t)nlal, sizeof(double));
    long *count_left = (long *)calloc((size_t)nlal, sizeof(long));
    long *count_right = (long *)malloc(sizeof(long) * (size_t)nlal);
    memcpy(count_right, p->count_right, sizeof(long) * (size_t)nl);
    /* get_levels_sum pcrpp.cpp:119-127 */
    for (long j = 0; j < len; ++j) now_right_sum[vals_sorted[j]] += stream[j];
    long now_left = 0, now_right = 0;
    for (long j = 0; j < len; ++j) {
        double now_cut = mm_sorted[j];
        long now_val = vals_sorted[j];
        long level;
        while (now_left < len && mm_sorted[now_left] <= now_cut + 1.0) {
            level = vals_sorted[now_left];
            now_left_sum[level] += stream[now_left];
            count_left[level] += 1;
            now_left += 1;
        }
        while (now_right < len && mm_sorted[now_right] < now_cut - 1.0) {
            level = vals_sorted[now_right];
            now_right_sum[level] -= stream[now_right];
            count_right[level] -= 1;
            now_right += 1;
        }
        double cc = 0.0;
        if (add1) {
            for (long k = 0; k <= now_val - 1; ++k)
                cc += (count_right[k] * (mm_sorted[j] - 1.0) - now_right_sum[k]);
            for (long k = now_val + 1; k < nl; ++k)
                cc += (count_left[k] * (mm_sorted[j] + 1.0) - now_left_sum[k]);
        } else {
            for (long k = 0; k <= now_val - 1; ++k)
                cc += (count_right[k] * stream[j] - now_right_sum[k]);
            for (long k = now_val + 1; k < nl; ++k)
                cc += (count_left[k] * stream[j] - now_left_sum[k]);
        }
        cc *= 2.0;
        c[j] = cc;
        if (cntL) for (long k = 0; k < nl; ++k) cntL[j * nl + k] = count_left[k];
        if (cntR) for (long k = 0; k < nl; ++k) cntR[j * nl + k] = count_right[k];
    }
    free(now_right_sum); free(now_left_sum); free(count_left); free(count_right);
}

/* objective sweep, objective_new pcrpp.cpp:388-407 == objective_u_new :552-571 (without the reg term) */
static double sweep_objective(const infor_ui *p) {
    long len = p->len, nl = p->num_levels;
    long nlal = nl > 0 ? nl : 1;
    const double *mm_sorted = p->mm_sorted;
    const long *vals_sorted = p->vals_sorted;
    long now_left = 0;
    long *count_left = (long *)calloc((size_t)nlal, sizeof(long));
    double *now_left_sum = (double *)calloc((size_t)nlal, sizeof(double));
    double *now_left_sqsum = (double *)calloc((size_t)nlal, sizeof(double));
    double res = 0.0;
    for (long j = 0; j < len; ++j) {
        double now_cut = mm_sorted[j];
        long now_val = vals_sorted[j];
        long level;
        while (now_left < len && mm_sorted[now_left] <= now_cut + 1.0) {
            level = vals_sorted[now_left];
            now_left_sum[level] += (mm_sorted[now_left] - 1.0);
            /* pow(x, 2.0) is folded to x*x by g++ -O3 */
            now_left_sqsum[level] += (mm_sorted[now_left] - 1.0) * (mm_sorted[now_left] - 1.0);
            count_left[level] += 1;
            now_left += 1;
        }
        for (long k = now_val + 1; k < nl; ++k)
            res += (count_left[k] * (now_cut * now_cut) - 2.0 * now_cut * now_left_sum[k] + now_left_sqsum[k]);
    }
    free(count_left); free(now_left_sum); free(now_left_sqsum);
    return res;
}

/* Per-level window counters of one segment (the loop locals of pcrpp.cpp:206-229).  levels_out gets the
   GLOBAL level index used by the CUDA path when level_map != NULL (level_map[k] = global index of the
   user's k-th local level), so that the integer counts can be compared bit-exactly. */
void orc_level_counts(const double *mm, const double *vals, long len, long *num_levels,
                      double *mm_sorted, long *perm, long *level_sorted, long *cntL, long *cntR) {
    infor_ui *p = build_infor(mm, vals, NULL, len);
    double *c = (double *)malloc(sizeof(double) * (size_t)(len > 0 ? len : 1));
    sweep_coeff(p, p->mm_sorted, 1, c, cntL, cntR);
    *num_levels = p->num_levels;
    for (long j = 0; j < len; ++j) { mm_sorted[j] = p->mm_sorted[j]; perm[j] = p->perm[j]; level_sorted[j] = p->vals_sorted[j]; }
    free(c); infor_free(p);
}

/* ---------------------------------------------------------------- Primal-CR++ V side */

/* obtain_g_new pcrpp.cpp:140-249 : g = lambda*V + sum_i sum_j c_ij e_{p_j} U_i^T */
void orc_obtain_g_new(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                      const double *U, const double *V, int r, const double *m, double lambda, double *g) {
    (void)nnz;
    for (long i = 0; i < d2 * r; ++i) g[i] = V[i] * lambda;  /* copy_mat_t(V, lambda) util.cpp:281-299 */
    for (long i = 0; i < d1; ++i) {
        long start = index[i], len = index[i + 1] - index[i];
        infor_ui *p = build_infor(m + start, vals + start, rows + start, len);
        double *c = (double *)malloc(sizeof(double) * (size_t)(len > 0 ? len : 1));
        sweep_coeff(p, p->mm_sorted, 1, c, NULL, NULL);
        for (long j = 0; j < len; ++j) {
            long q = p->d2bar_sorted[j];
            for (long k = 0; k < r; ++k) g[q * r + k] += c[j] * U[i * r + k];
        }
        free(c); infor_free(p);
    }
}

/* compute_Ha_new pcrpp.cpp:252-332 */
void orc_compute_Ha_new(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                        const double *a, const double *m, const double *U, int r, double lambda, double *Ha) {
    (void)nnz;
    for (long i = 0; i < d2 * r; ++i) Ha[i] = a[i] * lambda;  /* copy_vec_t(a, lambda) */
    for (long i = 0; i < d1; ++i) {
        long start = index[i], len = index[i + 1] - index[i];
        long nalloc = len > 0 ? len : 1;
        double *b = (double *)malloc(sizeof(double) * (size_t)nalloc);
        for (long k = 0; k < len; ++k) b[k] = dot_fwd(U + i * r, a + rows[start + k] * r, r);
        infor_ui *p = build_infor(m + start, vals + start, rows + start, len);
        double *b_sorted = (double *)malloc(sizeof(double) * (size_t)nalloc);
        for (long j = 0; j < len; ++j) b_sorted[j] = b[p->perm[j]];   /* get_sorted_b :109-117 */
        double *c = (double *)malloc(sizeof(double) * (size_t)nalloc);
        sweep_coeff(p, b_sorted, 0, c, NULL, NULL);
        for (long j = 0; j < len; ++j) {
            long q = p->d2bar_sorted[j];
            for (long ii = 0; ii < r; ++ii) { double tmp = c[j] * U[i * r + ii]; Ha[q * r + ii] += tmp; }
        }
        free(b); free(b_sorted); free(c); infor_free(p);
    }
}

/* objective_new pcrpp.cpp:361-412 */
double orc_objective_new(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                         const double *m, const double *U, const double *V, int r, double lambda) {
    (void)nnz; (void)rows;
    double res = 0.0;
    double norm_U = norm_mat(U, d1, r), norm_V = norm_mat(V, d2, r);
    for (long i = 0; i < d1; ++i) {
        long start = index[i], len = index[i + 1] - index[i];
        infor_ui *p = build_infor(m + start, vals + start, NULL, len);
        res += sweep_objective(p);
        infor_free(p);
    }
    res += lambda * (norm_U + norm_V) / 2.0;
    return res;
}

/* solve_delta_new pcrpp.cpp:335-358 (== solve_delta pcr.cpp:248-277 with compute_Ha).
   hv(ctx, p, Hp) evaluates the Hessian-vector product.  Returns the number of CG iterations run. */
typedef void (*hv_fn)(void *ctx, const double *p, double *Hp);

static int cg_solve(const double *g, long n, hv_fn hv, void *ctx, double *delta) {
    double *rr = (double *)malloc(sizeof(double) * (size_t)n);
    double *p = (double *)malloc(sizeof(double) * (size_t)n);
    double *Hp = (double *)malloc(sizeof(double) * (size_t)n);
    for (long i = 0; i < n; ++i) { delta[i] = 0.0; rr[i] = g[i] * -1.0; p[i] = g[i]; }
    double err = sqrt(norm_vec(rr, n)) * 0.01;
    int its = 0;
    for (int k = 1; k <= 10; ++k) {
        hv(ctx, p, Hp);
        ++its;
        double prod_p_Hp = dot_rev(p, Hp, n);
        double alpha = -1.0 * dot_rev(rr, p, n) / prod_p_Hp;
        for (long i = 0; i < n; ++i) delta[i] = delta[i] * 1.0 + p[i] * alpha;   /* add_vec_vec util.cpp:346-355 */
        for (long i = 0; i < n; ++i) rr[i] = rr[i] * 1.0 + Hp[i] * alpha;
        if (sqrt(norm_vec(rr, n)) < err) break;
        double b = dot_rev(rr, Hp, n) / prod_p_Hp;
        for (long i = 0; i < n; ++i) p[i] = rr[i] * -1.0 + p[i] * b;
    }
    free(rr); free(p); free(Hp);
    return its;
}

typedef struct {
    long d1, d2, nnz; const long *index, *rows; const double *vals, *m, *U; int r; double lambda;
} vctx_t;

static void hv_V_pp(void *c, const double *p, double *Hp) {
    vctx_t *x = (vctx_t *)c;
    orc_compute_Ha_new(x->d1, x->d2, x->nnz, x->index, x->rows, x->vals, p, x->m, x->U, x->r, x->lambda, Hp);
}

/* stats[0] = V-side CG iterations, stats[1] = line-search trials, stats[2] = 1 if a trial was accepted */
/* update_V_new pcrpp.cpp:415-444; m_out (nnz) receives the scores of the LAST trial */
void orc_update_V_new(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                      double lambda, double stepsize, int r, const double *U, double *V, double *now_obj,
                      double *m_out, long *stats) {
    long n = d2 * r;
    double *m = m_out;
    orc_comp_m(d1, d2, nnz, index, rows, U, V, r, m);
    double *g = (double *)malloc(sizeof(double) * (size_t)n);
    orc_obtain_g_new(d1, d2, nnz, index, rows, vals, U, V, r, m, lambda, g);
    double *delta = (double *)malloc(sizeof(double) * (size_t)n);
    vctx_t ctx = { d1, d2, nnz, index, rows, vals, m, U, r, lambda };
    int its = cg_solve(g, n, hv_V_pp, &ctx, delta);
    double prev_obj = orc_objective_new(d1, d2, nnz, index, rows, vals, m, U, V, r, lambda);
    double *V_new = (double *)malloc(sizeof(double) * (size_t)n);
    int trials = 0, accepted = 0;
    for (int iter = 0; iter < 20; ++iter) {
        for (long i = 0; i < n; ++i) V_new[i] = V[i];
        for (long i = 0; i < n; ++i) V_new[i] -= stepsize * delta[i];     /* mat_substract_vec util.cpp:395-408 */
        orc_comp_m(d1, d2, nnz, index, rows, U, V_new, r, m);
        *now_obj = orc_objective_new(d1, d2, nnz, index, rows, vals, m, U, V_new, r, lambda);
        ++trials;
        if (*now_obj < prev_obj) { memcpy(V, V_new, sizeof(double) * (size_t)n); accepted = 1; break; }
        else stepsize /= 2.0;
    }
    if (stats) { stats[0] = its; stats[1] = trials; stats[2] = accepted; }
    free(g); free(delta); free(V_new);
}

/* ---------------------------------------------------------------- Primal-CR++ U side */

/* obtain_g_u_new pcrpp.cpp:493-539 */
static void g_u_new(const infor_ui *p, const double *V, int r, double lambda, const double *ui, double *g) {
    if (p->len == 0) { for (int k = 0; k < r; ++k) g[k] = 0.0; return; }
    for (int k = 0; k < r; ++k) g[k] = ui[k] * lambda;
    double *c = (double *)malloc(sizeof(double) * (size_t)p->len);
    sweep_coeff(p, p->mm_sorted, 1, c, NULL, NULL);
    for (long j = 0; j < p->len; ++j) {
        const double *vp = V + p->d2bar_sorted[j] * r;
        for (int k = 0; k < r; ++k) g[k] = g[k] * 1.0 + vp[k] * c[j];   /* add_vec_vec(g, V[p], 1.0, c) */
    }
    free(c);
}

/* objective_u_new pcrpp.cpp:542-573 */
static double obj_u_new(const infor_ui *p, const double *ui, int r, double lambda) {
    double res = 0.0;
    res += lambda / 2.0 * norm_vec(ui, r);
    res += sweep_objective(p);   /* same accumulation: res starts at the reg term, then += per (j,k) */
    return res;
}

/* NOTE: the reference accumulates `res += term` per (j, level) starting FROM the regulariser; the helper
   above adds the sweep total to the regulariser instead.  The two differ by fp64 rounding only
   (<= 1 ulp of the total per term); tests compare at 1e-12 relative.  Same remark for objective_new,
   where the reference reduces per-thread partial sums under OpenMP anyway. */

typedef struct { const infor_ui *p; const double *V; int r; double lambda; } uctx_t;

/* obtain_Hs_new pcrpp.cpp:576-625 */
static void hv_u_pp(void *c, const double *s, double *Hs) {
    uctx_t *x = (uctx_t *)c;
    const infor_ui *p = x->p;
    int r = x->r;
    for (int k = 0; k < r; ++k) Hs[k] = s[k] * x->lambda;
    long len = p->len;
    long nalloc = len > 0 ? len : 1;
    double *b_sorted = (double *)malloc(sizeof(double) * (size_t)nalloc);
    for (long k = 0; k < len; ++k) b_sorted[k] = dot_rev(s, x->V + p->d2bar_sorted[k] * r, r);  /* dot() :593 */
    double *cf = (double *)malloc(sizeof(double) * (size_t)nalloc);
    sweep_coeff(p, b_sorted, 0, cf, NULL, NULL);
    for (long j = 0; j < len; ++j) {
        const double *vp = x->V + p->d2bar_sorted[j] * r;
        for (int k = 0; k < r; ++k) Hs[k] = Hs[k] * 1.0 + vp[k] * cf[j];
    }
    free(b_sorted); free(cf);
}

/* update_u_new pcrpp.cpp:779-815.  ustats[0] += CG its * len, ustats[1] += LS trials * len,
   ustats[2] += 1 if skipped by the norm test, ustats[3] += total CG its, ustats[4] += total LS trials */
static void update_u_new(long i, const long *index, const long *rows, const double *vals, const double *V,
                         const double *m, int r, double lambda, double stepsize, const double *ui,
                         double *ui_out, double *obj_u, long *ustats) {
    long start = index[i], len = index[i + 1] - index[i];
    infor_ui *p = build_infor(m + start, vals + start, rows + start, len);
    double *g = (double *)malloc(sizeof(double) * (size_t)r);
    g_u_new(p, V, r, lambda, ui, g);
    double prev_obj = obj_u_new(p, ui, r, lambda);
    if (norm_vec(g, r) < 0.0001) {
        *obj_u = prev_obj;
        for (int k = 0; k < r; ++k) ui_out[k] = ui[k];
        if (ustats) ustats[2] += 1;
        free(g); infor_free(p);
        return;
    }
    double *delta = (double *)malloc(sizeof(double) * (size_t)r);
    uctx_t ctx = { p, V, r, lambda };
    int its = cg_solve(g, r, hv_u_pp, &ctx, delta);
    long nalloc = len > 0 ? len : 1;
    double *mm = (double *)malloc(sizeof(double) * (size_t)nalloc);
    int trials = 0;
    for (int iter = 0; iter < 20; ++iter) {
        for (int k = 0; k < r; ++k) ui_out[k] = ui[k] * 1.0 + delta[k] * (-stepsize);
        /* compute_mm_old pcrpp.cpp:728-744 */
        for (long j = 0; j < len; ++j) {
            const double *vp = V + rows[start + j] * r;
            double res = 0.0;
            for (int k = 0; k < r; ++k) res += ui_out[k] * vp[k];
            mm[j] = res;
        }
        /* update_infor_ui :684-726 */
        infor_ui *pn = build_infor(mm, vals + start, rows + start, len);
        *obj_u = obj_u_new(pn, ui_out, r, lambda);
        infor_free(pn);
        ++trials;
        if (*obj_u < prev_obj) break; else stepsize /= 2.0;
    }
    if (ustats) { ustats[0] += its * len; ustats[1] += trials * len; ustats[3] += its; ustats[4] += trials; }
    free(mm); free(delta); free(g); infor_free(p);
}

/* update_U_new pcrpp.cpp:818-838 (race-free: obj_u_new is per user, i.e. the -n 1 behaviour) */
void orc_update_U_new(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                      const double *m, double lambda, double stepsize, int r, const double *V, double *U,
                      double *now_obj, long *ustats) {
    (void)nnz;
    double total_obj_new = 0.0;
    double *U_new = (double *)malloc(sizeof(double) * (size_t)(d1 * r > 0 ? d1 * r : 1));
    if (ustats) for (int q = 0; q < 5; ++q) ustats[q] = 0;
    for (long i = 0; i < d1; ++i) {
        double obj_u = 0.0;
        update_u_new(i, index, rows, vals, V, m, r, lambda, stepsize, U + i * r, U_new + i * r, &obj_u, ustats);
        total_obj_new += obj_u;
    }
    total_obj_new += lambda / 2.0 * norm_mat(V, d2, r);
    *now_obj = total_obj_new;
    memcpy(U, U_new, sizeof(double) * (size_t)(d1 * r));
    free(U_new);
}

/* per-user pieces exported for stage tests (obtain_g_u_new / objective_u_new / obtain_Hs_new) */
void orc_user_stage(long len, const long *rows, const double *vals, const double *m, const double *V, int r,
                    double lambda, const double *ui, const double *s, double *g, double *obj, double *Hs) {
    infor_ui *p = build_infor(m, vals, rows, len);
    g_u_new(p, V, r, lambda, ui, g);
    *obj = obj_u_new(p, ui, r, lambda);
    uctx_t ctx = { p, V, r, lambda };
    hv_u_pp(&ctx, s, Hs);
    infor_free(p);
}

/* ---------------------------------------------------------------- evaluation */

typedef struct { double key; long idx; } dk_t;
static int desc_cmp(const void *a, const void *b) {
    const dk_t *x = (const dk_t *)a, *y = (const dk_t *)b;
    if (x->key > y->key) return -1;
    if (x->key < y->key) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);
}

/* compute_pairwise_error_ndcg util.cpp:434-542 from given scores (score[e] of rating e, CSR order).
   out[0] = pairwise error, out[1] = ndcg.
   counts (optional, 4 longs): total error_comps, total num_comps, users with >=1 pair, users with >=1 rating.
   per_user_err (optional, d1 longs) = error_comps_i.
   per_user_ndcg (optional, d1 doubles) = dcg / dcg_max of the user (NaN when dcg_max is 0), 0 for an empty row */
void orc_eval_scores(long d1, const long *index, const double *vals, const double *scores, int ndcg_k, double *out,
                     long *counts, long *per_user_err, double *per_user_ndcg) {
    double sum_error = 0.0, ndcg_sum = 0.0;
    long total_count = 0, total_pair_d1 = 0, tot_err = 0, tot_cmp = 0;
    for (long i = 0; i < d1; ++i) {
        long start = index[i], end = index[i + 1] - 1, len = end - start + 1;
        if (per_user_err) per_user_err[i] = 0;
        if (per_user_ndcg) per_user_ndcg[i] = 0.0;
        if (len == 0) continue; else total_count += 1;
        const double *score = scores + start;
        long error_comps_i = 0, num_comps_i = 0;
        for (long j = start; j < end; ++j) {
            double val_j = vals[j];
            for (long k = j + 1; k <= end; ++k) {
                double val_k = vals[k];
                if (score[j - start] >= score[k - start] && val_j < val_k) error_comps_i++;
                if (score[j - start] <= score[k - start] && val_j > val_k) error_comps_i++;
                num_comps_i++;
            }
        }
        if (num_comps_i != 0) {
            sum_error += (double)error_comps_i / (double)num_comps_i;
            total_pair_d1++;
        }
        tot_err += error_comps_i; tot_cmp += num_comps_i;
        if (per_user_err) per_user_err[i] = error_comps_i;
        dk_t *bs = (dk_t *)malloc(sizeof(dk_t) * (size_t)len), *bv = (dk_t *)malloc(sizeof(dk_t) * (size_t)len);
        for (long k = 0; k < len; ++k) { bs[k].key = score[k]; bs[k].idx = k; bv[k].key = vals[start + k]; bv[k].idx = k; }
        qsort(bs, (size_t)len, sizeof(dk_t), desc_cmp);
        qsort(bv, (size_t)len, sizeof(dk_t), desc_cmp);
        double dcg = 0.0, dcg_max = 0.0;
        long nowk = ndcg_k;
        if (len < nowk) nowk = len;
        for (long k = 1; k <= nowk; ++k) {
            long id1 = bs[k - 1].idx;
            dcg += (pow(2.0, vals[start + id1]) - 1.0) / log2((double)k + 1.0);
            long id2 = bv[k - 1].idx;
            dcg_max += (pow(2.0, vals[start + id2]) - 1.0) / log2((double)k + 1.0);
        }
        ndcg_sum += dcg / dcg_max;
        if (per_user_ndcg) per_user_ndcg[i] = dcg / dcg_max;
        free(bs); free(bv);
    }
    out[0] = sum_error / (double)total_pair_d1;
    out[1] = ndcg_sum / (double)total_count;
    if (counts) { counts[0] = tot_err; counts[1] = tot_cmp; counts[2] = total_pair_d1; counts[3] = total_count; }
}

/* compute_pairwise_error_ndcg util.cpp:434-542 at the factors (U, V): the scores are U_i . V_j (dot_rev), then as above */
void orc_eval(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
              const double *U, const double *V, int r, int ndcg_k, double *out, long *counts, long *per_user_err,
              double *per_user_ndcg) {
    (void)d2;
    double *score = (double *)malloc(sizeof(double) * (size_t)(nnz > 0 ? nnz : 1));
    for (long i = 0; i < d1; ++i)
        for (long e = index[i]; e < index[i + 1]; ++e) score[e] = dot_rev(U + i * r, V + rows[e] * r, r);
    orc_eval_scores(d1, index, vals, score, ndcg_k, out, counts, per_user_err, per_user_ndcg);
    free(score);
}

/* ---------------------------------------------------------------- Primal-CR (pcr.cpp), O(len^2) pair loops */

/* objective pcr.cpp:5-43 */
double orc_pcr_objective(long d1, long d2, const long *index, const double *vals, const double *m,
                         const double *U, const double *V, int r, double lambda) {
    double res = 0;
    double norm_U = norm_mat(U, d1, r), norm_V = norm_mat(V, d2, r);
    for (long i = 0; i < d1; ++i) {
        long start = index[i], end = index[i + 1] - 1;
        for (long j = start; j <= end - 1; ++j) {
            double val_j = vals[j];
            for (long k = j + 1; k <= end; ++k) {
                double val_k = vals[k];
                if (val_j == val_k) continue;
                double mask = m[j] - m[k];
                if (val_j < val_k) mask = -mask;
                if (mask < 1.0) res += (1.0 - mask) * (1.0 - mask);
            }
        }
    }
    res += lambda * (norm_U + norm_V) / 2.0;
    return res;
}

/* obtain_g pcr.cpp:102-164 */
void orc_pcr_obtain_g(long d1, long d2, const long *index, const long *rows, const double *vals,
                      const double *U, const double *V, int r, const double *m, double lambda, double *g) {
    for (long i = 0; i < d2 * r; ++i) g[i] = V[i] * lambda;
    for (long i = 0; i < d1; ++i) {
        long start = index[i], end = index[i + 1] - 1, len = end - start + 1;
        double *t = (double *)calloc((size_t)(len > 0 ? len : 1), sizeof(double));
        for (long j = start; j <= end - 1; ++j) {
            double val_j = vals[j];
            for (long k = j + 1; k <= end; ++k) {
                double val_k = vals[k];
                double y_ijk = 1.0;
                if (val_j == val_k) continue; else if (val_j < val_k) y_ijk = -1.0;
                double mask = m[j] - m[k];
                mask *= y_ijk;
                if (mask < 1.0) {
                    double s_jk = 2.0 * (mask - 1);
                    t[j - start] += s_jk * y_ijk;
                    t[k - start] -= s_jk * y_ijk;
                }
            }
        }
        for (long k = 0; k < len; ++k) {
            long j = rows[start + k];
            double c = t[k];
            for (int kk = 0; kk < r; kk++) g[j * r + kk] += c * U[i * r + kk];
        }
        free(t);
    }
}

/* compute_Ha pcr.cpp:167-243 */
void orc_pcr_compute_Ha(long d1, long d2, const long *index, const long *rows, const double *vals,
                        const double *a, const double *m, const double *U, int r, double lambda, double *Ha) {
    for (long i = 0; i < d2 * r; ++i) Ha[i] = a[i] * lambda;
    for (long i = 0; i < d1; ++i) {
        long start = index[i], end = index[i + 1] - 1, len = end - start + 1;
        long nalloc = len > 0 ? len : 1;
        double *b = (double *)malloc(sizeof(double) * (size_t)nalloc);
        for (long k = 0; k < len; ++k) b[k] = dot_fwd(U + i * r, a + rows[start + k] * r, r);
        double *cpvals = (double *)calloc((size_t)nalloc, sizeof(double));
        for (long j = start; j < end; ++j) {
            double val_j = vals[j];
            for (long k = j + 1; k <= end; ++k) {
                double val_k = vals[k];
                if (val_j == val_k) continue;
                double mask = m[j] - m[k];
                if (val_k > val_j) mask = -mask;
                if (mask < 1.0) {
                    double ddd = b[j - start] - b[k - start];
                    ddd *= 2;
                    cpvals[j - start] += ddd;
                    cpvals[k - start] -= ddd;
                }
            }
        }
        for (long k = 0; k < len; ++k) {
            long q = rows[start + k];
            double c = cpvals[k];
            for (long j = 0; j < r; j++) Ha[q * r + j] += c * U[i * r + j];
        }
        free(b); free(cpvals);
    }
}

typedef struct { long d1, d2; const long *index, *rows; const double *vals, *m, *U; int r; double lambda; } pvctx_t;
static void hv_V_pcr(void *c, const double *p, double *Hp) {
    pvctx_t *x = (pvctx_t *)c;
    orc_pcr_compute_Ha(x->d1, x->d2, x->index, x->rows, x->vals, p, x->m, x->U, x->r, x->lambda, Hp);
}

/* update_V pcr.cpp:279-330 */
void orc_pcr_update_V(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                      double lambda, double stepsize, int r, const double *U, double *V, double *now_obj,
                      double *m_out, long *stats) {
    long n = d2 * r;
    double *m = m_out;
    orc_comp_m(d1, d2, nnz, index, rows, U, V, r, m);
    double *g = (double *)malloc(sizeof(double) * (size_t)n);
    orc_pcr_obtain_g(d1, d2, index, rows, vals, U, V, r, m, lambda, g);
    double *delta = (double *)malloc(sizeof(double) * (size_t)n);
    pvctx_t ctx = { d1, d2, index, rows, vals, m, U, r, lambda };
    int its = cg_solve(g, n, hv_V_pcr, &ctx, delta);
    double prev_obj = orc_pcr_objective(d1, d2, index, vals, m, U, V, r, lambda);
    double *V_new = (double *)malloc(sizeof(double) * (size_t)n);
    int trials = 0, accepted = 0;
    for (int iter = 0; iter < 20; ++iter) {
        for (long i = 0; i < n; ++i) V_new[i] = V[i];
        for (long i = 0; i < n; ++i) V_new[i] -= stepsize * delta[i];
        orc_comp_m(d1, d2, nnz, index, rows, U, V_new, r, m);
        *now_obj = orc_pcr_objective(d1, d2, index, vals, m, U, V_new, r, lambda);
        ++trials;
        if (*now_obj < prev_obj) { memcpy(V, V_new, sizeof(double) * (size_t)n); accepted = 1; break; }
        else stepsize /= 2.0;
    }
    if (stats) { stats[0] = its; stats[1] = trials; stats[2] = accepted; }
    free(g); free(delta); free(V_new);
}

/* objective_u pcr.cpp:396-427 */
static double pcr_objective_u(const double *mm, const double *ui, const double *vals, long len, int r, double lambda) {
    double res = 0.0;
    res += lambda / 2.0 * norm_vec(ui, r);
    for (long j = 0; j + 1 < len; ++j) {
        double val_j = vals[j];
        for (long k = j + 1; k < len; ++k) {
            double val_k = vals[k];
            if (val_j == val_k) continue;
            double mask = mm[j] - mm[k];
            if (val_j < val_k) mask = -mask;
            if (mask < 1.0) res += (1.0 - mask) * (1.0 - mask);
        }
    }
    return res;
}

typedef struct { long len; const long *rows; const double *vals; const double *D; const double *V; int r; double lambda; } puctx_t;

/* obtain_Hs pcr.cpp:430-496: active set taken from D (built by obtain_g_u from m) */
static void hv_u_pcr(void *c, const double *s, double *Hs) {
    puctx_t *x = (puctx_t *)c;
    int r = x->r; long len = x->len;
    for (int k = 0; k < r; ++k) Hs[k] = s[k] * x->lambda;
    long nalloc = len > 0 ? len : 1;
    double *b = (double *)malloc(sizeof(double) * (size_t)nalloc);
    for (long k = 0; k < len; ++k) {
        const double *vp = x->V + x->rows[k] * r;
        double res = 0.0;
        for (int kk = 0; kk < r; ++kk) res += s[kk] * vp[kk];
        b[k] = res;
    }
    double *cpvals = (double *)calloc((size_t)nalloc, sizeof(double));
    long cc = 0;
    for (long j = 0; j + 1 < len; ++j) {
        double val_j = x->vals[j];
        for (long k = j + 1; k < len; ++k) {
            double val_k = x->vals[k];
            if (val_j == val_k) continue;
            if (x->D[cc] > 0.0) {
                double ddd = b[j] - b[k];
                ddd *= 2.0;
                cpvals[j] += ddd;
                cpvals[k] -= ddd;
            }
            cc++;
        }
    }
    for (long k = 0; k < len; ++k) {
        const double *vp = x->V + x->rows[k] * r;
        for (int kk = 0; kk < r; ++kk) Hs[kk] = Hs[kk] * 1.0 + vp[kk] * cpvals[k];
    }
    free(b); free(cpvals);
}

/* update_u pcr.cpp:523-585 (with obtain_g_u :332-394 inlined) */
static void pcr_update_u(long i, const long *index, const long *rows, const double *vals, const double *V,
                         const double *m, int r, double lambda, double stepsize, const double *ui,
                         double *ui_out, double *obj_u, long *ustats) {
    long start = index[i], len = index[i + 1] - index[i];
    size_t num_pairs = (size_t)(len * (len - 1) / 2);
    double *D = (double *)malloc(sizeof(double) * (num_pairs > 0 ? num_pairs : 1));
    for (size_t q = 0; q < num_pairs; ++q) D[q] = -1.0;
    long cc = 0;
    double *g = (double *)malloc(sizeof(double) * (size_t)r);
    for (int k = 0; k < r; ++k) g[k] = ui[k] * lambda;
    long nalloc = len > 0 ? len : 1;
    double *t = (double *)calloc((size_t)nalloc, sizeof(double));
    for (long j = 0; j + 1 < len; ++j) {
        double val_j = vals[start + j];
        for (long k = j + 1; k < len; ++k) {
            double val_k = vals[start + k];
            if (val_j == val_k) continue;
            double mask = m[start + j] - m[start + k];
            if (val_k > val_j) mask = -mask;
            if (mask < 1.0) {
                D[cc] = 1.0;
                double s_jk = 2 * (1 - mask);
                if (val_k > val_j) s_jk = -s_jk;
                t[j] -= s_jk;
                t[k] += s_jk;
            }
            cc++;
        }
    }
    for (long k = 0; k < len; ++k) {
        const double *vp = V + rows[start + k] * r;
        for (int kk = 0; kk < r; ++kk) g[kk] = g[kk] * 1.0 + vp[kk] * t[k];
    }
    free(t);
    /* compute_mm pcr.cpp:83-99 with the CURRENT ui */
    double *mm = (double *)malloc(sizeof(double) * (size_t)nalloc);
    for (long j = 0; j < len; ++j) {
        const double *vp = V + rows[start + j] * r;
        double res = 0.0;
        for (int k = 0; k < r; ++k) res += ui[k] * vp[k];
        mm[j] = res;
    }
    double prev_obj = pcr_objective_u(mm, ui, vals + start, len, r, lambda);
    if (cc == 0 || norm_vec(g, r) < 0.0001) {
        *obj_u = prev_obj;
        for (int k = 0; k < r; ++k) ui_out[k] = ui[k];
        if (ustats) ustats[2] += 1;
        free(D); free(mm); free(g);
        return;
    }
    double *delta = (double *)malloc(sizeof(double) * (size_t)r);
    puctx_t ctx = { len, rows + start, vals + start, D, V, r, lambda };
    int its = cg_solve(g, r, hv_u_pcr, &ctx, delta);
    int trials = 0;
    for (int iter = 0; iter < 20; ++iter) {
        for (int k = 0; k < r; ++k) ui_out[k] = ui[k] * 1.0 + delta[k] * (-stepsize);
        for (long j = 0; j < len; ++j) {
            const double *vp = V + rows[start + j] * r;
            double res = 0.0;
            for (int k = 0; k < r; ++k) res += ui_out[k] * vp[k];
            mm[j] = res;
        }
        *obj_u = pcr_objective_u(mm, ui_out, vals + start, len, r, lambda);
        ++trials;
        if (*obj_u < prev_obj) break; else stepsize /= 2.0;
    }
    if (ustats) { ustats[0] += its * len; ustats[1] += trials * len; ustats[3] += its; ustats[4] += trials; }
    free(D); free(mm); free(g); free(delta);
}

/* update_U pcr.cpp:587-611 (race-free) */
void orc_pcr_update_U(long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
                      const double *m, double lambda, double stepsize, int r, const double *V, double *U,
                      double *now_obj, long *ustats) {
    (void)nnz;
    double total_obj_new = 0.0;
    double *U_new = (double *)malloc(sizeof(double) * (size_t)(d1 * r > 0 ? d1 * r : 1));
    if (ustats) for (int q = 0; q < 5; ++q) ustats[q] = 0;
    for (long i = 0; i < d1; ++i) {
        double obj_u = 0.0;
        pcr_update_u(i, index, rows, vals, V, m, r, lambda, stepsize, U + i * r, U_new + i * r, &obj_u, ustats);
        total_obj_new += obj_u;
    }
    total_obj_new += lambda / 2.0 * norm_mat(V, d2, r);
    *now_obj = total_obj_new;
    memcpy(U, U_new, sizeof(double) * (size_t)(d1 * r));
    free(U_new);
}

/* ---------------------------------------------------------------- drivers: pcrpp() pcrpp.cpp:841-901, pcr() pcr.cpp:616-704
   solver: 1 = Primal-CR, 2 = Primal-CR++.  obj[0..maxiter] receives "Iter i ... obj" values;
   evals (optional, (maxiter+1)*4 doubles) = train err, train ndcg, test err, test ndcg per iteration;
   counters (optional, maxiter*8 longs) = per iteration: V CG its, V LS trials, V accepted,
   sum(len*cg_i), sum(len*ls_i), users skipped, sum cg_i, sum ls_i. */
void orc_train(int solver, long d1, long d2, long nnz, const long *index, const long *rows, const double *vals,
               long nnz_t, const long *index_t, const long *rows_t, const double *vals_t,
               double *U, double *V, int r, double lambda, double stepsize, int maxiter, int do_predict,
               int ndcg_k, double *obj, double *evals, long *counters) {
    double *m = (double *)malloc(sizeof(double) * (size_t)(nnz > 0 ? nnz : 1));
    orc_comp_m(d1, d2, nnz, index, rows, U, V, r, m);
    double now_obj = solver == 2 ? orc_objective_new(d1, d2, nnz, index, rows, vals, m, U, V, r, lambda)
                                 : orc_pcr_objective(d1, d2, index, vals, m, U, V, r, lambda);
    obj[0] = now_obj;
    for (int iter = 0; iter <= maxiter; ++iter) {
        if (iter > 0) {
            long st[3] = {0, 0, 0}, us[5] = {0, 0, 0, 0, 0};
            if (solver == 2) {
                orc_update_V_new(d1, d2, nnz, index, rows, vals, lambda, stepsize, r, U, V, &now_obj, m, st);
                orc_update_U_new(d1, d2, nnz, index, rows, vals, m, lambda, stepsize, r, V, U, &now_obj, us);
            } else {
                orc_pcr_update_V(d1, d2, nnz, index, rows, vals, lambda, stepsize, r, U, V, &now_obj, m, st);
                orc_pcr_update_U(d1, d2, nnz, index, rows, vals, m, lambda, stepsize, r, V, U, &now_obj, us);
            }
            obj[iter] = now_obj;
            if (counters) {
                long *c = counters + (iter - 1) * 8;
                c[0] = st[0]; c[1] = st[1]; c[2] = st[2]; c[3] = us[0]; c[4] = us[1]; c[5] = us[2]; c[6] = us[3]; c[7] = us[4];
            }
        }
        if (evals) {
            double *e = evals + iter * 4;
            e[0] = e[1] = e[2] = e[3] = 0.0;
            if (do_predict) {
                double o[2];
                orc_eval(d1, d2, nnz, index, rows, vals, U, V, r, ndcg_k, o, NULL, NULL, NULL);
                e[0] = o[0]; e[1] = o[1];
                if (nnz_t != 0) {
                    orc_eval(d1, d2, nnz_t, index_t, rows_t, vals_t, U, V, r, ndcg_k, o, NULL, NULL, NULL);
                    e[2] = o[0]; e[3] = o[1];
                }
            }
        }
    }
    free(m);
}
