// queries.cu -- the one-shot queries of the C ABI (include/primalcr.h): prediction, top-N recommendation, similar rows and
// held-out ranks on the GPU, and the host-only ranking metrics.  A GPU query checks its arguments (scalars, then the
// device, then the id and CSR scans), opens a Session, uploads, makes one launcher call and downloads.
#include "kernels.h"
#include "abi.h"
#include "../host/loader.hpp"
#include "../host/rankmetrics.hpp"

namespace {

void require_device(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        throw pcr::Error(PRIMALCR_ECUDA, "no CUDA device available: libprimalcr_b200 has no CPU fallback");
    PCR_REQUIRE(device >= 0 && device < ndev, "bad device ordinal");
}

// U (d1 x k) and V (d2 x k) of the kernels of k_topn.cu
void check_factors(const double *U, int64_t d1, const double *V, int64_t d2, int k) {
    PCR_REQUIRE(k >= 1 && k <= 256, "rank k out of range [1, 256]");
    PCR_REQUIRE(d1 >= 0 && d2 >= 0 && d1 <= INT32_MAX && d2 <= INT32_MAX, "d1 / d2 out of range");
    PCR_REQUIRE((U || d1 == 0) && (V || d2 == 0), "null factor matrix");
}

// every id a kernel reads through is checked before anything runs
void check_ids(const int32_t *ids, int64_t n, int64_t bound, const char *msg) {
    bool bad = false;
#pragma omp parallel for reduction(|| : bad) schedule(static)
    for (int64_t t = 0; t < n; ++t) bad = bad || ids[t] < 0 || ids[t] >= bound;
    PCR_REQUIRE(!bad, msg);
}

// the exclusion CSR of primalcr_recommend / primalcr_similar / primalcr_rank_heldout: both pointers or neither, ascending
// rows -> its nnz
int64_t check_exclusion(int64_t d1, int64_t d2, const int64_t *excl_row_ptr, const int32_t *excl_item) {
    if (!excl_row_ptr) return 0;
    const std::string err = pcrhost::csr_error("exclusion", d1, d2, excl_row_ptr, excl_item, true);
    PCR_REQUIRE(err.empty(), err);
    return excl_row_ptr[d1];
}

// Argument checks of a top-N call (primalcr_recommend, primalcr_similar): rows users[0..n_users) of U (users NULL: every
// row) against the d2 rows of V, with an optional d1 x d2 exclusion CSR -> the exclusion's nnz.
int64_t check_topn(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int64_t *excl_row_ptr,
                   const int32_t *excl_item, const int32_t *users, int64_t n_users, int topn, const int32_t *items_out,
                   int device) {
    check_factors(U, d1, V, d2, k);
    PCR_REQUIRE(topn >= 1 && topn <= 256, "topn out of range [1, 256]");
    PCR_REQUIRE(n_users >= 0 && (users || n_users == d1), "users == NULL requires n_users == d1");
    PCR_REQUIRE(n_users == 0 || items_out, "null items_out");
    PCR_REQUIRE((excl_row_ptr == nullptr) == (excl_item == nullptr), "excl_row_ptr and excl_item must both be given or both be NULL");
    require_device(device);
    if (users) check_ids(users, n_users, d1, "user id out of range");
    return check_exclusion(d1, d2, excl_row_ptr, excl_item);
}

// One query call's device state: a non-blocking stream and buffers from plain cudaMalloc.  The destructor drains and
// destroys the stream before the members (the buffers) are released, on every exit, exceptions included; the stream is
// the last thing the constructor creates, so a constructor that throws leaves nothing behind.
struct Session {
    pcr::DevPool pool;
    pcr::Profiler prof;
    pcr::Ctx ctx{nullptr, &prof, 0, nullptr};     // no ticket: the query launchers schedule no work dynamically

    explicit Session(int device) {
        PCR_CUDA(cudaSetDevice(device));
        PCR_CUDA(cudaDeviceGetAttribute(&ctx.sms, cudaDevAttrMultiProcessorCount, device));
        PCR_CUDA(cudaStreamCreateWithFlags(&ctx.stream, cudaStreamNonBlocking));
    }
    ~Session() { cudaStreamSynchronize(ctx.stream); cudaStreamDestroy(ctx.stream); }
    Session(const Session &) = delete; Session &operator=(const Session &) = delete;

    template <class T> T *upload(const T *host, size_t n) {
        T *dev = pool.alloc<T>(n);
        if (n) PCR_CUDA(cudaMemcpyAsync(dev, host, sizeof(T) * n, cudaMemcpyHostToDevice, ctx.stream));
        return dev;
    }
    template <class T> void download(T *host, const T *dev, size_t n) {
        if (n) PCR_CUDA(cudaMemcpyAsync(host, dev, sizeof(T) * n, cudaMemcpyDeviceToHost, ctx.stream));
    }
    void sync() { PCR_CUDA(cudaStreamSynchronize(ctx.stream)); }
};

}  // namespace

extern "C" {

// ---- prediction (pmf-predict.cpp:57-64) ---------------------------------------------------------------
int primalcr_predict(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int32_t *user,
                     const int32_t *item, int64_t n, double *out, int device) {
    API_BEGIN
    PCR_REQUIRE(U && V && (n == 0 || (user && item && out)) && k >= 1 && d1 >= 0 && d2 >= 0, "bad argument");
    require_device(device);
    check_ids(user, n, d1, "user/item id out of range");
    check_ids(item, n, d2, "user/item id out of range");
    Session s(device);
    const int ld = pcr::ceil16(k);
    const double *Uc = s.upload(U, (size_t)d1 * k), *Vc = s.upload(V, (size_t)d2 * k);
    const int32_t *ud = s.upload(user, (size_t)n), *id = s.upload(item, (size_t)n);
    double *Ud = s.pool.alloc<double>((size_t)d1 * ld), *Vd = s.pool.alloc<double>((size_t)d2 * ld);
    double *od = s.pool.alloc<double>((size_t)n);
    pcr::k_pad_copy(s.ctx, Uc, d1, k, ld, Ud); pcr::k_pad_copy(s.ctx, Vc, d2, k, ld, Vd);
    pcr::k_dots(s.ctx, Ud, ud, Vd, id, n, ld, k, nullptr, od, 0.0);
    s.download(out, od, (size_t)n);
    s.sync();
    API_END
}

// ---- top-N recommendation ---------------------------------------------------------------------------------------
int primalcr_recommend(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int64_t *excl_row_ptr,
                       const int32_t *excl_item, const int32_t *users, int64_t n_users, int topn, int32_t *items_out,
                       double *scores_out, int device) {
    API_BEGIN
    const int64_t ex_nnz = check_topn(U, d1, V, d2, k, excl_row_ptr, excl_item, users, n_users, topn, items_out, device);
    if (n_users == 0) return PRIMALCR_OK;
    Session s(device);
    const size_t n_out = (size_t)n_users * topn;
    const double *Ud = s.upload(U, (size_t)d1 * k), *Vd = s.upload(V, (size_t)d2 * k);
    int32_t *ud = users ? s.upload(users, (size_t)n_users) : s.pool.alloc<int32_t>((size_t)n_users);
    if (!users) pcr::k_iota32(s.ctx, ud, n_users);
    const pcr::i64 *exp_d = excl_row_ptr ? s.upload((const pcr::i64 *)excl_row_ptr, (size_t)d1 + 1) : nullptr;
    const int32_t *exi_d = excl_row_ptr ? s.upload(excl_item, (size_t)ex_nnz) : nullptr;
    int32_t *itd = s.pool.alloc<int32_t>(n_out);
    double *scd = scores_out ? s.pool.alloc<double>(n_out) : nullptr;
    pcr::k_topn(s.ctx, Ud, Vd, d2, k, exp_d, exi_d, ud, n_users, topn, itd, scd);
    s.download(items_out, itd, n_out);
    if (scores_out) s.download(scores_out, scd, n_out);
    s.sync();
    API_END
}

// ---- similar items / users ---------------------------------------------------------------------------------------
int primalcr_similar(const double *M, int64_t n, int k, int measure, const int64_t *excl_row_ptr, const int32_t *excl_id,
                     const int32_t *queries, int64_t n_queries, int topn, int32_t *ids_out, double *scores_out, int device) {
    API_BEGIN
    PCR_REQUIRE(measure == PRIMALCR_SIM_DOT || measure == PRIMALCR_SIM_COSINE, "unknown similarity measure");
    const int64_t ex_nnz = check_topn(M, n, M, n, k, excl_row_ptr, excl_id, queries, n_queries, topn, ids_out, device);
    if (n_queries == 0) return PRIMALCR_OK;
    Session s(device);
    const bool cosine = measure == PRIMALCR_SIM_COSINE;
    const size_t n_out = (size_t)n_queries * topn;
    const double *Md = s.upload(M, (size_t)n * k);
    int32_t *qd = queries ? s.upload(queries, (size_t)n_queries) : s.pool.alloc<int32_t>((size_t)n_queries);
    if (!queries) pcr::k_iota32(s.ctx, qd, n_queries);
    const pcr::i64 *exp_d = excl_row_ptr ? s.upload((const pcr::i64 *)excl_row_ptr, (size_t)n + 1) : nullptr;
    const int32_t *exi_d = excl_row_ptr ? s.upload(excl_id, (size_t)ex_nnz) : nullptr;
    int32_t *itd = s.pool.alloc<int32_t>(n_out);
    double *scd = scores_out ? s.pool.alloc<double>(n_out) : nullptr;
    double *norms = cosine ? s.pool.alloc<double>((size_t)n) : nullptr;
    pcr::k_similar(s.ctx, Md, n, k, cosine, norms, exp_d, exi_d, qd, n_queries, topn, itd, scd);
    s.download(ids_out, itd, n_out);
    if (scores_out) s.download(scores_out, scd, n_out);
    s.sync();
    API_END
}

// ---- held-out ranking evaluation --------------------------------------------------------------------------------
int primalcr_rank_heldout(const double *U, int64_t d1, const double *V, int64_t d2, int k, const int64_t *excl_row_ptr,
                          const int32_t *excl_item, const int64_t *ho_row_ptr, const int32_t *ho_item, int32_t *rank_out,
                          double *score_out, int device) {
    API_BEGIN
    check_factors(U, d1, V, d2, k);
    PCR_REQUIRE(ho_row_ptr, "null ho_row_ptr");
    PCR_REQUIRE((excl_row_ptr == nullptr) == (excl_item == nullptr), "excl_row_ptr and excl_item must both be given or both be NULL");
    require_device(device);
    const int64_t nnz = ho_row_ptr[d1];
    PCR_REQUIRE(nnz == 0 || (ho_item && rank_out), "null ho_item or rank_out");
    const std::string err = pcrhost::csr_error("held-out", d1, d2, ho_row_ptr, ho_item, false);
    PCR_REQUIRE(err.empty(), err);
    const int64_t ex_nnz = check_exclusion(d1, d2, excl_row_ptr, excl_item);
    if (nnz == 0) return PRIMALCR_OK;
    // units: a user and at most RANK_UNIT consecutive entries of its row; they tile [0, nnz) in order
    std::vector<int32_t> unit_user;
    std::vector<pcr::i64> unit_beg;
    for (int64_t u = 0; u < d1; ++u)
        for (int64_t e = ho_row_ptr[u]; e < ho_row_ptr[u + 1]; e += pcr::RANK_UNIT) { unit_user.push_back((int32_t)u); unit_beg.push_back(e); }
    unit_beg.push_back(nnz);
    const int64_t n_units = (int64_t)unit_user.size();
    Session s(device);
    const double *Ud = s.upload(U, (size_t)d1 * k), *Vd = s.upload(V, (size_t)d2 * k);
    const int32_t *hid = s.upload(ho_item, (size_t)nnz), *uud = s.upload(unit_user.data(), (size_t)n_units);
    const pcr::i64 *ubd = s.upload(unit_beg.data(), (size_t)n_units + 1);
    const pcr::i64 *exp_d = excl_row_ptr ? s.upload((const pcr::i64 *)excl_row_ptr, (size_t)d1 + 1) : nullptr;
    const int32_t *exi_d = excl_row_ptr ? s.upload(excl_item, (size_t)ex_nnz) : nullptr;
    int32_t *rkd = s.pool.alloc<int32_t>((size_t)nnz);
    double *scd = score_out ? s.pool.alloc<double>((size_t)nnz) : nullptr;
    pcr::k_rank_heldout(s.ctx, Ud, Vd, d2, k, exp_d, exi_d, hid, uud, ubd, n_units, rkd, scd);
    s.download(rank_out, rkd, (size_t)nnz);
    if (score_out) s.download(score_out, scd, (size_t)nnz);
    s.sync();
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

}  // extern "C"
