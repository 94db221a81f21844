// rankmetrics.hpp -- top-N ranking metrics from the catalog ranks of held-out entries (primalcr_rank_heldout), on the
// host.  This is the one implementation behind primalcr_rank_metrics, so the C ABI, the Python API and primalcr-rankeval
// report the same numbers.  The definitions are in include/primalcr.h.
#pragma once
#include "loader.hpp"

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <limits>
#include <string>
#include <utility>
#include <vector>

namespace pcrhost {

struct RankMetrics {
    std::vector<double> recall, precision, ndcg;    // [n_cutoffs]
    double mrr = 0.0, auc = 0.0;
    int64_t n_users = 0;
};

// Returns "" and fills `out`, or what is wrong with the arguments.  excl_row_ptr / excl_item may both be NULL (nothing
// excluded); ho_item, ho_rating and rank may be NULL only when there are no held-out entries.
inline std::string rank_metrics(int64_t d1, int64_t d2, const int64_t *excl_row_ptr, const int32_t *excl_item,
                                const int64_t *ho_row_ptr, const int32_t *ho_item, const double *ho_rating,
                                const int32_t *rank, double min_rating, const int32_t *cutoffs, int n_cutoffs,
                                RankMetrics &out) {
    if (d1 < 0 || d2 < 0 || d1 > INT32_MAX || d2 > INT32_MAX) return "d1 / d2 out of range";
    if (n_cutoffs < 0 || (n_cutoffs > 0 && !cutoffs)) return "bad cutoffs";
    for (int c = 0; c < n_cutoffs; ++c)
        if (cutoffs[c] < 1) return "cutoffs must be >= 1";
    if (std::isnan(min_rating)) return "min_rating is NaN";
    if ((excl_row_ptr == nullptr) != (excl_item == nullptr)) return "excl_row_ptr and excl_item must both be given or both be NULL";
    if (!ho_row_ptr) return "null ho_row_ptr";
    std::string err;
    if (excl_row_ptr && !(err = csr_error("exclusion", d1, d2, excl_row_ptr, excl_item, true)).empty()) return err;
    const int64_t nnz = ho_row_ptr[d1];
    if (nnz > 0 && (!ho_item || !ho_rating || !rank)) return "null ho_item, ho_rating or rank";
    if (!(err = csr_error("held-out", d1, d2, ho_row_ptr, ho_item, false)).empty()) return err;
    bool bad_rank = false;
#pragma omp parallel for reduction(|| : bad_rank) schedule(static)
    for (int64_t e = 0; e < nnz; ++e) bad_rank = bad_rank || rank[e] < 0 || rank[e] > d2;
    if (bad_rank) return "rank out of range [0, d2]";

    // per user: recall / precision / ndcg at every cutoff, then mrr, auc; NaN marks "not evaluated"
    const int nc = n_cutoffs, W = 3 * nc + 2;
    std::vector<double> per((size_t)d1 * W);
    std::vector<char> evaluated((size_t)d1, 0), has_auc((size_t)d1, 0);
#pragma omp parallel
    {
        std::vector<std::pair<int32_t, int64_t>> ent;     // (item, entry) of the user's ranked entries
        std::vector<int64_t> rel;                         // ranks of the relevant items, ascending
#pragma omp for schedule(dynamic, 1024)
        for (int64_t u = 0; u < d1; ++u) {
            ent.clear(); rel.clear();
            for (int64_t e = ho_row_ptr[u]; e < ho_row_ptr[u + 1]; ++e)
                if (rank[e] > 0) ent.emplace_back(ho_item[e], e);
            std::sort(ent.begin(), ent.end());
            for (size_t a = 0; a < ent.size();) {         // one distinct item: its largest rating, its smallest rank
                size_t b = a;
                double rt = -std::numeric_limits<double>::infinity();
                int64_t rk = INT64_MAX;
                for (; b < ent.size() && ent[b].first == ent[a].first; ++b) {
                    rt = std::max(rt, ho_rating[ent[b].second]);
                    rk = std::min(rk, (int64_t)rank[ent[b].second]);
                }
                if (rt >= min_rating) rel.push_back(rk);
                a = b;
            }
            if (rel.empty()) continue;
            std::sort(rel.begin(), rel.end());
            const int64_t nr = (int64_t)rel.size();
            double *o = per.data() + (size_t)u * W;
            for (int c = 0; c < nc; ++c) {
                const int64_t N = cutoffs[c];
                const int64_t hits = std::upper_bound(rel.begin(), rel.end(), N) - rel.begin();
                double dcg = 0.0, idcg = 0.0;
                for (int64_t q = 0; q < hits; ++q) dcg += 1.0 / std::log2((double)rel[q] + 1.0);
                for (int64_t p = 1; p <= std::min(N, nr); ++p) idcg += 1.0 / std::log2((double)p + 1.0);
                o[c] = (double)hits / (double)nr;
                o[nc + c] = (double)hits / (double)N;
                o[2 * nc + c] = dcg / idcg;
            }
            o[3 * nc] = 1.0 / (double)rel[0];
            int64_t cand = d2;                             // C_u: d2 minus the distinct items of the exclusion row
            if (excl_row_ptr)
                for (int64_t e = excl_row_ptr[u]; e < excl_row_ptr[u + 1]; ++e)
                    cand -= (e == excl_row_ptr[u] || excl_item[e] != excl_item[e - 1]);
            const int64_t nn = cand - nr;
            if (nn > 0) {
                double s = 0.0;
                for (int64_t q = 0; q < nr; ++q) {
                    const int64_t pos = std::lower_bound(rel.begin(), rel.end(), rel[q]) - rel.begin();
                    s += (double)(nn - (rel[q] - 1 - pos));
                }
                o[3 * nc + 1] = s / ((double)nr * (double)nn);
                has_auc[(size_t)u] = 1;
            }
            evaluated[(size_t)u] = 1;
        }
    }
    // plain means over users, summed in ascending user order
    std::vector<double> sum((size_t)W, 0.0);
    int64_t n = 0, n_auc = 0;
    for (int64_t u = 0; u < d1; ++u) {
        if (!evaluated[(size_t)u]) continue;
        const double *o = per.data() + (size_t)u * W;
        for (int j = 0; j <= 3 * nc; ++j) sum[(size_t)j] += o[j];
        ++n;
        if (has_auc[(size_t)u]) { sum[(size_t)3 * nc + 1] += o[3 * nc + 1]; ++n_auc; }
    }
    const double nan = std::numeric_limits<double>::quiet_NaN();
    out.recall.assign((size_t)nc, nan); out.precision.assign((size_t)nc, nan); out.ndcg.assign((size_t)nc, nan);
    for (int c = 0; c < nc && n > 0; ++c) {
        out.recall[(size_t)c] = sum[(size_t)c] / (double)n;
        out.precision[(size_t)c] = sum[(size_t)nc + c] / (double)n;
        out.ndcg[(size_t)c] = sum[(size_t)2 * nc + c] / (double)n;
    }
    out.mrr = n > 0 ? sum[(size_t)3 * nc] / (double)n : nan;
    out.auc = n_auc > 0 ? sum[(size_t)3 * nc + 1] / (double)n_auc : nan;
    out.n_users = n;
    return "";
}

}  // namespace pcrhost
