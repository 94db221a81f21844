// primalcr-rankeval -- whole-catalog ranking metrics of a trained model on a data directory's test set, through the C ABI
// (primalcr_rank_heldout on the GPU, then primalcr_rank_metrics on the host):
//     primalcr-rankeval [-n cutoffs (default 10, comma-separated)] [-r min_rating] [-d device] data_dir model
// The training ratings of data_dir are excluded from every user's candidates and its test ratings are the held-out set;
// test ratings >= min_rating are relevant (default: all).  Prints one "name value" line per metric ("%.17g"):
// recall@N, precision@N and ndcg@N per cutoff, then mrr, auc and n_users (the number of evaluated users).
#include "../host/cli.hpp"
#include "../host/model.hpp"
#include "primalcr.h"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <vector>

static void usage() {
    printf("Usage: primalcr-rankeval [-n cutoffs (default 10, e.g. 5,10,20)] [-r min_rating] [-d device] data_dir model\n");
}

int main(int argc, char **argv) {
    std::vector<int32_t> cutoffs;
    double min_rating = -INFINITY;
    int device = 0;
    int i = 1;
    for (; i < argc && argv[i][0] == '-'; i += 2) {
        if (i + 1 >= argc) { usage(); return 1; }
        switch (argv[i][1]) {
            case 'n': {
                cutoffs.clear();
                for (const char *p = argv[i + 1]; *p;) {
                    char *end;
                    const long n = strtol(p, &end, 10);
                    if (end == p || n < 1 || n > INT32_MAX || (*end && *end != ',')) {
                        fprintf(stderr, "bad cutoff list: %s\n", argv[i + 1]); return 1;
                    }
                    cutoffs.push_back((int32_t)n);
                    p = *end ? end + 1 : end;
                }
                break;
            }
            case 'r': min_rating = atof(argv[i + 1]); break;
            case 'd': device = atoi(argv[i + 1]); break;
            default: fprintf(stderr, "unknown option: -%c\n", argv[i][1]); usage(); return 1;
        }
    }
    if (argc - i != 2) { usage(); return 1; }
    const char *data_dir = argv[i], *model_path = argv[i + 1];
    if (cutoffs.empty()) cutoffs.push_back(10);

    std::vector<double> W, H;
    long d1 = 0, k = 0, d2 = 0;
    if (!pcrhost::read_model(model_path, W, d1, H, d2, k)) { fprintf(stderr, "can't read model file %s\n", model_path); return 1; }
    pcrhost::DataDir data;
    if (!pcrhost::load_model_dir(data_dir, d1, d2, data)) return 1;
    if (!data.has_test) { fprintf(stderr, "%s has no test set to evaluate\n", data_dir); return 1; }

    const pcrhost::Csr &X = data.train, &T = data.test;
    std::vector<int32_t> rank((size_t)T.row_ptr[d1]);
    int rc = primalcr_rank_heldout(W.data(), d1, H.data(), d2, (int)k, X.row_ptr.data(), X.item.data(), T.row_ptr.data(),
                                   T.item.data(), rank.data(), nullptr, device);
    if (rc != 0) { fprintf(stderr, "primalcr_rank_heldout failed (%d): %s\n", rc, primalcr_last_error()); return 1; }
    const int nc = (int)cutoffs.size();
    std::vector<double> recall(nc), precision(nc), ndcg(nc);
    double mrr = 0.0, auc = 0.0;
    int64_t n_users = 0;
    rc = primalcr_rank_metrics(d1, d2, X.row_ptr.data(), X.item.data(), T.row_ptr.data(), T.item.data(), T.rating.data(),
                               rank.data(), min_rating, cutoffs.data(), nc, recall.data(), precision.data(), ndcg.data(),
                               &mrr, &auc, &n_users);
    if (rc != 0) { fprintf(stderr, "primalcr_rank_metrics failed (%d): %s\n", rc, primalcr_last_error()); return 1; }
    for (int c = 0; c < nc; ++c) {
        printf("recall@%d %.17g\n", cutoffs[c], recall[c]);
        printf("precision@%d %.17g\n", cutoffs[c], precision[c]);
        printf("ndcg@%d %.17g\n", cutoffs[c], ndcg[c]);
    }
    printf("mrr %.17g\nauc %.17g\nn_users %lld\n", mrr, auc, (long long)n_users);
    return 0;
}
