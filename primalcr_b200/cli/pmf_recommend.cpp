// primalcr-recommend -- top-N items per user from a trained model, on the GPU through the C ABI (primalcr_recommend):
//     primalcr-recommend [-n topN (default 10)] [-e data_dir] [-u users_file] [-d device] model output_file
// -e: exclude the training ratings of data_dir (the reference's meta + ratings layout); its d1 / d2 must match the model.
// -u: one 1-based user id per line (default: every user).
// Writes one "user item score" line per recommendation: 1-based ids, "%.17g" scores (the doubles round-trip), users in
// request order, best first; padding entries (fewer eligible items than topN) are not written.
#include "../host/loader.hpp"
#include "../host/model.hpp"
#include "primalcr.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

static void usage() {
    printf("Usage: primalcr-recommend [-n topN (default 10)] [-e data_dir] [-u users_file] [-d device] model output_file\n");
}

int main(int argc, char **argv) {
    int topn = 10, device = 0;
    const char *data_dir = nullptr, *users_file = nullptr;
    int i = 1;
    for (; i < argc && argv[i][0] == '-'; i += 2) {
        if (i + 1 >= argc) { usage(); return 1; }
        switch (argv[i][1]) {
            case 'n': topn = atoi(argv[i + 1]); break;
            case 'e': data_dir = argv[i + 1]; break;
            case 'u': users_file = argv[i + 1]; break;
            case 'd': device = atoi(argv[i + 1]); break;
            default: fprintf(stderr, "unknown option: -%c\n", argv[i][1]); usage(); return 1;
        }
    }
    if (argc - i != 2) { usage(); return 1; }
    const char *model_path = argv[i], *out_path = argv[i + 1];

    std::vector<double> W, H;
    long d1 = 0, k = 0, d2 = 0;
    if (!pcrhost::read_model(model_path, W, d1, H, d2, k)) { fprintf(stderr, "can't read model file %s\n", model_path); return 1; }

    pcrhost::DataDir data;
    if (data_dir) {
        try { data = pcrhost::load_dir(data_dir); }
        catch (const std::exception &ex) { fprintf(stderr, "can't load %s: %s\n", data_dir, ex.what()); return 1; }
        if (data.train.d1 != d1 || data.train.d2 != d2) {
            fprintf(stderr, "%s is %lld x %lld, the model is %ld x %ld\n", data_dir, (long long)data.train.d1,
                    (long long)data.train.d2, d1, d2);
            return 1;
        }
    }

    std::vector<int32_t> users;
    if (users_file) {
        FILE *fp = fopen(users_file, "r");
        if (!fp) { fprintf(stderr, "can't open users file %s\n", users_file); return 1; }
        long u;
        while (fscanf(fp, "%ld", &u) == 1) {
            if (u < 1 || u > d1) { fprintf(stderr, "user %ld out of range [1, %ld]\n", u, d1); fclose(fp); return 1; }
            users.push_back((int32_t)(u - 1));
        }
        fclose(fp);
    }
    const int64_t n_users = users_file ? (int64_t)users.size() : (int64_t)d1;

    std::vector<int32_t> items((size_t)n_users * (topn > 0 ? topn : 0));
    std::vector<double> scores(items.size());
    const int rc = primalcr_recommend(W.data(), d1, H.data(), d2, (int)k,
                                      data_dir ? data.train.row_ptr.data() : nullptr,
                                      data_dir ? data.train.item.data() : nullptr,
                                      users_file ? users.data() : nullptr, n_users, topn, items.data(), scores.data(), device);
    if (rc != 0) { fprintf(stderr, "primalcr_recommend failed (%d): %s\n", rc, primalcr_last_error()); return 1; }

    FILE *out = fopen(out_path, "wb");
    if (!out) { fprintf(stderr, "can't open output file %s\n", out_path); return 1; }
    for (int64_t q = 0; q < n_users; ++q) {
        const long u = users_file ? (long)users[q] + 1 : (long)q + 1;
        for (int j = 0; j < topn; ++j) {
            const size_t t = (size_t)q * topn + j;
            if (items[t] < 0) break;
            fprintf(out, "%ld %d %.17g\n", u, items[t] + 1, scores[t]);
        }
    }
    fclose(out);
    return 0;
}
