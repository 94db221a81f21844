// primalcr-recommend -- top-N items per user from a trained model, on the GPU through the C ABI (primalcr_recommend):
//     primalcr-recommend [-n topN (default 10)] [-e data_dir] [-u users_file] [-d device] model output_file
// -e: exclude the training ratings of data_dir (the reference's meta + ratings layout); its d1 / d2 must match the model.
// -u: one 1-based user id per line (default: every user).
// Writes one "user item score" line per recommendation: 1-based ids, "%.17g" scores (the doubles round-trip), users in
// request order, best first; padding entries (fewer eligible items than topN) are not written.
#include "../host/cli.hpp"
#include "../host/model.hpp"
#include "primalcr.h"

#include <cstdio>
#include <cstdlib>
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
    if (data_dir && !pcrhost::load_model_dir(data_dir, d1, d2, data)) return 1;
    std::vector<int32_t> users;
    if (users_file && !pcrhost::read_ids(users_file, d1, "user", users)) return 1;
    const int64_t n_users = users_file ? (int64_t)users.size() : (int64_t)d1;

    std::vector<int32_t> items((size_t)n_users * (topn > 0 ? topn : 0));
    std::vector<double> scores(items.size());
    const int rc = primalcr_recommend(W.data(), d1, H.data(), d2, (int)k,
                                      data_dir ? data.train.row_ptr.data() : nullptr,
                                      data_dir ? data.train.item.data() : nullptr,
                                      users_file ? users.data() : nullptr, n_users, topn, items.data(), scores.data(), device);
    if (rc != 0) { fprintf(stderr, "primalcr_recommend failed (%d): %s\n", rc, primalcr_last_error()); return 1; }

    if (!pcrhost::write_topn(out_path, users_file ? users.data() : nullptr, n_users, topn, items, scores)) return 1;
    return 0;
}
