// primalcr-similar -- the most similar items (or users) of a trained model, on the GPU through the C ABI (primalcr_similar):
//     primalcr-similar [-s items|users] [-m cosine|dot] [-n topN (default 10)] [-q ids_file] [-d device] model output_file
// -s: rank the rows of V (items, the default) or of U (users) against each other.
// -m: cosine (the default) or dot product of the factor rows.
// -q: one 1-based item / user id per line (default: every one).
// Writes one "query neighbour score" line per neighbour: 1-based ids, "%.17g" scores (the doubles round-trip), queries in
// request order, best first; a query is never its own neighbour, and padding entries (fewer than topN rows) are not written.
#include "../host/cli.hpp"
#include "../host/model.hpp"
#include "primalcr.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

static void usage() {
    printf("Usage: primalcr-similar [-s items|users] [-m cosine|dot] [-n topN (default 10)] [-q ids_file] [-d device] "
           "model output_file\n");
}

int main(int argc, char **argv) {
    int topn = 10, device = 0, measure = PRIMALCR_SIM_COSINE;
    bool users_side = false;
    const char *ids_file = nullptr;
    int i = 1;
    for (; i < argc && argv[i][0] == '-'; i += 2) {
        if (i + 1 >= argc) { usage(); return 1; }
        const char *v = argv[i + 1];
        switch (argv[i][1]) {
            case 's':
                if (!strcmp(v, "items")) users_side = false;
                else if (!strcmp(v, "users")) users_side = true;
                else { fprintf(stderr, "-s takes items or users, got %s\n", v); usage(); return 1; }
                break;
            case 'm':
                if (!strcmp(v, "cosine")) measure = PRIMALCR_SIM_COSINE;
                else if (!strcmp(v, "dot")) measure = PRIMALCR_SIM_DOT;
                else { fprintf(stderr, "-m takes cosine or dot, got %s\n", v); usage(); return 1; }
                break;
            case 'n': topn = atoi(v); break;
            case 'q': ids_file = v; break;
            case 'd': device = atoi(v); break;
            default: fprintf(stderr, "unknown option: -%c\n", argv[i][1]); usage(); return 1;
        }
    }
    if (argc - i != 2) { usage(); return 1; }
    const char *model_path = argv[i], *out_path = argv[i + 1];

    std::vector<double> W, H;
    long d1 = 0, k = 0, d2 = 0;
    if (!pcrhost::read_model(model_path, W, d1, H, d2, k)) { fprintf(stderr, "can't read model file %s\n", model_path); return 1; }
    const std::vector<double> &M = users_side ? W : H;
    const long n = users_side ? d1 : d2;

    std::vector<int32_t> queries;
    if (ids_file && !pcrhost::read_ids(ids_file, n, "id", queries)) return 1;
    const int64_t n_queries = ids_file ? (int64_t)queries.size() : (int64_t)n;

    std::vector<int32_t> ids((size_t)n_queries * (topn > 0 ? topn : 0));
    std::vector<double> scores(ids.size());
    const int rc = primalcr_similar(M.data(), n, (int)k, measure, nullptr, nullptr, ids_file ? queries.data() : nullptr,
                                    n_queries, topn, ids.data(), scores.data(), device);
    if (rc != 0) { fprintf(stderr, "primalcr_similar failed (%d): %s\n", rc, primalcr_last_error()); return 1; }

    if (!pcrhost::write_topn(out_path, ids_file ? queries.data() : nullptr, n_queries, topn, ids, scores)) return 1;
    return 0;
}
