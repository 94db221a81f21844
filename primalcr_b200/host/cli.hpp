// cli.hpp -- what the query CLIs (primalcr-recommend, primalcr-similar, primalcr-rankeval) share.  Each helper prints its
// error to stderr and returns false; the caller then exits with status 1.
#pragma once
#include "loader.hpp"

#include <cstdio>
#include <vector>

namespace pcrhost {

// one 1-based id per line of the file at path, each in [1, n] -> 0-based ids; `what` names an id in the messages
inline bool read_ids(const char *path, long n, const char *what, std::vector<int32_t> &ids) {
    FILE *fp = fopen(path, "r");
    if (!fp) { fprintf(stderr, "can't open %ss file %s\n", what, path); return false; }
    long v;
    while (fscanf(fp, "%ld", &v) == 1) {
        if (v < 1 || v > n) { fprintf(stderr, "%s %ld out of range [1, %ld]\n", what, v, n); fclose(fp); return false; }
        ids.push_back((int32_t)(v - 1));
    }
    fclose(fp);
    return true;
}

// the data directory at path, whose ratings must be d1 x d2 like the model
inline bool load_model_dir(const char *path, long d1, long d2, DataDir &data) {
    try { data = load_dir(path); }
    catch (const std::exception &ex) { fprintf(stderr, "can't load %s: %s\n", path, ex.what()); return false; }
    if (data.train.d1 != d1 || data.train.d2 != d2) {
        fprintf(stderr, "%s is %lld x %lld, the model is %ld x %ld\n", path, (long long)data.train.d1,
                (long long)data.train.d2, d1, d2);
        return false;
    }
    return true;
}

// the n_rows x topn result of a top-N call as "row id score" lines: 1-based ids, "%.17g" scores (the doubles round-trip);
// row q is rows[q] (rows NULL: q), and a row's padding (id -1) is not written
inline bool write_topn(const char *path, const int32_t *rows, int64_t n_rows, int topn, const std::vector<int32_t> &ids,
                       const std::vector<double> &scores) {
    FILE *out = fopen(path, "wb");
    if (!out) { fprintf(stderr, "can't open output file %s\n", path); return false; }
    for (int64_t q = 0; q < n_rows; ++q) {
        const long r = rows ? (long)rows[q] + 1 : (long)q + 1;
        for (int j = 0; j < topn; ++j) {
            const size_t t = (size_t)q * topn + j;
            if (ids[t] < 0) break;
            fprintf(out, "%ld %d %.17g\n", r, ids[t] + 1, scores[t]);
        }
    }
    fclose(out);
    return true;
}

}  // namespace pcrhost
