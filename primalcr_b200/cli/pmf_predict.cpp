// primalcr-predict -- same command line and output as omp-pmf-predict (pmf-predict.cpp:6-67):
//     primalcr-predict test_file model output_file
// prints one "%lf" per test line: U[i-1] . V[j-1].  The dot products are evaluated on the GPU in one batch through
// the C ABI (primalcr_predict); the model layout is the reference's (load_mat_t util.cpp:56-79).
#include "../host/loader.hpp"
#include "../host/model.hpp"
#include "primalcr.h"

#include <cstdio>
#include <vector>

int main(int argc, char **argv) {
    if (argc != 4) { printf("Usage: primalcr-predict test_file model output_file\n"); return 1; }
    FILE *model_fp = fopen(argv[2], "rb");
    if (!model_fp) { fprintf(stderr, "can't open model file %s\n", argv[2]); return 1; }
    FILE *out = fopen(argv[3], "wb");
    if (!out) { fprintf(stderr, "can't open output file %s\n", argv[3]); return 1; }
    std::vector<double> W, H;
    long d1 = 0, k = 0, d2 = 0, k2 = 0;
    if (!pcrhost::read_matrix(model_fp, W, d1, k) || !pcrhost::read_matrix(model_fp, H, d2, k2) || k != k2) { fprintf(stderr, "bad model file %s\n", argv[2]); return 1; }
    fclose(model_fp);
    pcrhost::Triples t;
    try { t = pcrhost::parse_file(argv[1], -1); }
    catch (const std::exception &ex) { fprintf(stderr, "can't open test file %s\n", argv[1]); return 1; }
    std::vector<double> pred(t.u.size());
    const int rc = primalcr_predict(W.data(), d1, H.data(), d2, (int)k, t.u.data(), t.i.data(), (int64_t)t.u.size(), pred.data(), 0);
    if (rc != 0) { fprintf(stderr, "primalcr_predict failed (%d): %s\n", rc, primalcr_last_error()); return 1; }
    for (double v : pred) fprintf(out, "%lf\n", v);
    fclose(out);
    return 0;
}
