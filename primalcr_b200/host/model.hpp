// model.hpp -- the model file primalcr-train writes (save_mat_t util.cpp:30-51): U then V, each as a long row count, a
// long column count and the row-major doubles.
#pragma once
#include <cstdio>
#include <vector>

namespace pcrhost {

// one matrix of the model file (load_mat_t util.cpp:56-79); false on a short read or a bad shape
inline bool read_matrix(FILE *fp, std::vector<double> &M, long &rows, long &k) {
    if (fread(&rows, sizeof(long), 1, fp) != 1 || fread(&k, sizeof(long), 1, fp) != 1) return false;
    if (rows < 0 || k < 1) return false;
    M.resize((size_t)rows * k);
    return fread(M.data(), sizeof(double), (size_t)rows * k, fp) == (size_t)rows * k;
}

// U (d1 x k) and V (d2 x k) from the file at path; false when it cannot be opened or read, or the two k differ
inline bool read_model(const char *path, std::vector<double> &U, long &d1, std::vector<double> &V, long &d2, long &k) {
    FILE *fp = fopen(path, "rb");
    if (!fp) return false;
    long k2 = 0;
    const bool ok = read_matrix(fp, U, d1, k) && read_matrix(fp, V, d2, k2) && k == k2;
    fclose(fp);
    return ok;
}

}  // namespace pcrhost
