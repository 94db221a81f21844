// loader.hpp -- fast host loader for the reference's data directory format (replaces the serial fgets+sscanf+std::sort
// of load() util.cpp:6-25 / smat_t::load_from_iterator util.h:201-271 / testset_t::load util.h:360-371).
//
//   data_dir/meta : "m n" / "nnz_train train_file" / optional "nnz_test test_file"        (util.cpp:9-21)
//   ratings files : "user item rating" per line, 1-based ids                               (util.h:126, 367)
//
// The file is mmap'ed, split at line boundaries into one chunk per thread and parsed with hand-rolled integer / strtod
// scanners; training entries are bucketed by user (counting sort) and ordered by item inside a user, which is the order
// smat_t's `sort(perm, SparseComp)` (util.h:240) produces; the test set keeps file order inside a user and must be
// grouped by user like convert(testset_t&) requires (util.cpp:257-266).
#pragma once
#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <stdexcept>
#include <string>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

namespace pcrhost {

struct Csr {
    int64_t d1 = 0, d2 = 0, nnz = 0;
    std::vector<int64_t> row_ptr;
    std::vector<int32_t> item;
    std::vector<double> rating;
};

struct Triples { std::vector<int32_t> u, i; std::vector<double> r; };

// Checks a caller's d1-row CSR over items [0, d2) (row_ptr: d1+1 entries; ascending: the items of a row must not
// decrease, repeats allowed).  item == NULL checks the row pointers only.  Returns "" when it is well formed, else what is
// wrong, prefixed with `what`.
inline std::string csr_error(const char *what, int64_t d1, int64_t d2, const int64_t *row_ptr, const int32_t *item,
                             bool ascending) {
    if (row_ptr[0] != 0) return std::string(what) + ": row_ptr[0] must be 0";
    bool bad_ptr = false, bad_item = false, descending = false;
#pragma omp parallel for reduction(|| : bad_ptr, bad_item, descending) schedule(dynamic, 4096)
    for (int64_t u = 0; u < d1; ++u) {
        const int64_t a = row_ptr[u], b = row_ptr[u + 1];
        if (b < a) { bad_ptr = true; continue; }
        if (!item) continue;
        for (int64_t e = a; e < b; ++e) {
            if (item[e] < 0 || item[e] >= d2) { bad_item = true; break; }
            if (ascending && e > a && item[e] < item[e - 1]) { descending = true; break; }
        }
    }
    if (bad_ptr) return std::string(what) + ": row_ptr decreases";
    if (bad_item) return std::string(what) + ": item id out of range";
    if (descending) return std::string(what) + ": row items must ascend";
    return "";
}

inline void parse_chunk(const char *p, const char *end, Triples &out) {
    while (p < end) {
        while (p < end && (*p == ' ' || *p == '\t' || *p == '\r' || *p == '\n')) ++p;
        if (p >= end) break;
        long a = 0, b = 0;
        bool neg = false;
        if (*p == '-') { neg = true; ++p; }
        while (p < end && *p >= '0' && *p <= '9') a = a * 10 + (*p++ - '0');
        if (neg) a = -a;
        while (p < end && (*p == ' ' || *p == '\t')) ++p;
        neg = false;
        if (p < end && *p == '-') { neg = true; ++p; }
        while (p < end && *p >= '0' && *p <= '9') b = b * 10 + (*p++ - '0');
        if (neg) b = -b;
        while (p < end && (*p == ' ' || *p == '\t')) ++p;
        // rating: plain decimals "[-]ddd[.ddd]" with <= 15 significant digits are converted exactly (integer mantissa
        // divided by an exactly representable power of ten = the correctly rounded value, i.e. what strtod / sscanf
        // "%lf" return); anything else (exponents, inf, nan, long mantissas) goes through strtod
        const char *q = p;
        bool rneg = false;
        if (q < end && (*q == '-' || *q == '+')) { rneg = *q == '-'; ++q; }
        unsigned long long mant = 0; int nd = 0, frac = 0;
        while (q < end && *q >= '0' && *q <= '9') { mant = mant * 10 + (unsigned)(*q++ - '0'); ++nd; }
        if (q < end && *q == '.') { ++q; while (q < end && *q >= '0' && *q <= '9') { mant = mant * 10 + (unsigned)(*q++ - '0'); ++nd; ++frac; } }
        const bool at_end = q >= end || *q == '\n' || *q == '\r' || *q == ' ' || *q == '\t';
        double v;
        if (nd > 0 && nd <= 15 && at_end) {
            static const double p10[16] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15};
            v = (double)mant / p10[frac];
            if (rneg) v = -v;
            while (q < end && *q != '\n') ++q;
        } else {
            q = p;
            while (q < end && *q != '\n') ++q;
            char buf[64];
            size_t len = (size_t)(q - p);
            if (len > 63) len = 63;
            memcpy(buf, p, len); buf[len] = 0;
            v = strtod(buf, nullptr);
        }
        out.u.push_back((int32_t)(a - 1)); out.i.push_back((int32_t)(b - 1)); out.r.push_back(v);
        p = q;
    }
}

// parses at most `limit` entries (the reference reads exactly the count given in meta); the result stays split into the
// per-thread parts, in file order
inline std::vector<Triples> parse_file_parts(const std::string &path, int64_t limit) {
    int fd = open(path.c_str(), O_RDONLY);
    if (fd < 0) throw std::runtime_error("cannot open " + path);
    struct stat st; fstat(fd, &st);
    const size_t size = (size_t)st.st_size;
    std::vector<Triples> part;
    if (size == 0) { close(fd); return part; }
    const char *base = (const char *)mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (base == MAP_FAILED) { close(fd); throw std::runtime_error("mmap failed for " + path); }
    int nt = 1;
#ifdef _OPENMP
    nt = omp_get_max_threads();
#endif
    if ((size_t)nt > size / 65536 + 1) nt = (int)(size / 65536 + 1);
    std::vector<size_t> cut(nt + 1, size);
    cut[0] = 0;
    for (int t = 1; t < nt; ++t) {
        size_t c = size / nt * t;
        while (c < size && base[c] != '\n') ++c;
        cut[t] = c < size ? c + 1 : size;
    }
    part.resize(nt);
#pragma omp parallel for schedule(static, 1)
    for (int t = 0; t < nt; ++t) {
        const size_t guess = (cut[t + 1] - cut[t]) / 12 + 16;
        part[t].u.reserve(guess); part[t].i.reserve(guess); part[t].r.reserve(guess);
        parse_chunk(base + cut[t], base + cut[t + 1], part[t]);
    }
    munmap((void *)base, size); close(fd);
    if (limit >= 0) {                       // keep the first `limit` entries of the file
        int64_t left = limit;
        for (auto &p : part) {
            const int64_t n = std::min<int64_t>((int64_t)p.u.size(), left);
            p.u.resize((size_t)n); p.i.resize((size_t)n); p.r.resize((size_t)n);
            left -= n;
        }
    }
    return part;
}

inline Triples concat_parts(const std::vector<Triples> &part) {
    Triples all;
    size_t total = 0;
    for (auto &p : part) total += p.u.size();
    all.u.resize(total); all.i.resize(total); all.r.resize(total);
    std::vector<size_t> off(part.size() + 1, 0);
    for (size_t t = 0; t < part.size(); ++t) off[t + 1] = off[t] + part[t].u.size();
#pragma omp parallel for schedule(static, 1)
    for (int64_t t = 0; t < (int64_t)part.size(); ++t) {
        std::copy(part[t].u.begin(), part[t].u.end(), all.u.begin() + off[t]);
        std::copy(part[t].i.begin(), part[t].i.end(), all.i.begin() + off[t]);
        std::copy(part[t].r.begin(), part[t].r.end(), all.r.begin() + off[t]);
    }
    return all;
}

inline Triples parse_file(const std::string &path, int64_t limit) { return concat_parts(parse_file_parts(path, limit)); }

// CSR sorted by (user, item): the order of smat_t::load_from_iterator util.h:240-247.  Parallel two-pass counting sort
// straight from the parsed parts: per-part user histograms -> offsets (file order is kept inside a user, so duplicates
// stay in file order like the reference's stable handling) -> every part scatters into its own slots.
inline Csr build_train_csr(int64_t d1, int64_t d2, const std::vector<Triples> &part) {
    Csr X; X.d1 = d1; X.d2 = d2;
    const int64_t np = (int64_t)part.size();
    X.nnz = 0;
    for (auto &p : part) X.nnz += (int64_t)p.u.size();
    X.row_ptr.assign(d1 + 1, 0);
    X.item.resize(X.nnz); X.rating.resize(X.nnz);
    if (np == 0) return X;
    std::vector<std::vector<int64_t>> off((size_t)np, std::vector<int64_t>());
    std::atomic<bool> bad(false);
#pragma omp parallel for schedule(static, 1)
    for (int64_t t = 0; t < np; ++t) {
        off[t].assign((size_t)d1, 0);
        const Triples &p = part[t];
        for (size_t e = 0; e < p.u.size(); ++e) {
            if (p.u[e] < 0 || p.u[e] >= d1 || p.i[e] < 0 || p.i[e] >= d2) { bad.store(true); break; }
            off[t][p.u[e]]++;
        }
    }
    if (bad.load()) throw std::runtime_error("rating id out of range");
#pragma omp parallel for schedule(static, 4096)
    for (int64_t u = 0; u < d1; ++u) {
        int64_t c = 0;
        for (int64_t t = 0; t < np; ++t) c += off[t][u];
        X.row_ptr[u + 1] = c;
    }
    for (int64_t u = 0; u < d1; ++u) X.row_ptr[u + 1] += X.row_ptr[u];
#pragma omp parallel for schedule(static, 4096)
    for (int64_t u = 0; u < d1; ++u) {
        int64_t run = X.row_ptr[u];
        for (int64_t t = 0; t < np; ++t) { const int64_t c = off[t][u]; off[t][u] = run; run += c; }
    }
#pragma omp parallel for schedule(static, 1)
    for (int64_t t = 0; t < np; ++t) {
        const Triples &p = part[t];
        std::vector<int64_t> &o = off[t];
        for (size_t e = 0; e < p.u.size(); ++e) { const int64_t q = o[p.u[e]]++; X.item[q] = p.i[e]; X.rating[q] = p.r[e]; }
    }
#pragma omp parallel for schedule(dynamic, 256)
    for (int64_t u = 0; u < d1; ++u) {
        const int64_t a = X.row_ptr[u], b = X.row_ptr[u + 1];
        bool sorted = true;
        for (int64_t e = a + 1; e < b; ++e) if (X.item[e] < X.item[e - 1]) { sorted = false; break; }
        if (sorted) continue;
        std::vector<std::pair<int32_t, double>> tmp((size_t)(b - a));
        for (int64_t e = a; e < b; ++e) tmp[e - a] = std::make_pair(X.item[e], X.rating[e]);
        std::stable_sort(tmp.begin(), tmp.end(), [](const std::pair<int32_t, double> &x, const std::pair<int32_t, double> &y) { return x.first < y.first; });
        for (int64_t e = a; e < b; ++e) { X.item[e] = tmp[e - a].first; X.rating[e] = tmp[e - a].second; }
    }
    return X;
}
inline Csr build_train_csr(int64_t d1, int64_t d2, const Triples &t) {
    std::vector<Triples> one(1, t);
    return build_train_csr(d1, d2, one);
}

// convert(testset_t&, d1, d2) util.cpp:250-274, literally: file order, entries lumped while T[cc].i <= j
inline Csr build_test_csr(int64_t d1, int64_t d2, const Triples &t) {
    Csr X; X.d1 = d1; X.d2 = d2;
    const int64_t nnz = (int64_t)t.u.size();
    X.row_ptr.assign(d1 + 1, 0); X.item.resize(nnz); X.rating.resize(nnz);
    int64_t cc = 0;
    for (int64_t j = 0; j < d1; ++j) {
        X.row_ptr[j] = cc;
        for (; cc < nnz; ++cc) {
            if (t.u[cc] > j) break;
            X.item[cc] = t.i[cc]; X.rating[cc] = t.r[cc];
        }
    }
    X.row_ptr[d1] = cc; X.nnz = cc;
    X.item.resize(cc); X.rating.resize(cc);
    return X;
}

struct DataDir { Csr train, test; bool has_test = false; };

inline DataDir load_dir(const std::string &dir) {
    FILE *fp = fopen((dir + "/meta").c_str(), "r");
    if (!fp) throw std::runtime_error("cannot open " + dir + "/meta");
    long m = 0, n = 0, nnz = 0, nnz_t = 0;
    char buf[1024], buf2[1024];
    if (fscanf(fp, "%ld %ld", &m, &n) != 2 || fscanf(fp, "%ld %1023s", &nnz, buf) != 2) { fclose(fp); throw std::runtime_error("bad meta file"); }
    const bool has_test = fscanf(fp, "%ld %1023s", &nnz_t, buf2) == 2;
    fclose(fp);
    DataDir d;
    d.train = build_train_csr(m, n, parse_file_parts(dir + "/" + buf, nnz));
    d.has_test = has_test;
    if (has_test) d.test = build_test_csr(m, n, parse_file(dir + "/" + buf2, nnz_t));
    else { d.test.d1 = m; d.test.d2 = n; d.test.row_ptr.assign(m + 1, 0); }
    return d;
}

}  // namespace pcrhost
