// k_setup.cu -- one-time preprocessing on the device (replaces convert() util.cpp:219-274 and the CSR->CSC
// transpose of smat_t::load_from_iterator util.h:259-270).
// CUB (shipped with the CUDA toolkit) is used here only for the scan and the radix sort of the CSC build; the heavy
// users are sorted by k_hsort.cu, the per-iteration hot kernels are in k_core.cu.
#include "kernels.h"
#include <cub/cub.cuh>

namespace pcr {

#define LAUNCH(ctx, name, bytes, kernel, grid, block, smem, ...)                         \
    do {                                                                                 \
        (ctx).prof->begin(name, (ctx).stream, (double)(bytes));                          \
        kernel<<<(grid), (block), (smem), (ctx).stream>>>(__VA_ARGS__);                  \
        (ctx).prof->end((ctx).stream);                                                   \
        PCR_CUDA(cudaGetLastError());                                                    \
    } while (0)

static inline unsigned grid_for(i64 n, int per_block, int max_blocks) {
    i64 b = (n + per_block - 1) / per_block;
    if (b < 1) b = 1;
    if (b > max_blocks) b = max_blocks;
    return (unsigned)b;
}

// user_out[e] = the row that contains CSR position e (binary search in row_ptr)
__global__ void expand_users_kernel(const i64 *__restrict__ row_ptr, i64 d1, i64 nnz, int32_t *__restrict__ out) {
    for (i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (i64)gridDim.x * blockDim.x) {
        i64 a = 0, b = d1;                 // last u with row_ptr[u] <= e
        while (b - a > 1) { const i64 mid = (a + b) >> 1; if (row_ptr[mid] <= e) a = mid; else b = mid; }
        out[e] = (int32_t)a;
    }
}
void k_expand_users(Ctx &c, const i64 *row_ptr, i64 d1, i64 nnz, int32_t *user_out) {
    if (nnz <= 0) return;
    LAUNCH(c, "expand_users", 0.0, expand_users_kernel, grid_for(nnz, 256, c.sms * 16), 256, 0, row_ptr, d1, nnz, user_out);
}

// level index of lround(rating) in the ascending table (find_levels pcrpp.cpp:38-49 + remap :182-189)
__global__ void levels_kernel(const double *__restrict__ rating, i64 nnz, const i64 *__restrict__ table, int T,
                              uint8_t *__restrict__ out, int *__restrict__ bad) {
    for (i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (i64)gridDim.x * blockDim.x) {
        const i64 v = llround(rating[e]);
        int k = 0, hi = T;                      // the table is strictly ascending: lower bound
        while (k < hi) { const int mid = (k + hi) >> 1; if (table[mid] < v) k = mid + 1; else hi = mid; }
        if (k == T || table[k] != v) { atomicOr(bad, 1); k = 0; }
        if ((double)v != rating[e] && !(*reinterpret_cast<volatile int *>(bad) & 2)) atomicOr(bad, 2);
        out[e] = (uint8_t)k;
    }
}
void k_levels(Ctx &c, const double *rating, i64 nnz, const i64 *table_dev, int T, uint8_t *level_out, int *bad_flag) {
    if (nnz <= 0) return;
    LAUNCH(c, "levels", 0.0, levels_kernel, grid_for(nnz, 256, c.sms * 16), 256, 0, rating, nnz, table_dev, T, level_out, bad_flag);
}

__global__ void iota32_kernel(int32_t *out, i64 n) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) out[i] = (int32_t)i;
}
void k_iota32(Ctx &c, int32_t *out, i64 n) {
    if (n <= 0) return;
    LAUNCH(c, "iota32", 0.0, iota32_kernel, grid_for(n, 256, c.sms * 16), 256, 0, out, n);
}

// number of entries whose id lies outside [0, bound): checked BEFORE any kernel indexes with them
__global__ void count_out_of_range_kernel(const int32_t *__restrict__ idx, i64 n, i64 bound, int *__restrict__ bad) {
    int local = 0;
    for (i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (i64)gridDim.x * blockDim.x)
        if (idx[e] < 0 || (i64)idx[e] >= bound) local = 1;
    if (local) atomicOr(bad, 1);
}
void k_check_range(Ctx &c, const int32_t *idx, i64 n, i64 bound, int *bad_flag) {
    if (n <= 0) return;
    LAUNCH(c, "check_range", 0.0, count_out_of_range_kernel, grid_for(n, 256, c.sms * 16), 256, 0, idx, n, bound, bad_flag);
}

__global__ void hist_kernel(const int32_t *__restrict__ item, i64 nnz, unsigned long long *__restrict__ counts) {
    for (i64 e = (i64)blockIdx.x * blockDim.x + threadIdx.x; e < nnz; e += (i64)gridDim.x * blockDim.x)
        atomicAdd(&counts[item[e]], 1ull);
}
__global__ void gather_i32_kernel(const int32_t *__restrict__ src, const int32_t *__restrict__ idx, i64 n, int32_t *__restrict__ out) {
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) out[i] = src[idx[i]];
}

void k_build_csc(Ctx &c, DevPool &pool, const int32_t *item, const int32_t *user, i64 nnz, i64 d2,
                 i64 *col_ptr, int32_t *csc2csr, int32_t *csc_user) {
    PCR_CUDA(cudaMemsetAsync(col_ptr, 0, sizeof(i64) * (size_t)(d2 + 1), c.stream));
    if (nnz <= 0) return;
    // histogram -> exclusive scan = col_ptr
    unsigned long long *counts = nullptr;
    counts = (unsigned long long *)pool.raw_alloc(sizeof(unsigned long long) * (size_t)(d2 + 1));
    PCR_CUDA(cudaMemsetAsync(counts, 0, sizeof(unsigned long long) * (size_t)(d2 + 1), c.stream));
    LAUNCH(c, "csc_hist", 0.0, hist_kernel, grid_for(nnz, 256, c.sms * 16), 256, 0, item, nnz, counts);
    void *tmp = nullptr; size_t tb = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb, (const i64 *)counts, col_ptr, (int)(d2 + 1), c.stream);
    tmp = pool.raw_alloc(tb > 0 ? tb : 1);
    c.prof->begin("csc_scan(cub)", c.stream, 0.0);
    PCR_CUDA(cub::DeviceScan::ExclusiveSum(tmp, tb, (const i64 *)counts, col_ptr, (int)(d2 + 1), c.stream));
    c.prof->end(c.stream);
    PCR_CUDA(cudaStreamSynchronize(c.stream));
    pool.raw_free(tmp); pool.raw_free(counts);
    // stable radix sort of (item -> CSR position): users stay ascending inside an item
    int32_t *keys_out = nullptr, *iota = nullptr;
    keys_out = (int32_t *)pool.raw_alloc(sizeof(int32_t) * (size_t)nnz);
    iota = (int32_t *)pool.raw_alloc(sizeof(int32_t) * (size_t)nnz);
    k_iota32(c, iota, nnz);
    int bits = 1;
    while (bits < 31 && ((i64)1 << bits) < d2) ++bits;
    tmp = nullptr; tb = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tb, item, keys_out, (const int32_t *)iota, csc2csr, nnz, 0, bits, c.stream);
    tmp = pool.raw_alloc(tb > 0 ? tb : 1);
    c.prof->begin("csc_sort(cub)", c.stream, 0.0);
    PCR_CUDA(cub::DeviceRadixSort::SortPairs(tmp, tb, item, keys_out, (const int32_t *)iota, csc2csr, nnz, 0, bits, c.stream));
    c.prof->end(c.stream);
    LAUNCH(c, "csc_users", 0.0, gather_i32_kernel, grid_for(nnz, 256, c.sms * 16), 256, 0, user, csc2csr, nnz, csc_user);
    PCR_CUDA(cudaStreamSynchronize(c.stream));
    pool.raw_free(tmp); pool.raw_free(keys_out); pool.raw_free(iota);
}

__global__ void csc_block_bounds_kernel(const i64 *__restrict__ col_ptr, const int32_t *__restrict__ csc_user, i64 d2, int nb,
                                        i64 block_users, i64 *__restrict__ bpos) {
    const i64 total = d2 * (nb + 1);
    for (i64 t = (i64)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (i64)gridDim.x * blockDim.x) {
        const i64 p = t / (nb + 1); const int j = (int)(t - p * (nb + 1));
        i64 a = col_ptr[p], b = col_ptr[p + 1];
        const i64 key = (i64)j * block_users;
        while (a < b) { const i64 mid = (a + b) >> 1; if ((i64)csc_user[mid] < key) a = mid + 1; else b = mid; }
        bpos[t] = a;
    }
}
void k_csc_block_bounds(Ctx &c, const i64 *col_ptr, const int32_t *csc_user, i64 d2, int nb, i64 block_users, i64 *bpos) {
    if (d2 <= 0) return;
    LAUNCH(c, "csc_block_bounds", 0.0, csc_block_bounds_kernel, grid_for(d2 * (nb + 1), 256, c.sms * 16), 256, 0, col_ptr, csc_user, d2, nb, block_users, bpos);
}

}  // namespace pcr
