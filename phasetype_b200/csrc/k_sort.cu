/*
 * k_sort.cu -- observation layout for the MHRS sweep: y in decreasing order.
 *
 * The number of rejection attempts an observation needs is Geometric(survival(y)), so its cost is known in
 * advance up to noise.  The lane phase of k_mhrs.cu walks the observations in layout order; with the expensive
 * ones first, the stream ends on the cheapest observations and the grid drains in microseconds instead of
 * handing a hundred thousand half-done observations to the tail.  Paths are keyed by the GLOBAL observation
 * index (perm carries it along), so the layout changes nothing in the results.
 * Done once per engine, on the device (CUB radix sort: 64-bit keys, 32-bit payload).  Method 64 with groups
 * (pht_engine_set_groups) adds a stable pass by group id over that permutation, so each group is a contiguous range
 * still ordered by decreasing y.
 */
#include <cub/device/device_radix_sort.cuh>
#include "engine_internal.h"

__global__ void k_iota(uint32_t *v, long l) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < l) v[i] = (uint32_t)i;
}
__global__ void k_gather_u8(const uint8_t *src, const uint32_t *perm, uint8_t *dst, long l) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < l) dst[i] = src[perm[i]];
}
__global__ void k_gather_f64(const double *src, const uint32_t *perm, double *dst, long l) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < l) dst[i] = src[perm[i]];
}

/* ys[i] = y[perm[i]] non-increasing, cs[i] = cens[perm[i]]; all pointers device memory of length l */
cudaError_t pht_sort_by_y_desc(const double *y, const uint8_t *cens, long l, double *ys, uint8_t *cs, uint32_t *perm, cudaStream_t st) {
    if (l <= 0) return cudaSuccess;
    uint32_t *idx = nullptr; void *tmp = nullptr; size_t tmp_bytes = 0;
    cudaError_t e = pht_dev_alloc((void **)&idx, sizeof(uint32_t) * (size_t)l, st);
    if (e != cudaSuccess) return e;
    const int threads = 256; const unsigned blocks = (unsigned)((l + threads - 1) / threads);
    k_iota<<<blocks, threads, 0, st>>>(idx, l);
    e = cub::DeviceRadixSort::SortPairsDescending(nullptr, tmp_bytes, y, ys, idx, perm, (int)l, 0, 64, st);
    if (e == cudaSuccess) e = pht_dev_alloc(&tmp, tmp_bytes ? tmp_bytes : 1, st);
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairsDescending(tmp, tmp_bytes, y, ys, idx, perm, (int)l, 0, 64, st);
    if (e == cudaSuccess) { k_gather_u8<<<blocks, threads, 0, st>>>(cens, perm, cs, l); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    pht_dev_free(tmp, st);
    pht_dev_free(idx, st);
    return e;
}

__global__ void k_group_keys(const uint32_t *perm_y, const uint8_t *group, uint8_t *keys, uint32_t *idx, long l) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < l) { const uint32_t k = perm_y ? perm_y[i] : (uint32_t)i; idx[i] = k; keys[i] = group[k]; }
}

/* groups (method 64): a second, stable pass over the y-descending permutation, by group id ascending (8-bit keys) */
cudaError_t pht_sort_by_group(const uint32_t *perm_y, const uint8_t *group, const double *y, const uint8_t *cens, long l,
                              double *ys, uint8_t *cs, uint32_t *perm, cudaStream_t st) {
    if (l <= 0) return cudaSuccess;
    uint32_t *idx = nullptr; uint8_t *keys = nullptr, *keys_out = nullptr; void *tmp = nullptr; size_t tmp_bytes = 0;
    cudaError_t e = pht_dev_alloc((void **)&idx, sizeof(uint32_t) * (size_t)l, st);
    if (e == cudaSuccess) e = pht_dev_alloc((void **)&keys, (size_t)l, st);
    if (e == cudaSuccess) e = pht_dev_alloc((void **)&keys_out, (size_t)l, st);
    const int threads = 256; const unsigned blocks = (unsigned)((l + threads - 1) / threads);
    if (e == cudaSuccess) { k_group_keys<<<blocks, threads, 0, st>>>(perm_y, group, keys, idx, l); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys_out, idx, perm, (int)l, 0, 8, st);
    if (e == cudaSuccess) e = pht_dev_alloc(&tmp, tmp_bytes ? tmp_bytes : 1, st);
    if (e == cudaSuccess) e = cub::DeviceRadixSort::SortPairs(tmp, tmp_bytes, keys, keys_out, idx, perm, (int)l, 0, 8, st);
    if (e == cudaSuccess) { k_gather_f64<<<blocks, threads, 0, st>>>(y, perm, ys, l); e = cudaGetLastError(); }
    if (e == cudaSuccess) { k_gather_u8<<<blocks, threads, 0, st>>>(cens, perm, cs, l); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    pht_dev_free(tmp, st); pht_dev_free(keys_out, st); pht_dev_free(keys, st); pht_dev_free(idx, st);
    return e;
}

/* interval bounds into the sorted layout (pht_engine_set_upper): the sort itself stays as it is */
cudaError_t pht_gather_f64(const double *src, const uint32_t *perm, double *dst, long l, cudaStream_t st) {
    if (l <= 0) return cudaSuccess;
    const int threads = 256; const unsigned blocks = (unsigned)((l + threads - 1) / threads);
    k_gather_f64<<<blocks, threads, 0, st>>>(src, perm, dst, l);
    return cudaGetLastError();
}
