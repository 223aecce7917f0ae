// transpose.cu — the transposed operator: a second handle over A^T, built on the device from the CSR of an existing
// handle, so that the gradient dB = A^T · dC runs through the same plan and kernels as the forward product.
//
// No reference counterpart: PA4 is forward only (SURVEY.md §8f-3 lists the transposed product as the optional
// remaining half of the stacked-GNN step). The transposed CSR keeps, inside every row (= column of A), the nonzeros
// in A's storage order — ascending row of A — so each output element is again ONE in-order FMA chain, fully specified
// and restated on the CPU by oracle_spmm_t_f32 (oracle/spmm_oracle.c).
//
// Construction (all on the device, no host copy of idx/val): histogram of the columns -> exclusive scan = ptr of A^T;
// stable LSD radix sort of the nonzero positions by column (cub::DeviceRadixSort — preprocessing only, not on the
// hot path) -> `perm`; idx_t[k] = row of A of nonzero perm[k], val_t[k] = val[perm[k]]. `perm` is kept so that
// spmm_b200_refresh_values can re-gather the values after the caller re-weights the edges.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <new>

#include "common.h"

namespace spmm_b200 {

namespace {

__global__ void __launch_bounds__(256) col_histogram_kernel(const int *idx, long long nnz, int *count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride) atomicAdd(count + idx[i], 1);
}

// one warp per row of A: the row id of each of its nonzeros, and the identity permutation
__global__ void __launch_bounds__(256) expand_rows_kernel(const int *ptr, int num_v, int *row_of, int *pos) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= num_v) return;
    for (int i = ptr[gw] + lane; i < ptr[gw + 1]; i += 32) {
        row_of[i] = (int)gw;
        pos[i] = i;
    }
}

// one warp per row of A: (row, column) as one 64-bit sort key per nonzero, and the identity permutation
__global__ void __launch_bounds__(256) row_col_keys_kernel(const int *ptr, const int *idx, int num_v, unsigned long long *key, int *pos) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= num_v) return;
    for (int i = ptr[gw] + lane; i < ptr[gw + 1]; i += 32) {
        key[i] = ((unsigned long long)gw << 32) | (unsigned int)idx[i];
        pos[i] = i;
    }
}

__global__ void __launch_bounds__(256) gather_t_kernel(const int *perm, const int *row_of, const float *val, long long nnz, int *idx_t,
                                                       float *val_t) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < nnz; k += stride) {
        const int i = perm[k];
        if (idx_t) idx_t[k] = row_of[i];
        val_t[k] = val[i];
    }
}

// Radix key bits that cover [0, n): at least 1, at most 31.
int key_bits(long long n) {
    int bits = 1;
    while (bits < 31 && (1ll << bits) < n) ++bits;
    return bits;
}

// Pool blocks (pool.cu) that one construction borrows, stream-ordered on `s`; create_derived frees them however it ends.
struct Scratch {
    cudaStream_t s;
    void *p[5] = {};   // the most one construction borrows (the transposed one)
    int n = 0;
    template <class T>
    cudaError_t alloc(T **ptr, size_t bytes) {
        const cudaError_t e = pool_alloc((void **)ptr, bytes, s);
        if (e == cudaSuccess) p[n++] = *ptr;
        return e;
    }
    void drop() {
        for (int i = 0; i < n; ++i) pool_free(p[i], s);
    }
};

// What the transposed and the column-sorted handle share: the argument check, a new handle whose t_idx / t_val / t_perm
// (max(1, nnz) each) come from the current device's pool, one failure path that leaves no handle and no scratch behind,
// and the synchronise before the handle is returned. build(t, scratch) queues the rest on the stream and sets t's d_ptr,
// num_v and b_rows; it returns 0 or a status code.
template <class Build>
int create_derived(spmm_b200_handle *h, int feat_in, void *stream, spmm_b200_t *out, const char *who, Build build) {
    if (!h || !out || feat_in < 0) {
        set_error("%s: bad arguments", who);
        return SPMM_B200_EINVAL;
    }
    spmm_b200_handle *t = new (std::nothrow) spmm_b200_handle();
    if (!t) {
        set_error("%s: out of host memory", who);
        return SPMM_B200_ENOMEM;
    }
    cudaStream_t s = (cudaStream_t)stream;
    Scratch scratch{s};
    const int rc = [&]() {
        const size_t cnt = (size_t)std::max<long long>(1, h->num_e);
        SB_CUDA(cudaGetDevice(&t->t_device));
        SB_CUDA(pool_alloc((void **)&t->t_idx, sizeof(int) * cnt, s));
        SB_CUDA(pool_alloc((void **)&t->t_val, sizeof(float) * cnt, s));
        SB_CUDA(pool_alloc((void **)&t->t_perm, sizeof(int) * cnt, s));
        const int rc = build(t, scratch);
        if (rc) return rc;
        SB_CUDA(cudaStreamSynchronize(s));
        return 0;
    }();
    if (rc) {
        cudaStreamSynchronize(s);   // whatever was queued may still read the scratch
        cudaGetLastError();
        scratch.drop();
        spmm_b200_destroy(t);
        return rc;
    }
    scratch.drop();
    t->d_idx = t->t_idx;
    t->d_val = t->t_val;
    t->num_e = h->num_e;
    t->feat = feat_in;
    t->t_src = h;
    *out = t;
    return 0;
}

}  // namespace

// values of the transposed CSR from the source handle's current val (spmm_b200_refresh_values on a transposed handle)
int regather_transposed_values(spmm_b200_handle *t, cudaStream_t stream) {
    if (!t->t_src || t->num_e == 0) return 0;
    gather_t_kernel<<<stride_grid(t->num_e), 256, 0, stream>>>(t->t_perm, nullptr, t->t_src->d_val, t->num_e, nullptr, t->t_val);
    SB_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" int spmm_b200_create_transposed(spmm_b200_t h, int feat_in, void *stream, spmm_b200_t *out) {
    return create_derived(h, feat_in, stream, out, "spmm_b200_create_transposed", [&](spmm_b200_handle *t, Scratch &scratch) {
        cudaStream_t s = scratch.s;
        const int rows_t = h->b_rows > 0 ? h->b_rows : h->num_v;   // rows of A^T = columns of A = rows of B
        const long long nnz = h->num_e;
        SB_CUDA(pool_alloc((void **)&t->t_ptr, sizeof(int) * ((size_t)rows_t + 1), s));
        SB_CUDA(cudaMemsetAsync(t->t_ptr, 0, sizeof(int) * ((size_t)rows_t + 1), s));
        t->d_ptr = t->t_ptr;
        t->num_v = rows_t;
        t->b_rows = h->num_v;   // A^T gathers rows of dC, which has as many rows as A
        if (nnz == 0) return 0;
        // a column outside [0, rows_t) would corrupt the histogram: same check as preprocess
        int *bad = nullptr, *row_of = nullptr, *pos = nullptr, *keys_out = nullptr, h_bad = 0;
        void *tmp = nullptr;
        SB_CUDA(scratch.alloc(&bad, sizeof(int)));
        SB_CUDA(cudaMemsetAsync(bad, 0, sizeof(int), s));
        const int rc = launch_check_cols(h->d_idx, nnz, rows_t, bad, s);
        if (rc) return rc;
        SB_CUDA(cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, s));
        SB_CUDA(cudaStreamSynchronize(s));
        if (h_bad) {
            set_error("CSR idx holds a column outside [0, %d)", rows_t);
            return SPMM_B200_EINVAL;
        }
        SB_CUDA(scratch.alloc(&row_of, sizeof(int) * (size_t)nnz));
        SB_CUDA(scratch.alloc(&pos, sizeof(int) * (size_t)nnz));
        SB_CUDA(scratch.alloc(&keys_out, sizeof(int) * (size_t)nnz));
        // ptr of A^T: counts shifted by one, then an inclusive scan in place == exclusive scan of the counts
        col_histogram_kernel<<<stride_grid(nnz), 256, 0, s>>>(h->d_idx, nnz, t->t_ptr + 1);
        SB_CUDA(cudaGetLastError());
        size_t scan_bytes = 0, sort_bytes = 0;
        SB_CUDA(cub::DeviceScan::InclusiveSum(nullptr, scan_bytes, t->t_ptr + 1, t->t_ptr + 1, rows_t, s));
        const int bits = key_bits(rows_t);
        SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, h->d_idx, keys_out, pos, t->t_perm, (int)nnz, 0, bits, s));
        SB_CUDA(scratch.alloc(&tmp, std::max(scan_bytes, sort_bytes)));
        SB_CUDA(cub::DeviceScan::InclusiveSum(tmp, scan_bytes, t->t_ptr + 1, t->t_ptr + 1, rows_t, s));
        const long long threads = (long long)h->num_v * 32;
        if (h->num_v > 0) expand_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(h->d_ptr, h->num_v, row_of, pos);
        SB_CUDA(cudaGetLastError());
        // stable: equal columns keep A's storage order, i.e. ascending row of A
        SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, sort_bytes, h->d_idx, keys_out, pos, t->t_perm, (int)nnz, 0, bits, s));
        gather_t_kernel<<<stride_grid(nnz), 256, 0, s>>>(t->t_perm, row_of, h->d_val, nnz, t->t_idx, t->t_val);
        SB_CUDA(cudaGetLastError());
        return 0;
    });
}

// The column-sorted operator: a second handle over the SAME matrix whose rows are stored in ascending column order
// (equal columns keep their storage order: the radix sort is stable). For CSR inputs whose rows are not column-sorted —
// which the plan otherwise keeps in one column block, because splitting an unsorted row at band boundaries would reorder
// its FMA chain (preprocess.cu) — this is the opt-in that gives them the L2-resident bands: outputs then associate in
// column order, i.e. they equal the reference run on the sorted CSR bit for bit and the reference run on the original
// order within the split-row tolerance. Shares ptr with `h` (borrowed), owns idx / val / perm (pool.cu).
extern "C" int spmm_b200_create_column_sorted(spmm_b200_t h, int feat_in, void *stream, spmm_b200_t *out) {
    return create_derived(h, feat_in, stream, out, "spmm_b200_create_column_sorted", [&](spmm_b200_handle *t, Scratch &scratch) {
        cudaStream_t s = scratch.s;
        const long long nnz = h->num_e;
        t->d_ptr = h->d_ptr;   // same rows, same lengths
        t->num_v = h->num_v;
        t->b_rows = h->b_rows;
        if (nnz == 0) return 0;
        unsigned long long *key_in = nullptr, *key_out = nullptr;
        int *pos = nullptr;
        void *tmp = nullptr;
        SB_CUDA(scratch.alloc(&key_in, sizeof(unsigned long long) * (size_t)nnz));
        SB_CUDA(scratch.alloc(&key_out, sizeof(unsigned long long) * (size_t)nnz));
        SB_CUDA(scratch.alloc(&pos, sizeof(int) * (size_t)nnz));
        const long long threads = (long long)h->num_v * 32;
        row_col_keys_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(h->d_ptr, h->d_idx, h->num_v, key_in, pos);
        SB_CUDA(cudaGetLastError());
        const int bits = 32 + key_bits(h->num_v);
        size_t sort_bytes = 0;
        SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, key_in, key_out, pos, t->t_perm, (int)nnz, 0, bits, s));
        SB_CUDA(scratch.alloc(&tmp, sort_bytes));
        // stable: nonzeros of one row with the same column keep their storage order
        SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp, sort_bytes, key_in, key_out, pos, t->t_perm, (int)nnz, 0, bits, s));
        // idx_sorted[k] = idx[perm[k]], val_sorted[k] = val[perm[k]]
        gather_t_kernel<<<stride_grid(nnz), 256, 0, s>>>(t->t_perm, h->d_idx, h->d_val, nnz, t->t_idx, t->t_val);
        SB_CUDA(cudaGetLastError());
        return 0;
    });
}
