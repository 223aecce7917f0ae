// rows.cuh — how the row-wise kernels (edge_softmax.cu, reduce.cu) split a CSR's rows (internal, not installed).
//
// Every call makes two launches of kRowBlock threads per CTA over all rows; each kernel skips the other's rows, split
// at a threshold of nonzeros that each file sets for itself.
//   Warp launch (rows up to the threshold): warp w takes the contiguous rows [first_row(w * chunk),
//     first_row((w + 1) * chunk)), first_row(d) being the first row r with ptr[r] + r >= d, so every warp gets about
//     `chunk` rows + nonzeros. chunk = (rows + nonzeros) / (kWarpWaves ranges per resident warp, 32 warps per SM
//     assumed), rounded up and at least kMinChunk.
//   Long-row launch (rows above the threshold, one CTA each): CTA b scans the stripes b, b + gridDim.x, ... of kRowBlock
//     rows, marks a stripe's long rows with one ballot per warp and takes them in row order; min(stripes, 4 x SMs)
//     CTAs. No list of long rows, no workspace.
#ifndef HPC_B200_ROWS_CUH_
#define HPC_B200_ROWS_CUH_

#include "common.h"

namespace spmm_b200 {

namespace {

constexpr int kRowBlock = 256;             // threads per CTA of both launches, and rows per stripe
constexpr int kRowWarps = kRowBlock / 32;
constexpr int kWarpWaves = 4;              // row ranges per resident warp (32 per SM assumed): a short tail
constexpr long long kMinChunk = 256;       // rows + nonzeros per warp at least

// first row r in [0, num_v] with ptr[r] + r >= d
__device__ int first_row(const int *ptr, int num_v, long long d) {
    int lo = 0, hi = num_v;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((long long)__ldg(ptr + mid) + mid >= d) hi = mid;
        else lo = mid + 1;
    }
    return lo;
}

// The calling warp's rows [r0, r1) in the warp launch.
// tid defaults to threadIdx.x read at the call site. nvcc bounds each threadIdx.x read by the __launch_bounds__ of the
// function that contains it before it inlines anything. In a kernel that bound is kRowBlock, in a device function it
// is 1024, even a __forceinline__ one. With the tighter bound w's add compiles to an OR, and other index arithmetic
// simplifies too. Reading threadIdx.x inside these helpers instead changes the SASS of 14 of the 20 row-wise kernels
// (sm_100a, CUDA 12.9). Reading it inside a long-row body changes the four reduce_long_kernel instances.
template <class Args>
__device__ __forceinline__ void warp_rows(const Args &a, int &r0, int &r1, unsigned tid = threadIdx.x) {
    const long long w = (long long)blockIdx.x * kRowWarps + (tid >> 5);
    r0 = first_row(a.ptr, a.num_v, w * a.chunk);
    r1 = first_row(a.ptr, a.num_v, (w + 1) * a.chunk);
}

// body(r) for every row r of more than min_len nonzeros, in the long-row launch's order. Called by the whole CTA, and
// so is body, which may synchronise the CTA. long_mask is the kernel's __shared__ unsigned[kRowWarps]. tid: as in
// warp_rows. body is a lambda, that is, a device function, so it should use a thread index the kernel has read rather
// than threadIdx.x.
template <class Args, class Body>
__device__ __forceinline__ void for_long_rows(const Args &a, int min_len, unsigned *long_mask, Body body,
                                              unsigned tid = threadIdx.x) {
    const int lane = tid & 31, warp = tid >> 5;
    for (long long r0 = (long long)blockIdx.x * kRowBlock; r0 < a.num_v; r0 += (long long)gridDim.x * kRowBlock) {
        const long long rr = r0 + tid;
        const bool is_long = rr < a.num_v && __ldg(a.ptr + rr + 1) - __ldg(a.ptr + rr) > min_len;
        const unsigned bm = __ballot_sync(0xffffffffu, is_long);
        if (lane == 0) long_mask[warp] = bm;
        __syncthreads();
        for (int sw = 0; sw < kRowWarps; ++sw)
            for (unsigned rest = long_mask[sw]; rest; rest &= rest - 1) body((int)r0 + sw * 32 + __ffs(rest) - 1);
        __syncthreads();   // long_mask is rewritten by the next stripe
    }
}

// The grids of both launches and the warp launch's chunk, for the current device.
struct RowGrid {
    unsigned warp_blocks, long_blocks;
    long long chunk;
};
int row_grid(int num_v, long long num_e, RowGrid *g) {
    int sms = 0;
    SB_CUDA(query_sm_count(&sms));
    if (sms <= 0) sms = 1;
    const long long d = num_e + num_v;
    const long long target = (long long)sms * 32 * kWarpWaves;
    g->chunk = (d + target - 1) / target;
    if (g->chunk < kMinChunk) g->chunk = kMinChunk;
    const long long warps = (d + g->chunk - 1) / g->chunk;
    g->warp_blocks = (unsigned)((warps + kRowWarps - 1) / kRowWarps);
    const long long stripes = ((long long)num_v + kRowBlock - 1) / kRowBlock;
    g->long_blocks = (unsigned)(stripes < (long long)sms * 4 ? stripes : (long long)sms * 4);
    return 0;
}

}  // namespace

}  // namespace spmm_b200
#endif
