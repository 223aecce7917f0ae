// sddmm.cu — SDDMM over the operator's sparsity pattern (spmm_b200_sddmm): for every nonzero e of row r,
//     out[e] = sum_j x_row[r * K + j] * x_col[idx[e] * K + j]
// With x_row = dC and x_col = B this is dL/dval of C = A·B, the gradient the forward product and the transposed
// operator leave out; with x_row = X_dst and x_col = X_src it is the score of an attention edge. No reference
// counterpart (PA4 is forward only); restated on the CPU by oracle_sddmm_f32 (tests/sddmm_oracle.c).
//
// Summation order (depends on K alone, so the bits do not change with any plan option, row partition or column-block
// layout). K % 4 == 0: Q = K/4 float4 groups, L = min(32, pow2ceil(Q)) lanes. Lane l starts from 0.0f and, for
// q = l, l+L, ... < Q and t = 0..3, computes s_l = fmaf(x_row[4q+t], x_col[4q+t], s_l). Then for o = L/2, L/4, ..., 1
// every lane sets s_l = s_l + s_(l xor o), and out[e] = s_0. K % 4 != 0: the same with scalar columns (Q = K,
// L = min(32, pow2ceil(K)), one fmaf per column). Built -ftz=true: every FMA and add flushes subnormals.
//
// Work split: equal chunks of nonzeros per warp (merge path), not a warp per row — rows range from empty to 21 657
// nonzeros on the reddit shape. A warp binary-searches the segment its chunk starts in and walks on from there.
// With several column blocks the nonzeros are walked band-major, in the virtual order "band 0 of every row, then band
// 1 of every row, ...": the x_col band in flight stays in the L2, as in the forward passes, and since no output
// depends on another band the one launch needs no waiting between bands. The prefix of that virtual order (an
// exclusive scan of the (band, row) lengths from the plan's split array) is built on the device by the first call
// after preprocess; with one block it is ptr itself.
#include <cub/device/device_scan.cuh>

#include "common.h"

namespace spmm_b200 {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kBlock = 256;
constexpr int kWaves = 8;          // chunks per resident warp: a short tail, and a narrow window over the bands
constexpr int kMinChunk = 128;     // nonzeros per warp at least: keeps the binary search small next to the walk

struct SddmmArgs {
    const int *vp;        // [n_seg + 1] virtual start of every (band, row) segment, band-major (ptr with one band)
    const int *start;     // [n_seg] CSR position where segment s starts (the plan's split array, or ptr)
    const int *idx;
    const float *x_row;   // num_v x K
    const float *x_col;   // b_rows x K
    float *out;           // num_e
    int num_v, n_seg, nnz, feat, chunk;
};

__device__ __forceinline__ int ld_stream_s32(const int *p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}

// The walk of one lane group over the virtual positions: the segment s holding the current position, its row, its
// virtual end and the offset from virtual to CSR position. Positions only grow, so a cursor steps forward.
struct Cursor {
    int s, row, end, off;
    __device__ __forceinline__ void init(const SddmmArgs &a, int v) {
        int lo = 0, hi = a.n_seg;   // vp[lo] <= v < vp[hi]: the last segment that starts at or before v (not empty)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (__ldg(a.vp + mid) <= v) lo = mid;
            else hi = mid;
        }
        s = lo;
        row = lo % a.num_v;
        end = __ldg(a.vp + lo + 1);
        off = __ldg(a.start + lo) - __ldg(a.vp + lo);
    }
    // CSR position of virtual position v (>= the previous one)
    __device__ __forceinline__ int pos(const SddmmArgs &a, int v) {
        if (v >= end) {
            int beg;
            do {
                beg = end;
                ++s;
                if (++row == a.num_v) row = 0;
                end = __ldg(a.vp + s + 1);
            } while (v >= end);
            off = __ldg(a.start + s) - beg;
        }
        return v + off;
    }
};

__device__ __forceinline__ void fma_dot4(float &s, const float4 &x, const float4 &y) {
    s = fmaf(x.x, y.x, s);
    s = fmaf(x.y, y.y, s);
    s = fmaf(x.z, y.z, s);
    s = fmaf(x.w, y.w, s);
}

// K % 4 == 0 and K <= 512. LANES lanes per entry (L of the order above), each owning VEC float4 of the row;
// 32 / LANES lane groups take alternate entries, U entries per group in flight. The row's x_row slice stays in
// registers; the first new row of a batch is fetched together with the batch's gathers.
template <int LANES, int VEC, int U>
__global__ void __launch_bounds__(kBlock) sddmm_kernel(const __grid_constant__ SddmmArgs a) {
    constexpr int G = 32 / LANES;
    const int lane = threadIdx.x & 31;
    const int l = lane % LANES, g = lane / LANES;
    const long long v0 = ((long long)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) * a.chunk;
    if (v0 >= a.nnz) return;
    const int vend = (int)min((long long)a.nnz, v0 + a.chunk);
    const int Q = a.feat >> 2;
    const float4 *xr4 = reinterpret_cast<const float4 *>(a.x_row) + l;
    const float4 *xc4 = reinterpret_cast<const float4 *>(a.x_col) + l;
    bool qok[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) qok[v] = l + v * LANES < Q;

    Cursor cur;
    cur.init(a, (int)v0);
    float4 xr[VEC], xn[VEC];
    int row_xr = -1, row_xn = -1;
    for (int vb = (int)v0; vb < vend; vb += G * U) {
        int pos[U], row[U], col[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int v = vb + u * G + g;
            pos[u] = v < vend ? cur.pos(a, v) : -1;
            row[u] = cur.row;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) col[u] = pos[u] >= 0 ? ld_stream_s32(a.idx + pos[u]) : 0;
        float4 b[U][VEC];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const float4 *src = xc4 + (size_t)col[u] * Q;
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (qok[v]) b[u][v] = __ldg(src + v * LANES);
        }
        int want = -1;
#pragma unroll
        for (int u = U - 1; u >= 0; --u)
            if (pos[u] >= 0 && row[u] != row_xr) want = row[u];
        if (want >= 0 && want != row_xn) {
            const float4 *src = xr4 + (size_t)want * Q;
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (qok[v]) xn[v] = __ldg(src + v * LANES);
            row_xn = want;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (pos[u] >= 0 && row[u] != row_xr) {
                if (row[u] == row_xn) {
#pragma unroll
                    for (int v = 0; v < VEC; ++v) xr[v] = xn[v];
                } else {   // a second new row inside one batch (short rows)
                    const float4 *src = xr4 + (size_t)row[u] * Q;
#pragma unroll
                    for (int v = 0; v < VEC; ++v)
                        if (qok[v]) xr[v] = __ldg(src + v * LANES);
                }
                row_xr = row[u];
            }
            float s = 0.f;
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (qok[v]) fma_dot4(s, xr[v], b[u][v]);
#pragma unroll
            for (int o = LANES / 2; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
            if (l == 0 && pos[u] >= 0) a.out[pos[u]] = s;
        }
    }
}

// K % 4 != 0 (V4 = false: scalar columns) and K > 512 (V4 = true): the same order with a runtime lane count, one entry
// per lane group at a time, x_row read per entry.
template <bool V4>
__global__ void __launch_bounds__(kBlock) sddmm_generic_kernel(const __grid_constant__ SddmmArgs a, int lanes) {
    const int G = 32 / lanes;
    const int lane = threadIdx.x & 31;
    const int l = lane % lanes, g = lane / lanes;
    const long long v0 = ((long long)blockIdx.x * (kBlock / 32) + (threadIdx.x >> 5)) * a.chunk;
    if (v0 >= a.nnz) return;
    const int vend = (int)min((long long)a.nnz, v0 + a.chunk);
    const int Q = V4 ? a.feat >> 2 : a.feat;
    Cursor cur;
    cur.init(a, (int)v0);
    for (int vb = (int)v0; vb < vend; vb += G) {
        const int v = vb + g;
        const int pos = v < vend ? cur.pos(a, v) : -1;
        float s = 0.f;
        if (pos >= 0) {
            const size_t col = (size_t)ld_stream_s32(a.idx + pos);
            if (V4) {
                const float4 *xr = reinterpret_cast<const float4 *>(a.x_row) + (size_t)cur.row * Q;
                const float4 *xc = reinterpret_cast<const float4 *>(a.x_col) + col * Q;
                for (int q = l; q < Q; q += lanes) fma_dot4(s, __ldg(xr + q), __ldg(xc + q));
            } else {
                const float *xr = a.x_row + (size_t)cur.row * Q;
                const float *xc = a.x_col + col * Q;
                for (int q = l; q < Q; q += lanes) s = fmaf(__ldg(xr + q), __ldg(xc + q), s);
            }
        }
        for (int o = lanes / 2; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
        if (l == 0 && pos >= 0) a.out[pos] = s;
    }
}

// (band, row) segment lengths of the band-major order; len[n_seg] = 0 so that an exclusive scan ends on the total
__global__ void __launch_bounds__(256) band_len_kernel(const int *split, int num_v, long long n_seg, int *len) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i <= n_seg; i += stride)
        len[i] = i < n_seg ? split[i + num_v] - split[i] : 0;
}

int pow2_lanes(int q) {
    int l = 1;
    while (l < q && l < 32) l <<= 1;
    return l;
}

// the fast kernel's shape for K % 4 == 0, K <= 512: lanes = L, vec = float4 per lane (1, 2 or 4), u = entries in flight
struct Shape {
    int lanes, vec, u;
};
Shape fast_shape(int K) {
    const int q = K / 4, l = pow2_lanes(q);
    const int need = (q + l - 1) / l;
    const int vec = need <= 1 ? 1 : need <= 2 ? 2 : 4;
    return {l, vec, vec == 4 ? 2 : 4};
}

template <int LANES, int VEC, int U>
void *fast_fn() {
    return reinterpret_cast<void *>(&sddmm_kernel<LANES, VEC, U>);
}
void *kernel_fn(int K) {
    if (K % 4 != 0) return reinterpret_cast<void *>(&sddmm_generic_kernel<false>);
    if (K > 512) return reinterpret_cast<void *>(&sddmm_generic_kernel<true>);
    const Shape sh = fast_shape(K);
    switch (sh.lanes * 10 + sh.vec) {
        case 11: return fast_fn<1, 1, 4>();
        case 21: return fast_fn<2, 1, 4>();
        case 41: return fast_fn<4, 1, 4>();
        case 81: return fast_fn<8, 1, 4>();
        case 161: return fast_fn<16, 1, 4>();
        case 321: return fast_fn<32, 1, 4>();
        case 322: return fast_fn<32, 2, 4>();
        case 324: return fast_fn<32, 4, 2>();
        default: return nullptr;
    }
}

// First call after preprocess: the band-major prefix (several column blocks; allocated from the pool, freed with the
// plan) and the chunk size from the kernel's occupancy.
int prepare(spmm_b200_handle *h, cudaStream_t stream) {
    Plan &p = h->plan;
    const int K = h->feat;
    if (p.n_col_blocks > 1 && !p.d_sddmm_vp) {
        const long long n_seg = (long long)p.n_col_blocks * h->num_v;
        int *len = nullptr, *vp = nullptr;
        void *tmp = nullptr;
        size_t tmp_bytes = 0;
        SB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, len, vp, (int)(n_seg + 1), stream));
        SB_CUDA(pool_alloc((void **)&vp, sizeof(int) * (size_t)(n_seg + 1), stream));
        cudaError_t e = pool_alloc((void **)&len, sizeof(int) * (size_t)(n_seg + 1), stream);
        if (e == cudaSuccess) e = pool_alloc(&tmp, tmp_bytes, stream);
        if (e == cudaSuccess) {
            const long long blocks = (n_seg + 256) / 256;
            band_len_kernel<<<(unsigned)(blocks < 2048 ? blocks : 2048), 256, 0, stream>>>(p.d_split, h->num_v, n_seg, len);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, len, vp, (int)(n_seg + 1), stream);
        pool_free(tmp, stream);
        pool_free(len, stream);
        if (e != cudaSuccess) {
            pool_free(vp, stream);
            return cuda_fail(e, "sddmm band prefix", __FILE__, __LINE__);
        }
        p.d_sddmm_vp = vp;
    }
    if (p.sddmm_chunk == 0) {
        int per_sm = 0, dev = 0, sms = 0;
        void *fn = kernel_fn(K);
        if (!fn) {
            set_error("spmm_b200_sddmm: no kernel for feat_in = %d", K);
            return SPMM_B200_EINVAL;
        }
        SB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, kBlock, 0));
        SB_CUDA(cudaGetDevice(&dev));
        SB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        const long long warps = (long long)(per_sm > 0 ? per_sm : 1) * (kBlock / 32) * (sms > 0 ? sms : 1);
        long long chunk = (h->num_e + kWaves * warps - 1) / (kWaves * warps);
        if (chunk < kMinChunk) chunk = kMinChunk;
        chunk = (chunk + 127) / 128 * 128;   // whole batches (32 / lanes groups x entries in flight) of every shape
        p.sddmm_chunk = (int)(chunk < 0x40000000ll ? chunk : 0x40000000ll);
    }
    return 0;
}

}  // namespace

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" int spmm_b200_sddmm(spmm_b200_t h, const float *x_row, const float *x_col, float *out, void *stream) {
    if (!h) {
        set_error("spmm_b200_sddmm: null handle");
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.ready) {
        set_error("spmm_b200_sddmm: preprocess has not been called");
        return SPMM_B200_ESTATE;
    }
    if (h->num_e == 0) return 0;
    const int K = h->feat;
    if (!out || (K > 0 && (!x_row || !x_col))) {
        set_error("spmm_b200_sddmm: null x_row / x_col / out");
        return SPMM_B200_EINVAL;
    }
    if (K > 0 && K % 4 == 0 && (((uintptr_t)x_row | (uintptr_t)x_col) & 15)) {
        set_error("spmm_b200_sddmm: x_row / x_col must be 16-byte aligned");
        return SPMM_B200_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    if (K == 0) {
        SB_CUDA(cudaMemsetAsync(out, 0, sizeof(float) * (size_t)h->num_e, s));
        return 0;
    }
    int rc = prepare(h, s);
    if (rc) return rc;
    const Plan &p = h->plan;
    SddmmArgs a;
    const bool banded = p.n_col_blocks > 1;
    a.vp = banded ? p.d_sddmm_vp : h->d_ptr;
    a.start = banded ? p.d_split : h->d_ptr;
    a.idx = h->d_idx;
    a.x_row = x_row;
    a.x_col = x_col;
    a.out = out;
    a.num_v = h->num_v;
    a.n_seg = (banded ? p.n_col_blocks : 1) * h->num_v;
    a.nnz = h->num_e;
    a.feat = K;
    a.chunk = p.sddmm_chunk;
    const long long warps = ((long long)h->num_e + a.chunk - 1) / a.chunk;
    const unsigned grid = (unsigned)((warps + kBlock / 32 - 1) / (kBlock / 32));
    if (K % 4 != 0) {
        sddmm_generic_kernel<false><<<grid, kBlock, 0, s>>>(a, pow2_lanes(K));
    } else if (K > 512) {
        sddmm_generic_kernel<true><<<grid, kBlock, 0, s>>>(a, pow2_lanes(K / 4));
    } else {
        const Shape sh = fast_shape(K);
        switch (sh.lanes * 10 + sh.vec) {
            case 11: sddmm_kernel<1, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 21: sddmm_kernel<2, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 41: sddmm_kernel<4, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 81: sddmm_kernel<8, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 161: sddmm_kernel<16, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 321: sddmm_kernel<32, 1, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 322: sddmm_kernel<32, 2, 4><<<grid, kBlock, 0, s>>>(a); break;
            case 324: sddmm_kernel<32, 4, 2><<<grid, kBlock, 0, s>>>(a); break;
            default:
                set_error("spmm_b200_sddmm: unsupported shape lanes=%d vec=%d", sh.lanes, sh.vec);
                return SPMM_B200_EINVAL;
        }
    }
    SB_CUDA(cudaGetLastError());
    return 0;
}
