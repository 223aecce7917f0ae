// edge_softmax.cu — softmax over each row's nonzeros (spmm_b200_edge_softmax) and its gradient
// (spmm_b200_edge_softmax_backward). With the scores of sddmm(X_dst, X_src) this is the normalisation of dot-product
// graph attention; hpc_b200.GraphAttention chains sddmm -> edge_softmax -> run. Restated on the CPU by
// tests/softmax_oracle.c.
//
// Contract, per row r with nonzeros at CSR positions ptr[r] .. ptr[r+1]-1 (n of them):
//   forward   m = max s[e] (exact in any order); out[e] = exp(s[e] - m) / S, S = sum exp(s[e] - m)
//   backward  d = sum p[e] * dp[e];               ds[e]  = p[e] * (dp[e] - d)
// Special values (forward): a row holding a NaN or +inf is NaN throughout (out = 0x7fffffff); a row whose scores are
// all -inf is 0 throughout (masking; torch.softmax gives NaN there); otherwise a -inf score gives 0.
//
// Order (depends on n alone, so the bits do not change with any plan option, row partition or handle). The row's
// positions are cut into tiles of T = 256. In tile t, lane l of 32 builds a chain from 0.0f over the positions
// t*T + l + 32*j, j = 0..7, that are < n:  forward  c_l = c_l + x (x = exp(s - m), in j order),
//                                          backward c_l = fmaf(p, dp, c_l).
// Then for o = 16, 8, 4, 2, 1 every lane sets c_l = c_l + c_(l xor o); the tile sum is c_0 (every lane holds it).
// The row sum starts from 0.0f and adds the tile sums in tile order. out = x / S is the IEEE-rounded division;
// ds = p * (dp - d) is a rounded subtraction, then a rounded multiply (never contracted). Built -ftz=true: every add,
// FMA, multiply, division and subtraction flushes subnormal inputs and outputs to signed zero.
//
// exp (sm_exp below, restated bit for bit by the oracle) is computed from fmaf, multiplies and integer bit operations,
// not expf / __expf: both end in the hardware's ex2.approx, which a CPU cannot restate. Cody–Waite reduction
// x = k ln2 + r (k = round(x log2 e), ln2 split in a 16-bit head and a tail), a degree-7 Taylor polynomial in Horner
// form (|r| <= 0.35: truncation below 0.13 ulp), then a multiply by 2^k built from exponent bits. Defined for x <= 0:
// exp(0) = exp(-0) = 1 exactly (single-edge rows give 1), -inf and every result below FLT_MIN give +0, and every float
// in [-87.5, 0] is within 2 ulp of the fp64 exp (checked exhaustively by tests/test_edge_softmax_oracle.py).
//
// Work split (rows run from 0 to 154 828 nonzeros on the shapes of hpc_b200/shapes.py), as rows.cuh describes. Rows of
// at most 1024 nonzeros: one warp each, scores kept in registers (HBM reads every input once). Longer rows: one CTA
// each (8 warps take the tiles round-robin, tile sums are folded in tile order through shared memory); the passes
// after the first re-read the row from the L2. No atomics, no workspace, no allocation.
#include <cfloat>
#include <cstdint>

#include "rows.cuh"

namespace spmm_b200 {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kTile = 256;                   // T of the order above
constexpr int kPer = kTile / 32;             // positions per lane per tile
constexpr int kRegTiles = 4;                 // a warp keeps rows of up to kRegTiles tiles in registers
constexpr int kWarpMax = kRegTiles * kTile;  // longer rows go to the CTA path
constexpr int kRound = 64;                   // tile sums folded per round in the CTA path

struct SoftmaxArgs {
    const int *ptr;
    const float *a;   // scores (forward) or p (backward)
    const float *b;   // dp (backward)
    float *out;       // out (forward) or ds (backward)
    int num_v;
    long long chunk;  // rows + nonzeros per warp (warp path)
};

__device__ __forceinline__ float sm_exp(float x) {
    if (x < -88.0f) return 0.0f;   // below FLT_MIN (also -inf)
    const float kf = __fsub_rn(fmaf(x, 1.44269504f, 12582912.0f), 12582912.0f);   // round(x log2 e)
    const int k = (int)kf;
    if (k < -126) return 0.0f;
    float r = fmaf(kf, -0.693145751953125f, x);   // exact: the head has 16 significant bits
    r = fmaf(kf, -1.428606765330187e-6f, r);
    float p = 1.98412698e-4f;   // 1/7!
    p = fmaf(p, r, 1.38888889e-3f);
    p = fmaf(p, r, 8.33333333e-3f);
    p = fmaf(p, r, 4.16666667e-2f);
    p = fmaf(p, r, 1.66666667e-1f);
    p = fmaf(p, r, 0.5f);
    p = fmaf(p, r, 1.0f);
    p = fmaf(p, r, 1.0f);
    const float y = __fmul_rn(p, __int_as_float((k + 127) << 23));
    return y < FLT_MIN ? 0.0f : y;
}

__device__ __forceinline__ float warp_sum(float c) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c = __fadd_rn(c, __shfl_xor_sync(kFull, c, o));
    return c;
}

__device__ __forceinline__ bool is_bad(float x) { return x != x || x == INFINITY; }

// Rows of 1 .. kWarpMax nonzeros, one warp each, in contiguous ranges of about `chunk` rows + nonzeros per warp.
template <bool BWD>
__global__ void __launch_bounds__(kRowBlock) softmax_warp_kernel(const __grid_constant__ SoftmaxArgs a) {
    const int lane = threadIdx.x & 31;
    int r0, r1;
    warp_rows(a, r0, r1);
    int beg = r0 < r1 ? __ldg(a.ptr + r0) : 0;
    for (int r = r0; r < r1; ++r) {
        const int end = __ldg(a.ptr + r + 1);
        const int n = end - beg;
        const float *x = a.a + beg;
        float *out = a.out + beg;
        beg = end;
        if (n == 0 || n > kWarpMax) continue;
        float v[kRegTiles][kPer];
        if (!BWD) {
            float m = -INFINITY;
            bool bad = false;
#pragma unroll
            for (int t = 0; t < kRegTiles; ++t) {
                if (t * kTile >= n) break;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    const int i = t * kTile + j * 32 + lane;
                    v[t][j] = i < n ? __ldcs(x + i) : -INFINITY;
                    m = fmaxf(m, v[t][j]);
                    bad |= is_bad(v[t][j]);
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
            bad = __any_sync(kFull, bad);
            if (bad || m == -INFINITY) {
                const float fill = bad ? __int_as_float(0x7fffffff) : 0.0f;
                for (int i = lane; i < n; i += 32) __stcs(out + i, fill);
                continue;
            }
            float S = 0.0f;
#pragma unroll
            for (int t = 0; t < kRegTiles; ++t) {
                if (t * kTile >= n) break;
                float c = 0.0f;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    if (t * kTile + j * 32 + lane < n) {
                        v[t][j] = sm_exp(__fsub_rn(v[t][j], m));
                        c = __fadd_rn(c, v[t][j]);
                    }
                }
                S = __fadd_rn(S, warp_sum(c));
            }
#pragma unroll
            for (int t = 0; t < kRegTiles; ++t) {
                if (t * kTile >= n) break;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    const int i = t * kTile + j * 32 + lane;
                    if (i < n) __stcs(out + i, __fdiv_rn(v[t][j], S));
                }
            }
        } else {
            const float *dp = a.b + (x - a.a);
            float g[kRegTiles][kPer];
            float D = 0.0f;
#pragma unroll
            for (int t = 0; t < kRegTiles; ++t) {
                if (t * kTile >= n) break;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    const int i = t * kTile + j * 32 + lane;
                    v[t][j] = i < n ? __ldcs(x + i) : 0.0f;
                    g[t][j] = i < n ? __ldcs(dp + i) : 0.0f;
                }
                float c = 0.0f;
#pragma unroll
                for (int j = 0; j < kPer; ++j)
                    if (t * kTile + j * 32 + lane < n) c = fmaf(v[t][j], g[t][j], c);
                D = __fadd_rn(D, warp_sum(c));
            }
#pragma unroll
            for (int t = 0; t < kRegTiles; ++t) {
                if (t * kTile >= n) break;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    const int i = t * kTile + j * 32 + lane;
                    if (i < n) __stcs(out + i, __fmul_rn(v[t][j], __fsub_rn(g[t][j], D)));
                }
            }
        }
    }
}

// Rows of more than kWarpMax nonzeros, one CTA each (the long-row launch of rows.cuh).
template <bool BWD>
__global__ void __launch_bounds__(kRowBlock) softmax_long_kernel(const __grid_constant__ SoftmaxArgs a) {
    __shared__ unsigned long_mask[kRowWarps];
    __shared__ float red_m[kRowWarps];
    __shared__ int red_bad[kRowWarps];
    __shared__ float tsum[kRound];
    __shared__ float total;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for_long_rows(a, kWarpMax, long_mask, [&](int r) {
        const int beg = __ldg(a.ptr + r), n = __ldg(a.ptr + r + 1) - beg;
        const float *x = a.a + beg;
        const float *dp = BWD ? a.b + beg : nullptr;
        float *out = a.out + beg;
        // pass 1 (forward): max and the NaN / +inf flag
        float m = 0.0f;
        if (!BWD) {
            m = -INFINITY;
            int bad = 0;
            for (int i = tid; i < n; i += kRowBlock) {
                const float s = x[i];
                m = fmaxf(m, s);
                bad |= is_bad(s);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(kFull, m, o));
            bad = __any_sync(kFull, bad);
            if (lane == 0) {
                red_m[warp] = m;
                red_bad[warp] = bad;
            }
            __syncthreads();
            for (int k = 0; k < kRowWarps; ++k) {
                m = fmaxf(m, red_m[k]);
                bad |= red_bad[k];
            }
            __syncthreads();
            if (bad || m == -INFINITY) {
                const float fill = bad ? __int_as_float(0x7fffffff) : 0.0f;
                for (int i = tid; i < n; i += kRowBlock) out[i] = fill;
                return;
            }
        }
        // pass 2: tile sums in tile order
        const int nt = (n + kTile - 1) / kTile;
        float S = 0.0f;
        for (int t0 = 0; t0 < nt; t0 += kRound) {
            const int t1 = min(nt, t0 + kRound);
            for (int t = t0 + warp; t < t1; t += kRowWarps) {
                float xa[kPer], xb[kPer];
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    const int i = t * kTile + j * 32 + lane;
                    xa[j] = i < n ? x[i] : 0.0f;
                    if (BWD) xb[j] = i < n ? dp[i] : 0.0f;
                }
                float c = 0.0f;
#pragma unroll
                for (int j = 0; j < kPer; ++j) {
                    if (t * kTile + j * 32 + lane < n)
                        c = BWD ? fmaf(xa[j], xb[j], c) : __fadd_rn(c, sm_exp(__fsub_rn(xa[j], m)));
                }
                c = warp_sum(c);
                if (lane == 0) tsum[t - t0] = c;
            }
            __syncthreads();
            if (tid == 0)
                for (int t = t0; t < t1; ++t) S = __fadd_rn(S, tsum[t - t0]);
            __syncthreads();
        }
        if (tid == 0) total = S;
        __syncthreads();
        S = total;
        // pass 3: outputs
        for (int i = tid; i < n; i += kRowBlock)
            out[i] = BWD ? __fmul_rn(x[i], __fsub_rn(dp[i], S)) : __fdiv_rn(sm_exp(__fsub_rn(x[i], m)), S);
        __syncthreads();   // `total` is rewritten by the next row
    });
}

template <bool BWD>
int launch(spmm_b200_t h, const float *x, const float *y, float *out, cudaStream_t s) {
    RowGrid gr;
    const int rc = row_grid(h->num_v, h->num_e, &gr);
    if (rc) return rc;
    SoftmaxArgs a;
    a.ptr = h->d_ptr;
    a.a = x;
    a.b = y;
    a.out = out;
    a.num_v = h->num_v;
    a.chunk = gr.chunk;
    softmax_warp_kernel<BWD><<<gr.warp_blocks, kRowBlock, 0, s>>>(a);
    SB_CUDA(cudaGetLastError());
    softmax_long_kernel<BWD><<<gr.long_blocks, kRowBlock, 0, s>>>(a);
    SB_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" int spmm_b200_edge_softmax(spmm_b200_t h, const float *scores, float *out, void *stream) {
    if (!h) {
        set_error("spmm_b200_edge_softmax: null handle");
        return SPMM_B200_EINVAL;
    }
    if (h->num_e == 0) return 0;
    if (!scores || !out) {
        set_error("spmm_b200_edge_softmax: null scores / out");
        return SPMM_B200_EINVAL;
    }
    return launch<false>(h, scores, nullptr, out, (cudaStream_t)stream);
}

extern "C" int spmm_b200_edge_softmax_backward(spmm_b200_t h, const float *p, const float *dp, float *ds, void *stream) {
    if (!h) {
        set_error("spmm_b200_edge_softmax_backward: null handle");
        return SPMM_B200_EINVAL;
    }
    if (h->num_e == 0) return 0;
    if (!p || !dp || !ds) {
        set_error("spmm_b200_edge_softmax_backward: null p / dp / ds");
        return SPMM_B200_EINVAL;
    }
    return launch<true>(h, p, dp, ds, (cudaStream_t)stream);
}
