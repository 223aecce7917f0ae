// reduce.cu — amax / amin aggregation over the operator's rows (spmm_b200_reduce) and its gradient on the transposed
// operator (spmm_b200_reduce_backward): the max aggregators of GNN layers (GraphSAGE pooling, PNA, DGL's u_mul_e_max),
// with torch.sparse.mm(A, B, "amax" | "amin") semantics. Restated on the CPU by tests/reduce_oracle.c.
//
// Forward contract, per row r, column j < K and nonzero e of r: the message is m(e, j) = val[e] * vin[idx[e]*K + j],
// one rounded multiply (flush-to-zero build). vout[r*K + j] is the message of the winner, arg[r*K + j] its CSR position.
// The winner is the maximum of a total order on (message, position): a NaN ranks above every number (amax and amin
// alike, so NaN propagates as in torch.amax); among numbers the larger (amax) or smaller (amin) wins; equal values,
// -0 == +0 included, go to the smaller position. Since the order is total, the bits do not depend on how a row is split
// over lanes, warps, CTAs or column-block passes. An empty row gives +0.0f and arg = -1.
//
// Column blocks (several column blocks imply ascending columns in every row): pass b walks the positions
// [split[b][r], split[b+1][r]) and gathers only band b of B, which stays in the L2. A pass whose row already holds a
// winner from earlier bands (split[b][r] > ptr[r]) replaces it only when its own winner is strictly better, or a NaN
// replacing a number: its positions are all larger, so that keeps the tie rule without reading arg.
//
// Backward contract (on t = the transposed handle): with Aᵀ row c holding entries k in storage order (ascending row of
// A), e = perm[k], r = t_idx[k], entry k matches column j when arg[r*K + j] == e.
//   db[c, j]: the row is cut into tiles of kTile consecutive entries; a tile computes s = fmaf(val[e], dc[r*K + j], s)
//             from 0.0f over its matching entries in order (the others are skipped); db = 0.0f + tile sums, in tile
//             order. The order depends on the length of the Aᵀ row alone; rows nothing matches give +0.0f.
//   dval[e]:  sddmm's order (sddmm.cu) with x_row = dc[r], x_col = vin[c], the terms of non-matching columns skipped.
// No atomics: every element of db belongs to one Aᵀ row and every e to one entry, so each is written once, and the sums
// are bit-reproducible like every other kernel of the library.
//
// Work split (forward and backward alike): lane groups of L lanes cover one slice of the columns (L lanes x VEC units
// of W = 4 or 1 columns, the lane shape of sddmm); K % 4 == 0 and K <= 512 is one slice, wider or scalar K loops over
// slices. dval's bits rely on L being sddmm's: both take it from pow2_lanes / fast_lane_shape (common.h). Rows are split
// as rows.cuh describes, at kWarpMax (forward) and kBwdWarpMax (backward) nonzeros. Forward: the 32 / L groups of a warp
// take interleaved nonzeros of one row, keep a running (value, position) per column in registers and fold with
// shuffles. Backward: the groups take different rows of Aᵀ, since each tile is one in-order chain. Long rows, one CTA
// each: forward warps interleave nonzeros and fold through shared memory; backward lane groups take whole tiles
// round-robin and the tile sums are added in tile order through shared memory. Built -ftz=true. No atomics, no
// workspace, no allocation.
#include <cstdint>

#include "rows.cuh"

namespace spmm_b200 {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kWarpMax = 2048;          // forward: rows with more nonzeros go to the CTA path
constexpr int kTile = 1024;             // T of the backward order (tests/reduce_oracle.c: REDUCE_TILE)
constexpr int kBwdWarpMax = 4 * kTile;  // backward: longer Aᵀ rows go to the CTA path
constexpr int kMaxSlice = 512;          // columns per slice at most (32 lanes x 4 float4)

struct ReduceArgs {
    const int *ptr, *idx;
    const float *val, *vin;
    float *vout;
    int *arg;               // NULL: values only
    const int *s0, *s1;     // this pass's range in row r: [s0[r], s1[r]) (ptr, ptr + 1 with one column block)
    int band, num_v, feat, lanes, n_slices;
    bool amax;
    long long chunk;        // rows + nonzeros per warp
};

struct BwdArgs {
    const int *ptr, *idx, *perm;   // Aᵀ
    const float *val;              // the source handle's live values, indexed by e = perm[k]
    const float *dc, *vin;
    const int *arg;
    float *db, *dval;              // either may be NULL
    int num_v, feat, lanes, n_slices;
    long long chunk;
};

template <int W>
__device__ __forceinline__ void ldf(float (&d)[W], const float *base, size_t unit) {
    if constexpr (W == 4) {
        const float4 f = __ldg(reinterpret_cast<const float4 *>(base) + unit);
        d[0] = f.x, d[1] = f.y, d[2] = f.z, d[3] = f.w;
    } else {
        d[0] = __ldg(base + unit);
    }
}

template <int W>
__device__ __forceinline__ void ldi(int (&d)[W], const int *base, size_t unit) {
    if constexpr (W == 4) {
        const int4 f = __ldg(reinterpret_cast<const int4 *>(base) + unit);
        d[0] = f.x, d[1] = f.y, d[2] = f.z, d[3] = f.w;
    } else {
        d[0] = __ldg(base + unit);
    }
}

template <int W>
__device__ __forceinline__ void stf(float *base, size_t unit, const float (&d)[W]) {
    if constexpr (W == 4) reinterpret_cast<float4 *>(base)[unit] = make_float4(d[0], d[1], d[2], d[3]);
    else base[unit] = d[0];
}

template <int W>
__device__ __forceinline__ void sti(int *base, size_t unit, const int (&d)[W]) {
    if constexpr (W == 4) reinterpret_cast<int4 *>(base)[unit] = make_int4(d[0], d[1], d[2], d[3]);
    else base[unit] = d[0];
}

// m, at a larger position than the current winner v, replaces it
__device__ __forceinline__ bool later_wins(float m, float v, bool amax) {
    return (m != m && v == v) || (amax ? m > v : m < v);
}

// the total order: (v1, p1) ranks above (v2, p2); p < 0 is "no entry" and ranks below everything
__device__ __forceinline__ bool beats(float v1, int p1, float v2, int p2, bool amax) {
    if (p2 < 0) return p1 >= 0;
    if (p1 < 0) return false;
    const bool n1 = v1 != v1, n2 = v2 != v2;
    if (n1 != n2) return n1;
    if (!n1 && v1 != v2) return amax ? v1 > v2 : v1 < v2;
    return p1 < p2;
}

// ---- forward ---------------------------------------------------------------------------------------------------

// One lane group's walk over the positions first, first + step, ... of [pb, pe) for the slice starting at column unit
// u0 (+ the lane's units l + v*L): the running winner per column. p = -1 where the group met no entry.
template <int W, int VEC, int U>
__device__ __forceinline__ void fwd_walk(const ReduceArgs &a, int pb, int pe, int first, int step, size_t u0,
                                         const bool (&ok)[VEC], float (&v)[VEC][W], int (&p)[VEC][W]) {
    const int L = a.lanes;
    const size_t row_units = (size_t)(a.feat / W);
#pragma unroll
    for (int i = 0; i < VEC; ++i)
#pragma unroll
        for (int t = 0; t < W; ++t) v[i][t] = 0.0f, p[i][t] = -1;
    bool have = false;
    for (int e0 = pb + first; e0 < pe; e0 += step * U) {
        int col[U];
        float w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int e = e0 + u * step;
            col[u] = e < pe ? __ldg(a.idx + e) : -1;
            w[u] = e < pe ? __ldg(a.val + e) : 0.0f;
        }
        float b[U][VEC][W];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < VEC; ++i)
                if (col[u] >= 0 && ok[i]) ldf<W>(b[u][i], a.vin, (size_t)col[u] * row_units + u0 + i * L);
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (col[u] < 0) continue;
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                if (!ok[i]) continue;
#pragma unroll
                for (int t = 0; t < W; ++t) {
                    const float m = __fmul_rn(w[u], b[u][i][t]);
                    if (!have || later_wins(m, v[i][t], a.amax)) v[i][t] = m, p[i][t] = e0 + u * step;
                }
            }
            have = true;
        }
    }
}

// Stores one unit (W columns) of a row's result for this pass: unconditionally (first band, or no earlier entry), or,
// when the row holds a winner from earlier bands, only where this pass's winner is strictly better.
template <int W>
__device__ __forceinline__ void fwd_store(const ReduceArgs &a, size_t unit, const float (&v)[W], const int (&p)[W],
                                          bool combine) {
    if (!combine) {
        stf<W>(a.vout, unit, v);
        if (a.arg) sti<W>(a.arg, unit, p);
        return;
    }
#pragma unroll
    for (int t = 0; t < W; ++t) {
        const size_t o = unit * W + t;
        if (later_wins(v[t], a.vout[o], a.amax)) {
            a.vout[o] = v[t];
            if (a.arg) a.arg[o] = p[t];
        }
    }
}

// +0.0f / -1 for the units u0 + l, u0 + l + L, ... < end of an empty row
template <int W>
__device__ __forceinline__ void fwd_store_empty(const ReduceArgs &a, size_t u0, size_t end, int l, int L) {
    float z[W];
    int m[W];
#pragma unroll
    for (int t = 0; t < W; ++t) z[t] = 0.0f, m[t] = -1;
    for (size_t u = u0 + l; u < end; u += L) {
        stf<W>(a.vout, u, z);
        if (a.arg) sti<W>(a.arg, u, m);
    }
}

template <int W, int VEC>
__device__ __forceinline__ void fold_groups(float (&v)[VEC][W], int (&p)[VEC][W], int L, bool amax) {
    for (int o = L; o < 32; o <<= 1) {
#pragma unroll
        for (int i = 0; i < VEC; ++i)
#pragma unroll
            for (int t = 0; t < W; ++t) {
                const float ov = __shfl_xor_sync(kFull, v[i][t], o);
                const int op = __shfl_xor_sync(kFull, p[i][t], o);
                if (beats(ov, op, v[i][t], p[i][t], amax)) v[i][t] = ov, p[i][t] = op;
            }
    }
}

// Rows of at most kWarpMax nonzeros: one warp per row of its range, the groups interleaving the row's nonzeros.
template <int W, int VEC, int U>
__global__ void __launch_bounds__(kRowBlock) reduce_warp_kernel(const __grid_constant__ ReduceArgs a) {
    const int lane = threadIdx.x & 31, L = a.lanes, G = 32 / L;
    const int l = lane % L, g = lane / L;
    int r0, r1;
    warp_rows(a, r0, r1);
    const size_t row_units = (size_t)(a.feat / W);
    const int slice_units = L * VEC;
    for (int r = r0; r < r1; ++r) {
        const int rb = __ldg(a.ptr + r);
        if (__ldg(a.ptr + r + 1) - rb > kWarpMax) continue;
        const int pb = __ldg(a.s0 + r), pe = __ldg(a.s1 + r);
        if (pb == pe) {
            if (a.band == 0 && g == 0) fwd_store_empty<W>(a, (size_t)r * row_units, (size_t)(r + 1) * row_units, l, L);
            continue;
        }
        const bool combine = a.band > 0 && pb > rb;
        for (int s = 0; s < a.n_slices; ++s) {
            const size_t u0 = (size_t)s * slice_units + l;
            bool ok[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) ok[i] = u0 + i * L < row_units;
            float v[VEC][W];
            int p[VEC][W];
            fwd_walk<W, VEC, U>(a, pb, pe, g, G, u0, ok, v, p);
            fold_groups<W, VEC>(v, p, L, a.amax);
            if (g == 0) {
#pragma unroll
                for (int i = 0; i < VEC; ++i)
                    if (ok[i]) fwd_store<W>(a, (size_t)r * row_units + u0 + i * L, v[i], p[i], combine);
            }
        }
    }
}

// Rows of more than kWarpMax nonzeros, one CTA each (the long-row launch of rows.cuh). The warps interleave the row's
// nonzeros; their winners meet in shared memory.
template <int W, int VEC, int U>
__global__ void __launch_bounds__(kRowBlock) reduce_long_kernel(const __grid_constant__ ReduceArgs a) {
    __shared__ unsigned long_mask[kRowWarps];
    __shared__ float red_v[kRowWarps][kMaxSlice];
    __shared__ int red_p[kRowWarps][kMaxSlice];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, L = a.lanes, G = 32 / L;
    const int l = lane % L, g = lane / L;
    const size_t row_units = (size_t)(a.feat / W);
    const int slice_units = L * VEC;
    for_long_rows(a, kWarpMax, long_mask, [&](int r) {
        const int rb = __ldg(a.ptr + r);
        const int pb = __ldg(a.s0 + r), pe = __ldg(a.s1 + r);
        if (pb == pe) {
            if (a.band == 0) fwd_store_empty<W>(a, (size_t)r * row_units, (size_t)(r + 1) * row_units, tid, kRowBlock);
            return;
        }
        const bool combine = a.band > 0 && pb > rb;
        for (int s = 0; s < a.n_slices; ++s) {
            const size_t u0 = (size_t)s * slice_units + l;
            bool ok[VEC];
#pragma unroll
            for (int i = 0; i < VEC; ++i) ok[i] = u0 + i * L < row_units;
            float v[VEC][W];
            int p[VEC][W];
            fwd_walk<W, VEC, U>(a, pb, pe, warp * G + g, kRowWarps * G, u0, ok, v, p);
            fold_groups<W, VEC>(v, p, L, a.amax);
            if (g == 0) {
#pragma unroll
                for (int i = 0; i < VEC; ++i)
#pragma unroll
                    for (int t = 0; t < W; ++t) {
                        const int j = (l + i * L) * W + t;   // column inside the slice
                        red_v[warp][j] = v[i][t];
                        red_p[warp][j] = p[i][t];
                    }
            }
            __syncthreads();
            const int cols = slice_units * W;
            const size_t c0 = (size_t)s * cols;
            for (int j = tid; j < cols && c0 + j < (size_t)a.feat; j += kRowBlock) {
                float bv = red_v[0][j];
                int bp = red_p[0][j];
                for (int k = 1; k < kRowWarps; ++k)
                    if (beats(red_v[k][j], red_p[k][j], bv, bp, a.amax)) bv = red_v[k][j], bp = red_p[k][j];
                const size_t o = (size_t)r * a.feat + c0 + j;
                if (!combine || later_wins(bv, a.vout[o], a.amax)) {
                    a.vout[o] = bv;
                    if (a.arg) a.arg[o] = bp;
                }
            }
            __syncthreads();   // red_v / red_p are rewritten by the next slice or row
        }
    });
}

// ---- backward --------------------------------------------------------------------------------------------------

// One tile [kb, ke) of an Aᵀ row c, for the slice at unit u0 (+ the lane's units l + v*L): s = the tile's chain per
// column (db). With x (vin[c]'s slice, the whole row: one slice) also dval of every entry, in sddmm's order over the
// group's L lanes (gmask); that order holds only while layout() takes L from sddmm's lane rule (common.h).
template <int W, int VEC, int U>
__device__ __forceinline__ void bwd_tile(const BwdArgs &a, int kb, int ke, size_t u0, const bool (&ok)[VEC],
                                         float (&s)[VEC][W], const float (&x)[VEC][W], bool with_dval, int l,
                                         unsigned gmask) {
    const int L = a.lanes;
    const size_t row_units = (size_t)(a.feat / W);
#pragma unroll
    for (int i = 0; i < VEC; ++i)
#pragma unroll
        for (int t = 0; t < W; ++t) s[i][t] = 0.0f;
    for (int k0 = kb; k0 < ke; k0 += U) {
        int e[U], r[U];
        float w[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int k = k0 + u;
            e[u] = k < ke ? __ldg(a.perm + k) : -1;
            r[u] = k < ke ? __ldg(a.idx + k) : 0;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) w[u] = e[u] >= 0 ? __ldg(a.val + e[u]) : 0.0f;
        int am[U][VEC][W];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                if (e[u] >= 0 && ok[i]) ldi<W>(am[u][i], a.arg, (size_t)r[u] * row_units + u0 + i * L);
                else
#pragma unroll
                    for (int t = 0; t < W; ++t) am[u][i][t] = -1;
            }
        float d[U][VEC][W];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int i = 0; i < VEC; ++i)
#pragma unroll
                for (int t = 0; t < W; ++t)
                    d[u][i][t] = am[u][i][t] == e[u] && e[u] >= 0
                                     ? __ldg(a.dc + ((size_t)r[u] * row_units + u0 + i * L) * W + t) : 0.0f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (e[u] < 0) continue;   // uniform over the group
            float sd = 0.0f;
#pragma unroll
            for (int i = 0; i < VEC; ++i)
#pragma unroll
                for (int t = 0; t < W; ++t)
                    if (am[u][i][t] == e[u]) {
                        s[i][t] = fmaf(w[u], d[u][i][t], s[i][t]);
                        sd = fmaf(d[u][i][t], x[i][t], sd);
                    }
            if (with_dval) {
                for (int o = L / 2; o > 0; o >>= 1) sd += __shfl_xor_sync(gmask, sd, o);
                if (l == 0) a.dval[e[u]] = sd;
            }
        }
    }
}

// dval of the entries first, first + step, ... of [kb, ke) of Aᵀ row c when K spans several slices: sddmm's order over
// the group's L lanes, each lane walking all its units.
template <int W>
__device__ __forceinline__ void bwd_dval_walk(const BwdArgs &a, int c, int kb, int ke, int first, int step, int l,
                                              unsigned gmask) {
    const int L = a.lanes;
    const size_t row_units = (size_t)(a.feat / W);
    const float *xc = a.vin + (size_t)c * a.feat;
    for (int k = kb + first; k < ke; k += step) {
        const int e = __ldg(a.perm + k);
        const size_t r = (size_t)__ldg(a.idx + k);
        float sd = 0.0f;
        for (size_t q = l; q < row_units; q += L) {
            int am[W];
            ldi<W>(am, a.arg, r * row_units + q);
#pragma unroll
            for (int t = 0; t < W; ++t)
                if (am[t] == e) sd = fmaf(__ldg(a.dc + (r * row_units + q) * W + t), __ldg(xc + q * W + t), sd);
        }
        for (int o = L / 2; o > 0; o >>= 1) sd += __shfl_xor_sync(gmask, sd, o);
        if (l == 0) a.dval[e] = sd;
    }
}

// Aᵀ rows of at most kBwdWarpMax entries: the warp's groups take the rows of its range round-robin, each row walked
// tile by tile by one group.
template <int W, int VEC, int U>
__global__ void __launch_bounds__(kRowBlock) reduce_bwd_warp_kernel(const __grid_constant__ BwdArgs a) {
    const int lane = threadIdx.x & 31, L = a.lanes, G = 32 / L;
    const int l = lane % L, g = lane / L;
    const unsigned gmask = L == 32 ? kFull : ((1u << L) - 1) << (g * L);
    int r0, r1;
    warp_rows(a, r0, r1);
    const size_t row_units = (size_t)(a.feat / W);
    const int slice_units = L * VEC;
    const bool fused = a.n_slices == 1;
    for (int c = r0 + g; c < r1; c += G) {
        const int kb = __ldg(a.ptr + c), ke = __ldg(a.ptr + c + 1);
        if (ke - kb > kBwdWarpMax) continue;
        if (a.db || (fused && a.dval)) {
            for (int s = 0; s < a.n_slices; ++s) {
                const size_t u0 = (size_t)s * slice_units + l;
                bool ok[VEC];
                float x[VEC][W], tot[VEC][W], ts[VEC][W];
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    ok[i] = u0 + i * L < row_units;
#pragma unroll
                    for (int t = 0; t < W; ++t) x[i][t] = 0.0f, tot[i][t] = 0.0f;
                    if (ok[i] && fused && a.dval) ldf<W>(x[i], a.vin, (size_t)c * row_units + u0 + i * L);
                }
                for (int tb = kb; tb < ke; tb += kTile) {
                    bwd_tile<W, VEC, U>(a, tb, min(ke, tb + kTile), u0, ok, ts, x, fused && a.dval, l, gmask);
#pragma unroll
                    for (int i = 0; i < VEC; ++i)
#pragma unroll
                        for (int t = 0; t < W; ++t) tot[i][t] = __fadd_rn(tot[i][t], ts[i][t]);
                }
                if (a.db)
#pragma unroll
                    for (int i = 0; i < VEC; ++i)
                        if (ok[i]) stf<W>(a.db, (size_t)c * row_units + u0 + i * L, tot[i]);
            }
        }
        if (a.dval && !fused) bwd_dval_walk<W>(a, c, kb, ke, 0, 1, l, gmask);
    }
}

// Aᵀ rows of more than kBwdWarpMax entries, one CTA each (the long-row launch of rows.cuh). The CTA's lane groups take
// the tiles round-robin, kRowWarps * G tiles per round; the tile sums of a round are added in tile order through shared
// memory.
template <int W, int VEC, int U>
__global__ void __launch_bounds__(kRowBlock, 1) reduce_bwd_long_kernel(const __grid_constant__ BwdArgs a) {
    constexpr int kSumCols = kRowWarps * 32 * VEC * W;   // workers (kRowWarps * G) x slice columns (L * VEC * W)
    __shared__ unsigned long_mask[kRowWarps];
    __shared__ float tsum[kSumCols];
    __shared__ float acc[kMaxSlice];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, L = a.lanes, G = 32 / L;
    const int l = lane % L, g = lane / L;
    const int worker = warp * G + g, n_workers = kRowWarps * G;
    const unsigned gmask = L == 32 ? kFull : ((1u << L) - 1) << (g * L);
    const size_t row_units = (size_t)(a.feat / W);
    const int slice_units = L * VEC, cols = slice_units * W;
    const bool fused = a.n_slices == 1;
    for_long_rows(a, kBwdWarpMax, long_mask, [&](int c) {
        const int kb = __ldg(a.ptr + c), ke = __ldg(a.ptr + c + 1);
        const int nt = (ke - kb + kTile - 1) / kTile;
        if (a.db || (fused && a.dval)) {
            for (int s = 0; s < a.n_slices; ++s) {
                const size_t u0 = (size_t)s * slice_units + l;
                const size_t c0 = (size_t)s * cols;
                bool ok[VEC];
                float x[VEC][W], ts[VEC][W];
#pragma unroll
                for (int i = 0; i < VEC; ++i) {
                    ok[i] = u0 + i * L < row_units;
#pragma unroll
                    for (int t = 0; t < W; ++t) x[i][t] = 0.0f;
                    if (ok[i] && fused && a.dval) ldf<W>(x[i], a.vin, (size_t)c * row_units + u0 + i * L);
                }
                for (int j = tid; j < cols; j += kRowBlock) acc[j] = 0.0f;
                for (int t0 = 0; t0 < nt; t0 += n_workers) {
                    const int t = t0 + worker;
                    if (t < nt) {
                        bwd_tile<W, VEC, U>(a, kb + t * kTile, min(ke, kb + (t + 1) * kTile), u0, ok, ts, x,
                                            fused && a.dval, l, gmask);
#pragma unroll
                        for (int i = 0; i < VEC; ++i)
#pragma unroll
                            for (int q = 0; q < W; ++q) tsum[worker * cols + (l + i * L) * W + q] = ts[i][q];
                    }
                    __syncthreads();
                    const int n_here = min(n_workers, nt - t0);
                    for (int j = tid; j < cols; j += kRowBlock)
                        for (int k = 0; k < n_here; ++k) acc[j] = __fadd_rn(acc[j], tsum[k * cols + j]);
                    __syncthreads();
                }
                if (a.db)
                    for (int j = tid; j < cols && c0 + j < (size_t)a.feat; j += kRowBlock)
                        a.db[(size_t)c * a.feat + c0 + j] = acc[j];
                __syncthreads();   // acc is reset by the next slice or row
            }
        }
        if (a.dval && !fused) bwd_dval_walk<W>(a, c, kb, ke, worker, n_workers, l, gmask);
    });
}

// ---- host --------------------------------------------------------------------------------------------------------

// The lane shape: W columns per unit, L lanes, VEC units per lane and slice. L is sddmm's (common.h), which dval's bits
// rely on. K % 4 == 0, K <= 512: sddmm's fast shape (one slice); K % 4 == 0, K > 512: 32 lanes x 4 float4; K % 4 != 0:
// sddmm's scalar lane count, 4 columns per lane.
struct Layout {
    int w, lanes, vec, n_slices;
};
Layout layout(int K) {
    Layout s;
    if (K % 4 == 0 && K <= 512) {
        const LaneShape f = fast_lane_shape(K);
        s = {4, f.lanes, f.vec, 1};
    } else if (K % 4 == 0) {
        s = {4, pow2_lanes(K / 4), 4, 0};
    } else {
        s = {1, pow2_lanes(K), 4, 0};
    }
    const int cols = s.lanes * s.vec * s.w;
    s.n_slices = (K + cols - 1) / cols;
    return s;
}

template <int W, int VEC, int U>
void launch_fwd(const ReduceArgs &a, const RowGrid &gr, cudaStream_t s) {
    reduce_warp_kernel<W, VEC, U><<<gr.warp_blocks, kRowBlock, 0, s>>>(a);
    reduce_long_kernel<W, VEC, U><<<gr.long_blocks, kRowBlock, 0, s>>>(a);
}

template <int W, int VEC, int U>
void launch_bwd(const BwdArgs &a, const RowGrid &gr, cudaStream_t s) {
    reduce_bwd_warp_kernel<W, VEC, U><<<gr.warp_blocks, kRowBlock, 0, s>>>(a);
    reduce_bwd_long_kernel<W, VEC, U><<<gr.long_blocks, kRowBlock, 0, s>>>(a);
}

// the four instantiations: (W, VEC) = (4, 1), (4, 2), (4, 4), (1, 4); U = entries in flight per lane group
template <class F1, class F2, class F4, class FS>
int dispatch(const Layout &ly, F1 f1, F2 f2, F4 f4, FS fs) {
    if (ly.w == 1) fs();
    else if (ly.vec == 1) f1();
    else if (ly.vec == 2) f2();
    else f4();
    SB_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" int spmm_b200_reduce(spmm_b200_t h, int op, const float *vin, float *vout, int *arg, void *stream) {
    if (!h) {
        set_error("spmm_b200_reduce: null handle");
        return SPMM_B200_EINVAL;
    }
    if (op != SPMM_B200_REDUCE_AMAX && op != SPMM_B200_REDUCE_AMIN) {
        set_error("spmm_b200_reduce: op must be SPMM_B200_REDUCE_AMAX or SPMM_B200_REDUCE_AMIN, got %d", op);
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.ready) {
        set_error("spmm_b200_reduce: preprocess has not been called");
        return SPMM_B200_ESTATE;
    }
    const int K = h->feat;
    if (K == 0 || h->num_v == 0) return 0;
    if (!vout || (h->num_e > 0 && !vin)) {
        set_error("spmm_b200_reduce: null vin / vout");
        return SPMM_B200_EINVAL;
    }
    if (K % 4 == 0 && (((uintptr_t)vin | (uintptr_t)vout | (uintptr_t)arg) & 15)) {
        set_error("spmm_b200_reduce: vin / vout / arg must be 16-byte aligned");
        return SPMM_B200_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const Layout ly = layout(K);
    RowGrid gr;
    int rc = row_grid(h->num_v, h->num_e, &gr);
    if (rc) return rc;
    const Plan &p = h->plan;
    const int nb = p.n_col_blocks > 1 ? p.n_col_blocks : 1;
    ReduceArgs a;
    a.ptr = h->d_ptr;
    a.idx = h->d_idx;
    a.val = h->d_val;
    a.vin = vin;
    a.vout = vout;
    a.arg = arg;
    a.num_v = h->num_v;
    a.feat = K;
    a.lanes = ly.lanes;
    a.n_slices = ly.n_slices;
    a.amax = op == SPMM_B200_REDUCE_AMAX;
    a.chunk = gr.chunk;
    for (int b = 0; b < nb; ++b) {
        a.band = b;
        a.s0 = nb > 1 ? p.d_split + (size_t)b * h->num_v : h->d_ptr;
        a.s1 = nb > 1 ? p.d_split + (size_t)(b + 1) * h->num_v : h->d_ptr + 1;
        rc = dispatch(ly, [&] { launch_fwd<4, 1, 4>(a, gr, s); }, [&] { launch_fwd<4, 2, 4>(a, gr, s); },
                      [&] { launch_fwd<4, 4, 2>(a, gr, s); }, [&] { launch_fwd<1, 4, 4>(a, gr, s); });
        if (rc) return rc;
    }
    return 0;
}

extern "C" int spmm_b200_reduce_backward(spmm_b200_t t, const float *dc, const int *arg, const float *vin, float *db,
                                         float *dval, void *stream) {
    if (!t) {
        set_error("spmm_b200_reduce_backward: null handle");
        return SPMM_B200_EINVAL;
    }
    if (!t->t_ptr || !t->t_src || !t->t_perm) {
        set_error("spmm_b200_reduce_backward: the handle is not a transposed operator (spmm_b200_create_transposed)");
        return SPMM_B200_EINVAL;
    }
    const int K = t->feat;
    if (t->t_src->feat != K) {
        set_error("spmm_b200_reduce_backward: feat_in %d of the transposed operator differs from the source's %d", K,
                  t->t_src->feat);
        return SPMM_B200_EINVAL;
    }
    if (K == 0 || t->num_v == 0 || (!db && !dval)) return 0;
    if ((t->num_e > 0 && (!dc || !arg)) || (dval && t->num_e > 0 && !vin)) {
        set_error("spmm_b200_reduce_backward: null dc / arg, or null vin with dval");
        return SPMM_B200_EINVAL;
    }
    if (K % 4 == 0 && (((uintptr_t)dc | (uintptr_t)arg | (uintptr_t)vin | (uintptr_t)db) & 15)) {
        set_error("spmm_b200_reduce_backward: dc / arg / vin / db must be 16-byte aligned");
        return SPMM_B200_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    const Layout ly = layout(K);
    RowGrid gr;
    int rc = row_grid(t->num_v, t->num_e, &gr);
    if (rc) return rc;
    BwdArgs a;
    a.ptr = t->t_ptr;
    a.idx = t->t_idx;
    a.perm = t->t_perm;
    a.val = t->t_src->d_val;
    a.dc = dc;
    a.vin = vin;
    a.arg = arg;
    a.db = db;
    a.dval = t->num_e > 0 ? dval : nullptr;
    a.num_v = t->num_v;
    a.feat = K;
    a.lanes = ly.lanes;
    a.n_slices = ly.n_slices;
    a.chunk = gr.chunk;
    if (!a.db && !a.dval) return 0;
    return dispatch(ly, [&] { launch_bwd<4, 1, 4>(a, gr, s); }, [&] { launch_bwd<4, 2, 4>(a, gr, s); },
                    [&] { launch_bwd<4, 4, 2>(a, gr, s); }, [&] { launch_bwd<1, 4, 4>(a, gr, s); });
}
