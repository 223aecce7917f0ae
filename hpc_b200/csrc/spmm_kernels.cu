// spmm_kernels.cu — sm_100a kernels of the CSR SpMM engine.
//
// Replaces spmm_kernel_ref (PA4/handout/src/spmm_ref.cu:3-17: one thread per row, serial over
// K and over the row) and the student's SpmmOptKernel (PA4/workspace/src/spmm_opt.cu:9-35:
// one CTA per <=256-nnz task, atomicAdd into a pre-zeroed vout).
//
//   spmm_kernel        one launch per column block (two, one per row half, with two-stream launches), one warp task per
//                      warp: heavy segments and light-row stream tasks in the order the plan schedules them.
//     light stream     rows kept whole are packed (header + {col,val} entries) into a stream panel cut into
//                      equal-sized warp tasks; LANES lanes cooperate on one row, each owning VEC float4 of the
//                      feature slice, so a warp walks 32/LANES interleaved lanes of rows at once. The task's
//                      panel is staged into shared memory with 1-D TMA (cp.async.bulk + mbarrier, double
//                      buffered); B rows are gathered with 128-bit loads that stay in flight across row
//                      boundaries; every output element is one in-order FMA chain from 0.0f in CSR order — the
//                      same chain as spmm_ref.cu:10-14 — so these rows are bit-identical to the reference.
//     heavy segments   rows longer than seg_len are cut into nnz-balanced segments (one warp each), staged the
//                      same way; the 32/LANES lane groups take alternate nonzeros and are combined by warp
//                      shuffles; the warp finishing a row's last segment adds the partial rows in segment
//                      order (deterministic, no float atomics, vout never needs pre-zeroing).
//   spmm_scalar_kernel K % 4 != 0 fallback: warp per row, scalar lanes over the columns, same chain.
//
// fp32 CUDA cores only: SpMM is a gather, not a dense contraction.
#include <stdio.h>

#include "common.h"

namespace spmm_b200 {

namespace {

constexpr unsigned kFull = 0xffffffffu;
constexpr int kChunk = 128;   // panel entries per TMA stage (1 KB)
constexpr int kStages = 2;

// ---- memory helpers ------------------------------------------------------------------------

// col/val are streamed exactly once per slice: keep them out of L1 so B rows stay there.
__device__ __forceinline__ int ld_stream_s32(const int *p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ float ld_stream_f32(const float *p) {
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_c_row(float *p, const float4 &v) {
    __stcs(reinterpret_cast<float4 *>(p), v);
}
// A finished C row piece. Passes that are not the last keep the suspended chain in vout; the final pass stores the
// row to cfinal (vout, or run_host's pinned host buffer) and, in stacked-layer mode, to every rank's copy of the next
// layer's B — one multimem.st through the NVLS multicast address when there is one, else one st.global per
// peer-mapped buffer.
__device__ __forceinline__ void st_final(const CommonArgs &c, bool final, int row, int col, const float4 &v) {
    if (!final) {
        st_c_row(c.vout + (size_t)row * c.feat + col, v);
        return;
    }
    st_c_row(c.cfinal + (size_t)row * c.feat + col, v);
    if (c.n_gather) {
        const size_t off = (size_t)(c.gather_row0 + row) * c.feat + col;
        if (c.gather_mc) {
            asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(c.gather_mc + off), "f"(v.x),
                         "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
        } else {
            for (int t = 0; t < c.n_gather; ++t) *reinterpret_cast<float4 *>(c.gather[t] + off) = v;
        }
    }
}
__device__ __forceinline__ void fma4(float4 &acc, const float4 &b, float v) {
    acc.x = fmaf(b.x, v, acc.x);
    acc.y = fmaf(b.y, v, acc.y);
    acc.z = fmaf(b.z, v, acc.z);
    acc.w = fmaf(b.w, v, acc.w);
}

__device__ __forceinline__ uint32_t smem_u32(const void *p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
                 "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(smem_u32(bar)), "r"(parity)
            : "memory");
    } while (!done);
}
// 1-D TMA: global -> shared, completion counted in bytes on the mbarrier.
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, uint32_t bytes,
                                             uint64_t *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
            "r"(smem_u32(dst)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// ---- the SpMM kernel ------------------------------------------------------------------------
//
// Warp tasks (equal-sized, TMA-staged spans of a {col,val} panel) are either light-stream tasks or heavy segments, in
// the order the plan wants them scheduled. spmm_kernel runs one task per warp, scheduled by the hardware; a launch
// covers one column block (or one row half of it, with two-stream launches), and a later block's pass continues the
// chains the earlier one left in C because the launches over the same rows are ordered on one stream.
//
// TUNE selects the gathers kept in flight per lane group and the register cap (option "tune";
// measurements in profiles/r01_sweep.md):
//   0: 4 gathers in flight per lane group: <= 64 registers when a lane owns one float4 (4 CTAs of 256 threads
//      per SM), <= 80 when it owns two (K >= 256; 3 CTAs/SM)                                     [default]
//   1: 2 gathers in flight, <= 64 registers
// Measured and dropped: 8 in flight at K < 256; 2/VEC at 48 registers (spills); L1::no_allocate or
// L2::evict_last on B rows; gathering B rows into a shared-memory ring with cp.async or with one 1-D TMA copy
// per row (both ~35 % slower than register gathers on every shape).
// FULL: every lane's columns are inside the slice (K a multiple of the slice width): no column predicates.
// LIVE (option "live_values"): a staged entry's .y word is the nonzero's position p and the weight is c.val[p], loaded in
// the same batch as the entry's B-row gather (both depend on the staged entry alone). Headers and nops load nothing.
template <int TUNE, int VEC>
struct Tune {
    static constexpr int kMinBlocks = (TUNE == 0 && VEC == 2) ? 3 : 4;
    static constexpr int kUnroll = TUNE == 1 ? 2 : 4;   // gathers in flight per lane group
};

// A warp's staging pipeline: kStages chunks of shared memory, one mbarrier each, initialised by the warp before its
// task. The task waits for chunk k on stage k % kStages with phase parity (k / kStages) & 1: the barriers start in
// phase 0, and a warp runs exactly one task, so they are never reused.
struct Pipe {
    int2 *buf;
    uint64_t *bars;
};
__device__ __forceinline__ void pipe_init(const Pipe &p, int lane) {
    if (lane == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) mbar_init(&p.bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
}
// After the last chunk of a task has been consumed by every lane (the chunk loops end with __syncwarp): one plain
// arrival completes each idle barrier's current phase, so both end the task in an even phase. A warp runs one task, so
// nothing depends on that; the arrivals stay because the code the compiler generates with them is faster: without them
// reddit K=32 took 0.8246 instead of 0.8195 ms per run (B200, 1000 W), and spmm_kernel<32, 2, 0, false> spills 24 bytes.
__device__ __forceinline__ void pipe_finish(const Pipe &p, int nchunks, int lane) {
    static_assert(kStages == 2, "phase bookkeeping below is written for two stages");
    if (lane == 0) {
        if (((nchunks + 1) >> 1) & 1) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&p.bars[0])) : "memory");
        if ((nchunks >> 1) & 1) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&p.bars[1])) : "memory");
    }
}
__device__ __forceinline__ void pipe_issue(const Pipe &p, int k, const int2 *src, uint32_t entries) {
    const int s = k % kStages;
    mbar_expect_tx(&p.bars[s], entries * 8u);
    tma_bulk_g2s(p.buf + s * kChunk, src, entries * 8u, &p.bars[s]);
}
__device__ __forceinline__ const int2 *pipe_wait(const Pipe &p, int k) {
    const int s = k % kStages;
    mbar_wait(&p.bars[s], (uint32_t)(k / kStages) & 1u);
    return p.buf + s * kChunk;
}

// Light rows as a stream: a warp walks one task of the light panel, staged through shared
// memory by 1-D TMA exactly like a heavy segment. Lane group g reads entries g, g+GROUPS, ... of the task:
// a header starts a new row (the previous row's accumulator is stored first), a nonzero is one B-row gather
// and one in-order FMA, a nop is padding. Rows never span lane groups, so every row is still one FMA chain in
// CSR order (bit-exact), but gathers stay in flight across row boundaries and no load depends on a
// per-row descriptor.
template <int LANES, int VEC, int TUNE, bool FULL, bool LIVE>
__device__ __forceinline__ void light_stream(const CommonArgs &c, const BandArgs &bd, bool accumulate, bool final, int slice, int2 td,
                                             int lane, const Pipe &pipe) {
    constexpr int GROUPS = 32 / LANES;
    constexpr int U = Tune<TUNE, VEC>::kUnroll;
    const int l = lane % LANES;
    const int g = lane / LANES;
    const int len = td.y * GROUPS;
    const int nchunks = (len + kChunk - 1) / kChunk;
    const int2 *src = bd.lpanel + td.x;

    if (lane == 0) {
        pipe_issue(pipe, 0, src, (uint32_t)min(kChunk, len));   // len is a multiple of 4 * GROUPS
        if (nchunks > 1) pipe_issue(pipe, 1, src + kChunk, (uint32_t)min(kChunk, len - kChunk));
    }

    const int K = c.feat;
    const int col0 = slice * c.kslice + l * 4;
    const int col_end = min(K, (slice + 1) * c.kslice);
    // panel entries carry the B row's offset in float4 units (col * K/4), so a gather address is one multiply-add
    const float4 *bbase = reinterpret_cast<const float4 *>(c.vin + col0);
    float4 acc[VEC];
    bool colok[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        colok[v] = FULL || col0 + v * LANES * 4 < col_end;
    }
    int cur_row = -1;
    auto flush_row = [&]() {
        if (cur_row >= 0) {
#pragma unroll
            for (int v = 0; v < VEC; ++v)
                if (colok[v]) st_final(c, final, cur_row, col0 + v * LANES * 4, acc[v]);
        }
    };

    for (int k = 0; k < nchunks; ++k) {
        const int2 *stage = pipe_wait(pipe, k);
        const int n = min(kChunk, len - k * kChunk);
        const int2 *ep = stage + g;   // this lane group's entries: ep[0], ep[GROUPS], ...
        for (int t0 = 0; t0 < n; t0 += GROUPS * U, ep += GROUPS * U) {
            float4 b[U][VEC];
            int2 cv[U];
            float lw[U];   // LIVE: the weights, defined for nonzero entries only
#pragma unroll
            for (int u = 0; u < U; ++u) {
                cv[u] = ep[u * GROUPS];   // in range: a task is padded to a multiple of 4 steps
                if (cv[u].x >= 0) {
                    const float4 *brow = bbase + (unsigned)cv[u].x;
                    if (LIVE) lw[u] = ld_stream_f32(c.val + (unsigned)cv[u].y);
#pragma unroll
                    for (int v = 0; v < VEC; ++v)
                        if (colok[v]) b[u][v] = __ldg(brow + v * LANES);
                }
            }
            bool hdr = false;
#pragma unroll
            for (int u = 0; u < U; ++u) hdr |= cv[u].x < -1;   // headers are 0x80000000 | row; nop is -1
            if (!__any_sync(kFull, hdr)) {
                // common case for long rows: nonzeros (and padding) only — straight-line predicated FMAs
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float w = LIVE ? lw[u] : __int_as_float(cv[u].y);
#pragma unroll
                    for (int v = 0; v < VEC; ++v)
                        if (cv[u].x >= 0 && colok[v]) fma4(acc[v], b[u][v], w);
                }
            } else {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (cv[u].x >= 0) {
                        const float w = LIVE ? lw[u] : __int_as_float(cv[u].y);
#pragma unroll
                        for (int v = 0; v < VEC; ++v)
                            if (colok[v]) fma4(acc[v], b[u][v], w);   // CSR order within the row: bit-exact chain
                    } else if (cv[u].x != -1) {
                        flush_row();   // header: the previous row of this lane group is complete
                        cur_row = cv[u].x & 0x7fffffff;
                        if (accumulate) {
                            const float *crow = c.vout + (size_t)cur_row * K + col0;
#pragma unroll
                            for (int v = 0; v < VEC; ++v)
                                if (colok[v]) acc[v] = __ldcg(reinterpret_cast<const float4 *>(crow + v * LANES * 4));
                        } else {
#pragma unroll
                            for (int v = 0; v < VEC; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
                        }
                    }
                }
            }
        }
        __syncwarp();   // every lane is done reading this stage before it is refilled
        if (lane == 0 && k + kStages < nchunks)
            pipe_issue(pipe, k + kStages, src + (size_t)(k + kStages) * kChunk, (uint32_t)min(kChunk, len - (k + kStages) * kChunk));
    }
    pipe_finish(pipe, nchunks, lane);
    flush_row();
}

template <int LANES, int VEC, int TUNE, bool FULL, bool LIVE>
__device__ __forceinline__ void heavy_segment(const CommonArgs &c, const BandArgs &bd, bool accumulate, bool final, int slice, int seg,
                                              int lane, const Pipe &pipe) {
    constexpr int GROUPS = 32 / LANES;
    constexpr int U = Tune<TUNE, VEC>::kUnroll;
    const int l = lane % LANES;
    const int g = lane / LANES;
    const SegDesc d = bd.seg_desc[seg];
    const int plen = (d.len + 4 * GROUPS - 1) / (4 * GROUPS) * (4 * GROUPS);   // the panel span, padded with nops
    const int nchunks = (plen + kChunk - 1) / kChunk;
    const int2 *src = bd.panel + d.panel_off;

    if (lane == 0) {
        pipe_issue(pipe, 0, src, (uint32_t)min(kChunk, plen));
        if (nchunks > 1) pipe_issue(pipe, 1, src + kChunk, (uint32_t)min(kChunk, plen - kChunk));
    }

    const int K = c.feat;
    const int col0 = slice * c.kslice + l * 4;
    const int col_end = min(K, (slice + 1) * c.kslice);
    // panel entries carry the B row's offset in float4 units (col * K/4), so a gather address is one multiply-add
    const float4 *bbase = reinterpret_cast<const float4 *>(c.vin + col0);
    float4 acc[VEC];
    bool colok[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
        acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        colok[v] = FULL || col0 + v * LANES * 4 < col_end;
    }

    for (int k = 0; k < nchunks; ++k) {
        const int2 *e = pipe_wait(pipe, k);
        const int n = min(kChunk, plen - k * kChunk);
        for (int t0 = 0; t0 < n; t0 += GROUPS * U) {
            float4 b[U][VEC];
            float wt[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int2 cv = e[t0 + u * GROUPS + g];   // in range: the span is padded to whole batches
                ok[u] = cv.x >= 0;                        // nop entries are {-1, 0}
                // a nop gathers row 0 (always a valid address) and is ignored below: every b[u][v] is defined in every
                // iteration, which keeps the register allocator from carrying the batch across iterations
                const float4 *brow = bbase + (ok[u] ? (unsigned)cv.x : 0u);
#pragma unroll
                for (int v = 0; v < VEC; ++v)
                    if (colok[v]) b[u][v] = __ldg(brow + v * LANES);
                if (LIVE) wt[u] = ok[u] ? ld_stream_f32(c.val + (unsigned)cv.y) : 0.f;   // a nop loads nothing
                else wt[u] = __int_as_float(cv.y);
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
#pragma unroll
                for (int v = 0; v < VEC; ++v)
                    if (ok[u] && colok[v]) fma4(acc[v], b[u][v], wt[u]);
            }
        }
        __syncwarp();   // every lane is done reading this stage before it is refilled
        if (lane == 0 && k + kStages < nchunks)
            pipe_issue(pipe, k + kStages, src + (size_t)(k + kStages) * kChunk, (uint32_t)min(kChunk, plen - (k + kStages) * kChunk));
    }

    pipe_finish(pipe, nchunks, lane);
    // combine the lane groups (fixed tree => deterministic)
#pragma unroll
    for (int off = LANES; off < 32; off <<= 1) {
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
            acc[v].x += __shfl_xor_sync(kFull, acc[v].x, off);
            acc[v].y += __shfl_xor_sync(kFull, acc[v].y, off);
            acc[v].z += __shfl_xor_sync(kFull, acc[v].z, off);
            acc[v].w += __shfl_xor_sync(kFull, acc[v].w, off);
        }
    }
    if (g == 0) {
        float *prow = bd.part + (size_t)seg * K + col0;
#pragma unroll
        for (int v = 0; v < VEC; ++v)
            if (colok[v]) __stcg(reinterpret_cast<float4 *>(prow + v * LANES * 4), acc[v]);
        __threadfence();   // partial visible device-wide before this segment is counted
    }
    __syncwarp();

    // Segment reduction without a second launch and without float atomics: the warp that
    // finishes a row's last outstanding segment adds the partials IN SEGMENT ORDER, so the
    // result does not depend on which warp that is. The counter returns to zero for the next run.
    const int hrow = bd.seg_hrow[seg];
    const int s0 = bd.heavy_seg0[hrow], s1 = bd.heavy_seg0[hrow + 1];
    int last = 0;
    if (lane == 0) {
        int *cnt = bd.seg_count + (size_t)hrow * c.n_slices + slice;
        last = atomicAdd(cnt, 1) == s1 - s0 - 1;
        if (last) *cnt = 0;
    }
    last = __shfl_sync(kFull, last, 0);
    if (!last) return;
    // acquire side, executed by every lane that is about to read the other warps' partials (the writers fenced
    // after their stores and before the counter was bumped)
    __threadfence();
    const float *crow = c.vout + (size_t)d.row * K;
    for (int col = slice * c.kslice + lane * 4; col < col_end; col += 128) {
        const float *p = bd.part + (size_t)s0 * K + col;
        float4 sum = accumulate ? __ldcg(reinterpret_cast<const float4 *>(crow + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
        for (int sgm = s0; sgm < s1; ++sgm, p += K) {
            const float4 x = __ldcg(reinterpret_cast<const float4 *>(p));
            sum.x += x.x;
            sum.y += x.y;
            sum.z += x.z;
            sum.w += x.w;
        }
        st_final(c, final, d.row, col, sum);
    }
}

template <int LANES, int VEC, int TUNE, bool FULL, bool LIVE>
__global__ void __launch_bounds__(256, Tune<TUNE, VEC>::kMinBlocks) spmm_kernel(const __grid_constant__ RunArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    const long long gw = (long long)blockIdx.x * nwarps + warp;
    // one task list per feature slice, in the order the plan wants them scheduled
    const int slice = (int)(gw / a.b.n_utask);
    if (slice >= a.c.n_slices) return;
    const int2 td = __ldg(a.b.utask + (gw - (long long)slice * a.b.n_utask));
    const Pipe pipe = {reinterpret_cast<int2 *>(smem_raw) + (size_t)warp * kStages * kChunk,
                       reinterpret_cast<uint64_t *>(smem_raw + (size_t)nwarps * kStages * kChunk * sizeof(int2)) + warp * kStages};
    pipe_init(pipe, lane);
    if (td.x < 0) heavy_segment<LANES, VEC, TUNE, FULL, LIVE>(a.c, a.b, a.b.accumulate != 0, a.b.final != 0, slice, -1 - td.x, lane, pipe);
    else light_stream<LANES, VEC, TUNE, FULL, LIVE>(a.c, a.b, a.b.accumulate != 0, a.b.final != 0, slice, td, lane, pipe);
}

// K % 4 != 0: scalar lanes over the feature columns, one warp per row, same in-order chain. It reads idx/val at run time;
// with live values on a derived handle the weight of position i is val[perm[i]].
__global__ void __launch_bounds__(256) spmm_scalar_kernel(const __grid_constant__ RunArgs ra) {
    const CommonArgs &a = ra.c;
    const int lane = threadIdx.x & 31;
    const long long gw = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (gw >= ra.b.n_light) return;
    const int4 d = __ldg(ra.b.light_desc + gw);
    const int row = d.x, begin = d.y, deg = d.z;
    const int K = a.feat;
    for (int cb = 0; cb < K; cb += 32) {
        const int col = cb + lane;
        float acc = 0.f;
        for (int base = 0; base < deg; base += 32) {
            int c = 0;
            float w = 0.f;
            if (base + lane < deg) {
                const int i = begin + base + lane;
                c = ld_stream_s32(a.idx + i);
                w = ld_stream_f32(a.val + (a.perm ? ld_stream_s32(a.perm + i) : i));
            }
            const int n = min(32, deg - base);
            for (int t = 0; t < n; ++t) {
                const int ct = __shfl_sync(kFull, c, t);
                const float wt = __shfl_sync(kFull, w, t);
                if (col < K) acc = fmaf(__ldg(a.vin + (size_t)ct * K + col), wt, acc);
            }
        }
        if (col < K) a.vout[(size_t)row * K + col] = acc;
    }
}

// ---- preprocessing / support kernels ---------------------------------------------------------

// one warp per row: position of every column-block boundary inside the row (binary search by lane b),
// and a check that the row's columns ascend (otherwise the blocks are not contiguous)
struct BandBounds {
    int begin[kMaxSplitBands + 1];
};
__global__ void __launch_bounds__(256) split_rows_kernel(const int *ptr, const int *idx, int num_v, int nb,
                                                         const BandBounds bands, int *split, int *unsorted) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= num_v) return;
    const int begin = ptr[gw], end = ptr[gw + 1];
    bool bad = false;
    for (int i = begin + lane; i + 1 < end; i += 32) bad |= idx[i] > idx[i + 1];
    if (__any_sync(kFull, bad) && lane == 0) atomicExch(unsorted, 1);
    for (int b = lane; b <= nb; b += 32) {
        int pos;
        if (b == 0) pos = begin;
        else if (b == nb) pos = end;
        else {
            const int target = bands.begin[b];   // first position with idx >= target
            int lo = begin, hi = end;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (idx[mid] < target) lo = mid + 1;
                else hi = mid;
            }
            pos = lo;
        }
        split[(size_t)b * num_v + gw] = pos;
    }
}

// every column index must address a row of B: one pass over idx at plan time (a bad index would otherwise turn
// into an out-of-bounds gather in every run)
__global__ void __launch_bounds__(256) check_cols_kernel(const int *idx, long long nnz, int b_rows, int *bad) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    bool any = false;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += stride) {
        const int c = idx[i];
        any |= c < 0 || c >= b_rows;
    }
    if (__any_sync(kFull, any) && (threadIdx.x & 31) == 0) atomicExch(bad, 1);
}

// The .y word of the staged entry of CSR position i: the value bits, or (live values) the position the run reads its
// weight from — i itself, or perm[i] on a derived handle (a position in the source handle's CSR).
__device__ __forceinline__ int staged_word(int i, const float *val, const int *perm, bool live) {
    return live ? (perm ? perm[i] : i) : __float_as_int(val[i]);
}

// one warp per light row: header at its slot, nonzeros at stride `groups` after it (the panel was preset to nops)
__global__ void __launch_bounds__(256) build_lpanel_kernel(const int4 *light_desc, int n_light, int groups, int k4,
                                                           const int *idx, const float *val, const int *perm, bool live,
                                                           int2 *lpanel) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= n_light) return;
    const int4 d = light_desc[gw];   // {row, begin, deg, dst}
    if (lane == 0) lpanel[d.w] = make_int2((int)(0x80000000u | (unsigned)d.x), 0);
    for (int t = lane; t < d.z; t += 32)
        lpanel[(size_t)d.w + (size_t)(1 + t) * groups] = make_int2(idx[d.y + t] * k4, staged_word(d.y + t, val, perm, live));
}

// one warp per segment: gather its {col * k4, val} pairs into the panel, nop entries in the padding
__global__ void __launch_bounds__(256) build_panel_kernel(const SegDesc *seg, int n_seg, int k4, int pad, const int *idx,
                                                          const float *val, const int *perm, bool live, int2 *panel) {
    const long long gw = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gw >= n_seg) return;
    const SegDesc d = seg[gw];
    const int padded = (d.len + pad - 1) / pad * pad;
    for (int t = lane; t < padded; t += 32) {
        int2 e = make_int2(-1, 0);
        if (t < d.len) e = make_int2(idx[d.nnz_begin + t] * k4, staged_word(d.nnz_begin + t, val, perm, live));
        panel[(size_t)d.panel_off + t] = e;
    }
}

// splitmix64 finaliser; fill = Irwin-Hall(8 x 16 bit) scaled — see oracle/spmm_oracle.c
// (oracle_fill_normal) for the definition both sides implement.
__device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ int sum16x4(uint64_t a) {
    return (int)(a & 0xFFFF) + (int)((a >> 16) & 0xFFFF) + (int)((a >> 32) & 0xFFFF) + (int)(a >> 48);
}
__global__ void __launch_bounds__(256) fill_normal_kernel(float *dst, long long n, uint64_t key, float scale,
                                                          float mean) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const uint64_t x = mix64(key + 2ull * (uint64_t)i);
        const uint64_t y = mix64(key + 2ull * (uint64_t)i + 1ull);
        const int t = sum16x4(x) + sum16x4(y) - 262140;
        dst[i] = __fadd_rn(__fmul_rn((float)t, scale), mean);   // separate mul and add, as the oracle
    }
}

// validate_float (PA4/handout/src/valid.cu:3-13) with an IEEE divide and a 64-bit counter
__global__ void __launch_bounds__(256) valid_kernel(const float *y, const float *y2, long long num,
                                                    unsigned long long *count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned int local = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < num; i += stride) {
        const float q = __fdiv_rn(y[i] - y2[i], y[i]);
        if ((double)fabsf(q) > 1e-2) ++local;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) local += __shfl_xor_sync(kFull, local, off);
    if ((threadIdx.x & 31) == 0 && local) atomicAdd(count, (unsigned long long)local);
}

// per warp: kStages chunks + their mbarriers
size_t task_smem(int block) { return (size_t)(block / 32) * kStages * (kChunk * sizeof(int2) + sizeof(uint64_t)); }

template <int LANES, int VEC, int TUNE, bool FULL, bool LIVE>
void launch_tuned(const RunArgs &a, int block, cudaStream_t stream) {
    const int warps = block / 32;
    const long long tasks = (long long)a.b.n_utask * a.c.n_slices;
    spmm_kernel<LANES, VEC, TUNE, FULL, LIVE><<<(unsigned)((tasks + warps - 1) / warps), block, task_smem(block), stream>>>(a);
}

template <int LANES, int VEC, bool LIVE>
void launch_shape(const RunArgs &a, int block, int tune, bool full, cudaStream_t stream) {
    if (tune == 1) {
        if (full) launch_tuned<LANES, VEC, 1, true, LIVE>(a, block, stream);
        else launch_tuned<LANES, VEC, 1, false, LIVE>(a, block, stream);
    } else {
        if (full) launch_tuned<LANES, VEC, 0, true, LIVE>(a, block, stream);
        else launch_tuned<LANES, VEC, 0, false, LIVE>(a, block, stream);
    }
}

template <int LANES, int VEC>
void launch_shape(const RunArgs &a, const Plan &p, bool full, cudaStream_t stream) {
    if (p.live) launch_shape<LANES, VEC, true>(a, p.block, p.tune, full, stream);
    else launch_shape<LANES, VEC, false>(a, p.block, p.tune, full, stream);
}

int launch_lanes(const Plan &p, const RunArgs &a, bool full, cudaStream_t stream) {
    switch (p.lanes * 10 + p.vec) {
        case 11: launch_shape<1, 1>(a, p, full, stream); break;
        case 21: launch_shape<2, 1>(a, p, full, stream); break;
        case 41: launch_shape<4, 1>(a, p, full, stream); break;
        case 81: launch_shape<8, 1>(a, p, full, stream); break;
        case 161: launch_shape<16, 1>(a, p, full, stream); break;
        case 321: launch_shape<32, 1>(a, p, full, stream); break;
        case 322: launch_shape<32, 2>(a, p, full, stream); break;
        default:
            set_error("unsupported kernel shape lanes=%d vec=%d", p.lanes, p.vec);
            return SPMM_B200_EINVAL;
    }
    return 0;
}

template <int LANES, int VEC>
int slots_shape(int block, int tune) {
    int nb = 0;
    const size_t smem = task_smem(block);
    // the LIVE instances keep the same register caps (DESIGN.md §3), so the snapshot kernel's occupancy stands for both
    const cudaError_t e = tune == 1 ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, spmm_kernel<LANES, VEC, 1, true, false>, block, smem)
                                    : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, spmm_kernel<LANES, VEC, 0, true, false>, block, smem);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return nb;
}

int ctas_per_sm(int lanes, int vec, int tune, int block) {
    switch (lanes * 10 + vec) {
        case 11: return slots_shape<1, 1>(block, tune);
        case 21: return slots_shape<2, 1>(block, tune);
        case 41: return slots_shape<4, 1>(block, tune);
        case 81: return slots_shape<8, 1>(block, tune);
        case 161: return slots_shape<16, 1>(block, tune);
        case 321: return slots_shape<32, 1>(block, tune);
        case 322: return slots_shape<32, 2>(block, tune);
        default: return 0;
    }
}

void fill_common(CommonArgs &c, const spmm_b200_handle *h, const float *vin, float *vout, float *cfinal, const float *val) {
    const Plan &p = h->plan;
    c.idx = h->d_idx;
    c.val = h->d_val;
    c.perm = nullptr;
    if (p.live) {   // positions index the value source: the handle's own CSR, or the source's on a derived handle
        c.val = val ? val : h->t_src ? h->t_src->d_val : h->d_val;
        c.perm = h->t_src ? h->t_perm : nullptr;
    }
    c.vin = vin;
    c.vout = vout;
    c.cfinal = cfinal ? cfinal : vout;
    c.feat = h->feat;
    c.kslice = p.kslice;
    c.n_slices = p.n_slices;
    c.n_gather = h->n_gather;
    for (int t = 0; t < kMaxGather; ++t) c.gather[t] = h->gather[t];
    c.gather_mc = h->gather_mc;
    c.gather_row0 = h->gather_row0;
}

void fill_band(BandArgs &b, const Plan &p, int blk) {
    const BlockPlan &bp = p.blocks[blk];
    b.light_desc = bp.d_light_desc;
    b.n_light = bp.n_light;
    b.utask = bp.d_utask;
    b.n_utask = bp.n_utask;
    b.lpanel = bp.d_lpanel;
    b.seg_desc = bp.d_seg_desc;
    b.seg_hrow = bp.d_seg_hrow;
    b.heavy_seg0 = bp.d_heavy_seg0;
    b.seg_count = bp.d_seg_count;
    b.panel = bp.d_panel;
    b.part = bp.d_part;
    b.accumulate = blk > 0;
    b.final = blk + 1 == p.n_col_blocks;   // only the last pass produces final rows
}

}  // namespace

int launch_spmm(spmm_b200_handle *h, const float *vin, float *vout, cudaStream_t stream,
                int *launches, const cudaEvent_t *band_ready, float *cfinal, const float *val) {
    const Plan &p = h->plan;
    *launches = 0;
    if (h->num_v == 0 || h->feat == 0) return 0;
    const bool full = !p.scalar && h->feat % (p.lanes * p.vec * 4) == 0 && p.kslice == p.lanes * p.vec * 4;
    // Two-stream launches: every pass goes out as two kernels, the first half of the row groups on the caller's stream and
    // the second half on a stream of the handle's. A pass only depends on the previous pass over the SAME rows, so each
    // stream is its own chain, and while one kernel drains its last wave the other stream's kernel fills the freed SMs:
    // the tail of every launch overlaps the next one without any synchronisation inside the kernels.
    const bool two = p.split_streams && !p.scalar;
    if (two) {
        if (!h->aux_stream) {
            SB_CUDA(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
            SB_CUDA(cudaEventCreateWithFlags(&h->aux_fork, cudaEventDisableTiming));
            SB_CUDA(cudaEventCreateWithFlags(&h->aux_join, cudaEventDisableTiming));
        }
        SB_CUDA(cudaEventRecord(h->aux_fork, stream));
        SB_CUDA(cudaStreamWaitEvent(h->aux_stream, h->aux_fork, 0));
    }
    for (int blk = 0; blk < p.n_col_blocks; ++blk) {
        const BlockPlan &bp = p.blocks[blk];
        if (band_ready) {
            SB_CUDA(cudaStreamWaitEvent(stream, band_ready[blk], 0));
            if (two) SB_CUDA(cudaStreamWaitEvent(h->aux_stream, band_ready[blk], 0));
        }
        if (bp.n_light == 0 && bp.n_seg == 0) continue;
        RunArgs a;
        fill_common(a.c, h, vin, vout, cfinal, val);
        fill_band(a.b, p, blk);
        if (p.scalar) {
            const int warps = p.block / 32;
            spmm_scalar_kernel<<<(unsigned)((a.b.n_light + warps - 1) / warps), p.block, 0, stream>>>(a);
            ++*launches;
            continue;
        }
        const int n = bp.n_utask, cut = two ? bp.split_task : n;
        for (int half = 0; half < 2; ++half) {
            const int t0 = half ? cut : 0, t1 = half ? n : cut;
            if (t1 <= t0) continue;
            RunArgs b = a;
            b.b.utask = a.b.utask + t0;
            b.b.n_utask = t1 - t0;
            int rc = launch_lanes(p, b, full, half ? h->aux_stream : stream);
            if (rc) return rc;
            ++*launches;
        }
    }
    if (two) {
        SB_CUDA(cudaEventRecord(h->aux_join, h->aux_stream));
        SB_CUDA(cudaStreamWaitEvent(stream, h->aux_join, 0));
    }
    SB_CUDA(cudaGetLastError());
    return 0;
}

// warps the device keeps resident for this kernel shape (0 when it cannot be queried, e.g. no device)
int resident_warps(int lanes, int vec, int tune, int block) {
    return ctas_per_sm(lanes, vec, tune, block) * (block / 32) * sm_count();
}

int launch_check_cols(const int *d_idx, long long nnz, int b_rows, int *d_bad, cudaStream_t stream) {
    if (nnz == 0) return 0;
    check_cols_kernel<<<stride_grid(nnz), 256, 0, stream>>>(d_idx, nnz, b_rows, d_bad);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_split_rows(const int *d_ptr, const int *d_idx, int num_v, int n_col_blocks, const int *band_begin,
                      int *d_split, int *d_unsorted, cudaStream_t stream) {
    if (num_v == 0) return 0;
    if (n_col_blocks > kMaxSplitBands) {
        set_error("too many column blocks: %d > %d", n_col_blocks, kMaxSplitBands);
        return SPMM_B200_EINVAL;
    }
    BandBounds bands;
    for (int b = 0; b <= kMaxSplitBands; ++b) bands.begin[b] = band_begin[b < n_col_blocks ? b : n_col_blocks];
    const long long threads = (long long)num_v * 32;
    split_rows_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(d_ptr, d_idx, num_v, n_col_blocks, bands, d_split,
                                                                            d_unsorted);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_build_lpanel(const int4 *d_light_desc, int n_light, int groups, int k4, const int *d_idx, const float *d_val,
                        const int *perm, bool live, int2 *d_lpanel, cudaStream_t stream) {
    if (n_light == 0) return 0;
    const long long threads = (long long)n_light * 32;
    build_lpanel_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(d_light_desc, n_light, groups, k4, d_idx,
                                                                              d_val, perm, live, d_lpanel);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_build_panel(const SegDesc *d_seg, int n_seg, int k4, int pad, const int *d_idx, const float *d_val,
                       const int *perm, bool live, int2 *d_panel, cudaStream_t stream) {
    if (n_seg == 0) return 0;
    const long long threads = (long long)n_seg * 32;
    build_panel_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, stream>>>(d_seg, n_seg, k4, pad, d_idx, d_val, perm,
                                                                             live, d_panel);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_fill_normal(float *d_dst, long long n, uint64_t seed, uint64_t stream_id, float mean,
                       float stddev, cudaStream_t stream) {
    if (n <= 0) return 0;
    // host copy of mix64 for the key
    auto hmix = [](uint64_t z) {
        z += 0x9E3779B97F4A7C15ull;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    };
    const uint64_t key = hmix(seed ^ hmix(stream_id * 0x632BE59BD9B4E019ull + 0x1234567ull));
    const float scale = (float)((double)stddev / 53510.0);
    fill_normal_kernel<<<stride_grid(n), 256, 0, stream>>>(d_dst, n, key, scale, mean);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_valid(const float *d_y, const float *d_y2, long long num, unsigned long long *d_count,
                 cudaStream_t stream) {
    if (num <= 0) return 0;
    valid_kernel<<<stride_grid(num), 256, 0, stream>>>(d_y, d_y2, num, d_count);
    SB_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace spmm_b200
