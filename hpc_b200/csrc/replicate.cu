// replicate.cu — sharded host I/O for the multi-GPU driver: B is replicated over NVLink, not N times over PCIe.
//
// No reference counterpart (the reference is single-GPU; SURVEY.md §8e: "each GPU gets ... full B replicated").
// One process per GPU. Every rank holds a full-size copy of B in symmetric (peer-mapped) memory. Per call, rank g
// uploads only ITS slice of B rows from the host, pushes that slice into every other rank's copy — one
// `multimem.st` per 16 bytes through the NVLS multicast address when there is one, else one `st.global` per peer —
// and a device-side flag barrier over the same peer mappings orders the pushes against the SpMM passes. PCIe then
// carries 4·b_rows·K/N bytes in and 4·rows_g·K bytes out per rank instead of the whole B on every rank.
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <vector>

#include "common.h"

namespace spmm_b200 {

namespace {

struct PtrTable {
    float *p[kMaxGather];
};
struct FlagTable {
    unsigned int *p[kMaxGather];
};

__device__ __forceinline__ void st_release_sys(unsigned int *p, unsigned int v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int *p) {
    unsigned int v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// grid-stride float4 copy of this rank's slice into the peers' copies of B
__global__ void __launch_bounds__(256) push_rows_kernel(const float4 *__restrict__ src, long long off4, long long n4, int n,
                                                        const __grid_constant__ PtrTable tg, int skip, float *mc) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 v = __ldcs(src + i);
        if (mc) {
            asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(reinterpret_cast<float4 *>(mc) + off4 + i),
                         "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                         : "memory");
        } else {
            for (int t = 0; t < n; ++t)
                if (t != skip) reinterpret_cast<float4 *>(tg.p[t])[off4 + i] = v;
        }
    }
}

// one thread per rank: publish my arrival everywhere, then wait for everybody's in my own flag array.
// Epochs only grow (one per call and phase), compared wrap-safe.
__global__ void xrank_barrier_kernel(const __grid_constant__ FlagTable fl, int world, int rank, int phase, unsigned int epoch) {
    const int t = threadIdx.x;
    if (t >= world) return;
    __threadfence_system();   // whatever this stream wrote before (peer pushes of the previous kernel) is visible first
    st_release_sys(fl.p[t] + phase * world + rank, epoch);
    const unsigned int *mine = fl.p[rank] + phase * world + t;
    while ((int)(ld_acquire_sys(mine) - epoch) < 0) __nanosleep(64);
}

}  // namespace

int launch_push_rows(const float *src, long long off, long long count, int n, float *const *targets, int skip, float *mc,
                     cudaStream_t stream) {
    if (count <= 0) return 0;
    if ((count & 3) || (off & 3) || ((uintptr_t)src & 15)) {
        set_error("push_rows: slice must be 16-byte aligned and a multiple of 4 floats");
        return SPMM_B200_EINVAL;
    }
    PtrTable tg;
    for (int t = 0; t < kMaxGather; ++t) tg.p[t] = t < n ? targets[t] : nullptr;
    int sms = sm_count();
    if (sms <= 0) sms = 148;
    const long long n4 = count / 4;
    long long blocks = (n4 + 255) / 256;
    if (blocks > 8ll * sms) blocks = 8ll * sms;
    push_rows_kernel<<<(unsigned)blocks, 256, 0, stream>>>(reinterpret_cast<const float4 *>(src), off / 4, n4, n, tg, skip, mc);
    SB_CUDA(cudaGetLastError());
    return 0;
}

int launch_xrank_barrier(unsigned int *const *flags, int world, int rank, int phase, unsigned int epoch, cudaStream_t stream) {
    FlagTable fl;
    for (int t = 0; t < kMaxGather; ++t) fl.p[t] = t < world ? flags[t] : nullptr;
    xrank_barrier_kernel<<<1, 32, 0, stream>>>(fl, world, rank, phase, epoch);
    SB_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" {

int spmm_b200_set_replicate(spmm_b200_t h, int world, int rank, float *const *peers_b, float *multicast_b,
                            unsigned int *const *peers_flags) {
    if (!h || world < 0 || world > kMaxGather || (world > 0 && (rank < 0 || rank >= world || !peers_b || !peers_flags))) {
        set_error("spmm_b200_set_replicate: bad arguments (world <= %d)", kMaxGather);
        return SPMM_B200_EINVAL;
    }
    for (int t = 0; t < world; ++t)
        if (!peers_b[t] || ((uintptr_t)peers_b[t] & 15) || !peers_flags[t]) {
            set_error("spmm_b200_set_replicate: buffer %d is null or not 16-byte aligned", t);
            return SPMM_B200_EINVAL;
        }
    h->rep_world = world;
    h->rep_rank = world > 0 ? rank : 0;
    for (int t = 0; t < kMaxGather; ++t) {
        h->rep_b[t] = t < world ? peers_b[t] : nullptr;
        h->rep_flags[t] = t < world ? peers_flags[t] : nullptr;
    }
    h->rep_mc = world > 0 ? multicast_b : nullptr;
    h->rep_epoch = 0;
    return 0;
}

// B is cut into n_chunks equal row chunks by a rule every rank evaluates identically (b_rows and feat_in only: about
// kBandBytes each, the column-block band size, so chunks and bands coincide whenever a rank's plan uses column blocks);
// rank g brings in the g-th of `world` equal pieces of every chunk.
static int replicate_chunks(long long b_rows, int feat) {
    const long long bytes = b_rows * feat * 4ll;
    long long n = (bytes + kBandBytes - 1) / kBandBytes;
    if (n < 1) n = 1;
    if (n > 16) n = 16;
    if (n > b_rows) n = b_rows > 0 ? b_rows : 1;
    return (int)n;
}

int spmm_b200_run_host_sharded(spmm_b200_t h, const float *h_vin, float *h_vout, void *stream) {
    if (!h || !h_vin || !h_vout) {
        set_error("spmm_b200_run_host_sharded: null argument");
        return SPMM_B200_EINVAL;
    }
    if (h->rep_world <= 0) {
        set_error("spmm_b200_run_host_sharded: spmm_b200_set_replicate has not been called");
        return SPMM_B200_ESTATE;
    }
    if (!h->plan.ready) {
        set_error("spmm_b200_run_host_sharded: preprocess has not been called");
        return SPMM_B200_ESTATE;
    }
    if (h->feat % 4 != 0 || h->feat == 0) {
        set_error("spmm_b200_run_host_sharded: needs feat_in %% 4 == 0");
        return SPMM_B200_EINVAL;
    }
    const int b_rows = h->b_rows > 0 ? h->b_rows : h->num_v;
    const int world = h->rep_world, rank = h->rep_rank;
    const Plan &p = h->plan;
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)h->num_v * h->feat;
    if (h->stage_elems < n) {
        cudaFree(h->d_stage_out);
        h->d_stage_out = nullptr;
        h->stage_elems = 0;
        if (n) SB_CUDA(cudaMalloc((void **)&h->d_stage_out, n * sizeof(float)));
        h->stage_elems = n;
    }
    const int n_chunks = replicate_chunks(b_rows, h->feat);
    const int chunk_rows = (b_rows + n_chunks - 1) / n_chunks;
    if (!h->copy_stream) {
        int lo = 0, hi = 0;
        SB_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
        // above the passes: a pending push or barrier must not queue behind the CTAs of a pass that does not need it
        SB_CUDA(cudaStreamCreateWithPriority(&h->copy_stream, cudaStreamNonBlocking, hi));
    }
    while ((int)h->band_events.size() < std::max(n_chunks, p.n_col_blocks) + 1) {
        cudaEvent_t e;
        SB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->band_events.push_back(e);
    }
    float *local_b = h->rep_b[rank];
    cudaStream_t c = h->copy_stream;
    int rc;
    // SPMM_B200_TRACE_HOST=1: device timestamps of the call's phases on stderr (rank 0 and the last rank)
    static const bool trace = getenv("SPMM_B200_TRACE_HOST") != nullptr;
    cudaEvent_t tev[24] = {nullptr};
    int n_tev = 0;
    auto stamp = [&](cudaStream_t st) {
        if (!trace || n_tev >= 24) return;
        if (cudaEventCreate(&tev[n_tev]) == cudaSuccess) cudaEventRecord(tev[n_tev++], st);
    };
    stamp(s);
    // the copy stream starts behind whatever is queued on the caller's stream (the previous call's passes)
    SB_CUDA(cudaEventRecord(h->band_events[n_chunks], s));
    SB_CUDA(cudaStreamWaitEvent(c, h->band_events[n_chunks], 0));
    // phase 0: every rank is done gathering from its copy of B (previous call) before anybody overwrites a row of it
    const unsigned int call = ++h->rep_epoch;
    if ((rc = launch_xrank_barrier(h->rep_flags, world, rank, 0, call, c))) return rc;
    stamp(c);
    long long h2d = 0;
    for (int ck = 0; ck < n_chunks; ++ck) {
        const long long c0 = std::min<long long>(b_rows, (long long)ck * chunk_rows), c1 = std::min<long long>(b_rows, c0 + chunk_rows);
        const long long r0 = c0 + (c1 - c0) * rank / world, r1 = c0 + (c1 - c0) * (rank + 1) / world;
        const long long off = r0 * h->feat, cnt = (r1 - r0) * h->feat;
        if (cnt) {
            SB_CUDA(cudaMemcpyAsync(local_b + off, h_vin + off, (size_t)cnt * sizeof(float), cudaMemcpyHostToDevice, c));
            if ((rc = launch_push_rows(local_b + off, off, cnt, world, h->rep_b, rank, h->rep_mc, c))) return rc;
            h2d += cnt * 4;
        }
        // phase 1, one epoch per chunk: every rank's piece of this chunk has landed everywhere
        const unsigned int epoch = (call - 1) * (unsigned int)n_chunks + (unsigned int)ck + 1u;
        stamp(c);
        if ((rc = launch_xrank_barrier(h->rep_flags, world, rank, 1, epoch, c))) return rc;
        SB_CUDA(cudaEventRecord(h->band_events[ck], c));
        stamp(c);
    }
    h->rep_h2d_bytes = h2d;
    if (n) {
        // pass b gathers from B rows [col_begin, col_end): it waits for the last chunk that holds any of them
        std::vector<cudaEvent_t> ready((size_t)p.n_col_blocks);
        for (int b = 0; b < p.n_col_blocks; ++b) {
            const int last_row = std::max(0, std::min(b_rows, p.blocks[b].col_end) - 1);
            ready[b] = h->band_events[std::min(n_chunks - 1, last_row / chunk_rows)];
        }
        float *out_map = host_out_mapping(h, h_vout);   // pinned output: the last pass stores final rows straight into it
        if ((rc = launch_spmm(h, local_b, h->d_stage_out, s, &h->plan.launches, ready.data(), out_map))) return rc;
        if (!out_map) SB_CUDA(cudaMemcpyAsync(h_vout, h->d_stage_out, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    } else {
        SB_CUDA(cudaStreamWaitEvent(s, h->band_events[n_chunks - 1], 0));
    }
    stamp(s);
    SB_CUDA(cudaStreamSynchronize(s));
    SB_CUDA(cudaStreamSynchronize(c));
    if (trace && n_tev > 1 && (rank == 0 || rank == world - 1)) {
        fprintf(stderr, "[run_host_sharded rank %d] ms since call start: barrier0 done", rank);
        for (int i = 1; i < n_tev; ++i) {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, tev[0], tev[i]);
            if (i == n_tev - 1) fprintf(stderr, " | passes + C out done %.3f", ms);
            else if (i == 1) fprintf(stderr, " %.3f | chunks (pushed, landed everywhere):", ms);
            else fprintf(stderr, " %.3f", ms);
        }
        fprintf(stderr, "\n");
    }
    for (int i = 0; i < n_tev; ++i) cudaEventDestroy(tev[i]);
    return 0;
}

long long spmm_b200_replicate_h2d_bytes(spmm_b200_t h) { return h ? h->rep_h2d_bytes : 0; }

}  // extern "C"
