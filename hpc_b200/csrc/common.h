// common.h — internal declarations shared by the engine's translation units (not installed).
#ifndef HPC_B200_COMMON_H_
#define HPC_B200_COMMON_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

#include "spmm_b200.h"

namespace spmm_b200 {

// Error plumbing: the reference aborts in checkCudaErrors (PA4/handout/include/util.h:63-84);
// the C ABI records the message and returns the code instead.
void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define SB_CUDA(call)                                                              \
    do {                                                                           \
        cudaError_t e__ = (call);                                                  \
        if (e__ != cudaSuccess) return ::spmm_b200::cuda_fail(e__, #call, __FILE__, __LINE__); \
    } while (0)

constexpr int kMaxGather = 16;

// One heavy-row segment: `len` nonzeros of `row` starting at CSR position `nnz_begin`,
// staged at panel[panel_off .. panel_off + len rounded up to whole gather batches, 4 * (32 / lanes) entries).
struct SegDesc {
    int row;
    int panel_off;
    int len;
    int nnz_begin;
};

constexpr int kMaxBands = 16;    // cap of the automatic number of column blocks
// Bytes of B per column-block band, and per chunk of run_host_sharded's upload of B, so that chunks and bands coincide
constexpr long long kBandBytes = 48ll << 20;
constexpr int kMaxRowGroups = 64;

// What every pass of a run shares.
struct CommonArgs {
    const int *idx;           // scalar fallback kernel only (the vectorised kernels read the staged panels)
    const float *val;         // scalar kernel; with live values also the vectorised kernels: val[panel .y word]
    const int *perm;          // live values on a derived handle (scalar kernel): the weight of position i is val[perm[i]]
    const float *vin;
    float *vout;              // C: partial chains between column-block passes, and final rows unless cfinal differs
    float *cfinal;            // where FINAL rows are stored (= vout, or device-mapped pinned host memory: run_host's zero-copy output)
    int feat;                 // K
    int kslice;               // feature columns per slice
    int n_slices;
    // stacked-layer epilogue: final rows also go to every rank's copy of the next layer's B
    int n_gather;             // 0 = off
    float *gather[kMaxGather];   // peer-mapped (or local) buffers of b_rows x K floats
    float *gather_mc;         // NVLS multicast address of the same buffers, or NULL
    long long gather_row0;    // this handle's first row inside those buffers
};

// One column block (band of B rows) of the plan.
struct BandArgs {
    const int4 *light_desc;   // {row, begin, deg, dst} in processing order (scalar kernel; dst: header slot in lpanel)
    int n_light;
    const int2 *utask;        // warp tasks of one slice in scheduling order: {lpanel offset, steps per lane group}
                              // for a light-stream task, {-1 - segment, 0} for a heavy segment
    int n_utask;
    const int2 *lpanel;       // light rows as a stream: header {0x80000000|row, 0}, then {col, val}..., nop = {-1, -1}
                              // (live values: {col, position} instead of {col, val})
    const SegDesc *seg_desc;
    const int *seg_hrow;      // segment -> index of its row in heavy_rows
    const int *heavy_seg0;    // heavy row -> first segment (prefix, n_heavy + 1)
    int *seg_count;           // [n_heavy][n_slices] finished-segment counters, zero between runs
    const int2 *panel;
    float *part;              // [n_seg][K] partial sums
    int accumulate;           // 1: continue the chains from vout (column blocks after the first)
    int final;                // 1: this pass delivers final rows (cfinal, stacked-layer targets)
};

// One launch per column block.
struct RunArgs {
    CommonArgs c;
    BandArgs b;
};

// The plan of one column block (the whole matrix when there is a single block): its counts and its device arrays.
struct BlockPlan {
    int col_begin = 0, col_end = 0;   // B rows [col_begin, col_end) are gathered in this pass
    int reorder = 1, light_steps = 0;
    int n_light = 0, n_heavy = 0, n_seg = 0, n_ltask = 0, n_utask = 0;
    long long panel_len = 0, lpanel_len = 0;
    int split_task = 0;            // first task of the second half of the row groups (two-stream launches); 0 / n_utask: no split
    int4 *d_light_desc = nullptr;
    int2 *d_utask = nullptr, *d_lpanel = nullptr, *d_panel = nullptr;
    SegDesc *d_seg_desc = nullptr;
    int *d_heavy_seg0 = nullptr, *d_seg_hrow = nullptr, *d_seg_count = nullptr;
    float *d_part = nullptr;
};

struct Plan {
    bool ready = false;
    int device = -1;   // the device the plan's arrays live on (the current device at preprocess)
    int seg_len = 0, kslice = 0, n_slices = 0, block = 128, lanes = 0, vec = 0, tune = 0, light_steps = 0;
    bool scalar = false;   // K % 4 != 0: scalar fallback kernel, no segments
    bool live = false;     // option "live_values": panels stage positions, runs read the weights from a value array
    int n_col_blocks = 1;
    long long slots = 0;   // warps the device keeps resident for the chosen kernel shape
    int *d_split = nullptr;   // [(n_col_blocks+1)][num_v] start of each column block inside each row
    std::vector<BlockPlan> blocks;
    int launches = 0;
    int n_groups = 1;               // row groups: contiguous row ranges planned independently, never spanned by a task
    std::vector<int> group_row;     // [n_groups + 1] first row of each group
    bool split_streams = false;     // every pass as two launches (row-group halves) on two streams: each tail overlaps the next launch
    // arenas: one allocation per array kind, band after band (the per-band pointers above point into them)
    int2 *d_lpanel_all = nullptr, *d_panel_all = nullptr;
    float *d_part_all = nullptr;
    int *d_seg_count_all = nullptr;
    // spmm_b200_sddmm (sddmm.cu), set up by its first call after preprocess
    int *d_sddmm_vp = nullptr;      // [n_col_blocks * num_v + 1] band-major prefix of the (band, row) lengths (several blocks)
    int sddmm_chunk = 0;            // nonzeros per warp (0: not set up yet)
};

}  // namespace spmm_b200

struct spmm_b200_handle {
    const int *d_ptr = nullptr;
    const int *d_idx = nullptr;
    const float *d_val = nullptr;
    int num_v = 0, num_e = 0, feat = 0;
    long long opt_seg_len = 0, opt_kslice = 0, opt_block = 128, opt_reorder = -1, opt_tune = 0, opt_col_blocks = 0, opt_light_steps = 0,
              opt_zero_copy = 1, opt_row_groups = 0, opt_split_streams = -1, opt_host_bands = 0, opt_live_values = 0;
    int plan_select = 0;   // which column block plan_info / plan_copy describe
    spmm_b200::Plan plan;
    float *d_stage_in = nullptr, *d_stage_out = nullptr;
    size_t stage_elems = 0, stage_in_elems = 0;
    cudaStream_t copy_stream = nullptr;          // run_host: H2D of B bands
    cudaStream_t aux_stream = nullptr;           // two-stream launches: the second row half
    cudaEvent_t aux_fork = nullptr, aux_join = nullptr;
    std::vector<cudaEvent_t> band_events;
    int n_gather = 0;
    float *gather[spmm_b200::kMaxGather] = {nullptr};
    float *gather_mc = nullptr;
    long long gather_row0 = 0;
    int b_rows = 0;   // rows of B (0 = num_v); > num_v for a row partition of a larger graph
    // sharded host I/O over NVLink (replicate.cu): every rank's copy of B and flag words, as mapped in this process
    int rep_world = 0, rep_rank = 0;
    float *rep_b[spmm_b200::kMaxGather] = {nullptr};
    float *rep_mc = nullptr;
    unsigned int *rep_flags[spmm_b200::kMaxGather] = {nullptr};
    unsigned int rep_epoch = 0;
    long long rep_h2d_bytes = 0;   // host-to-device bytes of the last run_host_sharded call
    // transposed operator (transpose.cu): the CSR of A^T is owned by this handle; t_src is the handle it was built from
    int *t_ptr = nullptr, *t_idx = nullptr, *t_perm = nullptr;
    int t_device = -1;   // the device whose pool (pool.cu) these arrays came from
    float *t_val = nullptr;
    const spmm_b200_handle *t_src = nullptr;
};

namespace spmm_b200 {

// capi.cu
float *host_out_mapping(const spmm_b200_handle *h, float *h_vout);

// preprocess.cu
int build_plan(spmm_b200_handle *h, cudaStream_t stream);
void free_plan(Plan &p);
// pool.cu: plan arrays (and the transposed operator's CSR) come from a library-owned CUDA memory pool per device that
// keeps freed blocks for the next plan; all three act on the CURRENT device.
cudaError_t pool_alloc(void **ptr, size_t bytes, cudaStream_t stream);
void pool_free(void *ptr, cudaStream_t stream);
int trim_pool_memory();
int refresh_panels(spmm_b200_handle *h, cudaStream_t stream);

// spmm_kernels.cu
// band_ready: NULL, or one event per column block that the stream waits on before that block's pass
// (run_host uploads B band by band on a second stream while earlier passes compute)
// cfinal: NULL, or where the final rows go instead of vout (the last pass stores them there; earlier passes keep
// their partial chains in vout)
// val: a live plan's value array (spmm_b200_run_values); NULL = the handle's value source (d_val, or t_src's on a
// derived handle). Ignored by a snapshot plan.
int launch_spmm(spmm_b200_handle *h, const float *vin, float *vout, cudaStream_t stream,
                int *launches, const cudaEvent_t *band_ready = nullptr, float *cfinal = nullptr, const float *val = nullptr);
int resident_warps(int lanes, int vec, int tune, int block);
int launch_check_cols(const int *d_idx, long long nnz, int b_rows, int *d_bad, cudaStream_t stream);
// band_begin[0..n_col_blocks]: first B row of every column block (band_begin[n] = b_rows), at most kMaxSplitBands blocks
constexpr int kMaxSplitBands = 64;
int launch_split_rows(const int *d_ptr, const int *d_idx, int num_v, int n_col_blocks, const int *band_begin,
                      int *d_split, int *d_unsorted, cudaStream_t stream);
// The .y word of a staged entry: the value bits of d_val[i] (live = false), or the position i — perm[i] when perm is
// non-NULL — (live = true, d_val is not read).
int launch_build_lpanel(const int4 *d_light_desc, int n_light, int groups, int k4, const int *d_idx, const float *d_val,
                        const int *perm, bool live, int2 *d_lpanel, cudaStream_t stream);
int launch_build_panel(const SegDesc *d_seg, int n_seg, int k4, int pad, const int *d_idx, const float *d_val,
                       const int *perm, bool live, int2 *d_panel, cudaStream_t stream);
int launch_fill_normal(float *d_dst, long long n, uint64_t seed, uint64_t stream_id, float mean,
                       float stddev, cudaStream_t stream);
int launch_valid(const float *d_y, const float *d_y2, long long num, unsigned long long *d_count,
                 cudaStream_t stream);

// transpose.cu
int regather_transposed_values(spmm_b200_handle *t, cudaStream_t stream);

// replicate.cu
// Push `count` floats at src (16-byte aligned, count % 4 == 0) to the same offset `off` of every buffer in targets[0..n)
// except targets[skip] (skip < 0: none) — or, when mc is non-NULL, once through that NVLS multicast address.
int launch_push_rows(const float *src, long long off, long long count, int n, float *const *targets, int skip, float *mc,
                     cudaStream_t stream);
// Cross-rank barrier on `stream`: phase-th flag word of this rank is set to `epoch` in every rank's flag array, then the
// kernel waits until every rank's word in the local array has reached `epoch`. flags[r] = uint32[2 * world] of rank r.
int launch_xrank_barrier(unsigned int *const *flags, int world, int rank, int phase, unsigned int epoch, cudaStream_t stream);

// Packs light rows (costs = deg + 1 entries each, in plan order) into stream tasks of `groups` interleaved lane-group
// lanes with about `steps` entries each; dst[i] = lpanel slot of row i's header. Returns the lpanel length.
long long pack_light_host(const int *cost, int n, int groups, int steps, int *dst, std::vector<int2> &tasks);

// The current device's SM count, or the error of the failed query.
inline cudaError_t query_sm_count(int *sms) {
    int dev = 0;
    const cudaError_t e = cudaGetDevice(&dev);
    return e != cudaSuccess ? e : cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
}

// The current device's SM count, or 0 when it cannot be queried (the error is cleared).
inline int sm_count() {
    int sms = 0;
    if (query_sm_count(&sms) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return sms;
}

// Grid of a grid-stride support kernel of 256-thread blocks over n elements: one block per 256, at most 16 per SM of the
// current device (148 SMs, a B200's, when it cannot be queried), at least 1.
inline int stride_grid(long long n) {
    const int sms = sm_count();
    const long long cap = 16ll * (sms > 0 ? sms : 148), blocks = (n + 255) / 256;
    return (int)(blocks < 1 ? 1 : blocks < cap ? blocks : cap);
}

// Lanes per row slice of q units (float4 or columns): the power of two >= q, at most 32. This is the L of sddmm's
// summation order (sddmm.cu), which reduce_backward's dval (reduce.cu) must follow bit for bit.
inline int pow2_lanes(int q) {
    int l = 1;
    while (l < q && l < 32) l <<= 1;
    return l;
}

// The one-slice lane shape of K % 4 == 0, K <= 512 (sddmm_kernel, reduce.cu's float4 kernels): L lanes of vec float4.
struct LaneShape {
    int lanes, vec;   // vec: 1, 2 or 4
};
inline LaneShape fast_lane_shape(int K) {
    const int q = K / 4, l = pow2_lanes(q), need = (q + l - 1) / l;
    return {l, need <= 1 ? 1 : need <= 2 ? 2 : 4};
}

// lanes/vec choice for a slice width (shared by plan + launch)
inline void shape_for_kslice(int kslice, int *lanes, int *vec) {
    // kslice is a multiple of 4; lanes*vec*4 >= kslice, lanes a power of two <= 32
    const int q = (kslice + 3) / 4;   // float4 per row slice
    *lanes = pow2_lanes(q);
    *vec = (q + *lanes - 1) / *lanes;   // 1 for kslice <= 128, 2 for 256
}

}  // namespace spmm_b200
#endif
