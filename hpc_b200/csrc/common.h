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

constexpr int kMaxBands = 16;    // column blocks one persistent launch can carry
constexpr int kMaxRowGroups = 64;

// What every pass of a run shares.
struct CommonArgs {
    const int *idx;           // scalar fallback kernel only (the vectorised kernels read the staged panels)
    const float *val;
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

// One persistent launch for all column blocks: warps draw tickets; ticket order is band-major. `all` addresses the
// bands' arrays as ONE set (each array is a single allocation, band after band), and the ticket list carries absolute
// positions, so nothing in the task bodies is indexed by band.
struct PersistArgs {
    CommonArgs c;
    BandArgs all;             // lpanel / panel / seg_desc / seg_hrow / heavy_seg0 / seg_count / part over all bands
    const int4 *ptask;        // per ticket: {lpanel offset, or -1 - segment; steps; row group | accumulate << 16 | final << 17;
                              //              completed tasks of that row group the task waits for}
    int total;                // tickets
    unsigned int *ctr;        // counters, one per 128-byte line (kCtrStride words apart): [0] ticket, [1] exited warps,
                              // [2 + g] completed tasks of row group g — zero between runs — then the watchdog's line
    int n_groups;
    int batch;                // tickets a warp draws at once while the launch is far from its end (1 over its last stretch)
};
constexpr int kCtrStride = 32;   // words between counters: each on its own L2 line (same-line atomics serialise)
inline size_t ctr_words(int n_groups) { return (size_t)(2 + n_groups + 1) * kCtrStride; }

// The plan of one column block (the whole matrix when there is a single block).
struct BlockPlan {
    int col_begin = 0, col_end = 0;   // B rows [col_begin, col_end) are gathered in this pass
    int n_light = 0, n_heavy = 0, n_seg = 0;
    long long panel_len = 0;
    int *d_row_perm = nullptr;
    int4 *d_light_desc = nullptr;
    int2 *d_ltask = nullptr;
    int2 *d_utask = nullptr;
    int n_utask = 0;
    int2 *d_lpanel = nullptr;
    int n_ltask = 0;
    int light_steps = 0;
    int reorder = 1;
    long long lpanel_len = 0;
    int *d_heavy_rows = nullptr;
    int *d_heavy_seg0 = nullptr;
    SegDesc *d_seg_desc = nullptr;
    int *d_seg_hrow = nullptr;
    int *d_seg_count = nullptr;
    int2 *d_panel = nullptr;
    float *d_part = nullptr;
    std::vector<int> task_group;   // host: row group of every utask entry (persistent launch)
    int split_task = 0;            // first task of the second half of the row groups (two-stream launches); 0 / n_utask: no split
};

struct Plan {
    bool ready = false;
    int device = -1;   // the device the plan's arrays live on (the current device at preprocess)
    int seg_len = 0, kslice = 0, n_slices = 0, block = 128, lanes = 0, vec = 0, tune = 0, light_steps = 0;
    bool scalar = false;   // K % 4 != 0: scalar fallback kernel, no segments
    int n_col_blocks = 1;
    long long slots = 0;   // warps the device keeps resident for the chosen kernel shape
    int *d_split = nullptr;   // [(n_col_blocks+1)][num_v] start of each column block inside each row
    std::vector<BlockPlan> blocks;
    int launches = 0;
    // persistent single launch (all column blocks in one kernel)
    bool persistent = false;
    int n_groups = 1;               // row groups: band b+1's tasks of a group wait for band b's tasks of the same group
    std::vector<int> group_row;     // [n_groups + 1] first row of each group
    unsigned int *d_ctr = nullptr;  // ticket, exited warps, per-group completion counters, watchdog (ctr_words)
    int persist_grid = 0;           // CTAs of the persistent launch (all co-resident)
    int ticket_batch = 1;           // tickets drawn at once far from the end of the launch
    bool split_streams = false;     // every pass as two launches (row-group halves) on two streams: each tail overlaps the next launch
    int n_ptask = 0;
    int4 *d_ptask = nullptr;        // the ticket list
    SegDesc *d_pseg_desc = nullptr; // segments of all bands with absolute panel offsets
    int *d_pseg_hrow = nullptr;     // segment -> absolute heavy-row index
    int *d_pheavy_seg0 = nullptr;   // absolute heavy row -> absolute first segment (n_heavy + 1 entries per band)
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
              opt_zero_copy = 1, opt_persistent = -1, opt_row_groups = 0, opt_ticket_batch = 0, opt_split_streams = -1, opt_host_bands = 0;
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
int launch_spmm(spmm_b200_handle *h, const float *vin, float *vout, cudaStream_t stream,
                int *launches, const cudaEvent_t *band_ready = nullptr, float *cfinal = nullptr);
int resident_warps(int lanes, int vec, int tune, int block);
int persistent_grid(int lanes, int vec, int tune, int block);   // CTAs that are co-resident for the persistent kernel
int launch_check_cols(const int *d_idx, long long nnz, int b_rows, int *d_bad, cudaStream_t stream);
// band_begin[0..n_col_blocks]: first B row of every column block (band_begin[n] = b_rows), at most kMaxSplitBands blocks
constexpr int kMaxSplitBands = 64;
int launch_split_rows(const int *d_ptr, const int *d_idx, int num_v, int n_col_blocks, const int *band_begin,
                      int *d_split, int *d_unsorted, cudaStream_t stream);
int launch_build_lpanel(const int4 *d_light_desc, int n_light, int groups, int k4, const int *d_idx, const float *d_val,
                        int2 *d_lpanel, cudaStream_t stream);
int launch_build_panel(const SegDesc *d_seg, int n_seg, int k4, int pad, const int *d_idx, const float *d_val,
                       int2 *d_panel, cudaStream_t stream);
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
// cut[0..n_cut): ascending row positions before which the open task is closed (row-group boundaries), or NULL.
long long pack_light_host(const int *cost, int n, int groups, int steps, int *dst, std::vector<int2> &tasks,
                          const int *cut = nullptr, int n_cut = 0);

// lanes/vec choice for a slice width (shared by plan + launch)
inline void shape_for_kslice(int kslice, int *lanes, int *vec) {
    // kslice is a multiple of 4; lanes*vec*4 >= kslice, lanes a power of two <= 32
    int q = (kslice + 3) / 4;   // float4 per row slice
    int l = 1;
    while (l < q && l < 32) l <<= 1;
    *lanes = l;
    *vec = (q + l - 1) / l;     // 1 for kslice <= 128, 2 for 256
}

}  // namespace spmm_b200
#endif
