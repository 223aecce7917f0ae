/*
 * spmm_b200.h — C ABI of the B200-native CSR SpMM engine (C = A·B, A sparse CSR fp32,
 * B/C dense row-major fp32 with leading dimension K).
 *
 * This header is the drop-in boundary for the SpMM operator of liblaf/hpc PA4. Every entry
 * point cites the reference interface it replaces (paths relative to the reference root).
 * Plain pointers and sizes only; no C++ / torch types. All functions return 0 on success or
 * a non-zero status (a cudaError_t value when a CUDA call failed, a negative SPMM_B200_E*
 * code otherwise) and never exit or throw; spmm_b200_last_error() gives the text.
 *
 * Ownership (PA4/handout/test/main.cpp:11-16, test/test_spmm.cu:16-28): ptr/idx/val/vin/vout
 * are DEVICE pointers owned by the caller and borrowed for the handle's lifetime; everything
 * preprocess allocates is owned by the handle and released by spmm_b200_destroy.
 */
#ifndef SPMM_B200_H_
#define SPMM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SPMM_B200_EINVAL (-1)   /* bad argument */
#define SPMM_B200_ESTATE (-2)   /* call protocol violated (run before preprocess, ...) */
#define SPMM_B200_EIO (-3)      /* graph file missing / malformed */
#define SPMM_B200_ENOMEM (-4)   /* host allocation failed */

typedef struct spmm_b200_handle *spmm_b200_t;

/* ---- operator: class SpMM (PA4/handout/include/spmm_base.h:8-46) ------------------------- */

/* SpMM::SpMM(CSR *g, int feat_in)  (spmm_base.h:14-21; struct CSR: include/util.h:120-129).
 * d_ptr int32[num_v+1], d_idx int32[num_e], d_val f32[num_e]: device pointers. */
int spmm_b200_create(const int *d_ptr, const int *d_idx, const float *d_val, int num_v, int num_e,
                     int feat_in, spmm_b200_t *out);

/* SpMM::set_feat (spmm_base.h:26-29). Invalidates the plan: preprocess must be called again. */
int spmm_b200_set_feat(spmm_b200_t h, int feat_in);

/* Tunables, set before preprocess. Unknown names return SPMM_B200_EINVAL.
 *   "seg_len"   nonzeros per heavy-row segment; rows longer than this are split (0 = auto)
 *   "kslice"    feature columns per pass over the graph (0 = auto; else multiple of 4)
 *   "block"     threads per CTA (multiple of 32)
 *   "reorder"   1 = degree-bucketed row order, 0 = natural order, -1 (default) = natural for single-block plans when a
 *               full warp serves each row (K >= 128) and the graph is at least 8 waves of tasks long, else bucketed
 *   "light_steps" entries per lane group and stream task (0 = auto: 64 / groups, at least 16;
 *               128 on very large graphs at K >= 128; smaller on graphs of fewer than 4 waves of tasks, to
 *               fill whole waves of resident warps)
 *   "col_blocks" passes over A, each gathering from one band of B rows that fits the L2
 *               (0 = auto: 1 unless B is larger than the L2 and rows are long); needs ascending
 *               columns inside each row, otherwise falls back to 1
 *   "split_streams" -1 (default) = with several column blocks every pass goes out as two launches, the two halves of
 *               the rows, on two streams (each tail overlaps the next launch), 0 = one launch per column block, 1 = on
 *   "row_groups" contiguous row groups, balanced by nonzeros, that no task spans (0 = auto: 16 in natural row order, 2
 *               in bucketed order with several column blocks, else 1; at most 64): the unit of parallel planning and of
 *               the two-stream launches
 *   "host_bands" 1 = lay the column blocks out for spmm_b200_run_host: the last block takes the last 40 % of B's rows
 *               (its pass is bound by the PCIe transfer of C anyway), the blocks before it share the rest (the first
 *               pass starts sooner, the rest finishes under the upload of B); 10..90 = that percentage instead of 40.
 *               0 (default) = equal blocks, best for run(). Rows split into segments sum in a different association
 *               than with equal blocks (same tolerance); whole rows stay bit-exact
 *   "zero_copy" run_host / run_host_sharded: 1 (default) = when the output buffer is pinned host memory the last pass
 *               stores final rows straight into it (no separate device-to-host copy), 0 = always copy
 *   "tune"      measured kernel variant, 0 (default) or 1, see hpc_b200/csrc/spmm_kernels.cu
 *   "live_values" 0 (default) = the plan stages the edge values (SNAPSHOT, see preprocess); 1 = the plan stages each
 *               nonzero's position instead and every run reads the weights at run time from a value array
 *               (spmm_b200_run_values). On a handle from create_transposed / create_column_sorted the positions are
 *               those of the source handle's CSR, so one value array drives both. Part of the plan: changing it
 *               invalidates the plan
 *   "b_rows"    rows of B when A is a row block of a larger graph (0 = num_v). Part of the plan (column bounds
 *               check, 32-bit offset guard, column-block bands, run_host's copy of B): changing it after
 *               preprocess invalidates the plan
 * The reference's counterpart are the compile-time constants kBatchSize / kTasksPerBlock
 * (PA4/workspace/src/spmm_opt.cu:6-7). */
int spmm_b200_set_option(spmm_b200_t h, const char *name, long long value);

/* SpMM::preprocess(float *vin, float *vout)  (spmm_base.h:31; student version
 * PA4/workspace/src/spmm_opt.cu:37-69). Builds the plan: degree-bucketed row order, heavy-row
 * segments, staged col/val panels. vin/vout are hints only and are not written (the student's
 * preprocess zeroes vout, spmm_opt.cu:67-68; this engine's run overwrites vout instead).
 * Runs on `stream` and synchronises it before returning.
 * SNAPSHOT: for feat_in % 4 == 0 the plan stages a copy of idx/val ({col, val} panels) and run() reads only that
 * copy — unlike the reference's SpMMOpt::run, which reads idx/val at run time (PA4/workspace/src/spmm_opt.cu:22-25).
 * A caller that rewrites d_val in place afterwards (or d_idx, if the plan has a single column block and no row changes
 * its length) must call spmm_b200_refresh_values before the next run; any other change of the structure needs a new
 * preprocess. With option live_values = 1 run, run_host and run_host_sharded instead read the values at run time, as
 * the reference does: d_val, or on a derived handle the source handle's d_val (refresh_values is then needed only after
 * d_idx changes). */
int spmm_b200_preprocess(spmm_b200_t h, const float *vin, float *vout, void *stream);

/* Re-stages the plan's {col, val} panels from the caller's current d_idx / d_val (same ptr), asynchronously on
 * `stream`: two small kernels per column block, no host work, no new plan (GNN edge re-weighting between layers).
 * No reference counterpart (the reference reads idx/val live). On a live_values plan it re-stages idx and the positions. */
int spmm_b200_refresh_values(spmm_b200_t h, void *stream);

/* SpMM::run(float *vin, float *vout)  (spmm_base.h:32; PA4/handout/src/spmm_ref.cu:27-30).
 * Asynchronous on `stream` (a cudaStream_t; NULL = the default stream, as in the reference).
 * Fully overwrites vout[num_v*feat_in]; does not depend on its previous contents. Runs of one handle must not
 * overlap in time (they share the handle's partial-row workspace): issue them on one stream, or synchronise.
 * With several column blocks half of the launches go out on a second stream owned by the handle, forked from and
 * joined back to `stream` by events inside the call: to the caller everything is ordered on `stream` (also under
 * CUDA-graph capture). */
int spmm_b200_run(spmm_b200_t h, const float *vin, float *vout, void *stream);

/* C = A_val * B: run with the edge values of this call (no reference counterpart; DGL's u_mul_e_sum). val[p] is the
 * value of the nonzero at CSR position p, a device array of num_e floats — on a handle from create_transposed /
 * create_column_sorted, p is a position in the SOURCE handle's CSR and val holds the source's num_e floats. Needs a
 * plan built with option live_values = 1 (SPMM_B200_ESTATE otherwise, and without preprocess); val == NULL while
 * num_e > 0: SPMM_B200_EINVAL. Everything else is run's: asynchronous on `stream`, fully overwrites vout, column
 * blocks, two-stream launches, the stacked-layer epilogue and the alignment rules; capturable into a CUDA graph (the
 * graph reads val's contents at replay). The bits equal those of a snapshot plan with the same options after its
 * values are set to val and refreshed. */
int spmm_b200_run_values(spmm_b200_t h, const float *val, const float *vin, float *vout, void *stream);

/* run, plus the device time of its kernel in milliseconds (CUDA events on `stream` around the
 * launch). Synchronises. Counterpart of getCUDATime (PA4/handout/include/util.h:131-139). */
int spmm_b200_run_profiled(spmm_b200_t h, const float *vin, float *vout, void *stream, float *ms);

/* Stacked-layer epilogue (no reference counterpart; SURVEY.md 8e/8f-3). Besides vout, every finished C row r is
 * also stored at targets[t] + (row_offset + r) * feat_in for each t < n_targets — e.g. every rank's copy of the next
 * layer's B, mapped through NVLink peer memory — or, when `multicast` is non-NULL, once through that NVLS multicast
 * address of the same buffers (multimem.st). The all-gather of C then needs no separate collective: after the
 * kernel and a cross-rank barrier every rank holds the full C. Targets are device pointers, 16-byte aligned, of
 * b_rows * feat_in floats; n_targets <= 16; 0 switches the mode off. */
int spmm_b200_set_gather(spmm_b200_t h, int n_targets, float *const *targets, float *multicast, long long row_offset);

/* The transposed operator (no reference counterpart — PA4 is forward only; SURVEY.md 8f-3): a new handle over A^T,
 * built on the device from h's CSR, for the gradient dB = A^T * dC through the same plan and kernels. Inside a row of
 * A^T (a column of A) the nonzeros keep A's storage order (ascending row), so every output element is one in-order
 * FMA chain. The new handle OWNS its CSR arrays; its num_v = h's b_rows (rows of B), its b_rows = h's num_v, so
 * run(out, dC[num_v x feat_in], dB[b_rows x feat_in]). Use it like any handle (set_option, preprocess, run, destroy);
 * destroy it before h. spmm_b200_refresh_values on it re-reads h's current values. Synchronises `stream`. */
int spmm_b200_create_transposed(spmm_b200_t h, int feat_in, void *stream, spmm_b200_t *out);

/* SDDMM over the operator's sparsity pattern (no reference counterpart; PA4 is forward only). For every nonzero e of
 * row r (CSR position order, e in [0, num_e)):
 *     out[e] = sum_j x_row[r * feat_in + j] * x_col[idx[e] * feat_in + j]
 * in the fixed order documented in hpc_b200/csrc/sddmm.cu (results depend on feat_in only, not on any plan option).
 * x_row: num_v x feat_in (e.g. dC), x_col: b_rows x feat_in (e.g. B), out: num_e floats, fully overwritten.
 * With x_row = dC and x_col = B, out is dL/dval of C = A*B. Reads the caller's d_ptr / d_idx (not val), and no
 * workspace that run uses. Works on any handle (row block, transposed, column-sorted); out follows THAT handle's CSR
 * positions. x_row / x_col must be 16-byte aligned when feat_in % 4 == 0. num_e == 0: returns 0 without a CUDA call;
 * feat_in == 0: out is set to +0.0f. Needs preprocess (SPMM_B200_ESTATE otherwise); set_feat, the b_rows option and a
 * new preprocess invalidate it as they invalidate run. Asynchronous on `stream`. The first call after preprocess on a
 * plan with several column blocks allocates its band prefix (from the library's pool, on `stream`): make that call
 * before capturing sddmm into a CUDA graph. */
int spmm_b200_sddmm(spmm_b200_t h, const float *x_row, const float *x_col, float *out, void *stream);

/* Row-wise softmax over the operator's pattern (no reference counterpart), in h's CSR position order: for every
 * nonzero e of row r
 *     out[e] = exp(s[e] - m_r) / sum_{e' in r} exp(s[e'] - m_r),   m_r = max_{e' in r} s[e']
 * in the fixed order documented in hpc_b200/csrc/edge_softmax.cu: it depends on the row's length alone, not on any
 * plan option. Special values follow torch.softmax (a -inf score gives 0; a NaN or +inf anywhere in a row makes the
 * whole row NaN) except that a row whose scores are all -inf gives zeros (masking; torch gives NaN).
 * Reads only h's ptr (a valid CSR: ptr[0] = 0, nondecreasing, ptr[num_v] = num_e): needs no preprocess, works on every
 * handle (row block, transposed: normalising over a column of A, column-sorted). scores / out: num_e floats; out must
 * not overlap scores. Asynchronous on `stream`, allocates nothing (capturable into a CUDA graph). num_e == 0: returns
 * 0 without a CUDA call. A null handle, or null arrays with num_e > 0: SPMM_B200_EINVAL. */
int spmm_b200_edge_softmax(spmm_b200_t h, const float *scores, float *out, void *stream);

/* The gradient of spmm_b200_edge_softmax: with p its output and dp = dL/dp,
 *     ds[e] = p[e] * (dp[e] - sum_{e' in r} p[e'] * dp[e'])
 * in the same order. ds must not overlap p or dp. Same contract as spmm_b200_edge_softmax otherwise. */
int spmm_b200_edge_softmax_backward(spmm_b200_t h, const float *p, const float *dp, float *ds, void *stream);

/* amax / amin aggregation over the operator's rows (no reference counterpart; torch.sparse.mm(A, B, "amax" | "amin")).
 * For every row r, column j < feat_in and nonzero e of r the message is m(e, j) = val[e] * vin[idx[e] * feat_in + j]
 * (one rounded multiply, subnormals flushed to zero); vout[r * feat_in + j] is the message of the winning nonzero and
 * arg[r * feat_in + j] its CSR position (arg may be NULL). The winner is the maximum of a total order on (message,
 * position): a NaN ranks above every number (for amax and amin alike, so NaN propagates as in torch.amax); among
 * numbers the larger (AMAX) or smaller (AMIN) value wins; equal values, -0 == +0 included, go to the smaller CSR
 * position. The bits therefore depend on no plan option. An empty row gives +0.0f and arg = -1.
 * vin: b_rows x feat_in, vout / arg: num_v x feat_in, fully overwritten (also when num_e == 0); 16-byte aligned when
 * feat_in % 4 == 0. feat_in == 0: returns 0 without a CUDA call. Reads the caller's CURRENT d_ptr / d_idx / d_val, not
 * the plan's staged copy: no spmm_b200_refresh_values is needed after the values change. Needs preprocess (it validates
 * the columns against b_rows; SPMM_B200_ESTATE otherwise); set_feat, the b_rows option and a new preprocess invalidate
 * it as they invalidate run. Works on every handle (row block, transposed, column-sorted); outputs follow THAT handle's
 * CSR positions. With several column blocks it makes one pass per band of B, as run does. Asynchronous on `stream`, no
 * atomics, allocates nothing (capturable into a CUDA graph). The stacked-layer epilogue (set_gather), run_host and
 * set_replicate do not apply. A null handle, a bad op, or null arrays with work to do: SPMM_B200_EINVAL. */
#define SPMM_B200_REDUCE_AMAX 1
#define SPMM_B200_REDUCE_AMIN 2
int spmm_b200_reduce(spmm_b200_t h, int op, const float *vin, float *vout, int *arg, void *stream);

/* The gradient of spmm_b200_reduce, on t = spmm_b200_create_transposed(h, feat_in, ...) (any other handle, a
 * column-sorted one included, gives SPMM_B200_EINVAL; t needs no preprocess). dc: num_v x feat_in of h (dL/dvout), arg:
 * the forward's arg (required). With A^T row c holding entries k in storage order, e = perm[k] and r = the row of A of
 * entry k, entry k matches column j when arg[r * feat_in + j] == e:
 *     db[c, j] = sum over matching entries of val[e] * dc[r * feat_in + j]      (b_rows x feat_in; +0.0f if none)
 *     dval[e]  = sum over matching columns j of dc[r * feat_in + j] * vin[c * feat_in + j]      (num_e, h's positions)
 * in the fixed orders documented in hpc_b200/csrc/reduce.cu (db: tiles of 1024 entries; dval: sddmm's order with the
 * non-matching terms skipped), so the bits do not depend on any option. val is h's CURRENT d_val. db and dval are each
 * optional (NULL); vin (the forward's B) is needed only with dval. Arrays 16-byte aligned when feat_in % 4 == 0.
 * Asynchronous on `stream`, no atomics, allocates nothing (capturable into a CUDA graph). */
int spmm_b200_reduce_backward(spmm_b200_t t, const float *dc, const int *arg, const float *vin, float *db, float *dval,
                              void *stream);

/* The column-sorted operator (no reference counterpart): a new handle over the SAME matrix with every row stored in
 * ascending column order (stable: equal columns keep their storage order), built on the device. A CSR whose rows are
 * not column-sorted is otherwise kept in ONE column block — splitting an unsorted row at band boundaries would reorder
 * its FMA chain — and loses the L2-resident bands on large graphs; this is the opt-in: outputs equal the reference
 * run on the sorted CSR bit for bit (whole rows), and the reference run on the original order within the split-row
 * tolerance 1e-5 * sum|terms|. Borrows h's ptr, owns idx / val; use it like any handle, destroy it before h.
 * spmm_b200_refresh_values on it re-reads h's current values. Synchronises `stream`. */
int spmm_b200_create_column_sorted(spmm_b200_t h, int feat_in, void *stream, spmm_b200_t *out);

/* SpMMOpt::~SpMMOpt (PA4/workspace/include/spmm_opt.h:18-20). Waits for the device to finish what still reads the plan.
 * The plan's arrays go back to a memory pool the library keeps per device (cudaMemPool, release threshold = max), from
 * which the next preprocess on that device takes them: creating, re-planning and destroying operators does not pay the
 * driver's allocate / release cost again and again. SPMM_B200_POOL=0 in the environment selects plain cudaMalloc/cudaFree. */
int spmm_b200_destroy(spmm_b200_t h);

/* Hands the pooled memory that no live plan uses on the CURRENT device back to the driver (no reference counterpart;
 * the reference's cudaFree in ~SpMMOpt does it per operator). Synchronises the device. */
int spmm_b200_trim_memory(void);

/* Host-buffer convenience for callers that hold B and C on the host: H2D(vin) → run → D2H(vout)
 * on `stream`, then synchronise. The handle keeps device staging buffers of num_v*feat_in floats. With column
 * blocks B is uploaded band by band on a second stream while earlier passes compute; when h_vout is pinned
 * (cudaHostAlloc / cudaHostRegister) the last pass stores the final rows straight into it over PCIe.
 * (The reference's harness keeps everything on the device; this is the end-to-end call that
 * bench.py times as `e2e`.) */
int spmm_b200_run_host(spmm_b200_t h, const float *h_vin, float *h_vout, void *stream);

const char *spmm_b200_last_error(void);

/* Number of kernels the last spmm_b200_run launched (for bench.py's gpu_launches). */
int spmm_b200_launches_per_run(spmm_b200_t h);

/* ---- plan introspection (parity tests: plan must equal the CPU oracle bit for bit) --------- */

typedef struct {
    int num_v, num_e, feat_in;
    int seg_len;        /* effective nonzeros per segment */
    int kslice;         /* effective feature columns per pass */
    int n_slices;       /* ceil(feat_in / kslice) */
    int block;          /* threads per CTA */
    int n_light;        /* rows handled whole (row_perm length) */
    int n_heavy;        /* rows split into segments */
    int n_seg;          /* total segments */
    long long panel_len; /* entries (8 bytes each) in the staged col/val panel */
    int lanes;          /* lanes cooperating on one row in the light kernel */
    int vec;            /* float4 per lane */
    int n_ltask;        /* light-stream tasks (one warp each) */
    int n_utask;        /* all warp tasks of one feature slice: n_ltask + n_seg */
    long long lpanel_len; /* entries in the light stream panel */
    int light_steps;    /* target entries per lane group and task (selected block) */
    int reorder;        /* row order in effect for the selected block: 1 bucketed, 0 natural */
    int resident_warps; /* warps the device keeps resident for the kernel shape (sizes small graphs' tasks) */
    int n_col_blocks;   /* passes over A, one per band of B rows (1 = the whole matrix at once) */
    int col_begin, col_end; /* band of B rows of the selected column block */
    int persistent;     /* always 0: the single-launch mode it reported was removed; kept so that the layout of this
                           struct, and every reader of it, stays as it was */
    int n_row_groups;   /* row groups: contiguous row ranges balanced by nonzeros that no task spans (1 = whole bands) */
    int n_tickets;      /* always 0, for the same reason as `persistent` */
} spmm_b200_plan_info_t;

/* With n_col_blocks > 1 the plan holds one set of arrays per column block; plan_info / plan_copy
 * describe the block chosen here (0 after preprocess). n_light .. panel_len are per block. */
int spmm_b200_plan_select(spmm_b200_t h, int col_block);

int spmm_b200_plan_info(spmm_b200_t h, spmm_b200_plan_info_t *info);

/* Copy one plan array to the host. which:
 *   0 row_perm   int32[n_light]     light rows in processing order
 *   1 heavy_rows int32[n_heavy]     heavy rows in processing order
 *   2 heavy_seg0 int32[n_heavy+1]   first segment of each heavy row (prefix)
 *   3 seg_desc   int32[n_seg*4]     {row, panel_off, len, nnz_begin} per segment
 *   4 panel      int32[panel_len*2] {col * feat_in/4, float bits of val} pairs, segment-major (the column is stored as
 *                                   the B row's offset in float4 units, so a gather address is one multiply-add);
 *                                   each segment is padded with nops {-1, 0} to a multiple of 4 * (32 / lanes) entries
 *   5 light_desc int32[n_light*4]   {row, first CSR position, nonzeros, slot of its header in lpanel} per light
 *                                   row, same order as row_perm
 *   8 ltask      int32[n_ltask*2]   {lpanel offset, steps per lane group} per light-stream task
 *  10 utask      int32[n_utask*2]   the warp tasks of one feature slice in scheduling order: a light-stream task as in
 *                                   ltask, a heavy segment as {-1 - segment, 0}. Bucketed rows: segments first, then the
 *                                   light tasks; natural order: merged by the row each task starts with
 *   9 lpanel     int32[lpanel_len*2] light rows as a stream of {x, y} entries: header {0x80000000|row, 0},
 *                                   nonzero {col * feat_in/4, float bits of val}, nop {-1, -1}; within a task, entry j
 *                                   of lane group g sits at offset + j*groups + g; tasks are padded to 4-step multiples
 *   6 seg_hrow   int32[n_seg]       index into heavy_rows of each segment's row
 *   7 split      int32[(n_col_blocks+1)*num_v]  block-major: CSR position where column block b starts
 *                                   in row r (empty when n_col_blocks == 1)
 *  12 group_row  int32[n_row_groups+1] first row of each row group (row g's bound: first row with ptr >= g*nnz/groups)
 * Returns SPMM_B200_EINVAL when `bytes` is not the exact size. */
int spmm_b200_plan_copy(spmm_b200_t h, int which, void *host_dst, size_t bytes);

/* The row part of the plan computed from a HOST ptr array, no GPU needed (the same routine
 * preprocess uses after copying ptr to the host). Call once with the array arguments NULL to
 * get the counts, then with row_perm int32[n_light], heavy_rows int32[n_heavy], heavy_seg0
 * int32[n_heavy+1 (0 if none)], seg_desc int32[n_seg*4]. seg_len <= 0 selects the automatic
 * value for nnz = h_ptr[num_v] and feat_in. */
int spmm_b200_plan_host(const int *h_ptr, int num_v, int feat_in, long long seg_len, int reorder, int *row_perm,
                        int *n_light, int *heavy_rows, int *n_heavy, int *heavy_seg0, int *seg_desc,
                        int *n_seg, long long *panel_len);

/* The light-stream packing rule on the host (tests): cost[i] = nonzeros + 1 of the i-th light row in plan order;
 * dst int32[n] receives each row's header slot, ltask int32[2*n_ltask] the tasks (call with ltask = dst = NULL
 * first to get n_ltask / lpanel_len). groups = 32 / lanes. */
int spmm_b200_pack_light_host(const int *cost, int n, int groups, int steps, int *dst, int *ltask, int *n_ltask,
                              long long *lpanel_len);

/* ---- support (device pointers) ------------------------------------------------------------ */

/* allocate<float>'s fill (PA4/handout/include/data.h:24-37: curandGenerateNormal(0, 0.1)):
 * counter-based N(mean, stddev) fill, element i of (seed, stream_id) identical to the CPU
 * oracle's generator. */
int spmm_b200_fill_normal(float *d_dst, long long n, uint64_t seed, uint64_t stream_id, float mean,
                          float stddev, void *stream);

/* valid(float *y, float *y2, int num) (PA4/handout/src/valid.cu:3-13,41-56): number of elements
 * with |(y - y2) / y| > 1e-2 (IEEE divide). Synchronises. */
int spmm_b200_valid(const float *d_y, const float *d_y2, long long num, long long *mismatches,
                    void *stream);

/* ---- graphs (host pointers) ---------------------------------------------------------------- */

/* Synthetic stand-in for the OGB/DGL graphs the reference loads from ~/PA4/data
 * (PA4/handout/script/run_all.sh:11): power-law row degrees rescaled to exactly `nnz` with
 * maximum `max_deg` (the per-graph figure PA4/workspace/phase_2.log pins), columns drawn from
 * a popularity-skewed + local mixture, unique and ascending within a row.
 *   tail_k      degree weight = u^(-tail_k/4), tail_k in 1..4 (Pareto alpha = 4/tail_k)
 *   zero_ppm    fraction of empty rows, parts per million
 *   local_ppm   fraction of a row's columns drawn from the window [r-window, r+window]
 * ptr int32[num_v+1] and idx int32[nnz] are caller-allocated host arrays. */
int spmm_b200_gen_graph(int num_v, long long nnz, int max_deg, int tail_k, int zero_ppm,
                        int local_ppm, int window, uint64_t seed, int *ptr, int *idx);

/* Degrees only (first half of the above), deg int32[num_v]. */
int spmm_b200_gen_degrees(int num_v, long long nnz, int max_deg, int tail_k, int zero_ppm,
                          uint64_t seed, int *deg);

/* Host threads used by the OpenMP parts of the library (the generator above); overrides OMP_NUM_THREADS. */
int spmm_b200_set_host_threads(int n);

/* load_graph (PA4/handout/src/data.cu:3-66): <dir>/<dset>.config ("num_v num_e"),
 * <dset>.graph (text: num_v+1 ptr ints then num_e idx ints), binary caches
 * <dset>.graph.ptrdump / .edgedump (int32), written on first text read.
 * Pass ptr = idx = NULL to query the sizes only. */
int spmm_b200_load_graph(const char *datadir, const char *dset, int *num_v, int *num_e, int *ptr,
                         int *idx);

/* Writes <dset>.config plus either the text .graph (text != 0) or the two binary dumps. */
int spmm_b200_write_graph(const char *datadir, const char *dset, int num_v, int num_e,
                          const int *ptr, const int *idx, int text);

/* ---- multi-GPU (no reference counterpart; SURVEY.md §8e) ------------------------------------- */

/* nnz-balanced contiguous row partition: bounds[g] = first row r with ptr[r] >= g*nnz/parts
 * (64-bit arithmetic), bounds[0] = 0, bounds[parts] = num_v. h_ptr is a host array. */
int spmm_b200_partition_rows(const int *h_ptr, int num_v, int parts, int *bounds);

/* Cost-balanced variant: a row costs its nonzeros plus row_cost — the plan's per-row overhead (one header entry
 * per column block, whose C row is read and written there; spmm_b200_plan_row_cost gives the automatic plan's
 * figure). bounds[g] = first row r with ptr[r] + row_cost*r >= g*(nnz + row_cost*num_v)/parts. row_cost = 0 is
 * spmm_b200_partition_rows. */
int spmm_b200_partition_rows_weighted(const int *h_ptr, int num_v, int parts, int row_cost, int *bounds);

/* Column blocks the automatic plan uses for a graph of num_v rows and nnz nonzeros against a B of b_rows x feat_in
 * (= header entries per row of the staged plan): the row_cost to balance a partition with. */
int spmm_b200_plan_row_cost(int num_v, long long nnz, int b_rows, int feat_in);

/* Rebase one partition: out_ptr[i] = h_ptr[row_begin + i] - h_ptr[row_begin], i in [0, rows]. */
int spmm_b200_rebase_ptr(const int *h_ptr, int row_begin, int row_end, int *out_ptr);

/* ---- sharded host I/O, one process per GPU (hpc_b200/csrc/replicate.cu) ------------------------------------
 * The end-to-end call for a row partition over `world` ranks: B is replicated over NVLink instead of being uploaded
 * whole by every rank. peers_b[r] is rank r's full copy of B (b_rows * feat_in floats, 16-byte aligned) as mapped
 * into THIS process (symmetric / peer-mapped memory; peers_b[rank] is the local one), multicast_b the NVLS multicast
 * address of the same buffers or NULL, peers_flags[r] rank r's 2 * world zero-initialised uint32 flag words, mapped
 * the same way. world <= 16; world = 0 switches the mode off. Allocation and address exchange are the caller's
 * (bench.py: torch.distributed._symmetric_memory). */
int spmm_b200_set_replicate(spmm_b200_t h, int world, int rank, float *const *peers_b, float *multicast_b,
                            unsigned int *const *peers_flags);

/* Collective over the ranks (every rank calls it once per step, in the same order). h_vin is the WHOLE B on the
 * host (b_rows * feat_in floats), of which this rank reads only its share: B is cut into equal row chunks of about
 * 48 MB by a rule all ranks evaluate identically, and rank g uploads the g-th of `world` equal pieces of every chunk,
 * stores it into every rank's copy of B (multimem.st through the multicast address, else one peer store per rank) and
 * joins a cross-rank flag barrier per chunk — all on a second, high-priority stream, so that the upload and
 * replication of later chunks overlap the column-block passes over earlier ones. The rank's block of C (num_v *
 * feat_in floats) goes to h_vout: stored straight into it by the last pass when it is pinned, else copied.
 * Synchronises. PCIe carries about 4*b_rows*feat_in/world bytes in and 4*num_v*feat_in bytes out per rank. */
int spmm_b200_run_host_sharded(spmm_b200_t h, const float *h_vin, float *h_vout, void *stream);

/* Host-to-device bytes the last spmm_b200_run_host_sharded call of this handle copied (bench.py's accounting). */
long long spmm_b200_replicate_h2d_bytes(spmm_b200_t h);

/* ---- multi-GPU driver, one process and N devices (hpc_b200/csrc/multi.cu; SURVEY.md §8e) -------------------
 * No reference counterpart (single GPU; `// extern ncclComm_t* comms;`, PA4/handout/include/util.h:30). */
typedef struct spmm_b200_mg *spmm_b200_mg_t;

/* HOST CSR arrays of the whole graph. Rows are cut into n_devices contiguous blocks balanced by nnz
 * (spmm_b200_partition_rows), each block is uploaded to its device (devices[g], or g when devices is NULL; the same
 * device may be listed more than once), which also gets a full-size B, its block of C and one operator handle with
 * b_rows = num_v. n_devices <= 16. Peer access between the devices is switched on when they offer it. */
int spmm_b200_mg_create(const int *h_ptr, const int *h_idx, const float *h_val, int num_v, int num_e, int feat_in,
                        int n_devices, const int *devices, spmm_b200_mg_t *out);
/* spmm_b200_set_option on every device's handle. */
int spmm_b200_mg_set_option(spmm_b200_mg_t m, const char *name, long long value);
/* spmm_b200_preprocess on every device. */
int spmm_b200_mg_preprocess(spmm_b200_mg_t m);
/* n_devices, bounds int32[n_devices + 1] (device g owns rows [bounds[g], bounds[g+1])), whether peer access is on.
 * Any of the outputs may be NULL. */
int spmm_b200_mg_info(spmm_b200_mg_t m, int *n_devices, int *bounds, int *peer_access);
/* Device g's buffers: its full B (num_v * feat_in), its block of C, the full C (NULL until set_fused / allgather /
 * swap allocated it) and its operator handle. Any of the outputs may be NULL. */
int spmm_b200_mg_device_buffers(spmm_b200_mg_t m, int g, float **d_b, float **d_c_block, float **d_c_full, spmm_b200_t *op);
/* Host buffers in and out: h_vin = B (num_v * feat_in), h_vout = C (num_v * feat_in), pinned for overlap. Device g
 * uploads rows [g*num_v/N, (g+1)*num_v/N) of B and stores them into every device's copy through peer mappings
 * (cudaMemcpyPeerAsync without peer access), every device runs its block and downloads it. Synchronises. */
int spmm_b200_mg_run_host(spmm_b200_mg_t m, const float *h_vin, float *h_vout);
/* Device-resident step: C block = A block x (the device's B buffer) on every device, asynchronously. */
int spmm_b200_mg_run(spmm_b200_mg_t m);
/* Waits for everything queued on every device. */
int spmm_b200_mg_sync(spmm_b200_mg_t m);
/* Stacked layers without a collective: with on != 0 every following mg_run also stores each finished C row into
 * every device's full C (spmm_b200_set_gather over the peer mappings); after mg_sync the full C is complete
 * everywhere. Needs peer access and feat_in % 4 == 0. */
int spmm_b200_mg_set_fused(spmm_b200_mg_t m, int on);
/* The baseline for the same step: all-gather-v of the C blocks into every device's full C with NCCL (one grouped
 * ncclBroadcast per row block; libnccl.so.2 is opened on first use), asynchronously on the devices' streams. */
int spmm_b200_mg_allgather(spmm_b200_mg_t m);
/* Next layer: the full C becomes B and the old B becomes the full-C buffer (after mg_sync). */
int spmm_b200_mg_swap(spmm_b200_mg_t m);
int spmm_b200_mg_destroy(spmm_b200_mg_t m);

#ifdef __cplusplus
}
#endif
#endif /* SPMM_B200_H_ */
