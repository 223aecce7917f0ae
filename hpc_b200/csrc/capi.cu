// capi.cu — the extern "C" layer declared in include/spmm_b200.h.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <new>

#include "common.h"

namespace spmm_b200 {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
    // same information the reference prints before exiting (PA4/handout/include/util.h:63-84)
    set_error("Cuda failure: %s (%d) in %s at %s:%d", cudaGetErrorString(e), (int)e, what, file, line);
    return (int)e;
}

}  // namespace spmm_b200

using namespace spmm_b200;

extern "C" {

const char *spmm_b200_last_error(void) { return g_err; }

int spmm_b200_create(const int *d_ptr, const int *d_idx, const float *d_val, int num_v, int num_e,
                     int feat_in, spmm_b200_t *out) {
    if (!out || num_v < 0 || num_e < 0 || feat_in < 0 || (num_v > 0 && !d_ptr) ||
        (num_e > 0 && (!d_idx || !d_val))) {
        set_error("spmm_b200_create: bad arguments");
        return SPMM_B200_EINVAL;
    }
    spmm_b200_handle *h = new (std::nothrow) spmm_b200_handle();
    if (!h) {
        set_error("spmm_b200_create: out of host memory");
        return SPMM_B200_ENOMEM;
    }
    h->d_ptr = d_ptr;
    h->d_idx = d_idx;
    h->d_val = d_val;
    h->num_v = num_v;
    h->num_e = num_e;
    h->feat = feat_in;
    *out = h;
    return 0;
}

int spmm_b200_set_feat(spmm_b200_t h, int feat_in) {
    if (!h || feat_in < 0) {
        set_error("spmm_b200_set_feat: bad arguments");
        return SPMM_B200_EINVAL;
    }
    if (h->n_gather > 0 && feat_in % 4 != 0) {
        // the scalar fallback kernel has no stacked-layer epilogue: refuse rather than drop it silently
        set_error("spmm_b200_set_feat: the gather epilogue is on and needs feat_in %% 4 == 0 (switch it off first)");
        return SPMM_B200_EINVAL;
    }
    h->feat = feat_in;
    free_plan(h->plan);
    return 0;
}

int spmm_b200_set_option(spmm_b200_t h, const char *name, long long value) {
    if (!h || !name) {
        set_error("spmm_b200_set_option: null argument");
        return SPMM_B200_EINVAL;
    }
    if (!strcmp(name, "seg_len") && value >= 0) h->opt_seg_len = value;
    else if (!strcmp(name, "kslice") && value >= 0 && value % 4 == 0) h->opt_kslice = value;
    else if (!strcmp(name, "block") && value >= 32 && value <= 256 && value % 32 == 0) h->opt_block = value;
    else if (!strcmp(name, "reorder") && value >= -1 && value <= 1) h->opt_reorder = value;
    else if (!strcmp(name, "tune") && value >= 0 && value <= 1) h->opt_tune = value;
    else if (!strcmp(name, "light_steps") && value >= 0 && value <= 65536) h->opt_light_steps = value;
    else if (!strcmp(name, "col_blocks") && value >= 0 && value <= 64) h->opt_col_blocks = value;
    else if (!strcmp(name, "row_groups") && value >= 0 && value <= kMaxRowGroups) h->opt_row_groups = value;
    else if (!strcmp(name, "split_streams") && value >= -1 && value <= 1) h->opt_split_streams = value;
    else if (!strcmp(name, "host_bands") && (value == 0 || value == 1 || (value >= 10 && value <= 90))) h->opt_host_bands = value;
    else if (!strcmp(name, "live_values") && value >= 0 && value <= 1) h->opt_live_values = value;
    else if (!strcmp(name, "zero_copy") && value >= 0 && value <= 1) {
        h->opt_zero_copy = value;   // run_host only; not part of the plan
        return 0;
    }
    else if (!strcmp(name, "b_rows") && value >= 0 && value <= 0x7fffffffll) {
        // the plan depends on it (column bounds check, 32-bit offset guard, column-block bands)
        if ((int)value != h->b_rows) h->plan.ready = false;
        h->b_rows = (int)value;
        return 0;
    }
    else {
        set_error("spmm_b200_set_option: unknown option or bad value: %s = %lld", name, value);
        return SPMM_B200_EINVAL;
    }
    h->plan.ready = false;
    return 0;
}

int spmm_b200_set_gather(spmm_b200_t h, int n_targets, float *const *targets, float *multicast, long long row_offset) {
    if (!h || n_targets < 0 || n_targets > kMaxGather || (n_targets > 0 && !targets) || row_offset < 0) {
        set_error("spmm_b200_set_gather: bad arguments");
        return SPMM_B200_EINVAL;
    }
    if (n_targets > 0 && h->feat % 4 != 0) {
        set_error("spmm_b200_set_gather: needs feat_in %% 4 == 0");
        return SPMM_B200_EINVAL;
    }
    for (int t = 0; t < n_targets; ++t)
        if (!targets[t] || ((uintptr_t)targets[t] & 15)) {
            set_error("spmm_b200_set_gather: target %d is null or not 16-byte aligned", t);
            return SPMM_B200_EINVAL;
        }
    h->n_gather = n_targets;
    for (int t = 0; t < kMaxGather; ++t) h->gather[t] = t < n_targets ? targets[t] : nullptr;
    h->gather_mc = n_targets > 0 ? multicast : nullptr;
    h->gather_row0 = row_offset;
    return 0;
}

int spmm_b200_preprocess(spmm_b200_t h, const float *vin, float *vout, void *stream) {
    (void)vin;
    (void)vout;
    if (!h) {
        set_error("spmm_b200_preprocess: null handle");
        return SPMM_B200_EINVAL;
    }
    return build_plan(h, (cudaStream_t)stream);
}

// argument checks shared by run and run_profiled
static int check_run_args(const char *who, spmm_b200_t h, const float *vin, const float *vout) {
    if (!h) {
        set_error("%s: null handle", who);
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.ready) {
        set_error("%s: preprocess has not been called", who);
        return SPMM_B200_ESTATE;
    }
    if ((size_t)h->num_v * h->feat > 0 && (!vin || !vout)) {
        set_error("%s: null vin/vout", who);
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.scalar && (((uintptr_t)vin | (uintptr_t)vout) & 15)) {
        set_error("%s: vin/vout must be 16-byte aligned", who);
        return SPMM_B200_EINVAL;
    }
    return 0;
}

int spmm_b200_refresh_values(spmm_b200_t h, void *stream) {
    if (!h) {
        set_error("spmm_b200_refresh_values: null handle");
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.ready) {
        set_error("spmm_b200_refresh_values: preprocess has not been called");
        return SPMM_B200_ESTATE;
    }
    // a transposed handle first re-gathers its values from the handle it was built from
    int rc = regather_transposed_values(h, (cudaStream_t)stream);
    if (rc) return rc;
    return refresh_panels(h, (cudaStream_t)stream);
}

int spmm_b200_run(spmm_b200_t h, const float *vin, float *vout, void *stream) {
    int rc = check_run_args("spmm_b200_run", h, vin, vout);
    if (rc) return rc;
    return launch_spmm(h, vin, vout, (cudaStream_t)stream, &h->plan.launches);
}

int spmm_b200_run_values(spmm_b200_t h, const float *val, const float *vin, float *vout, void *stream) {
    int rc = check_run_args("spmm_b200_run_values", h, vin, vout);
    if (rc) return rc;
    if (!h->plan.live) {
        set_error("spmm_b200_run_values: the plan stages its values; set option live_values = 1 before preprocess");
        return SPMM_B200_ESTATE;
    }
    if (h->num_e > 0 && !val) {
        set_error("spmm_b200_run_values: null val");
        return SPMM_B200_EINVAL;
    }
    return launch_spmm(h, vin, vout, (cudaStream_t)stream, &h->plan.launches, nullptr, nullptr, val);
}

int spmm_b200_run_profiled(spmm_b200_t h, const float *vin, float *vout, void *stream, float *ms) {
    if (!ms) {
        set_error("spmm_b200_run_profiled: null argument");
        return SPMM_B200_EINVAL;
    }
    int rc = check_run_args("spmm_b200_run_profiled", h, vin, vout);
    if (rc) return rc;
    cudaEvent_t ev[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; ++i) {
        cudaError_t ce = cudaEventCreate(&ev[i]);
        if (ce != cudaSuccess) {
            if (i == 1) cudaEventDestroy(ev[0]);
            SB_CUDA(ce);
        }
    }
    cudaStream_t s = (cudaStream_t)stream;
    cudaError_t e = cudaEventRecord(ev[0], s);
    rc = launch_spmm(h, vin, vout, s, &h->plan.launches);
    if (e == cudaSuccess) e = cudaEventRecord(ev[1], s);
    if (e == cudaSuccess) e = cudaEventSynchronize(ev[1]);
    if (rc == 0 && e == cudaSuccess) e = cudaEventElapsedTime(ms, ev[0], ev[1]);
    for (int i = 0; i < 2; ++i) cudaEventDestroy(ev[i]);
    if (rc) return rc;
    SB_CUDA(e);
    return 0;
}

}  // extern "C"

namespace spmm_b200 {
// run_host's output path: when h_vout is pinned (device-mapped) host memory the last pass stores the final rows
// straight into it over PCIe — the download then overlaps the pass instead of following it (measured on the reddit
// shape, K=256: 9.3 ms vs 10.3 ms for run + copy, profiles/r02_zero_copy_probe.json). Pageable memory, a misaligned
// pointer, the scalar fallback kernel or option zero_copy = 0: NULL, and the caller copies C out afterwards.
float *host_out_mapping(const spmm_b200_handle *h, float *h_vout) {
    if (!h->opt_zero_copy || h->plan.scalar || ((uintptr_t)h_vout & 15)) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, h_vout) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    if (at.type != cudaMemoryTypeHost || !at.devicePointer) return nullptr;
    return static_cast<float *>(at.devicePointer);
}
}  // namespace spmm_b200

extern "C" {

int spmm_b200_run_host(spmm_b200_t h, const float *h_vin, float *h_vout, void *stream) {
    if (!h || !h_vin || !h_vout) {
        set_error("spmm_b200_run_host: null argument");
        return SPMM_B200_EINVAL;
    }
    if (!h->plan.ready) {
        set_error("spmm_b200_run_host: preprocess has not been called");
        return SPMM_B200_ESTATE;
    }
    const size_t n = (size_t)h->num_v * h->feat;
    const size_t nb = (size_t)(h->b_rows > 0 ? h->b_rows : h->num_v) * h->feat;
    if (n == 0) return 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (h->stage_elems < n || h->stage_in_elems < nb) {
        cudaFree(h->d_stage_in);
        cudaFree(h->d_stage_out);
        h->d_stage_in = h->d_stage_out = nullptr;
        h->stage_elems = h->stage_in_elems = 0;
        SB_CUDA(cudaMalloc((void **)&h->d_stage_in, nb * sizeof(float)));
        SB_CUDA(cudaMalloc((void **)&h->d_stage_out, n * sizeof(float)));
        h->stage_elems = n;
        h->stage_in_elems = nb;
    }
    int rc;
    const Plan &p = h->plan;
    float *out_map = host_out_mapping(h, h_vout);
    if (p.n_col_blocks > 1) {
        // Column block b only gathers from its band of B rows: upload the bands in order on a second stream and
        // let each pass wait for its own band, so the PCIe transfer of later bands overlaps the earlier passes.
        if (!h->copy_stream) SB_CUDA(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
        while ((int)h->band_events.size() < p.n_col_blocks) {
            cudaEvent_t e;
            SB_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
            h->band_events.push_back(e);
        }
        // the copy stream must not run ahead of work already queued on the caller's stream
        SB_CUDA(cudaEventRecord(h->band_events[0], s));
        SB_CUDA(cudaStreamWaitEvent(h->copy_stream, h->band_events[0], 0));
        for (int b = 0; b < p.n_col_blocks; ++b) {
            const size_t off = (size_t)p.blocks[b].col_begin * h->feat;
            const size_t cnt = (size_t)(p.blocks[b].col_end - p.blocks[b].col_begin) * h->feat;
            SB_CUDA(cudaMemcpyAsync(h->d_stage_in + off, h_vin + off, cnt * sizeof(float), cudaMemcpyHostToDevice,
                                    h->copy_stream));
            SB_CUDA(cudaEventRecord(h->band_events[b], h->copy_stream));
        }
        rc = launch_spmm(h, h->d_stage_in, h->d_stage_out, s, &h->plan.launches, h->band_events.data(), out_map);
    } else {
        SB_CUDA(cudaMemcpyAsync(h->d_stage_in, h_vin, nb * sizeof(float), cudaMemcpyHostToDevice, s));
        rc = launch_spmm(h, h->d_stage_in, h->d_stage_out, s, &h->plan.launches, nullptr, out_map);
    }
    if (rc) return rc;
    if (!out_map) SB_CUDA(cudaMemcpyAsync(h_vout, h->d_stage_out, n * sizeof(float), cudaMemcpyDeviceToHost, s));
    SB_CUDA(cudaStreamSynchronize(s));
    return 0;
}

int spmm_b200_destroy(spmm_b200_t h) {
    if (!h) return 0;
    free_plan(h->plan);
    if (h->t_ptr || h->t_idx || h->t_val || h->t_perm) {   // the transposed operator's CSR: back to its device's pool
        int cur = -1;
        const bool hop = h->t_device >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != h->t_device && cudaSetDevice(h->t_device) == cudaSuccess;
        cudaDeviceSynchronize();
        pool_free(h->t_ptr, cudaStreamLegacy);
        pool_free(h->t_idx, cudaStreamLegacy);
        pool_free(h->t_val, cudaStreamLegacy);
        pool_free(h->t_perm, cudaStreamLegacy);
        if (hop) cudaSetDevice(cur);
    }
    cudaFree(h->d_stage_in);
    cudaFree(h->d_stage_out);
    for (cudaEvent_t e : h->band_events) cudaEventDestroy(e);
    if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
    if (h->aux_stream) cudaStreamDestroy(h->aux_stream);
    if (h->aux_fork) cudaEventDestroy(h->aux_fork);
    if (h->aux_join) cudaEventDestroy(h->aux_join);
    delete h;
    return 0;
}

int spmm_b200_trim_memory(void) { return trim_pool_memory(); }

int spmm_b200_launches_per_run(spmm_b200_t h) { return h ? h->plan.launches : 0; }

int spmm_b200_plan_select(spmm_b200_t h, int col_block) {
    if (!h || !h->plan.ready || col_block < 0 || col_block >= h->plan.n_col_blocks) {
        set_error("spmm_b200_plan_select: no such column block");
        return SPMM_B200_EINVAL;
    }
    h->plan_select = col_block;
    return 0;
}

int spmm_b200_plan_info(spmm_b200_t h, spmm_b200_plan_info_t *info) {
    if (!h || !info || !h->plan.ready) {
        set_error("spmm_b200_plan_info: no plan");
        return h && info ? SPMM_B200_ESTATE : SPMM_B200_EINVAL;
    }
    const Plan &p = h->plan;
    const BlockPlan &b = p.blocks[h->plan_select];
    info->num_v = h->num_v;
    info->num_e = h->num_e;
    info->feat_in = h->feat;
    info->seg_len = p.seg_len;
    info->kslice = p.kslice;
    info->n_slices = p.n_slices;
    info->block = p.block;
    info->n_light = b.n_light;
    info->n_heavy = b.n_heavy;
    info->n_seg = b.n_seg;
    info->panel_len = b.panel_len;
    info->lanes = p.lanes;
    info->vec = p.vec;
    info->n_ltask = b.n_ltask;
    info->n_utask = b.n_utask;
    info->lpanel_len = b.lpanel_len;
    info->light_steps = b.light_steps;
    info->resident_warps = (int)p.slots;
    info->reorder = b.reorder;
    info->n_col_blocks = p.n_col_blocks;
    info->col_begin = b.col_begin;
    info->col_end = b.col_end;
    info->persistent = 0;
    info->n_row_groups = p.n_groups;
    info->n_tickets = 0;
    return 0;
}

int spmm_b200_plan_copy(spmm_b200_t h, int which, void *host_dst, size_t bytes) {
    if (!h || !h->plan.ready) {
        set_error("spmm_b200_plan_copy: no plan");
        return SPMM_B200_ESTATE;
    }
    const Plan &pl = h->plan;
    const BlockPlan &p = pl.blocks[h->plan_select];
    const void *src = nullptr;
    size_t want = 0;
    switch (which) {
        case 0: src = p.d_light_desc; want = sizeof(int) * (size_t)p.n_light; break;
        case 1: src = p.d_seg_desc; want = sizeof(int) * (size_t)p.n_heavy; break;
        case 2: src = p.d_heavy_seg0; want = p.n_heavy ? sizeof(int) * ((size_t)p.n_heavy + 1) : 0; break;
        case 3: src = p.d_seg_desc; want = sizeof(SegDesc) * (size_t)p.n_seg; break;
        case 4: src = p.d_panel; want = sizeof(int2) * (size_t)p.panel_len; break;
        case 5: src = p.d_light_desc; want = sizeof(int4) * (size_t)p.n_light; break;
        case 6: src = p.d_seg_hrow; want = sizeof(int) * (size_t)p.n_seg; break;
        case 8: src = p.d_utask; want = sizeof(int2) * (size_t)p.n_ltask; break;
        case 10: src = p.d_utask; want = sizeof(int2) * (size_t)p.n_utask; break;
        case 9: src = p.d_lpanel; want = sizeof(int2) * (size_t)p.lpanel_len; break;
        case 7:
            src = pl.d_split;
            want = pl.n_col_blocks > 1 ? sizeof(int) * (size_t)(pl.n_col_blocks + 1) * h->num_v : 0;
            break;
        case 12: {
            want = pl.group_row.empty() ? 0 : sizeof(int) * pl.group_row.size();
            if (bytes != want) break;
            if (want) memcpy(host_dst, pl.group_row.data(), want);
            return 0;
        }
        default: set_error("spmm_b200_plan_copy: unknown array %d", which); return SPMM_B200_EINVAL;
    }
    if (bytes != want) {
        set_error("spmm_b200_plan_copy: array %d is %zu bytes, caller gave %zu", which, want, bytes);
        return SPMM_B200_EINVAL;
    }
    if (want == 0) return 0;
    if (!src) {
        set_error("spmm_b200_plan_copy: array %d is empty", which);
        return SPMM_B200_ESTATE;
    }
    // No kernel reads arrays 0, 1 and 8, so the device does not keep them. They are projections of the arrays that `src` is:
    // row_perm[i] == light_desc[i].x; heavy_rows[i] == seg_desc[heavy_seg0[i]].row; ltask == the entries of utask with x >= 0
    // (not a heavy segment) in their order: planning takes the light tasks in sequence in either row order, and the row
    // groups' concatenation shifts both arrays by the same offsets.
    int *out = static_cast<int *>(host_dst);
    if (which == 0) {
        std::vector<int4> light((size_t)p.n_light);
        SB_CUDA(cudaMemcpy(light.data(), src, sizeof(int4) * light.size(), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < light.size(); ++i) out[i] = light[i].x;
    } else if (which == 1) {
        std::vector<SegDesc> segs((size_t)p.n_seg);
        std::vector<int> seg0((size_t)p.n_heavy);
        SB_CUDA(cudaMemcpy(segs.data(), src, sizeof(SegDesc) * segs.size(), cudaMemcpyDeviceToHost));
        SB_CUDA(cudaMemcpy(seg0.data(), p.d_heavy_seg0, sizeof(int) * seg0.size(), cudaMemcpyDeviceToHost));
        for (size_t i = 0; i < seg0.size(); ++i) out[i] = segs[(size_t)seg0[i]].row;
    } else if (which == 8) {
        std::vector<int2> utask((size_t)p.n_utask);
        SB_CUDA(cudaMemcpy(utask.data(), src, sizeof(int2) * utask.size(), cudaMemcpyDeviceToHost));
        int2 *ltask = static_cast<int2 *>(host_dst);
        for (size_t i = 0, n = 0; i < utask.size() && n < (size_t)p.n_ltask; ++i)
            if (utask[i].x >= 0) ltask[n++] = utask[i];
    } else {
        SB_CUDA(cudaMemcpy(host_dst, src, want, cudaMemcpyDeviceToHost));
    }
    return 0;
}

int spmm_b200_fill_normal(float *d_dst, long long n, uint64_t seed, uint64_t stream_id, float mean,
                          float stddev, void *stream) {
    if (n < 0 || (n > 0 && !d_dst)) {
        set_error("spmm_b200_fill_normal: bad arguments");
        return SPMM_B200_EINVAL;
    }
    return launch_fill_normal(d_dst, n, seed, stream_id, mean, stddev, (cudaStream_t)stream);
}

int spmm_b200_valid(const float *d_y, const float *d_y2, long long num, long long *mismatches, void *stream) {
    if (!mismatches || num < 0 || (num > 0 && (!d_y || !d_y2))) {
        set_error("spmm_b200_valid: bad arguments");
        return SPMM_B200_EINVAL;
    }
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long *d_count = nullptr;
    SB_CUDA(cudaMalloc((void **)&d_count, sizeof(unsigned long long)));
    cudaError_t e = cudaMemsetAsync(d_count, 0, sizeof(unsigned long long), s);
    int rc = 0;
    if (e == cudaSuccess) rc = launch_valid(d_y, d_y2, num, d_count, s);
    unsigned long long host = 0;
    if (e == cudaSuccess && rc == 0)
        e = cudaMemcpyAsync(&host, d_count, sizeof(host), cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess && rc == 0) e = cudaStreamSynchronize(s);
    cudaFree(d_count);
    if (rc) return rc;
    SB_CUDA(e);
    *mismatches = (long long)host;
    return 0;
}

}  // extern "C"
