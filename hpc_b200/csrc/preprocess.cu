// preprocess.cu — builds the execution plan of one (CSR, K) pair.
//
// Takes the place of the student's SpMMOpt::preprocess (PA4/workspace/src/spmm_opt.cu:37-69:
// copy ptr to the host, cut every row into <=256-nnz tasks, random_shuffle, upload, memset
// vout). The plan here is deterministic and fully specified so the CPU oracle
// (oracle/plan_oracle.py) can restate it and the tests compare bit for bit:
//
//   deg(r)    = ptr[r+1] - ptr[r]
//   heavy(r)  = deg(r) > seg_len
//   bucket(r) = bit length of deg(r)                      (0 for an empty row)
//   order     = rows by (bucket descending, r ascending)  (natural order when reorder = 0)
//   row_perm  = the non-heavy rows in that order
//   heavy rows, in that order, are cut into nseg = ceil(deg/seg_len) nnz-balanced segments
//               [begin + floor(j*deg/nseg), begin + floor((j+1)*deg/nseg)),  j = 0..nseg-1
//   panel     = the segments' {col * K/4, val} pairs back to back, each segment padded with nop entries {-1, 0} to a
//               multiple of 4 * (32 / lanes) entries (whole gather batches, 16-byte granules for the TMA copies)
//   lpanel    = the rows of row_perm as a stream: per row a header {0x80000000 | row, 0} and its {col, val}
//               entries, packed into equal-sized warp tasks by pack_light_host (rule stated there)
//   column blocks: when B exceeds the L2 (auto_col_blocks), every row is split at the band boundaries
//               (split[b][r]) and the whole plan above is built once per block over [split[b][r], split[b+1][r])
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <vector>

#include "common.h"

namespace spmm_b200 {

// SPMM_B200_PREP_TRACE=1: per-phase wall times of preprocess on stderr (tools/prep_probe.py)
struct PrepTrace {
    bool on = getenv("SPMM_B200_PREP_TRACE") != nullptr;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void lap(const char *what) {
        if (!on) return;
        auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[prep] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

void free_plan(Plan &p) {
    // the arrays came from the library's pool of p.device (pool.cu): wait, like cudaFree would, for whatever still reads the
    // plan, then hand them back in the order of the legacy stream
    int cur = -1;
    const bool hop = p.device >= 0 && cudaGetDevice(&cur) == cudaSuccess && cur != p.device && cudaSetDevice(p.device) == cudaSuccess;
    if (p.d_split || !p.blocks.empty()) cudaDeviceSynchronize();
    auto release = [](void *q) { pool_free(q, cudaStreamLegacy); };
    for (BlockPlan &b : p.blocks) {
        release(b.d_light_desc);
        release(b.d_utask);
        release(b.d_heavy_seg0);
        release(b.d_seg_desc);
        release(b.d_seg_hrow);
        // d_lpanel, d_panel, d_part, d_seg_count point into the arenas below
    }
    release(p.d_lpanel_all);
    release(p.d_panel_all);
    release(p.d_part_all);
    release(p.d_seg_count_all);
    release(p.d_split);
    release(p.d_sddmm_vp);
    if (hop) cudaSetDevice(cur);
    p = Plan();
}

static inline int bit_length(unsigned x) { return x ? 32 - __builtin_clz(x) : 0; }

int auto_seg_len(long long nnz, int lanes) {
    // Rows longer than this are cut into nnz-balanced segments, one warp each, their col/val
    // staged through shared memory by TMA. Measured on B200 (profiles/r01_sweep.md):
    //  * a full warp per row (K >= 128): equal-sized staged work units beat whole-row warps from
    //    ~256 nonzeros up on every graph shape;
    //  * narrower lane groups (K < 128): a segment carries only lanes*16 bytes per nonzero, so the
    //    per-segment partial + counter cost wants longer segments on big graphs (reddit K=32:
    //    1024), while small graphs are tail-bound and want short ones (arxiv K=32: 128):
    //    next power of two of nnz/65536, clamped to [128, 1024].
    if (lanes >= 32) return 256;
    long long t = nnz / 65536;
    int l = 128;
    while (l < t && l < 1024) l <<= 1;
    return l;
}

int auto_kslice(int num_v, int feat) {
    (void)num_v;
    if (feat % 4 != 0) return feat;
    // Measured on B200 (profiles/r01_sweep.md): narrower feature slices never paid for the extra
    // passes over col/val — the 126 MB L2 keeps the hot B rows even when B is larger than L2 —
    // so a pass covers up to 256 columns (32 lanes x 2 float4).
    return feat < 256 ? ((feat + 3) & ~3) : 256;
}

// Column blocks: when B does not fit the L2, A is processed as n column blocks (C = sum_b A[:, b]·B[b, :]),
// one pass each, so that every pass gathers from an L2-resident band of B and HBM sees B about once.
// Worth it only while a row still has enough nonzeros per block to amortise re-reading its C row.
int auto_col_blocks(long long b_rows, int feat, long long nnz, int num_v) {
    const long long b_bytes = b_rows * feat * 4ll;
    if (feat % 4 != 0 || num_v <= 0 || b_bytes <= (96ll << 20)) return 1;
    long long nb = (b_bytes + kBandBytes - 1) / kBandBytes;
    if (nb > 16) return 1;
    if (nnz / num_v / nb < 64) return 1;
    return (int)nb;
}

// Host-only core of the plan (also exported as spmm_b200_plan_host for CPU-side tests).
// Row r owns CSR positions [rb[r], re[r]) (rb = ptr, re = ptr + 1 for the whole matrix; a column block
// passes its own bounds). skip_empty drops rows with no nonzero in the block (passes after the first).
// `pad`: every segment's panel span is padded (with nop entries) to a multiple of `pad` entries: 4 gather steps
// of all lane groups, so the kernel reads whole batches without bounds checks.
int plan_rows_host(const int *rb, const int *re, int M, int seg_len, int reorder, int skip_empty, int pad,
                   std::vector<int> &row_perm, std::vector<int> &heavy_rows, std::vector<int> &heavy_seg0,
                   std::vector<SegDesc> &segs, long long *panel_len_out, int row0 = 0, int row1 = -1) {
    // a row range [row0, row1) may be planned on its own (row groups are planned in parallel and concatenated)
    if (row1 < 0) row1 = M;
    const int base = row0, count = row1 - row0;
    // stable counting sort by bucket, descending
    std::vector<int> order((size_t)count);
    if (reorder) {
        size_t cnt[34] = {0};
        for (int r = row0; r < row1; ++r) {
            const int d = re[r] - rb[r];
            if (d < 0) {
                set_error("CSR ptr decreases at row %d", r);
                return SPMM_B200_EINVAL;
            }
            ++cnt[bit_length((unsigned)d)];
        }
        size_t start[34];
        size_t run = 0;
        for (int b = 33; b >= 0; --b) {
            start[b] = run;
            run += cnt[b];
        }
        for (int r = row0; r < row1; ++r) order[start[bit_length((unsigned)(re[r] - rb[r]))]++] = r;
    } else {
        for (int r = 0; r < count; ++r) order[r] = base + r;
    }

    row_perm.clear();
    heavy_rows.clear();
    heavy_seg0.clear();
    segs.clear();
    row_perm.reserve(count);
    long long panel_len = 0;
    for (int k = 0; k < count; ++k) {
        const int r = order[k];
        const int begin = rb[r];
        const int d = re[r] - begin;
        if (d == 0 && skip_empty) continue;
        if (d <= seg_len) {
            row_perm.push_back(r);
            continue;
        }
        heavy_rows.push_back(r);
        heavy_seg0.push_back((int)segs.size());
        const int nseg = (int)(((long long)d + seg_len - 1) / seg_len);
        for (int j = 0; j < nseg; ++j) {
            const int b = begin + (int)((long long)j * d / nseg);
            const int e = begin + (int)((long long)(j + 1) * d / nseg);
            SegDesc s;
            s.row = r;
            s.panel_off = (int)panel_len;
            s.len = e - b;
            s.nnz_begin = b;
            segs.push_back(s);
            panel_len += (s.len + pad - 1) / pad * pad;
        }
    }
    if (!heavy_rows.empty()) heavy_seg0.push_back((int)segs.size());
    if (panel_len > 0x7fffffffll) {
        set_error("panel too large");
        return SPMM_B200_EINVAL;
    }
    *panel_len_out = panel_len;
    return 0;
}

// Light rows as a stream. Rows are taken in plan order; each costs deg + 1 entries (a header carrying the row id,
// then its nonzeros). A task has `groups` lanes (one per lane group of the warp). A row goes to the least-filled
// lane of the current task (lowest index on ties); if that lane is non-empty and the row would take it past
// `steps` entries, the task is closed and the row opens the next one. A task's lanes are interleaved in the
// panel — entry j of lane g sits at off + j*groups + g — and padded with nops to the longest lane rounded up to a
// multiple of 4 steps (whole gather batches; it also keeps every task on a 16-byte boundary).
long long pack_light_host(const int *cost, int n, int groups, int steps, int *dst, std::vector<int2> &tasks) {
    tasks.clear();
    std::vector<int> fill((size_t)groups, 0);
    long long off = 0;
    auto close_task = [&]() {
        int mx = 0;
        for (int x : fill) mx = std::max(mx, x);
        mx = (mx + 3) & ~3;   // whole batches of 4 steps: the kernel reads a task without bounds checks
        tasks.push_back(make_int2((int)off, mx));
        off += (long long)mx * groups;
        std::fill(fill.begin(), fill.end(), 0);
    };
    for (int i = 0; i < n; ++i) {
        int g = 0;
        for (int q = 1; q < groups; ++q)
            if (fill[q] < fill[g]) g = q;
        if (fill[g] > 0 && fill[g] + cost[i] > steps) {
            close_task();
            g = 0;
        }
        dst[i] = (int)(off + (long long)fill[g] * groups + g);
        fill[g] += cost[i];
    }
    bool any = false;
    for (int x : fill) any |= x > 0;
    if (any) close_task();
    return off;
}

// Entries per lane group and stream task: 64 per warp task, at least 16 per lane group; 128 when a full warp
// serves each row and the block is longer than 64 waves (measured, profiles/r01_sweep.md: arxiv K=256 0.142 / 0.155 ms
// at 64 / 128; reddit K=256 6.28 / 6.14 ms; products K=256 12.45 / 12.09 ms; K=32 shapes flat from 8 to 64). Small graphs are quantised by waves — 1.1 waves of tasks
// take as long as 2 — so when the light rows amount to fewer than 4 waves of default-sized tasks the size is
// chosen to fill a whole number of waves of the warps the device keeps resident (`slots`, minus the heavy
// segments that run beside them).
int auto_light_steps(int groups, long long total_cost, long long slots, long long heavy_tasks) {
    int dflt = 64 / groups;
    if (dflt < 16) dflt = 16;
    if (slots <= 0 || total_cost <= 0) return dflt;
    if (groups == 1 && total_cost >= 64ll * slots * 64) return 128;   // very large graphs: fewer, longer tasks
    long long avail = slots - heavy_tasks % slots;
    if (avail < slots / 2) avail = slots;
    const long long per_wave = avail * groups * (long long)dflt;
    if (total_cost >= 4 * per_wave) return dflt;
    const long long waves = (total_cost + per_wave - 1) / per_wave;
    long long st = (total_cost + waves * avail * groups - 1) / (waves * avail * groups);
    st += st / 16 + 1;   // head-room: lanes are filled to within one row of the target
    if (st < 16) st = 16;
    return (int)(st < dflt ? st : dflt);
}

// The host arrays of one column block, from host planning to their upload (the block's counts go to its BlockPlan).
struct BlockArrays {
    std::vector<int4> light;
    std::vector<int2> utask;
    std::vector<SegDesc> segs;
    std::vector<int> heavy_seg0, seg_hrow;
    int rc = 0;
    char err[256] = "";   // set_error keeps one message per thread, and the blocks are planned on several
};

// The row groups (contiguous row ranges) are planned independently of each other — a task never spans a group bound, and
// the row order (natural or degree buckets) applies INSIDE a group — so planning group by group and concatenating
// (offsets shifted by what precedes) is the whole plan. The groups run in parallel on the host (OpenMP), which is what
// brings preprocess for the products shape (2.4 M rows) from ~75 ms of serial host work to a few ms. One group is the
// ungrouped plan.
static void plan_block_groups(const spmm_b200_handle *h, const int *rb, const int *re, int skip_empty, int reorder, const int *group_row,
                              int n_groups, BlockPlan &bp, BlockArrays &a) {
    const Plan &p = h->plan;
    const int M = h->num_v;
    const int groups = 32 / p.lanes, pad = 4 * groups;
    struct Part {
        std::vector<int> row_perm, heavy_rows, heavy_seg0, cost, dst;
        std::vector<SegDesc> segs;
        std::vector<int2> ltasks, utask;
        long long panel_len = 0, lpanel_len = 0, total_cost = 0;
        int rc = 0;
    };
    std::vector<Part> part((size_t)n_groups);
#pragma omp parallel for schedule(dynamic, 1)
    for (int g = 0; g < n_groups; ++g) {
        Part &x = part[g];
        x.rc = plan_rows_host(rb, re, M, p.seg_len, reorder, skip_empty, pad, x.row_perm, x.heavy_rows, x.heavy_seg0, x.segs, &x.panel_len,
                              group_row[g], group_row[g + 1]);
        x.cost.resize(x.row_perm.size());
        for (size_t i = 0; i < x.row_perm.size(); ++i) {
            x.cost[i] = re[x.row_perm[i]] - rb[x.row_perm[i]] + 1;
            x.total_cost += x.cost[i];
        }
    }
    long long total = 0, n_seg = 0;
    for (Part &x : part) {
        if (x.rc) {
            a.rc = x.rc;
            snprintf(a.err, sizeof(a.err), "row planning failed");
            return;
        }
        total += x.total_cost;
        n_seg += (long long)x.segs.size();
    }
    int steps = p.light_steps;
    if (h->opt_light_steps <= 0) steps = auto_light_steps(groups, total, p.slots, n_seg * p.n_slices);
    bp.light_steps = steps;
#pragma omp parallel for schedule(dynamic, 1)
    for (int g = 0; g < n_groups; ++g) {
        Part &x = part[g];
        const int n = (int)x.row_perm.size();
        x.dst.resize((size_t)n);
        x.lpanel_len = pack_light_host(x.cost.data(), n, groups, steps, x.dst.data(), x.ltasks);
        x.utask.reserve(x.ltasks.size() + x.segs.size());
        if (reorder) {
            // degree buckets: the heavy segments (the longest rows) first, then the light tasks
            for (size_t si = 0; si < x.segs.size(); ++si) x.utask.push_back(make_int2(-1 - (int)si, 0));
            for (const int2 &t : x.ltasks) x.utask.push_back(t);
            continue;
        }
        // natural order: light tasks and heavy segments merged by the row they start with, so that a heavy row runs next
        // to its neighbours (whose B rows it shares in L2) instead of ahead of everything
        size_t li = 0, si = 0, first_i = 0;
        while (li < x.ltasks.size() || si < x.segs.size()) {
            int lrow = 0x7fffffff;
            if (li < x.ltasks.size()) {
                while (first_i < (size_t)n && x.dst[first_i] < x.ltasks[li].x) ++first_i;
                if (first_i < (size_t)n) lrow = x.row_perm[first_i];
            }
            if (si < x.segs.size() && x.segs[si].row < lrow) {
                x.utask.push_back(make_int2(-1 - (int)si, 0));
                ++si;
            } else {
                x.utask.push_back(x.ltasks[li]);
                ++li;
            }
        }
    }
    // concatenate, shifting every offset by what precedes
    std::vector<long long> b_light((size_t)n_groups + 1, 0), b_heavy((size_t)n_groups + 1, 0), b_seg((size_t)n_groups + 1, 0),
        b_panel((size_t)n_groups + 1, 0), b_lpanel((size_t)n_groups + 1, 0), b_utask((size_t)n_groups + 1, 0);
    for (int g = 0; g < n_groups; ++g) {
        const Part &x = part[g];
        b_light[g + 1] = b_light[g] + (long long)x.row_perm.size();
        b_heavy[g + 1] = b_heavy[g] + (long long)x.heavy_rows.size();
        b_seg[g + 1] = b_seg[g] + (long long)x.segs.size();
        b_panel[g + 1] = b_panel[g] + x.panel_len;
        b_lpanel[g + 1] = b_lpanel[g] + x.lpanel_len;
        b_utask[g + 1] = b_utask[g] + (long long)x.utask.size();
    }
    bp.panel_len = b_panel[n_groups];
    bp.lpanel_len = b_lpanel[n_groups];
    if (bp.panel_len > 0x7fffffffll || bp.lpanel_len > 0x7fffffffll) {
        a.rc = SPMM_B200_EINVAL;
        snprintf(a.err, sizeof(a.err), "panel too large");
        return;
    }
    bp.n_light = (int)b_light[n_groups];
    bp.n_heavy = (int)b_heavy[n_groups];
    bp.n_seg = (int)b_seg[n_groups];
    bp.n_utask = (int)b_utask[n_groups];
    bp.n_ltask = bp.n_utask - bp.n_seg;   // every segment is one task
    bp.split_task = (int)b_utask[(n_groups + 1) / 2];   // the groups' tasks are contiguous, in group order
    a.light.resize((size_t)bp.n_light);
    a.heavy_seg0.resize(bp.n_heavy ? (size_t)bp.n_heavy + 1 : 0);
    a.segs.resize((size_t)bp.n_seg);
    a.seg_hrow.resize((size_t)bp.n_seg);
    a.utask.resize((size_t)bp.n_utask);
    if (bp.n_heavy) a.heavy_seg0[(size_t)bp.n_heavy] = bp.n_seg;
#pragma omp parallel for schedule(dynamic, 1)
    for (int g = 0; g < n_groups; ++g) {
        const Part &x = part[g];
        const int lp = (int)b_lpanel[g], pn = (int)b_panel[g], sg = (int)b_seg[g], hv = (int)b_heavy[g];
        for (size_t i = 0; i < x.row_perm.size(); ++i) {
            const int r = x.row_perm[i];
            a.light[(size_t)b_light[g] + i] = make_int4(r, rb[r], re[r] - rb[r], lp + x.dst[i]);
        }
        for (size_t i = 0; i < x.heavy_rows.size(); ++i) {
            a.heavy_seg0[(size_t)hv + i] = sg + x.heavy_seg0[i];
            for (int sgm = x.heavy_seg0[i]; sgm < x.heavy_seg0[i + 1]; ++sgm) a.seg_hrow[(size_t)sg + sgm] = hv + (int)i;
        }
        for (size_t i = 0; i < x.segs.size(); ++i) {
            SegDesc d = x.segs[i];
            d.panel_off += pn;
            a.segs[(size_t)sg + i] = d;
        }
        for (size_t i = 0; i < x.utask.size(); ++i) {
            const int2 u = x.utask[i];
            a.utask[(size_t)b_utask[g] + i] = u.x < 0 ? make_int2(-1 - (sg + (-1 - u.x)), 0) : make_int2(lp + u.x, u.y);
        }
    }
}

// The scalar fallback (K % 4 != 0) keeps every row whole in one group and reads idx/val at run time: its plan of a block
// is the row order alone.
static void plan_block_scalar(const spmm_b200_handle *h, const int *rb, const int *re, int skip_empty, int reorder, BlockPlan &bp,
                              BlockArrays &a) {
    const Plan &p = h->plan;
    std::vector<int> row_perm, heavy_rows;
    a.rc = plan_rows_host(rb, re, h->num_v, p.seg_len, reorder, skip_empty, 2, row_perm, heavy_rows, a.heavy_seg0, a.segs, &bp.panel_len);
    if (a.rc) {
        snprintf(a.err, sizeof(a.err), "%s", spmm_b200_last_error());
        return;
    }
    bp.n_light = (int)row_perm.size();
    bp.n_heavy = (int)heavy_rows.size();
    bp.n_seg = (int)a.segs.size();
    a.light.resize(row_perm.size());
    for (size_t i = 0; i < row_perm.size(); ++i) {
        const int r = row_perm[i];
        a.light[i] = make_int4(r, rb[r], re[r] - rb[r], 0);
    }
}

template <class T>
static int upload_vec(T **dst, const std::vector<T> &v, cudaStream_t stream) {
    if (v.empty()) return 0;
    SB_CUDA(pool_alloc((void **)dst, sizeof(T) * v.size(), stream));
    SB_CUDA(cudaMemcpyAsync(*dst, v.data(), sizeof(T) * v.size(), cudaMemcpyHostToDevice, stream));
    return 0;
}

// Kernel shape (feature slices, lanes x vec per row slice, segment length, resident warps) and the number of column blocks
// to aim for. The vectorised kernels address B with 32-bit float4 offsets.
static int plan_shape(spmm_b200_handle *h, int b_rows, int &nb) {
    Plan &p = h->plan;
    const int M = h->num_v, K = h->feat;
    p.block = (int)h->opt_block;
    p.scalar = (K % 4) != 0;
    p.kslice = h->opt_kslice > 0 ? (int)h->opt_kslice : auto_kslice(M, K);
    if (p.scalar) p.kslice = K;
    if (p.kslice > 256) p.kslice = 256;
    if (p.kslice > ((K + 3) & ~3)) p.kslice = (K + 3) & ~3;
    p.n_slices = (K + p.kslice - 1) / p.kslice;
    if (!p.scalar) shape_for_kslice(p.kslice, &p.lanes, &p.vec);
    p.seg_len = h->opt_seg_len > 0 ? (int)h->opt_seg_len : auto_seg_len(h->num_e, p.lanes);
    p.tune = (int)h->opt_tune;
    p.light_steps = h->opt_light_steps > 0 ? (int)h->opt_light_steps : 0;
    p.slots = p.scalar ? 0 : resident_warps(p.lanes, p.vec, p.tune, p.block);
    if (p.scalar) p.seg_len = 0x7fffffff;   // scalar fallback keeps every row whole
    if (!p.scalar && (long long)b_rows * (K / 4) > 0x7fffffffll) {
        set_error("B is too large for 32-bit row offsets: b_rows * feat_in / 4 = %lld >= 2^31", (long long)b_rows * (K / 4));
        return SPMM_B200_EINVAL;
    }
    nb = h->opt_col_blocks > 0 ? (int)h->opt_col_blocks : auto_col_blocks(b_rows, K, h->num_e, M);
    if (p.scalar || nb < 1) nb = 1;
    if (nb > kMaxBands && h->opt_col_blocks <= 0) nb = kMaxBands;
    if (nb > b_rows) nb = b_rows > 0 ? b_rows : 1;
    return 0;
}

// Band bounds: band b is B rows [bounds[b], bounds[b + 1]). Default: nb equal bands of ceil(b_rows / nb) rows. Option
// "host_bands" (the plan is meant for the host-buffer call, spmm_b200_run_host): the LAST band takes the last 40 % of B's
// rows and the bands before it share the rest. The last pass stores final rows over PCIe and is bound by that transfer
// whatever it computes, so it may as well carry half of the nonzeros (from a band that no longer fits the L2), while the
// small early bands let the first pass start sooner and finish the rest of the work under the upload of B.
static std::vector<int> band_bounds(int b_rows, int nb, long long host_bands) {
    std::vector<int> bounds;
    if (host_bands && nb >= 3) {
        // host_bands = 1: the last band is 40 % of B's rows (measured best on the reddit shape: e2e 10.31 -> 9.34 ms;
        // 30 %: 9.76, 50 %: 9.60, 60 %: 9.98 — profiles/r02_host_bands.jsonl); 10..90: that percentage
        const long long pct = host_bands >= 10 ? host_bands : 40;
        const int small = nb - 1, half = (int)((long long)b_rows * (100 - pct) / 100);
        const int per = (half + small - 1) / small;
        for (int b = 0; b < small && b * per < half; ++b) bounds.push_back(b * per);
        bounds.push_back(half);
        bounds.push_back(b_rows);
        return bounds;
    }
    const int cols_per_block = nb > 1 ? (b_rows + nb - 1) / nb : b_rows;
    if (nb > 1) nb = (b_rows + cols_per_block - 1) / cols_per_block;   // every band starts inside B (b_rows = 10, 7 bands -> 5 of 2 rows)
    for (int b = 0; b < nb; ++b) bounds.push_back(b * cols_per_block);
    bounds.push_back(b_rows);
    return bounds;
}

// CSR read and checks: ptr comes to the host and must hold num_e nonzeros in rows of non-negative degree (whatever the row
// order, a negative degree would turn into out-of-bounds panel slots). Behind the copy, one pass over idx sets flags[0]
// when a column is outside B; split_at_bands reads the flags back.
static int read_csr(const spmm_b200_handle *h, int b_rows, int *d_flags, std::vector<int> &ptr, cudaStream_t stream, PrepTrace &tr) {
    const int M = h->num_v;
    ptr.assign((size_t)M + 1, 0);
    SB_CUDA(cudaMemcpyAsync(ptr.data(), h->d_ptr, sizeof(int) * ((size_t)M + 1), cudaMemcpyDeviceToHost, stream));
    SB_CUDA(cudaMemsetAsync(d_flags, 0, 2 * sizeof(int), stream));
    const int rc = launch_check_cols(h->d_idx, h->num_e, b_rows, d_flags, stream);
    if (rc) return rc;
    SB_CUDA(cudaStreamSynchronize(stream));
    if (ptr[0] != 0 || ptr[M] != h->num_e) {
        set_error("CSR ptr is inconsistent: ptr[0]=%d ptr[num_v]=%d num_e=%d", ptr[0], ptr[M], h->num_e);
        return SPMM_B200_EINVAL;
    }
    for (int r = 0; r < M; ++r)
        if (ptr[r + 1] < ptr[r]) {
            set_error("CSR ptr decreases at row %d", r);
            return SPMM_B200_EINVAL;
        }
    tr.lap("ptr D2H + check_cols");
    return 0;
}

// Row split: with several bands every row is cut at the band bounds on the device (split[b][r]: where band b starts in
// row r) and the split comes to the host. That needs ascending columns inside a row: an unsorted CSR keeps one block.
static int split_at_bands(spmm_b200_handle *h, int b_rows, int *d_flags, std::vector<int> &band_begin, std::vector<int> &split,
                          cudaStream_t stream) {
    Plan &p = h->plan;
    const int M = h->num_v, nb = (int)band_begin.size() - 1;
    if (nb > 1) {
        SB_CUDA(pool_alloc((void **)&p.d_split, sizeof(int) * (size_t)(nb + 1) * M, stream));
        const int rc = launch_split_rows(h->d_ptr, h->d_idx, M, nb, band_begin.data(), p.d_split, d_flags + 1, stream);
        if (rc) return rc;
        split.resize((size_t)(nb + 1) * M);
        SB_CUDA(cudaMemcpyAsync(split.data(), p.d_split, sizeof(int) * split.size(), cudaMemcpyDeviceToHost, stream));
    }
    int flags[2] = {0, 0};
    SB_CUDA(cudaMemcpyAsync(flags, d_flags, sizeof(flags), cudaMemcpyDeviceToHost, stream));
    SB_CUDA(cudaStreamSynchronize(stream));
    if (flags[0]) {
        set_error("CSR idx holds a column outside [0, %d)", b_rows);
        return SPMM_B200_EINVAL;
    }
    if (nb > 1 && flags[1]) {
        pool_free(p.d_split, stream);
        p.d_split = nullptr;
        split.clear();
        band_begin = {0, b_rows};
    }
    return 0;
}

// Row order, one for every block. Degree buckets (longest rows first) shorten the tail of every launch and keep the lanes
// of a task balanced; natural order keeps neighbouring rows together, which lets a graph's locality hit in L2. Auto (option
// reorder = -1): natural order only when locality is what is at stake: ONE block (no column blocks — B is either small or
// far larger than the L2) in a launch of at least 8 waves of tasks with a full warp per row: measured 12.2 -> 11.3 ms on the
// products shape and the opposite (0.14 -> 0.19 ms) on the one-wave arxiv shape (profiles/r01_sweep.md). With column blocks
// every pass gathers from an L2-resident band whatever the order, and buckets win at every partition size of the reddit
// shape (6.04 vs 6.14 ms whole, 0.80 vs 0.92 ms for a 1/8 block: profiles/r02_notes.md).
// Row groups: contiguous row ranges balanced by nonzeros (the partition rule, spmm_b200_partition_rows), planned
// independently (in parallel) and never spanned by a task. Natural order: 16. Degree buckets with several blocks: 2 — the
// halves that go out on two streams. Otherwise 1.
static int order_rows(spmm_b200_handle *h, const std::vector<int> &ptr, int nb, int &reorder) {
    Plan &p = h->plan;
    const int M = h->num_v;
    const long long entries = (long long)h->num_e + M;   // the light stream of a single block: every nonzero, a header per row
    const bool natural = h->opt_reorder >= 0 ? h->opt_reorder == 0 : nb == 1 && p.lanes == 32 && p.slots > 0 && entries >= 8ll * p.slots * 64;
    reorder = !natural;
    long long g = h->opt_row_groups > 0 ? h->opt_row_groups : (natural ? 16 : (nb > 1 ? 2 : 1));
    if (p.scalar) g = 1;
    if (g > kMaxRowGroups) g = kMaxRowGroups;
    if (g > M) g = M;
    p.n_groups = (int)g;
    p.group_row.resize((size_t)p.n_groups + 1);
    return spmm_b200_partition_rows(ptr.data(), M, p.n_groups, p.group_row.data());
}

// Host planning of every block, independent of each other: row order, segments, light-stream packing, task order. Block b
// gathers from B rows [band_begin[b], band_begin[b + 1]) and owns CSR positions [split[b][r], split[b+1][r]) of row r.
static int plan_blocks_host(spmm_b200_handle *h, const std::vector<int> &ptr, const std::vector<int> &split,
                            const std::vector<int> &band_begin, int reorder, std::vector<BlockArrays> &arr) {
    Plan &p = h->plan;
    const int nb = p.n_col_blocks, M = h->num_v;
    // (several blocks: one host thread per block; a single block: its row groups in parallel — nested regions stay serial)
#pragma omp parallel for schedule(dynamic, 1) if (nb > 1)
    for (int b = 0; b < nb; ++b) {
        const int *rb = nb > 1 ? split.data() + (size_t)b * M : ptr.data();
        const int *re = nb > 1 ? split.data() + (size_t)(b + 1) * M : ptr.data() + 1;
        // passes after the first skip rows without nonzeros in their band — except the last pass, which lists every
        // row: it is the one that delivers final rows (to C, to the stacked-layer targets, to run_host's host buffer)
        const bool skip_empty = b > 0 && b + 1 != nb;
        p.blocks[b].col_begin = band_begin[b];
        p.blocks[b].col_end = band_begin[b + 1];
        p.blocks[b].reorder = reorder;
        if (p.scalar) plan_block_scalar(h, rb, re, skip_empty, reorder, p.blocks[b], arr[b]);
        else plan_block_groups(h, rb, re, skip_empty, reorder, p.group_row.data(), p.n_groups, p.blocks[b], arr[b]);
    }
    for (const BlockArrays &a : arr)
        if (a.rc) {
            set_error("%s", a.err);
            return a.rc;
        }
    if (h->opt_light_steps <= 0) p.light_steps = p.blocks[0].light_steps;   // reported by plan_info (block 0)
    return 0;
}

// Device upload: one pool allocation per array kind that kernels write (lpanel, panel, part, seg_count), block after block,
// then the arrays that kernels read, block by block (the host vectors must outlive the synchronisation of `stream`).
static int upload_plan(Plan &p, int K, const std::vector<BlockArrays> &arr, cudaStream_t stream, PrepTrace &tr) {
    long long lp_total = 0, pn_total = 0, seg_total = 0, heavy_total = 0, task_total = 0;
    for (const BlockPlan &bp : p.blocks) {
        lp_total += bp.lpanel_len;
        pn_total += bp.panel_len;
        seg_total += bp.n_seg;
        heavy_total += bp.n_heavy;
        task_total += bp.n_utask;
    }
    if (lp_total > 0x7fffffffll || pn_total > 0x7fffffffll || task_total * p.n_slices > 0x7fffffffll) {
        set_error("plan too large for 32-bit panel offsets (%lld light, %lld heavy entries)", lp_total, pn_total);
        return SPMM_B200_EINVAL;
    }
    if (lp_total) {
        SB_CUDA(pool_alloc((void **)&p.d_lpanel_all, sizeof(int2) * (size_t)lp_total, stream));
        SB_CUDA(cudaMemsetAsync(p.d_lpanel_all, 0xFF, sizeof(int2) * (size_t)lp_total, stream));   // nop entries
    }
    if (pn_total) SB_CUDA(pool_alloc((void **)&p.d_panel_all, sizeof(int2) * (size_t)pn_total, stream));
    if (seg_total) SB_CUDA(pool_alloc((void **)&p.d_part_all, sizeof(float) * (size_t)seg_total * K, stream));
    if (heavy_total) {
        // n_heavy x n_slices counters per band
        const size_t slots = (size_t)heavy_total * p.n_slices;
        SB_CUDA(pool_alloc((void **)&p.d_seg_count_all, sizeof(int) * slots, stream));
        SB_CUDA(cudaMemsetAsync(p.d_seg_count_all, 0, sizeof(int) * slots, stream));
    }
    tr.lap("arena allocation");
    long long lp_off = 0, pn_off = 0, seg_off = 0, heavy_off = 0;
    for (size_t b = 0; b < arr.size(); ++b) {
        BlockPlan &bp = p.blocks[b];
        int rc;
        if ((rc = upload_vec(&bp.d_light_desc, arr[b].light, stream)) || (rc = upload_vec(&bp.d_utask, arr[b].utask, stream)) ||
            (rc = upload_vec(&bp.d_seg_hrow, arr[b].seg_hrow, stream)) || (rc = upload_vec(&bp.d_heavy_seg0, arr[b].heavy_seg0, stream)) ||
            (rc = upload_vec(&bp.d_seg_desc, arr[b].segs, stream)))
            return rc;
        bp.d_lpanel = p.d_lpanel_all + lp_off;   // a block's empty slices are never read
        bp.d_panel = p.d_panel_all + pn_off;
        bp.d_part = p.d_part_all + seg_off * K;
        bp.d_seg_count = p.d_seg_count_all + heavy_off * p.n_slices;
        lp_off += bp.lpanel_len;
        pn_off += bp.panel_len;
        seg_off += bp.n_seg;
        heavy_off += bp.n_heavy;
    }
    return 0;
}

int build_plan(spmm_b200_handle *h, cudaStream_t stream) {
    Plan &p = h->plan;
    PrepTrace tr;
    free_plan(p);
    tr.lap("free the previous plan");
    h->plan_select = 0;
    p.live = h->opt_live_values != 0;
    const int M = h->num_v, K = h->feat;
    const int b_rows = h->b_rows > 0 ? h->b_rows : M;
    if (K == 0 || M == 0) {
        // nothing to compute (launch_spmm returns before touching the plan): an empty, ready plan of one empty block
        p.block = (int)h->opt_block;
        p.n_col_blocks = 1;
        p.blocks.resize(1);
        p.group_row = {0, M};
        p.ready = true;
        return 0;
    }
    SB_CUDA(cudaGetDevice(&p.device));   // the plan's arrays come from this device's pool (pool.cu)
    int nb = 1, rc;
    if ((rc = plan_shape(h, b_rows, nb))) return rc;
    std::vector<int> band_begin = band_bounds(b_rows, nb, h->opt_host_bands), ptr, split;

    int *d_flags = nullptr;   // [0] a column outside B, [1] a row whose columns are not ascending
    SB_CUDA(pool_alloc((void **)&d_flags, 2 * sizeof(int), stream));
    if (!(rc = read_csr(h, b_rows, d_flags, ptr, stream, tr))) rc = split_at_bands(h, b_rows, d_flags, band_begin, split, stream);
    pool_free(d_flags, stream);
    if (rc) return rc;
    tr.lap("split_rows + D2H");

    nb = (int)band_begin.size() - 1;
    p.n_col_blocks = nb;
    p.blocks.resize(nb);
    std::vector<BlockArrays> arr((size_t)nb);
    int reorder = 1;
    if ((rc = order_rows(h, ptr, nb, reorder)) || (rc = plan_blocks_host(h, ptr, split, band_begin, reorder, arr))) return rc;
    tr.lap("host planning (all blocks)");

    if ((rc = upload_plan(p, K, arr, stream, tr)) || (rc = refresh_panels(h, stream))) return rc;
    tr.lap("uploads + panel kernels queued");

    // Two-stream launches (option "split_streams": -1 auto = whenever there are several blocks).
    p.split_streams = !p.scalar && p.n_groups > 1 && (h->opt_split_streams == 1 || (h->opt_split_streams < 0 && nb > 1));
    if (p.split_streams && !h->aux_stream) {   // created here, not in run: run may be under CUDA-graph capture
        SB_CUDA(cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking));
        SB_CUDA(cudaEventCreateWithFlags(&h->aux_fork, cudaEventDisableTiming));
        SB_CUDA(cudaEventCreateWithFlags(&h->aux_join, cudaEventDisableTiming));
    }

    SB_CUDA(cudaStreamSynchronize(stream));   // host vectors go out of scope
    tr.lap("final sync");
    p.ready = true;
    return 0;
}

// Stage the {col, val} panels from the caller's idx/val (asynchronous on `stream`): at preprocess, and at refresh_values, as
// the plan's structure (row order, segments, tasks, slots) depends on ptr only: new edge values need no new plan. A live plan
// stages {col, position} instead — the position in the value source's CSR (t_perm on a derived handle) — and reads no val.
int refresh_panels(spmm_b200_handle *h, cudaStream_t stream) {
    Plan &p = h->plan;
    if (p.scalar || h->feat == 0 || h->num_v == 0) return 0;   // the scalar kernel reads idx/val at run time
    const int groups = 32 / p.lanes, pad = 4 * groups, k4 = h->feat / 4;
    const int *perm = p.live && h->t_src ? h->t_perm : nullptr;
    for (BlockPlan &bp : p.blocks) {
        int rc;
        if (bp.n_ltask > 0 &&
            (rc = launch_build_lpanel(bp.d_light_desc, bp.n_light, groups, k4, h->d_idx, h->d_val, perm, p.live, bp.d_lpanel, stream)))
            return rc;
        if (bp.n_seg > 0 &&
            (rc = launch_build_panel(bp.d_seg_desc, bp.n_seg, k4, pad, h->d_idx, h->d_val, perm, p.live, bp.d_panel, stream)))
            return rc;
    }
    return 0;
}

}  // namespace spmm_b200

extern "C" int spmm_b200_plan_row_cost(int num_v, long long nnz, int b_rows, int feat_in) {
    if (num_v <= 0 || feat_in <= 0) return 1;
    return spmm_b200::auto_col_blocks(b_rows > 0 ? b_rows : num_v, feat_in, nnz, num_v);
}

// Host-only plan for CPU-side callers and tests (declared in include/spmm_b200.h).
extern "C" int spmm_b200_plan_host(const int *h_ptr, int num_v, int feat_in, long long seg_len, int reorder, int *row_perm,
                                   int *n_light, int *heavy_rows, int *n_heavy, int *heavy_seg0, int *seg_desc,
                                   int *n_seg, long long *panel_len) {
    using namespace spmm_b200;
    if (!h_ptr || num_v < 0 || !n_light || !n_heavy || !n_seg || !panel_len) {
        set_error("spmm_b200_plan_host: bad arguments");
        return SPMM_B200_EINVAL;
    }
    int lanes = 32, vec = 1;
    if (feat_in > 0 && feat_in % 4 == 0) shape_for_kslice(auto_kslice(num_v, feat_in), &lanes, &vec);
    if (seg_len <= 0) seg_len = (feat_in % 4 != 0) ? 0x7fffffffll : auto_seg_len(h_ptr[num_v], lanes);
    const int pad = (feat_in % 4 != 0) ? 2 : 4 * (32 / lanes);
    if (seg_len > 0x7fffffffll) seg_len = 0x7fffffffll;
    std::vector<int> rp, hr, hs;
    std::vector<SegDesc> segs;
    int rc = plan_rows_host(h_ptr, h_ptr + 1, num_v, (int)seg_len, reorder, 0, pad, rp, hr, hs, segs, panel_len);
    if (rc) return rc;
    *n_light = (int)rp.size();
    *n_heavy = (int)hr.size();
    *n_seg = (int)segs.size();
    if (row_perm) std::copy(rp.begin(), rp.end(), row_perm);
    if (heavy_rows) std::copy(hr.begin(), hr.end(), heavy_rows);
    if (heavy_seg0) std::copy(hs.begin(), hs.end(), heavy_seg0);
    if (seg_desc && !segs.empty()) memcpy(seg_desc, segs.data(), sizeof(SegDesc) * segs.size());
    return 0;
}

// Host-only light-stream packing (declared in include/spmm_b200.h).
extern "C" int spmm_b200_pack_light_host(const int *cost, int n, int groups, int steps, int *dst, int *ltask,
                                         int *n_ltask, long long *lpanel_len) {
    using namespace spmm_b200;
    if (n < 0 || groups < 1 || groups > 32 || (groups & (groups - 1)) || steps < 1 || !n_ltask || !lpanel_len ||
        (n > 0 && !cost)) {
        set_error("spmm_b200_pack_light_host: bad arguments");
        return SPMM_B200_EINVAL;
    }
    std::vector<int> d((size_t)n);
    std::vector<int2> tasks;
    *lpanel_len = pack_light_host(cost, n, groups, steps, d.data(), tasks);
    *n_ltask = (int)tasks.size();
    if (dst) std::copy(d.begin(), d.end(), dst);
    if (ltask && !tasks.empty()) memcpy(ltask, tasks.data(), sizeof(int2) * tasks.size());
    return 0;
}
