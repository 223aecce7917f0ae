"""numpy restatement of the engine's preprocessing plan — TEST INFRASTRUCTURE ONLY.

The reference has no degree sort or panels; its only preprocessing is the student's fixed
256-nnz task split (PA4/workspace/src/spmm_opt.cu:43-54), which `student_split_check` below
uses as a cross-check for the segment cutter. Parity with the reference is therefore UNPINNED
for the plan by construction (SURVEY.md §8c); this file pins the product against an
independently written restatement of the plan's published definition:

  deg(r) = ptr[r+1]-ptr[r];  heavy(r) = deg(r) > seg_len;  bucket(r) = bit_length(deg(r))
  order  = rows by (bucket descending, row ascending), or natural order when reorder = 0
  row_perm = non-heavy rows in order; heavy rows in order are cut into
  nseg = ceil(deg/seg_len) segments [begin + j*deg//nseg, begin + (j+1)*deg//nseg);
  panel = segments' (col, val-bits) pairs back to back, each padded with nops to a multiple of 4 * (32 / lanes) entries.
  lpanel / ltask = the rows of row_perm as a stream of header + entries, packed into equal-sized tasks
  (pack_light); split / column blocks = rows cut at the boundaries of nb bands of B rows (split_rows),
  one plan per band.
"""
from __future__ import annotations

import numpy as np


def lanes_for(feat: int) -> int:
    """lanes cooperating on one row for the automatic slice width (32 when feat % 4 != 0)."""
    if feat % 4:
        return 32
    q = (auto_kslice(0, feat) + 3) // 4
    l = 1
    while l < q and l < 32:
        l <<= 1
    return l


def auto_seg_len(nnz: int, feat: int) -> int:
    if feat % 4:
        return 0x7FFFFFFF
    if lanes_for(feat) >= 32:
        return 256
    t = nnz // 65536
    l = 128
    while l < t and l < 1024:
        l <<= 1
    return l


def auto_kslice(num_v: int, feat: int) -> int:
    if feat % 4:
        return feat
    return (feat + 3) & ~3 if feat < 256 else 256


def bit_length(deg: np.ndarray) -> np.ndarray:
    out = np.zeros(deg.shape, np.int64)
    d = deg.astype(np.int64).copy()
    while np.any(d > 0):
        out += d > 0
        d >>= 1
    return out


def auto_col_blocks(b_rows: int, feat: int, nnz: int, num_v: int) -> int:
    """Passes over A, one per band of B rows: 1 unless B exceeds 96 MB; then ceil(B bytes / 48 MB),
    accepted when <= 16 and a row still averages >= 64 nonzeros per block."""
    b_bytes = b_rows * feat * 4
    if feat % 4 or num_v <= 0 or b_bytes <= (96 << 20):
        return 1
    nb = -(-b_bytes // (48 << 20))
    if nb > 16 or nnz // num_v // nb < 64:
        return 1
    return nb


def host_band_bounds(nb: int, b_rows: int, pct: int = 40):
    """Option host_bands: the last band is the last pct % of B's rows, the nb - 1 bands before it share the rest."""
    small, half = nb - 1, b_rows * (100 - pct) // 100
    per = -(-half // small)
    return [b * per for b in range(small) if b * per < half] + [half, b_rows]


def split_rows(ptr, idx, nb: int, b_rows: int, bounds=None) -> np.ndarray:
    """split[b, r] = first CSR position of row r whose column is >= the first B row of band b — b * ceil(b_rows / nb),
    or bounds[b] — (split[0] = ptr[r], split[nb] = ptr[r+1]); columns must ascend inside a row."""
    ptr = np.asarray(ptr, np.int64)
    idx = np.asarray(idx, np.int64)
    m = len(ptr) - 1
    cpb = -(-b_rows // nb)
    if bounds is None:
        bounds = [b * cpb for b in range(nb)]
    # rank of (row, column) pairs in the row-major, column-ascending order the CSR already has
    row_of = np.repeat(np.arange(m, dtype=np.int64), np.diff(ptr))
    keys = row_of * (b_rows + 1) + idx
    out = np.empty((nb + 1, m), np.int64)
    out[0], out[nb] = ptr[:-1], ptr[1:]
    for b in range(1, nb):
        out[b] = np.searchsorted(keys, np.arange(m, dtype=np.int64) * (b_rows + 1) + bounds[b], side="left")
    return out.astype(np.int32)


def row_groups_of(m: int, group_row) -> np.ndarray:
    """Row group of every row: group g owns rows [group_row[g], group_row[g+1]); one group when group_row is None."""
    if group_row is None:
        return np.zeros(m, np.int64)
    return np.searchsorted(np.asarray(group_row, np.int64), np.arange(m, dtype=np.int64), side="right") - 1


def plan(ptr, idx, val, seg_len: int, reorder: bool = True, rb=None, re=None, skip_empty: bool = False, k4: int = 1,
         pad: int = 2, group_row=None) -> dict:
    """Plan of the whole matrix (rb/re omitted) or of one column block (row r owns [rb[r], re[r])).
    k4 = feat // 4: panels store a column as the B row's offset in float4 units (col * k4).
    pad = 4 * (32 // lanes): every segment's span is padded with nop entries (-1, 0) to a multiple of it.
    group_row: row-group bounds; the row order (degree buckets or natural) applies inside each group, groups in order."""
    ptr = np.asarray(ptr, np.int64)
    m = len(ptr) - 1
    rb = ptr[:-1] if rb is None else np.asarray(rb, np.int64)
    re = ptr[1:] if re is None else np.asarray(re, np.int64)
    deg = re - rb
    if reorder:
        # by (row group, degree bucket descending, row): lexsort's last key is the primary one
        order = np.lexsort((np.arange(m), -bit_length(deg), row_groups_of(m, group_row)))
    else:
        order = np.arange(m)
    if skip_empty:
        order = order[deg[order] > 0]
    heavy_mask = deg[order] > seg_len
    row_perm = order[~heavy_mask].astype(np.int32)
    heavy_rows = order[heavy_mask].astype(np.int32)
    seg_desc, heavy_seg0, panel = [], [0], []
    off = 0
    for r in heavy_rows:
        d, begin = int(deg[r]), int(rb[r])
        nseg = -(-d // seg_len)
        for j in range(nseg):
            b = begin + j * d // nseg
            e = begin + (j + 1) * d // nseg
            seg_desc.append((int(r), off, e - b, b))
            cols = (np.asarray(idx[b:e], np.int64) * k4).astype(np.int32)
            bits = np.asarray(val[b:e], np.float32).view(np.int32)
            pairs = np.stack([cols, bits], axis=1)
            extra = -(e - b) % pad
            if extra:
                pairs = np.concatenate([pairs, np.tile(np.asarray([[-1, 0]], np.int32), (extra, 1))])
            panel.append(pairs)
            off += len(pairs)
        heavy_seg0.append(len(seg_desc))
    light_desc = np.stack([row_perm.astype(np.int64), rb[row_perm], deg[row_perm], np.zeros(len(row_perm), np.int64)],
                          axis=1).astype(np.int32).reshape(-1, 4)
    seg_hrow = np.repeat(np.arange(len(heavy_rows)), np.diff(heavy_seg0)).astype(np.int32) if len(heavy_rows) else np.zeros(0, np.int32)
    return {
        "light_desc": light_desc,
        "seg_hrow": seg_hrow,
        "row_perm": row_perm,
        "heavy_rows": heavy_rows,
        "heavy_seg0": np.asarray(heavy_seg0 if len(heavy_rows) else [], np.int32),
        "seg_desc": np.asarray(seg_desc, np.int32).reshape(-1, 4),
        "panel": np.concatenate(panel) if panel else np.zeros((0, 2), np.int32),
    }


def auto_light_steps(groups: int, total_cost: int, slots: int, heavy_tasks: int) -> int:
    """Default max(16, 64 // groups); graphs of fewer than 4 waves of such tasks get a size that fills a whole
    number of waves of the `slots` resident warps (less the heavy segments running beside them)."""
    dflt = max(16, 64 // groups)
    if slots <= 0 or total_cost <= 0:
        return dflt
    if groups == 1 and total_cost >= 64 * slots * 64:
        return 128
    avail = slots - heavy_tasks % slots
    if avail < slots // 2:
        avail = slots
    per_wave = avail * groups * dflt
    if total_cost >= 4 * per_wave:
        return dflt
    waves = -(-total_cost // per_wave)
    st = -(-total_cost // (waves * avail * groups))
    st += st // 16 + 1
    return min(max(st, 16), dflt)


def auto_reorder(lanes: int, total_cost: int, slots: int) -> bool:
    """Natural order (False) when a full warp serves each row and the block is >= 8 waves of 64-entry tasks."""
    return not (lanes == 32 and slots > 0 and total_cost >= 8 * slots * 64)


def pack_light(cost, groups: int, steps: int, cuts=()):
    """Light-stream packing. cost[i] = nonzeros + 1 of the i-th light row in plan order. A row goes to the
    least-filled lane of the current task (lowest index on ties); when that lane is non-empty and would exceed
    `steps`, the task is closed first. `cuts`: row positions before which an open task is closed (row-group
    boundaries: the groups are packed one by one). -> (dst slots, tasks [(offset, steps)], panel length)"""
    dst, tasks = [], []
    fill = [0] * groups
    off = 0
    cuts = set(int(c) for c in cuts)

    def close():
        nonlocal off, fill
        mx = (max(fill) + 3) // 4 * 4
        tasks.append((off, mx))
        off += mx * groups
        fill = [0] * groups

    for i, c in enumerate(int(x) for x in cost):
        if i in cuts and any(fill):
            close()
        g = fill.index(min(fill))
        if fill[g] > 0 and fill[g] + c > steps:
            close()
            g = 0
        dst.append(off + fill[g] * groups + g)
        fill[g] += c
    if any(fill):
        close()
    return np.asarray(dst, np.int32), np.asarray(tasks, np.int32).reshape(-1, 2), off


def light_stream(plan_dict, idx, val, groups: int, steps: int, k4: int = 1, group_row=None) -> dict:
    """light_desc with header slots, task list and the stream panel for a plan() result. group_row: the row-group
    bounds: no task spans a bound."""
    ld = plan_dict["light_desc"].copy()
    grp = row_groups_of(int(ld[:, 0].max()) + 1 if len(ld) else 0, group_row)[ld[:, 0]] if len(ld) else np.zeros(0, np.int64)
    cuts = [i for i in range(1, len(ld)) if grp[i] != grp[i - 1]]     # the light rows are group-major in either order
    dst, tasks, length = pack_light(ld[:, 2].astype(np.int64) + 1, groups, steps, cuts)
    ld[:, 3] = dst
    panel = np.full((length, 2), -1, np.int32)
    idx = np.asarray(idx, np.int32)
    bits = np.asarray(val, np.float32).view(np.int32)
    for row, begin, deg, d in ld:
        panel[d] = (np.uint32(0x80000000 | int(row)).astype(np.int32), 0)   # header
        if deg:
            sl = d + (1 + np.arange(deg)) * groups
            panel[sl, 0] = idx[begin:begin + deg].astype(np.int64) * k4
            panel[sl, 1] = bits[begin:begin + deg]
    return {"light_desc": ld, "ltask": tasks, "lpanel": panel}


def unified_tasks(plan_dict, stream_dict, reorder: bool, group_row=None) -> np.ndarray:
    """Scheduling order of the warp tasks of one slice: (lpanel offset, steps) for a light task, (-1 - segment, 0) for
    a heavy segment. Bucketed rows: per row group, all its segments, then its light tasks. Natural order: merged by
    first row (a light task's first row is the row whose header sits at its offset)."""
    ltask = stream_dict["ltask"]
    nseg = len(plan_dict["seg_desc"])
    heavy = [(-1 - s, 0) for s in range(nseg)]
    light = [tuple(int(x) for x in t) for t in ltask]
    ld = stream_dict["light_desc"]
    first_row = {int(d): int(r) for r, _, _, d in ld}          # header slot -> row
    if reorder:
        gr = np.asarray([0, 1 << 62] if group_row is None else group_row, np.int64)
        grp_of = lambda row: int(np.searchsorted(gr, row, side="right")) - 1
        keyed = [(grp_of(int(plan_dict["seg_desc"][s][0])), 0, s, heavy[s]) for s in range(nseg)] + \
                [(grp_of(first_row[t[0]]), 1, i, t) for i, t in enumerate(light)]
        keyed.sort(key=lambda k: k[:3])
        return np.asarray([k[3] for k in keyed], np.int32).reshape(-1, 2)
    keyed = [(first_row[t[0]], 1, t) for t in light] + [(int(plan_dict["seg_desc"][s][0]), 0, heavy[s]) for s in range(nseg)]
    keyed.sort(key=lambda k: (k[0], k[1]))                     # stable: a row's segments stay in order
    return np.asarray([k[2] for k in keyed], np.int32).reshape(-1, 2)


def task_groups(utask, light_desc, seg_desc, group_row) -> np.ndarray:
    """Row group of every task of one block's utask: that of the row the task starts with (a light task's first row is
    the row whose header sits at its offset)."""
    first_row = {int(d): int(r) for r, _, _, d in light_desc}
    rows = [int(seg_desc[-1 - x][0]) if x < 0 else first_row[int(x)] for x, _ in utask]
    return np.searchsorted(np.asarray(group_row, np.int64), np.asarray(rows, np.int64), side="right") - 1


def student_split_check(ptr, tasks) -> bool:
    """With seg_len = 256 a row of deg d yields ceil(d/256) pieces in both schemes
    (spmm_opt.cu:46 steps by kBatchSize; the plan balances the same number of pieces)."""
    ptr = np.asarray(ptr, np.int64)
    deg = np.diff(ptr)
    per_row = np.bincount(tasks[:, 0], minlength=len(deg))
    return bool(np.array_equal(per_row, -(-deg // 256)))


def partition_rows(ptr, parts: int, row_cost: int = 0) -> np.ndarray:
    """bounds[g] = first row r with ptr[r] + row_cost*r >= g*(nnz + row_cost*m)//parts (SURVEY.md §8e; row_cost = 0:
    balanced by nonzeros alone)."""
    ptr = np.asarray(ptr, np.int64)
    m = len(ptr) - 1
    ptr = ptr + row_cost * np.arange(m + 1, dtype=np.int64)
    nnz = int(ptr[m])
    b = [0]
    for g in range(1, parts):
        r = int(np.searchsorted(ptr, g * nnz // parts, side="left"))
        b.append(max(min(r, m), b[-1]))
    b.append(m)
    return np.asarray(b, np.int32)
