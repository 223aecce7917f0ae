"""De-risking probe: two-stream launches with BUCKETED row order — emulated with two handles over the two row halves of a
rank's block (each plans its own rows), run on two streams. Compared with one handle (bucketed per band, one stream)."""
import json, sys
import numpy as np, torch
sys.path.insert(0, ".")
import hpc_b200 as H

shape, K = "reddit", 256
ptr, idx = H.gen_named_graph(shape)
M, nnz = len(ptr) - 1, len(idx)
val = H.fill_normal(torch.empty(nnz, device="cuda"), 123, 1)
vin = H.fill_normal(torch.empty(M * K, device="cuda"), 123, 2)
d_idx = torch.from_numpy(idx).cuda()

def make(r0, r1, **opts):
    lptr = H.rebase_ptr(ptr, r0, r1)
    e0, e1 = int(ptr[r0]), int(ptr[r1])
    g = H.CSR(r1 - r0, e1 - e0, torch.from_numpy(lptr).cuda(), d_idx[e0:e1].clone(), val[e0:e1].clone())
    out = torch.empty((r1 - r0) * K, device="cuda")
    op = H.SpMMB200(g, K, b_rows=M, **opts)
    op.preprocess(vin, out)
    return op, out, g

for parts in (8, 4, 2, 1):
    bounds = H.partition_rows(ptr, parts)
    r0, r1 = int(bounds[0]), int(bounds[1])
    mid = int(H.partition_rows(H.rebase_ptr(ptr, r0, r1), 2)[1]) + r0
    res = {}
    for name, reorder in (("bucketed", 1), ("natural", 0), ("auto", -1)):
        one, out1, _g = make(r0, r1, split_streams=0, reorder=reorder)
        a_op, a_out, _ga = make(r0, mid, split_streams=0, reorder=reorder)
        b_op, b_out, _gb = make(mid, r1, split_streams=0, reorder=reorder)
        s1 = torch.cuda.Stream()
        def run_two():
            s1.wait_stream(torch.cuda.current_stream())
            # interleave the passes by issuing both runs; stream order keeps each half's chain
            a_op.run(vin, a_out)
            with torch.cuda.stream(s1):
                b_op.run(vin, b_out)
            torch.cuda.current_stream().wait_stream(s1)
        def timeit(fn):
            for _ in range(5): fn()
            ts = []
            for rep in range(3):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(); e0.record()
                for _ in range(20): fn()
                e1.record(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1) / 20)
            return round(float(np.mean(ts)), 4)
        t_one = timeit(lambda: one.run(vin, out1))
        t_two = timeit(run_two)
        torch.cuda.synchronize()
        eq = bool(torch.equal(torch.cat([a_out, b_out]), out1))
        res[name] = {"one_handle": t_one, "two_halves_two_streams": t_two, "ratio": round(t_two / t_one, 4), "bit_equal": eq}
        for o in (one, a_op, b_op): o.close()
    print(json.dumps({"parts": parts, **res}), flush=True)
