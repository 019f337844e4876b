import importlib, os, sys, time, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pkg = importlib.import_module("k8s-dra-driver_b200")
R=pkg.records
w = pkg.synth.cfg2()
for graph in (0, pkg.api.CFG_USE_GRAPH):
    ctx = pkg.api.Context(device=0, flags=graph)
    ctx.set_table(w.table); ctx.set_inventory(w.gpus, w.node_off)
    pc = pkg.api.PinnedBuffer(w.n_claim, R.CLAIM_DTYPE); pc.array[:] = w.claims
    po = pkg.api.PinnedBuffer(w.n_out, R.OUT_DTYPE)
    F = pkg.api.F_FRESH_INVENTORY
    for nm, fn in (("allocate()", lambda: ctx.allocate(pc.array, None, w.n_out, flags=F, out=po.array)),
                   ("allocate_raw()", lambda: ctx.allocate_raw(pc.ptr, w.n_claim, None, po.ptr, w.n_out, F))):
        for _ in range(20): fn()
        ts=[]
        for _ in range(300):
            t0=time.perf_counter(); fn(); ts.append(time.perf_counter()-t0)
        print("graph" if graph else "eager", nm, "median %.1f us  p10 %.1f" % (np.median(ts)*1e6, np.percentile(ts,10)*1e6))
    ctx.close()
# raw copies for scale
s = torch.cuda.Stream()
h = torch.empty(160000, dtype=torch.uint8).pin_memory(); d = torch.empty(160000, dtype=torch.uint8, device="cuda")
h2 = torch.empty(80000, dtype=torch.uint8).pin_memory()
with torch.cuda.stream(s):
    for nm, fn in (("H2D 160KB + sync", lambda: (d.copy_(h, non_blocking=True), s.synchronize())),
                   ("D2H 80KB + sync", lambda: (h2.copy_(d[:80000], non_blocking=True), s.synchronize())),
                   ("H2D + D2H + sync", lambda: (d.copy_(h, non_blocking=True), h2.copy_(d[:80000], non_blocking=True), s.synchronize()))):
        for _ in range(20): fn()
        ts=[]
        for _ in range(300):
            t0=time.perf_counter(); fn(); ts.append(time.perf_counter()-t0)
        print(nm, "median %.1f us" % (np.median(ts)*1e6))
