import importlib, os, sys, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
pkg = importlib.import_module("k8s-dra-driver_b200")
s = torch.cuda.Stream(); torch.cuda.set_stream(s)
ctx = pkg.api.Context(device=0, stream=s.cuda_stream)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
def timeit(w, n_claim, do_flush, reps=50):
    ctx.set_table(w.table); ctx.set_inventory(w.gpus, w.node_off)
    d_claims = torch.from_numpy(w.claims.view(np.uint8).copy()).cuda()
    d_out = torch.zeros(max(w.n_out,1) * 8, dtype=torch.uint8, device="cuda")
    ts=[]
    for it in range(reps+5):
        if do_flush: flush.fill_(1)
        a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
        a.record(s); ctx.allocate_device(d_claims.data_ptr(), n_claim, None, d_out.data_ptr(), max(n_claim,1), pkg.api.F_FRESH_INVENTORY); b.record(s)
        torch.cuda.synchronize()
        if it>=5: ts.append(a.elapsed_time(b)*1e3)
    return np.median(ts)
w = pkg.synth.cfg2()
print("stage=%s" % ("off" if os.environ.get("DRA_NO_STAGE") else "on"))
print("cfg2 full batch, flush:    %.2f us" % timeit(w, w.n_claim, True))
print("cfg2 full batch, no flush: %.2f us" % timeit(w, w.n_claim, False))
print("empty batch (0 claims, 126 CTAs), flush:    %.2f us" % timeit(w, 0, True))
print("empty batch (0 claims, 126 CTAs), no flush: %.2f us" % timeit(w, 0, False))

def noop(grid, block, smem, reps=50):
    ts=[]
    for it in range(reps+5):
        a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
        a.record(s); ctx.debug_noop(grid, block, smem); b.record(s)
        torch.cuda.synchronize()
        if it>=5: ts.append(a.elapsed_time(b)*1e3)
    return np.median(ts)
for g,b_,sm in [(1,32,0),(126,32,0),(126,256,0),(126,256,43*1024),(126,256,204*1024),(126,512,204*1024)]:
    print("noop <<<%d,%d,%dKB>>>: %.2f us" % (g,b_,sm//1024, noop(g,b_,sm)))
def two_events(reps=50):
    ts=[]
    for it in range(reps):
        a=torch.cuda.Event(enable_timing=True); b=torch.cuda.Event(enable_timing=True)
        a.record(s); b.record(s); torch.cuda.synchronize(); ts.append(a.elapsed_time(b)*1e3)
    return np.median(ts)
print("two events back to back: %.2f us" % two_events())
