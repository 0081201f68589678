"""Small fixed workloads for ncu captures.  usage: python scripts/ncu_targets.py k4|k3|k1|k2b
k4: codon scan on the C3 shape (2000 x 3 Mb, 2 populations);  k3: pairwise 2000 rows x 100 kb;
k1: one hybrid upload of 10000 x 200 kb pinned text (raw K1 + packed K1 kernels)"""
import ctypes, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import polyfasta_b200 as pf
from polyfasta_b200 import api
from polyfasta_b200._lib import lib, check

which = sys.argv[1]
ctx = pf.Context(0)
if which == "k4":
    aln = pf.Alignment.synthetic(ctx, 2000, 3_000_000, 3)
    aln.set_pops([list(range(0, 1000)), list(range(1000, 2000))])
    out = torch.zeros(2 * 71, dtype=torch.int64, device="cuda")
    for _ in range(3):
        aln.cds_stats_device(out.data_ptr())
    ctx.sync()
    print("k4", out[:6].tolist())
elif which == "k2g":
    # the site scan with sparse gaps: 2000 x 3 Mb at 10 gaps per 10^6 bases, then 10000 x 2 Mb at 100
    for n, L, ppm in ((2000, 3_000_000, 10), (10000, 2_000_000, 100)):
        aln = pf.Alignment.synthetic(ctx, n, L, 4)
        aln.poke_gaps(4, ppm)
        out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
        for _ in range(2):
            aln.site_stats_device(out.data_ptr())
        ctx.sync()
        print("k2g", n, L, ppm, out[:2].tolist())
        aln.free()
elif which == "k1":
    n, cols = 10000, 200_000
    d = torch.empty((n, cols), dtype=torch.uint8, device="cuda")
    api.synth_text_device(ctx, d.data_ptr(), cols, n, 4, 50000, 10000, 0, cols)
    ctx.sync()
    h = torch.empty((n, cols), dtype=torch.uint8, pin_memory=True)
    h.copy_(d)
    torch.cuda.synchronize()
    for _ in range(2):
        a = pf.Alignment.from_host_ptr(ctx, h.data_ptr(), n, cols, cols)
        ctx.sync()
        print("k1", ctx.ingest_stats())
        a.free()
elif which == "k2b":
    # the batched site scan on the C5 shape: 4,000 resident loci of 100 x 5 kb
    b = api.Batch(ctx)
    for i in range(4000):
        b.add_synthetic(100, 5000, 5 + i)
    b.stage()
    for _ in range(3):
        b.scan(jc=True)
    print("k2b", b.result(0)["S"], b.kernel_ms())
else:
    a = pf.Alignment.synthetic(ctx, 2000, 100_000, 3)
    out = torch.zeros(1, dtype=torch.int64, device="cuda")
    D = torch.zeros((2000, 2000), dtype=torch.int32, device="cuda")
    for _ in range(2):
        check(lib().pfa_pairwise_device(a.handle, ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(D.data_ptr())), ctx.handle)
    ctx.sync()
    print("k3", int(out[0]))
