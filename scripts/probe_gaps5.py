"""GPU-box probe: the compact validity area (PFA_VCOMPACT) and passes per slot of the validity-aware scans on gapped shards."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import polyfasta_b200 as pf

ctx = pf.Context(0)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)


def timed(fn, reps=10):
    fn(); stream.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(stream)
    for _ in range(reps):
        fn()
    b.record(stream); stream.synchronize()
    return a.elapsed_time(b) / reps


with torch.cuda.stream(stream):
    for n, L in [(10000, 2_000_000), (2000, 3_000_000)]:
        for ppm in (0, 1, 10, 100):
            aln = pf.Alignment.synthetic(ctx, n, L, 4)
            if ppm:
                aln.poke_gaps(4, ppm)
            out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
            cds = torch.zeros(71, dtype=torch.int64, device="cuda")
            row = []
            for compact, ms, mc in (("0", None, None), ("1", None, None)):
                os.environ["PFA_VCOMPACT"] = compact
                for k, v in (("PFA_SITE_TMA_M", ms), ("PFA_CDS_TMA_M", mc)):
                    os.environ.pop(k, None)
                    if v:
                        os.environ[k] = str(v)
                k2 = timed(lambda: aln.site_stats_device(out.data_ptr()))
                kn2 = ctx.last_kernel.split("passes_per_slot=")[1]
                k4 = timed(lambda: aln.cds_stats_device(cds.data_ptr()))
                kn4 = ctx.last_kernel.split("passes_per_slot=")[1]
                row.append("compact=%s K2 %.3f [m=%s] K4 %.3f [m=%s]" % (compact, k2, kn2.replace(" v_records_per_slot=", " vs="), k4, kn4.replace(" v_records_per_slot=", " vs=")))
            print("%d x %d %3d ppm: %s" % (n, L, ppm, " | ".join(row)), flush=True)
            aln.free()
