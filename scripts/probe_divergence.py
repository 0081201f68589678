"""GPU-box probe: cost of the divergence scan (d_xy between populations) next to the plain site scan.

CUDA events over 20 launches per timed block; the site scan (pfa_site_stats_device), the whole-alignment divergence
(pfa_divergence_device) and the divergence windows of 10 kb (pfa_divergence_windows_device) alternate in one run, three blocks
each, after one warm-up call of each.  Then, in a separate pass with torch.profiler (CUDA activities), the device time of every
kernel inside five pfa_divergence_device calls: the var-flags pass, the cub site list, the per-site kernel and the escape kernel.
Shapes (all larger than the 126 MB L2): C4 (bench.py's synthetic 10,000 x 10 Mb) split into two populations of 5,000 rows, the
C3 shape (2,000 x 3 Mb, two populations), and C4 with 10 gaps per 10^6 bases.

    python scripts/probe_divergence.py [--rows N --sites L]   (--rows / --sites: a small shape for a dry run)"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SEED, P_SEG_PPM, TRI_PPM = 4, 50_000, 10_000   # bench.py's synthetic parameters
C3_SEED = 3
REPS, BLOCKS = 20, 3
WINDOW = 10_000


def shapes(args):
    """(label, rows, sites, seed, gap_ppm) of every probed alignment; two populations: the halves"""
    if args.rows:
        return [("dry run %d x %d" % (args.rows, args.sites), args.rows, args.sites, SEED, 0),
                ("dry run %d x %d, 10 gaps per 10^6 bases" % (args.rows, args.sites), args.rows, args.sites, SEED, 10)]
    return [("C4 10,000 x 10 Mb, two populations of 5,000", 10_000, 10_000_000, SEED, 0),
            ("C3 shape 2,000 x 3 Mb, two populations of 1,000", 2_000, 3_000_000, C3_SEED, 0),
            ("C4 10,000 x 10 Mb, two populations, 10 gaps per 10^6 bases", 10_000, 10_000_000, SEED, 10)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--sites", type=int, default=0)
    args = ap.parse_args()
    todo = shapes(args)
    for label, n, L, seed, gaps in todo:
        print("%s: %d populations x %d rows, %d windows of %d" % (label, 2, n // 2, -(-L // WINDOW), WINDOW))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_divergence: no CUDA device")
    import polyfasta_b200 as pf
    from polyfasta_b200 import api

    ctx = pf.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)

    def timed(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(REPS):
            fn()
        b.record(stream)
        stream.synchronize()
        return a.elapsed_time(b) / REPS

    with torch.cuda.stream(stream):
        print("device: %s" % card(), flush=True)
        for label, n, L, seed, gaps in todo:
            aln = pf.Alignment.synthetic(ctx, n, L, seed, P_SEG_PPM, TRI_PPM)
            if gaps:
                aln.poke_gaps(seed, gaps)
            aln.set_pops([list(range(n // 2)), list(range(n // 2, n))])
            nwin = api.window_count(L, WINDOW, WINDOW)
            out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
            dv = torch.zeros(1, dtype=torch.int64, device="cuda")
            dw = torch.zeros(2 * nwin, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            runs = [("site scan", lambda: aln.site_stats_device(out.data_ptr())),
                    ("divergence", lambda: aln.divergence_device(dv.data_ptr())),
                    ("divergence windows 10 kb", lambda: aln.divergence_windows_device(WINDOW, WINDOW, dw.data_ptr()))]
            for _, fn in runs:   # warm-up: module loads, pool growth
                fn()
            stream.synchronize()
            ms = {name: [] for name, _ in runs}
            for _ in range(BLOCKS):
                for name, fn in runs:
                    ms[name].append(timed(fn))
            base = min(ms["site scan"])
            print("%s  [has_invalid=%d, D_xy=%d, planes %.2f GB]" % (label, aln.has_invalid, int(dv.cpu()[0]), aln.packed_bytes / 1e9), flush=True)
            for name, _ in runs:
                v = ms[name]
                print("  %-26s %s ms per call   ratio to the site scan %.3f" % (name, " ".join("%.4f" % x for x in v), min(v) / base), flush=True)
            # kernel by kernel inside one divergence call (a separate, profiled pass)
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    aln.divergence_device(dv.data_ptr())
                stream.synchronize()
            print(prof.key_averages().table(sort_by="device_time_total", row_limit=8), flush=True)
            aln.free()
            del out, dv, dw
            ctx.trim()


if __name__ == "__main__":
    main()
