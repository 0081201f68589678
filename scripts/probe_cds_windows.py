"""GPU-box probe: cost of the codon windows (pfa_cds_windows_device, --cds --window) next to the --cds scans.

CUDA events over 20 launches per timed block; K2 + K4 as --cds runs them (pfa_site_stats_device then pfa_cds_stats_device) and
pfa_cds_windows_device at W = 30,000, step = 15,000 alternate in one run, three blocks each, after one warm-up call of each.
Then, in a separate pass with torch.profiler (CUDA activities), the device time of every kernel inside five
pfa_cds_windows_device calls: K2 with the per-site H, K4 with the labels, the bins kernel, the scan and the window kernel.
Shapes (both larger than the 126 MB L2): the C3 shape (2,000 x 3 Mb, two populations of 1,000) and 10,000 x 2 Mb with 10 gaps per
10^6 bases (two populations of 5,000).

    python scripts/probe_cds_windows.py [--rows N --sites L]   (--rows / --sites: a small shape for a dry run)"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

P_SEG_PPM, TRI_PPM = 50_000, 10_000   # bench.py's synthetic parameters
REPS, BLOCKS = 20, 3
WINDOW, STEP = 30_000, 15_000


def shapes(args):
    """(label, rows, sites, seed, gap_ppm) of every probed alignment; two populations: the halves"""
    if args.rows:
        return [("dry run %d x %d" % (args.rows, args.sites), args.rows, args.sites, 3, 0),
                ("dry run %d x %d, 10 gaps per 10^6 bases" % (args.rows, args.sites), args.rows, args.sites, 4, 10)]
    return [("C3 shape 2,000 x 3 Mb, two populations of 1,000", 2_000, 3_000_000, 3, 0),
            ("10,000 x 2 Mb, two populations of 5,000, 10 gaps per 10^6 bases", 10_000, 2_000_000, 4, 10)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--sites", type=int, default=0)
    args = ap.parse_args()
    todo = shapes(args)
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_cds_windows: no CUDA device")
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
            nwin = api.window_count(L, WINDOW, STEP)
            site = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
            cds = torch.zeros(2 * api.PFA_CDS_LEN, dtype=torch.int64, device="cuda")
            win = torch.zeros(2 * nwin * api.PFA_CDS_WIN_LEN, dtype=torch.int64, device="cuda")
            torch.cuda.synchronize()
            runs = [("K2 + K4 (--cds)", lambda: (aln.site_stats_device(site.data_ptr()), aln.cds_stats_device(cds.data_ptr()))),
                    ("cds windows 30 kb / 15 kb", lambda: aln.cds_windows_device(WINDOW, STEP, win.data_ptr()))]
            for _, fn in runs:   # warm-up: module loads, pool growth
                fn()
            stream.synchronize()
            ms = {name: [] for name, _ in runs}
            for _ in range(BLOCKS):
                for name, fn in runs:
                    ms[name].append(timed(fn))
            base = min(ms[runs[0][0]])
            w = win.cpu().numpy().reshape(2, nwin, api.PFA_CDS_WIN_LEN)
            print("%s  [has_invalid=%d, planes %.2f GB, %d windows, S_s + S_n of the windows: %d]" %
                  (label, aln.has_invalid, aln.packed_bytes / 1e9, nwin, int(w[:, :, 2].sum() + w[:, :, 4].sum())), flush=True)
            for name, _ in runs:
                v = ms[name]
                print("  %-26s %s ms per call   ratio to K2 + K4 %.3f" % (name, " ".join("%.4f" % x for x in v), min(v) / base), flush=True)
            # kernel by kernel inside the windows call (a separate, profiled pass)
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for _ in range(5):
                    aln.cds_windows_device(WINDOW, STEP, win.data_ptr())
                stream.synchronize()
            print(prof.key_averages().table(sort_by="device_time_total", row_limit=10, max_name_column_width=70), flush=True)
            aln.free()
            del site, cds, win
            ctx.trim()


if __name__ == "__main__":
    main()
