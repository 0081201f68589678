"""GPU-box probe: cost of the haplotype classes (pfa_haplotypes_device) next to the plain site scan.

Alignments of rows drawn from 500 founders with a random base written at 0.1 % of the cells (so most rows are distinct and many
sites are variable), generated as text on the device with torch and uploaded from there.  Shapes: C4 (10,000 x 10 Mb), the C3
shape (2,000 x 3 Mb) and C4 with 10 gaps per 10^6 bases; one population of all rows.

Per shape:
  1. the first pfa_haplotypes_device call of the alignment (whole alignment), which also builds the cached row-major planes of
     the marked sites (K3's var-flags pass, cub site list, transpose) and the row-ordered exception list, timed with CUDA events
     inside a torch.profiler pass (CUDA activities) that splits it kernel by kernel;
  2. CUDA events over 20 launches per timed block, three blocks each, alternating: the site scan (pfa_site_stats_device), the
     whole alignment and windows of W = 10 kb every S = 5 kb, with the row-major planes cached;
  3. a separate torch.profiler pass over five warm calls of each haplotype form: hash, sort and verify.

    python scripts/probe_haplotypes.py [--rows N --sites L]   (--rows / --sites: a small shape for a dry run)"""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FOUNDERS, CHANGE = 500, 0.001
REPS, BLOCKS = 20, 3
WINDOW, STEP = 10_000, 5_000


def shapes(args):
    """(label, rows, sites, seed, gap_ppm) of every probed alignment"""
    if args.rows:
        return [("dry run %d x %d" % (args.rows, args.sites), args.rows, args.sites, 4, 0),
                ("dry run %d x %d, 10 gaps per 10^6 bases" % (args.rows, args.sites), args.rows, args.sites, 4, 10)]
    return [("C4 10,000 x 10 Mb, 500 founders, 0.1 % changes", 10_000, 10_000_000, 4, 0),
            ("C3 shape 2,000 x 3 Mb, 500 founders, 0.1 % changes", 2_000, 3_000_000, 3, 0),
            ("C4 10,000 x 10 Mb, 500 founders, 0.1 % changes, 10 gaps per 10^6 bases", 10_000, 10_000_000, 4, 10)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0]


def founder_text(torch, n, L, seed):
    """uint8 [n][L] upper-case text on the device: rows drawn from FOUNDERS random rows, then a random base at CHANGE of the cells"""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device="cuda")
    chunk = max(1, (1 << 29) // max(L, 1))   # rows per generation step: at most 4 GB of int64 indices
    F = torch.empty((FOUNDERS, L), dtype=torch.uint8, device="cuda")
    for f0 in range(0, FOUNDERS, chunk):
        f1 = min(FOUNDERS, f0 + chunk)
        F[f0:f1] = lut[torch.randint(0, 4, (f1 - f0, L), generator=g, device="cuda")]
    pick = torch.randint(0, FOUNDERS, (n,), generator=g, device="cuda")
    text = torch.empty((n, L), dtype=torch.uint8, device="cuda")
    for r0 in range(0, n, 8 * chunk):
        r1 = min(n, r0 + 8 * chunk)
        text[r0:r1] = F[pick[r0:r1]]
    del F
    flat = text.view(-1)
    todo = int(n * L * CHANGE)
    for c0 in range(0, todo, 1 << 26):
        m = min(1 << 26, todo - c0)
        flat[torch.randint(0, n * L, (m,), generator=g, device="cuda")] = lut[torch.randint(0, 4, (m,), generator=g, device="cuda")]
    return text


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--sites", type=int, default=0)
    args = ap.parse_args()
    todo = shapes(args)
    for label, n, L, seed, gaps in todo:
        print("%s: %d windows of %d every %d" % (label, -(-max(L - WINDOW, 0) // STEP) + 1, WINDOW, STEP))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_haplotypes: no CUDA device")
    import numpy as np
    from torch.profiler import ProfilerActivity, profile

    import polyfasta_b200 as pf
    from polyfasta_b200 import api

    ctx = pf.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)

    def events():
        return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        a, b = events()
        a.record(stream)
        for _ in range(REPS):
            fn()
        b.record(stream)
        stream.synchronize()
        return a.elapsed_time(b) / REPS

    with torch.cuda.stream(stream):
        print("device: %s" % card(), flush=True)
        for label, n, L, seed, gaps in todo:
            text = founder_text(torch, n, L, seed)
            torch.cuda.synchronize()
            aln = pf.Alignment.from_device_ptr(ctx, text.data_ptr(), n, L, L)
            ctx.sync()
            del text
            torch.cuda.empty_cache()
            if gaps:
                aln.poke_gaps(seed, gaps)
            nwin = api.window_count(L, WINDOW, STEP)
            out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
            rep1 = torch.zeros(n, dtype=torch.int32, device="cuda")
            repw = torch.zeros(nwin * n, dtype=torch.int32, device="cuda")
            torch.cuda.synchronize()
            aln.site_stats_device(out.data_ptr())   # warm-up of the site scan and the pool
            stream.synchronize()
            # 1. the first call: the row-major cache is built inside it
            a, b = events()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                a.record(stream)
                aln.haplotypes_device(L, L, rep1.data_ptr())
                b.record(stream)
                stream.synchronize()
            cold = a.elapsed_time(b)
            r = rep1.cpu().numpy()
            print("%s  [has_invalid=%d, planes %.2f GB, haplotypes %d of %d rows]" % (label, aln.has_invalid, aln.packed_bytes / 1e9,
                                                                                   len(np.unique(r)), n), flush=True)
            print("  first call, whole alignment (builds the row-major planes; under the profiler): %.4f ms" % cold)
            print(prof.key_averages().table(sort_by="device_time_total", row_limit=14), flush=True)
            # 2. warm calls against the site scan
            runs = [("site scan", lambda: aln.site_stats_device(out.data_ptr())),
                    ("haplotypes whole alignment", lambda: aln.haplotypes_device(L, L, rep1.data_ptr())),
                    ("haplotypes W 10 kb / S 5 kb", lambda: aln.haplotypes_device(WINDOW, STEP, repw.data_ptr()))]
            for _, fn in runs:
                fn()
            stream.synchronize()
            ms = {name: [] for name, _ in runs}
            for _ in range(BLOCKS):
                for name, fn in runs:
                    ms[name].append(timed(fn))
            base = min(ms["site scan"])
            for name, _ in runs:
                v = ms[name]
                print("  %-28s %s ms per call   ratio to the site scan %.3f" % (name, " ".join("%.4f" % x for x in v), min(v) / base), flush=True)
            # 3. kernel by kernel inside warm calls (a separate, profiled pass)
            for name, fn in runs[1:]:
                with profile(activities=[ProfilerActivity.CUDA]) as prof:
                    for _ in range(5):
                        fn()
                    stream.synchronize()
                print("  five warm calls: %s" % name)
                print(prof.key_averages().table(sort_by="device_time_total", row_limit=12), flush=True)
            aln.free()
            del out, rep1, repw
            ctx.trim()
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
