"""GPU-box probe: cost of the windowed site scan (K2 with the per-site H + the window reduction) against the plain K2 pass.

CUDA events over 20 launches per timed block; the plain pass (pfa_site_stats_device) and the windowed pass
(pfa_site_windows_device) alternate in one run, three blocks each.  Shapes: C4 (bench.py's synthetic 10,000 x 10 Mb, one
population) with window / step pairs from 1 kb to the whole alignment, C4 with 100 gaps per 10^6 bases, the C3 shape (2,000 x 3 Mb,
two populations), and the C3 shape with 100 gaps per 10^6 bases (two populations: gap-only sites take the whole-warp pass when
the per-site H is stored)."""
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import polyfasta_b200 as pf
from polyfasta_b200 import api

SEED, P_SEG_PPM, TRI_PPM = 4, 50_000, 10_000   # bench.py's synthetic parameters
C3_SEED = 3
REPS, BLOCKS = 20, 3

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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
        return q.stdout.strip().splitlines()[0]
    except (OSError, IndexError):
        return torch.cuda.get_device_name(0)


def probe(label, aln, windows):
    out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
    bufs = {w: torch.zeros(max(2 * aln.num_pops * api.window_count(aln.total_len, *w), 1), dtype=torch.int64, device="cuda")
            for w in windows}
    torch.cuda.synchronize()
    plain = lambda: aln.site_stats_device(out.data_ptr())
    runs = [("plain K2", plain)] + [("windows %d / %d" % w, (lambda w=w: aln.site_windows_device(w[0], w[1], bufs[w].data_ptr())))
                                    for w in windows]
    for _, fn in runs:   # warm-up: module loads, pool growth
        fn()
    stream.synchronize()
    ms = {name: [] for name, _ in runs}
    for _ in range(BLOCKS):
        for name, fn in runs:
            ms[name].append(timed(fn))
    base = min(ms["plain K2"])
    print("%s  [%s]" % (label, ctx.last_kernel.split(" grid=")[0]), flush=True)
    for name, _ in runs:
        v = ms[name]
        print("  %-20s %s ms per pass   ratio %.3f" % (name, " ".join("%.4f" % x for x in v), min(v) / base), flush=True)


with torch.cuda.stream(stream):
    print("device:", card(), flush=True)
    a = pf.Alignment.synthetic(ctx, 10_000, 10_000_000, SEED, P_SEG_PPM, TRI_PPM)
    probe("C4 10,000 x 10 Mb", a, [(10_000, 10_000), (100_000, 10_000), (1_000, 1_000), (1_000_000, 1_000_000), (10_000_000, 10_000_000)])
    a.poke_gaps(SEED, 100)
    probe("C4 10,000 x 10 Mb, 100 gaps per 10^6 bases", a, [(10_000, 10_000)])
    a.free()
    n = 2_000
    a = pf.Alignment.synthetic(ctx, n, 3_000_000, C3_SEED, P_SEG_PPM, TRI_PPM)
    a.set_pops([list(range(n // 2)), list(range(n // 2, n))])
    probe("C3 shape 2,000 x 3 Mb, two populations", a, [(10_000, 10_000), (1_000, 1_000), (3_000_000, 3_000_000)])
    a.poke_gaps(C3_SEED, 100)
    probe("C3 shape 2,000 x 3 Mb, two populations, 100 gaps per 10^6 bases", a, [(10_000, 10_000)])
    a.free()
