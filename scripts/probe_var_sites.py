"""GPU-box probe: the site scan over the list of sites where rows differ (pfa_var_sites_ensure + the list path of
pfa_site_scan_tma_kernel) against the dense scan of other builds of the library.

For every build given with --build NAME=ROOT (a tree whose polyfasta_b200 package is built), in a subprocess of its own:
  * C4 (bench.py's synthetic 10,000 x 10 Mb): the first scan of a fresh alignment (the list is built inside it) and the
    steady-state scan, CUDA events over 20 launches x 3 blocks after one warm-up; then, with torch.profiler (CUDA
    activities) in a separate pass, the device time of every kernel of the first scan of another fresh alignment: the
    var-flags pass and cub's select are the list build.
  * a density sweep: p_seg_ppm from 0 to 10^6 at n = 2,000 (10 Mb) and n = 10,000 (2 Mb), steady-state scan per point
    (every point is larger than the 126 MB L2).
Bytes the list path fetches = listed sites x planes x record bytes + 8 bytes per list entry; the rate on those bytes is the
honest bandwidth figure of that path (bench.py's roofline divides the 0.25 B/base that a dense scan must read).

    python scripts/probe_var_sites.py --build new=. --build parent=../parent [--rows N --sites L]  (small shape: dry run)"""
import argparse
import json
import os
import subprocess
import sys

SEED, P_SEG_PPM, TRI_PPM = 4, 50_000, 10_000  # bench.py's synthetic parameters
REPS, BLOCKS = 20, 3
SWEEP_PPM = [0, 1_000, 10_000, 50_000, 100_000, 200_000, 300_000, 400_000, 500_000, 700_000, 1_000_000]


def worker(args):
    sys.path.insert(0, os.path.abspath(args.worker))
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("probe_var_sites: no CUDA device")
    import polyfasta_b200 as pf
    ctx = pf.Context(0)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    res = {}

    def timed(fn, reps=REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(reps):
            fn()
        b.record(stream)
        stream.synchronize()
        return a.elapsed_time(b) / reps

    with torch.cuda.stream(stream):
        n, L = (args.rows, args.sites) if args.rows else (10_000, 10_000_000)
        aln = pf.Alignment.synthetic(ctx, n, L, SEED, P_SEG_PPM, TRI_PPM)
        out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        scan = lambda: aln.site_stats_device(out.data_ptr())  # noqa: E731
        first = timed(scan, 1)
        timed(scan, 1)
        steady = sorted(timed(scan) for _ in range(BLOCKS))
        res["c4"] = {"n": n, "L": L, "rec": aln.packed_bytes // (3 * L), "first_ms": first, "steady_ms": steady[len(steady) // 2],
                     "steady_all": steady, "kernel": ctx.last_kernel, "S": int(out[0].item())}
        aln.free()
        del out
        # the first scan of a fresh alignment under the profiler: kernel by kernel
        aln = pf.Alignment.synthetic(ctx, n, L, SEED, P_SEG_PPM, TRI_PPM)
        out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            aln.site_stats_device(out.data_ptr())
            stream.synchronize()
        kern = {}
        for ev in prof.events():
            if ev.device_type.name == "CUDA" and ev.device_time_total > 0 and "emcpy" not in ev.name and "emset" not in ev.name:
                kern[ev.name[:90]] = kern.get(ev.name[:90], 0.0) + ev.device_time_total / 1e3
        res["c4_first_kernels_ms"] = kern
        aln.free()
        del out
        sweep = []
        shapes = [(args.rows, args.sites)] if args.rows else [(2_000, 10_000_000), (10_000, 2_000_000)]
        for sn, sL in shapes:
            for ppm in SWEEP_PPM:
                a = pf.Alignment.synthetic(ctx, sn, sL, SEED, ppm, TRI_PPM)
                o = torch.zeros(a.site_len(), dtype=torch.int64, device="cuda")
                torch.cuda.synchronize()
                f = lambda: a.site_stats_device(o.data_ptr())  # noqa: E731
                timed(f, 2)
                ms = sorted(timed(f) for _ in range(2))[0]
                sweep.append({"n": sn, "L": sL, "ppm": ppm, "ms": ms, "S": int(o[0].item()), "kernel": ctx.last_kernel})
                a.free()
                del o
        res["sweep"] = sweep
    print("RESULT " + json.dumps(res), flush=True)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    except FileNotFoundError:
        return "unknown (no nvidia-smi)"
    return q.stdout.strip().splitlines()[0] if q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--build", action="append", default=[], help="NAME=ROOT")
    ap.add_argument("--rows", type=int, default=0)
    ap.add_argument("--sites", type=int, default=0)
    ap.add_argument("--worker", default=None)
    args = ap.parse_args()
    if args.worker:
        return worker(args)
    builds = [b.split("=", 1) for b in args.build] or [["this", "."]]
    print("device: %s" % card(), flush=True)
    results = {}
    for name, root in builds:
        cmd = [sys.executable, os.path.abspath(__file__), "--worker", root]
        if args.rows:
            cmd += ["--rows", str(args.rows), "--sites", str(args.sites)]
        p = subprocess.run(cmd, capture_output=True, text=True)
        line = [x for x in p.stdout.splitlines() if x.startswith("RESULT ")]
        if p.returncode or not line:
            sys.stderr.write(p.stdout + p.stderr)
            raise SystemExit("probe_var_sites: build %s failed" % name)
        results[name] = json.loads(line[0][7:])
    for name, r in results.items():
        c = r["c4"]
        rec = c["rec"]
        listed = " sites=" in c["kernel"]
        print("\n[%s] C4 %d x %d: %s" % (name, c["n"], c["L"], c["kernel"]))
        print("  first scan of a fresh alignment %.3f ms, steady-state scan %.3f ms (blocks %s)" % (
            c["first_ms"], c["steady_ms"], ", ".join("%.3f" % x for x in c["steady_all"])))
        fetched = (c["S"] * 2 * rec + 8 * c["S"]) if listed else c["L"] * 2 * rec
        print("  bytes fetched per scan %.3f GB (%s), %.0f GB/s on them" % (
            fetched / 1e9, "%d listed sites x 2 planes x %d B + the list" % (c["S"], rec) if listed else "every site x 2 planes x %d B" % rec,
            fetched / c["steady_ms"] / 1e6))
        build = 0.0
        for k, ms in sorted(r["c4_first_kernels_ms"].items(), key=lambda kv: -kv[1]):
            print("    first scan kernel %8.3f ms  %s" % (ms, k))
            if "var_flags" in k or "DeviceSelect" in k or "DeviceCompact" in k:
                build += ms
        print("  list build (var flags + select, device time) %.3f ms" % build)
    names = list(results)
    print("\ndensity sweep: steady-state scan ms (S = variable sites; * = the list path ran)")
    print("%6s %10s %8s %9s " % ("n", "sites", "ppm", "S") + " ".join("%14s" % x for x in names))
    for i, pt in enumerate(results[names[0]]["sweep"]):
        cells = []
        for x in names:
            q = results[x]["sweep"][i]
            cells.append("%13.3f%s" % (q["ms"], "*" if " sites=" in q["kernel"] else " "))
        print("%6d %10d %8d %9d " % (pt["n"], pt["L"], pt["ppm"], pt["S"]) + " ".join(cells))


if __name__ == "__main__":
    main()
