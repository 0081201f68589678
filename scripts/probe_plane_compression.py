"""Does compressible device memory make the planes cheaper to read?

For each kind of plane memory (PFA_PLANE_ALLOC = pool | vmm | compressible), alternated and repeated, this times the
read-only probe (`read_probe(2, 5)`: one streaming pass over the two base planes) on three inputs, and the site scan (K2)
itself on the first:
  c4      the C4 planes (10,000 x 10 Mb synthetic, 95 % monomorphic sites: most 128-byte lines are uniform)
  random  random ACGT text made on the device and encoded through from_device_ptr (incompressible: must not gain)
  allA    an all-A alignment (every line uniform)
The vmm arm is the same mapping without compression: it separates page-size or mapping effects from compression.
--sweep adds passes per slot (PFA_SITE_TMA_M 1..4) x slots per warp (PFA_SITE_TMA 1, 2) for K2 on C4, and PFA_CDS_TMA_M 1..4
for the codon scan (K4) on C3, pool against compressible planes.

  python scripts/probe_plane_compression.py [--reps 3] [--launches 10] [--sweep] [--small]
"""
import argparse
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KINDS = ("pool", "vmm", "compressible")


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,driver_version", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = "nvidia-smi unavailable: %s" % e
    print("card (name, power limit, max SM clock, driver):", out)
    try:
        cu = ctypes.CDLL("libcuda.so.1")
        cu.cuInit(0)
        ver, dev, attr = ctypes.c_int(), ctypes.c_int(), ctypes.c_int(-1)
        cu.cuDriverGetVersion(ctypes.byref(ver))
        cu.cuDeviceGet(ctypes.byref(dev), 0)
        cu.cuDeviceGetAttribute(ctypes.byref(attr), 107, dev)  # CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED
        print("CUDA driver API version %d, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED = %d" % (ver.value, attr.value))
    except OSError as e:
        print("libcuda not loadable: %s" % e)
    sys.stdout.flush()


def time_launches(torch, stream, fn, launches):
    fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(launches):
        fn()
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--launches", type=int, default=10)
    ap.add_argument("--sweep", action="store_true")
    ap.add_argument("--small", action="store_true", help="a tiny shape (rehearsal)")
    args = ap.parse_args()
    card()
    import torch
    import polyfasta_b200 as pf
    stream = torch.cuda.Stream()   # not the legacy default stream: set_stream(0) would mean the ctx's own stream
    torch.cuda.set_stream(stream)
    ctx = pf.default_context(0)
    ctx.set_stream(stream.cuda_stream)
    n, L = (10_000, 10_000_000) if not args.small else (1000, 200_000)
    tn, tL = (10_000, 1_000_000) if not args.small else (1000, 100_000)
    ld = (tL + 255) // 256 * 256
    lut = torch.tensor([ord(c) for c in "ACGT"], dtype=torch.uint8, device="cuda")
    rand_text = torch.empty((tn, ld), dtype=torch.uint8, device="cuda")
    torch.manual_seed(7)
    for r in range(0, tn, 200):
        rand_text[r:r + 200] = lut[torch.randint(0, 4, (min(200, tn - r), ld), device="cuda")]
    a_text = torch.full((tn, ld), ord("A"), dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    out = None
    results = {}
    print("inputs: c4 %d x %d (%.1f GB of planes), random / allA %d x %d (%.2f GB of planes); read_probe(2, 5) and K2 over %d launches"
          % (n, L, 3 * n * L / 8 / 1e9 * 1.024, tn, tL, 3 * tn * tL / 8 / 1e9 * 1.024, args.launches))
    for rep in range(args.reps):
        for kind in (KINDS if rep % 2 == 0 else KINDS[::-1]):
            os.environ["PFA_PLANE_ALLOC"] = kind
            row = {}
            c4 = pf.Alignment.synthetic(ctx, n, L, 4)
            got_kind = c4.plane_alloc
            if out is None:
                out = torch.zeros(c4.site_len(), dtype=torch.int64, device="cuda")
            row["c4_probe"] = c4.read_probe(2, 5)
            row["c4_k2"] = time_launches(torch, stream, lambda: c4.site_stats_device(out.data_ptr()), args.launches)
            kernel = ctx.last_kernel
            torch.cuda.synchronize()
            sh = (int(out[0]), int(out[1]))
            c4.free()
            ctx.trim()
            for name, text in (("random", rand_text), ("allA", a_text)):
                a = pf.Alignment.from_device_ptr(ctx, text.data_ptr(), tn, tL, ld)
                row[name + "_probe"] = a.read_probe(2, 5)
                row[name + "_kind"] = a.plane_alloc
                a.free()
                ctx.trim()
            results.setdefault(kind, []).append(row)
            print("rep %d %-12s granted=%-12s c4 probe %.3f ms  c4 K2 %.3f ms  random probe %.4f ms (%s)  allA probe %.4f ms (%s)  S,H=%s  %s"
                  % (rep, kind, got_kind, row["c4_probe"], row["c4_k2"], row["random_probe"], row["random_kind"], row["allA_probe"],
                     row["allA_kind"], sh, kernel))
            sys.stdout.flush()
    print("\nmedian over %d reps (ms), ratio to pool:" % args.reps)
    med = lambda xs: sorted(xs)[len(xs) // 2]  # noqa: E731
    for key in ("c4_probe", "c4_k2", "random_probe", "allA_probe"):
        base = med([r[key] for r in results["pool"]])
        print("  %-13s " % key + "  ".join("%s %.4f (%.3f; range %.4f-%.4f)" % (k, med([r[key] for r in results[k]]), med([r[key] for r in results[k]]) / base,
                                                                            min(r[key] for r in results[k]), max(r[key] for r in results[k])) for k in KINDS))
    if args.sweep:
        sweep(torch, stream, pf, ctx, args, n, L)
    os.environ.pop("PFA_PLANE_ALLOC", None)


def sweep(torch, stream, pf, ctx, args, n, L):
    print("\nsweep: K2 on c4 and K4 on c3 (2,000 x 3 Mb, two populations), pool against compressible planes, alternated")
    alns = {}
    for kind in ("pool", "compressible"):
        os.environ["PFA_PLANE_ALLOC"] = kind
        alns[kind] = pf.Alignment.synthetic(ctx, n, L, 4)
    out = torch.zeros(alns["pool"].site_len(), dtype=torch.int64, device="cuda")
    for rep in range(2):
        for slots in ("1", "2"):
            for m in ("1", "2", "3", "4"):
                os.environ["PFA_SITE_TMA"], os.environ["PFA_SITE_TMA_M"] = slots, m
                line = []
                for kind in ("pool", "compressible") if rep == 0 else ("compressible", "pool"):
                    ms = time_launches(torch, stream, lambda: alns[kind].site_stats_device(out.data_ptr()), args.launches)
                    line.append("%s %.3f" % (kind, ms))
                print("  rep %d K2 slots=%s passes_per_slot=%s: %s  (%s)" % (rep, slots, m, "  ".join(line), ctx.last_kernel.split(" grid=")[1]))
                sys.stdout.flush()
    for k in ("PFA_SITE_TMA", "PFA_SITE_TMA_M"):
        os.environ.pop(k)
    for a in alns.values():
        a.free()
    ctx.trim()
    cn, cL = (2000, 3_000_000) if not args.small else (200, 30_000)
    alns = {}
    for kind in ("pool", "compressible"):
        os.environ["PFA_PLANE_ALLOC"] = kind
        alns[kind] = pf.Alignment.synthetic(ctx, cn, cL, 3)
        alns[kind].set_pops([list(range(cn // 2)), list(range(cn // 2, cn))])
    d_cds = torch.zeros(2 * 71, dtype=torch.int64, device="cuda")
    for rep in range(2):
        for m in ("default", "1", "2", "3", "4"):
            if m == "default":
                os.environ.pop("PFA_CDS_TMA_M", None)
            else:
                os.environ["PFA_CDS_TMA_M"] = m
            line = []
            for kind in ("pool", "compressible") if rep == 0 else ("compressible", "pool"):
                ms = time_launches(torch, stream, lambda: alns[kind].cds_stats_device(d_cds.data_ptr()), 4 * args.launches)
                line.append("%s %.4f" % (kind, ms))
            print("  rep %d K4 passes_per_slot=%s: %s  (%s)" % (rep, m, "  ".join(line), ctx.last_kernel))
            sys.stdout.flush()
    os.environ.pop("PFA_CDS_TMA_M", None)
    for a in alns.values():
        a.free()
    ctx.trim()


if __name__ == "__main__":
    main()
