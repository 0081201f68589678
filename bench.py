#!/usr/bin/env python3
"""Benchmark of the PolyFastA hot path on B200:  python bench.py --gpus N --steps K --warmup W  [--impl reference] [--workload c4|c3|c5]
[--dump-outputs DIR]

Workloads (BASELINE.json configs; DESIGN.md section 4):

  c4 (default, the configuration the metric is quoted on): synthetic non-coding alignment of 10,000 sequences x 10 Mb (1e11
      aligned bases), pure ACGT, ~5 % segregating sites with a 1/k spectrum, 1 % of them tri-allelic; generated directly in
      packed form on the device (polyfasta_b200.synth is the numpy twin).  With N GPUs the COLUMNS are split in N contiguous
      ranges (strong scaling: the total stays 1e11 bases); the int64 vector [S, H, SFS] is summed over the shards inside the
      scan kernel's last block over NVLink peer memory (or with one NCCL all-reduce: --collective nccl).
      --gaps-ppm G turns G cells per million into '-' (sparse validity: the scans fetch only the flagged pieces of the v plane);
      --force-validity makes them read the whole validity plane (0.375 B/base, the worst case).
  c3: synthetic in-frame CDS alignment 2,000 x 3 Mb, two populations (the two halves of the rows), --cds --jc: one step = site
      scan (K2) + codon scan (K4) over the resident shard, columns split codon-aligned over the ranks.
  c5: --dir batch of 100,000 loci of 100 x 5 kb: locus i goes to rank i mod N, NO collective; one step = the segmented
      site scan + finalisation of every locus of the rank (batches of resident loci), rows gathered on rank 0.

  value       aligned bases/s = bases of the whole job * K / (device time of the K steps, max over ranks); inputs resident in HBM
  roofline    the dominant scan kernel: algorithmic bytes (what the scan must read: two bit-planes = 0.25 B/base for pure-ACGT
              input, three = 0.375 B/base otherwise; DESIGN.md) / its mean CUDA-event duration inside the timed region
  e2e         the same metric from HOST input through the public API: c4 / c3: pinned row-major text -> H2D -> K1 encode -> scans
              -> sum over shards -> D2H -> K5 finalise -> Python tuples; c5: FASTA files on disk -> the drop-in's --dir path -> rows
  cpu_baseline / --impl reference: the CPU oracle port (oracle/c, C + OpenMP, all host threads) on a bounded sample of the same
              workload, plus (cpu_baseline.python_1core) the pure-Python oracle on one core -- the reference itself is pure
              Python of that speed class (~1e7 bases/s on one core, BASELINE.md) and cannot travel to the GPU box.
"""
import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_SEQ = 10_000
N_SITES = 10_000_000
SEED = 4
P_SEG_PPM = 50_000
TRI_PPM = 10_000
C3_N, C3_SITES, C3_SEED = 2_000, 3_000_000, 3
C5_LOCI, C5_N, C5_SITES, C5_SEED = 100_000, 100, 5_000, 5
METRIC = "aligned bases/sec (seqs x sites)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c4", choices=["c4", "c3", "c5"])
    ap.add_argument("--n", type=int, default=0, help="rows (default: the workload's)")
    ap.add_argument("--sites", type=int, default=0, help="sites (default: the workload's)")
    ap.add_argument("--loci", type=int, default=C5_LOCI, help="c5: number of loci")
    ap.add_argument("--e2e-sites", type=int, default=1_000_000, help="c4: column slice used for the end-to-end leg")
    ap.add_argument("--e2e-loci", type=int, default=8_000, help="c5: loci written as FASTA files for the end-to-end leg")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-sample-sites", type=int, default=0, help="columns (c5: loci) of the CPU sample")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--collective", default="fused", choices=["fused", "nccl"],
                    help="N > 1: 'fused' = the scan kernel's last block sums the shard vectors over NVLink peer memory (pfa_xchg, the product "
                         "path); 'nccl' = scan kernel + torch.distributed all_reduce (comparison only)")
    ap.add_argument("--force-validity", action="store_true", help="c4: make the scan read the whole validity plane too (0.375 B/base)")
    ap.add_argument("--gaps-ppm", type=int, default=0, help="c4: gaps per million bases poked into the alignment (sparse validity)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last step computed as DIR/<name>.npy "
                    "(float64, at most 64 MB in all): c4 site_stats = [S, H, folded SFS]; c3 site_stats and cds_stats [population][71]; "
                    "c5 locus, S, H, sfs, pi_site, theta_site, tajimas_d (NaN for NA) per locus.  The inputs are seeded, so two builds "
                    "can be compared output for output")
    a = ap.parse_args()
    if a.dump_outputs and a.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    dn, ds = {"c4": (N_SEQ, N_SITES), "c3": (C3_N, C3_SITES), "c5": (C5_N, C5_SITES)}[a.workload]
    a.n = a.n or dn
    a.sites = a.sites or ds
    if not a.cpu_sample_sites:
        a.cpu_sample_sites = {"c4": 100_000, "c3": 60_000, "c5": 2_000}[a.workload]
    return a


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled through NVML every few ms DURING the timed region (B200_PROFILING.md)"""

    def __init__(self, index, period=0.004):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.sm, self.reasons, self.sm_max, self.power = [], 0, None, []
        self.stop_flag = threading.Event()
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def run(self):
        if self.h is None:
            return
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.reasons |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            self.stop_flag.wait(self.period)

    def finish(self):
        self.stop_flag.set()
        self.join()
        names = []
        if self.h is not None:
            nv = self.nv
            for nm, bit in (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                            ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap)):
                if self.reasons & bit:
                    names.append(nm)
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max, "reasons": names,
                "samples": len(self.sm), "power_w_max": max(self.power) if self.power else None}


def host_threads():
    """all host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which must not cap the CPU arm)"""
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------------------------
# CPU arms: the oracle port (C + OpenMP) and the pure-Python oracle, on a bounded sample of each workload
# ---------------------------------------------------------------------------------------------------------------------

class CpuSample:
    """one bounded sample of a workload for the CPU oracle: .run() is one pass, .bases its aligned bases, .text what it is"""

    def __init__(self, args):
        from oracle import c_oracle as co
        co.build()
        self.co, self.threads, self.wl = co, host_threads(), args.workload
        n, s = args.n, args.cpu_sample_sites
        if self.wl == "c4":
            self.mat = co.synth_text(SEED, n, args.sites, P_SEG_PPM, TRI_PPM, 0, s, threads=self.threads)
            self.bases = n * s
            self.text = "columns [0,%d) of the %d x %d alignment (%.1e bases)" % (s, n, args.sites, self.bases)
        elif self.wl == "c3":
            s = s // 3 * 3
            self.mat = co.synth_text(C3_SEED, n, args.sites, P_SEG_PPM, TRI_PPM, 0, s, threads=self.threads)
            self.pops = [list(range(n // 2)), list(range(n // 2, n))]
            self.bases = n * s
            self.text = "columns [0,%d) of the %d x %d CDS alignment, two populations, site + codon statistics (%.1e bases)" % (s, n, args.sites, self.bases)
        else:
            self.mats = [co.synth_text(C5_SEED + i, n, args.sites, P_SEG_PPM, TRI_PPM, 0, args.sites, threads=self.threads) for i in range(s)]
            self.bases = n * args.sites * s
            self.text = "loci [0,%d) of the %d loci of %d x %d (%.1e bases)" % (s, args.loci, n, args.sites, self.bases)

    def run(self):
        co, t = self.co, self.threads
        if self.wl == "c4":
            return co.site_stats(self.mat, threads=t)
        if self.wl == "c3":
            return [(co.site_stats(self.mat, rows, threads=t), co.cds_stats(self.mat, rows, threads=t)) for rows in self.pops]
        return [co.site_stats(m, threads=t) for m in self.mats]


def python_1core(args, seconds=4.0):
    """the pure-Python oracle (oracle/polyfasta_oracle.py: per-column loops over Python strings, the reference's speed class) on
    ONE core over a small slice of the workload -> dict for cpu_baseline.python_1core"""
    from oracle import c_oracle as co
    from oracle import polyfasta_oracle as orc
    n = args.n
    seed = {"c4": SEED, "c3": C3_SEED, "c5": C5_SEED}[args.workload]
    cols = min(args.sites, max(30, int(2.0e6 // n) // 3 * 3))
    mat = co.synth_text(seed, n, args.sites, P_SEG_PPM, TRI_PPM, 0, cols, threads=1)
    rows = [mat[i].tobytes().decode() for i in range(n)]
    t0 = time.perf_counter()
    passes = 0
    while passes < 1 or time.perf_counter() - t0 < seconds:
        orc.site_stats(rows, cols, want_sfs=True)
        if args.workload == "c3":
            orc.cds_stats(rows, cols)
        passes += 1
    dt = time.perf_counter() - t0
    return {"value": n * cols * passes / dt, "unit": "bases/s", "cores": 1,
            "sample": "columns [0,%d) x %d rows x %d passes, oracle/polyfasta_oracle.py (pure Python)" % (cols, n, passes)}


def workload_text(args):
    if args.workload == "c4":
        return "C4: synthetic non-coding alignment %d seqs x %d sites, site scan (S, H, folded SFS)" % (args.n, args.sites)
    if args.workload == "c3":
        return "C3: synthetic in-frame CDS alignment %d seqs x %d sites, two populations, --cds --jc (site scan + codon scan)" % (args.n, args.sites)
    return "C5: --dir batch of %d loci of %d seqs x %d sites, round-robin over the GPUs, no collective" % (args.loci, args.n, args.sites)


def run_reference(args, rank, print_json):
    """--impl reference: the CPU implementation of the path on the box's host cores; rank 0 only"""
    if rank != 0:
        return
    smp = CpuSample(args)
    for _ in range(args.warmup):
        smp.run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        smp.run()
    dt = time.perf_counter() - t0
    value = smp.bases * args.steps / dt
    sample_txt = smp.text + " per step, C+OpenMP oracle port"
    print_json({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "bases/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": workload_text(args), "sample": sample_txt},
        "cpu_baseline": {"value": value, "unit": "bases/s", "cores": smp.threads, "kind": "port", "sample": sample_txt},
        "e2e": {"value": value, "unit": "bases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference is pure Python (not on this box); its own functions ran at ~1e7 bases/s on one core in the build container (BASELINE.md)",
    })


def cpu_baseline(args):
    smp = CpuSample(args)
    smp.run()  # warm-up
    t0 = time.perf_counter()
    passes = 0
    while passes < 2 or time.perf_counter() - t0 < args.cpu_seconds:
        smp.run()
        passes += 1
    dt = time.perf_counter() - t0
    out = {"value": smp.bases * passes / dt, "unit": "bases/s", "cores": smp.threads, "kind": "port",
           "sample": "%s x %d passes, C+OpenMP oracle port (oracle/c)" % (smp.text, passes)}
    try:
        out["python_1core"] = python_1core(args)
    except Exception as e:   # the pure-Python figure is a courtesy line: never fail the bench for it
        out["python_1core"] = {"error": repr(e)}
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------------------------

class Env:
    """process-wide state of one rank: torch, the context on its stream, rank helpers"""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        import polyfasta_b200 as pf
        self.torch, self.dist, self.pf = torch, dist, pf
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.cpus = host_threads()
        if self.world > 1:
            from polyfasta_b200 import parallel
            parallel.bind_near_gpu(self.local_rank)   # pinned staging memory of this rank on the GPU's NUMA node
        self.ctx = pf.Context(self.local_rank)
        self.stream = torch.cuda.Stream()
        self.ctx.set_stream(self.stream.cuda_stream)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, x):
        if self.world == 1:
            return x
        t = self.torch.tensor([x], dtype=self.torch.float64, device="cuda")
        self.dist.all_reduce(t)
        return float(t.item())

    def shard(self, total, r=None):
        from polyfasta_b200 import parallel
        return parallel.shard_columns(total, self.world, self.rank if r is None else r)

    def timed_steps(self, args, step, fused_xchg=None):
        """W warm-up steps, then K timed ones between device events on the context's stream -> (elapsed ms, kernel ms, launches, clocks);
        step(ev) records ev[0] / ev[1] around its dominant kernel when ev is given"""
        torch, ctx, stream = self.torch, self.ctx, self.stream
        for _ in range(args.warmup):
            step(None)
        self.barrier()
        launches0 = ctx.launch_count
        sampler = ClockSampler(self.local_rank)
        sampler.start()
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if self.world > 1:
            # device-side rendezvous on the timing stream: the ranks leave the host barrier up to a millisecond apart, and
            # without it the first timed step of the early ranks would just measure that host skew
            sync_word = torch.zeros(1, dtype=torch.int64, device="cuda")
            if fused_xchg is not None:
                fused_xchg.allreduce(sync_word.data_ptr(), 1)
            else:
                self.dist.all_reduce(sync_word)
        t_start.record(stream)
        for i in range(args.steps):
            step(kev[i])
        t_end.record(stream)
        self.barrier()
        clocks = sampler.finish()
        launches = ctx.launch_count - launches0
        elapsed_ms = self.max_over_ranks(t_start.elapsed_time(t_end))
        try:
            kernel_ms = self.max_over_ranks(sum(a.elapsed_time(b) for a, b in kev) / args.steps)
        except Exception:   # the step times its kernels itself (c5)
            kernel_ms = None
        self.kev = kev
        return elapsed_ms, kernel_ms, launches, clocks


DUMP_LIMIT = 64 << 20


def dump_outputs(directory, arrays):
    """--dump-outputs: arrays {name: integer or float array} -> directory/<name>.npy in float64 (integers only where exact)"""
    import numpy as np
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        f = a.astype(np.float64)
        if a.dtype.kind in "iu" and not np.array_equal(f.astype(a.dtype), a):
            raise SystemExit("--dump-outputs: %s holds integers that float64 does not represent exactly" % name)
        out[name] = f
    total = sum(f.nbytes for f in out.values())
    if total > DUMP_LIMIT:
        raise SystemExit("--dump-outputs: %d bytes exceed the %d byte limit" % (total, DUMP_LIMIT))
    os.makedirs(directory, exist_ok=True)
    for name, f in out.items():
        np.save(os.path.join(directory, name + ".npy"), f)


def c5_outputs(args, env, batches):
    """the per-locus results of the last batched scan, gathered on rank 0 in locus order: every locus, or a fixed seeded sample
    of them where all would exceed DUMP_LIMIT"""
    import numpy as np
    half = args.n // 2
    cap = DUMP_LIMIT // (8 * (6 + half))
    pick = range(args.loci) if args.loci <= cap else np.random.default_rng(0).choice(args.loci, cap, replace=False).tolist()
    pick = set(pick)
    rows = []
    for bt, ids in batches:
        for j, i in enumerate(ids):
            if i in pick:
                r = bt.result(j, 0, want_sfs=True)
                _, pi, theta, d = r["poly"]
                rows.append((i, r["S"], r["H"], pi, theta, float("nan") if d == "NA" else d, r["sfs"]))
    if env.world > 1:
        got = [None] * env.world if env.rank == 0 else None
        env.dist.gather_object(rows, got, dst=0)
        rows = sorted((r for part in got for r in part), key=lambda r: r[0]) if env.rank == 0 else []
    col = lambda k: np.array([r[k] for r in rows])   # noqa: E731
    return {"locus": col(0), "S": col(1), "H": col(2), "sfs": np.array([r[6] for r in rows], dtype=np.int64).reshape(len(rows), half),
            "pi_site": col(3), "theta_site": col(4), "tajimas_d": col(5)}


def traffic_for(key):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu --set full capture of this shape, or None"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            t = json.load(f).get(key)
        return (t["dram_bytes_read"] + t["dram_bytes_write"]) if t else None
    except Exception:
        return None


def roofline(kernel, kernel_ms, algo_bytes, traffic, read_only_gbs=None):
    peak, peak_kind = measured_peak()
    achieved = algo_bytes / (kernel_ms * 1e-3) / 1e9
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
         "peak_kind": peak_kind, "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": algo_bytes}
    if read_only_gbs:
        r.update({"read_only_peak": read_only_gbs, "frac_of_read_only_peak": achieved / read_only_gbs,
                  "read_only_peak_kind": "pfa_read_probe_kernel over the same planes (padded bytes), measured in this run"})
    return r


def run_c4(args, env):
    torch, dist, pf, ctx, stream = env.torch, env.dist, env.pf, env.ctx, env.stream
    from polyfasta_b200 import api, parallel, synth
    rank, world = env.rank, env.world
    n, L = args.n, args.sites
    with torch.cuda.stream(stream):
        c0, c1 = env.shard(L)
        aln = pf.Alignment.synthetic(ctx, n, L, SEED, P_SEG_PPM, TRI_PPM, c0, c1)
        if args.gaps_ppm:
            aln.poke_gaps(SEED, args.gaps_ppm)
        if args.force_validity:
            aln.force_validity(True)
        whole_v = args.force_validity or os.environ.get("PFA_VFLAG") == "0"
        planes_read = 3 if (aln.has_invalid and (whole_v or not args.gaps_ppm)) else 2
        out = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
        fused = world > 1 and args.collective == "fused"
        xchg = parallel.connect_exchange(ctx, aln.site_len()) if fused else None
        ctx.sync()

        def step(ev):
            if ev:
                ev[0].record(stream)
            if fused:
                aln.site_stats_xchg(xchg, out.data_ptr())     # ONE launch: K2 + sum over the shards of all ranks
            else:
                aln.site_stats_device(out.data_ptr())
            if ev:
                ev[1].record(stream)
            if world > 1 and not fused:
                dist.all_reduce(out)

        elapsed_ms, kernel_ms, launches, clocks = env.timed_steps(args, step, xchg)
        kernel_name = ctx.last_kernel
        result = out.cpu().numpy().copy()
        if fused and xchg.timed_out():
            raise SystemExit("the NVLink exchange timed out on rank %d (a rank did not arrive)" % rank)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"site_stats": result})
        if os.environ.get("PFA_XCHG_STAMPS"):
            per = [a.elapsed_time(b) for a, b in env.kev]
            gaps = [env.kev[i][0].elapsed_time(env.kev[i + 1][0]) for i in range(args.steps - 1)]
            sys.stderr.write("rank %d kernel ms per step %s\nrank %d step-to-step ms %s\n" %
                             (rank, ["%.3f" % x for x in per], rank, ["%.3f" % x for x in gaps]))
            if fused:
                sys.stderr.write("rank %d exchange stages (ns): %s\n" % (rank, xchg.stamps()))

    value = n * L * args.steps / (elapsed_ms * 1e-3)
    my_sites = c1 - c0
    # algorithmic bytes: the two base planes, plus the validity plane when all of it has to be read; with sparse gaps only the
    # flagged 128-row pieces are needed -- they are left out of the algorithmic figure (an upper bound on the achieved rate)
    algo_bytes = n * my_sites * planes_read / 8.0
    traffic = traffic_for("C4 n=%d sites=%d gpus=%d planes=%d%s" % (n, L, world, planes_read, " gaps_ppm=%d" % args.gaps_ppm if args.gaps_ppm else ""))

    parity = "skipped"
    if rank == 0 and not args.no_check:
        if args.gaps_ppm == 0:
            want = synth.expected_site_stats(SEED, n, L, P_SEG_PPM, TRI_PPM)
            got = (int(result[0]), int(result[1]), [int(x) for x in result[2:]])
            if got != (want["S"], want["H"], want["sfs"]):
                raise SystemExit("PARITY FAILURE at full size: got S=%d H=%d, closed form S=%d H=%d" % (got[0], got[1], want["S"], want["H"]))
            parity = "S, H and the folded SFS of the %d x %d alignment equal the generator's closed form (S=%d)" % (n, L, want["S"])
    if args.gaps_ppm and not args.no_check:
        # no closed form with gaps: (a) the oracle on a column slice of the same gapped alignment, (b) the sparse-validity scan
        # against the same kernels reading the whole validity plane, on this rank's whole shard
        with torch.cuda.stream(stream):
            ref = torch.zeros_like(out)
            aln.force_validity(True)
            aln.site_stats_device(ref.data_ptr())
            aln.force_validity(False)
            mine = torch.zeros_like(out)
            aln.site_stats_device(mine.data_ptr())
            ctx.sync()
            if not torch.equal(ref, mine):
                raise SystemExit("PARITY FAILURE: sparse-validity scan != whole-plane scan on rank %d" % rank)
            if rank == 0:
                from oracle import c_oracle as co
                sl = min(2000, L)
                text = synth.poke_gaps(co.synth_text(SEED, n, L, P_SEG_PPM, TRI_PPM, 0, sl, threads=host_threads()), SEED, args.gaps_ppm)
                a2 = pf.Alignment.synthetic(ctx, n, L, SEED, P_SEG_PPM, TRI_PPM, 0, sl)
                a2.poke_gaps(SEED, args.gaps_ppm)
                got, want = a2.site_stats()[0], co.site_stats(text, threads=host_threads())
                a2.free()
                if (got["S"], got["H"], got["sfs"]) != (want["S"], want["H"], want["sfs"]):
                    raise SystemExit("PARITY FAILURE on the gapped slice against the oracle")
        parity = "gapped alignment: sparse-validity scan == whole-validity-plane scan on every shard; columns [0,%d) == C oracle" % min(2000, L)
    fin = ctx.finalize([(n, int(result[0]), int(result[1]), L, True)])[0]
    probe_ms = aln.read_probe(planes_read, 5)   # the read-only ceiling for exactly these bytes on this GPU (outside the timed region)
    read_only_gbs = aln.packed_bytes / 3 * planes_read / (probe_ms * 1e-3) / 1e9
    aln.free()
    ctx.trim()

    e2e = None
    if not args.no_e2e:
        with torch.cuda.stream(stream):
            es = min(args.e2e_sites, L)
            e0, e1 = env.shard(es)
            cols = e1 - e0
            ld = (cols + 255) // 256 * 256
            d_text = torch.empty((n, ld), dtype=torch.uint8, device="cuda")
            api.synth_text_device(ctx, d_text.data_ptr(), ld, n, SEED, P_SEG_PPM, TRI_PPM, e0, e1)
            ctx.sync()
            h_text = torch.empty((n, ld), dtype=torch.uint8, pin_memory=True)
            h_text.copy_(d_text)
            torch.cuda.synchronize()
            del d_text
            torch.cuda.empty_cache()
            h_out = torch.empty(out.numel(), dtype=torch.int64, pin_memory=True)
            ctx.set_host_threads(max(1, env.cpus // world))   # the ranks of one box share its cores

            def e2e_step():
                a = pf.Alignment.from_host_ptr(ctx, h_text.data_ptr(), n, cols, ld)   # H2D (pinned, chunked) + K1
                if fused:
                    a.site_stats_xchg(xchg, out.data_ptr())                          # K2 + sum over shards (NVLink)
                else:
                    a.site_stats_device(out.data_ptr())                              # K2
                    if world > 1:
                        dist.all_reduce(out)
                h_out.copy_(out, non_blocking=True)                                  # D2H
                stream.synchronize()
                r = ctx.finalize([(n, int(h_out[0]), int(h_out[1]), es, True)])[0]   # K5
                a.free()
                return r

            e2e_step()
            env.barrier()
            l0 = ctx.launch_count
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                r = e2e_step()
            env.barrier()
            dt = env.max_over_ranks(time.perf_counter() - t0)
            e2e_launches = (ctx.launch_count - l0) // args.e2e_steps
            if rank == 0 and not args.no_check:
                want = synth.expected_site_stats(SEED, n, L, P_SEG_PPM, TRI_PPM, 0, es)
                if (int(h_out[0]), int(h_out[1])) != (want["S"], want["H"]):
                    raise SystemExit("PARITY FAILURE in the end-to-end leg")
            ing = ctx.ingest_stats()   # the last step's upload on this rank (every rank's shard has the same shape)
            e2e = {"value": n * es * args.e2e_steps / dt, "unit": "bases/s",
                   "h2d_bytes_per_step": (ing["h2d_text_bytes"] + ing["h2d_packed_bytes"]) * world,
                   "d2h_bytes_per_step": (out.numel() * 8 + 32) * world, "ms_per_step": dt / args.e2e_steps * 1e3,
                   "sample": "columns [0,%d) of the workload as row-major text in pinned host memory (%.1e bases/step); "
                             "hybrid ingest (column chunks either as text over PCIe -> K1, or packed 4 bases/byte by host threads -> packed "
                             "K1) + K2 + sum over shards + D2H + K5 inside the timed region" % (es, n * es),
                   "gpu_launches_per_step": e2e_launches, "ingest": ing, "host_text_bytes_per_step": n * cols * world, "result": [r[0], r[1], r[2], r[3]]}

    cfg = {"workload": workload_text(args),
           "parallelism": ("columns split in %d contiguous ranges; " % world + ("the scan kernel's last block sums the int64 shard vectors "
                           "over NVLink peer memory (fused, no collective call)" if fused else "1 NCCL int64 all-reduce per step"))
           if world > 1 else "1 GPU",
           "l2": "inputs larger than L2 (%.1f GB of planes read per GPU per step)" % (algo_bytes / 1e9),
           "planes_read": planes_read, "seed": SEED, "p_seg_ppm": P_SEG_PPM, "tri_ppm": TRI_PPM}
    if args.gaps_ppm:
        cfg["gaps_ppm"] = args.gaps_ppm
        cfg["validity"] = "whole validity plane" if whole_v else "sparse: only flagged 128-row pieces of the validity plane are fetched"
    return {"value": value, "elapsed_ms": elapsed_ms, "scaling": "strong", "config": cfg,
            "roofline": roofline(kernel_name, kernel_ms, algo_bytes, traffic, read_only_gbs), "e2e": e2e, "launches": launches, "clocks": clocks,
            "parity": parity, "result": {"S": int(result[0]), "H": int(result[1]), "pi_site_jc": fin[1], "theta_site": fin[2], "tajimasD": fin[3]}}


def c3_rows(ctx, aln, site_vec, cds_vec, L, jc=True):
    """the --cds rows (as tuples) of both populations from the reduced vectors: K5 on the device"""
    import numpy as np
    from polyfasta_b200 import api
    site = aln.unpack_site(site_vec)
    raw = np.asarray(cds_vec).reshape(-1, api.PFA_CDS_LEN)
    ss = ctx.cds_ssites(raw)
    todo, rows = [], []
    for q, st in enumerate(site):
        c = aln.unpack_cds(raw[q])
        nsites = (L - c["missing"]) - float(ss[q])
        todo += [(st["n"], c["S_s"], c["H_s"], float(ss[q]), jc), (st["n"], c["S_n"], c["H_n"], nsites, jc)]
        rows.append((round(float(ss[q]), 2), round(nsites, 2), st["n"], c["nstops"]))
    fin = ctx.finalize(todo)
    return [rows[q] + fin[2 * q] + fin[2 * q + 1] for q in range(len(site))]


def run_c3(args, env):
    torch, dist, pf, ctx, stream = env.torch, env.dist, env.pf, env.ctx, env.stream
    from polyfasta_b200 import api, parallel
    import numpy as np
    rank, world = env.rank, env.world
    n, L = args.n, args.sites
    pops = [list(range(n // 2)), list(range(n // 2, n))]
    k = len(pops)
    with torch.cuda.stream(stream):
        c0, c1 = env.shard(L)
        aln = pf.Alignment.synthetic(ctx, n, L, C3_SEED, P_SEG_PPM, TRI_PPM, c0, c1)
        aln.set_pops(pops)
        d_site = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
        d_cds = torch.zeros(k * api.PFA_CDS_LEN, dtype=torch.int64, device="cuda")
        fused = world > 1 and args.collective == "fused"
        nsl = aln.site_len()
        xchg = parallel.connect_exchange(ctx, nsl + k * api.PFA_CDS_LEN) if fused else None
        d_both = torch.zeros(nsl + k * api.PFA_CDS_LEN, dtype=torch.int64, device="cuda")   # fused: [site vector | codon vectors]
        if fused:
            d_site, d_cds = d_both[:nsl], d_both[nsl:]
        ctx.sync()
        names = {}

        def step(ev):
            if fused:
                # ONE launch pair, ONE exchange: K2 leaves its shard vector in the exchange's buffer, K4's epilogue pushes both
                if ev:
                    ev[0].record(stream)
                aln.site_cds_stats_xchg(xchg, d_both.data_ptr())
                if ev:
                    ev[1].record(stream)
                return
            aln.site_stats_device(d_site.data_ptr())
            names["k2"] = ctx.last_kernel
            if ev:
                ev[0].record(stream)
            aln.cds_stats_device(d_cds.data_ptr())
            if ev:
                ev[1].record(stream)
            if world > 1:
                dist.all_reduce(d_site)
                dist.all_reduce(d_cds)

        elapsed_ms, kernel_ms, launches, clocks = env.timed_steps(args, step, xchg)
        names["k4"] = ctx.last_kernel
        site_vec, cds_vec = d_site.cpu().numpy().copy(), d_cds.cpu().numpy().copy()
        if fused and xchg.timed_out():
            raise SystemExit("the NVLink exchange timed out on rank %d" % rank)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"site_stats": site_vec, "cds_stats": cds_vec.reshape(k, api.PFA_CDS_LEN)})
    value = n * L * args.steps / (elapsed_ms * 1e-3)
    algo_bytes = n * (c1 - c0) * 2 / 8.0   # the codon scan reads the two base planes of the shard once (pure ACGT)
    if fused:
        algo_bytes *= 2                     # the timed pair is K2 + K4 (one exchange at the end): both read the two planes
    rows = c3_rows(ctx, aln, site_vec, cds_vec, L)
    parity = "skipped"
    if rank == 0 and not args.no_check:
        from oracle import c_oracle as co
        sl = min(args.cpu_sample_sites // 3 * 3, L)
        text = co.synth_text(C3_SEED, n, L, P_SEG_PPM, TRI_PPM, 0, sl, threads=host_threads())
        a2 = pf.Alignment.synthetic(ctx, n, L, C3_SEED, P_SEG_PPM, TRI_PPM, 0, sl)
        a2.set_pops(pops)
        gs, gc = a2.site_stats(), a2.cds_stats()
        a2.free()
        for q, r in enumerate(pops):
            ws, wc = co.site_stats(text, r, threads=host_threads()), co.cds_stats(text, r, threads=host_threads())
            if (gs[q]["S"], gs[q]["H"], gs[q]["sfs"]) != (ws["S"], ws["H"], ws["sfs"]) or any(gc[q][x] != wc[x] for x in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len")):
                raise SystemExit("PARITY FAILURE: C3 slice against the oracle, population %d" % q)
        parity = "columns [0,%d) of the workload, both populations: K2 and K4 (the same kernel instantiations) == C oracle, bit-exact" % sl
    probe_ms = aln.read_probe(2, 5)
    read_only_gbs = aln.packed_bytes / 3 * 2 / (probe_ms * 1e-3) / 1e9
    aln.free()
    ctx.trim()

    e2e = None
    if not args.no_e2e:
        with torch.cuda.stream(stream):
            cols = c1 - c0
            ld = (cols + 255) // 256 * 256
            d_text = torch.empty((n, ld), dtype=torch.uint8, device="cuda")
            api.synth_text_device(ctx, d_text.data_ptr(), ld, n, C3_SEED, P_SEG_PPM, TRI_PPM, c0, c1)
            ctx.sync()
            h_text = torch.empty((n, ld), dtype=torch.uint8, pin_memory=True)
            h_text.copy_(d_text)
            torch.cuda.synchronize()
            del d_text
            torch.cuda.empty_cache()
            h_site = torch.empty(d_site.numel(), dtype=torch.int64, pin_memory=True)
            h_cds = torch.empty(d_cds.numel(), dtype=torch.int64, pin_memory=True)
            ctx.set_host_threads(max(1, env.cpus // world))

            def e2e_step():
                a = pf.Alignment.from_host_ptr(ctx, h_text.data_ptr(), n, cols, ld)   # H2D (pinned, chunked) + K1 of this rank's columns
                a.set_pops(pops)
                if fused:
                    a.site_cds_stats_xchg(xchg, d_both.data_ptr())
                else:
                    a.site_stats_device(d_site.data_ptr())
                    a.cds_stats_device(d_cds.data_ptr())
                    if world > 1:
                        dist.all_reduce(d_site)
                        dist.all_reduce(d_cds)
                h_site.copy_(d_site, non_blocking=True)
                h_cds.copy_(d_cds, non_blocking=True)
                stream.synchronize()
                r = c3_rows(ctx, a, h_site.numpy(), h_cds.numpy(), L)
                a.free()
                return r

            e2e_step()
            env.barrier()
            l0 = ctx.launch_count
            t0 = time.perf_counter()
            for _ in range(args.e2e_steps):
                r = e2e_step()
            env.barrier()
            dt = env.max_over_ranks(time.perf_counter() - t0)
            if rank == 0 and not args.no_check and r != rows:
                raise SystemExit("PARITY FAILURE: end-to-end rows differ from the device-resident run")
            ing = ctx.ingest_stats()
            e2e = {"value": n * L * args.e2e_steps / dt, "unit": "bases/s",
                   "h2d_bytes_per_step": (ing["h2d_text_bytes"] + ing["h2d_packed_bytes"]) * world,
                   "d2h_bytes_per_step": (d_site.numel() + d_cds.numel()) * 8 * world, "ms_per_step": dt / args.e2e_steps * 1e3,
                   "sample": "the whole alignment as row-major text in pinned host memory (%.1e bases/step): hybrid ingest + K1 + K2 + K4 + sum over "
                             "shards + D2H + K5 rows of both populations inside the timed region" % (n * L),
                   "gpu_launches_per_step": (ctx.launch_count - l0) // args.e2e_steps, "ingest": ing, "host_text_bytes_per_step": n * cols * world}
    cfg = {"workload": workload_text(args),
           "parallelism": ("columns split codon-aligned in %d ranges; " % world + ("K2 and K4 each sum their int64 shard vectors over NVLink peer "
                           "memory in their last block" if fused else "2 NCCL int64 all-reduces per step")) if world > 1 else "1 GPU",
           "l2": "inputs larger than L2 (%.2f GB of planes read per GPU per scan, two scans per step)" % (algo_bytes / 1e9),
           "planes_read": 2, "seed": C3_SEED, "p_seg_ppm": P_SEG_PPM, "tri_ppm": TRI_PPM, "site_scan_kernel": names.get("k2")}
    return {"value": value, "elapsed_ms": elapsed_ms, "scaling": "strong", "config": cfg,
            "roofline": roofline(names["k4"] if not fused else "K2 + K4 back to back, one exchange: " + names["k4"], kernel_ms, algo_bytes, traffic_for("C3 n=%d sites=%d gpus=%d" % (n, L, world)), read_only_gbs),
            "e2e": e2e, "launches": launches, "clocks": clocks, "parity": parity,
            "result": {"rows": [list(r) for r in rows]}}


def run_c5(args, env):
    torch, dist, pf, ctx, stream = env.torch, env.dist, env.pf, env.ctx, env.stream
    from polyfasta_b200 import api, cli, parallel, synth
    rank, world = env.rank, env.world
    n, L, loci = args.n, args.sites, args.loci
    mine = [i for i in range(loci) if parallel.chunk_owner(i, world) == rank]   # locus i -> rank i mod world (SURVEY 8e.2)
    per_batch = int(os.environ.get("PFA_BENCH_BATCH", "10000"))
    batches = []
    with torch.cuda.stream(stream):
        for b0 in range(0, len(mine), per_batch):
            bt = api.Batch(ctx)
            for i in mine[b0:b0 + per_batch]:
                bt.add_synthetic(n, L, C5_SEED + i, P_SEG_PPM, TRI_PPM)
            bt.stage()                      # text generated on the device, encoded, dropped: the planes stay resident
            batches.append((bt, mine[b0:b0 + per_batch]))
        ctx.sync()
        ms_acc = []

        def step(ev):
            tot = 0.0
            for bt, _ in batches:
                bt.scan(jc=True)            # segmented K2b + K5b over the resident loci, results to the host, one sync
                tot += bt.kernel_ms()[0]
            ms_acc.append(tot)

        elapsed_ms, _, launches, clocks = env.timed_steps(args, step)
        # the segmented site kernel is timed inside the library (CUDA events around it, pfa_batch_kernel_ms)
        kernel_ms = env.max_over_ranks(sum(ms_acc[-args.steps:]) / args.steps)
        kernel_name = ctx.last_kernel or "pfa_batch_site_kernel"
        if args.dump_outputs:
            dumped = c5_outputs(args, env, batches)
            if rank == 0:
                dump_outputs(args.dump_outputs, dumped)
    my_bases = n * L * len(mine)
    value = n * L * loci * args.steps / (elapsed_ms * 1e-3)
    algo_bytes = my_bases * 2 / 8.0
    parity = "skipped"
    if not args.no_check:
        bad = 0
        for bt, ids in batches[:2]:
            for j in list(range(0, len(ids), max(1, len(ids) // 40)))[:50]:
                got = bt.result(j, 0, want_sfs=True)
                want = synth.expected_site_stats(C5_SEED + ids[j], n, L, P_SEG_PPM, TRI_PPM)
                bad += (got["S"], got["H"], got["sfs"]) != (want["S"], want["H"], want["sfs"])
        if env.sum_over_ranks(bad):
            raise SystemExit("PARITY FAILURE: batched loci differ from the generator's closed form")
        parity = "S, H and the folded SFS of ~100 loci per rank equal the generator's closed form"
    plane_bytes = sum(bt.shape()[1] for bt, _ in batches)
    first = batches[0][0].result(0, 0)
    for bt, _ in batches:
        bt.close()
    ctx.trim()

    e2e = None
    if not args.no_e2e:
        import shutil
        import tempfile
        import numpy as np
        e_loci = min(args.e2e_loci, loci)
        base = "/dev/shm" if os.path.isdir("/dev/shm") else None
        d = os.path.join(tempfile.gettempdir() if base is None else base, "pfa_bench_c5")
        my_files = [i for i in range(e_loci) if parallel.chunk_owner(i, world) == rank]
        if rank == 0:
            shutil.rmtree(d, ignore_errors=True)
            os.makedirs(d)
        env.barrier()
        ld = (L + 255) // 256 * 256
        heads = [(">indiv%d\n" % r).encode() for r in range(n)]
        with torch.cuda.stream(stream):
            buf = torch.empty((n, ld), dtype=torch.uint8, device="cuda")
            for i in my_files:               # every rank writes its own loci: one sequence per line, as the shipped examples
                api.synth_text_device(ctx, buf.data_ptr(), ld, n, C5_SEED + i, P_SEG_PPM, TRI_PPM, 0, L)
                ctx.sync()
                h = buf.cpu().numpy()
                with open(os.path.join(d, "locus%06d.fa" % i), "wb") as f:
                    f.write(b"".join(heads[r] + h[r, :L].tobytes() + b"\n" for r in range(n)))
            del buf
        env.barrier()
        paths = sorted(os.path.join(d, "locus%06d.fa" % i) for i in my_files)
        file_bytes = sum(os.path.getsize(p) for p in paths)

        class Collect:
            def __init__(self):
                self.rows = []

            def note(self, line):
                self.rows.append(line)

            def row(self, line, file, pop):
                self.rows.append(line)

        os.environ["POLYFASTA_DEVICES"] = str(env.local_rank)

        def e2e_step():
            sink = Collect()
            cli.run_files(paths, False, True, None, sink)      # the drop-in's --dir loop over this rank's loci
            if world > 1:
                got = [None] * world if rank == 0 else None
                dist.gather_object(sink.rows, got, dst=0)      # rows gathered on rank 0 (printed in sorted order there)
                return sum(len(x) for x in got) if rank == 0 else 0
            return len(sink.rows)

        e2e_step()
        env.barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            nrows = e2e_step()
        env.barrier()
        dt = env.max_over_ranks(time.perf_counter() - t0)
        if rank == 0 and nrows != e_loci:
            raise SystemExit("end-to-end leg: %d rows for %d loci" % (nrows, e_loci))
        env.barrier()
        if rank == 0:
            shutil.rmtree(d, ignore_errors=True)
        e2e = {"value": n * L * e_loci * args.e2e_steps / dt, "unit": "bases/s", "h2d_bytes_per_step": int(env.sum_over_ranks(len(my_files) * n * ((L + 31) // 32 * 32))),
               "d2h_bytes_per_step": e_loci * 64, "ms_per_step": dt / args.e2e_steps * 1e3, "us_per_locus": dt / args.e2e_steps / e_loci * 1e6,
               "sample": "loci [0,%d) of the workload as FASTA files in %s (%.1e bases/step, %.2f GB of files), locus i on rank i mod N: the drop-in's "
                         "--dir path (parallel read + parse + staging into pinned memory, one H2D + K1b + K2b + K5b per chunk of %d loci, rows "
                         "formatted, gathered on rank 0) inside the timed region" % (e_loci, d, n * L * e_loci, env.sum_over_ranks(file_bytes) / 1e9, cli.BATCH_FILES),
               "host_text_bytes_per_step": int(env.sum_over_ranks(file_bytes))}
    cfg = {"workload": workload_text(args), "parallelism": "locus i -> rank i mod %d, no collective; rows gathered on rank 0" % world if world > 1 else "1 GPU",
           "l2": "inputs larger than L2 (%.1f GB of planes resident per GPU, %.1f GB read per step)" % (3 * plane_bytes / 1e9, algo_bytes / 1e9),
           "loci_per_gpu": len(mine), "loci_per_resident_batch": per_batch, "planes_read": 2, "seed": "%d + locus" % C5_SEED,
           "record_layout": "n = 100 rows in 128-bit records: the planes hold 1.28 x the algorithmic bytes"}
    return {"value": value, "elapsed_ms": elapsed_ms, "scaling": "strong", "config": cfg,
            "roofline": roofline("%s (segmented over %d loci per launch)" % (kernel_name, per_batch), kernel_ms, algo_bytes,
                                 traffic_for("C5 n=%d sites=%d" % (n, L))),
            "e2e": e2e, "launches": launches, "clocks": clocks, "parity": parity,
            "result": {"locus0": {"S": first["S"], "H": first["H"], "poly": list(first["poly"])}}}


def main():
    args = parse_args()
    # rank 0 prints exactly ONE line on stdout; anything a library writes to fd 1 (NCCL's version banner) goes to stderr
    real_stdout = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    def print_json(obj):
        real_stdout.write(json.dumps(obj) + "\n")
        real_stdout.flush()

    if args.impl == "reference":
        run_reference(args, int(os.environ.get("RANK", "0")), print_json)
        return 0
    env = Env(args)
    res = {"c4": run_c4, "c3": run_c3, "c5": run_c5}[args.workload](args, env)
    cpu = None
    if env.rank == 0 and env.world == 1 and not args.no_cpu:
        cpu = cpu_baseline(args)
    if env.rank == 0:
        print_json({
            "metric": METRIC, "value": res["value"], "unit": "bases/s", "n_gpus": env.world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": res["elapsed_ms"] / args.steps, "higher_is_better": True, "scaling": res["scaling"],
            "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": res["config"], "roofline": res["roofline"],
            "cpu_baseline": cpu, "e2e": res["e2e"], "gpu_launches": res["launches"], "clocks": res["clocks"], "parity": res["parity"],
            "result": res["result"],
        })
    if env.world > 1:
        env.dist.barrier()
        env.dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
