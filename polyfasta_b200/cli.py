"""Drop-in command line of PolyFastA.py on top of the B200 library.

Flags, defaults, CSV columns, screen text, `#` data-error rows and exit codes follow the reference's main() and
print_result() (PolyFastA.py:13-225); all counting and the fp64 statistics run on the GPU.  `-p/--pops` implements
the semantics the reference intends (PolyFastA.py:123-134: header-substring match, one row per key in the given
order); the reference itself raises TypeError there under Python 3 (:126)."""
import argparse
import os
import sys

from . import api

DESCRIPTION = """
    Fast estimator of nucleotide diversity (theta_pi),
    Watterson's theta (theta_w), and Tajimas\'s D for coding and
    non-coding sequences\n"""

EPILOG = """

    It can also print a vector of the folded site frequency spectrum and
    correct theta_pi for multiple hits (jukes-cantor).

    Examples:
    python PolyFastA.py -f myAlignment.fas -p pop1,pop2
    \"-p pop1,pop2\" assumes that the alignment has sequences that are labeled:

    >pop1_ind1_XXX
    ATGC...
    >pop1_ind2_XXX
    ATGC...
    >pop2_ind1_XXX
    ATGC...
    >pop2_ind2_XXX

    Alignment is inframe cooding sequence:
    python PolyFastA.py -f myAlignment.fas -p pop1,pop2 --cds

    Want Jukes-Cantor corrected estimates for CDS:
    python PolyFastA.py -f myAlignment.fas -p pop1,pop2 --cds --jc

    FASTA files in directory:
    python PolyFastA.py -d myFastaDir/ --out allpoly.csv

    Read from pipe:
    python PolyFastA.py --pipe -p pop1,pop2

    The format is not strict but the identifier (e.g. pop1) needs to be somewhere in the header.\n"""

# (long, short, kwargs): the flag table of PolyFastA.py:51-77
FLAGS = [
    ("--file", "-f", dict(nargs="*", type=str, default="", help="one or several alignment files in FASTA format.")),
    ("--dir", "-d", dict(type=str, default=".", help="directory containing FASTA files only.")),
    ("--pops", "-p", dict(nargs="?", default=False, metavar="pop1,pop2,pop3", type=str,
                          help="split alignment by populations. A comma-separated list of strings that are found in the sequence headers.")),
    ("--out", "-o", dict(type=str, default="", help="name of output file. (default/empty will print to screen")),
    ("--pipe", "-i", dict(action="store_true", default=False, help="if FASTA file is being piped in from STDIN.")),
    ("--cds", "-c", dict(action="store_true", default=False,
                         help="the alignment is protein coding. Will split into synonymous and nonsynonymous sites.")),
    ("--silent", "-s", dict(action="store_true", default=False, help="suppress header and verbose output.")),
    ("--name", "-n", dict(type=str, default=False, help="name of the DNA region to show in output.")),
    ("--jc", None, dict(action="store_true", default=False, help="Jukes-Cantor correction for Pi.")),
]

HEADER_NONCDS = "file,seqlen,pop,N,seg_sites,pi,theta,tajimasD"
HEADER_WINDOWS = "file,window_start,window_end,seqlen,pop,N,seg_sites,pi,theta,tajimasD"
HEADER_DXY = "file,seqlen,pop1,pop2,N1,N2,dxy,da,Fst"
HEADER_DXY_WINDOWS = "file,window_start,window_end,seqlen,pop1,pop2,N1,N2,dxy,da,Fst"
HEADER_HAP = "file,seqlen,pop,N,haplotypes,Hd,Hd_var"
HEADER_HAP_WINDOWS = "file,window_start,window_end,seqlen,pop,N,haplotypes,Hd,Hd_var"
HEADER_CDS = ("file,sites_S,sites_N,pop,N,seg_sites_S,seg_sites_N,pi_S,pi_N,theta_S,theta_N,"
              "tajimasD_S,tajimasD_N,nstops")
HEADER_CDS_WINDOWS = ("file,window_start,window_end,sites_S,sites_N,pop,N,seg_sites_S,seg_sites_N,pi_S,pi_N,theta_S,theta_N,"
                      "tajimasD_S,tajimasD_N,nstops")


def build_parser():
    parser = argparse.ArgumentParser(prog="PolyFastA.py", formatter_class=argparse.RawTextHelpFormatter,
                                     description=DESCRIPTION, epilog=EPILOG)
    for long, short, kw in FLAGS:
        names = [long] if short is None else [long, short]
        parser.add_argument(*names, **kw)
    # beyond the reference: sliding windows along the alignment
    parser.add_argument("--window", type=int, default=None, metavar="W",
                        help="pi, theta and Tajima's D in windows of W alignment columns (one row per window and population;\n"
                             "window_start / window_end are 1-based and inclusive). With --cds: the synonymous and\n"
                             "nonsynonymous statistics per window; W and S must then be multiples of 3.")
    parser.add_argument("--step", type=int, default=None, metavar="S",
                        help="start a window every S columns (default: W). S > W skips the columns between windows.")
    # beyond the reference: divergence between populations
    parser.add_argument("--dxy", action="store_true", default=False,
                        help="d_xy, net divergence d_a and Hudson's F_ST between every pair of the -p populations (one row per\n"
                             "pair instead of the per-population rows; with --window, one row per window and pair). Not with --cds.")
    # beyond the reference: haplotype statistics
    parser.add_argument("--haplotypes", action="store_true", default=False,
                        help="number of distinct haplotypes (rows), Nei's haplotype diversity Hd and its variance per population\n"
                             "instead of the default statistics (with --window, per window). Not with --cds or --dxy.")
    return parser


def check_hap_args(parser, args):
    """the --haplotypes combinations that are errors"""
    if not args.haplotypes:
        return
    if args.cds:
        parser.error("--haplotypes does not work with --cds")
    if args.dxy:
        parser.error("--haplotypes does not work with --dxy")


def check_dxy_args(parser, args):
    """the --dxy combinations that are errors"""
    if not args.dxy:
        return
    if not args.pops:
        parser.error("--dxy needs -p/--pops")
    if args.cds:
        parser.error("--dxy does not work with --cds")


def check_window_args(parser, args):
    """the --window / --step combinations that are errors"""
    if args.step is not None and args.window is None:
        parser.error("--step needs --window")
    if args.window is None:
        return None
    step = args.window if args.step is None else args.step
    if args.window < 1 or step < 1:
        parser.error("--window and --step must be positive")
    if args.cds and (args.window % 3 or step % 3):
        parser.error("with --cds, --window and --step must be multiples of 3 (a window holds whole codons)")
    return args.window, step


class Sink:
    """where rows go: the screen, or --out (header truncates, everything else appends, plus the \\r progress text)"""

    def __init__(self, out, silent):
        self.out = out
        self.silent = silent

    def header(self, cds, windows=False, dxy=False, hap=False):
        if hap:
            line = HEADER_HAP_WINDOWS if windows else HEADER_HAP
        elif dxy:
            line = HEADER_DXY_WINDOWS if windows else HEADER_DXY
        else:
            line = (HEADER_CDS_WINDOWS if cds else HEADER_WINDOWS) if windows else HEADER_CDS if cds else HEADER_NONCDS
        if self.out:
            with open(self.out, "w") as o:
                o.write(line + "\n")
        else:
            print(line)

    def note(self, line):
        """`#` data-problem rows (PolyFastA.py:115-119,127-131,136-140)"""
        if self.out:
            with open(self.out, "a") as o:
                o.write(line + "\n")
        else:
            print(line)

    def row(self, line, file, pop):
        if self.out:
            with open(self.out, "a") as o:
                if not self.silent:
                    print("\r", f"Writting to {self.out}, pop: {pop:<10s}, parsing: {file:<15s}", end="", flush=True)
                o.write(line + "\n")
        else:
            print(line)


def poly_tail(S, poly):
    """the tail of a default or window row: S of the site scan, poly the tuple Context.finalize returns"""
    if S == 0:
        return ",0,0,0,NA"                                                                     # PolyFastA.py:187/:189
    return f",{poly[0]},{poly[1]},{poly[2]},{poly[3]}"                                         # :196/:198


def cds_tail(S, poly_s, poly_n, nstops):
    """the tail of a --cds or codon-window row: S of the site scan, poly_s / poly_n the synonymous / nonsynonymous tuples"""
    if S == 0:
        return ",0,0,0,NA,0,0,0,NA,0"                                                          # PolyFastA.py:160/:162
    s, m = poly_s, poly_n
    return f",{s[0]},{m[0]},{s[1]},{m[1]},{s[2]},{m[2]},{s[3]},{m[3]},{nstops}"                 # :178/:180


def format_rows(ctx, file, seqlen, cds, jc, pops, site, cdsst):
    """rows of print_result.no_header (PolyFastA.py:148-198) for the populations of one alignment.
    pops: list of (label, n); site: K2 results per population; cdsst: K4 results per population or None."""
    todo = []
    for q, (label, n) in enumerate(pops):
        if cds:
            c = cdsst[q]
            nsites = (seqlen - c["missing"]) - c["ssites"]
            if site[q]["S"]:
                todo.append((n, c["S_s"], c["H_s"], c["ssites"], jc))
                todo.append((n, c["S_n"], c["H_n"], nsites, jc))
        elif site[q]["S"]:
            todo.append((n, site[q]["S"], site[q]["H"], seqlen, jc))
    fin = iter(ctx.finalize(todo))
    lines = []
    for q, (label, n) in enumerate(pops):
        S = site[q]["S"]
        if cds:
            s, m = (next(fin), next(fin)) if S else (None, None)
            lines.append(cds_line(file, seqlen, label, n, S, cdsst[q], s, m))
        else:
            lines.append(f"{file},{seqlen},{label},{n}" + poly_tail(S, next(fin) if S else None))
    return lines


def window_rows(file, found, wins):
    """rows of one alignment in windows: wins = the list api.site_window_results returns.  Window by window, the populations in
    order; each row is the row format_rows gives for the window's columns alone, with the window's 1-based inclusive
    coordinates in front of seqlen (the window's length)."""
    return [f"{file},{w['start'] + 1},{w['end']},{w['seqlen']},{label},{n}" + poly_tail(p["S"], p["poly"])
            for w in wins for (label, _, n), p in zip(found, w["pops"])]


def cds_window_rows(file, found, wins):
    """--cds rows of one alignment in windows: wins = the list api.cds_window_results returns.  Window by window, the populations
    in order; each row is the --cds row format_rows gives for the window's columns alone, with the window's 1-based inclusive
    coordinates after the file's name"""
    lines = []
    for w in wins:
        for (label, _, n), p in zip(found, w["pops"]):
            c = p["cds"]
            head = f"{file},{w['start'] + 1},{w['end']},{round(c['ssites'], 2)},{round(c['nsites'], 2)},{label},{n}"
            lines.append(head + cds_tail(p["S"], p["poly_s"], p["poly_n"], c["nstops"]))
    return lines


def dxy_rows(file, found, wins, windowed):
    """--dxy rows of one alignment: wins = [dict(start, end, pairs=[dict(dxy, da, fst)])] (the list
    api.divergence_window_results returns, or the whole alignment's api.divergence_results as one window), start 0-based, end
    exclusive; the pairs in api.pop_pairs order.  windowed: the window's 1-based inclusive coordinates go in front of seqlen
    (the window's length)"""
    pairs = api.pop_pairs(len(found))
    lines = []
    for w in wins:
        start, end = w["start"], w["end"]
        head = f"{file},{start + 1},{end},{end - start}" if windowed else f"{file},{end - start}"
        for (x, y), d in zip(pairs, w["pairs"]):
            lines.append(head + f",{found[x][0]},{found[y][0]},{found[x][2]},{found[y][2]},{d['dxy']},{d['da']},{d['fst']}")
    return lines


def hap_rows(file, found, wins, windowed):
    """--haplotypes rows of one alignment: wins = the list api.haplotype_results returns (the whole alignment is one window).
    Window by window, the populations in order; windowed: the window's 1-based inclusive coordinates go in front of seqlen (the
    window's length)"""
    lines = []
    for w in wins:
        head = f"{file},{w['start'] + 1},{w['end']},{w['seqlen']}" if windowed else f"{file},{w['seqlen']}"
        for (label, _, n), p in zip(found, w["pops"]):
            lines.append(head + f",{label},{n},{p['h']},{p['Hd']},{p['Hd_var']}")
    return lines


class RankGroup:
    """the ranks of a torchrun launch (one process per GPU): rendezvous and row gathering go through torch.distributed
    (gloo, host plumbing only); the per-shard count vectors are summed inside the scan kernels over NVLink (api.Exchange)"""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.device = int(os.environ.get("LOCAL_RANK", str(self.rank)))
        self.host_cpus = os.cpu_count() or 1
        from . import parallel
        parallel.bind_near_gpu(self.device)
        if not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            dist.init_process_group("gloo", rank=self.rank, world_size=self.world)
        self.xchg = None
        # the in-kernel exchange maps every rank's buffer with CUDA IPC: one host, at most 16 ranks.  Anything else (several
        # nodes, more ranks) sums the small count vectors on the host through the rendezvous backend instead.
        import socket
        hosts = [None] * self.world
        dist.all_gather_object(hosts, socket.gethostname())
        self.fused = self.world <= 16 and len(set(hosts)) == 1 and os.environ.get("POLYFASTA_HOST_ALLREDUCE", "0") != "1"

    def parse_once(self, path, threads):
        """a large file every rank needs: rank 0 parses it with all host threads and hands the others the row layout (a few bytes
        per row); they map the file and adopt it.  Files that were not mapped in place are parsed by every rank."""
        blob = [None]
        fasta = None
        if self.rank == 0:
            fasta = api.parse_files([path], threads=max(threads, (os.cpu_count() or 1)))[0]
            blob = [fasta.export_layout() if isinstance(fasta, api.Fasta) else None]
        self.dist.broadcast_object_list(blob, src=0)
        if self.rank == 0:
            return fasta
        if blob[0] is None:
            return api.parse_files([path], threads=threads)[0]
        return api.Fasta.from_layout(path, blob[0])

    def exchange(self, ctx, words):
        """an exchange of at least `words` int64 (collective: every rank asks for the same size at the same point)"""
        from . import parallel
        if self.xchg is None or self.xchg.capacity < words:
            if self.xchg is not None:
                ctx.sync()
                self.dist.barrier()
                self.xchg.close()
            self.xchg = parallel.connect_exchange(ctx, max(words, 1 << 14))
        return self.xchg

    def close(self, ctx):
        if self.xchg is not None:
            ctx.sync()
            self.dist.barrier()
            self.xchg.close()
            self.xchg = None


XCHG_MAX_WORDS = 1 << 28   # the longest vector an exchange takes (pfa_xchg_create); longer window vectors go through the host


def sum_over_ranks(ctx, group, parts, fused=None):
    """parts: [(words, launch(d_ptr))], each launch writing this rank's int64 vector of `words` words into device memory;
    returns the sums over the ranks as host arrays, one per part.  The vectors travel in one exchange, or through the host
    collective when the group is not fused or they are longer than an exchange takes.  fused(xchg, d_ptr): one launch that
    computes every part and sums it over the ranks itself (the scan kernels' own exchange)."""
    import torch
    offs = [0]
    for n, _ in parts:
        offs.append(offs[-1] + n)
    words = max(offs[-1], 1)
    d_cnt = torch.zeros(words, dtype=torch.int64, device="cuda:%d" % ctx.device)
    d = d_cnt.data_ptr()

    def launch():
        for off, (_, part) in zip(offs, parts):
            part(d + 8 * off)

    torch.cuda.synchronize(ctx.device)
    if group.fused and words <= XCHG_MAX_WORDS:
        x = group.exchange(ctx, words)
        # the ranks meet on the host AFTER their uploads (parse + ingest times differ by seconds on cold files), so the wait
        # inside the kernels only has to cover launch skew
        ctx.sync()
        group.dist.barrier()
        if fused is not None:
            fused(x, d)
        else:
            launch()
            x.allreduce(d, words)
        ctx.sync()
        if x.timed_out():
            raise api.PolyFastaError(1, "a rank did not arrive at the exchange")
        h = d_cnt.cpu()
    else:
        launch()
        ctx.sync()
        h = d_cnt.cpu()
        group.dist.all_reduce(h)
    h = h.numpy()
    return [h[offs[i]:offs[i + 1]] for i in range(len(parts))]


BATCH_FILES = int(os.environ.get("POLYFASTA_BATCH_FILES", "512"))   # loci per batched GPU pass
SHARD_MIN_BYTES = int(os.environ.get("POLYFASTA_SHARD_MIN_BYTES", str(64 << 20)))   # files this large are column-sharded over the ranks
BATCH_BYTES = 1 << 30          # ... or this much text


def plan_populations(fasta, popkeys):
    """[(label, mask | None, rows)]: header-substring split (PolyFastA.py:123-125); no keys = one population 'NA'"""
    if popkeys is None:
        return [("NA", None, fasta.nseq)]
    plan = []
    for key in popkeys:
        mask, hits = api.match_mask(fasta, key)
        plan.append((key, mask, hits))
    return plan


def alignment_rows(ctx, fasta, file, cds, jc, found, window=None, dxy=False, group=None, hap=False):
    """rows of one alignment through the single-alignment kernels (large alignments, --cds, --window, --cds --window, --dxy and
    --haplotypes).  One process scans the whole alignment.  With `group`, every rank scans its codon-aligned column shard
    (SURVEY.md 8e.1), the integer vectors are summed over the ranks, and rank 0 finalises and formats them as one process does
    (the other ranks return None).  --haplotypes: the classes of the shards are not a sum; each rank writes its int32 rep array
    into its own slice of the vector and leaves the other slices zero, so the sum over the ranks gathers them, and rank 0 takes
    their meet (api.meet_classes)."""
    import numpy as np
    from functools import partial
    L, k = fasta.seqlen, len(found)
    sizes = [rows for _, _, rows in found]
    if group is None:
        aln = api.Alignment.from_fasta(ctx, fasta)
    else:
        from . import parallel
        aln = api.Alignment.from_fasta(ctx, fasta, *parallel.shard_columns(L, group.world, group.rank))
    try:
        if found[0][1] is not None:
            m = np.stack([mask for _, mask, _ in found])
            api.check(api.lib().pfa_aln_set_pops(aln.handle, m.ctypes.data, k), ctx.handle)
        P = len(api.pop_pairs(k))
        fused = None
        # (words, synchronous counts, asynchronous launch into device memory) of every vector the rows need
        if hap:
            W, step = window if window is not None else (max(L, 1), max(L, 1))
            nwin = api.window_count(L, W, step)
            half = (nwin * fasta.nseq + 1) // 2   # int64 words of one rank's slice
            rank, world = (0, 1) if group is None else (group.rank, group.world)
            parts = [(world * half, partial(aln.haplotype_classes, W, step),
                      lambda d: aln.haplotypes_device(W, step, d + 8 * half * rank))]
        elif window is None:
            parts = [(aln.site_len(), aln.site_counts, aln.site_stats_device)]
            if cds:   # K2 leaves its vector in the exchange's buffer, K4's epilogue pushes both: ONE exchange per alignment
                parts.append((k * api.PFA_CDS_LEN, aln.cds_counts, aln.cds_stats_device))
                fused = aln.site_cds_stats_xchg
            elif dxy:
                parts.append((P, aln.divergence_counts, aln.divergence_device))
            else:
                fused = aln.site_stats_xchg
        else:
            W, step = window
            nwin = api.window_count(L, W, step)
            if cds:
                parts = [(k * nwin * api.PFA_CDS_WIN_LEN, partial(aln.cds_window_counts, W, step), partial(aln.cds_windows_device, W, step))]
            else:
                parts = [(2 * k * nwin, partial(aln.site_window_counts, W, step), partial(aln.site_windows_device, W, step))]
            if dxy:
                parts.append((2 * P * nwin, partial(aln.divergence_window_counts, W, step), partial(aln.divergence_windows_device, W, step)))
        if group is None:
            vecs = [counts() for _, counts, _ in parts]
        else:
            vecs = sum_over_ranks(ctx, group, [(words, launch) for words, _, launch in parts], fused)
            if group.rank != 0:
                return None
        if hap:
            if group is None:
                reps = vecs
            else:
                reps = [vecs[0][r * half:(r + 1) * half].view(np.int32)[:nwin * fasta.nseq].reshape(nwin, fasta.nseq)
                        for r in range(group.world)]
            masks = None if found[0][1] is None else np.stack([mask for _, mask, _ in found])
            return hap_rows(file, found, api.haplotype_results(api.meet_classes(reps), masks, sizes, L, W, step), window is not None)
        if window is None:
            site = aln.unpack_site(vecs[0])
            if dxy:
                return dxy_rows(file, found, [{"start": 0, "end": L, "pairs": api.divergence_results(ctx, site, vecs[1], sizes, L, jc)}],
                                False)
            cdsst = api.cds_results(ctx, np.reshape(vecs[1], (k, api.PFA_CDS_LEN))) if cds else None
            return format_rows(ctx, file, L, cds, jc, [(label, rows) for label, _, rows in found], site, cdsst)
        if cds:
            wins = api.cds_window_results(ctx, np.reshape(vecs[0], (k, nwin, api.PFA_CDS_WIN_LEN)), sizes, L, W, step, jc)
            return cds_window_rows(file, found, wins)
        site = np.reshape(vecs[0], (k, nwin, 2))
        if dxy:
            wins = api.divergence_window_results(ctx, site, np.reshape(vecs[1], (P, nwin, 2)), sizes, L, W, step, jc)
            return dxy_rows(file, found, wins, True)
        return window_rows(file, found, api.site_window_results(ctx, site, sizes, L, W, step, jc))
    finally:
        aln.free()


def process_chunk(ctx, batch, items, cds, jc, popkeys, group=None, window=None, dxy=False, hap=False):
    """items: [(path, Fasta | exception)] in output order -> ordered actions ('stdout' | 'note' | 'row', ...).
    Small non-CDS loci of the chunk share ONE batched GPU pass; everything else goes through the single-alignment path.
    window = (W, step): every alignment goes through the single-alignment path (or the column shards of `group`) and gives
    its window rows after its '# Pop ... not found' notes.  dxy: the same, with one row per population pair (and window); a file
    with fewer than two populations found gives one more '#' note instead.  hap: the --haplotypes rows, through the same route."""
    actions = []
    pending = []   # (position in actions, locus, pop, file, seqlen, label, n)
    own_batch = None
    if batch is not None:
        batch.clear()
    for path, fasta in items:
        file = path.split("/")[-1]
        if isinstance(fasta, api.NotFasta):
            actions.append(("stdout", f"# file {path} is not FASTA!"))                         # PolyFastA.py:247
            continue
        if isinstance(fasta, Exception):
            actions.append(("raise", fasta))
            break
        if fasta.seqlen < 0:
            actions.append(("note", f"# Sequences do not have the same length: {file}"))        # :135-140
            continue
        if cds and fasta.seqlen % 3 != 0:
            actions.append(("note", f"# CDS sequence length is not a multiple of 3: {file}"))   # :114-119
        plan = plan_populations(fasta, popkeys)
        found = [p for p in plan if p[2] > 0]
        rows = iter(())
        if window is not None or dxy or hap:
            for label, mask, hits in plan:
                if hits == 0:
                    actions.append(("note", f"# Pop {label} string was not found in fasta headers."))   # :126-132
            if dxy and len(found) < 2:
                actions.append(("note", f"# Fewer than two populations found in {file}: no divergence rows."))
            elif found:
                lines = alignment_rows(ctx, fasta, file, cds, jc, found, window, dxy, group, hap)
                keys = ([f"{found[x][0]},{found[y][0]}" for x, y in api.pop_pairs(len(found))] if dxy
                        else [label for label, _, _ in found])
                for i, line in enumerate(lines or ()):
                    actions.append(("row", line, file, keys[i % len(keys)]))
            continue
        if found and (group is not None or cds or not api.Batch.fits(fasta)):
            rows = iter(alignment_rows(ctx, fasta, file, cds, jc, found, group=group) or [None] * len(found))
        elif found:
            import numpy as np
            masks = None if found[0][1] is None else np.stack([m for _, m, _ in found])
            if batch is None:   # a caller that expected only large alignments: stage the small one in a batch of our own
                batch = own_batch = api.Batch(ctx)
            locus = batch.add(fasta, masks)
        q = 0
        for label, mask, hits in plan:
            if hits == 0:
                actions.append(("note", f"# Pop {label} string was not found in fasta headers."))   # :126-132
            elif group is not None or cds or not api.Batch.fits(fasta):
                actions.append(("row", next(rows), file, label))
            else:
                pending.append((len(actions), locus, q, file, fasta.seqlen, label, hits))
                actions.append(None)
                q += 1
    if pending:
        batch.run(jc)
        for pos, locus, q, file, seqlen, label, n in pending:
            actions[pos] = ("row", noncds_line(file, seqlen, label, n, batch.result(locus, q)), file, label)
    for _, fasta in items:
        if isinstance(fasta, api.Fasta):
            fasta.close()
    if own_batch is not None:
        own_batch.close()
    return actions


def noncds_line(file, seqlen, label, n, r):
    """the default row of print_result.no_header (PolyFastA.py:187-198) from the batched results of one (locus, population)"""
    return f"{file},{seqlen},{label},{n}" + poly_tail(r["S"], r["poly"])


def cds_line(file, seqlen, label, n, S, c, poly_s, poly_n):
    """the --cds row of print_result.no_header (PolyFastA.py:160-180) of one population: S of the site scan, c its codon-scan
    results, poly_s / poly_n the synonymous / nonsynonymous tuples"""
    ssites = c["ssites"]
    nsites = (seqlen - c["missing"]) - ssites
    return f"{file},{round(ssites, 2)},{round(nsites, 2)},{label},{n}" + cds_tail(S, poly_s, poly_n, c["nstops"])


def process_chunk_native(ctx, batch, paths, jc, popkeys, threads, cds=False):
    """--dir chunk: ONE native call reads, parses, splits and stages every file (host threads), ONE batched GPU pass computes
    every (locus, population) -- the site scan and, with --cds, the codon scan -- then the rows are formatted in order"""
    from ._lib import PFA_BATCH_TOO_BIG, PFA_ERR_IO, PFA_ERR_NON_ASCII, PFA_ERR_NOT_FASTA, PFA_ERR_RAGGED, PFA_OK
    import time
    t0 = time.perf_counter()
    batch.clear()
    # files too large for the batched kernels skip the native staging (it would read and parse them only to refuse them)
    def _size(p):
        try:
            return os.path.getsize(p)
        except OSError:
            return 0
    big = [_size(p) > api.Batch.MAX_LOCUS_BYTES for p in paths]
    small_info = iter(batch.add_files([p for p, b in zip(paths, big) if not b], popkeys or (), threads))
    info = [{"status": PFA_BATCH_TOO_BIG} if b else next(small_info) for b in big]
    t1 = time.perf_counter()
    labels = popkeys if popkeys is not None else ["NA"]
    actions, pending = [], []
    for path, fi in zip(paths, info):
        file = path.split("/")[-1]
        st = fi["status"]
        if st == PFA_ERR_NOT_FASTA:
            actions.append(("stdout", f"# file {path} is not FASTA!"))
        elif st == PFA_ERR_IO:
            actions.append(("raise", OSError("cannot read %s" % path)))
            break
        elif st == PFA_ERR_NON_ASCII:
            actions.append(("raise", ValueError("%s: non-ASCII bytes in sequence lines are not supported" % path)))
            break
        elif st == PFA_ERR_RAGGED:
            actions.append(("note", f"# Sequences do not have the same length: {file}"))
        elif st == PFA_BATCH_TOO_BIG:
            actions.extend(process_chunk(ctx, None, [(path, api.parse_files([path], threads=threads)[0])], cds, jc, popkeys))
        elif st == PFA_OK:
            if cds and fi["L"] % 3 != 0:
                actions.append(("note", f"# CDS sequence length is not a multiple of 3: {file}"))   # :114-119
            q = 0
            for label, hits in zip(labels, fi["hits"]):
                if hits == 0:
                    actions.append(("note", f"# Pop {label} string was not found in fasta headers."))
                else:
                    pending.append((len(actions), fi["locus"], q, file, fi["L"], label, hits))
                    actions.append(None)
                    q += 1
        else:
            actions.append(("raise", api.PolyFastaError(st, "cannot process %s" % path)))
            break
    t2 = time.perf_counter()
    if pending:
        if os.environ.get("POLYFASTA_TIMING"):  # the three steps of Batch.run, timed one by one
            ta = time.perf_counter()
            batch.stage()
            tb = time.perf_counter()
            batch.scan(jc, cds)
            tc = time.perf_counter()
            batch.release()
            print("  gpu run: stage %.1f ms, scan %.1f ms, release %.1f ms" % ((tb - ta) * 1e3, (tc - tb) * 1e3, (time.perf_counter() - tc) * 1e3), file=sys.stderr)
        else:
            batch.run(jc, cds)
        t3 = time.perf_counter()
        for pos, locus, q, file, seqlen, label, n in pending:
            if cds:
                c = batch.result_cds(locus, q)
                line = cds_line(file, seqlen, label, n, batch.result(locus, q)["S"], c, c["poly_s"], c["poly_n"])
            else:
                line = noncds_line(file, seqlen, label, n, batch.result(locus, q))
            actions[pos] = ("row", line, file, label)
    else:
        t3 = t2
    if os.environ.get("POLYFASTA_TIMING"):
        print("chunk of %d files: add_files %.1f ms (%d threads), plan %.1f ms, gpu run %.1f ms, rows %.1f ms" %
              (len(paths), (t1 - t0) * 1e3, threads, (t2 - t1) * 1e3, (t3 - t2) * 1e3, (time.perf_counter() - t3) * 1e3), file=sys.stderr)
    return [a for a in actions if a is not None]


def emit(actions, sink):
    for a in actions:
        if a[0] == "stdout":
            print(a[1])
        elif a[0] == "note":
            sink.note(a[1])
        elif a[0] == "row":
            sink.row(a[1], a[2], a[3])
        elif a[0] == "raise":
            raise a[1]


def _file_size(p):
    try:
        return os.path.getsize(p)
    except OSError:
        return 0


def devices_from_env():
    """POLYFASTA_DEVICES=0,1,... (or POLYFASTA_DEVICE=0): the GPUs the --dir loci are spread over, round-robin by chunk"""
    spec = os.environ.get("POLYFASTA_DEVICES") or os.environ.get("POLYFASTA_DEVICE") or "0"
    return [int(x) for x in spec.split(",") if x.strip() != ""]


_SLOTS = {}


def run_files(paths, cds, jc, popkeys, sink, window=None, dxy=False, hap=False):
    """the per-file loop of PolyFastA.py:104-140 over sorted paths, in chunks; chunk i runs on device i mod G and the
    rows are emitted in the reference's order"""
    from concurrent.futures import ThreadPoolExecutor
    from . import parallel
    devs = devices_from_env()
    chunks = [ps for _, ps in parallel.plan_units(paths, [_file_size(p) for p in paths], None, BATCH_FILES, BATCH_BYTES)]
    if window is not None or dxy or hap:   # windows, divergence, haplotypes: file by file through the single-alignment path on the first listed device
        ctx = api.default_context(devs[0])
        for ps in chunks:
            emit(process_chunk(ctx, None, list(zip(ps, api.parse_files(ps))), cds, jc, popkeys, window=window, dxy=dxy, hap=hap), sink)
        return
    if len(chunks) > 1 and os.environ.get("POLYFASTA_DOUBLE_BUFFER", "1") != "0":
        devs = [d for d in devs for _ in (0, 1)]   # two slots per GPU: host staging of chunk i+1 overlaps the GPU pass of chunk i
    state = _SLOTS   # contexts and pinned staging buffers outlive one call (a process that runs several directories reuses them)

    def work(ci):
        slot = parallel.chunk_owner(ci, len(devs))   # one context + batch per listed device slot (a context is not re-entrant)
        key = (slot, devs[slot])
        if key not in state:
            ctx = api.Context(devs[slot])
            state[key] = (ctx, api.Batch(ctx))
        ctx, batch = state[key]
        threads = max(1, (os.cpu_count() or 1) // len(devs))
        return process_chunk_native(ctx, batch, chunks[ci], jc, popkeys, threads, cds)

    if len(devs) == 1 or len(chunks) == 1:
        for ci in range(len(chunks)):
            emit(work(ci), sink)
    else:
        # one worker thread per device (a context is not re-entrant); ctypes releases the GIL during library calls
        pools = [ThreadPoolExecutor(max_workers=1) for _ in devs]
        futs = [pools[parallel.chunk_owner(ci, len(devs))].submit(work, ci) for ci in range(len(chunks))]
        for f in futs:
            emit(f.result(), sink)
        for pl in pools:
            pl.shutdown()


def run_files_ranks(paths, cds, jc, popkeys, sink, group, window=None, dxy=False, hap=False):
    """the same loop under torchrun (one process per GPU).  Units in the reference's order: a file of at least
    SHARD_MIN_BYTES is ONE alignment scanned by ALL ranks in column shards (exchange fused into the kernels); the other
    files are grouped in chunks and chunk j goes to rank j mod world with no collective (SURVEY.md 8e.2).  Rank 0 gathers the
    finished rows and prints them in order."""
    from . import parallel
    ctx = api.Context(group.device)
    batch = api.Batch(ctx)
    threads = max(1, (os.cpu_count() or 1) // group.world)
    ctx.set_host_threads(threads)
    units = parallel.plan_units(paths, [_file_size(p) for p in paths], SHARD_MIN_BYTES, BATCH_FILES, BATCH_BYTES)
    mine, j = [], 0
    for ui, (kind, ps) in enumerate(units):
        if kind == "all":
            fasta = group.parse_once(ps[0], threads)
            acts = process_chunk(ctx, None, [(ps[0], fasta)], cds, jc, popkeys, group=group, window=window, dxy=dxy, hap=hap)
            if group.rank == 0:
                mine.append((ui, acts))
            continue
        if parallel.chunk_owner(j, group.world) == group.rank:
            if window is not None or dxy or hap:
                mine.append((ui, process_chunk(ctx, None, list(zip(ps, api.parse_files(ps, threads))), cds, jc, popkeys, window=window,
                                               dxy=dxy, hap=hap)))
            else:
                mine.append((ui, process_chunk_native(ctx, batch, ps, jc, popkeys, threads, cds)))
        j += 1
    group.close(ctx)
    gathered = parallel.gather_rows(mine)
    if group.rank == 0:
        for _, acts in gathered:
            emit(acts, sink)


def main(argv=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    window = check_window_args(parser, args)
    check_dxy_args(parser, args)
    check_hap_args(parser, args)
    if args.file == "" and args.dir == "." and not args.pipe:
        print("Both --file/-f and --dir/-d were not found.")
        r = input("Do you wish to run polySFS on all files in the current directory? [y|n]: ")
        if r != "y":
            parser.error(parser.print_help())
    if len(args.file) != 0 and args.dir != ".":
        parser.error("Run with either --file/-f or --dir/-d, but not both")
    elif len(args.file) == 0 and args.dir != ".":
        args.file = [args.dir + "/" + i for i in os.listdir(args.dir)]
    elif len(args.file) == 0 and args.dir == "." and args.pipe:
        args.file = [args.name] if args.name else ["stdin"]
    sink = Sink(args.out, args.silent)
    group = RankGroup() if int(os.environ.get("WORLD_SIZE", "1")) > 1 else None   # torchrun: one process per GPU
    if group is not None and group.rank != 0 and args.pipe:
        return 0   # stdin belongs to rank 0
    if group is not None and args.pipe:
        group = None
    if not args.silent and (group is None or group.rank == 0):
        sink.header(args.cds, window is not None, args.dxy, args.haplotypes)
    popkeys = args.pops.split(",") if args.pops else None
    paths = sorted(args.file)
    if paths and args.pipe:
        if not (args.file[0] == "stdin" or args.file[0] == args.name):
            parser.error("A FASTA file or multiple files cannot be used with the --pipe argument.")
        data = sys.stdin.buffer.read()
        ctx = api.default_context(devices_from_env()[0])
        batch = api.Batch(ctx)
        for path in paths:   # the reference reads stdin once per listed name; the second read is empty
            try:
                fasta = api.Fasta.from_bytes(data)
            except api.NotFasta as e:
                fasta = e
            emit(process_chunk(ctx, batch, [(path, fasta)], args.cds, args.jc, popkeys, window=window, dxy=args.dxy,
                               hap=args.haplotypes), sink)
            data = b""
    elif paths and group is not None:
        run_files_ranks(paths, args.cds, args.jc, popkeys, sink, group, window, args.dxy, args.haplotypes)
    elif paths:
        run_files(paths, args.cds, args.jc, popkeys, sink, window, args.dxy, args.haplotypes)
    if len(args.out) != 0 and not args.silent and (group is None or group.rank == 0):
        print("")
    return 0


if __name__ == "__main__":
    sys.exit(main())
