"""Per-site H out of the site scan (K2) and pi / theta / Tajima's D in sliding windows along the alignment.

The truth is the C oracle: per-site H from orc_site_stats, and every window's (S, H) is the oracle's result for the alignment
cut to the window's columns; pi / theta / D are K5 of those counts with seqlen = the window's length.  The CLI's window rows are
compared with the default CLI's rows for FASTA files that hold only the window's columns."""
import io
import os
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import polyfasta_b200 as pf
from polyfasta_b200 import api, cli, parallel, synth
from oracle import c_oracle as co
from test_gpu_parity import _random_text, _upper
from test_oracle_golden import check_poly

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _check_hsite(aln, up, pops, what):
    site = aln.site_stats(want_isvar=True, want_hsite=True)
    for q, rows in enumerate(pops):
        want = co.site_stats(up, rows, per_site=True)
        h = site[q]["hsite"]
        assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"]), (what, q)
        assert np.array_equal(h, want["hsite"]), (what, q)
        assert np.array_equal(site[q]["isvar"], (h > 0).astype(np.uint8)), (what, q)
        assert int(h.sum()) == want["H"] and int(np.count_nonzero(h)) == want["S"], (what, q)


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("n,L", [(100, 3000), (700, 2000), (2000, 1500), (10000, 400), (21000, 240)])
def test_hsite_against_c_oracle(ctx, n, L, p_junk):
    """every K2 path: TMA with narrow records (n = 100), the register kernel (700), TMA (2,000, 10,000), the streaming kernel
    (21,000); p_junk = 0.01 adds gaps / N / ? and IUPAC codes (the escape kernel)"""
    rng = np.random.default_rng(n * 7919 + L)
    text = _random_text(rng, n, L, p_junk=p_junk)
    up = _upper(text)
    aln = pf.Alignment.from_rows(ctx, text)
    for pops in ([list(range(n))], [list(range(n)), list(range(0, n, 2))], [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n))]):
        aln.set_pops(pops)
        _check_hsite(aln, up, pops, (n, L, p_junk, len(pops)))
    aln.free()


@pytest.mark.parametrize("n,L,k", [(2000, 1200, 6), (10000, 300, 20), (100, 2000, 40)])
def test_hsite_more_populations_than_lanes(ctx, n, L, k):
    """k larger than the lanes per site: the whole-warp second pass keeps those populations in shared memory"""
    rng = np.random.default_rng(k * 31 + n)
    for p_junk in (0.0, 0.01):
        text = _random_text(rng, n, L, p_junk=p_junk)
        aln = pf.Alignment.from_rows(ctx, text)
        pops = [list(range(q, n, q + 1)) for q in range(k)]
        aln.set_pops(pops)
        _check_hsite(aln, _upper(text), pops, (n, L, k, p_junk))
        aln.free()


@pytest.mark.parametrize("k", [1, 2, 3])
def test_hsite_gap_only_sites(ctx, k):
    """10,000 rows with 100 gaps per 10^6 bases: most variable sites are gap-only (valid rows show one base)"""
    seed, n, L = 99, 10000, 1200
    text = synth.poke_gaps(synth.text_matrix(seed, n, L), seed, 100)
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.has_invalid
    pops = [list(range(n)), list(range(0, n, 2)), list(range(100, 7000))][:k]
    aln.set_pops(pops)
    _check_hsite(aln, text, pops, k)
    aln.free()


GRID = [(10, 10), (30, 10), (7, 3), (3, 7), (1, 1), (100, 50), (5000, 1), (250, 1000)]


def _oracle_windows(up, pops, L, W, step, jc):
    out = []
    for i in range(api.window_count(L, W, step)):
        a, b = i * step, min(i * step + W, L)
        per = []
        for rows in pops:
            o = co.site_stats(np.ascontiguousarray(up[:, a:b]), rows, want_sfs=False)
            per.append((len(rows), o["S"], o["H"], co.finalize(len(rows), o["S"], o["H"], b - a, jc)))
        out.append((a, b, per))
    return out


@pytest.mark.parametrize("n,L", [(150, 1003), (2000, 700)])
def test_windows_against_oracle_slices(ctx, n, L):
    rng = np.random.default_rng(n + L)
    text = _random_text(rng, n, L, p_var=0.1, p_junk=0.02)
    up = _upper(text)
    pops = [list(range(n)), list(range(1, n, 3))]
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.num_escapes > 0 and aln.has_invalid
    aln.set_pops(pops)
    for W, step in GRID:
        for jc in (False, True):
            got = aln.site_windows(W, step, jc)
            want = _oracle_windows(up, pops, L, W, step, jc)
            assert len(got) == len(want) == api.window_count(L, W, step), (W, step)
            for g, (a, b, per) in zip(got, want):
                assert (g["start"], g["end"], g["seqlen"]) == (a, b, b - a)
                for p, (nq, S, H, poly) in zip(g["pops"], per):
                    assert (p["n"], p["S"], p["H"]) == (nq, S, H), (W, step, a)
                    check_poly(p["poly"], poly, nq, S, H)
    aln.free()


@pytest.mark.parametrize("W,step", [(12_001, 12_001), (5_000, 5_000), (6_144, 4_096), (4_100, 8_200), (9_000, 3_000)])
def test_large_windows_against_oracle_slices(ctx, W, step):
    """bins wider than one piece of the bin reduction (gcd(W, step) > 2,048 columns): several lane groups per bin add into it"""
    n, L = 300, 12_001
    rng = np.random.default_rng(W + step)
    text = _random_text(rng, n, L, p_junk=0.01)
    up = _upper(text)
    pops = [list(range(n)), list(range(0, n, 2))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    got = aln.site_windows(W, step)
    want = _oracle_windows(up, pops, L, W, step, False)
    assert len(got) == len(want)
    for g, (a, b, per) in zip(got, want):
        assert (g["start"], g["end"]) == (a, b)
        for p, (nq, S, H, poly) in zip(g["pops"], per):
            assert (p["S"], p["H"]) == (S, H), (W, step, a)
            check_poly(p["poly"], poly, nq, S, H)
    aln.free()


def _window_vec(aln, W, step):
    res = aln.site_windows(W, step)
    k = aln.num_pops
    return np.array([[[w["pops"][q]["S"], w["pops"][q]["H"]] for w in res] for q in range(k)], dtype=np.int64).reshape(-1)


@pytest.mark.parametrize("world,L", [(2, 4099), (3, 4099), (8, 4099), (2, 5), (4, 10), (8, 20)])
def test_window_shards_add_up(world, L):
    """the shards' partial vectors sum to the whole alignment's, on the host and through the exchange (ranks in one process)"""
    rng = np.random.default_rng(300 + world + L)
    n = 260
    text = _random_text(rng, n, L, p_junk=0.02)
    pops = [list(range(n)), list(range(1, n, 3))]
    ctxs = [pf.Context(0) for _ in range(world)]
    whole = pf.Alignment.from_rows(ctxs[0], text)
    whole.set_pops(pops)
    xs = [api.Exchange(c, 1 << 16) for c in ctxs]
    api.Exchange.connect_local(xs)
    shards = []
    for r in range(world):
        c0, c1 = parallel.shard_columns(L, world, r)
        a = pf.Alignment.from_rows(ctxs[r], text, c0, c1)
        a.set_pops(pops)
        assert a.total_len == L
        shards.append(a)
    for W, step in ((100, 100), (7, 3), (3, 7), (1000, 250), (4099, 4099), (2500, 5000)):
        want = _window_vec(whole, W, step)
        words = len(want)
        bufs = [torch.full((words,), -1, dtype=torch.int64, device="cuda") for _ in range(world)]
        torch.cuda.synchronize()
        for r in range(world):
            shards[r].site_windows_device(W, step, bufs[r].data_ptr())
        for c in ctxs:
            c.sync()
        parts = [b.cpu().numpy() for b in bufs]
        assert np.array_equal(sum(parts), want), (W, step)
        for r in range(world):
            xs[r].allreduce(bufs[r].data_ptr(), words)
        for c in ctxs:
            c.sync()
        for r in range(world):
            assert np.array_equal(bufs[r].cpu().numpy(), want), (W, step, r)
    assert not any(x.timed_out() for x in xs)
    for a in shards + [whole]:
        a.free()
    for x in xs:
        x.close()
    for c in ctxs:
        c.close()


def test_launch_plan_unchanged(ctx):
    """the per-site output changes neither the kernel choice nor the results of a plain scan"""
    for n, L, p_junk, k in ((10000, 600, 0.0, 1), (2000, 900, 0.01, 2), (700, 800, 0.01, 3), (21000, 100, 0.0, 2), (100, 900, 0.01, 2)):
        rng = np.random.default_rng(n + L)
        text = _random_text(rng, n, L, p_junk=p_junk)
        aln = pf.Alignment.from_rows(ctx, text)
        aln.set_pops([list(range(q, n, q + 1)) for q in range(k)])
        plain = aln.site_stats(want_isvar=True)
        kern = ctx.last_kernel
        aln.site_windows(50, 25)
        assert ctx.last_kernel == kern
        aln.site_stats(want_hsite=True)
        assert ctx.last_kernel == kern
        again = aln.site_stats(want_isvar=True)
        assert ctx.last_kernel == kern
        for a, b in zip(plain, again):
            assert (a["S"], a["H"], a["sfs"]) == (b["S"], b["H"], b["sfs"])
            assert np.array_equal(a["isvar"], b["isvar"])
        aln.free()


# ---- CLI -------------------------------------------------------------------------------------------------------------------

def _write_fasta(path, heads, text):
    with open(path, "wb") as f:
        for h, row in zip(heads, text):
            f.write((">%s\n" % h).encode() + row.tobytes() + b"\n")


def _run_cli(argv, stdin=None):
    buf = io.StringIO()
    old = sys.stdin
    try:
        if stdin is not None:
            sys.stdin = io.TextIOWrapper(io.BytesIO(stdin))
        with redirect_stdout(buf):
            assert cli.main(argv) == 0
    finally:
        sys.stdin = old
    return buf.getvalue()


@pytest.fixture(scope="module")
def cli_input(tmp_path_factory):
    d = tmp_path_factory.mktemp("win")
    rng = np.random.default_rng(4242)
    n, L = 40, 257
    text = _random_text(rng, n, L, p_var=0.08, p_junk=0.02)
    heads = ["pop%d_ind%d" % (i % 2, i) for i in range(n)]
    text[:, 100:140] = text[0, 100:140]   # a stretch without variation: windows with S = 0
    _write_fasta(d / "aln.fa", heads, text)
    return d, heads, text


def _window_reference(tmp, heads, text, W, step, extra):
    """the default CLI's rows (without the file's name) for FASTA files holding only each window's columns"""
    L = text.shape[1]
    rows = []
    for i in range(api.window_count(L, W, step)):
        a, b = i * step, min(i * step + W, L)
        sub = tmp / ("w%d_%d_%d" % (W, step, i))
        sub.mkdir(exist_ok=True)
        _write_fasta(sub / "aln.fa", heads, text[:, a:b])
        out = _run_cli(["-f", str(sub / "aln.fa"), "-s"] + extra)
        rows.extend((a + 1, b, line) for line in out.splitlines() if not line.startswith("#"))
    return rows


def _strip(line):
    f = line.split(",")
    return (int(f[1]), int(f[2])), ",".join([f[0]] + f[3:])


@pytest.mark.parametrize("extra", [[], ["-p", "pop1,nobody,pop0"], ["--jc"], ["-p", "pop0", "--jc"]])
def test_cli_windows_file_pipe_dir(cli_input, tmp_path, extra):
    d, heads, text = cli_input
    for W, step in ((50, 50), (64, 20), (30, 45)):
        want = _window_reference(tmp_path, heads, text, W, step, extra)
        out = _run_cli(["-f", str(d / "aln.fa"), "--window", str(W), "--step", str(step)] + extra)
        lines = out.splitlines()
        assert lines[0] == cli.HEADER_WINDOWS
        notes = [l for l in lines[1:] if l.startswith("#")]
        rows = [l for l in lines[1:] if not l.startswith("#")]
        assert lines[1: 1 + len(notes)] == notes   # notes first
        if "nobody" in extra:
            assert notes == ["# Pop nobody string was not found in fasta headers."]
        assert len(rows) == len(want)
        for line, (a, b, ref) in zip(rows, want):
            coords, rest = _strip(line)
            assert coords == (a, b) and rest == ref, (W, step, line, ref)
        # --pipe: the same rows under the name 'stdin'
        data = open(d / "aln.fa", "rb").read()
        piped = _run_cli(["--pipe", "-s", "--window", str(W), "--step", str(step)] + extra, stdin=data)
        assert piped.splitlines() == [l.replace("aln.fa,", "stdin,", 1) for l in lines[1:]]
        # -d: the files of the directory in sorted order, each through the single-alignment path
        dd = tmp_path / ("dir%d_%d" % (W, step))
        dd.mkdir()
        _write_fasta(dd / "a.fa", heads, text)
        _write_fasta(dd / "b.fa", heads[:20], text[:20, :199])
        got_d = _run_cli(["-d", str(dd), "-s", "--window", str(W), "--step", str(step)] + extra)
        want_d = (_run_cli(["-f", str(dd / "a.fa"), "-s", "--window", str(W), "--step", str(step)] + extra) +
                  _run_cli(["-f", str(dd / "b.fa"), "-s", "--window", str(W), "--step", str(step)] + extra))
        assert got_d == want_d


def test_cli_windows_out_file_and_errors(cli_input, tmp_path):
    d, _, _ = cli_input
    argv = ["-f", str(d / "aln.fa"), "--window", "40", "--step", "30", "-p", "pop0,pop1"]
    screen = _run_cli(argv)
    outp = tmp_path / "out.csv"
    _run_cli(argv + ["-o", str(outp)])
    assert open(outp).read() == screen
    with pytest.raises(SystemExit):
        cli.main(["-f", str(d / "aln.fa"), "--window", "40", "--cds"])


def test_cli_windows_without_window_unchanged(cli_input):
    """no --window: the default header and rows"""
    d, _, _ = cli_input
    out = _run_cli(["-f", str(d / "aln.fa"), "-p", "pop0,pop1"])
    assert out.splitlines()[0] == cli.HEADER_NONCDS and len(out.splitlines()) == 3


def test_cli_windows_under_two_ranks(tmp_path):
    """--window under two ranks: a column-sharded large file and -d loci; rank 0 prints what one process prints"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from test_gpu_xchg import _cli_worker, _free_port
    rng = np.random.default_rng(9)
    n, L = 60, 30001
    text = _random_text(rng, n, L, p_junk=0.002)
    d = tmp_path / "loci"
    d.mkdir()
    _write_fasta(d / "big.fa", ["pop%d_%d" % (i % 2, i) for i in range(n)], text)
    _write_fasta(d / "small.fa", ["pop%d_%d" % (i % 2, i) for i in range(20)], text[:20, :500])
    argvs = [["-f", str(d / "big.fa"), "--window", "1000", "--step", "700", "-p", "pop0,pop1,none"],
             ["-d", str(d), "--window", "333", "--jc"]]
    want = [_run_cli(a) for a in argvs]
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = _free_port()
    procs = [mpc.Process(target=_cli_worker, args=(r, 2, port, argvs, 1_000_000, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in range(2))
    for p in procs:
        p.join(60)
    assert got[0] == want
    assert all(o == "" for o in got[1])
