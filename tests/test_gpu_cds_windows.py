"""Synonymous and nonsynonymous statistics in sliding windows along a CDS alignment (pfa_cds_windows, --cds --window).

The truth for every window is the alignment cut to the window's columns: its 72-word vector must equal the C oracle's codon
vector plus the oracle's S of the cut, and the library's own cds_stats / site_stats of an alignment built from the cut text
(not a column shard: a shard's trailing partial column belongs to the last shard only).  pi / theta / D are K5 of those counts.
The CLI's window rows are compared with the --cds rows of FASTA files that hold only the window's columns."""
import io
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

WIN = api.PFA_CDS_WIN_LEN


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _oracle_vec(up, rows):
    """the 72 words of one population for the alignment `up` (already cut): the oracle's codon vector, then its S"""
    c = co.cds_stats(up, rows)
    v = [c["nstops"], c["missing"], c["S_s"], c["H_s"], c["S_n"], c["H_n"]] + [c["sum3_by_len"].get(l, 0) for l in range(65)]
    v.append(co.site_stats(up, rows, want_sfs=False)["S"])
    return np.array(v, dtype=np.int64), c


def _gpu_cut_vecs(ctx, text, pops):
    """the same words from the library: cds_stats + site_stats of an alignment built from the cut text alone"""
    a = pf.Alignment.from_rows(ctx, np.ascontiguousarray(text))
    a.set_pops(pops)
    cds, site = a.cds_stats(), a.site_stats()
    a.free()
    return [np.concatenate([c["raw"], [s["S"]]]).astype(np.int64) for c, s in zip(cds, site)]


def _check_windows(ctx, text, pops, grid, use_oracle=True, jc=False):
    up = _upper(text)
    L = text.shape[1]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    for W, step in grid:
        got = aln.cds_windows(W, step, jc)
        assert len(got) == api.window_count(L, W, step), (W, step)
        for i, g in enumerate(got):
            a, b = i * step, min(i * step + W, L)
            assert (g["start"], g["end"]) == (a, b)
            cut = np.ascontiguousarray(up[:, a:b])
            lib_vecs = _gpu_cut_vecs(ctx, text[:, a:b], pops)
            for q, rows in enumerate(pops):
                p = g["pops"][q]
                assert np.array_equal(p["cds"]["raw"], lib_vecs[q]), (W, step, i, q)
                assert p["S"] == lib_vecs[q][-1]
                if not use_oracle:
                    continue
                want, c = _oracle_vec(cut, rows)
                assert np.array_equal(p["cds"]["raw"], want), (W, step, i, q, p["cds"]["raw"] - want)
                n = len(rows)
                assert p["cds"]["ssites"] == pytest.approx(c["ssites"], rel=1e-12, abs=1e-12)
                check_poly(p["poly_s"], co.finalize(n, c["S_s"], c["H_s"], c["ssites"], jc), n, c["S_s"], c["H_s"])
                check_poly(p["poly_n"], co.finalize(n, c["S_n"], c["H_n"], c["nsites"], jc), n, c["S_n"], c["H_n"])
    aln.free()


def _pops(n, k):
    return [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n)), list(range(1, n, 3)), list(range(0, n // 2))][:k]


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("k", [1, 2, 5])
@pytest.mark.parametrize("L", [600, 601, 602])
def test_windows_against_cut_alignments(ctx, L, k, p_junk):
    """S < W, S = W, S > W, W >= L, and L % 3 = 0, 1, 2 (the trailing partial codon column is missing data of the last window)"""
    n = 150
    rng = np.random.default_rng(L * 10 + k + int(p_junk * 1000))
    text = _random_text(rng, n, L, p_var=0.08, p_junk=p_junk)
    grid = [(90, 30), (99, 99), (30, 60), (3, 3), (600, 300), (900, 3), (603, 603), (12, 9)]
    _check_windows(ctx, text, _pops(n, k), grid, jc=(L % 2 == 1))


@pytest.mark.parametrize("n,L", [(100, 903), (700, 601), (2000, 450), (13000, 152)])
def test_windows_row_count_paths(ctx, n, L):
    """every K2 / K4 kernel: TMA with narrow records (100), the register kernels (700), TMA (2,000), and beyond K4's TMA limit
    of 12,288 rows the streaming codon scan (13,000); with junk, so the validity plane and the escape kernels take part"""
    rng = np.random.default_rng(n + L)
    text = _random_text(rng, n, L, p_junk=0.01)
    grid = [(150, 75), (L - L % 3, 3 * (L // 6)), (3000, 3000)]
    _check_windows(ctx, text, _pops(n, 2), grid, use_oracle=n <= 2000)


@pytest.mark.parametrize("k", [1, 3])
def test_windows_sparse_gaps(ctx, k):
    """10,000 rows with 100 gaps per 10^6 bases (poke_gaps): most columns have no flagged validity cell and take the fast path"""
    seed, n, L = 77, 10000, 602
    text = synth.poke_gaps(synth.text_matrix(seed, n, L), seed, 100)
    _check_windows(ctx, text, [list(range(n)), list(range(0, n, 2)), list(range(100, 7000))][:k], [(60, 30), (300, 300)],
                   use_oracle=False)


def test_large_bins_cut_into_pieces(ctx):
    """bins much wider than one piece: many warps add into one bin"""
    n, L = 64, 30_002
    rng = np.random.default_rng(5)
    text = _random_text(rng, n, L, p_junk=0.005)
    _check_windows(ctx, text, _pops(n, 2), [(9_000, 6_000), (30_000, 15_000)], use_oracle=True)


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
def test_invariants(ctx, p_junk):
    """S = W: the windows add up to the whole alignment's codon vector and S; H_s and H_n are the per-site H at the labels"""
    n, L = 400, 3001
    rng = np.random.default_rng(11)
    text = _random_text(rng, n, L, p_junk=p_junk)
    pops = _pops(n, 3)
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    cds = aln.cds_stats(want_labels=True)
    site = aln.site_stats(want_hsite=True)
    for W in (3, 300, 999, 3003):
        wins = aln.cds_windows(W)
        for q in range(len(pops)):
            tot = sum(w["pops"][q]["cds"]["raw"] for w in wins)
            assert np.array_equal(tot[:api.PFA_CDS_LEN], cds[q]["raw"]), (W, q)
            assert tot[api.PFA_CDS_LEN] == site[q]["S"]
    for q in range(len(pops)):
        lab, h = cds[q]["labels"], site[q]["hsite"]
        assert int(h[lab == 1].sum()) == cds[q]["H_s"] and int(np.count_nonzero(lab == 1)) == cds[q]["S_s"]
        assert int(h[lab == 2].sum()) == cds[q]["H_n"] and int(np.count_nonzero(lab == 2)) == cds[q]["S_n"]
    aln.free()


def test_column_shards_add_up(ctx):
    """two codon-aligned column shards in one process: their device vectors add up to the unsharded vector"""
    n, L = 260, 4001
    rng = np.random.default_rng(3)
    text = _random_text(rng, n, L, p_junk=0.02)
    pops = _pops(n, 2)
    whole = pf.Alignment.from_rows(ctx, text)
    whole.set_pops(pops)
    shards = []
    for r in range(2):
        c0, c1 = parallel.shard_columns(L, 2, r)
        a = pf.Alignment.from_rows(ctx, text, c0, c1)
        a.set_pops(pops)
        shards.append(a)
    for W, step in ((300, 300), (99, 33), (33, 99), (4002, 4002), (3, 3)):
        nwin = api.window_count(L, W, step)
        want = np.stack([np.stack([w["pops"][q]["cds"]["raw"] for w in whole.cds_windows(W, step)]) for q in range(2)]).reshape(-1)
        bufs = [torch.full((len(want),), -1, dtype=torch.int64, device="cuda") for _ in range(2)]
        torch.cuda.synchronize()
        for a, b in zip(shards, bufs):
            a.cds_windows_device(W, step, b.data_ptr())
        ctx.sync()
        assert len(want) == 2 * nwin * WIN
        assert np.array_equal(bufs[0].cpu().numpy() + bufs[1].cpu().numpy(), want), (W, step)
    # a shard that does not start on a codon boundary, and windows that are not whole codons, are refused
    odd = pf.Alignment.from_rows(ctx, text, 1000, L)
    with pytest.raises(api.PolyFastaError):
        odd.cds_windows_device(300, 300, bufs[0].data_ptr())
    with pytest.raises(ValueError):
        whole.cds_windows(100, 99)
    with pytest.raises(api.PolyFastaError):
        whole.cds_windows_device(100, 100, bufs[0].data_ptr())
    for a in shards + [whole, odd]:
        a.free()


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
    d = tmp_path_factory.mktemp("cdswin")
    rng = np.random.default_rng(4243)
    n, L = 40, 259   # L % 3 = 1: the file's note, and a partial codon column in the last window
    text = _random_text(rng, n, L, p_var=0.08, p_junk=0.02)
    heads = ["pop%d_ind%d" % (i % 2, i) for i in range(n)]
    text[:, 99:141] = text[0, 99:141]   # a stretch without variation: windows with S = 0
    _write_fasta(d / "aln.fa", heads, text)
    return d, heads, text


def _cds_window_reference(tmp, heads, text, W, step, extra):
    """the --cds rows (without the file's name) for FASTA files holding only each window's columns"""
    L = text.shape[1]
    rows = []
    for i in range(api.window_count(L, W, step)):
        a, b = i * step, min(i * step + W, L)
        sub = tmp / ("w%d_%d_%d" % (W, step, i))
        sub.mkdir(exist_ok=True)
        _write_fasta(sub / "aln.fa", heads, text[:, a:b])
        out = _run_cli(["-f", str(sub / "aln.fa"), "-s", "--cds"] + extra)
        rows.extend((a + 1, b, line) for line in out.splitlines() if not line.startswith("#"))
    return rows


def _strip(line):
    f = line.split(",")
    return (int(f[1]), int(f[2])), ",".join([f[0]] + f[3:])


@pytest.mark.parametrize("extra", [[], ["-p", "pop1,nobody,pop0"], ["--jc"]])
def test_cli_cds_windows_file_pipe_dir(cli_input, tmp_path, extra):
    d, heads, text = cli_input
    for W, step in ((51, 51), (60, 21), (30, 45)):
        want = _cds_window_reference(tmp_path, heads, text, W, step, extra)
        out = _run_cli(["-f", str(d / "aln.fa"), "--cds", "--window", str(W), "--step", str(step)] + extra)
        lines = out.splitlines()
        assert lines[0] == cli.HEADER_CDS_WINDOWS
        notes = [l for l in lines[1:] if l.startswith("#")]
        rows = [l for l in lines[1:] if not l.startswith("#")]
        assert lines[1: 1 + len(notes)] == notes   # notes first
        assert notes[0] == "# CDS sequence length is not a multiple of 3: aln.fa"
        if "nobody" in extra:
            assert notes[1:] == ["# Pop nobody string was not found in fasta headers."]
        assert len(rows) == len(want)
        for line, (a, b, ref) in zip(rows, want):
            coords, rest = _strip(line)
            assert coords == (a, b) and rest == ref, (W, step, line, ref)
        data = open(d / "aln.fa", "rb").read()
        piped = _run_cli(["--pipe", "-s", "--cds", "--window", str(W), "--step", str(step)] + extra, stdin=data)
        assert piped.splitlines() == [l.replace("aln.fa", "stdin") for l in lines[1:]]
        dd = tmp_path / ("dir%d_%d" % (W, step))
        dd.mkdir()
        _write_fasta(dd / "a.fa", heads, text)
        _write_fasta(dd / "b.fa", heads[:20], text[:20, :198])
        argv = ["-s", "--cds", "--window", str(W), "--step", str(step)] + extra
        got_d = _run_cli(["-d", str(dd)] + argv)
        assert got_d == _run_cli(["-f", str(dd / "a.fa")] + argv) + _run_cli(["-f", str(dd / "b.fa")] + argv)
        assert _run_cli(["-f", str(dd / "a.fa"), str(dd / "b.fa")] + argv) == got_d


def test_cli_cds_windows_out_file_and_errors(cli_input, tmp_path, capsys):
    d, _, _ = cli_input
    argv = ["-f", str(d / "aln.fa"), "--cds", "--window", "42", "--step", "30", "-p", "pop0,pop1"]
    screen = _run_cli(argv)
    outp = tmp_path / "out.csv"
    _run_cli(argv + ["-o", str(outp)])
    assert open(outp).read() == screen
    for bad in (["--window", "40"], ["--window", "42", "--step", "20"]):
        with pytest.raises(SystemExit) as e:
            cli.main(["-f", str(d / "aln.fa"), "--cds"] + bad)
        assert e.value.code == 2
    with pytest.raises(SystemExit) as e:
        cli.main(["-f", str(d / "aln.fa"), "--cds", "--dxy", "-p", "pop0,pop1"])
    assert e.value.code == 2


def test_cli_cds_without_window_unchanged(cli_input):
    """plain --cds: the CDS header and one row per population, the rows format_rows gives for the whole-alignment results"""
    d, heads, text = cli_input
    out = _run_cli(["-f", str(d / "aln.fa"), "--cds", "-p", "pop0,pop1"])
    lines = out.splitlines()
    assert lines[0] == cli.HEADER_CDS and lines[1].startswith("#") and len(lines) == 4
    # the single window that covers everything carries the same row after its coordinates
    win = _run_cli(["-f", str(d / "aln.fa"), "--cds", "-s", "--window", "300", "-p", "pop0,pop1"]).splitlines()
    assert [_strip(l)[1] for l in win if not l.startswith("#")] == lines[2:]


def test_cli_cds_windows_under_two_ranks(tmp_path):
    """--cds --window under two ranks: a column-sharded large file and -d loci; rank 0 prints what one process prints"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from test_gpu_xchg import _cli_worker, _free_port
    rng = np.random.default_rng(19)
    n, L = 60, 30001
    text = _random_text(rng, n, L, p_junk=0.002)
    d = tmp_path / "loci"
    d.mkdir()
    _write_fasta(d / "big.fa", ["pop%d_%d" % (i % 2, i) for i in range(n)], text)
    _write_fasta(d / "small.fa", ["pop%d_%d" % (i % 2, i) for i in range(20)], text[:20, :500])
    argvs = [["-f", str(d / "big.fa"), "--cds", "--window", "999", "--step", "702", "-p", "pop0,pop1,none"],
             ["-d", str(d), "--cds", "--window", "333", "--jc"]]
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
