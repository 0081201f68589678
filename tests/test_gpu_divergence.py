"""Divergence between populations on the GPU: D_xy per pair and per site against the C oracle, the identity with K3's n x n
matrix, escape-only columns, windows against the alignment cut to each window's columns, column shards, and the CLI's --dxy."""
import io
import os
from contextlib import redirect_stdout

import numpy as np
import pytest
import torch

import polyfasta_b200 as pf
from divergence_oracle import divergence, divergence_c, divergence_rows, finalize, pairs, pi_site
from oracle import c_oracle as co
from oracle import polyfasta_oracle as orc
from polyfasta_b200 import api, cli, parallel, synth
from test_gpu_parity import _random_text, _upper
from test_oracle_golden import close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _device_vec(aln, words, fill):
    buf = torch.full((max(words, 1),), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    fill(buf.data_ptr())
    aln.ctx.sync()
    return buf.cpu().numpy()[:words]


def _dsite(aln):
    """per-site Dxy of every pair: windows of one column ([P][L][2], the D half)"""
    P, L = len(api.pop_pairs(aln.num_pops)), aln.total_len
    v = _device_vec(aln, 2 * P * L, lambda d: aln.divergence_windows_device(1, 1, d))
    return v.reshape(P, L, 2)


def _check_against_oracle(aln, up, pops, what):
    got = aln.divergence()
    P = len(pairs(len(pops)))
    ds = _dsite(aln)
    dev = _device_vec(aln, P, aln.divergence_device)
    assert len(got) == P
    for p, (x, y) in enumerate(pairs(len(pops))):
        D, want_ds = divergence_c(up, pops[x], pops[y], per_site=True)
        g = got[p]
        assert (g["x"], g["y"], g["n_x"], g["n_y"]) == (x, y, len(pops[x]), len(pops[y])), what
        assert g["D"] == D == int(dev[p]), (what, p)
        assert np.array_equal(ds[p, :, 1], want_ds), (what, p)
        assert np.array_equal(ds[p, :, 0], (want_ds > 0).astype(np.int64)), (what, p)


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("n,L", [(100, 3000), (700, 2000), (2000, 1500), (10000, 400), (21000, 240)])
def test_divergence_against_c_oracle(ctx, n, L, p_junk, k):
    """the row counts that select the different K2 paths; overlapping populations; p_junk = 0.01 adds gaps / N / ? and IUPAC
    codes (three planes and the escape kernel)"""
    rng = np.random.default_rng(n * 31 + L + k)
    text = _random_text(rng, n, L, p_junk=p_junk)
    up = _upper(text)
    pops = [list(range(0, n // 2)), list(range(n // 3, n)), list(range(0, n, 3))][:k]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    _check_against_oracle(aln, up, pops, (n, L, p_junk, k))
    aln.free()


def test_divergence_many_pairs(ctx):
    """k = 40: 780 pairs, most of them beyond the lanes of a warp; random overlapping populations"""
    n, L, k = 1000, 300, 40
    rng = np.random.default_rng(40)
    text = _random_text(rng, n, L, p_junk=0.01)
    up = _upper(text)
    pops = [np.flatnonzero(rng.random(n) < rng.uniform(0.02, 0.3)).tolist() for _ in range(k)]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    got = aln.divergence()
    for p, (x, y) in enumerate(pairs(k)):
        assert got[p]["D"] == divergence_c(up, pops[x], pops[y]), (x, y)
    ds = _dsite(aln)
    for p in (0, 100, 779):
        x, y = pairs(k)[p]
        assert np.array_equal(ds[p, :, 1], divergence_c(up, pops[x], pops[y], per_site=True)[1])
    aln.set_pops([list(range(i, n, 65)) for i in range(65)])
    with pytest.raises(pf.PolyFastaError):
        aln.divergence()
    aln.set_pops([list(range(n))])
    with pytest.raises(pf.PolyFastaError):
        aln.divergence()
    aln.free()


def test_divergence_equals_pairwise_matrix(ctx):
    n, L = 2000, 1500
    rng = np.random.default_rng(2000)
    text = _random_text(rng, n, L, p_junk=0.01)
    pops = [list(range(0, 1200)), list(range(900, n)), list(range(0, n, 7))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    _, mat = aln.pairwise(want_matrix=True)
    got = aln.divergence()
    for p, (x, y) in enumerate(pairs(3)):
        assert got[p]["D"] == int(mat[np.ix_(pops[x], pops[y])].astype(np.int64).sum()), (x, y)
    aln.free()


def test_escape_only_columns(ctx):
    """columns where every row holds an IUPAC code and the codes differ, and columns where one population is all R and the
    other all Y: the planes show one class there, so the var-flags pass does not mark them"""
    n, L = 300, 64
    rng = np.random.default_rng(7)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, L)][None, :].repeat(n, axis=0).copy()
    codes = np.frombuffer(b"RYKMSWrykm", dtype=np.uint8)
    for c in range(0, 20):
        text[:, c] = codes[rng.integers(0, len(codes), n)]
    text[: n // 2, 20:30] = ord("R")
    text[n // 2:, 20:30] = ord("Y")
    text[:, 30:34] = ord("K")            # one code everywhere: no divergence
    text[5, 40] = ord("N")
    up = _upper(text)
    pops = [list(range(n // 2)), list(range(n // 2, n)), list(range(0, n, 5))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    _check_against_oracle(aln, up, pops, "escape")
    assert aln.divergence()[0]["D"] > (n // 2) ** 2 * 10 - 1
    aln.free()


@pytest.mark.parametrize("k", [2, 3])
def test_gap_heavy(ctx, k):
    seed, n, L = 77, 10000, 900
    text = synth.poke_gaps(synth.text_matrix(seed, n, L), seed, 100)
    pops = [list(range(0, 6000)), list(range(5000, n)), list(range(0, n, 2))][:k]
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.has_invalid
    aln.set_pops(pops)
    _check_against_oracle(aln, text, pops, ("gaps", k))
    aln.free()


def _check_fin(got, want):
    """(dxy, da, fst) within 1e-12 of the oracle; da = dxy - hw and fst = 1 - hw / dxy cancel, so their error is bounded by
    1e-12 of the terms, not of the difference (the style of check_poly)"""
    if any(isinstance(x, str) for x in tuple(got) + tuple(want)):
        assert [isinstance(x, str) and x for x in got] == [isinstance(x, str) and x for x in want], (got, want)
    if isinstance(want[0], str):
        return
    assert close(got[0], want[0]), (got, want)
    hw = want[0] - want[1]
    assert abs(got[1] - want[1]) <= 1e-12 * max(abs(want[0]), abs(hw)), (got, want)
    if not isinstance(want[2], str):
        assert abs(got[2] - want[2]) <= 1e-12 * max(1.0, abs(1.0 - want[2])), (got, want)


GRID = [(10, 10), (30, 10), (7, 3), (3, 7), (1, 1), (100, 50), (5000, 1), (250, 1000), (257, 64)]


@pytest.mark.parametrize("n,L", [(150, 1003), (2000, 700)])
def test_windows_against_oracle_slices(ctx, n, L):
    """step < W, step > W, W not dividing L, gcd(W, step) = 1, W larger than L; every window's D is the oracle's for the
    alignment cut to the window's columns, dxy / da / fst the oracle formulas of the window's sums"""
    rng = np.random.default_rng(n + 3 * L)
    text = _random_text(rng, n, L, p_var=0.1, p_junk=0.02)
    up = _upper(text)
    pops = [list(range(n)), list(range(1, n, 3)), list(range(n // 2, n))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    for W, step in GRID:
        for jc in (False, True):
            got = aln.divergence_windows(W, step, jc)
            assert len(got) == api.window_count(L, W, step), (W, step)
            for i, g in enumerate(got):
                a, b = i * step, min(i * step + W, L)
                assert (g["start"], g["end"], g["seqlen"]) == (a, b, b - a)
                cut = np.ascontiguousarray(up[:, a:b])
                pis = []
                for rows in pops:
                    o = co.site_stats(cut, rows, want_sfs=False)
                    pis.append(co.finalize(len(rows), o["S"], o["H"], b - a, jc)[1])
                for p, (x, y) in enumerate(pairs(3)):
                    D = divergence_c(cut, pops[x], pops[y])
                    e = g["pairs"][p]
                    assert (e["x"], e["y"], e["D"]) == (x, y, D), (W, step, a, p)
                    _check_fin((e["dxy"], e["da"], e["fst"]), finalize(len(pops[x]), len(pops[y]), D, b - a, pis[x], pis[y], jc))
    aln.free()


def test_whole_alignment_counts_against_python_oracle(ctx):
    """the Python oracle end to end (pi from the reference's restatement) on a small alignment, and D from the synchronous C
    entry point"""
    rng = np.random.default_rng(5)
    n, L = 24, 120
    text = _random_text(rng, n, L, p_var=0.2, p_junk=0.05)
    seqs = [bytes(r).decode("latin-1") for r in _upper(text)]
    pops = [list(range(0, 10)), list(range(8, 24)), [3]]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    for jc in (False, True):
        got = aln.divergence(jc)
        D = np.zeros(3, dtype=np.int64)
        api.check(api.lib().pfa_divergence(aln.handle, D.ctypes.data), ctx.handle)
        for p, (x, y) in enumerate(pairs(3)):
            rx, ry = [seqs[i] for i in pops[x]], [seqs[i] for i in pops[y]]
            Dw = divergence(rx, ry, L)
            px, py = pi_site(rx, L, jc), pi_site(ry, L, jc)
            want = finalize(len(rx), len(ry), Dw, L, px, py, jc)
            g = got[p]
            assert g["D"] == Dw == int(D[p])
            assert close(g["pi_x"], px) and close(g["pi_y"], py)
            _check_fin((g["dxy"], g["da"], g["fst"]), want)
    aln.free()


def test_identical_populations_and_empty_population(ctx):
    rng = np.random.default_rng(11)
    n, L = 50, 200
    text = _random_text(rng, n, L, p_junk=0.02)
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops([[0], [0], list(range(n))])
    got = aln.divergence()
    assert got[0]["D"] == 0 and got[0]["dxy"] == 0.0 and got[0]["fst"] == "NA"
    aln.set_pops([[], list(range(n))])
    got = aln.divergence()
    assert got[0]["D"] == 0 and (got[0]["dxy"], got[0]["da"], got[0]["fst"]) == ("NA", "NA", "NA")
    aln.free()


@pytest.mark.parametrize("world,L", [(2, 4099), (3, 4099), (8, 4099), (2, 5), (4, 10)])
def test_shards_add_up(world, L):
    """the shards' per-pair and window vectors sum to the whole alignment's, on the host and through the exchange"""
    rng = np.random.default_rng(500 + world + L)
    n = 260
    text = _random_text(rng, n, L, p_junk=0.02)
    pops = [list(range(n)), list(range(1, n, 3)), list(range(100, 200))]
    P = len(pairs(3))
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
        shards.append(a)
    jobs = [(P, lambda a, d: a.divergence_device(d))]
    for W, step in ((100, 100), (7, 3), (3, 7), (1000, 250), (4099, 4099), (2500, 5000)):
        jobs.append((2 * P * api.window_count(L, W, step), lambda a, d, W=W, step=step: a.divergence_windows_device(W, step, d)))
    for words, fill in jobs:
        want = _device_vec(whole, words, lambda d: fill(whole, d))
        bufs = [torch.full((max(words, 1),), -1, dtype=torch.int64, device="cuda") for _ in range(world)]
        torch.cuda.synchronize()
        for r in range(world):
            fill(shards[r], bufs[r].data_ptr())
        for c in ctxs:
            c.sync()
        assert np.array_equal(sum(b.cpu().numpy()[:words] for b in bufs), want), words
        for r in range(world):
            xs[r].allreduce(bufs[r].data_ptr(), words)
        for c in ctxs:
            c.sync()
        for r in range(world):
            assert np.array_equal(bufs[r].cpu().numpy()[:words], want), (words, r)
    assert not any(x.timed_out() for x in xs)
    for a in shards + [whole]:
        a.free()
    for x in xs:
        x.close()
    for c in ctxs:
        c.close()


# ---- CLI -------------------------------------------------------------------------------------------------------------------

EXAMPLES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "example_theta_0.01")


def _run_cli(argv):
    buf = io.StringIO()
    with redirect_stdout(buf):
        assert cli.main(argv) == 0
    return buf.getvalue()


def _write_fasta(path, heads, text):
    with open(path, "wb") as f:
        for h, row in zip(heads, text):
            f.write((">%s\n" % h).encode() + row.tobytes() + b"\n")


def _parse(path):
    with open(path, "rb") as f:
        heads, seqs = orc.parse_fasta(f.read().decode("latin-1"))
    return heads, seqs


@pytest.mark.parametrize("jc", [False, True])
def test_cli_dxy_examples(jc):
    keys = ["indiv1", "indiv2"]
    out = _run_cli(["-d", EXAMPLES, "-p", ",".join(keys), "--dxy"] + (["--jc"] if jc else []))
    lines = out.splitlines()
    assert lines[0] == cli.HEADER_DXY
    files = sorted(os.listdir(EXAMPLES))
    assert len(lines) == 1 + len(files)
    for line, name in zip(lines[1:], files):
        heads, seqs = _parse(os.path.join(EXAMPLES, name))
        pops = [orc.pop_rows(heads, key) for key in keys]
        assert [len(p) for p in pops] == [11, 2]
        D, dxy, da, fst = divergence_rows(seqs, pops, jc)[0]
        f = line.split(",")
        assert f[:6] == [name, str(len(seqs[0])), "indiv1", "indiv2", "11", "2"]
        _check_fin([x if x == "NA" else float(x) for x in f[6:]], (dxy, da, fst))


def test_cli_dxy_windows_match_cut_files(tmp_path):
    """--dxy --window W --step S rows are the --dxy rows of files holding only each window's columns; --out writes the same"""
    rng = np.random.default_rng(4243)
    n, L = 40, 257
    text = _random_text(rng, n, L, p_var=0.08, p_junk=0.02)
    text[:, 100:140] = text[0, 100:140]
    heads = ["pop%d_ind%d" % (i % 3, i) for i in range(n)]
    _write_fasta(tmp_path / "aln.fa", heads, text)
    for W, step in ((50, 50), (64, 20), (30, 45)):
        for extra in ([], ["--jc"]):
            argv = ["-f", str(tmp_path / "aln.fa"), "-p", "pop0,nobody,pop1,pop2", "--dxy", "--window", str(W), "--step", str(step)] + extra
            lines = _run_cli(argv).splitlines()
            assert lines[0] == cli.HEADER_DXY_WINDOWS
            assert lines[1] == "# Pop nobody string was not found in fasta headers."
            rows = lines[2:]
            want = []
            for i in range(api.window_count(L, W, step)):
                a, b = i * step, min(i * step + W, L)
                sub = tmp_path / ("w%d_%d_%d" % (W, step, i))
                sub.mkdir(exist_ok=True)
                _write_fasta(sub / "aln.fa", heads, text[:, a:b])
                ref = _run_cli(["-f", str(sub / "aln.fa"), "-s", "-p", "pop0,nobody,pop1,pop2", "--dxy"] + extra).splitlines()
                want.extend((a + 1, b, r) for r in ref if not r.startswith("#"))
            assert len(rows) == len(want) == 3 * api.window_count(L, W, step)
            for line, (a, b, ref) in zip(rows, want):
                f = line.split(",")
                assert (int(f[1]), int(f[2])) == (a, b)
                assert ",".join([f[0]] + f[3:]) == ref, (W, step, line, ref)
            outp = tmp_path / ("out%d_%d_%d.csv" % (W, step, len(extra)))
            _run_cli(argv + ["-o", str(outp), "-s"])
            assert open(outp).read().splitlines() == lines[1:]


def test_cli_dxy_fewer_than_two_populations(tmp_path):
    rng = np.random.default_rng(1)
    text = _random_text(rng, 10, 30, p_junk=0.0)
    _write_fasta(tmp_path / "a.fa", ["pop0_%d" % i for i in range(10)], text)
    lines = _run_cli(["-f", str(tmp_path / "a.fa"), "-p", "pop0,popX", "--dxy"]).splitlines()
    assert lines == [cli.HEADER_DXY, "# Pop popX string was not found in fasta headers.",
                     "# Fewer than two populations found in a.fa: no divergence rows."]


def test_cli_dxy_under_two_ranks(tmp_path):
    """--dxy under two ranks: a column-sharded large file and -d loci; rank 0 prints what one process prints"""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from test_gpu_xchg import _cli_worker, _free_port
    rng = np.random.default_rng(19)
    n, L = 60, 30001
    text = _random_text(rng, n, L, p_junk=0.002)
    d = tmp_path / "loci"
    d.mkdir()
    _write_fasta(d / "big.fa", ["pop%d_%d" % (i % 3, i) for i in range(n)], text)
    _write_fasta(d / "small.fa", ["pop%d_%d" % (i % 3, i) for i in range(20)], text[:20, :500])
    argvs = [["-f", str(d / "big.fa"), "--dxy", "-p", "pop0,pop1,none,pop2"],
             ["-f", str(d / "big.fa"), "--dxy", "--window", "1000", "--step", "700", "-p", "pop0,pop1,pop2", "--jc"],
             ["-d", str(d), "--dxy", "--window", "333", "-p", "pop0,pop2"]]
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
