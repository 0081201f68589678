"""Haplotype classes on the GPU: rep against the oracle bit for bit over row counts, alphabets and hand-made differences,
windows against the alignment cut to each window's columns, the identity with K3's matrix, a hash collision reached by data,
column shards through meet_classes, and the CLI's --haplotypes."""
import io
import os

import numpy as np
import pytest

import haplotype_oracle as ho
import polyfasta_b200 as pf
from oracle import polyfasta_oracle as orc
from polyfasta_b200 import api, cli, parallel
from test_gpu_divergence import EXAMPLES, _parse, _run_cli, _write_fasta
from test_gpu_parity import _random_text

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _founder_text(rng, n, L, founders, changes, p_junk=0.0, junk=b"-N?RYKM."):
    """n rows drawn from `founders` random rows, `changes` point changes per row on average, optional junk and lower case:
    many identical rows"""
    F = rng.integers(0, 4, (founders, L))
    mat = F[rng.integers(0, founders, n)]
    k = rng.poisson(changes, n)
    for r in np.flatnonzero(k):
        cols = rng.integers(0, L, k[r])
        mat[r, cols] = (mat[r, cols] + rng.integers(1, 4, k[r])) % 4
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[mat]
    if p_junk:
        j = rng.random((n, L)) < p_junk
        text = np.where(j, np.frombuffer(junk, dtype=np.uint8)[rng.integers(0, len(junk), (n, L))], text)
        lo = (rng.random((n, L)) < 0.1) & (text >= 65) & (text <= 90)
        text = np.where(lo, text + 32, text)
    return np.ascontiguousarray(text.astype(np.uint8))


def _strings(text):
    return [bytes(r).decode("latin-1") for r in text]


def _classes(ctx, text, window=None, step=None):
    a = pf.Alignment.from_rows(ctx, text)
    try:
        return a.haplotype_classes(window, step)
    finally:
        a.free()


def _check_stats(entry, rows, pops):
    for q, members in enumerate(pops):
        want, got = ho.pop_stats(rows, members), entry["pops"][q]
        assert (got["n"], got["h"], got["s2"], got["s3"]) == (want["n"], want["h"], want["s2"], want["s3"])
        if want["n"] == 1:
            assert got["Hd"] == got["Hd_var"] == "NA"
        else:
            assert got["Hd"] == want["Hd"]
            assert abs(got["Hd_var"] - float(want["Hd_var"])) <= 1e-12 * abs(float(want["Hd_var"]))


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 2000, 10000])
def test_rep_against_oracle(ctx, n, p_junk):
    rng = np.random.default_rng(n + int(p_junk * 1000))
    L = 700 if n <= 2000 else 300
    text = _founder_text(rng, n, L, founders=max(1, n // 25), changes=0.5, p_junk=p_junk)
    rows = _strings(text)
    a = pf.Alignment.from_rows(ctx, text)
    up = np.where((text >= 97) & (text <= 122), text - 32, text)
    assert a.has_invalid == bool(np.isin(up, np.frombuffer(b"ACGT", dtype=np.uint8), invert=True).any())
    pops = [list(range(n)), list(range(0, n, 3)), [n - 1]]
    a.set_pops(pops)
    rep = a.haplotype_classes()
    assert rep.shape == (1, n) and rep.dtype == np.int32
    assert rep[0].tolist() == ho.rep(rows)
    _check_stats(a.haplotypes()[0], rows, pops)
    a.free()


def test_hand_made_differences(ctx):
    """rows that differ only by an IUPAC code, only by N vs -, only by case (equal), only at the last or the first column"""
    base = "ACGTRACGTNACGT-?ACGTACGTAC"
    L = len(base)
    rows = [base,
            base.replace("R", "Y"),          # R vs Y
            base.replace("N", "-", 1),        # N vs -
            base.lower(),                     # case only: equal to row 0
            base[:-1] + "G",                  # last column
            "T" + base[1:],                   # first column
            base.replace("R", "r"),           # case of an IUPAC code: equal to row 0
            base.replace("R", "K"),           # another IUPAC code
            base[:-1] + "N",                  # last column, N
            base.replace("?", "N")]           # ? vs N
    text = np.frombuffer("".join(rows).encode(), dtype=np.uint8).reshape(len(rows), L).copy()
    rep = _classes(ctx, text)
    assert rep[0].tolist() == ho.rep(rows) == [0, 1, 2, 0, 4, 5, 0, 7, 8, 9]


@pytest.mark.parametrize("kind", ["acgt", "gap", "iupac"])
def test_all_rows_identical(ctx, kind):
    row = {"acgt": "ACGTTGCA" * 50, "gap": "AC-TNG?A" * 50, "iupac": "ACRTYGWA" * 50}[kind]
    text = np.frombuffer((row * 300).encode(), dtype=np.uint8).reshape(300, len(row)).copy()
    assert not _classes(ctx, text).any()
    W = api.window_count(len(row), 37, 11)
    assert _classes(ctx, text, 37, 11).shape == (W, 300) and not _classes(ctx, text, 37, 11).any()


@pytest.mark.parametrize("W,S", [(50, 20), (64, 64), (30, 45), (1, 1), (333, 100), (5000, 7), (700, 700)])
@pytest.mark.parametrize("p_junk", [0.0, 0.02])
def test_windows_equal_cut_alignments(ctx, W, S, p_junk):
    rng = np.random.default_rng(W * 7 + S)
    n, L = 150, 700
    text = _founder_text(rng, n, L, founders=8, changes=0.3, p_junk=p_junk)
    # differences that lie only at a window's first or last column
    text[5] = text[4]
    text[5, 100] = ord("A") if text[4, 100] != ord("A") else ord("C")
    text[7] = text[6]
    text[7, 99] = ord("N") if text[6, 99] != ord("N") else ord("-")
    got = _classes(ctx, text, W, S)
    nwin = api.window_count(L, W, S)
    assert got.shape == (nwin, n)
    for i in range(nwin):
        a, b = i * S, min(i * S + W, L)
        cut = np.ascontiguousarray(text[:, a:b])
        assert got[i].tolist() == ho.rep(_strings(cut)), (i, a, b)
        if i % 17 == 0:
            assert np.array_equal(got[i], _classes(ctx, cut)[0])


def test_windows_results_against_oracle(ctx):
    rng = np.random.default_rng(5)
    n, L, W, S = 90, 400, 120, 50
    text = _founder_text(rng, n, L, founders=5, changes=0.4, p_junk=0.01)
    rows = _strings(text)
    pops = [list(range(0, n, 2)), [3], list(range(n))]
    a = pf.Alignment.from_rows(ctx, text)
    a.set_pops(pops)
    res = a.haplotypes(W, S)
    a.free()
    assert len(res) == api.window_count(L, W, S)
    for i, w in enumerate(res):
        s, e = i * S, min(i * S + W, L)
        assert (w["start"], w["end"], w["seqlen"]) == (s, e, e - s)
        _check_stats(w, ho.window_rows(rows, s, e), pops)


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
def test_pairwise_identity(ctx, p_junk):
    """within each population, the pairs with K3's d_ij > 0 are (n^2 - sum c^2) / 2"""
    rng = np.random.default_rng(77)
    n, L = 300, 900
    text = _founder_text(rng, n, L, founders=12, changes=0.6, p_junk=p_junk)
    pops = [list(range(n)), list(range(1, n, 4)), list(range(0, 200))]
    a = pf.Alignment.from_rows(ctx, text)
    a.set_pops(pops)
    _, D = a.pairwise(want_matrix=True)
    res = a.haplotypes()[0]
    a.free()
    for q, members in enumerate(pops):
        m = np.asarray(members)
        sub = D[np.ix_(m, m)]
        diff = int(np.count_nonzero(np.triu(sub, 1)))
        p = res["pops"][q]
        assert 2 * diff == p["n"] ** 2 - p["s2"]


def test_hash_collision_by_data(ctx):
    """two rows whose words of one plane follow the Thue-Morse sequence and its complement over 2,048 words collide under every
    odd-base polynomial hash mod 2^64 (prod_{j<11} (1 - B^{2^j}) = 0 mod 2^64); a third row makes all 65,536 sites variable"""
    words = 2048
    L = 32 * words
    tm = np.array([bin(j).count("1") & 1 for j in range(words)], dtype=np.uint8)
    bit = np.repeat(tm, 32)                    # plane b0 of row 0: the Thue-Morse word sequence (all ones / all zeros)
    # b0 = bit 0 of the code A0 C1 G2 T3: row 0 is C where the bit is set, A elsewhere; row 1 the complement; b1 stays 0
    r0 = np.where(bit == 1, ord("C"), ord("A")).astype(np.uint8)
    r1 = np.where(bit == 1, ord("A"), ord("C")).astype(np.uint8)
    r2 = np.full(L, ord("G"), dtype=np.uint8)  # differs from both everywhere: every site is marked
    text = np.stack([r0, r1, r2, r1.copy(), r0.copy()])
    rep = _classes(ctx, text)[0].tolist()
    assert rep == [0, 1, 2, 1, 0]
    # the same rows in windows (word-aligned and not), and as a column shard pair
    rep_w = _classes(ctx, text, 8192, 4096)
    for i in range(rep_w.shape[0]):
        a, b = i * 4096, min(i * 4096 + 8192, L)
        assert rep_w[i].tolist() == ho.rep(_strings(text[:, a:b]))


@pytest.mark.parametrize("world", [2, 3, 8])
def test_shards_meet_to_whole(ctx, world):
    rng = np.random.default_rng(world)
    n, L = 200, 2400
    text = _founder_text(rng, n, L, founders=10, changes=0.8, p_junk=0.01)
    text[:, 300 * world: 300 * world + 300] = text[0, 300 * world: 300 * world + 300]   # a stretch without a marked site
    text[:, :L // world] = text[0, :L // world]                                         # the first shard: no marked site
    whole = _classes(ctx, text)
    for W, S in ((None, None), (500, 333), (L, L), (97, 97)):
        want = _classes(ctx, text, W, S)
        reps = []
        for r in range(world):
            c0, c1 = parallel.shard_columns(L, world, r)
            a = pf.Alignment.from_rows(ctx, text, c0, c1)
            reps.append(a.haplotype_classes(W, S))
            a.free()
        assert not reps[0].any()
        got = api.meet_classes(reps)
        assert np.array_equal(got, want), (world, W, S)
    assert np.array_equal(whole[0], np.asarray(ho.rep(_strings(text)), dtype=np.int32))


def test_shard_device_entry_point(ctx):
    import torch
    rng = np.random.default_rng(3)
    text = _founder_text(rng, 64, 1000, founders=6, changes=0.5, p_junk=0.01)
    a = pf.Alignment.from_rows(ctx, text, 300, 700)
    nwin = a.window_count(200, 150)
    buf = torch.full((nwin * 64,), -1, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    a.haplotypes_device(200, 150, buf.data_ptr())
    ctx.sync()
    got = buf.cpu().numpy().reshape(nwin, 64)
    assert np.array_equal(got, a.haplotype_classes(200, 150))
    for i in range(nwin):   # windows outside [300, 700) are one class in this shard
        s, e = max(i * 150, 300), min(i * 150 + 200, 700)
        assert got[i].tolist() == (ho.rep(_strings(text[:, s:e])) if e > s else [0] * 64)
    a.free()


# ---- CLI -------------------------------------------------------------------------------------------------------------------

def _hap_line(file, seqlen, label, st):
    return f"{file},{seqlen},{label},{st['n']},{st['h']},{st['Hd']},{float(st['Hd_var']) if st['Hd_var'] != 'NA' else 'NA'}"


def test_cli_examples():
    keys = ["indiv1", "indiv2"]
    lines = _run_cli(["-d", EXAMPLES, "-p", ",".join(keys), "--haplotypes"]).splitlines()
    assert lines[0] == cli.HEADER_HAP
    files = sorted(os.listdir(EXAMPLES))
    assert len(lines) == 1 + 2 * len(files)
    want = []
    for name in files:
        heads, seqs = _parse(os.path.join(EXAMPLES, name))
        for key in keys:
            want.append(_hap_line(name, len(seqs[0]), key, ho.pop_stats(seqs, orc.pop_rows(heads, key))))
    assert lines[1:] == want
    one = _run_cli(["-f", os.path.join(EXAMPLES, "file1.fa"), "--haplotypes", "--jc"]).splitlines()
    heads, seqs = _parse(os.path.join(EXAMPLES, "file1.fa"))
    assert one == [cli.HEADER_HAP, _hap_line("file1.fa", len(seqs[0]), "NA", ho.pop_stats(seqs, range(len(seqs))))]


def test_cli_windows_match_cut_files(tmp_path):
    """--haplotypes --window W --step S rows are the --haplotypes rows of files holding only each window's columns; --out writes
    the same"""
    rng = np.random.default_rng(4243)
    n, L = 40, 257
    text = _random_text(rng, n, L, p_var=0.01, p_junk=0.005)
    text[:, 100:140] = text[0, 100:140]
    heads = ["pop%d_ind%d" % (i % 3, i) for i in range(n)]
    _write_fasta(tmp_path / "aln.fa", heads, text)
    for W, step in ((50, 50), (64, 20), (30, 45), (300, 10)):
        argv = ["-f", str(tmp_path / "aln.fa"), "-p", "pop0,nobody,pop1,pop2", "--haplotypes", "--window", str(W), "--step", str(step)]
        lines = _run_cli(argv).splitlines()
        assert lines[0] == cli.HEADER_HAP_WINDOWS
        assert lines[1] == "# Pop nobody string was not found in fasta headers."
        want = []
        for i in range(api.window_count(L, W, step)):
            a, b = i * step, min(i * step + W, L)
            sub = tmp_path / ("w%d_%d_%d" % (W, step, i))
            sub.mkdir(exist_ok=True)
            _write_fasta(sub / "aln.fa", heads, text[:, a:b])
            ref = _run_cli(["-f", str(sub / "aln.fa"), "-s", "-p", "pop0,nobody,pop1,pop2", "--haplotypes"]).splitlines()
            want.extend((a + 1, b, r) for r in ref if not r.startswith("#"))
        rows = lines[2:]
        assert len(rows) == len(want) == 3 * api.window_count(L, W, step)
        for line, (a, b, ref) in zip(rows, want):
            f = line.split(",")
            assert (int(f[1]), int(f[2])) == (a, b)
            assert ",".join([f[0]] + f[3:]) == ref, (W, step, line, ref)
        outp = tmp_path / ("out%d_%d.csv" % (W, step))
        _run_cli(argv + ["-o", str(outp), "-s"])
        assert open(outp).read().splitlines() == lines[1:]


def test_cli_pipe(tmp_path, monkeypatch):
    path = os.path.join(EXAMPLES, "file3.fa")
    data = open(path, "rb").read()

    class _Stdin:
        buffer = io.BytesIO(data)
    monkeypatch.setattr("sys.stdin", _Stdin())
    lines = _run_cli(["--pipe", "-n", "locus", "-p", "indiv1,zzz", "--haplotypes"]).splitlines()
    heads, seqs = _parse(path)
    assert lines == [cli.HEADER_HAP, "# Pop zzz string was not found in fasta headers.",
                     _hap_line("locus", len(seqs[0]), "indiv1", ho.pop_stats(seqs, orc.pop_rows(heads, "indiv1")))]


def test_cli_two_ranks_one_gpu(tmp_path):
    """--haplotypes through the column-sharded route, two ranks on one GPU summing on the host: rank 0 prints exactly what one
    process prints, rank 1 nothing"""
    import torch.multiprocessing as mp
    from test_gpu_cli_routes import _free_port, _worker
    rng = np.random.default_rng(31)
    n, L = 60, 30001
    text = _founder_text(rng, n, L, founders=9, changes=1.5, p_junk=0.002)
    path = tmp_path / "big.fa"
    _write_fasta(path, ["pop%d_%d" % (i % 3, i) for i in range(n)], text)
    base = ["-f", str(path), "-p", "pop0,nobody,pop1,pop2", "--haplotypes"]
    argvs = [base, base + ["--window", "900", "--step", "600"], ["-f", str(path), "--haplotypes", "--window", "20000"]]
    want = [_run_cli(a) for a in argvs]
    assert want[0].count("\n") == 5
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = _free_port()
    procs = [mpc.Process(target=_worker, args=(r, port, argvs, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=600) for _ in range(2))
    for p in procs:
        p.join(60)
    assert got[0] == want
    assert all(o == "" for o in got[1])
