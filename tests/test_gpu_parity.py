"""GPU parity tests: the CUDA path, called through the C ABI, against (a) the golden vectors produced by the unmodified
reference, (b) the CPU oracles on seeded inputs, (c) size-independent properties at the benchmark's full size.
Integers are compared bit-exactly; fp64 statistics within rel 1e-12 (D: see test_oracle_golden.check_poly)."""
import io
import math
import os
import random
import subprocess
import sys
from contextlib import redirect_stdout

import numpy as np
import pytest

import polyfasta_b200 as pf
from polyfasta_b200 import cli, synth
from conftest import GOLDEN, ROOT, load_golden
from oracle import c_oracle as co
from oracle import polyfasta_oracle as orc
from test_oracle_golden import check_poly, close

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _pops_present(heads, keys):
    plan = [(k, list(range(len(heads))) if k == "NA" else orc.pop_rows(heads, k)) for k in keys]
    return [(k, r) for k, r in plan if r]


def _check_alignment(ctx, heads, seqs, L, pops, file, check_rows=True):
    present = _pops_present(heads, [k for k, rec in pops.items() if rec is not None])
    if not present:
        return
    aln = pf.Alignment.from_strings(ctx, seqs)
    aln.set_pops([r for _, r in present])
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    pw = aln.pairwise() if len(seqs) <= 64 else None
    aln.free()
    for q, (key, rows) in enumerate(present):
        rec = pops[key]
        st = site[q]
        assert (st["n"], st["S"], st["H"]) == (rec["n"], rec["S"], rec["H"]), (file, key)
        assert np.flatnonzero(st["isvar"]).tolist() == rec["pos"], (file, key)
        assert st["sfs"] == (rec["sfs"] if rec["S"] else [0] * (rec["n"] // 2)), (file, key)
        if pw is not None:
            assert 2 * pw[q] == rec["H"], (file, key)
        for jc in (0, 1):
            got = ctx.finalize([(st["n"], st["S"], st["H"], L, jc)])[0]
            check_poly(got, rec["poly_jc%d" % jc], st["n"], st["S"], st["H"])
        c = rec.get("cds")
        if c is None:
            continue
        g = cds[q]
        for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n"):
            assert g[k] == c[k], (file, key, k)
        assert np.flatnonzero(g["labels"] == 1).tolist() == sorted(c["S_pos"]), (file, key)
        assert np.flatnonzero(g["labels"] == 2).tolist() == sorted(c["N_pos"]), (file, key)
        assert {str(k): v for k, v in g["sum3_by_len"].items()} == {k: v for k, v in c["sum3_by_len"].items() if v}
        assert close(g["ssites"], c["count_syn"]), (file, key)
        if check_rows:
            for is_cds in (0, 1):
                for jc in (0, 1):
                    want = rec["row_cds%d_jc%d" % (is_cds, jc)].rstrip("\n")
                    got = cli.format_rows(ctx, file, L, bool(is_cds), bool(jc), [(key, len(rows))], [st], [g] if is_cds else None)[0]
                    _rows_close(got, want)


def _rows_close(got, want):
    g, w = got.split(","), want.split(",")
    assert len(g) == len(w), (got, want)
    for i, (x, y) in enumerate(zip(g, w)):
        if x != y:
            if len(g) == 14 and i in (1, 2):
                # sites_S / sites_N are printed as round(x, 2) (PolyFastA.py:178): when the exact value is a tie such
                # as 8.875 the reference's running float sum (:307) decides the last digit.  The unrounded values are
                # compared to 1e-12 separately (ssites); here one unit in the last printed place is allowed.
                assert abs(float(x) - float(y)) <= 0.01 + 1e-9, (got, want)
            else:
                assert math.isclose(float(x), float(y), rel_tol=2e-11), (got, want)


def test_example_loci(ctx):
    """C1/C2: the shipped loci, whole file and header-substring populations, against the reference's own numbers"""
    for fn, entry in load_golden("kat_examples.json").items():
        f = pf.Fasta.from_file(os.path.join(GOLDEN, "example_theta_0.01", fn))
        seqs = [f.row(i) for i in range(f.nseq)]
        _check_alignment(ctx, f.headers, seqs, entry["seqlen"], entry["pops"], fn)


def test_random_cases(ctx):
    """220 random alignments with gaps / N / IUPAC / '?' / lower case / stops"""
    for ci, case in enumerate(load_golden("random_cases.json")):
        f = pf.Fasta.from_bytes(case["text"])
        seqs = [f.row(i) for i in range(f.nseq)]
        _check_alignment(ctx, f.headers, seqs, case["seqlen"], case["pops"], "case%d.fa" % ci)


def test_finalize_cases(ctx):
    recs = load_golden("finalize_cases.json")
    got = ctx.finalize([(r["n"], r["S"], r["H"], r["seqlen"], r["jc"]) for r in recs])
    for g, r in zip(got, recs):
        check_poly(g, r["out"], r["n"], r["S"], r["H"])


def test_cli_golden(tmp_path):
    """the drop-in command line against the reference's captured stdout / --out files"""
    env = dict(os.environ, PYTHONPATH=ROOT, PYTHONHASHSEED="0")
    for rec in load_golden("cli_examples.json"):
        args = list(rec["args"])
        outp = str(tmp_path / "out.csv")
        if "@OUT@" in args:
            with open(outp, "w") as f:
                f.write("PRE-EXISTING LINE\n")
            args[args.index("@OUT@")] = outp
        stdin = None
        if rec["stdin"]:
            with open(os.path.join(GOLDEN, "example_theta_0.01", "file1.fa"), "rb") as f:
                stdin = f.read()
        p = subprocess.run([sys.executable, os.path.join(ROOT, "PolyFastA.py")] + args, input=stdin, capture_output=True,
                           env=env, cwd=GOLDEN)
        assert p.returncode == rec["rc"], (args, p.stderr.decode())
        _text_close(p.stdout.decode().replace(outp, "@OUT@"), rec["stdout"], args)
        if "outfile" in rec:
            with open(outp) as f:
                _text_close(f.read(), rec["outfile"], args)


def _text_close(got, want, what):
    gl, wl = got.split("\n"), want.split("\n")
    assert len(gl) == len(wl), (what, got, want)
    for g, w in zip(gl, wl):
        if g != w:
            _rows_close(g, w)


def test_cli_pops(tmp_path):
    """-p: rows per key in key order, '# Pop ... not found' rows, overlapping keys (reference rows via print_result)"""
    kat = load_golden("kat_examples.json")
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "PolyFastA.py"), "-d", "example_theta_0.01", "-p",
                        "indiv1,nothere,indiv2", "--jc", "-s"], capture_output=True, text=True, env=env, cwd=GOLDEN)
    assert p.returncode == 0, p.stderr
    want = []
    for fn in sorted(kat):
        want.append(kat[fn]["pops"]["indiv1"]["row_cds0_jc1"].rstrip("\n"))
        want.append("# Pop nothere string was not found in fasta headers.")
        want.append(kat[fn]["pops"]["indiv2"]["row_cds0_jc1"].rstrip("\n"))
    _text_close(p.stdout, "\n".join(want) + "\n", "pops")


def _random_text(rng, n, L, p_var=0.05, p_junk=0.01, junk=b"-N?RYKM.", lower=0.1):
    anc = rng.integers(0, 4, L)
    mat = np.repeat(anc[None, :], n, axis=0)
    var = rng.random(L) < p_var
    k = rng.integers(1, max(n, 2), L)
    der = (anc + rng.integers(1, 4, L)) % 4
    perm_rank = rng.random((n, L)).argsort(axis=0)
    mat = np.where(var[None, :] & (perm_rank < k[None, :]), der[None, :], mat)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[mat]
    j = rng.random((n, L)) < p_junk
    text = np.where(j, np.frombuffer(junk, dtype=np.uint8)[rng.integers(0, len(junk), (n, L))], text)
    lo = rng.random((n, L)) < lower
    text = np.where(lo & (text >= 65) & (text <= 90), text + 32, text).astype(np.uint8)
    return np.ascontiguousarray(text)


def _upper(mat):
    return np.where((mat >= 97) & (mat <= 122), mat - 32, mat).astype(np.uint8)


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("n,L", [(1, 50), (2, 333), (31, 1000), (32, 999), (33, 1001), (127, 700), (128, 701), (129, 650),
                                 (300, 5000), (1000, 6001), (2049, 3000), (5000, 1500), (10001, 600),
                                 (300, 1), (300, 2), (300, 4), (2000, 1), (2000, 2), (2000, 4)])
def test_against_c_oracle(ctx, n, L, p_junk):
    """seeded alignments of many shapes (word / chunk boundary cases for n), three overlapping populations.
    p_junk = 0: pure ACGT, i.e. the two-plane (HAS_V = false) instantiations every throughput figure is quoted on;
    p_junk = 0.01: gaps / N / ? / IUPAC codes, the three-plane instantiations plus the escape kernels.
    L = 1, 2: codon shards without a whole codon column (only the trailing partial one) through the TMA codon scan"""
    rng = np.random.default_rng(n * 1000003 + L)
    text = _random_text(rng, n, L, p_junk=p_junk)
    up = _upper(text)
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n))]
    pops = [p for p in pops if p]
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.has_invalid == bool((~np.isin(up, np.frombuffer(b"ACGT", dtype=np.uint8))).any())
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    aln.free()
    for q, rows in enumerate(pops):
        want = co.site_stats(up, rows, per_site=True)
        assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"]), (n, L, q)
        assert np.array_equal(site[q]["isvar"], want["isvar"])
        wc = co.cds_stats(up, rows, want_labels=True)
        for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
            assert cds[q][k] == wc[k], (n, L, q, k)
        assert np.array_equal(cds[q]["labels"], wc["labels"])
        assert math.isclose(cds[q]["ssites"], wc["ssites"], rel_tol=1e-12) or cds[q]["ssites"] == wc["ssites"]


def test_gappy_and_escape_heavy(ctx):
    """every column holds non-ACGT symbols; many distinct escape bytes per column; whole-column escapes"""
    rng = np.random.default_rng(77)
    n, L = 150, 900
    text = _random_text(rng, n, L, p_var=0.3, p_junk=0.4, junk=b"-N?RYKMSWBDHV.* x", lower=0.3)
    text[:, 10] = ord("R")
    text[:, 11] = ord("-")
    text[: n // 2, 12] = ord("Y")
    text[n // 2:, 12] = ord("r")
    up = _upper(text)
    pops = [list(range(n)), list(range(0, n, 3)), list(range(5, 40))]
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.num_escapes > 0 and aln.has_invalid
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    pw = aln.pairwise()
    aln.free()
    for q, rows in enumerate(pops):
        want = co.site_stats(up, rows, per_site=True)
        assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"])
        assert np.array_equal(site[q]["isvar"], want["isvar"])
        wc = co.cds_stats(up, rows, want_labels=True)
        for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
            assert cds[q][k] == wc[k], (q, k)
        assert np.array_equal(cds[q]["labels"], wc["labels"])
        assert 2 * pw[q] == want["H"]


def test_column_shards_add_up(ctx):
    """the integer vectors of column shards (codon-aligned) sum to the whole: what the multi-GPU all-reduce relies on"""
    rng = np.random.default_rng(5)
    n, L = 400, 3001
    text = _random_text(rng, n, L)
    pops = [list(range(n)), list(range(0, n, 2))]
    whole = pf.Alignment.from_rows(ctx, text)
    whole.set_pops(pops)
    ws, wc = whole.site_stats(), whole.cds_stats()
    whole.free()
    for parts in (2, 4, 8):
        per = (L // parts) // 3 * 3
        bounds = [i * per for i in range(parts)] + [L]
        acc_s = None
        acc_c = None
        for i in range(parts):
            sh = pf.Alignment.from_rows(ctx, text, bounds[i], bounds[i + 1])
            sh.set_pops(pops)
            s, c = sh.site_stats(), sh.cds_stats()
            sh.free()
            vs = [np.array([x["S"], x["H"]] + x["sfs"]) for x in s]
            vc = [x["raw"] for x in c]
            acc_s = vs if acc_s is None else [a + b for a, b in zip(acc_s, vs)]
            acc_c = vc if acc_c is None else [a + b for a, b in zip(acc_c, vc)]
        for q in range(len(pops)):
            assert acc_s[q].tolist() == [ws[q]["S"], ws[q]["H"]] + ws[q]["sfs"]
            assert np.array_equal(acc_c[q], wc[q]["raw"])


def test_synthetic_generator_matches_numpy_twin(ctx):
    """device generator == numpy twin (planes bit for bit), and the kernels == the closed form"""
    for n, L, seed in [(20, 1000, 1), (100, 5000, 5), (129, 777, 9), (1000, 3000, 4)]:
        dev = pf.Alignment.synthetic(ctx, n, L, seed, 100000, 50000)
        host = pf.Alignment.from_rows(ctx, synth.text_matrix(seed, n, L, 100000, 50000))
        for pl in range(3):
            assert np.array_equal(dev.plane(pl), host.plane(pl)), (n, L, pl)
        got = dev.site_stats()[0]
        want = synth.expected_site_stats(seed, n, L, 100000, 50000)
        assert (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"])
        dev.free()
        host.free()


def test_full_size_closed_form(ctx):
    """C4's row count (10,000) at 2 Mb (2e10 bases): the site scan against the generator's closed form, whole and in
    8 column shards; the same check runs at the full 10 Mb inside bench.py"""
    n, L, seed = 10000, 2_000_000, 4
    want = synth.expected_site_stats(seed, n, L)
    a = pf.Alignment.synthetic(ctx, n, L, seed)
    got = a.site_stats()[0]
    a.free()
    assert (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"])
    tot = np.zeros(2 + n // 2, dtype=np.int64)
    per = L // 8
    for i in range(8):
        sh = pf.Alignment.synthetic(ctx, n, L, seed, col_begin=i * per, col_end=L if i == 7 else (i + 1) * per)
        r = sh.site_stats()[0]
        sh.free()
        tot += np.array([r["S"], r["H"]] + r["sfs"])
    assert tot.tolist() == [want["S"], want["H"]] + want["sfs"]


def test_mirror_api_reads_like_the_reference(ctx):
    kat = load_golden("kat_examples.json")["file1.fa"]
    d = pf.readfasta(os.path.join(GOLDEN, "example_theta_0.01", "file1.fa"), False)
    pos, var = pf.getvarsites(d, 1000)
    rec = kat["pops"]["NA"]
    assert pos == rec["pos"] and len(var) == 87 and len(var[0]) == 20
    check_poly(pf.polymorphism(var, 1000, False), rec["poly_jc0"], 20, rec["S"], rec["H"])
    assert pf.getsfs(var) == rec["sfs_ref"]
    cs, S, N, nstops, missing = pf.getvarCDSsites(d, 1000)
    c = rec["cds"]
    assert (S, N, nstops, missing) == (sorted(c["S_pos"]), sorted(c["N_pos"]), c["nstops"], c["missing"])
    assert close(cs, c["count_syn"])
    haplo = list(map(list, zip(*var)))
    assert pf.nucleotide_diversity3(haplo) * (20 * 19 // 2) * 2 == pytest.approx(rec["H"], rel=1e-15)


def test_edge_shapes(ctx):
    """empty alignment, single row, single site, no variation"""
    a = pf.Alignment.from_strings(ctx, ["", ""])
    assert a.site_stats()[0]["S"] == 0 and a.cds_stats()[0]["missing"] == 0
    a.free()
    a = pf.Alignment.from_strings(ctx, ["ACGTAC"])
    s = a.site_stats()[0]
    assert (s["n"], s["S"], s["H"], s["sfs"]) == (1, 0, 0, [])
    a.free()
    a = pf.Alignment.from_strings(ctx, ["A", "C", "A"])
    s = a.site_stats()[0]
    assert (s["S"], s["H"], s["sfs"]) == (1, 4, [1])
    c = a.cds_stats()[0]
    assert c["missing"] == 3 and c["nstops"] == 0
    a.free()
    assert ctx.finalize([(5, 0, 0, 10, False)]) == [(0, 0, 0, "NA")]


def test_batch_path_matches_single_alignment_path(ctx):
    """the batched --dir path (K1b/K2b/K5b, one sync) == the single-alignment kernels == the C oracle, for loci of mixed
    shapes, populations and symbol content in one batch"""
    rng = np.random.default_rng(123)
    shapes = [(20, 1000), (100, 5000), (3, 7), (1, 40), (33, 65), (128, 300), (129, 301), (700, 900), (2100, 257), (16, 0), (50, 31)]
    batch = pf.api.Batch(ctx)
    loci = []
    for i, (n, L) in enumerate(shapes):
        text = _random_text(rng, n, L, p_junk=(0.0 if i % 3 == 0 else 0.02)) if L else np.zeros((n, 0), dtype=np.uint8)
        pops = None if i % 2 == 0 else [p for p in (list(range(0, n, 2)), list(range(n // 2, n)), list(range(n))) if p]
        loci.append((text, pops, batch.add_rows(text, pops)))
    batch.run(jc=True)
    for text, pops, idx in loci:
        n, L = text.shape
        up = _upper(text)
        for q, rows in enumerate(pops or [list(range(n))]):
            got = batch.result(idx, q, want_sfs=True)
            want = co.site_stats(up, rows) if L else {"S": 0, "H": 0, "sfs": [0] * (len(rows) // 2)}
            assert (got["n"], got["S"], got["H"], got["sfs"]) == (len(rows), want["S"], want["H"], want["sfs"]), (n, L, q)
            ref = ctx.finalize([(len(rows), want["S"], want["H"], L, True)])[0]
            assert got["poly"] == ref, (n, L, q)
    # reuse of the same batch object
    batch.clear()
    idx = batch.add_rows(loci[1][0], None)
    batch.run(jc=False)
    assert batch.result(idx)["S"] == co.site_stats(_upper(loci[1][0]))["S"]
    batch.close()


def test_batch_golden_examples(ctx):
    """C2: the 10 shipped loci in ONE batch, with the substring populations, against the reference's rows"""
    kat = load_golden("kat_examples.json")
    batch = pf.api.Batch(ctx)
    slots = []
    for fn in sorted(kat):
        f = pf.Fasta.from_file(os.path.join(GOLDEN, "example_theta_0.01", fn))
        masks = np.stack([pf.api.match_mask(f, key)[0] for key in ("indiv1", "indiv2", "indiv")])
        slots.append((fn, batch.add(f, masks)))
    batch.run(jc=True)
    for fn, idx in slots:
        for q, key in enumerate(("indiv1", "indiv2", "indiv")):
            rec = kat[fn]["pops"][key]
            got = batch.result(idx, q, want_sfs=True)
            assert (got["n"], got["S"], got["H"]) == (rec["n"], rec["S"], rec["H"])
            check_poly(got["poly"], rec["poly_jc1"], rec["n"], rec["S"], rec["H"])
    batch.close()


def test_cli_dir_on_two_contexts(tmp_path):
    """--dir with POLYFASTA_DEVICES naming two contexts (the same GPU twice on a 1-GPU box): chunks are processed by two
    worker threads and the rows still come out in the reference's sorted() order"""
    import polyfasta_b200.cli as cli_mod
    d = tmp_path / "loci"
    d.mkdir()
    rng = np.random.default_rng(8)
    want = {}
    for i in range(23):
        n, L = int(rng.integers(2, 40)), int(rng.integers(10, 400))
        text = _upper(_random_text(rng, n, L, lower=0.0))
        with open(d / ("locus%d.fa" % i), "w") as f:
            for r in range(n):
                f.write(">s%d\n%s\n" % (r, text[r].tobytes().decode()))
        rows = [text[r].tobytes().decode() for r in range(n)]
        want["locus%d.fa" % i] = orc.noncds_row("locus%d.fa" % i, L, "NA", rows, True)
    env = dict(os.environ, PYTHONPATH=ROOT, POLYFASTA_DEVICES="0,0", POLYFASTA_BATCH_FILES="4")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "PolyFastA.py"), "-d", str(d), "--jc", "-s"], capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    lines = p.stdout.strip().split("\n")
    assert [ln.split(",")[0] for ln in lines] == sorted(want)
    for ln in lines:
        _rows_close(ln, want[ln.split(",")[0]])


def _planes(a):
    return [a.plane(i) for i in range(3)]


@pytest.mark.parametrize("pinned", [False, True])
@pytest.mark.parametrize("n,L,c0,c1", [(33, 70000, 0, None), (260, 40001, 0, None), (1000, 9000, 1200, 8190), (129, 30011, 3, 30011)])
def test_hybrid_ingest_matches_plain_upload(ctx, monkeypatch, n, L, c0, c1, pinned):
    """large host inputs are split in column chunks between a raw lane (text over PCIe, K1) and a packed lane (host threads
    pack 4 bases per byte, pfa_encode_packed_kernel); chunks holding non-ACGT symbols fall back to the raw lane.  The planes,
    the exception list and every statistic must not depend on which lane a chunk took."""
    rng = np.random.default_rng(n + L)
    clean = _random_text(rng, n, L, p_junk=0.0)
    some = clean.copy()
    some[rng.integers(0, n, 40), rng.integers(L // 2, L, 40)] = np.frombuffer(b"-NR?n", dtype=np.uint8)[rng.integers(0, 5, 40)]
    gappy = _random_text(rng, n, L, p_junk=0.05)
    gaps_only = _random_text(rng, n, L, p_junk=0.03, junk=b"-Nn?")   # no escape symbols: packed with a validity bitmap (VBMI hosts)
    monkeypatch.setenv("PFA_INGEST_CHUNK_MB", "1")
    pops = [list(range(n)), list(range(0, n, 2))]
    import torch

    def upload(text):
        # pageable numpy memory: packed lane first, dirty chunks through pinned bounce buffers; pinned memory: the two lanes
        # race for the chunks and the raw lane copies straight from the source
        if not pinned:
            return pf.Alignment.from_rows(ctx, text, c0, c1)
        t = torch.from_numpy(text).pin_memory()
        a = pf.Alignment.from_host_ptr(ctx, t.data_ptr(), n, L, L, c0, L if c1 is None else c1)
        ctx.sync()
        return a

    for name, text in (("clean", clean), ("some", some), ("gappy", gappy), ("gaps_only", gaps_only)):
        monkeypatch.setenv("PFA_INGEST_HYBRID", "0")
        plain = pf.Alignment.from_rows(ctx, text, c0, c1)
        # mode 2: every chunk is offered to the packer first (deterministic); mode 1: the lanes race for the chunks
        monkeypatch.setenv("PFA_INGEST_HYBRID", "2")
        hyb = upload(text)
        st = ctx.ingest_stats()
        assert st["raw_chunks"] + st["packed_chunks"] >= 2, st
        if name == "clean":
            assert st["raw_chunks"] == 0 and st["dirty_chunks"] == 0, st
        if name == "some":
            assert st["packed_chunks"] > 0 and 0 < st["dirty_chunks"] <= st["raw_chunks"], st
        if name == "gappy":
            assert st["packed_chunks"] == 0 and st["dirty_chunks"] >= 1, st
        if name == "gaps_only":   # hosts without AVX-512 VBMI treat these chunks as dirty
            assert st["packed_chunks_with_validity"] == st["packed_chunks"] > 0 or st["packed_chunks"] == 0, st
        monkeypatch.setenv("PFA_INGEST_HYBRID", "1")
        race = upload(text)
        for x, y, z in zip(_planes(plain), _planes(hyb), _planes(race)):
            assert np.array_equal(x, y) and np.array_equal(x, z), name
        assert race.num_escapes == plain.num_escapes
        race.free()
        assert plain.num_escapes == hyb.num_escapes and plain.has_invalid == hyb.has_invalid
        plain.set_pops(pops)
        hyb.set_pops(pops)
        a, b = plain.site_stats(), hyb.site_stats()
        ca, cb = plain.cds_stats(), hyb.cds_stats()
        for q in range(2):
            assert (a[q]["S"], a[q]["H"], a[q]["sfs"]) == (b[q]["S"], b[q]["H"], b[q]["sfs"])
            assert np.array_equal(ca[q]["raw"], cb[q]["raw"])
        if name == "some":
            up = _upper(text[:, c0:c1])
            want = co.site_stats(up, pops[1])
            assert (b[1]["S"], b[1]["H"], b[1]["sfs"]) == (want["S"], want["H"], want["sfs"])
        plain.free()
        hyb.free()


def test_large_file_rows_in_place(ctx, tmp_path, monkeypatch):
    """files of 64 MB and more are parsed in place: the rows stay inside the file buffer at arbitrary offsets and the
    uploader gathers them (packed lane, dirty chunks through pinned bounce buffers).  Forced here on a small file with
    wrapped lines, headers of different lengths and a few non-ACGT symbols; column shards included."""
    rng = np.random.default_rng(99)
    n, L = 90, 20000
    text = _random_text(rng, n, L, p_junk=0.0)
    text[rng.integers(0, n, 25), rng.integers(L // 3, L, 25)] = np.frombuffer(b"-NRy?", dtype=np.uint8)[rng.integers(0, 5, 25)]
    path = tmp_path / "big.fa"
    with open(path, "wb") as f:
        for i in range(n):
            f.write((">pop%d_%d%s\n" % (i % 2, i, "x" * (i % 7))).encode())
            row = text[i].tobytes()
            w = 60 if i % 3 else 977
            for o in range(0, L, w):
                f.write(row[o:o + w] + b"\n")
    monkeypatch.setenv("PFA_INGEST_CHUNK_MB", "1")
    ref = pf.Fasta.from_file(str(path))
    pops = [list(range(n)), [i for i, h in enumerate(ref.headers) if "pop1" in h]]
    want = []
    for c0, c1 in ((0, L), (0, 9999), (9999, L)):
        a = pf.Alignment.from_fasta(ctx, ref, c0, c1)
        a.set_pops(pops)
        want.append((a.site_stats(), a.cds_stats(), [a.plane(i) for i in range(3)], a.num_escapes))
        a.free()
    monkeypatch.setenv("PFA_BIG_FILE_MIN", "1")
    big = pf.Fasta.from_file(str(path))
    assert big.headers == ref.headers and big.seqlen == L and [big.row(i) for i in (0, 1, n - 1)] == [ref.row(i) for i in (0, 1, n - 1)]
    for (c0, c1), (ws, wc, wp, we) in zip(((0, L), (0, 9999), (9999, L)), want):
        a = pf.Alignment.from_fasta(ctx, big, c0, c1)
        st = ctx.ingest_stats()
        assert st["packed_chunks"] + st["raw_chunks"] >= 1
        a.set_pops(pops)
        gs, gc = a.site_stats(), a.cds_stats()
        for x, y in zip(wp, [a.plane(i) for i in range(3)]):
            assert np.array_equal(x, y)
        assert a.num_escapes == we
        for q in range(2):
            assert (gs[q]["S"], gs[q]["H"], gs[q]["sfs"]) == (ws[q]["S"], ws[q]["H"], ws[q]["sfs"])
            assert np.array_equal(gc[q]["raw"], wc[q]["raw"])
        a.free()
    up = _upper(text)
    o = co.site_stats(up, pops[1])
    assert (want[0][0][1]["S"], want[0][0][1]["H"]) == (o["S"], o["H"])


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
@pytest.mark.parametrize("n,L", [(21000, 240), (13000, 303)])
def test_streaming_scan_kernels(ctx, n, L, p_junk):
    """alignments with more rows than the TMA kernels take (K2: 20,480, K4: 12,288) go through the streaming two-pass
    kernels, one warp per site or codon column.  Same checks as test_against_c_oracle, plus the exchange epilogue
    (world = 1) on this path."""
    rng = np.random.default_rng(n + 7 * L)
    text = _random_text(rng, n, L, p_junk=p_junk)
    up = _upper(text)
    pops = [list(range(n)), list(range(0, n, 3))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    import torch
    from polyfasta_b200 import parallel
    x = parallel.connect_exchange(ctx, max(aln.site_len(), 71 * 2))
    d_s = torch.zeros(aln.site_len(), dtype=torch.int64, device="cuda")
    d_c = torch.zeros(71 * 2, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    aln.site_stats_xchg(x, d_s.data_ptr())
    aln.cds_stats_xchg(x, d_c.data_ptr())
    ctx.sync()
    fused_s, fused_c = d_s.cpu().numpy(), d_c.cpu().numpy().reshape(2, 71)
    off = aln.site_offsets()
    aln.free()
    x.close()
    for q, rows in enumerate(pops):
        want = co.site_stats(up, rows, per_site=True)
        assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"]), (n, L, q)
        assert np.array_equal(site[q]["isvar"], want["isvar"])
        assert fused_s[off[q]: off[q + 1]].tolist() == [want["S"], want["H"]] + want["sfs"]
        wc = co.cds_stats(up, rows, want_labels=True)
        for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
            assert cds[q][k] == wc[k], (n, L, q, k)
        assert np.array_equal(cds[q]["labels"], wc["labels"])
        assert np.array_equal(fused_c[q], cds[q]["raw"])


def _check_site_cds(site, cds, up, pops, what):
    for q, rows in enumerate(pops):
        want = co.site_stats(up, rows, per_site=True)
        assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"]), (what, q)
        if "isvar" in site[q]:
            assert np.array_equal(site[q]["isvar"], want["isvar"]), (what, q)
        wc = co.cds_stats(up, rows, want_labels=True)
        for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
            assert cds[q][k] == wc[k], (what, q, k)
        if "labels" in cds[q]:
            assert np.array_equal(cds[q]["labels"], wc["labels"]), (what, q)
        assert math.isclose(cds[q]["ssites"], wc["ssites"], rel_tol=1e-12), (what, q)


@pytest.mark.parametrize("pops_kind", ["halves", "one"])
def test_c3_shape_pure_acgt(ctx, pops_kind):
    """C3's shape (2,000 rows, in-frame CDS, two populations = the two halves) at 300 kb, pure ACGT from the synthetic
    generator: the instantiations C3's figures are quoted on -- pfa_cds_scan_tma_kernel<8,2,HAS_V=false,MULTI,512> and
    pfa_site_scan_tma_kernel<4,4,false,MULTI> -- against the C oracle, bit-exact (PolyFastA.py:252-261, 284-315)"""
    n, L, seed = 2000, 300_000, 3
    text = co.synth_text(seed, n, L)
    pops = [list(range(n // 2)), list(range(n // 2, n))] if pops_kind == "halves" else [list(range(n))]
    aln = pf.Alignment.from_rows(ctx, text)
    assert not aln.has_invalid and aln.num_escapes == 0
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    aln.free()
    _check_site_cds(site, cds, text, pops, "c3")
    assert sum(c["S_s"] + c["S_n"] for c in cds) > 1000   # the case does exercise the variable-column paths


@pytest.mark.parametrize("n,L,k", [(200, 30_000, 2), (640, 9_000, 3), (2000, 6_000, 2), (5000, 1_500, 1), (100, 60_000, 2)])
def test_pure_acgt_multi_population_shapes(ctx, n, L, k):
    """pure-ACGT (two-plane) register / TMA kernels over the lanes-per-site and chunks-per-lane cases the launcher picks
    between (Wq = 2 ... 40), with 1-3 populations of unequal size that do not cover all rows"""
    rng = np.random.default_rng(n * 31 + L)
    text = _random_text(rng, n, L, p_var=0.08, p_junk=0.0, lower=0.05)
    up = _upper(text)
    pops = [list(range(0, n // 2)), list(range(n // 2 + 3, n)), list(range(1, n, 3))][:k]
    aln = pf.Alignment.from_rows(ctx, text)
    assert not aln.has_invalid
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    aln.free()
    _check_site_cds(site, cds, up, pops, (n, L, k))


def _brute_pairwise(up):
    """d_ij by one-hot matrix products over the variable columns: an independent numpy restatement of the pairwise loop
    of nucleotide_diversity3 (PolyFastA.py:469-479)"""
    var = (up != up[0:1, :]).any(axis=0)
    sub = up[:, var]
    same = np.zeros((up.shape[0], up.shape[0]), dtype=np.float64)
    for sym in np.unique(sub):
        x = (sub == sym).astype(np.float32)
        same += x @ x.T
    return (int(var.sum()) - np.rint(same)).astype(np.int32)


@pytest.mark.parametrize("n,L,p_junk", [(2000, 20_000, 0.0), (2000, 20_000, 0.002), (333, 5_000, 0.02), (64, 100_000, 0.0)])
def test_pairwise_matrix(ctx, n, L, p_junk):
    """K3: the n x n matrix of pairwise differences against a numpy brute force and the C oracle (matrix and sums per
    population), at the profiled shape (2,000 rows) with the variable-site compaction at a large L
    (PolyFastA.py:468-480)"""
    rng = np.random.default_rng(n + L)
    text = _random_text(rng, n, L, p_var=0.05, p_junk=p_junk, lower=0.1)
    up = _upper(text)
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 4, n // 2))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    sums, mat = aln.pairwise(want_matrix=True)
    only_sums = aln.pairwise()
    site = aln.site_stats()
    aln.free()
    brute = _brute_pairwise(up)
    assert np.array_equal(mat, brute)
    tot, omat = co.pairwise_sum(up, None, want_matrix=True)
    assert np.array_equal(mat, omat)
    assert only_sums == sums
    for q, rows in enumerate(pops):
        r = np.asarray(rows)
        assert sums[q] == int(np.triu(brute[np.ix_(r, r)], 1).sum(dtype=np.int64)), q
        assert 2 * sums[q] == site[q]["H"], q
    assert sums[0] == tot


def test_integration_stub_runs_as_printed(ctx):
    """the reference-side ctypes stub of INTEGRATION.md (Option B), executed as printed, against the reference's rows"""
    with open(os.path.join(ROOT, "INTEGRATION.md")) as f:
        md = f.read()
    a = md.index("```python\n# --- PolyFastA.py, after the imports") + len("```python\n")
    code = md[a: md.index("```", a)].replace('"libpolyfasta_b200.so"', repr(pf._lib.SO_PATH))
    ns = {}
    exec(compile(code, "INTEGRATION.md", "exec"), ns)
    assert isinstance(ns["_pfa"].pfa_global_error(), bytes)
    kat = load_golden("kat_examples.json")
    for fn in ("file1.fa", "file7.fa"):
        d = pf.readfasta(os.path.join(GOLDEN, "example_theta_0.01", fn), False)
        rec = kat[fn]["pops"]["NA"]
        for jc in (False, True):
            check_poly(ns["polymorphism_gpu"](d, 1000, jc), rec["poly_jc%d" % jc], 20, rec["S"], rec["H"])
    assert ns["polymorphism_gpu"]({"a": "ACGT", "b": "ACGT"}, 4, False) == (0, 0, 0, "NA")


def test_batch_exception_list_overflow_retries(ctx, tmp_path):
    """loci holding far more symbols outside ACGT-N? than the batched path sizes its exception list for ('.', '*', dense
    IUPAC codes: all alleles in the reference, PolyFastA.py:256-258): K1b is re-run with a list of the exact size instead
    of failing the chunk; through the API and through --dir"""
    rng = np.random.default_rng(31)
    batch = pf.api.Batch(ctx)
    loci = []
    for n, L in [(200, 2000), (64, 3000), (300, 700)]:
        text = _random_text(rng, n, L, p_var=0.2, p_junk=0.35, junk=b"RYKMSW.*BDHV")
        loci.append((text, batch.add_rows(text, [list(range(n)), list(range(0, n, 2))])))
    assert sum(int((~np.isin(_upper(t), np.frombuffer(b"ACGT-N?", dtype=np.uint8))).sum()) for t, _ in loci) > (1 << 16)
    batch.run(jc=False)
    for text, idx in loci:
        up = _upper(text)
        for q, rows in enumerate([list(range(text.shape[0])), list(range(0, text.shape[0], 2))]):
            got, want = batch.result(idx, q, want_sfs=True), co.site_stats(up, rows)
            assert (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"])
    batch.close()
    d = tmp_path / "dense"
    d.mkdir()
    want = {}
    for i in range(3):
        n, L = 250, 600
        text = _upper(_random_text(rng, n, L, p_junk=0.5, junk=b"RYKMSW.*", lower=0.0))
        rows = [text[r].tobytes().decode() for r in range(n)]
        with open(d / ("l%d.fa" % i), "w") as f:
            f.write("".join(">s%d\n%s\n" % (r, s) for r, s in enumerate(rows)))
        want["l%d.fa" % i] = orc.noncds_row("l%d.fa" % i, L, "NA", rows, False)
    env = dict(os.environ, PYTHONPATH=ROOT)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "PolyFastA.py"), "-d", str(d), "-s"], capture_output=True, text=True, env=env)
    assert p.returncode == 0, p.stderr
    for ln in p.stdout.strip().split("\n"):
        _rows_close(ln, want[ln.split(",")[0]])


def test_batch_many_short_rows(ctx, tmp_path):
    """files with many short rows need more staging space than their size (every row is padded to 32 bytes): they are staged
    in a second round instead of silently leaving the batched path"""
    rng = np.random.default_rng(32)
    d = tmp_path / "short"
    d.mkdir()
    paths, texts = [], []
    for i in range(6):
        n, L = (1500, 6) if i % 2 == 0 else (40, 300)
        text = _upper(_random_text(rng, n, L, p_var=0.5, lower=0.0))
        with open(d / ("s%d.fa" % i), "w") as f:
            f.write("".join(">%d\n%s\n" % (r, text[r].tobytes().decode()) for r in range(n)))
        paths.append(str(d / ("s%d.fa" % i)))
        texts.append(text)
    batch = pf.api.Batch(ctx)
    info = batch.add_files(paths)
    assert [fi["status"] for fi in info] == [0] * 6 and sorted(fi["locus"] for fi in info) == list(range(6))
    batch.run(jc=False)
    for fi, text in zip(info, texts):
        got, want = batch.result(fi["locus"], 0, want_sfs=True), co.site_stats(text)
        assert (fi["n"], fi["L"]) == text.shape and (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"])
    batch.close()


@pytest.mark.parametrize("p_junk", [0.0, 0.01])
def test_batch_of_narrow_loci_tma_scan(ctx, monkeypatch, p_junk):
    """every locus of the batch has at most 128 rows: the batched site scan runs as pfa_batch_site_tma_kernel on the contiguous
    site records of the whole batch (slots of 128 / 96 sites that span many tiny loci, loci that span many slots, empty loci, a
    last slot that is not full; with non-ACGT symbols the validity plane travels too).  Against the C oracle, and the per-lane
    kernel (PFA_BATCH_TMA=0) must book the same numbers."""
    rng = np.random.default_rng(77 + int(p_junk * 100))
    shapes = [(100, 5000), (3, 1), (128, 700), (20, 0), (64, 33), (5, 2), (2, 129), (90, 4097), (128, 95), (17, 640), (1, 50)] + \
             [(int(rng.integers(2, 129)), int(rng.integers(1, 60))) for _ in range(40)]
    loci = []
    for i, (n, L) in enumerate(shapes):
        text = _random_text(rng, n, L, p_junk=p_junk, p_var=0.1) if L else np.zeros((n, 0), dtype=np.uint8)
        pops = None if i % 3 else [p for p in (list(range(0, n, 2)), list(range(n // 2, n)), list(range(n))) if p]
        loci.append((text, pops))
    results = []
    for tma in ("1", "0"):   # 1: forced (small batches take the per-lane kernel by default)
        monkeypatch.setenv("PFA_BATCH_TMA", tma)
        batch = pf.api.Batch(ctx)
        idx = [batch.add_rows(text, pops) for text, pops in loci]
        batch.run(jc=False)
        results.append([[batch.result(i, q, want_sfs=True) for q in range(len(pops or [0]))] for i, (text, pops) in zip(idx, loci)])
        batch.close()
    for (text, pops), got_tma, got_lane in zip(loci, *results):
        n, L = text.shape
        up = _upper(text)
        for q, rows in enumerate(pops or [list(range(n))]):
            want = co.site_stats(up, rows) if L else {"S": 0, "H": 0, "sfs": [0] * (len(rows) // 2)}
            for got in (got_tma[q], got_lane[q]):
                assert (got["n"], got["S"], got["H"], got["sfs"]) == (len(rows), want["S"], want["H"], want["sfs"]), (n, L, q)


def test_batch_codon_scan(ctx):
    """K4b: the segmented codon scan of the batched --dir --cds path == the single-alignment K4 == the C oracle, for loci of
    mixed shapes (lengths not divisible by 3, shorter than a codon, more rows than one tile column handles), populations and
    symbol content (escape symbols inside codon columns) in one batch; repeated scans of one staged batch agree"""
    rng = np.random.default_rng(321)
    shapes = [(20, 1000), (100, 5000), (3, 7), (1, 40), (33, 65), (128, 300), (129, 301), (700, 902), (2100, 257), (16, 0), (50, 31), (9, 2),
              (40, 3), (300, 1535)]
    batch = pf.api.Batch(ctx)
    loci = []
    for i, (n, L) in enumerate(shapes):
        junk = 0.0 if i % 3 == 0 else 0.02
        text = _random_text(rng, n, L, p_var=0.1, p_junk=junk) if L else np.zeros((n, 0), dtype=np.uint8)
        pops = None if i % 2 == 0 else [p for p in (list(range(0, n, 2)), list(range(n // 2, n)), list(range(n))) if p]
        loci.append((text, pops, batch.add_rows(text, pops)))
    batch.stage()
    for rep in range(2):
        batch.scan(jc=True, cds=True)
        for text, pops, idx in loci:
            n, L = text.shape
            up = _upper(text)
            for q, rows in enumerate(pops or [list(range(n))]):
                got = batch.result_cds(idx, q)
                want = co.cds_stats(up, rows) if L else {"nstops": 0, "missing": 0, "S_s": 0, "H_s": 0, "S_n": 0, "H_n": 0, "sum3_by_len": {}, "ssites": 0.0}
                for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
                    assert got[k] == want[k], (n, L, q, k, rep)
                assert math.isclose(got["ssites"], want["ssites"], rel_tol=1e-12) or got["ssites"] == want["ssites"]
                site = batch.result(idx, q)
                ws = co.site_stats(up, rows) if L else {"S": 0, "H": 0}
                assert (site["S"], site["H"]) == (ws["S"], ws["H"])
                nsites = (L - got["missing"]) - got["ssites"]
                ref = ctx.finalize([(len(rows), got["S_s"], got["H_s"], got["ssites"], True), (len(rows), got["S_n"], got["H_n"], nsites, True)])
                assert [got["poly_s"], got["poly_n"]] == ref, (n, L, q)
    batch.release()
    batch.close()


@pytest.mark.parametrize("n,L,gap_ppm,k", [(2000, 60_000, 100, 2), (10_000, 6_000, 100, 1), (10_000, 3_000, 2_000, 2), (700, 50_001, 30, 3),
                                          (4100, 9_000, 5, 2), (12_000, 3_003, 400, 1), (2000, 30_000, 100, 6), (10_000, 6_000, 10, 3)])
def test_sparse_validity_flags(ctx, monkeypatch, n, L, gap_ppm, k):
    """alignments with a FEW gaps: the TMA scans fetch only the flagged 128-row pieces of the validity plane (per-site flag
    words written by the encoders, pfa_slot_issue).  The gapped synthetic alignment is built twice -- on the device (generator +
    pfa_aln_poke_gaps) and from the numpy twin's text through the encoder -- the planes must agree bit for bit, and K2 / K4 of
    both must equal the C oracle on that text (gaps are alleles in the site scan, PolyFastA.py:256-258, and make a codon
    unclean, :301).  With PFA_VFLAG=0 (whole validity plane fetched) the results must not change."""
    seed = 11 + n
    text = synth.poke_gaps(synth.text_matrix(seed, n, L), seed, gap_ppm)
    assert (text == ord("-")).sum() > 0
    # six populations on groups of four lanes: the gap sites of populations 4 and 5 go through shared-memory atomics
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n // 2)), list(range(1, n, 3)), list(range(n // 2, n)), list(range(5, n, 7))][:k]
    dev = pf.Alignment.synthetic(ctx, n, L, seed)
    dev.poke_gaps(seed, gap_ppm)
    host = pf.Alignment.from_rows(ctx, text)
    assert dev.has_invalid and host.has_invalid
    for pl in range(3):
        assert np.array_equal(dev.plane(pl), host.plane(pl)), pl
    res = []
    for aln, flag in ((dev, "1"), (host, "1"), (host, "0")):
        monkeypatch.setenv("PFA_VFLAG", flag)
        aln.set_pops(pops)
        res.append((aln.site_stats(want_isvar=True), aln.cds_stats(want_labels=True), ctx.last_kernel))
    dev.free()
    host.free()
    for site, cds, _ in res:
        _check_site_cds(site, cds, text, pops, (n, L, gap_ppm))
    assert "HAS_V=1" in res[0][2]


@pytest.mark.parametrize("n,L,gap_ppm,k", [(2000, 30_000, 300, 2), (10_000, 4_002, 100, 1), (5000, 9_000, 50, 3)])
def test_validity_area_overflow(ctx, monkeypatch, n, L, gap_ppm, k):
    """the slots of the sparse-validity scans hold the validity records of a FRACTION of their sites (sized from the density
    of flagged sites); flagged sites beyond that are read from global memory when they are scanned.  Forced here: an eighth of
    the sites (PFA_VDIV=8) on alignments in which a third to most of the sites hold a gap -- most flagged sites overflow."""
    seed = 5 + n
    text = synth.poke_gaps(synth.text_matrix(seed, n, L), seed, gap_ppm)
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n // 2))][:k]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    res = []
    for vdiv in ("8", "2", "1"):
        monkeypatch.setenv("PFA_VDIV", vdiv)
        res.append((aln.site_stats(want_isvar=True), aln.cds_stats(want_labels=True)))
        assert "v_records_per_slot" in ctx.last_kernel
    aln.free()
    for site, cds in res:
        _check_site_cds(site, cds, text, pops, (n, L, gap_ppm))


@pytest.mark.parametrize("n,L", [(20, 300_000), (64, 200_000), (200, 100_000), (380, 60_000), (1100, 30_000)])
def test_narrow_records_many_variable_sites(ctx, n, L):
    """records handled by 1-2 lanes per site (every lane of a warp its own site, no shuffle inside a pass) with a third of the
    sites variable, three populations: lanes leave the second pass at different times, and the refill of the warp's
    shared-memory slot must wait for all of them (a missing warp barrier double-counted sites here)"""
    rng = np.random.default_rng(n + L)
    text = _random_text(rng, n, L, p_var=0.3, p_junk=0.0, lower=0.0)
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n))]
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    for rep in range(3):
        site = aln.site_stats()
        cds = aln.cds_stats()
        for q, rows in enumerate(pops):
            want = co.site_stats(text, rows)
            assert (site[q]["S"], site[q]["H"], site[q]["sfs"]) == (want["S"], want["H"], want["sfs"]), (n, L, q, rep)
            wc = co.cds_stats(text, rows)
            for k in ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len"):
                assert cds[q][k] == wc[k], (n, L, q, k, rep)
    aln.free()


@pytest.mark.parametrize("n,L,k", [(2000, 60_000, 2), (5000, 9_000, 1), (700, 30_003, 3), (2000, 30_000, 3), (10_000, 6_000, 2)])
def test_missing_data_runs_in_cds(ctx, n, L, k):
    """what a real CDS alignment holds: gaps aligned to codons, runs of N across codon borders, a few '?' and IUPAC codes, on top
    of the base variation -- the codon scan's missing-data-only path (valid rows of every site show one base; only the flagged
    cells are read) and the site scan's gap-only path against the C oracle"""
    rng = np.random.default_rng(n + L + k)
    text = synth.text_matrix(21, n, L).copy()
    for _ in range(400):
        r, c = int(rng.integers(0, n)), int(rng.integers(0, L // 3)) * 3
        text[r, c: c + 3 * int(rng.integers(1, 4))] = ord("-")
    for _ in range(150):
        r, c = int(rng.integers(0, n)), int(rng.integers(0, L))
        text[r, c: c + int(rng.integers(1, 12))] = ord("N")
    rr, cc = rng.integers(0, n, 60), rng.integers(0, L, 60)
    text[rr, cc] = np.frombuffer(b"?RY", dtype=np.uint8)[rng.integers(0, 3, 60)]
    text[: n // 2, 300:306] = ord("-")      # a gap carried by half of the rows: more flagged cells than the short path takes
    text[:, 600:603] = ord("-")             # a codon column nobody shows
    # gap-only columns are settled in pass 1 when every population keeps a clean row; here no row is clean (first half
    # misses site 900, second half site 901) although each site shows one base among its valid rows, ...
    text[:, 900:903] = np.frombuffer(b"ACG", dtype=np.uint8)
    text[: n // 2, 900] = ord("-")
    text[n // 2:, 901] = ord("N")
    # ... and here the third population (rows n/3 .. n/2) loses all its rows while the others keep theirs
    text[:, 1200:1203] = np.frombuffer(b"TGA", dtype=np.uint8)
    text[n // 3: n // 2, 1201] = ord("-")
    pops = [list(range(n)), list(range(0, n, 2)), list(range(n // 3, n // 2))][:k]
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.has_invalid
    aln.set_pops(pops)
    site = aln.site_stats(want_isvar=True)
    cds = aln.cds_stats(want_labels=True)
    aln.free()
    _check_site_cds(site, cds, text, pops, (n, L, k))
