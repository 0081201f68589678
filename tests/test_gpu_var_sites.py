"""The site scan over the list of sites where rows differ: on sparse pure-ACGT shapes the TMA site scan fetches only the
listed sites (ctx.last_kernel names the list, "sites=listed/ns").  Results against the generator's closed form and the C
oracle: S, H and the SFS of one to six populations (some not covering every row), isvar, the per-site H, windows, the codon
scan after it, gaps poked in after a first scan (the list is dropped and rebuilt), IUPAC codes, an all-monomorphic shard
through the exchange, and the divergence and haplotype scans that share the list."""
import numpy as np
import pytest
import torch

import haplotype_oracle as ho
import polyfasta_b200 as pf
from oracle import c_oracle as co
from polyfasta_b200 import parallel, synth
from test_gpu_divergence import _check_against_oracle

pytestmark = pytest.mark.gpu

SEED = 11
CDS_KEYS = ("nstops", "missing", "S_s", "H_s", "S_n", "H_n", "sum3_by_len")


@pytest.fixture(scope="module")
def ctx():
    return pf.default_context(0)


def _listed(ctx):
    return " sites=" in ctx.last_kernel


def _pops(n, k):
    """k populations; from two on, some rows belong to none and some to two"""
    if k == 1:
        return [list(range(n))]
    if k == 2:
        return [list(range(0, n // 2)), list(range(n // 3, n - 7))]
    return [list(range(q, n - 3, k + 1)) for q in range(k - 1)] + [list(range(0, n // 5))]


def _check_sites(aln, text, pops, what):
    got = aln.site_stats(want_isvar=True, want_hsite=True)
    for q, rows in enumerate(pops):
        want = co.site_stats(text, rows, per_site=True)
        g = got[q]
        assert (g["S"], g["H"], g["sfs"]) == (want["S"], want["H"], want["sfs"]), (what, q)
        assert np.array_equal(g["isvar"], want["isvar"]), (what, q)
        assert np.array_equal(g["hsite"], want["hsite"]), (what, q)
    return got


@pytest.mark.parametrize("p_seg_ppm", [0, 1_000, 50_000, 300_000])
@pytest.mark.parametrize("n", [1281, 2000, 10000, 20480])
def test_synthetic_closed_form(ctx, n, p_seg_ppm):
    """records of 11 to 160 chunks; at most 5 % variable sites takes the list, a list of no site included"""
    L = 40_000 if n <= 2000 else 8_000
    aln = pf.Alignment.synthetic(ctx, n, L, SEED, p_seg_ppm)
    got = aln.site_stats()[0]
    kern = ctx.last_kernel
    want = synth.expected_site_stats(SEED, n, L, p_seg_ppm)
    assert (got["S"], got["H"], got["sfs"]) == (want["S"], want["H"], want["sfs"])
    if p_seg_ppm <= 50_000:
        assert kern.endswith(" sites=%d/%d" % (want["S"], L)), kern
    # a second scan reuses the list
    again = aln.site_stats()[0]
    assert (again["S"], again["H"], again["sfs"]) == (got["S"], got["H"], got["sfs"])
    aln.free()


@pytest.mark.parametrize("k", [1, 2, 6])
@pytest.mark.parametrize("n", [2000, 10000])
def test_populations_per_site_windows_cds(ctx, n, k):
    """isvar, per-site H and windows on the list path, then the codon scan of the same alignment"""
    L = 6_000
    text = synth.text_matrix(SEED, n, L, 50_000)
    pops = _pops(n, k)
    aln = pf.Alignment.synthetic(ctx, n, L, SEED, 50_000)
    aln.set_pops(pops)
    got = _check_sites(aln, text, pops, (n, k))
    assert _listed(ctx), ctx.last_kernel
    W, S = 1000, 500
    counts = aln.site_window_counts(W, S)
    for q in range(k):
        for w in range(counts.shape[1]):
            s0, s1 = w * S, min(w * S + W, L)
            assert counts[q, w, 0] == int(got[q]["isvar"][s0:s1].sum()), (q, w)
            assert counts[q, w, 1] == int(got[q]["hsite"][s0:s1].sum()), (q, w)
    cds = aln.cds_stats()
    for q, rows in enumerate(pops):
        want = co.cds_stats(text, rows)
        assert all(cds[q][key] == want[key] for key in CDS_KEYS), q
    aln.free()


@pytest.mark.parametrize("gap_ppm", [10, 100])
@pytest.mark.parametrize("n", [2000, 10000])
def test_gaps_after_first_scan(ctx, n, gap_ppm):
    """poke_gaps writes the planes after the list was built: the next scans see the gap sites (the site scan walks every site
    of a shard with invalid rows; the divergence scan takes the rebuilt list)"""
    L = 6_000
    aln = pf.Alignment.synthetic(ctx, n, L, SEED, 50_000)
    aln.site_stats()
    assert _listed(ctx), ctx.last_kernel
    aln.poke_gaps(SEED, gap_ppm)
    text = synth.poke_gaps(synth.text_matrix(SEED, n, L, 50_000), SEED, gap_ppm)
    pops = _pops(n, 2)
    aln.set_pops(pops)
    _check_sites(aln, text, pops, (n, gap_ppm))
    assert not _listed(ctx), ctx.last_kernel
    _check_against_oracle(aln, text, pops, (n, gap_ppm))
    cds = aln.cds_stats()
    for q, rows in enumerate(pops):
        want = co.cds_stats(text, rows)
        assert all(cds[q][key] == want[key] for key in CDS_KEYS), q
    aln.free()


def _sparse_junk_text(rng, n, L):
    """ACGT with 3 % variable columns, plus columns of gaps / N / ? / IUPAC codes: some with a few such rows, some where
    every row shows one code, some where every row shows an IUPAC code but not the same one (only the escape bytes differ)"""
    anc = rng.integers(0, 4, L)
    mat = np.frombuffer(b"ACGT", dtype=np.uint8)[np.repeat(anc[None, :], n, axis=0)].copy()
    var = np.flatnonzero(rng.random(L) < 0.03)
    for c in var:
        rows = rng.choice(n, int(rng.integers(1, n)), replace=False)
        mat[rows, c] = b"ACGT"[(anc[c] + 1 + int(rng.integers(0, 3))) % 4]
    junk = np.frombuffer(b"-N?RYKM.", dtype=np.uint8)
    cols = rng.choice(L, 60, replace=False)
    for i, c in enumerate(cols):
        if i % 3 == 0:
            rows = rng.choice(n, int(rng.integers(1, 20)), replace=False)
            mat[rows, c] = junk[rng.integers(0, len(junk), len(rows))]
        elif i % 3 == 1:
            mat[:, c] = junk[i % len(junk)]
        else:
            mat[:, c] = ord("R")
            mat[rng.choice(n, int(rng.integers(1, n)), replace=False), c] = ord("Y")
    return np.ascontiguousarray(mat)


@pytest.mark.parametrize("n", [2000, 10000])
def test_iupac_from_rows(ctx, n):
    rng = np.random.default_rng(n + 17)
    L = 3_000
    text = _sparse_junk_text(rng, n, L)
    aln = pf.Alignment.from_rows(ctx, text)
    assert aln.has_invalid and aln.num_escapes > 0
    pops = _pops(n, 2)
    aln.set_pops(pops)
    _check_sites(aln, text, pops, n)
    assert not _listed(ctx), ctx.last_kernel
    _check_against_oracle(aln, text, pops, n)
    aln.free()


def test_all_monomorphic_exchange(ctx):
    """a shard without a variable site: an empty list, the kernel still runs the exchange"""
    n, L = 2000, 9_000
    aln = pf.Alignment.synthetic(ctx, n, L, SEED, 0)
    x = parallel.connect_exchange(ctx, aln.site_len())
    d_out = torch.full((aln.site_len(),), -1, dtype=torch.int64, device="cuda:0")
    torch.cuda.synchronize()
    aln.site_stats_xchg(x, d_out.data_ptr())
    ctx.sync()
    assert ctx.last_kernel.endswith(" sites=0/%d" % L), ctx.last_kernel
    assert not x.timed_out() and d_out.cpu().tolist() == [0] * aln.site_len()
    x.close()
    aln.free()


@pytest.mark.parametrize("n", [1281, 2000])
def test_dense_alignment_scans_dense(ctx, n):
    """uniform random text: every site varies, the scan reads every record"""
    rng = np.random.default_rng(n)
    text = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, (n, 2000))]
    aln = pf.Alignment.from_rows(ctx, np.ascontiguousarray(text))
    _check_sites(aln, text, [list(range(n))], n)
    assert not _listed(ctx), ctx.last_kernel
    aln.free()


@pytest.mark.parametrize("junk", [False, True])
def test_divergence_haplotypes_share_the_list(ctx, junk):
    """the divergence and haplotype scans after a site scan that built the list, against their oracles"""
    n, L = 2000, 2_500
    rng = np.random.default_rng(5 + junk)
    text = _sparse_junk_text(rng, n, L) if junk else synth.text_matrix(SEED, n, L, 50_000)
    pops = _pops(n, 2)
    aln = pf.Alignment.from_rows(ctx, text)
    aln.set_pops(pops)
    _check_sites(aln, text, pops, junk)
    assert _listed(ctx) != junk, ctx.last_kernel
    _check_against_oracle(aln, text, pops, junk)
    rows = [bytes(r).decode("latin-1") for r in text]
    assert aln.haplotype_classes()[0].tolist() == ho.rep(rows)
    hap = aln.haplotypes()[0]
    for q, members in enumerate(pops):
        want, got = ho.pop_stats(rows, members), hap["pops"][q]
        assert (got["n"], got["h"], got["s2"], got["s3"]) == (want["n"], want["h"], want["s2"], want["s3"])
    aln.free()
