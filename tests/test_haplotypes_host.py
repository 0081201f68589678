"""Haplotype statistics without a GPU: the oracle against a literal pair loop, the CLI's argument errors and headers, the C-ABI
exports, api.meet_classes and api.haplotype_results."""
from fractions import Fraction

import numpy as np
import pytest

import haplotype_oracle as ho
from polyfasta_b200 import _lib, api, cli


def _random_rows(rng, n, L, alphabet="ACGT", founders=4):
    base = ["".join(rng.choice(list(alphabet), L)) for _ in range(founders)]
    rows = []
    for _ in range(n):
        r = list(base[rng.integers(0, founders)])
        if rng.random() < 0.3:
            r[rng.integers(0, L)] = rng.choice(list(alphabet))
        rows.append("".join(r))
    return rows


@pytest.mark.parametrize("seed", range(6))
def test_oracle_against_pair_loop(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 40))
    rows = _random_rows(rng, n, 12, alphabet="ACGTacgt-N?RY")
    pops = [list(range(n)), [i for i in range(n) if i % 3], [0, n - 1]]
    rep = ho.rep(rows)
    for r, x in enumerate(rep):
        assert x <= r and rows[x].upper() == rows[r].upper()
        assert all(rows[j].upper() != rows[r].upper() for j in range(x))
    for members in pops:
        st = ho.pop_stats(rows, members)
        m = len(members)
        assert st["n"] == m and st["h"] == len({rows[i].upper() for i in members})
        pairs = ho.differing_pairs(rows, members)
        assert st["s2"] == m * m - 2 * pairs   # Hd C(n,2) = pairs, exactly, before the one rounding
        assert st["Hd"] == (pairs / (m * (m - 1) // 2) if m > 1 else "NA")


def test_oracle_single_row_and_case():
    st = ho.pop_stats(["ACGT"], [0])
    assert (st["n"], st["h"], st["Hd"], st["Hd_var"]) == (1, 1, "NA", "NA")
    assert ho.rep(["acgt", "ACGT", "ACGA", "AcGa"]) == [0, 0, 2, 2]


@pytest.mark.parametrize("argv", [["-f", "x.fa", "--haplotypes", "--cds"],
                                  ["-f", "x.fa", "-p", "a,b", "--haplotypes", "--dxy"],
                                  ["-f", "x.fa", "--haplotypes", "--cds", "--window", "9"]])
def test_cli_haplotype_argument_errors(argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    assert "--haplotypes" in capsys.readouterr().err


def test_cli_haplotype_headers(capsys):
    assert cli.HEADER_HAP == "file,seqlen,pop,N,haplotypes,Hd,Hd_var"
    assert cli.HEADER_HAP_WINDOWS == "file,window_start,window_end,seqlen,pop,N,haplotypes,Hd,Hd_var"
    cli.Sink("", False).header(False, False, False, True)
    cli.Sink("", False).header(False, True, False, True)
    assert capsys.readouterr().out.splitlines() == [cli.HEADER_HAP, cli.HEADER_HAP_WINDOWS]


def test_haplotype_exports():
    for name in ("pfa_haplotypes_device", "pfa_haplotypes"):
        assert name in _lib.EXPORTS
        assert hasattr(_lib.lib(), name)


def _canonical(keys):
    """rep of rows from per-row hashable keys"""
    first = {}
    return [first.setdefault(k, i) for i, k in enumerate(keys)]


@pytest.mark.parametrize("seed", range(8))
def test_meet_classes_random_partitions(seed):
    rng = np.random.default_rng(100 + seed)
    nwin, n = int(rng.integers(1, 5)), int(rng.integers(1, 300))
    shards = int(rng.integers(1, 4))
    labels = rng.integers(0, int(rng.integers(1, 6)), (shards, nwin, n))
    reps = [np.array([_canonical(labels[s, w]) for w in range(nwin)], dtype=np.int32) for s in range(shards)]
    want = np.array([_canonical(list(zip(*[labels[s, w] for s in range(shards)]))) for w in range(nwin)], dtype=np.int32)
    got = api.meet_classes(reps)
    assert got.dtype == np.int32 and np.array_equal(got, want)


def test_meet_classes_identity_one_class_and_three_way():
    n = 50
    ident = np.arange(n, dtype=np.int32)[None, :]
    one = np.zeros((1, n), dtype=np.int32)
    a = np.array([_canonical([i % 2 for i in range(n)])], dtype=np.int32)
    b = np.array([_canonical([i % 3 for i in range(n)])], dtype=np.int32)
    c = np.array([_canonical([i % 5 for i in range(n)])], dtype=np.int32)
    assert np.array_equal(api.meet_classes([a]), a)
    assert np.array_equal(api.meet_classes([a, one]), a)
    assert np.array_equal(api.meet_classes([one, a]), a)
    assert np.array_equal(api.meet_classes([ident, a]), ident)
    assert np.array_equal(api.meet_classes([one, one]), one)
    want = np.array([_canonical([i % 30 for i in range(n)])], dtype=np.int32)
    assert np.array_equal(api.meet_classes([a, b, c]), want)


def _check_against_oracle(rows, rep, pops, start, end, entry):
    for q, members in enumerate(pops):
        want = ho.pop_stats(rows, members)
        got = entry["pops"][q]
        assert (got["n"], got["h"], got["s2"], got["s3"]) == (want["n"], want["h"], want["s2"], want["s3"])
        if want["n"] == 1:
            assert got["Hd"] == "NA" and got["Hd_var"] == "NA"
        else:
            assert got["Hd"] == want["Hd"]
            assert abs(Fraction(got["Hd_var"]) - want["Hd_var"]) <= Fraction(1, 10 ** 12) * abs(want["Hd_var"])


def test_haplotype_results_hand_made():
    rows = ["AAAA", "AAAA", "CCCC", "AAAA", "GGGG", "CCCC", "TTTT"]
    rep = np.array([ho.rep(rows)], dtype=np.int32)
    assert rep.tolist() == [[0, 0, 2, 0, 4, 2, 6]]
    pops = [list(range(7)), [0, 1, 3], [2], [2, 4, 5, 6]]
    masks = api.rows_to_masks(1, pops)
    res = api.haplotype_results(rep, masks, [len(p) for p in pops], 4, 4, 4)
    assert len(res) == 1 and (res[0]["start"], res[0]["end"], res[0]["seqlen"]) == (0, 4, 4)
    _check_against_oracle(rows, rep, pops, 0, 4, res[0])
    p = res[0]["pops"]
    assert (p[0]["h"], p[0]["s2"], p[0]["s3"]) == (4, 9 + 4 + 1 + 1, 27 + 8 + 1 + 1)
    assert p[0]["Hd"] == (49 - 15) / 42
    assert p[1]["Hd"] == 0.0 and p[1]["Hd_var"] == 0.0 and p[1]["h"] == 1
    assert (p[2]["n"], p[2]["h"], p[2]["Hd"], p[2]["Hd_var"]) == (1, 1, "NA", "NA")


def test_haplotype_results_windows_and_all_rows():
    rng = np.random.default_rng(7)
    n, L, W, S = 40, 23, 7, 5
    rows = _random_rows(rng, n, L, alphabet="AC", founders=6)
    nwin = api.window_count(L, W, S)
    spans = [(i * S, min(i * S + W, L)) for i in range(nwin)]
    rep = np.array([ho.rep(ho.window_rows(rows, s, e)) for s, e in spans], dtype=np.int32)
    res = api.haplotype_results(rep, None, [n], L, W, S)
    assert [(w["start"], w["end"], w["seqlen"]) for w in res] == [(s, e, e - s) for s, e in spans]
    for (s, e), w in zip(spans, res):
        _check_against_oracle(ho.window_rows(rows, s, e), rep, [list(range(n))], s, e, w)


def test_hap_rows_format():
    found = [("p1", None, 3), ("p2", None, 1)]
    wins = [{"start": 0, "end": 10, "seqlen": 10, "pops": [{"h": 2, "Hd": 0.5, "Hd_var": 0.25}, {"h": 1, "Hd": "NA", "Hd_var": "NA"}]}]
    assert cli.hap_rows("f.fa", found, wins, False) == ["f.fa,10,p1,3,2,0.5,0.25", "f.fa,10,p2,1,1,NA,NA"]
    assert cli.hap_rows("f.fa", found, wins, True) == ["f.fa,1,10,10,p1,3,2,0.5,0.25", "f.fa,1,10,10,p2,1,1,NA,NA"]
