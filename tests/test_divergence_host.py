"""Divergence between populations without a GPU: the oracles against a literal double loop, the float formulas, and the CLI's
argument errors and headers."""
import math

import numpy as np
import pytest

from divergence_oracle import divergence, divergence_c, finalize, pairs
from polyfasta_b200 import api, cli


def _random_seqs(rng, n, L, alphabet=b"ACGTACGTACGT-N?RYKMacgtn"):
    mat = np.frombuffer(alphabet, dtype=np.uint8)[rng.integers(0, len(alphabet), (n, L))]
    up = np.where((mat >= 97) & (mat <= 122), mat - 32, mat).astype(np.uint8)
    return up, [bytes(r).decode("latin-1") for r in up]


def _double_loop(seqs, X, Y, L):
    return sum(1 for i in X for j in Y for p in range(L) if seqs[i][p] != seqs[j][p])


@pytest.mark.parametrize("seed", range(12))
def test_python_oracle_against_double_loop(seed):
    """gaps, N, ?, IUPAC codes and lower case (folded to upper case as the reader does); overlapping and identical populations"""
    rng = np.random.default_rng(seed)
    n, L = int(rng.integers(2, 14)), int(rng.integers(1, 40))
    up, seqs = _random_seqs(rng, n, L)
    X = sorted(set(rng.integers(0, n, int(rng.integers(1, n + 1))).tolist()))
    Y = sorted(set(rng.integers(0, n, int(rng.integers(1, n + 1))).tolist()))
    for a, b in ((X, Y), (X, X), (Y, X), (list(range(n)), X)):
        rx, ry = [seqs[i] for i in a], [seqs[i] for i in b]
        D, ds = divergence(rx, ry, L, per_site=True)
        assert D == _double_loop(seqs, a, b, L) == sum(ds)
        for p in range(L):
            assert ds[p] == sum(1 for i in a for j in b if seqs[i][p] != seqs[j][p])


@pytest.mark.parametrize("seed", range(6))
def test_c_oracle_against_python_oracle(seed):
    rng = np.random.default_rng(100 + seed)
    n, L = int(rng.integers(2, 60)), int(rng.integers(1, 300))
    up, seqs = _random_seqs(rng, n, L)
    X = list(range(0, n, 2))
    Y = list(range(n // 3, n))
    D, ds = divergence([seqs[i] for i in X], [seqs[i] for i in Y], L, per_site=True)
    Dc, dsc = divergence_c(up, X, Y, per_site=True)
    assert Dc == D and dsc.tolist() == ds
    assert divergence_c(up, X, X) == divergence([seqs[i] for i in X], [seqs[i] for i in X], L)


def test_identical_rows_do_not_diverge():
    seqs = ["ACGTRY-N?", "ACGTRY-N?"]
    assert divergence(seqs[:1], seqs[1:], 9) == 0
    assert divergence(["R"], ["Y"], 1) == 1 and divergence(["R", "R"], ["Y"], 1) == 2


def test_finalize_formulas():
    # plain: dxy = D / (nx ny) / L, da = dxy - (pi_x + pi_y) / 2, fst = 1 - hw / dxy
    dxy, da, fst = finalize(4, 5, 30, 100, 0.01, 0.03, False)
    assert dxy == (30 / 20) / 100
    assert da == dxy - 0.5 * (0.01 + 0.03)
    assert fst == 1 - 0.02 / dxy
    # Jukes-Cantor on dxy, with K5's rule: a non-positive argument keeps the uncorrected value
    d_jc = finalize(4, 5, 30, 100, 0.01, 0.03, True)[0]
    assert d_jc == -0.75 * math.log(1 - (4. / 3.) * ((30 / 20) / 100))
    assert finalize(1, 1, 100, 100, 0.0, 0.0, True)[0] == 1.0   # x = 1 - 4/3 < 0
    # no differences: F_ST undefined
    assert finalize(3, 3, 0, 50, 0.0, 0.0, False) == (0.0, 0.0, "NA")
    assert finalize(3, 3, 0, 50, 0.01, 0.0, False) == (0.0, -0.005, "NA")
    # an empty population or no columns: every field undefined
    assert finalize(0, 3, 0, 50, 0.0, 0.0, False) == ("NA", "NA", "NA")
    assert finalize(2, 3, 0, 0, 0.0, 0.0, False) == ("NA", "NA", "NA")


def test_pair_order():
    assert pairs(4) == api.pop_pairs(4) == [(0, 1), (0, 2), (0, 3), (1, 2), (1, 3), (2, 3)]
    assert api.pop_pairs(1) == [] and len(api.pop_pairs(64)) == 2016


@pytest.mark.parametrize("argv,needle", [(["-f", "x.fa", "--dxy"], "-p"),
                                         (["-f", "x.fa", "--dxy", "-p", "a,b", "--cds"], "--cds")])
def test_cli_dxy_argument_errors(argv, needle, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    err = capsys.readouterr().err
    assert "--dxy" in err and needle in err


def test_cli_dxy_headers(tmp_path, capsys):
    assert cli.HEADER_DXY == "file,seqlen,pop1,pop2,N1,N2,dxy,da,Fst"
    assert cli.HEADER_DXY_WINDOWS == "file,window_start,window_end,seqlen,pop1,pop2,N1,N2,dxy,da,Fst"
    for windows, want in ((False, cli.HEADER_DXY), (True, cli.HEADER_DXY_WINDOWS)):
        cli.Sink("", False).header(False, windows, True)
        assert capsys.readouterr().out == want + "\n"
        out = tmp_path / "h.csv"
        cli.Sink(str(out), False).header(False, windows, True)
        assert out.read_text() == want + "\n"


def test_cli_dxy_rows_from_results():
    found = [("p0", None, 3), ("p1", None, 2), ("p2", None, 4)]
    fins = [{"dxy": dxy, "da": da, "fst": fst} for dxy, da, fst in ((0.25, 0.125, 0.5), (0.0, 0.0, "NA"), (1.5, -0.25, 0.75))]
    assert cli.dxy_rows("f.fa", found, [{"start": 0, "end": 10, "pairs": fins}], False) == [
        "f.fa,10,p0,p1,3,2,0.25,0.125,0.5", "f.fa,10,p0,p2,3,4,0.0,0.0,NA", "f.fa,10,p1,p2,2,4,1.5,-0.25,0.75"]
    assert cli.dxy_rows("f.fa", found[:2], [{"start": 5, "end": 9, "pairs": fins[:1]}], True) == ["f.fa,6,9,4,p0,p1,3,2,0.25,0.125,0.5"]
