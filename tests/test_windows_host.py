"""Sliding windows without a GPU: the window count and the CLI's argument errors."""
import pytest

from polyfasta_b200 import api, cli
from polyfasta_b200._lib import lib


def _windows_loop(L, W, step):
    """the windows by their definition: starts 0, step, 2 step, ... below L; the first window that reaches L is the last"""
    out = []
    start = 0
    while start < L:
        end = min(start + W, L)
        out.append((start, end))
        if end == L:
            break
        start += step
    return out


CASES = [(L, W, s) for L in (0, 1, 2, 9, 10, 11, 29, 30, 31, 100, 1000, 1001, 999)
         for (W, s) in ((10, 10), (30, 10), (7, 3), (3, 7), (5, 20), (1, 1), (2000, 1), (2000, 500), (1, 2))]


@pytest.mark.parametrize("L,W,step", CASES)
def test_window_count_matches_definition(L, W, step):
    want = len(_windows_loop(L, W, step))
    assert api.window_count(L, W, step) == want
    assert lib().pfa_window_count(L, W, step) == want


def test_window_count_formula_large():
    L = 10_000_000
    for W, s in ((10_000, 10_000), (100_000, 10_000), (1000, 1000), (7, 3), (3, 7)):
        want = min(1 + -(-max(0, L - W) // s), -(-L // s))
        assert api.window_count(L, W, s) == want


@pytest.mark.parametrize("L,W,step", [(10, 0, 1), (10, 1, 0), (10, -3, 2), (-1, 5, 5)])
def test_window_count_bad_arguments(L, W, step):
    assert lib().pfa_window_count(L, W, step) == -1
    with pytest.raises(ValueError):
        api.window_count(L, W, step)


@pytest.mark.parametrize("argv", [["-f", "x.fa", "--window", "10", "--cds"],
                                  ["-f", "x.fa", "--step", "5"],
                                  ["-f", "x.fa", "--window", "0"],
                                  ["-f", "x.fa", "--window", "-4"],
                                  ["-f", "x.fa", "--window", "10", "--step", "0"],
                                  ["-f", "x.fa", "--window", "10", "--step", "-1"]])
def test_cli_window_argument_errors(argv, capsys):
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    err = capsys.readouterr().err
    assert "--window" in err or "--step" in err


def test_cli_window_parser_defaults():
    p = cli.build_parser()
    a = p.parse_args(["-f", "x.fa", "--window", "100"])
    assert cli.check_window_args(p, a) == (100, 100)
    a = p.parse_args(["-f", "x.fa", "--window", "100", "--step", "25"])
    assert cli.check_window_args(p, a) == (100, 25)
    a = p.parse_args(["-f", "x.fa"])
    assert cli.check_window_args(p, a) is None
