"""--cds --window without a GPU: the argument rules, the header and the exported entry points."""
import pytest

from polyfasta_b200 import _lib, api, cli


@pytest.mark.parametrize("argv", [["-f", "x.fa", "--cds", "--window", "10"],
                                  ["-f", "x.fa", "--cds", "--window", "40"],
                                  ["-f", "x.fa", "--cds", "--window", "9", "--step", "4"],
                                  ["-f", "x.fa", "--cds", "--window", "8", "--step", "9"],
                                  ["-f", "x.fa", "--cds", "--window", "0"],
                                  ["-f", "x.fa", "--cds", "--window", "9", "--step", "-3"]])
def test_cli_cds_window_not_whole_codons(argv, capsys):
    """window and step are whole codons under --cds; anything else is a parser error that names --window"""
    with pytest.raises(SystemExit) as e:
        cli.main(argv)
    assert e.value.code == 2
    assert "--window" in capsys.readouterr().err


def test_cli_cds_window_parser_accepts_multiples_of_three():
    p = cli.build_parser()
    a = p.parse_args(["-f", "x.fa", "--cds", "--window", "300"])
    assert cli.check_window_args(p, a) == (300, 300)
    a = p.parse_args(["-f", "x.fa", "--cds", "--window", "30000", "--step", "15000"])
    assert cli.check_window_args(p, a) == (30000, 15000)
    a = p.parse_args(["-f", "x.fa", "--window", "10", "--step", "7"])   # without --cds any positive W and S
    assert cli.check_window_args(p, a) == (10, 7)


def test_cli_cds_dxy_still_an_error(capsys):
    for argv in (["-f", "x.fa", "--cds", "--dxy", "-p", "a,b"], ["-f", "x.fa", "--cds", "--dxy", "-p", "a,b", "--window", "9"]):
        with pytest.raises(SystemExit) as e:
            cli.main(argv)
        assert e.value.code == 2
    assert "--dxy" in capsys.readouterr().err


def test_cds_window_header():
    assert cli.HEADER_CDS_WINDOWS.split(",") == (["file", "window_start", "window_end"] + cli.HEADER_CDS.split(",")[1:])
    assert api.PFA_CDS_WIN_LEN == _lib.PFA_CDS_LEN + 1 == 72


def test_cds_window_entry_points_exported():
    L = _lib.lib()
    for name in ("pfa_cds_windows_device", "pfa_cds_windows"):
        assert name in _lib.EXPORTS and hasattr(L, name)
