"""--devices of the command line: a list of CUDA ordinals or `all`, and the refusals argparse reports (no GPU needed: the
number of visible devices is stubbed)."""
import pytest

from solaraxionraytracing_b200 import __main__ as cli


@pytest.fixture
def eight_gpus(monkeypatch):
    monkeypatch.setattr(cli, "visible_devices", lambda: 8)


def test_parse_devices_list_and_all():
    assert cli.parse_devices("0,1,2,3", 8) == [0, 1, 2, 3]
    assert cli.parse_devices("5,2", 8) == [5, 2]
    assert cli.parse_devices("all", 4) == [0, 1, 2, 3]
    assert cli.parse_devices("all", 1) == [0]


@pytest.mark.parametrize("text,n,match", [("1,1", 8, "listed twice"), ("0,2,0", 8, "listed twice"),
                                          ("8", 8, "does not exist"), ("-1", 8, "does not exist"),
                                          ("0,1", 1, "does not exist"), ("all", 0, "no CUDA device"),
                                          ("0;1", 8, "comma-separated"), ("", 8, "comma-separated")])
def test_parse_devices_refusals(text, n, match):
    with pytest.raises(ValueError, match=match):
        cli.parse_devices(text, n)


def test_parse_args(eight_gpus):
    assert cli.parse_args(["--devices", "0,1,2,3"]).devices == [0, 1, 2, 3]
    assert cli.parse_args(["--devices", "all"]).devices == list(range(8))
    assert cli.parse_args(["--devices", "3", "--device", "0"]).devices == [3]   # --device at its default
    plain = cli.parse_args([])
    assert plain.devices is None and plain.device == 0


@pytest.mark.parametrize("argv,match", [(["--devices", "0,0"], "listed twice"),
                                        (["--devices", "9"], "does not exist"),
                                        (["--devices", "0,1", "--device", "2"], "exclude each other")])
def test_parse_args_refusals(eight_gpus, capsys, argv, match):
    with pytest.raises(SystemExit) as e:
        cli.parse_args(argv)
    assert e.value.code == 2
    assert match in capsys.readouterr().err
