"""`main.py --defense` rejects malformed --beta and unsupported --MI_type values before any device work (no GPU needed)."""
import pytest


@pytest.mark.parametrize("beta", [None, "0.1,0.1,0.1,0.1", "0.1,0.1,0.1,0.1,0.1,0.1", "0.1,0.1,x,0.1,0.1",
                                  "0.1,0.1,nan,0.1,0.1", ""])
def test_defense_rejects_malformed_beta(beta):
    from mcgra_b200 import main as cli
    argv = ["--dataset", "synthetic:50:8:2", "--defense"] + ([] if beta is None else ["--beta", beta])
    with pytest.raises(ValueError, match="--beta"):
        cli.main(argv)


@pytest.mark.parametrize("mi", ["KDE", "IXZ", "HSIC"])
def test_defense_rejects_unsupported_mi_type(mi):
    from mcgra_b200 import main as cli
    with pytest.raises(SystemExit):
        cli.main(["--dataset", "synthetic:50:8:2", "--defense", "--beta", "0.1,0.1,0.1,0.1,0.1", "--MI_type", mi])


def test_parse_beta_keys():
    from mcgra_b200 import main as cli
    assert cli.parse_beta("1,2,3,4,5e-3") == {"layer-0": 1.0, "layer-1": 2.0, "layer-2": 3.0, "layer_inter-0": 4.0,
                                              "layer_inter-1": 5e-3}
