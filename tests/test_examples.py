"""examples/demos.py: argument parsing and the data-set loaders (no device needed for either)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "examples"))
# GINGR_REFERENCE: a checkout of the Scala GiNGR project, whose example data files are read here
REF_DATA = os.path.join(os.environ["GINGR_REFERENCE"], "examples", "data") if os.environ.get("GINGR_REFERENCE") else ""


def test_demo_cli_and_synthetic_dataset(capsys):
    import demos
    with pytest.raises(SystemExit) as e:
        demos.main(["--help"])
    assert e.value.code == 0 and "multires" in capsys.readouterr().out
    with pytest.raises(SystemExit):
        demos.main(["nonsense"])
    R = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    a = demos.load_dataset("synthetic", None)
    b = demos.load_dataset("synthetic", None, (R, np.array([1.0, 2.0, 3.0])))
    assert a["ref"][0].shape == (2000, 3) and a["target"][1].max() < len(a["target"][0]) and a["ref_lms"] is None
    assert np.allclose(b["target"][0], a["target"][0] @ R.T + [1.0, 2.0, 3.0])


@pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="GINGR_REFERENCE does not name a GiNGR checkout")
def test_demo_datasets_from_the_reference_files():
    import demos
    f = demos.load_dataset("femur", REF_DATA)
    assert f["ref"][0].shape == (1622, 3) and f["target"][0].shape[1] == 3 and f["kernel"] == (50.0, 70.0)
    assert {l.id for l in f["ref_lms"]} == {l.id for l in f["target_lms"]} and len(f["ref_lms"]) == 6
    off = (np.eye(3), np.array([50.0, 50.0, 50.0]))
    g = demos.load_dataset("femur", REF_DATA, off)
    assert np.allclose(g["target"][0], f["target"][0] + 50.0)
    assert np.allclose(g["target_lms"][0].point, f["target_lms"][0].point + 50.0)
    b = demos.load_dataset("bunny", REF_DATA, off)
    assert b["ref"][0].shape == (35393, 3) and b["target"][0].shape == (35393, 3) and b["kernel"] == (20.0, 40.0)
    d = np.linalg.norm(b["target"][0] - 50.0 - b["ref"][0], axis=1)
    assert 0.0 < d.mean() < 20.0                                  # the synthetic stand-in for the missing target.ply
