"""Wire / disk formats (gingr_b200/io.py, SURVEY.md 8f item 3): round trips, the reference's JSON layouts, and -- when
the reference tree is mounted -- its own example files (the femur fixtures of tests/golden were generated from them)."""
import pathlib
import dataclasses
import json
import os

import numpy as np
import pytest

# GINGR_REFERENCE: a checkout of the Scala GiNGR project, whose example data files are read here
REF_DATA = os.path.join(os.environ["GINGR_REFERENCE"], "examples", "data") if os.environ.get("GINGR_REFERENCE") else ""
needs_reference = pytest.mark.skipif(not os.path.isdir(REF_DATA), reason="GINGR_REFERENCE does not name a GiNGR checkout")


def _tetra():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1.5]], dtype=np.float64)
    t = np.array([[0, 2, 1], [0, 1, 3], [1, 2, 3], [0, 3, 2]], dtype=np.int32)
    return v, t


def test_model_fitting_parameters_json_layout(tmp_path):
    from gingr_b200 import api, io
    p = api.ModelFittingParameters(1.25, np.array([1.0, -2.0, 3.5]), (0.1, -0.2, 0.3), np.array([0.5, -1.5, 2.0]))
    obj = io.parameters_to_json(p)
    # spray-json jsonFormatN field names (ModelFittingParameters.scala:97-104)
    assert set(obj) == {"scale", "pose", "shape"} and obj["scale"] == {"s": 1.25}
    assert obj["pose"]["rotation"]["angles"] == {"phi": 0.1, "theta": -0.2, "psi": 0.3}
    assert obj["pose"]["rotation"]["center"] == [0.0, 0.0, 0.0] and obj["pose"]["translation"] == [1.0, -2.0, 3.5]
    assert obj["shape"] == {"parameters": [0.5, -1.5, 2.0]}
    f = str(tmp_path / "pars.json")
    io.save_parameters(p, f)
    q, c = io.load_parameters(f)
    assert q.scale == p.scale and tuple(q.euler) == tuple(p.euler) and c == (0.0, 0.0, 0.0)
    assert np.array_equal(q.translation, p.translation) and np.array_equal(q.shape, p.shape)
    with pytest.raises(ValueError):
        io.parameters_from_json({"scale": {"s": 1.0}})


def test_json_state_logger_records(tmp_path):
    from gingr_b200 import api, io
    pars = api.ModelFittingParameters(1.0, np.array([1.0, 2.0, 3.0]), (0.01, 0.02, 0.03), np.array([0.1, 0.2]))
    st = api.GeneralRegistrationState(pars, np.zeros((4, 3)), generatedBy="InformedProposal")
    lg = io.JSONStateLogger(lambda s: {"Prior": -1.5, "Distance": -10.0}, str(tmp_path / "log.json"))
    lg.accept(st)
    lg.reject(st)
    lg.accept(st)
    lg.write()
    raw = json.loads(pathlib.Path(tmp_path / "log.json").read_text())
    assert [r["index"] for r in raw] == [0, 1, 2] and [r["status"] for r in raw] == [True, False, True]
    assert set(raw[0]) == {"index", "name", "logvalue", "status", "modelParameters", "translation", "rotation",
                           "rotationCenter", "scaling", "datetime"}                       # jsonLogFormat :36-47
    assert raw[0]["logvalue"] == {"Prior": -1.5, "Distance": -10.0, "product": -11.5}
    assert raw[1]["modelParameters"] == [] and raw[1]["translation"] == [] and raw[1]["scaling"] == 1.0
    assert raw[0]["rotation"] == [0.01, 0.02, 0.03] and raw[0]["rotationCenter"] == [0.0, 0.0, 0.0]
    recs = io.JSONStateLogger.load(str(tmp_path / "log.json"))
    last = io.JSONStateLogger.last_accepted_parameters(recs)
    assert np.array_equal(last.shape, pars.shape) and tuple(last.euler) == tuple(pars.euler)
    assert lg.accepted == 2 and lg.rejected == 1 and lg.generatedBy == {"InformedProposal"}


def test_landmarks_round_trip_and_correspondences(tmp_path):
    from gingr_b200 import io
    cov = np.diag([4.0, 9.0, 1.0])
    lms = [io.Landmark("A", np.array([0.1, 0.0, 0.0]), cov), io.Landmark("B", np.array([0.9, 0.1, 0.0]), None),
           io.Landmark("only-model", np.array([5.0, 5.0, 5.0]), None)]
    f = str(tmp_path / "lm.json")
    io.write_landmarks(lms, f)
    back = io.read_landmarks(f)
    assert [b.id for b in back] == ["A", "B", "only-model"] and back[1].covariance is None
    assert np.allclose(back[0].covariance, cov, atol=1e-12) and np.array_equal(back[0].point, lms[0].point)
    v, _ = _tetra()
    tgt = [io.Landmark("B", np.array([7.0, 7.0, 7.0]), None), io.Landmark("A", np.array([8.0, 8.0, 8.0]), None)]
    pids, pts, covs = io.landmark_correspondences(back, tgt, v)
    assert pids.tolist() == [0, 1] and np.array_equal(pts, [[8.0, 8.0, 8.0], [7.0, 7.0, 7.0]])
    assert np.allclose(covs[0], cov) and np.array_equal(covs[1], np.eye(3))


@pytest.mark.parametrize("binary", [True, False])
def test_ply_round_trip(tmp_path, binary):
    from gingr_b200 import io
    v, t = _tetra()
    f = str(tmp_path / "m.ply")
    io.write_ply(f, v, t, binary=binary)
    v2, t2 = io.read_mesh(f)
    assert np.array_equal(v2, v) and np.array_equal(t2, t) and v2.dtype == np.float64 and t2.dtype == np.int32


def test_stl_round_trip_merges_vertices(tmp_path):
    from gingr_b200 import io
    v, t = _tetra()
    f = str(tmp_path / "m.stl")
    io.write_stl(f, v, t)
    v2, t2 = io.read_mesh(f)
    assert v2.shape == (4, 3) and t2.shape == (4, 3)             # 12 corners merged into 4 vertices
    assert np.array_equal(v2[t2], v[t])                          # same geometry, first-appearance vertex order
    ascii_stl = "solid s\n" + "".join(
        "facet normal 0 0 0\n outer loop\n" + "".join(f"  vertex {p[0]} {p[1]} {p[2]}\n" for p in v[tri]) + " endloop\nendfacet\n"
        for tri in t) + "endsolid s\n"
    g = str(tmp_path / "a.stl")
    pathlib.Path(g).write_text(ascii_stl)
    v3, t3 = io.read_stl(g)
    assert np.array_equal(v3[t3], v[t])
    with pytest.raises(ValueError):
        pathlib.Path(g).write_bytes(b"garbage" * 20)
        io.read_stl(g)


@needs_reference
def test_reference_example_files():
    from gingr_b200 import io
    v, t = io.read_mesh(os.path.join(REF_DATA, "femur", "femur.stl"))
    assert v.shape == (1622, 3) and t.shape == (3240, 3) and t.max() == 1621          # SURVEY.md 8c fixtures
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "femur_golden.npz"))
    key = [k for k in gold.files if "ref" in k.lower() and gold[k].shape == (1622, 3)]
    if key:
        assert np.array_equal(gold[key[0]], v)
    bv, bt = io.read_mesh(os.path.join(REF_DATA, "bunny", "bunny.ply"))
    assert bv.shape == (35393, 3) and bt.shape == (70782, 3) and bt.min() == 0 and bt.max() == 35392
    lm = io.read_landmarks(os.path.join(REF_DATA, "femur", "femur.json"))
    assert len(lm) == 6 and lm[0].id == "L0" and lm[0].covariance is None
    arm = io.read_landmarks(os.path.join(REF_DATA, "armadillo", "armadillo.json"))
    assert arm[0].covariance is not None and np.allclose(arm[0].covariance, 25.0 * np.eye(3))
    tl = io.read_landmarks(os.path.join(REF_DATA, "femur", "femur_target.json"))
    pids, pts, covs = io.landmark_correspondences(lm, tl, v)
    assert len(pids) == 6 and np.all(covs == np.eye(3))


def test_statistical_model_file_round_trip(tmp_path):
    """The cached-GPMM file (DemoDatasetLoader.scala:40-53 role): lossless round trip, reference file naming, and the
    reference's Try semantics (any unreadable / foreign / inconsistent file reads as 'absent')."""
    from gingr_b200 import io
    rng = np.random.default_rng(5)
    v, t = _tetra()
    basis, _ = np.linalg.qr(rng.normal(size=(12, 5)))
    var = np.sort(rng.uniform(0.1, 9.0, 5))[::-1].copy()
    mean = rng.normal(size=12)
    p = str(tmp_path / io.model_file_name("femur", 100, "Gauss", io.gauss_kernel_printpars(50, 70)))
    assert os.path.basename(p) == "femur_dec-100_Gauss_50.0_70.0.h5.json"                     # DemoDatasetLoader.scala:47
    assert io.model_file_name("bunny", None, "GaussMix", "") == "bunny_dec-full_GaussMix_.h5.json"
    io.write_statistical_model(p, v, t, mean, basis, var)
    ref, tri, m2, b2, v2 = io.read_statistical_model(p)
    assert np.array_equal(ref, v) and np.array_equal(tri, t) and tri.dtype == np.int32
    assert np.array_equal(m2, mean) and np.array_equal(b2, basis) and np.array_equal(v2, var)   # bit-exact, f64 kept
    doc = json.loads(pathlib.Path(p).read_text())
    assert doc["representer"]["points"]["shape"] == [3, 4] and doc["representer"]["cells"]["shape"] == [3, 4]
    assert doc["model"]["pcaBasis"]["shape"] == [12, 5] and doc["model"]["noiseVariance"] == 0.0
    # point cloud model (no cells)
    q = str(tmp_path / "cloud.h5.json")
    io.write_statistical_model(q, v, None, mean, basis, var)
    assert io.read_statistical_model(q)[1].shape == (0, 3)
    # failures
    with pytest.raises(OSError):
        io.read_statistical_model(str(tmp_path / "missing.h5.json"))
    (tmp_path / "foreign.h5.json").write_text(json.dumps({"format": "something else"}))
    with pytest.raises(ValueError):
        io.read_statistical_model(str(tmp_path / "foreign.h5.json"))
    doc["model"]["pcaVariance"]["shape"] = [4]
    (tmp_path / "bad.h5.json").write_text(json.dumps(doc))
    with pytest.raises(ValueError):
        io.read_statistical_model(str(tmp_path / "bad.h5.json"))
    with pytest.raises(ValueError):
        io.write_statistical_model(q, v, t, mean[:-1], basis, var)
    with pytest.raises(ValueError):
        io.write_statistical_model(q, v, t + 1, mean, basis, var)


def test_logger_statistics_and_precomputed_values():
    from gingr_b200 import api, io
    lg = io.JSONStateLogger()
    p = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.arange(3.0))
    s = api.GeneralRegistrationState(p, np.zeros((1, 3)), generatedBy="CPD")
    lg.accept(s, {"Prior": -1.5, "Distance": -2.0})
    lg.reject(dataclasses.replace(s, generatedBy="RandomShape-0.1"), {"Prior": -3.0, "Distance": -4.0})
    lg.reject(dataclasses.replace(s, generatedBy="CPD"), {"Prior": -3.0, "Distance": -4.0})
    assert lg.totalSamples == 3 and lg.log[0].logvalue == {"Prior": -1.5, "Distance": -2.0, "product": -3.5}
    assert lg.log[1].modelParameters == [] and lg.log[1].name == "RandomShape-0.1" and not lg.log[1].status
    assert lg.percentRejected == 0.67 and abs(lg.percentAccepted - 0.33) < 1e-12       # 2/3 -> 0.67 (HALF_UP, two decimals)
    assert lg.percentAcceptedOfType("CPD") == 0.5 and lg.percentAcceptedOfType("RandomShape-0.1") == 0.0
    assert lg.percentAcceptedOfType("CPD", last=1) == 0.0
    lg2 = io.JSONStateLogger()
    for k in range(8):
        (lg2.reject if k == 0 else lg2.accept)(s, {})
    assert lg2.percentRejected == 0.13                                                  # 0.125 rounds half UP


def test_malformed_mesh_files_raise_value_error(tmp_path):
    """MeshIO.readMesh returns a failed Try on unreadable files; here every malformed file is a ValueError (never an
    IndexError / UnicodeDecodeError, never a mesh with dangling indices)."""
    from gingr_b200 import io
    hdr = (b"ply\nformat ascii 1.0\nelement vertex 3\nproperty float x\nproperty float y\nproperty float z\n"
           b"element face 1\nproperty list uchar int vertex_indices\nend_header\n")
    cases = {
        "empty.stl": b"",
        "garbage.stl": bytes(range(256)) * 3,
        "truncated.stl": b"\0" * 80 + (5).to_bytes(4, "little") + b"\0" * 60,
        "ragged.stl": b"solid x\nfacet normal 0 0 1\nouter loop\nvertex 0 0 0\nvertex 1 0\nvertex 0 1 0\nendloop\nendfacet\nendsolid x\n",
        "two_corners.stl": b"solid x\nvertex 0 0 0\nvertex 1 0 0\nendsolid x\n",
        "empty.ply": b"",
        "header_only.ply": b"ply\nformat ascii 1.0\n",
        "short_body.ply": hdr + b"0 0 0\n1 0 0\n",
        "short_face.ply": hdr + b"0 0 0\n1 0 0\n0 1 0\n3 0 1\n",
        "dangling_index.ply": hdr + b"0 0 0\n1 0 0\n0 1 0\n3 0 1 7\n",
        "quad.ply": hdr.replace(b"vertex 3", b"vertex 4") + b"0 0 0\n1 0 0\n1 1 0\n0 1 0\n4 0 1 2 3\n",
        "binary_truncated.ply": hdr.replace(b"ascii", b"binary_little_endian") + b"\0" * 20,
        "unknown_format.ply": hdr.replace(b"ascii", b"binary_middle_endian") + b"\0" * 64,
        "mesh.obj": b"v 0 0 0\n",
    }
    for name, data in cases.items():
        p = tmp_path / name
        p.write_bytes(data)
        with pytest.raises(ValueError):
            io.read_mesh(str(p))
    good = tmp_path / "ok.ply"
    good.write_bytes(hdr + b"0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n")
    v, t = io.read_mesh(str(good))
    assert v.shape == (3, 3) and t.tolist() == [[0, 1, 2]]


def test_malformed_landmark_files_raise_value_error(tmp_path):
    from gingr_b200 import io
    bad = ['{"id": "A"}', '[{"id": "A"}]', '[{"id": "A", "coordinates": [1, 2]}]', '[3]',
           '[{"id": "A", "coordinates": [1, 2, 3], "uncertainty": {"stddevs": [1, 2], "pcvectors": [[1, 0, 0], [0, 1, 0], [0, 0, 1]]}}]',
           '[{"id": "A", "coordinates": [1, 2, 3], "uncertainty": {"stddevs": [1, 2, 3]}}]']
    for k, text in enumerate(bad):
        p = tmp_path / f"lm{k}.json"
        p.write_text(text)
        with pytest.raises(ValueError):
            io.read_landmarks(str(p))
    ok = tmp_path / "ok.json"
    ok.write_text('[{"id": "A", "coordinates": [1, 2, 3], "uncertainty": {"stddevs": [1, 2, 3], "pcvectors": [[0, 1, 0], [1, 0, 0], [0, 0, 1]]}}]')
    lm = io.read_landmarks(str(ok))[0]
    assert lm.id == "A" and np.allclose(np.diag(lm.covariance), [4.0, 1.0, 9.0])
