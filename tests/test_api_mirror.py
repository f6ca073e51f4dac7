"""The Python mirror of the reference's configuration / state classes (gingr_b200/api.py): names and DEFAULTS must be the
reference's (checked against the Scala sources when the reference tree is mounted), and the POD round trips are lossless.
No GPU."""
import pathlib
import dataclasses
import os
import re

import numpy as np
import pytest

# GINGR_REFERENCE: a checkout of the Scala GiNGR project, the sources these defaults are checked against
REF = os.path.join(os.environ["GINGR_REFERENCE"], "src", "main", "scala", "gingr") if os.environ.get("GINGR_REFERENCE") else ""
needs_reference = pytest.mark.skipif(not os.path.isdir(REF), reason="GINGR_REFERENCE does not name a GiNGR checkout")


def _case_class_defaults(path, name):
    """{field: default literal} of `case class name(...)` in a Scala file (fields with a default only)."""
    src = pathlib.Path(path).read_text()
    start = src.index("case class " + name)
    depth, i = 0, src.index("(", start)
    j = i
    while True:
        if src[j] == "(":
            depth += 1
        elif src[j] == ")":
            depth -= 1
            if depth == 0:
                break
        j += 1
    body = src[i + 1:j]
    out = {}
    for m in re.finditer(r"(?:override val\s+)?(\w+)\s*:\s*[^=,()]+(?:\[[^\]]*\])?\s*=\s*([^,\n]+)", body):
        out[m.group(1)] = m.group(2).strip()
    return out


def _num(s):
    return float(s.replace("1e-10", "1e-10"))


@needs_reference
def test_configuration_defaults_are_the_references():
    from gingr_b200 import api
    cpd = _case_class_defaults(os.path.join(REF, "api/registration/config/CPD.scala"), "CpdConfiguration")
    c = api.CpdConfiguration()
    assert int(cpd["maxIterations"]) == c.maxIterations and _num(cpd["threshold"]) == c.threshold
    assert cpd["useLandmarkCorrespondence"] == "true" and c.useLandmarkCorrespondence is True
    assert cpd["initialSigma"] == "None" and c.initialSigma is None
    assert _num(cpd["w"]) == c.w and _num(cpd["lambda"]) == c.lambda_
    icp = _case_class_defaults(os.path.join(REF, "api/registration/config/ICP.scala"), "IcpConfiguration")
    k = api.IcpConfiguration()
    assert int(icp["maxIterations"]) == k.maxIterations and _num(icp["threshold"]) == k.threshold
    assert _num(icp["initialSigma"]) == k.initialSigma and _num(icp["endSigma"]) == k.endSigma
    assert icp["reverseCorrespondenceDirection"] == "false" and k.reverseCorrespondenceDirection is False
    assert icp["correspondenceMethod"] == "TriangularClosestPoint" and k.correspondenceMethod == api.TRIANGULAR_CLOSEST_POINT
    assert k.sigmaStep == (k.initialSigma - k.endSigma) / k.maxIterations                      # ICP.scala:65
    gs = _case_class_defaults(os.path.join(REF, "api/GeneralRegistrationState.scala"), "GeneralRegistrationState")
    s = api.GeneralRegistrationState(api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(2)), np.zeros((1, 3)))
    assert _num(gs["sigma2"]) == s.sigma2 and _num(gs["stepLength"]) == s.stepLength
    assert gs["globalTransformation"] == "RigidTransforms" and s.globalTransformation == api.RIGID_TRANSFORMS
    assert int(gs["iteration"]) == s.iteration and gs["status"] == "FittingStatuses.None" and s.status == api.STATUS_NONE
    ps = _case_class_defaults(os.path.join(REF, "api/GingrAlgorithm.scala"), "ProbabilisticSettings")
    assert _num(ps["randomMixture"]) == api.ProbabilisticSettings().randomMixture
    gen = pathlib.Path(os.path.join(REF, "api/sampling/Generator.scala")).read_text()
    assert "defaultTranslation = 0.1" in gen and "defaultRotation = 0.01" in gen and "Seq(1.0, 0.1, 0.01)" in gen
    p = api.ProbabilisticSettings()
    assert p.translationSdev == (0.1, 0.1, 0.1) and p.rotationSdev == (0.01, 0.01, 0.01) and p.shapeSteps == (1.0, 0.1, 0.01)


@needs_reference
def test_enumerations_follow_the_reference_order():
    from gingr_b200 import api
    fs = pathlib.Path(os.path.join(REF, "api/FittingStatuses.scala")).read_text()
    order = re.search(r"val\s+(\w+)\s*,\s*(\w+)\s*,\s*(\w+)\s*,\s*(\w+)\s*=\s*Value", fs)
    assert order and [x for x in order.groups()] == ["None", "MaxIteration", "Converged", "ModelFlexibilityError"]
    assert (api.STATUS_NONE, api.STATUS_MAX_ITERATION, api.STATUS_CONVERGED, api.STATUS_MODEL_FLEXIBILITY_ERROR) == (0, 1, 2, 3)
    icp = pathlib.Path(os.path.join(REF, "api/registration/config/ICP.scala")).read_text()
    names = re.findall(r"case object (\w+ClosestPoint) extends ICPCorrespondenceMethod", icp)
    assert set(names) == {"TriangularClosestPoint", "AlongNormalClosestPoint", "PointcloudClosestPoint"}
    modes = pathlib.Path(os.path.join(REF, "api/sampling/evaluators/IndependentPointDistanceEvaluator.scala")).read_text()
    assert re.findall(r"case object (\w+) extends EvaluationMode", modes) == ["ModelToTargetEvaluation", "TargetToModelEvaluation", "SymmetricEvaluation"]
    assert (api.EVAL_MODEL_TO_TARGET, api.EVAL_TARGET_TO_MODEL, api.EVAL_SYMMETRIC) == (0, 1, 2)


def test_state_and_config_pod_round_trips():
    from gingr_b200 import api
    pars = api.ModelFittingParameters(1.25, np.array([1.0, -2.0, 3.5]), (0.1, -0.2, 0.3), np.linspace(-1, 1, 7))
    st = api.GeneralRegistrationState(pars, np.zeros((4, 3)), sigma2=2.5, globalTransformation=api.SIMILARITY_TRANSFORMS,
                                      stepLength=0.5, generatedBy="x", iteration=7, status=api.STATUS_CONVERGED)
    pod, alpha = st.to_pod()
    assert pod.rank == 7 and pod.iteration == 7 and pod.status == api.STATUS_CONVERGED and pod.sigma2 == 2.5
    assert tuple(pod.center) == (0.0, 0.0, 0.0) and pod.step_length == 0.5
    back = api.GeneralRegistrationState.from_pod(pod, alpha, st.fit, "x")
    assert back.modelParameters.scale == 1.25 and tuple(back.modelParameters.euler) == (0.1, -0.2, 0.3)
    assert np.array_equal(back.modelParameters.translation, pars.translation) and np.array_equal(back.modelParameters.shape, pars.shape)
    assert (back.sigma2, back.stepLength, back.iteration, back.status, back.globalTransformation) == (2.5, 0.5, 7, api.STATUS_CONVERGED, api.SIMILARITY_TRANSFORMS)
    c = api.CpdConfiguration(maxIterations=33, w=0.2, lambda_=2.0, initialSigma=4.0, useLandmarkCorrespondence=False).to_pod()
    assert (c.algorithm, c.max_iterations, c.w, c.lambda_, c.has_initial_sigma, c.initial_sigma, c.use_landmark_correspondence) == (api.ALGO_CPD, 33, 0.2, 2.0, 1, 4.0, 0)
    assert api.CpdConfiguration().to_pod().has_initial_sigma == 0
    k = api.IcpConfiguration(initialSigma=9.0, endSigma=3.0, reverseCorrespondenceDirection=True,
                             correspondenceMethod=api.ALONG_NORMAL_CLOSEST_POINT).to_pod()
    assert (k.algorithm, k.initial_sigma, k.end_sigma, k.reverse_correspondence_direction, k.correspondence_method) == (api.ALGO_ICP, 9.0, 3.0, 1, api.ALONG_NORMAL_CLOSEST_POINT)
    m = api.ProbabilisticSettings(uncertainty=2.0, mode=api.EVAL_SYMMETRIC, randomMixture=0.25, shapeSteps=(2.0, 0.2, 0.02)).to_pod()
    assert (m.uncertainty, m.evaluation_mode, m.random_mixture, tuple(m.shape_sdev)) == (2.0, 2, 0.25, (2.0, 0.2, 0.02))


def test_convergence_closures_match_the_reference():
    from gingr_b200 import api
    a = api.GeneralRegistrationState(api.ModelFittingParameters(1.0, np.zeros(3), (0, 0, 0), np.zeros(1)), np.zeros((1, 3)), sigma2=1.0)
    b = dataclasses.replace(a, sigma2=1.0 + 5e-11)
    c = dataclasses.replace(a, sigma2=1.1)
    cpd, icp = api.CpdConfiguration(), api.IcpConfiguration()
    assert cpd.converged(a, b, cpd.threshold) and not cpd.converged(a, c, cpd.threshold)      # CPD.scala:106-110
    assert not icp.converged(a, a, icp.threshold)                                             # ICP.scala:57-58: never


def test_maximum_point_distance_is_the_brute_force_value():
    """PointSetHelper.maximumPointDistance (GPMMHelper.scala:76-81): hull pairing above the limit must give the literal
    all-pairs maximum bit for bit -- also for points all on the hull, flat sets and duplicated points."""
    from gingr_b200 import api
    rng = np.random.default_rng(3)
    sphere = rng.normal(size=(2500, 3))
    sphere /= np.linalg.norm(sphere, axis=1)[:, None]
    flat = np.c_[rng.normal(size=(2500, 2)), np.zeros(2500)]
    blob = rng.normal(size=(3000, 3)) * [30.0, 10.0, 5.0]
    dup = np.repeat(blob[:1500], 2, axis=0)
    for pts in (sphere, flat, blob, dup):
        lit = api.maximum_point_distance(pts, brute_force_limit=10 ** 9)
        assert api.maximum_point_distance(pts, brute_force_limit=16) == lit
        i, j = rng.integers(0, len(pts), 2)
        assert lit >= np.linalg.norm(pts[i] - pts[j]) * (1 - 1e-15)
    tiny = np.array([[0.0, 0, 0], [3.0, 4.0, 0.0]])
    assert api.maximum_point_distance(tiny) == 5.0 and api.maximum_point_distance(tiny[:1]) == 0.0


def test_simple_registrator_attaches_the_json_logger_when_asked(tmp_path):
    """SimpleRegistrator.run (SimpleRegistrator.scala:127-158): probabilistic runs carry a JSONStateLogger that is written
    to logFileFittingParameters, the callback is the chain-state logger, and the returned fit is the FULL model's
    instance.  Wiring only (fake registration object, no device)."""
    from gingr_b200 import api, io
    pars = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.arange(2.0))
    st = api.GeneralRegistrationState(pars, np.zeros((2, 3)))
    calls = {}

    class FakeReg:
        def __init__(self, ctx, model, target, config):
            self.config = config

        def initializeState(self, general=None, globalTransformation=None):
            calls["init"] = (general, globalTransformation)
            return st

        def runProbabilistic(self, state, settings, seed=0, acceptRejectLogger=None, callBackLogger=None):
            calls["settings"] = settings
            calls["loggers"] = (acceptRejectLogger, callBackLogger)
            if acceptRejectLogger is not None:
                acceptRejectLogger.accept(state, {"Prior": -1.0, "Distance": -2.0})
                acceptRejectLogger.reject(dataclasses.replace(state, generatedBy="CPD"), {"Prior": -3.0, "Distance": -4.0})
            if callBackLogger is not None:
                callBackLogger(state)
            return dataclasses.replace(state, status=api.STATUS_MAX_ITERATION)

        def run(self, state, callback=None):
            calls["det"] = callback
            return dataclasses.replace(state, status=api.STATUS_CONVERGED)

        def close(self):
            calls["closed"] = calls.get("closed", 0) + 1

    class FakeModel:
        def instance(self, p):
            return np.full((5, 3), 7.0)

    log = str(tmp_path / "fit.json")
    sr = api.SimpleRegistrator(None, FakeReg, api.CpdConfiguration(), FakeModel(), None, evaluatorUncertainty=2.0,
                               evaluationMode=api.EVAL_SYMMETRIC, logFileFittingParameters=log)
    seen = []
    out = sr.run(probabilistic=True, randomMixture=0.25, callback=seen.append, seed=3)
    assert out.fit.shape == (5, 3) and out.status == api.STATUS_MAX_ITERATION and calls["closed"] == 1
    s = calls["settings"]
    assert (s.uncertainty, s.mode, s.randomMixture) == (2.0, api.EVAL_SYMMETRIC, 0.25)
    assert calls["loggers"][0] is sr.jsonLogger and len(seen) == 1
    recs = io.JSONStateLogger.load(log)
    assert [r.status for r in recs] == [True, False] and recs[1].name == "CPD" and recs[0].logvalue["product"] == -3.0
    # no log file, no callback: the chain is left on the device (no per-step logger)
    sr2 = api.SimpleRegistrator(None, FakeReg, api.CpdConfiguration(), FakeModel(), None)
    sr2.run(probabilistic=True)
    assert calls["loggers"] == (None, None) and sr2.jsonLogger is None
    # deterministic: callback goes to run(), and a handed-over state is re-initialised with iteration 0 / status None
    g = dataclasses.replace(st, iteration=9, status=api.STATUS_CONVERGED)
    out = sr2.run(generalState=g, globalTransformation=api.SIMILARITY_TRANSFORMS, callback=seen.append)
    assert calls["det"] is not None and out.status == api.STATUS_CONVERGED
    assert calls["init"][0].iteration == 0 and calls["init"][0].status == api.STATUS_NONE
    # the hand-over keeps the state's OWN transformation type; the call argument is ignored when a generalState is given
    # (SimpleRegistrator.scala:76-82, :93-95, :135-137)
    assert calls["init"][0].globalTransformation == st.globalTransformation != api.SIMILARITY_TRANSFORMS
    gs = dataclasses.replace(st, globalTransformation=api.SIMILARITY_TRANSFORMS)
    sr2.run(generalState=gs)                                   # default argument RIGID must not overwrite SIMILARITY
    assert calls["init"][0].globalTransformation == api.SIMILARITY_TRANSFORMS


def test_gingr_interface_options_reach_the_registration(monkeypatch):
    """simple/GingrInterface.scala:20-64 -> SimpleRegistrator: landmarks are resolved on the run model's reference, the
    initial transform seeds the pose, evaluatedPoints becomes the evaluator's point subsets."""
    from gingr_b200 import api, io
    calls = {}
    pars = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(2))
    st = api.GeneralRegistrationState(pars, np.zeros((2, 3)))

    class FakeReg:
        name = "CPD"

        def __init__(self, ctx, model, target, config):
            calls["config"] = config

        def setLandmarks(self, pids, points, cov=None):
            calls["lm"] = (np.asarray(pids), np.asarray(points), np.asarray(cov))

        def initializeState(self, general=None, globalTransformation=None, rotation=None, translation=None):
            calls["init"] = (general, globalTransformation, rotation, translation)
            return st

        def runProbabilistic(self, state, settings, seed=0, acceptRejectLogger=None, callBackLogger=None):
            calls["settings"] = settings
            return state

        def run(self, state, callback=None):
            return state

        def close(self):
            pass

    class FakeModel:
        M = 10
        reference = np.array([[float(k), 0.0, 0.0] for k in range(10)])

        def instance(self, p):
            return np.zeros((10, 3))

    class FakeTarget:
        N = 1000
        points = np.random.default_rng(0).uniform(size=(1000, 3)) * 50.0

    monkeypatch.setattr(api, "CpdRegistration", FakeReg)
    monkeypatch.setattr(api, "IcpRegistration", FakeReg)
    cov = np.diag([1.0, 2.0, 3.0])
    mlm = [io.Landmark("A", np.array([2.2, 0.1, 0.0]), cov), io.Landmark("B", np.array([7.6, 0.0, 0.0]), None),
           io.Landmark("only-model", np.zeros(3), None)]
    tlm = [io.Landmark("B", np.array([1.0, 1.0, 1.0]), None), io.Landmark("A", np.array([5.0, 5.0, 5.0]), None)]
    R = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    gi = api.GingrInterface(None, FakeModel(), FakeTarget(), initialModelParameterTransform=(R, [1.0, 2.0, 3.0]),
                            modelLandmarks=mlm, targetLandmarks=tlm, evaluatorUncertainty=3.0, evaluatedPoints=4,
                            evaluationMode=api.EVAL_TARGET_TO_MODEL)
    sr = gi.CPD(api.CpdConfiguration(w=0.2))
    assert isinstance(sr, api.SimpleRegistrator) and calls == {}
    sr.run(probabilistic=True, randomMixture=0.1)
    assert calls["config"].w == 0.2
    pids, pts, covs = calls["lm"]
    assert list(pids) == [2, 8] and np.array_equal(pts, [[5.0, 5.0, 5.0], [1.0, 1.0, 1.0]])     # matched by id, nearest reference vertex
    assert np.array_equal(covs[0], cov) and np.array_equal(covs[1], np.eye(3))
    assert calls["init"][0] is None and calls["init"][2] is R and list(calls["init"][3]) == [1.0, 2.0, 3.0]
    s = calls["settings"]
    assert (s.uncertainty, s.mode, s.randomMixture) == (3.0, api.EVAL_TARGET_TO_MODEL, 0.1)
    assert list(s.modelPointIds) == [0, 1, 2, 3]
    tids = np.asarray(s.targetPointIds)
    assert tids.dtype == np.int32 and 2 <= len(tids) <= 8 and np.all(np.diff(tids) > 0) and tids.max() < 1000
    # a handed-over state wins over the initial transform (combineStates, SimpleRegistrator.scala:76-82)
    gi.ICP().run(generalState=st)
    assert calls["init"][0] is not None and calls["init"][2] is None
    assert isinstance(calls["config"], api.IcpConfiguration)


def test_run_decimated_accepts_point_counts(monkeypatch):
    """runDecimated(modelPoints, targetPoints, ...) (SimpleRegistrator.scala:58-70): integer arguments decimate the model's
    reference and the target on the host, then re-reference / upload; tuples are taken as given."""
    from gingr_b200 import api, synthetic
    made = {}
    rv, rt = synthetic.sphere_mesh(400)
    tv, tt = synthetic.sphere_mesh(500)

    class FakeModel:
        M, reference, triangles = 400, rv, rt

        def newReference(self, pts, tri=None):
            made["ref"] = (np.asarray(pts), np.asarray(tri))
            return self

        def instance(self, p):
            return np.zeros((400, 3))

        def close(self):
            made["model_closed"] = True

    class FakeTarget:
        def __init__(self, ctx=None, pts=tv, tri=tt):
            self.points, self.triangles, self.N = np.asarray(pts), np.asarray(tri), len(pts)
            made.setdefault("targets", []).append(self)

        def close(self):
            made["target_closed"] = True

    pars = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(2))
    st = api.GeneralRegistrationState(pars, np.zeros((2, 3)))

    class FakeReg:
        def __init__(self, ctx, model, target, config):
            made["run_target"] = target

        def initializeState(self, general=None, globalTransformation=None):
            return st

        def run(self, state, callback=None):
            return state

        def close(self):
            pass

    monkeypatch.setattr(api, "Target", FakeTarget)
    sr = api.SimpleRegistrator(None, FakeReg, api.CpdConfiguration(), FakeModel(), FakeTarget())
    sr.runDecimated(60, 80)
    assert made["ref"][0].shape == (60, 3) and made["ref"][1].max() == 59
    assert made["run_target"].N == 80 and made["run_target"] is not sr.target
    assert made["model_closed"] and made["target_closed"]
    sr.runDecimated((rv[:50], None), (tv[:70], None))
    assert made["ref"][0].shape == (50, 3) and made["run_target"].N == 70


def test_model_constructor_rejects_inconsistent_arrays_before_touching_the_library():
    from gingr_b200 import api
    ref = np.zeros((4, 3))
    with pytest.raises(ValueError):
        api.Model(None, ref, np.zeros(12), np.zeros((11, 2)), np.ones(2))          # basis rows != 3M
    with pytest.raises(ValueError):
        api.Model(None, ref, np.zeros(9), np.zeros((12, 2)), np.ones(2))           # mean length != 3M
    with pytest.raises(ValueError):
        api.Model.gaussianMixture(None, ref, None, [1.0, 2.0], [1.0])


def test_minimum_point_distance_and_the_automatic_template_model(monkeypatch):
    """minimumPointDistance is the brute-force value; automaticGPMMfromTemplate (registration/utils/GPMMHelper.scala:38-68)
    passes the reference's three (sigma, scaling) pairs and relativeTolerance 0.1 to the device builder."""
    from gingr_b200 import api
    rng = np.random.default_rng(6)
    for pts in (rng.normal(size=(700, 3)) * 20.0, np.c_[rng.normal(size=(500, 2)), np.zeros(500)], rng.uniform(size=(5, 3))):
        d = np.sqrt(((pts[:, None] - pts[None]) ** 2).sum(-1))
        np.fill_diagonal(d, np.inf)
        got = api.minimum_point_distance(pts)
        assert abs(got - d.min()) <= 1e-15 * d.min()
    dup = np.r_[pts, pts[:1]]
    assert api.minimum_point_distance(dup) == 0.0
    with pytest.raises(ValueError):
        api.minimum_point_distance(pts[:1])
    seen = {}
    monkeypatch.setattr(api.Model, "gaussianMixture", staticmethod(lambda ctx, ref, tri, sig, sc, tol, cap=0: seen.update(sig=sig, sc=sc, tol=tol)))
    ref = rng.normal(size=(300, 3)) * 10.0
    api.Model.automaticGPMMfromTemplate(None, ref, None)
    dmax, dmin = api.maximum_point_distance(ref), api.minimum_point_distance(ref)
    assert seen["sig"] == [dmax / 4.0, dmax / 8.0, dmin * 5.0] and seen["sc"] == [dmax / 8.0, dmax / 16.0, dmin * 2.5]
    assert seen["tol"] == 0.1


def test_print_status_sentences(capsys):
    from gingr_b200 import api
    p = api.ModelFittingParameters(1.0, np.zeros(3), (0.0, 0.0, 0.0), np.zeros(1))
    s = api.GeneralRegistrationState(p, np.zeros((1, 3)), iteration=4)
    assert s.statusText() == "Initial state - no iterations performed!"
    assert dataclasses.replace(s, status=api.STATUS_CONVERGED).statusText() == "Fitting converged after 5 accepted iterations!"
    assert dataclasses.replace(s, status=api.STATUS_MAX_ITERATION).statusText() == "Fitting finished the MaxIterations with (5) accepted iterations!"
    dataclasses.replace(s, status=api.STATUS_MODEL_FLEXIBILITY_ERROR).printStatus()
    assert capsys.readouterr().out == "Model not flexible enough to compute posterior model - finished after 5 accepted iterations!\n"
    if os.path.isdir(REF):
        src = pathlib.Path(os.path.join(REF, "api/GeneralRegistrationState.scala")).read_text()
        for frag in ("Initial state - no iterations performed!", "Fitting converged after ", "Fitting finished the MaxIterations with (",
                     "Model not flexible enough to compute posterior model - finished after "):
            assert frag in src
