"""Wire / disk formats around the hot path (SURVEY.md 8f item 3): what a user of the reference exchanges with the Scala
tooling.  Host-side only (numpy + json); nothing here touches the device.

  ModelFittingParameters JSON   api/ModelFittingParameters.scala:75-105 (spray-json formats), :145-160 (save / load)
  jsonLogFormat / JSONStateLogger   api/sampling/loggers/JSONStateLogger.scala:36-47 (record), :95-140 (accept / reject),
                                    the log file is a JSON array of the records
  scalismo landmark JSON        examples/data/femur/femur.json, armadillo/*.json (id, coordinates, uncertainty{stddevs, pcvectors})
  binary / ASCII STL, PLY       examples/data/femur/*.stl, examples/data/bunny/bunny.ply (MeshIO.readMesh in
                                examples/DemoDatasetLoader.scala:60-76); STL vertices are merged when bit-identical, as
                                scalismo's STL reader does
"""
from __future__ import annotations

import datetime
import json
import struct
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np


# ---------------------------------------------------------------------------------------------
# ModelFittingParameters <-> JSON
# ---------------------------------------------------------------------------------------------
def parameters_to_json(pars, center=(0.0, 0.0, 0.0)) -> dict:
    """spray-json layout of ModelFittingParameters(scale: ScaleParameter, pose: PoseParameters, shape: ShapeParameters)
    with jsonFormatN field names (ModelFittingParameters.scala:97-104).  `pars`: api.ModelFittingParameters."""
    phi, theta, psi = (float(v) for v in pars.euler)
    return {
        "scale": {"s": float(pars.scale)},
        "pose": {
            "translation": [float(v) for v in pars.translation],
            "rotation": {"angles": {"phi": phi, "theta": theta, "psi": psi}, "center": [float(v) for v in center]},
        },
        "shape": {"parameters": [float(v) for v in np.asarray(pars.shape, dtype=float)]},
    }


def parameters_from_json(obj: dict):
    from .api import ModelFittingParameters
    try:
        ang = obj["pose"]["rotation"]["angles"]
        center = obj["pose"]["rotation"]["center"]
        pars = ModelFittingParameters(float(obj["scale"]["s"]), np.asarray(obj["pose"]["translation"], dtype=float),
                                      (float(ang["phi"]), float(ang["theta"]), float(ang["psi"])),
                                      np.asarray(obj["shape"]["parameters"], dtype=float))
    except (KeyError, TypeError) as e:
        raise ValueError(f"not a ModelFittingParameters JSON object: {e}")
    if len(pars.translation) != 3 or len(center) != 3:
        raise ValueError("translation and rotation centre must have 3 components")
    return pars, tuple(float(v) for v in center)


def save_parameters(pars, path: str, center=(0.0, 0.0, 0.0)) -> None:
    """ModelFittingParameters.save (:145-153): pretty-printed JSON."""
    with open(path, "w") as f:
        json.dump(parameters_to_json(pars, center), f, indent=2)


def load_parameters(path: str):
    """ModelFittingParameters.load (:155-160).  Returns (parameters, rotation centre)."""
    with open(path) as f:
        return parameters_from_json(json.load(f))


# ---------------------------------------------------------------------------------------------
# JSON state log
# ---------------------------------------------------------------------------------------------
@dataclass
class JsonLogRecord:
    """jsonLogFormat (JSONStateLogger.scala:36-47)."""
    index: int
    name: str
    logvalue: Dict[str, float]
    status: bool
    modelParameters: List[float]
    translation: List[float]
    rotation: List[float]
    rotationCenter: List[float]
    scaling: float
    datetime: str


class JSONStateLogger:
    """AcceptRejectLogger of the reference (JSONStateLogger.scala:49-190): an accepted sample stores its parameters, a
    rejected one only its log values ("the rejected state will contain the same parameters as the previous accepted
    state", :118).  `evaluate(state) -> {"Prior": .., "Distance": ..}`; "product" is added as their sum (:101-104)."""

    def __init__(self, evaluate=None, path: Optional[str] = None):
        self.evaluate = evaluate
        self.path = path
        self.log: List[JsonLogRecord] = []
        self.accepted = 0
        self.rejected = 0
        self.generatedBy = set()

    def _values(self, state, values=None) -> Dict[str, float]:
        if values is not None:
            ev = {k: float(v) for k, v in values.items()}
        else:
            ev = dict(self.evaluate(state)) if self.evaluate is not None else {}
        ev["product"] = float(sum(ev.values()))
        return ev

    def _now(self) -> str:
        return datetime.datetime.now().strftime("%Y-%m-%d %H:%M:%S")

    def accept(self, state, values=None) -> None:
        """values: the evaluators' log values when the caller already holds them (the device chain does), else
        evaluate(state) is called."""
        p = state.modelParameters
        self.generatedBy.add(state.generatedBy)
        self.log.append(JsonLogRecord(self.accepted + self.rejected, state.generatedBy, self._values(state, values), True,
                                      [float(v) for v in p.shape], [float(v) for v in p.translation],
                                      [float(v) for v in p.euler], [float(v) for v in getattr(p, "center", (0.0, 0.0, 0.0))],
                                      float(p.scale), self._now()))
        self.accepted += 1

    def reject(self, state, values=None) -> None:
        p = state.modelParameters
        self.generatedBy.add(state.generatedBy)
        self.log.append(JsonLogRecord(self.accepted + self.rejected, state.generatedBy, self._values(state, values), False,
                                      [], [], [], [], float(p.scale), self._now()))
        self.rejected += 1

    # acceptance statistics (JSONStateLogger.scala:86, :142-147, :186-196)
    @property
    def totalSamples(self) -> int:
        return self.accepted + self.rejected

    @property
    def percentRejected(self) -> float:
        """rejected / total rounded HALF_UP to two decimals (:142-145)."""
        import decimal
        if self.totalSamples == 0:
            return float("nan")
        q = decimal.Decimal(repr(self.rejected / self.totalSamples)).quantize(decimal.Decimal("0.01"), rounding=decimal.ROUND_HALF_UP)
        return float(q)

    @property
    def percentAccepted(self) -> float:
        return 1.0 - self.percentRejected

    def percentAcceptedOfType(self, name: str, last: Optional[int] = None) -> float:
        recs = [r for r in (self.log if last is None else self.log[-last:]) if r.name == name]
        return sum(1 for r in recs if r.status) / len(recs) if recs else float("nan")

    def to_json(self) -> list:
        return [r.__dict__.copy() for r in self.log]

    def write(self, path: Optional[str] = None) -> None:
        with open(path or self.path, "w") as f:
            json.dump(self.to_json(), f, indent=2)

    @staticmethod
    def load(path: str) -> List[JsonLogRecord]:
        with open(path) as f:
            data = json.load(f)
        if not isinstance(data, list):
            raise ValueError("a JSON state log is an array of records")
        out = []
        for d in data:
            try:
                out.append(JsonLogRecord(int(d["index"]), str(d["name"]), {k: float(v) for k, v in d["logvalue"].items()},
                                         bool(d["status"]), list(d["modelParameters"]), list(d["translation"]),
                                         list(d["rotation"]), list(d["rotationCenter"]), float(d["scaling"]), str(d["datetime"])))
            except (KeyError, TypeError) as e:
                raise ValueError(f"not a jsonLogFormat record: {e}")
        return out

    @staticmethod
    def last_accepted_parameters(records: Sequence[JsonLogRecord]):
        """The parameters of the chain's current state: the last record with status = true."""
        from .api import ModelFittingParameters
        for r in reversed(records):
            if r.status:
                return ModelFittingParameters(r.scaling, np.asarray(r.translation, float), tuple(r.rotation),
                                              np.asarray(r.modelParameters, float))
        return None


# ---------------------------------------------------------------------------------------------
# landmarks
# ---------------------------------------------------------------------------------------------
@dataclass
class Landmark:
    id: str
    point: np.ndarray                    # [3]
    covariance: Optional[np.ndarray]     # [3, 3] = P diag(stddev^2) P^T from uncertainty{stddevs, pcvectors}, or None


def read_landmarks(path: str) -> List[Landmark]:
    """scalismo LandmarkIO.readLandmarksJson3D layout."""
    with open(path) as f:
        data = json.load(f)
    if not isinstance(data, list):
        raise ValueError(f"{path}: a landmark file is a JSON array")
    out = []
    for d in data:
        try:
            cov = None
            u = d.get("uncertainty")
            if u is not None:
                sd = np.asarray(u["stddevs"], dtype=float)
                pcs = np.asarray(u["pcvectors"], dtype=float)      # rows = principal axes
                if sd.shape != (3,) or pcs.shape != (3, 3):
                    raise ValueError("uncertainty needs 3 stddevs and 3 x 3 pcvectors")
                cov = pcs.T @ np.diag(sd ** 2) @ pcs
            point = np.asarray(d["coordinates"], dtype=float)
            if point.shape != (3,):
                raise ValueError("coordinates need 3 components")
            out.append(Landmark(str(d["id"]), point, cov))
        except (KeyError, TypeError, AttributeError) as e:
            raise ValueError(f"{path}: not a scalismo landmark record ({type(e).__name__}: {e})")
    return out


def write_landmarks(landmarks: Sequence[Landmark], path: str) -> None:
    data = []
    for lm in landmarks:
        d = {"id": lm.id, "coordinates": [float(v) for v in lm.point]}
        if lm.covariance is not None:
            w, v = np.linalg.eigh(np.asarray(lm.covariance, dtype=float))
            d["uncertainty"] = {"stddevs": [float(np.sqrt(max(x, 0.0))) for x in w], "pcvectors": [[float(c) for c in v[:, k]] for k in range(3)]}
        data.append(d)
    with open(path, "w") as f:
        json.dump(data, f, indent=2)


def landmark_correspondences(model_landmarks: Sequence[Landmark], target_landmarks: Sequence[Landmark], reference_points):
    """GeneralRegistrationState.landmarkCorrespondences (GeneralRegistrationState.scala:43-62): landmarks matched by id,
    (nearest REFERENCE vertex id, target landmark point, the model landmark's covariance or I3) -- the arguments of
    GingrAlgorithm.setLandmarks / gingr_registration_set_landmarks."""
    ref = np.asarray(reference_points, dtype=float).reshape(-1, 3)
    tgt = {lm.id: lm for lm in target_landmarks}
    pids, pts, covs = [], [], []
    for lm in model_landmarks:
        if lm.id not in tgt:
            continue
        d = np.sum((ref - lm.point[None, :]) ** 2, axis=1)
        pids.append(int(np.argmin(d)))                      # lowest index on ties
        pts.append(tgt[lm.id].point)
        covs.append(np.eye(3) if lm.covariance is None else lm.covariance)
    return np.asarray(pids, dtype=np.int32), np.asarray(pts, dtype=float).reshape(-1, 3), np.asarray(covs, dtype=float).reshape(-1, 3, 3)


# ---------------------------------------------------------------------------------------------
# meshes
# ---------------------------------------------------------------------------------------------
def _merge_vertices(corners: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
    """[T, 3, 3] float32 triangle corners -> (vertices [n, 3] float64 in order of first appearance, triangles [T, 3])."""
    flat = np.ascontiguousarray(corners.reshape(-1, 3))
    key = flat.view([("x", flat.dtype), ("y", flat.dtype), ("z", flat.dtype)]).reshape(-1)
    _, first, inverse = np.unique(key, return_index=True, return_inverse=True)
    order = np.argsort(first)                               # unique entries by first appearance
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    verts = flat[first[order]].astype(np.float64)
    tri = rank[inverse].reshape(-1, 3).astype(np.int32)
    return verts, tri


def read_stl(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """Binary or ASCII STL -> (vertices [n, 3] float64, triangles [T, 3] int32); identical corners are merged."""
    with open(path, "rb") as f:
        raw = f.read()
    if len(raw) >= 84:
        (nt,) = struct.unpack_from("<I", raw, 80)
        if len(raw) == 84 + 50 * nt:
            rec = np.frombuffer(raw, dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]), count=nt, offset=84)
            return _merge_vertices(rec["v"])
    try:
        text = raw.decode("ascii", errors="strict")
    except UnicodeDecodeError:
        text = ""
    if not text.lstrip().startswith("solid"):
        raise ValueError(f"{path}: neither a binary STL (size mismatch) nor an ASCII STL")
    vals = [ln.split()[1:4] for ln in text.splitlines() if ln.strip().startswith("vertex")]
    try:
        corners = np.asarray(vals, dtype=np.float32)
    except ValueError:
        raise ValueError(f"{path}: malformed ASCII STL (vertex records)")
    if corners.size == 0 or corners.ndim != 2 or corners.shape[1] != 3 or corners.shape[0] % 3 != 0:
        raise ValueError(f"{path}: malformed ASCII STL")
    return _merge_vertices(corners.reshape(-1, 3, 3))


def write_stl(path: str, vertices, triangles) -> None:
    """Binary STL (facet normals computed from the corners)."""
    v = np.asarray(vertices, dtype=np.float32)
    t = np.asarray(triangles, dtype=np.int64).reshape(-1, 3)
    c = v[t]
    n = np.cross(c[:, 1] - c[:, 0], c[:, 2] - c[:, 0])
    ln = np.linalg.norm(n, axis=1, keepdims=True)
    n = np.where(ln > 0, n / np.where(ln > 0, ln, 1), 0).astype(np.float32)
    rec = np.zeros(len(t), dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]))
    rec["n"], rec["v"] = n, c
    with open(path, "wb") as f:
        f.write(b"gingr-b200".ljust(80, b" "))
        f.write(struct.pack("<I", len(t)))
        f.write(rec.tobytes())


_PLY_TYPES = {"char": "i1", "int8": "i1", "uchar": "u1", "uint8": "u1", "short": "i2", "int16": "i2", "ushort": "u2",
              "uint16": "u2", "int": "i4", "int32": "i4", "uint": "u4", "uint32": "u4", "float": "f4", "float32": "f4",
              "double": "f8", "float64": "f8"}


def read_ply(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """PLY (ascii, binary_little_endian or binary_big_endian) with a vertex element (x, y, z + any other scalar
    properties) and a face element with one list property of triangles -> (vertices float64, triangles int32).
    A truncated, inconsistent or non-triangle file raises ValueError (scalismo's MeshIO returns a failed Try)."""
    try:
        verts, tris = _read_ply(path)
    except (IndexError, KeyError, UnicodeDecodeError) as e:
        raise ValueError(f"{path}: malformed PLY ({type(e).__name__}: {e})")
    if verts is None:
        raise ValueError(f"{path}: no vertex element")
    tris = np.zeros((0, 3), dtype=np.int32) if tris is None else tris
    if tris.size and (tris.min() < 0 or tris.max() >= verts.shape[0]):
        raise ValueError(f"{path}: face index out of range")
    return verts, tris


def _read_ply(path: str):
    with open(path, "rb") as f:
        raw = f.read()
    end = raw.find(b"end_header")
    if not raw.startswith(b"ply") or end < 0:
        raise ValueError(f"{path}: not a PLY file")
    header = raw[:end].decode("ascii").splitlines()
    body = raw[raw.index(b"\n", end) + 1:]
    fmt, elements = None, []
    for ln in header:
        tok = ln.split()
        if not tok:
            continue
        if tok[0] == "format":
            fmt = tok[1]
        elif tok[0] == "element":
            elements.append({"name": tok[1], "count": int(tok[2]), "props": []})
        elif tok[0] == "property":
            if tok[1] == "list":
                elements[-1]["props"].append(("list", tok[2], tok[3], tok[4]))
            else:
                elements[-1]["props"].append(("scalar", tok[1], tok[2]))
    if fmt not in ("ascii", "binary_little_endian", "binary_big_endian"):
        raise ValueError(f"{path}: unsupported PLY format {fmt}")
    verts, tris = None, None
    if fmt == "ascii":
        lines = body.decode("ascii").split("\n")
        pos = 0
        for el in elements:
            rows = [ln.split() for ln in lines[pos:pos + el["count"]]]
            pos += el["count"]
            if el["name"] == "vertex":
                names = [p[2] for p in el["props"]]
                ix = [names.index(c) for c in ("x", "y", "z")]
                verts = np.asarray([[float(r[i]) for i in ix] for r in rows], dtype=np.float64).reshape(-1, 3)
            elif el["name"] == "face":
                for r in rows:
                    if int(r[0]) != 3:
                        raise ValueError(f"{path}: only triangle faces are supported")
                    if len(r) < 4:
                        raise ValueError(f"{path}: truncated face record")
                tris = np.asarray([[int(v) for v in r[1:4]] for r in rows], dtype=np.int32).reshape(-1, 3)
            if len(rows) != el["count"] or any(len(r) == 0 for r in rows):
                raise ValueError(f"{path}: element {el['name']} has fewer records than its header says")
        return verts, tris
    bo = "<" if fmt == "binary_little_endian" else ">"
    off = 0
    for el in elements:
        if all(p[0] == "scalar" for p in el["props"]):
            dt = np.dtype([(p[2], bo + _PLY_TYPES[p[1]]) for p in el["props"]])
            arr = np.frombuffer(body, dtype=dt, count=el["count"], offset=off)
            off += dt.itemsize * el["count"]
            if el["name"] == "vertex":
                verts = np.stack([arr["x"], arr["y"], arr["z"]], axis=1).astype(np.float64)
        else:
            if len(el["props"]) != 1:
                raise ValueError(f"{path}: element {el['name']} mixes list and scalar properties")
            _, ct, it, _ = el["props"][0]
            dt = np.dtype([("n", bo + _PLY_TYPES[ct]), ("v", bo + _PLY_TYPES[it], 3)])
            arr = np.frombuffer(body, dtype=dt, count=el["count"], offset=off)     # valid when every face is a triangle
            if el["count"] and not np.all(arr["n"] == 3):
                raise ValueError(f"{path}: only triangle faces are supported")
            off += dt.itemsize * el["count"]
            if el["name"] == "face":
                tris = arr["v"].astype(np.int32)
    return verts, tris


def write_ply(path: str, vertices, triangles, binary: bool = True) -> None:
    v = np.asarray(vertices, dtype=np.float32).reshape(-1, 3)
    t = np.asarray(triangles, dtype=np.int32).reshape(-1, 3)
    hdr = ["ply", "format binary_little_endian 1.0" if binary else "format ascii 1.0", "comment gingr-b200",
           f"element vertex {len(v)}", "property float x", "property float y", "property float z",
           f"element face {len(t)}", "property list uchar int vertex_indices", "end_header"]
    with open(path, "wb") as f:
        f.write(("\n".join(hdr) + "\n").encode("ascii"))
        if binary:
            f.write(v.astype("<f4").tobytes())
            rec = np.zeros(len(t), dtype=np.dtype([("n", "u1"), ("v", "<i4", 3)]))
            rec["n"], rec["v"] = 3, t
            f.write(rec.tobytes())
        else:
            for p in v:
                f.write(f"{float(p[0])!r} {float(p[1])!r} {float(p[2])!r}\n".encode("ascii"))
            for q in t:
                f.write(f"3 {q[0]} {q[1]} {q[2]}\n".encode("ascii"))


def read_mesh(path: str) -> Tuple[np.ndarray, np.ndarray]:
    """MeshIO.readMesh by extension (.stl, .ply)."""
    low = path.lower()
    if low.endswith(".stl"):
        return read_stl(path)
    if low.endswith(".ply"):
        return read_ply(path)
    raise ValueError(f"unsupported mesh format: {path}")


# ---------------------------------------------------------------------------------------------
# Statistical model file (the cached GPMM of examples/DemoHelper/DemoDatasetLoader.scala:40-53)
# ---------------------------------------------------------------------------------------------
# The reference caches its low-rank models through scalismo's StatisticalModelIO as "<name>_dec-<n>_<kernel>_<pars>.h5.json".
# That container is defined inside scalismo 1.0-RC1 (build.sbt:40), which is not in the reference tree, and the tree
# holds no sample file, so its byte layout cannot be pinned here: NOT interchangeable with scalismo's reader until
# checked against a real file.  What is kept is the statismo group / dataset naming the format descends from
# (/representer/points [3, M], /representer/cells [3, T], /model/mean [3M], /model/pcaBasis [3M, r] orthonormal,
# /model/pcaVariance [r], /model/noiseVariance) inside a JSON document, with every dataset stored as
# {"dtype", "shape", "base64"} of little-endian row-major data.  Doubles are stored as doubles (scalismo narrows to
# float32), so a reloaded model is bit-identical to the one that was written.
MODEL_FILE_FORMAT = "gingr_b200.statistical_model.v1"


def _dataset(a: np.ndarray, dtype: str) -> dict:
    import base64
    arr = np.ascontiguousarray(np.asarray(a).astype(dtype, copy=False))
    return {"dtype": dtype, "shape": list(arr.shape), "base64": base64.b64encode(arr.tobytes()).decode("ascii")}


def _from_dataset(d: dict) -> np.ndarray:
    import base64
    arr = np.frombuffer(base64.b64decode(d["base64"]), dtype=d["dtype"])
    shape = tuple(int(s) for s in d["shape"])
    if arr.size != int(np.prod(shape, dtype=np.int64)):
        raise ValueError("statistical model file: dataset size does not match its shape")
    return arr.reshape(shape).copy()


def model_file_name(name: str, decimate: Optional[int], kernel_name: str, printpars: str) -> str:
    """File name of the cached model, DemoDatasetLoader.scala:46-47 (kernel names / parameter strings:
    simple/SimpleModels.scala:25-52, e.g. GaussKernel(50, 70) -> ("Gauss", "50.0_70.0"))."""
    dec = "full" if decimate is None else str(int(decimate))
    return f"{name}_dec-{dec}_{kernel_name}_{printpars}.h5.json"


def gauss_kernel_printpars(scaling: float, sigma: float) -> str:
    """GaussKernel.printpars (SimpleModels.scala:37-40): scaling.toString + "_" + sigma.toString."""
    return f"{float(scaling)!r}_{float(sigma)!r}"


def write_statistical_model(path: str, reference_points, triangles, mean, basis, variance, noise_variance: float = 0.0) -> None:
    """StatisticalModelIO.writeStatisticalTriangleMeshModel3D's role (DemoDatasetLoader.scala:51); see the layout note above."""
    ref = np.asarray(reference_points, dtype=np.float64).reshape(-1, 3)
    m = ref.shape[0]
    mean = np.asarray(mean, dtype=np.float64).reshape(-1)
    basis = np.asarray(basis, dtype=np.float64)
    variance = np.asarray(variance, dtype=np.float64).reshape(-1)
    if mean.shape[0] != 3 * m or basis.shape != (3 * m, variance.shape[0]):
        raise ValueError("statistical model: mean must be [3M], basis [3M, r], variance [r]")
    tri = np.zeros((0, 3), np.int32) if triangles is None else np.asarray(triangles, dtype=np.int32).reshape(-1, 3)
    if tri.size and (tri.min() < 0 or tri.max() >= m):
        raise ValueError("statistical model: triangle index out of range")
    doc = {
        "format": MODEL_FILE_FORMAT,
        "version": {"majorVersion": 0, "minorVersion": 9},
        "representer": {"name": "gingr_b200", "datasetType": "POLYGON_MESH",
                        "points": _dataset(ref.T, "<f8"), "cells": _dataset(tri.T, "<i4")},
        "model": {"mean": _dataset(mean, "<f8"), "pcaBasis": _dataset(basis, "<f8"),
                  "pcaVariance": _dataset(variance, "<f8"), "noiseVariance": float(noise_variance)},
    }
    with open(path, "w") as f:
        json.dump(doc, f)


def read_statistical_model(path: str):
    """-> (reference points [M, 3], triangles [T, 3] int32, mean [3M], basis [3M, r], variance [r]).  Raises (the
    reference's Try fails, DemoDatasetLoader.scala:48) on a missing, foreign or inconsistent file."""
    with open(path) as f:
        doc = json.load(f)
    if not isinstance(doc, dict) or doc.get("format") != MODEL_FILE_FORMAT:
        raise ValueError(f"{path}: not a {MODEL_FILE_FORMAT} file")
    ref = _from_dataset(doc["representer"]["points"]).T.copy()
    tri = _from_dataset(doc["representer"]["cells"]).T.astype(np.int32).copy()
    mean = _from_dataset(doc["model"]["mean"])
    basis = _from_dataset(doc["model"]["pcaBasis"])
    var = _from_dataset(doc["model"]["pcaVariance"])
    m = ref.shape[0]
    if ref.ndim != 2 or ref.shape[1] != 3 or mean.shape != (3 * m,) or basis.shape != (3 * m, var.shape[0]):
        raise ValueError(f"{path}: inconsistent dataset shapes")
    if tri.size and (tri.min() < 0 or tri.max() >= m):
        raise ValueError(f"{path}: triangle index out of range")
    return ref, tri, mean, basis, var


def load_or_create_model(ctx, directory: str, name: str, reference_points, triangles, kernelSelect,
                         decimate: Optional[int] = None, relativeTolerance: float = 0.01):
    """DataSetLoader.model(decimate, kernelSelect, ...) (DemoDatasetLoader.scala:40-53): read the cached model when its
    file exists, else build it ON THE DEVICE (api.SimpleTriangleModels3D.create) and write the file.  The caller passes
    the (already decimated) reference; kernelSelect is api.GaussKernel / api.GaussSymKernel / api.InvLapKernel / api.GaussMixKernel; -> gingr_b200.api.Model."""
    import os
    from . import api
    path = os.path.join(directory, model_file_name(name, decimate, kernelSelect.name, kernelSelect.printpars))
    try:
        ref, tri, mean, basis, var = read_statistical_model(path)
        return api.Model(ctx, ref, mean, basis, var, tri if tri.size else None)
    except (OSError, ValueError, KeyError):
        pass
    model = api.SimpleTriangleModels3D.create(ctx, reference_points, triangles, kernelSelect, relativeTolerance)
    ref, mean, basis, var = model.download()
    write_statistical_model(path, ref, triangles, mean, basis, var)
    return model


def load_or_create_gauss_model(ctx, directory: str, name: str, reference_points, triangles, scaling: float, sigma: float,
                               decimate: Optional[int] = None, relativeTolerance: float = 0.01):
    """load_or_create_model with GaussKernel(scaling, sigma)."""
    from . import api
    return load_or_create_model(ctx, directory, name, reference_points, triangles, api.GaussKernel(scaling, sigma), decimate,
                                relativeTolerance)
