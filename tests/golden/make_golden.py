"""Generate tests/golden/femur_golden.npz.

INPUTS come from the reference's own example data, examples/data/femur/{femur,femur_target}.stl and their landmark
JSONs in the GiNGR checkout that GINGR_REFERENCE names (the data of examples/DemoICP.scala:11-17 and
examples/DemoCPD.scala:11-17).  The vertices / triangles / landmarks are committed in the fixture, so the tests that
read it need no such checkout.

OUTPUTS are those of the CPU oracle (oracle/) at the time of generation: the reference itself cannot run here (no
JVM, scalismo and Breeze absent), so these are REGRESSION vectors on real data -- they pin the oracle and the CUDA
path to each other across commits and machines; they are not outputs of the Scala code.  Parity stays "unpinned" in
the sense of DESIGN.md.

    GINGR_REFERENCE=<GiNGR checkout> python tests/golden/make_golden.py
"""
import json
import os
import struct
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def read_binary_stl(path):
    """Binary STL -> (vertices float64 [V,3] de-duplicated in first-occurrence order, triangles int32 [T,3])."""
    raw = open(path, "rb").read()
    (ntri,) = struct.unpack_from("<I", raw, 80)
    rec = np.frombuffer(raw, dtype=np.dtype([("n", "<f4", 3), ("v", "<f4", (3, 3)), ("a", "<u2")]), count=ntri, offset=84)
    pts = rec["v"].reshape(-1, 3)
    uniq, first, inv = np.unique(pts, axis=0, return_index=True, return_inverse=True)
    order = np.argsort(first)                      # first-occurrence order (a mesh reader's natural numbering)
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    verts = uniq[order].astype(np.float64)
    tri = rank[inv.reshape(-1)].reshape(-1, 3).astype(np.int32)
    return verts, tri


def landmarks(path):
    lm = json.load(open(path))
    return [l["id"] for l in lm], np.array([l["coordinates"] for l in lm], dtype=np.float64)


def femur_gpmm(ref, rank=50, seed=7):
    """Low-rank GPMM on the femur reference: Gaussian-kernel features (sigma = 70 as in DemoDatasetLoader.scala:113),
    QR-orthonormalised, variance 50^2 * 0.9^k.  Stands in for approximateGPCholesky (SURVEY.md A7)."""
    from gingr_b200 import synthetic
    mean, basis, var = synthetic.make_gpmm(ref, rank, seed, lambda0=2500.0, decay=0.9, kernel_sigma=70.0)
    return mean, basis, var


def main():
    if not os.environ.get("GINGR_REFERENCE"):
        sys.exit("make_golden.py: set GINGR_REFERENCE to a GiNGR checkout; its examples/data/femur holds the input meshes")
    data = os.path.join(os.environ["GINGR_REFERENCE"], "examples", "data", "femur")
    from oracle import oracle
    oracle.build()
    rv, rt = read_binary_stl(os.path.join(data, "femur.stl"))
    tv, tt = read_binary_stl(os.path.join(data, "femur_target.stl"))
    ids_r, lm_r = landmarks(os.path.join(data, "femur.json"))
    ids_t, lm_t = landmarks(os.path.join(data, "femur_target.json"))
    common = [i for i in ids_r if i in ids_t]
    lm_r = np.array([lm_r[ids_r.index(i)] for i in common])
    lm_t = np.array([lm_t[ids_t.index(i)] for i in common])
    out = dict(ref_v=rv, ref_t=rt, tgt_v=tv, tgt_t=tt, lm_ref=lm_r, lm_tgt=lm_t)
    print("femur", rv.shape, rt.shape, "target", tv.shape, tt.shape, "landmarks", common)

    # ---- C2: DemoCPD on the decimated femur (uniform subsampling in place of scalismo's decimate) ----------
    sub_r, sub_t = rv[::16], tv[::16]
    mean, basis, var = femur_gpmm(sub_r)
    P1, Pt1, PX = oracle.P_reductions(oracle.cpd_P(sub_r, sub_t, 1.0, 0.0), sub_t)       # sigma2 = 1 (DemoCPD.scala:21)
    out.update(c2_P1=P1, c2_Pt1=Pt1, c2_PX=PX)
    m = oracle.Gpmm(sub_r, mean, basis, var, None)
    lm_pid, _ = oracle.nearest_vertex(lm_r, sub_r)
    lms = oracle.Landmarks(lm_pid.astype(np.int32), lm_t, np.tile(np.eye(3), (len(common), 1, 1)))
    algo = oracle.CpdAlgorithm(oracle.CpdConfig(max_iterations=100))
    st = algo.initialize(oracle.initial_state(m, sub_t, None, global_transformation=oracle.RIGID_TRANSFORMS, landmarks=lms))
    out["c2_sigma2_0"] = st.sigma2
    for it in range(1, 21):
        st = oracle.propose(algo, st)
        if it in (1, 5, 20):
            out[f"c2_alpha_{it}"] = st.params.shape.copy()
            out[f"c2_sigma2_{it}"] = st.sigma2
            out[f"c2_pose_{it}"] = np.concatenate([[st.params.scale], st.params.translation, st.params.euler])
            out[f"c2_fit_{it}"] = st.fit.copy()

    # ---- C1: DemoICP on the full femur meshes (1622 vertices, 3240 triangles) ---------------------------
    mean, basis, var = femur_gpmm(rv)
    cp, w, md, idx = oracle.closest_point_correspondence(oracle.METHOD_TRIANGULAR, rv, rt, tv, tt)
    out.update(c1_idx=idx.astype(np.int32), c1_w=w.astype(np.uint8), c1_cp=cp, c1_mean_dist=md)
    m = oracle.Gpmm(rv, mean, basis, var, rt)
    algo = oracle.IcpAlgorithm(oracle.IcpConfig(max_iterations=100, initial_sigma=1.0, end_sigma=1.0))
    st = algo.initialize(oracle.initial_state(m, tv, tt, global_transformation=oracle.NO_TRANSFORMS))
    for it in range(1, 4):
        st = oracle.propose(algo, st)
        out[f"c1_alpha_{it}"] = st.params.shape.copy()
        out[f"c1_fit_{it}"] = st.fit.copy()
    np.savez_compressed(os.path.join(HERE, "femur_golden.npz"), **out)
    print("wrote", os.path.join(HERE, "femur_golden.npz"), os.path.getsize(os.path.join(HERE, "femur_golden.npz")), "bytes")


if __name__ == "__main__":
    main()
