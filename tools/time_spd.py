"""Cholesky + back substitution alone through gingr_spd_solve (CUDA events inside the library).
usage: python tools/time_spd.py [n ...]   env GINGR_CUDA_LIB selects a variant build"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from gingr_b200 import api
ns = [int(a) for a in sys.argv[1:]] or [50, 200, 520, 2000]
ctx = api.Context(0)
out = {"lib": os.environ.get("GINGR_CUDA_LIB", "default")}
for n in ns:
    rng = np.random.default_rng(n)
    Q = rng.normal(size=(n, n + 8))
    A = Q @ Q.T / (n + 8) + np.eye(n) * 1e-3
    b = rng.normal(size=(1, n))
    api.spd_solve(ctx, A, b, reps=3)
    o = api.spd_solve(ctx, A, b, reps=20)
    L = np.linalg.cholesky(A)
    out[str(n)] = {"ms": round(o["ms"], 4), "err_L": float(np.max(np.abs(o["L"] - L)) / np.abs(L).max()),
                   "resid": float(np.max(np.abs(A @ o["x"] - b[0])))}
print(json.dumps(out))
