import hashlib
import os
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run by the driver with -m gpu)")


_cases = {}


def get_case(name, scan_index=0):
    """Session cache of synthetic cases (map generation is the slow part)."""
    from superodom_b200 import synth
    key = (name, scan_index)
    if key not in _cases:
        base = (name, "map")
        if base not in _cases:
            _cases[base] = synth.make_map_for(name)
        scene, map_xyzi = _cases[base]
        _cases[key] = synth.make_case_on(scene, map_xyzi, name, scan_index)
    return _cases[key]


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle as O
    O.build()
    return O


@pytest.fixture(scope="session")
def gpu_api():
    from superodom_b200 import api
    lib = api.load_library()          # raises if the extension is missing: no silent fallback
    assert lib.so_device_available(), "no sm_100 device visible"
    return api


def quat_angle(qa, qb):
    """rotation angle between two unit quaternions (xyzw), sign-insensitive"""
    d = abs(float(np.dot(qa, qb)))
    return 2.0 * np.arccos(min(1.0, d))


# ---------------------------------------------------------------------------------------------------------------
# Stored outputs of the reference's own octree k-NN (tests/golden/reference_octree.npz, tests/golden/make_reference_octree.py)
# ---------------------------------------------------------------------------------------------------------------
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# (case, max_surface_features, scan stride) of the octree-in-the-loop registrations.  The 131 072- and 240 000-point scans are
# taken every 2nd point: with the whole scans reference_octree.npz grows from 196 KB to 342 KB, more than a reviewable patch
# of the repository carries (a binary diff is base85, 5/4 of the file)
OCTREE_CASES = [("cfg1", 2000, 1), ("cfg1", 0, 1), ("cfg2", 0, 2), ("cfg3", 0, 2)]
REGISTRATION_FIELDS = ("pose", "pose_opt", "iter_n_surf", "iter_lm_steps", "iter_lm_successful", "iter_lm_termination",
                       "iter_cost", "hist_obs", "hist_reject_plane", "cov")
_reference = {}


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def x_dominant_map():
    """Block-local cloud with a dominant x extent and x, y, z value ranges far apart: the layout on which the
    reference octree's two bugs (flann/octree.h:383-385 bbox, :984-1001 inside()) cannot fire."""
    rng = np.random.default_rng(11)
    n = 40000
    x = rng.uniform(77.0, 123.0, n)
    y = rng.uniform(-9.0, 9.0, n)
    z = np.where(rng.uniform(size=n) < 0.5, -1.8, rng.uniform(-1.8, 5.0, n))
    y = np.where(rng.uniform(size=n) < 0.3, np.round(y / 4.5) * 4.5, y)
    p = np.stack([x, y, z], 1) + rng.normal(0, 0.02, size=(n, 3))
    return np.concatenate([p, np.ones((n, 1))], 1).astype(np.float32)


def octree_pin_queries(x_map, cfg1_map):
    """k-NN queries near the points of x_dominant_map() and of the cfg1 warehouse map"""
    rng = np.random.default_rng(2)
    qx = x_map[::13, :3] + rng.normal(0, 0.1, size=x_map[::13, :3].shape).astype(np.float32)
    qc = cfg1_map[::37, :3] + rng.normal(0, 0.1, size=cfg1_map[::37, :3].shape).astype(np.float32)
    return qx, qc


def hall_queries(hall_map):
    """queries near every 7th point of the hall map, then 500 scattered up to 30 m away"""
    rng = np.random.default_rng(0)
    base = hall_map[::7, :3]
    q = base + rng.normal(0, 0.12, size=base.shape).astype(np.float32)
    return np.concatenate([q, rng.uniform(-30, 30, size=(500, 3)).astype(np.float32) + q.mean(0)])


def knn_trace(om, scan, pose, plane_res, cap, knn_mode):
    """neighbour ids the oracle's correspondence step finds at `pose` ([n, 5], -1 for points the sampling skips): one ICP
    iteration's rows of OracleMap.register(nn_trace=...)"""
    c = om.correspond(scan, pose, plane_res, cap, knn_mode, n_threads=8)[0]
    return np.where(c["status"][:, None] < 0, -1, c["nn"])


def _reference_octree():
    if not _reference:
        with np.load(os.path.join(GOLDEN, "reference_octree.npz")) as z:
            _reference.update({k: z[k] for k in z.files})
    return _reference


def reference_knn(key, om, q):
    """The reference octree's k-NN (ids int64, d2 float32) of queries q in the oracle map om, rebuilt from the exact search."""
    g = _reference_octree()
    assert digest(q) == g[key + "/queries_sha"], "queries changed: regenerate tests/golden/reference_octree.npz"
    idx, d2, _ = om.knn(q, 5, 0)
    rows = g[key + "/rows"]
    idx[rows], d2[rows] = g[key + "/idx"], g[key + "/d2"]
    assert digest(idx, d2) == g[key + "/sha"], f"{key}: exact search + stored rows != the stored reference output"
    return idx, d2


def reference_registration(key, om, scan, prior, cfg, cap):
    """The registration with the reference octree in the loop on (om's map, scan, prior): its result fields, its neighbour ids
    per ICP iteration ([n_iterations, n, 5] int64, the injection input of so_register_injected) and its correspondence status
    codes at the prior, rebuilt from the exact search at the stored per-iteration poses plus the rows where the octree differs."""
    g = _reference_octree()
    p = key + "/"
    assert digest(om.xyzi, scan, prior) == g[p + "inputs_sha"], "synthetic case changed: regenerate tests/golden/reference_octree.npz"
    n, splits = int(g[p + "n_iterations"]), g[p + "row_splits"]
    trace = np.stack([knn_trace(om, scan, g[p + "poses"][k], cfg["plane_res"], cap, 0) for k in range(n)])
    for k in range(n):
        trace[k][g[p + "rows"][splits[k]:splits[k + 1]]] = g[p + "nn"][splits[k]:splits[k + 1]]
    assert digest(trace) == g[p + "trace_sha"], f"{key}: exact search + stored rows != the stored reference trace"
    status = om.correspond(scan, prior, cfg["plane_res"], cap, 0, n_threads=8)[0]["status"]
    status[g[p + "status_rows"]] = g[p + "status"]
    assert digest(status) == g[p + "status_sha"], f"{key}: stored reference status codes not reproduced"
    result = types.SimpleNamespace(n_iterations=n, **{f: g[p + f] for f in REGISTRATION_FIELDS})
    return result, trace, status
