"""Property tests (hypothesis) of the oracle's restated third-party arithmetic against numpy: these functions carry the
"parity unpinned" part of the oracle (Eigen / Ceres / tf2 restatements), so they are checked over random inputs, not only on
the scenes the registration tests happen to produce."""
import numpy as np
import pytest
from hypothesis import given, settings, strategies as st
from hypothesis.extra import numpy as hnp

finite = st.floats(min_value=-50.0, max_value=50.0, allow_nan=False, allow_infinity=False, width=64)
# the plane fit solves on map points, which are float32: entries whose squares underflow in double (|x| < 1e-154) never reach it
point_coords = st.floats(min_value=-50.0, max_value=50.0, allow_nan=False, allow_infinity=False, width=32)


@settings(max_examples=60, deadline=None)
@given(hnp.arrays(np.float64, (5, 3), elements=point_coords))
def test_colpiv_qr_matches_lstsq_when_well_conditioned(oracle_mod, A):
    b = -np.ones(5)
    s = np.linalg.svd(A, compute_uv=False)
    if s[-1] < 1e-6 * max(s[0], 1e-300):
        return                                   # rank handling is Eigen-specific; covered by the dedicated test
    x = oracle_mod.colpiv_qr_solve(A, b)
    ref = np.linalg.lstsq(A, b, rcond=None)[0]
    assert np.allclose(x, ref, rtol=1e-8, atol=1e-8 * np.abs(ref).max())


@settings(max_examples=60, deadline=None)
@given(hnp.arrays(np.float64, (3, 3), elements=finite))
def test_sym_eig_matches_eigh(oracle_mod, M):
    S = M @ M.T                                   # scatter-like: symmetric positive semi-definite
    w, V = oracle_mod.sym_eig(S)
    wr = np.linalg.eigvalsh(S)
    scale = max(np.abs(wr).max(), 1e-300)
    assert np.all(np.diff(w) >= -1e-12 * scale) and np.allclose(w, wr, atol=1e-10 * scale)
    assert np.allclose(V @ np.diag(w) @ V.T, S, atol=1e-9 * scale) and np.allclose(V.T @ V, np.eye(3), atol=1e-10)


@settings(max_examples=60, deadline=None)
@given(hnp.arrays(np.float64, (7,), elements=finite), hnp.arrays(np.float64, (6,), elements=st.floats(-0.2, 0.2, width=64)))
def test_pose_plus_is_translation_add_and_right_multiplied_rotation(oracle_mod, x, d):
    q = x[3:]
    n = np.linalg.norm(q)
    if n < 1e-3:
        return
    x = x.copy()
    x[3:] = q / n
    y = oracle_mod.pose_plus(x, d)
    assert np.allclose(y[:3], x[:3] + d[:3], atol=1e-12) and abs(np.linalg.norm(y[3:]) - 1) < 1e-12
    from scipy.spatial.transform import Rotation as R
    dq = np.r_[d[3:] / 2.0, 1.0]
    exp = (R.from_quat(x[3:]) * R.from_quat(dq / np.linalg.norm(dq))).as_quat()
    assert min(np.abs(y[3:] - exp).max(), np.abs(y[3:] + exp).max()) < 1e-12


@settings(max_examples=40, deadline=None)
@given(st.integers(2, 400), st.integers(1, 9), st.floats(0.0, 3.0, width=32), st.integers(0, 2 ** 31 - 1))
def test_extract_uniform_is_a_subsequence_of_the_stride(oracle_mod, n, skip, block_range, seed):
    rng = np.random.default_rng(seed)
    pts = np.zeros((n, 8), np.float32)
    pts[:, :3] = rng.normal(0, 2, (n, 3)).astype(np.float32)
    dup = rng.random(n) < 0.3
    dup[0] = False
    pts[dup, :3] = pts[np.flatnonzero(dup) - 1, :3]                 # exact repeats of the predecessor are dropped
    pts[:, 5] = np.arange(n, dtype=np.float32)                      # time column = index, so the output names its source
    out = oracle_mod.extract_uniform(pts, 5, skip, block_range)
    src = out[:, 3].astype(int)
    assert np.all(np.diff(src) > 0) and np.all((src - 1) % skip == 0) and np.all(src >= 1)
    assert np.array_equal(out[:, :3], pts[src, :3])
    cand = np.arange(1, n, skip)
    dropped = np.setdiff1d(cand, src)
    d = pts[dropped, :3] - pts[dropped - 1, :3]
    assert np.all((np.abs(d[:, 0]) <= 1e-7) & (np.abs(d[:, 1]) <= 1e-7))   # a dropped point never moved in x or y


@settings(max_examples=25, deadline=None)
@given(st.integers(0, 2 ** 31 - 1))
def test_deskew_of_a_static_sensor_is_the_identity_and_inverts_under_reversed_motion(oracle_mod, seed):
    from superodom_b200 import synth
    d = synth.make_raw_sweep(300, seed=seed % 100000, with_defects=False)
    pts, st_, sp, t0 = d["points"], d["sample_times"], d["sample_poses"], d["start_time"]
    still = np.tile(sp[len(sp) // 2], (len(sp), 1))
    out, _, past = oracle_mod.deskew(pts, 5, t0, st_, still)
    assert past == 0 and np.abs(out[:, :3] - pts[:, :3]).max() <= 4e-6        # float32 store of an identity motion
    moved, start, _ = oracle_mod.deskew(pts, 5, t0, st_, sp)
    assert np.abs(moved[:, :3] - pts[:, :3]).max() > 1e-3
    # points stamped exactly at the sweep start do not move
    first = pts.copy()
    first[:, 5] = 0.0
    out0, _, _ = oracle_mod.deskew(first, 5, t0, st_, sp)
    assert np.abs(out0[:, :3] - first[:, :3]).max() <= 8e-6
