"""Accuracy of the device's small symmetric eigen-solvers: the 6x6 pseudo-inverse of the covariance step and the two 3x3 block
eigenproblems behind pos_err / pos_dir / pos_inv_cond and the ori_* fields, against a 50-digit mpmath restatement of the same
operations on the device's own H, at a bar derived from cond(H) instead of from what the device happened to produce.

Besides the warehouse cases (tiny, cfg1, hall) the scenes include weakly observable geometry, the case these outputs exist to
diagnose: a 140 m corridor whose ends lie beyond the scan's 30 m range, so translation along it is pinned only by the roughness
of the map (cond(H) ~ 2e3 at 2 cm map noise, ~ 2e4 at 5 mm), the same corridor with one pillar, and a 1 mm-noise corridor in
which the plane fit's lambda0 < 1e-6 gate (LidarSlam.cpp:772) rejects about 40 % of the points.  Exactly degenerate problems
(cond(H) >~ 1e10) are out of scope: there a pseudo-inverse of the normal equations and Ceres' SVD of J legitimately cut
different directions.

test_corridor_scene_premises runs on the CPU (oracle only), so a scene that drifts out of its intended conditioning is caught
before GPU time is spent on it."""
import numpy as np
import pytest

from conftest import get_case

EPS = np.finfo(np.float64).eps
CUT_RATIO = 1e-7                  # Ceres DENSE_SVD null-space rule: singular-value ratio s_i / s_max < sqrt(1e-14)
RMAX = 30.0                       # scan range of the corridor scenes: the corridor's ends stay out of sight
CORRIDOR_ROOM = np.array([-70.0, 70.0, -2.0, 2.0, -1.8, 3.0])
PILLAR = np.array([[9.0, 9.8, 1.0, 1.6, -1.8, 3.0]])        # faces >= 1 m from the origin (plane fit A n = -1)

# name: (map noise sigma, pillar, cond(H) range at the prior, share of processed points the lambda0 gate rejects)
CORRIDORS = {
    "corridor_20mm": (0.02, False, (5e2, 1e4), (0.0, 0.05)),
    "corridor_5mm": (0.005, False, (5e3, 1e5), (0.0, 0.05)),
    "corridor_5mm_pillar": (0.005, True, (2e2, 5e3), (0.0, 0.05)),
    "corridor_1mm": (0.001, False, (5e3, 2e5), (0.3, 0.55)),
}
# (case, max_surface_features) of the isolated covariance-step check
COV_CASES = [("tiny", 0), ("cfg1", 2000), ("cfg1", 0), ("hall", 0)] + [(name, 0) for name in CORRIDORS]
_corridors = {}


def corridor_case(name):
    """Corridor scene, map (voxel-filtered at planeRes 0.2), VLP-16 scan cut at 30 m, truth and prior; cached per session."""
    if name not in _corridors:
        from superodom_b200 import synth
        noise, pillar, _, _ = CORRIDORS[name]
        scene = synth.Scene(room=CORRIDOR_ROOM.copy(), boxes=PILLAR.copy() if pillar else np.zeros((0, 6)))
        raw = synth.sample_surfaces(scene, 0.2, seed=31, noise=noise)
        map_xyzi = synth.voxel_filter_blocks(np.concatenate([raw, np.ones((len(raw), 1), np.float32)], 1), 0.2)
        pose_true = np.r_[3.3, 0.25, 0.1, synth.quat_from_rotvec(np.array([0.0, 0.0, 0.12]))]
        scan = synth.make_scan(scene, "vlp16", pose_true, 4100, rmax=RMAX)
        prior = synth.perturb_pose(pose_true, 4200, dt=0.05, dth_deg=0.5)
        _corridors[name] = dict(scene=scene, map_xyzi=map_xyzi, scan_xyzi=scan, pose_true=pose_true, pose_prior=prior,
                                cfg=dict(plane_res=0.2, max_iterations=5))
    return _corridors[name]


def any_case(name):
    return corridor_case(name) if name in CORRIDORS else get_case(name)


def _ctx(api, case):
    ctx = api.Context(max_map_points=max(1 << 20, len(case["map_xyzi"]) + 1024), max_scan_points=262144,
                      plane_res=case["cfg"]["plane_res"])
    ctx.map_set_points(case["map_xyzi"])
    return ctx


# ---------------------------------------------------------------------------------------------------------------
# 50-digit reference of the covariance step (ceres::Covariance DENSE_SVD on H, then EstimateRegistrationError)
# ---------------------------------------------------------------------------------------------------------------
def _eigsy(mp, M):
    """ascending eigenvalues (list of mpf) and eigenvectors (mp.matrix, columns) of a symmetric mp.matrix"""
    E, Q = mp.eigsy(M)
    order = sorted(range(M.rows), key=lambda k: E[k])
    V = mp.matrix(M.rows, M.rows)
    for c, k in enumerate(order):
        for i in range(M.rows):
            V[i, c] = Q[i, k]
    return [E[k] for k in order], V


def covariance_reference(H):
    """-> dict of float64 results of the covariance step on the float64 matrix H, computed with 50 significant digits."""
    from mpmath import mp
    with mp.workdps(50):
        return _covariance_reference(mp, H)


def _covariance_reference(mp, H):
    A = mp.matrix([[mp.mpf(float(H[i, j])) for j in range(6)] for i in range(6)])
    w, V = _eigsy(mp, A)
    lmax = w[5]
    inv = [mp.mpf(0)] * 6
    ratios = []
    cut = False
    for k in range(5, -1, -1):                          # descending singular values: a cut direction cuts every smaller one
        ratio = mp.sqrt(w[k] / lmax) if w[k] > 0 else mp.mpf(0)
        ratios.append(float(ratio))
        cut = cut or ratio < CUT_RATIO
        inv[k] = mp.mpf(0) if cut else 1 / w[k]
    C = mp.matrix(6, 6)
    for i in range(6):
        for j in range(6):
            C[i, j] = mp.fsum(V[i, k] * inv[k] * V[j, k] for k in range(6))
    out = dict(cov=np.array([[float(C[i, j]) for j in range(6)] for i in range(6)]), cond=float(w[5] / w[0]),
               min_ratio=min(ratios), H_eig=np.array([float(x) for x in w]))
    for key, o, scale in (("pos", 0, mp.mpf(1)), ("ori", 3, 180 / mp.pi)):
        B = mp.matrix([[C[o + i, o + j] for j in range(3)] for i in range(3)])
        e, E = _eigsy(mp, B)
        out[key + "_eig"] = np.array([float(x) for x in e])
        out[key + "_err"] = float(mp.sqrt(e[2]) * scale)
        out[key + "_inv_cond"] = float(mp.sqrt(e[0] / e[2]))
        out[key + "_dir"] = np.array([float(E[i, 2]) for i in range(3)])
    return out


def assert_covariance_matches(r, ref, rel_bar):
    """r: an IcpResult.  cov within rel_bar * max|cov| per entry; the block eigen results within what that cov error (plus a
    backward-stable 3x3 solve) allows; the largest-eigenvalue directions, up to sign, where the eigen-gap defines them."""
    cg, co = np.array(r.cov).reshape(6, 6), ref["cov"]
    err = np.abs(cg - co).max() / np.abs(co).max()
    assert err <= rel_bar, f"cov: max|dC|/max|C| = {err:.3e} > {rel_bar:.3e} (cond(H) = {ref['cond']:.3e})"
    delta = rel_bar * np.abs(co).max()                  # per-entry error bound of cov
    for key, unit in (("pos", 1.0), ("ori", 180.0 / np.pi)):
        e = ref[key + "_eig"]
        tol = 3.0 * delta + 16.0 * EPS * e[2]           # ||dB||_2 <= 3 max|dB_ij|, plus the block solver's own rounding
        got_err = getattr(r, key + "_err" if key == "pos" else "ori_err_deg")
        bar = unit * tol / (2.0 * np.sqrt(e[2])) + 4.0 * EPS * ref[key + "_err"]
        assert abs(got_err - ref[key + "_err"]) <= bar, (key, got_err, ref[key + "_err"], bar)
        got_ic = getattr(r, key + "_inv_cond")
        bar = ref[key + "_inv_cond"] * (0.5 * tol * (1.0 / e[0] + 1.0 / e[2]) + 4.0 * EPS)
        assert abs(got_ic - ref[key + "_inv_cond"]) <= bar, (key, got_ic, ref[key + "_inv_cond"], bar)
        gap = e[2] - e[1]
        if gap > 1e3 * tol:                             # direction error <= ||dB|| / gap
            d = np.array(getattr(r, key + "_dir"))
            dd = min(np.abs(d - ref[key + "_dir"]).max(), np.abs(d + ref[key + "_dir"]).max())
            assert dd <= 4.0 * tol / gap + 8.0 * EPS, (key, dd, tol / gap)


def cov_bar(cond):
    return 16.0 * EPS * cond


# ---------------------------------------------------------------------------------------------------------------
# CPU: the scenes are what they are meant to be
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", list(CORRIDORS))
def test_corridor_scene_premises(oracle_mod, name):
    """cond(H) of the correspondences at the prior lies in the scene's intended range (far from the exactly degenerate
    regime and from the cut rule), the corridor's ends are out of the scan's sight, and the lambda0 < 1e-6 gate rejects
    the intended share of the processed points."""
    case = corridor_case(name)
    _, _, (clo, chi), (glo, ghi) = CORRIDORS[name]
    assert np.linalg.norm(case["scan_xyzi"][:, :3], axis=1).max() < RMAX
    assert min(case["pose_true"][0] - CORRIDOR_ROOM[0], CORRIDOR_ROOM[1] - case["pose_true"][0]) > RMAX + 5.0
    om = oracle_mod.OracleMap(case["map_xyzi"])
    oc, _, ohr = om.correspond(case["scan_xyzi"], case["pose_prior"], 0.2, 0, 0, n_threads=8)
    H = oracle_mod.evaluate(oc, case["pose_prior"], 0.2)[0]
    w = np.linalg.eigvalsh(H)
    assert w[0] > 0 and clo <= w[-1] / w[0] <= chi, (name, w[-1] / w[0])
    processed = (oc["status"] >= 0).sum()
    lam0 = (oc["status"] == 3) & (oc["eigval"][:, 0] < 1e-6)
    share = lam0.sum() / processed
    assert glo <= share <= ghi, (name, share)
    assert ohr[0] > 10000


def test_covariance_reference_on_known_spectra():
    """The mpmath reference itself: a matrix with a chosen spectrum and eigenbasis gives back the pseudo-inverse, the cut and
    the block results computed independently in float64 from the construction."""
    rng = np.random.default_rng(5)
    Q, _ = np.linalg.qr(rng.normal(size=(6, 6)))
    for lam in ([1e-2, 0.3, 2.0, 5.0, 40.0, 1e3], [1e-13, 0.3, 2.0, 5.0, 40.0, 1e3]):
        lam = np.array(lam)
        H = (Q * lam) @ Q.T
        H = 0.5 * (H + H.T)
        ref = covariance_reference(H)
        keep = np.sqrt(lam / lam.max()) >= CUT_RATIO
        C = (Q[:, keep] / lam[keep]) @ Q[:, keep].T
        assert np.abs(ref["cov"] - C).max() <= 1e-9 * np.abs(C).max()
        assert keep.all() == (ref["min_ratio"] >= CUT_RATIO)
        e, E = np.linalg.eigh(C[:3, :3])
        assert abs(ref["pos_err"] - np.sqrt(e[2])) <= 1e-9 * np.sqrt(e[2])
        assert min(np.abs(ref["pos_dir"] - E[:, 2]).max(), np.abs(ref["pos_dir"] + E[:, 2]).max()) < 1e-6


# ---------------------------------------------------------------------------------------------------------------
# GPU: the covariance step alone, on the device's own H
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name,cap", COV_CASES)
def test_covariance_step_against_extended_precision(gpu_api, oracle_mod, name, cap):
    """One ICP iteration (max_icp_iters=1): its correspondences are those of correspond() at the prior, and the covariance is
    taken from H at the accepted pose.  That H (re-evaluated through evaluate()) is checked to be the one the step used, then
    the device's cov and error fields are compared with the 50-digit pseudo-inverse and block eigen-decompositions of it."""
    case = any_case(name)
    pr = case["cfg"]["plane_res"]
    ctx = _ctx(gpu_api, case)
    r = ctx.register(case["scan_xyzi"], case["pose_prior"], 1, cap)
    assert r.status == 0 and r.n_iterations == 1
    gc, _, _ = ctx.correspond(case["scan_xyzi"], case["pose_prior"], cap)
    ok = gc["status"] == 0
    assert ok.sum() == r.iter_n_surf[0]
    H, g, cost = ctx.evaluate(np.array(r.pose_opt))
    assert abs(cost - r.iter_cost[0]) <= 1e-12 * r.iter_cost[0], (cost, r.iter_cost[0])          # the H at the step's final pose
    om = oracle_mod.OracleMap(case["map_xyzi"])
    oc, _, _ = om.correspond(case["scan_xyzi"], case["pose_prior"], pr, cap, 0, n_threads=8)
    assert np.array_equal(gc["status"].astype(np.int64), np.where(oc["status"] < 0, 255, oc["status"]))
    oH = oracle_mod.evaluate(oc, np.array(r.pose_opt), pr)[0]
    assert np.abs(H - oH).max() <= 1e-10 * np.abs(oH).max()
    assert np.array_equal(H, H.T)
    ref = covariance_reference(H)
    assert ref["cond"] < 1e10 and ref["min_ratio"] > 100 * CUT_RATIO, (ref["cond"], ref["min_ratio"])     # no direction near the cut
    assert_covariance_matches(r, ref, cov_bar(ref["cond"]))
    ctx.close()


# ---------------------------------------------------------------------------------------------------------------
# GPU: whole registrations on the corridor scenes against the oracle
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CORRIDORS))
def test_corridor_registration_parity(gpu_api, oracle_mod, name):
    case = corridor_case(name)
    ctx = _ctx(gpu_api, case)
    om = oracle_mod.OracleMap(case["map_xyzi"])
    r = ctx.register(case["scan_xyzi"], case["pose_prior"], 5, 0)
    ro = om.register(case["scan_xyzi"], case["pose_prior"], 0.2, 5, 0, knn_mode=0, n_threads=8)
    assert r.status == ro.status == 0
    assert list(r.hist_obs) == list(ro.hist_obs) and list(r.hist_reject_plane) == list(ro.hist_reject_plane)
    n = ro.n_iterations
    assert r.n_iterations == n
    for f in ("iter_n_surf", "iter_lm_steps", "iter_lm_successful", "iter_lm_termination"):
        assert list(getattr(r, f)[:n]) == list(getattr(ro, f)[:n]), f
    assert np.allclose(r.iter_cost[:n], ro.iter_cost[:n], rtol=1e-9)
    for a, b in ((r.pose, ro.pose), (r.pose_opt, ro.pose_opt)):
        a, b = np.array(a), np.array(b)
        assert np.abs(a[:3] - b[:3]).max() <= 1e-4
        assert 2.0 * np.arccos(min(1.0, abs(float(np.dot(a[3:], b[3:]))))) <= 1e-4
    cg, co = np.array(r.cov).reshape(6, 6), np.array(ro.cov).reshape(6, 6)
    assert np.abs(cg - co).max() <= 1e-6 * np.abs(co).max()
    for f in ("pos_err", "pos_inv_cond", "ori_err_deg", "ori_inv_cond"):
        assert abs(getattr(r, f) - getattr(ro, f)) <= 1e-6 * abs(getattr(ro, f)), f
    for key, o in (("pos", 0), ("ori", 3)):
        e = np.linalg.eigvalsh(co[o:o + 3, o:o + 3])
        if e[2] - e[1] > 1e-3 * e[2]:
            assert abs(abs(np.dot(getattr(r, key + "_dir"), getattr(ro, key + "_dir"))) - 1) < 1e-6, key
    processed = sum(ro.hist_reject_plane)
    lo, hi = CORRIDORS[name][3]
    if lo > 0:                                           # the low-noise corridor: the PCA gate really rejects a large share
        assert r.hist_reject_plane[3] >= lo * processed, (r.hist_reject_plane[3], processed)
    ctx.close()
