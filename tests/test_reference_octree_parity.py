"""Parity against the reference's REAL k-NN path: nanoflann::Octree::knnNeighbors (flann/octree.h:1004-1055, called from
LocalMap::nearestKSearchSurf, LocalMap.h:509-521), on the BASELINE configurations.  Its outputs come from
tests/golden/reference_octree.npz, written by tests/golden/make_reference_octree.py with the octree compiled verbatim into the
oracle (conftest.reference_registration rebuilds them and checks their SHA-256).  The cfg2 / cfg3 scans are taken every 8th
point (conftest.OCTREE_CASES) so that the stored neighbour rows stay small.

The reference octree is not an exact k-NN (`inside()` tests x on all three axes, the root bbox update compares x against
the y/z maxima and writes min[2] for max[2]: octree.h:383-385,984-1001); this library searches exactly inside the block
(SURVEY Appendix C).  Two statements are proven here, per configuration:

  (A) INJECTION: with the octree's own neighbour sets fed into the GPU stages after the search (so_register_injected), the
      GPU registration equals the octree-in-the-loop oracle: same accept/reject counts, same ICP and LM trip counts, pose
      within the north-star tolerance (1e-4 m / 1e-4 rad; observed ~1e-12).  Hence the k-NN is the ONLY deviation.
  (B) BOUND: the deviation the exact search causes -- GPU exact vs octree-in-the-loop -- is recorded (mismatching queries,
      |dpos|, |drot|) and bounded (<= 5e-4 m / 5e-4 rad), and the exact result is not farther from ground truth than the
      octree result beyond that bound.  The numbers are printed.
"""
import json

import numpy as np
import pytest

from conftest import OCTREE_CASES, get_case, quat_angle, reference_registration

pytestmark = pytest.mark.gpu

CASES = [(name, cap) for name, cap, _ in OCTREE_CASES]
STRIDE = {(name, cap): stride for name, cap, stride in OCTREE_CASES}


def _ctx(api, case):
    ctx = api.Context(max_map_points=len(case["map_xyzi"]) + 1024, max_scan_points=262144, plane_res=case["cfg"]["plane_res"])
    ctx.map_set_points(case["map_xyzi"])
    return ctx


def _record(key, row):
    print(f"[octree-parity] {key}: {json.dumps(row)}")


def _reference(oracle_mod, name, cap):
    case = get_case(name)
    scan = case["scan_xyzi"][::STRIDE[(name, cap)]]
    om = oracle_mod.OracleMap(case["map_xyzi"], ref_octree=False)
    ro, trace, status = reference_registration(f"{name}_cap{cap}", om, scan, case["pose_prior"], case["cfg"], cap)
    return case, scan, om, ro, trace, status


@pytest.mark.parametrize("name,cap", CASES)
def test_injected_reference_octree_neighbours_reproduce_the_reference_path(gpu_api, oracle_mod, name, cap):
    case, scan, om, ro, trace, _ = _reference(oracle_mod, name, cap)
    cfg, prior = case["cfg"], case["pose_prior"]
    n = ro.n_iterations
    ctx = _ctx(gpu_api, case)
    r = ctx.register_injected(scan, prior, cfg["max_iterations"], trace, cap)
    assert r.status == 0
    # (A) identical control flow and counts, pose far inside the tolerance
    assert r.n_iterations == n
    assert list(r.iter_n_surf[:n]) == list(ro.iter_n_surf[:n])
    assert list(r.iter_lm_steps[:n]) == list(ro.iter_lm_steps[:n])
    assert list(r.iter_lm_successful[:n]) == list(ro.iter_lm_successful[:n])
    assert list(r.iter_lm_termination[:n]) == list(ro.iter_lm_termination[:n])
    assert list(r.hist_obs) == list(ro.hist_obs) and list(r.hist_reject_plane) == list(ro.hist_reject_plane)
    pg, po = np.array(r.pose), np.array(ro.pose)
    dpos, drot = float(np.abs(pg[:3] - po[:3]).max()), float(quat_angle(pg[3:], po[3:]))
    assert dpos <= 1e-4 and drot <= 1e-4, (dpos, drot)
    assert dpos <= 1e-9 and drot <= 1e-7, ("expected ~1e-12: the stages after the search are the same arithmetic", dpos, drot)
    assert np.allclose(r.iter_cost[:n], ro.iter_cost[:n], rtol=1e-9)
    cg, co = np.array(r.cov).reshape(6, 6), np.array(ro.cov).reshape(6, 6)
    assert np.abs(cg - co).max() <= 1e-6 * np.abs(co).max()
    _record(f"{name}_cap{cap}_injected", {"icp_iterations": n, "dpos_m": dpos, "drot_rad": drot, "n_ok_last": int(ro.iter_n_surf[n - 1])})
    ctx.close()


@pytest.mark.parametrize("name,cap", CASES)
def test_exact_knn_deviation_from_reference_octree_is_bounded(gpu_api, oracle_mod, name, cap):
    case, scan, om, ro, trace, status2 = _reference(oracle_mod, name, cap)                                  # reference octree in the loop
    cfg, prior, truth = case["cfg"], case["pose_prior"], case["pose_true"]
    ctx = _ctx(gpu_api, case)
    r = ctx.register(scan, prior, cfg["max_iterations"], cap)                                                # exact in-block k-NN
    assert r.status == 0
    pg, po = np.array(r.pose), np.array(ro.pose)
    dpos, drot = float(np.linalg.norm(pg[:3] - po[:3])), float(quat_angle(pg[3:], po[3:]))
    eg = float(np.linalg.norm(pg[:3] - truth[:3]))
    eo = float(np.linalg.norm(po[:3] - truth[:3]))
    # mismatch rate of the neighbour sets at the prior pose (first ICP iteration)
    oc0, _, _ = om.correspond(scan, prior, cfg["plane_res"], cap, 0, n_threads=8)
    searched = (oc0["status"] >= 0) & (oc0["status"] != 1)
    mism = searched & (np.sort(trace[0], 1) != np.sort(oc0["nn"], 1)).any(1)
    gates = searched & (status2 != oc0["status"])
    row = {"queries": int(searched.sum()), "octree_wrong_neighbour_sets": int(mism.sum()), "mismatch_rate": float(mism.sum() / max(1, searched.sum())),
           "gate_flips": int(gates.sum()), "dpos_gpu_exact_vs_octree_m": dpos, "drot_rad": drot, "err_vs_truth_gpu_exact_m": eg,
           "err_vs_truth_octree_m": eo, "icp_iterations_gpu": int(r.n_iterations), "icp_iterations_octree": int(ro.n_iterations)}
    _record(f"{name}_cap{cap}_exact_vs_octree", row)
    assert dpos <= 5e-4 and drot <= 5e-4, row
    assert eg <= eo + 5e-4, row
    assert row["mismatch_rate"] <= 0.05, row
    ctx.close()
