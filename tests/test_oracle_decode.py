"""Pins oracle/decode_ref.py + oracle/pnp_ref.py against the golden vectors the
unmodified reference produced (tests/golden/decode_*.npz, gpfit_moments.npz) and
against cv2.solvePnPGeneric directly."""
import copy

import numpy as np
import pytest

from centerpose_b200 import _lib as L
from centerpose_b200 import synth
from oracle import decode_ref, pnp_ref
from tests.util import DETS_KEYS, compare_records, decode_case_geometry, decode_case_inputs, golden, oracle_records

CASES = ["decode_rep1_3obj", "decode_rep1_10obj_noisy", "decode_rep0_3obj", "decode_rep4_2obj", "decode_rep4_5pts_epnp",
         "decode_track_rep1_3obj", "decode_rep1_3obj_modern_torch", "decode_cls3_rep1_6obj", "decode_scale075_rep1_3obj",
         "decode_scale125_rep0_nonms"]


def _params(g):
    _, _, scales, nms = decode_case_geometry(g)
    return decode_ref.DecodeParams(K=100, rep_mode=int(g["rep_mode"]), use_moments=bool(int(g["tracking"])),
                                   balance=2.0, vis_thresh=float(g["vis_thresh"]), category=str(g["category"]),
                                   modern_bool=bool(int(g["modern_bool"])) if "modern_bool" in g.files else False,
                                   nms=nms, num_scales=len(scales))


def _check_golden(name):
    g = golden(name)
    hb, truths = decode_case_inputs(g)
    prm = _params(g)
    c, s, scales, _ = decode_case_geometry(g)
    for b in range(int(g["batch"])):
        dets, recs = oracle_records({k: v[b] for k, v in hb.items()}, prm, g["cam"], 512, 512, c, s, L, scale=scales[0])
        valid = g["dets%d_scores" % b][:, 0] > 0.05          # the tied sub-threshold tail is order-undefined
        for k in DETS_KEYS:
            want = g["dets%d_%s" % (b, k)]
            tol = 2e-6 if k in ("kps_displacement_std", "obj_scale_uncertainty") else 0.0
            assert np.abs(dets[k][valid] - want[valid]).max() <= tol, (name, b, k)
        want_recs = g["records%d" % b]
        assert recs.shape == want_recs.shape
        assert (recs[:, L.P_SRC_INDEX] == want_recs[:, L.P_SRC_INDEX]).all()      # same detections, same order
        compare_records(recs, want_recs, L, tol_px=1e-9, tol_q=1e-6)


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference_golden(name):
    _check_golden(name)


def test_oracle_matches_live_reference():
    """Three single planted frames -- five objects whose two keypoint estimates disagree by 2 px, the tracking heads,
    rep_mode 3 -- against what the reference's decode, post-process, soft-NMS and PnP returned for them."""
    for name in ("decode_rep1_5obj", "decode_track_rep1_2obj", "decode_rep3_3obj"):
        _check_golden(name)


def test_pnp_matches_cv2():
    """SOLVEPNP_ITERATIVE (cuboid_pnp_solver.py:165-171) is the arithmetic oracle for the PnP stage."""
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(5)
    cam = synth.default_camera(512, 512)
    worst_q = worst_t = 0.0
    for trial in range(60):
        scale = np.array([rng.uniform(0.3, 2), rng.uniform(0.5, 1.5), rng.uniform(0.3, 2)], np.float32)
        V = pnp_ref.cuboid_vertices(scale)
        R = synth._rand_rot(rng)
        tz = rng.uniform(2.5, 7)
        t = np.array([rng.uniform(-.3, .3) * tz, rng.uniform(-.3, .3) * tz, tz])
        pts = np.repeat(pnp_ref.project(V, R, t, cam), 2, axis=0) + rng.normal(0, rng.choice([0.0, 1.0, 4.0]), (16, 2))
        for j in range(8):
            if rng.uniform() < 0.3:
                pts[2 * j + 1] = [-10000, -10000]
        sol = pnp_ref.solve_pnp(pts, V, cam, opencv_return=True)
        ok = pts[:, 0] > -5000
        X = np.array([V[i // 2] for i in range(16)])[ok]
        _, rv, tv, err = cv2.solvePnPGeneric(X, pts[ok], cam, np.zeros((4, 1)), flags=cv2.SOLVEPNP_ITERATIVE)
        q = pnp_ref.mat_to_quat(pnp_ref.rodrigues(rv[0].reshape(3)))
        q2 = np.asarray(sol["quaternion"])
        if q @ q2 < 0:
            q2 = -q2
        worst_q = max(worst_q, np.abs(q - q2).max())
        worst_t = max(worst_t, np.abs(tv[0].reshape(3) - sol["location"]).max() / np.linalg.norm(tv[0]))
        assert abs(sol["reproj_err"] - err.flatten()[0]) <= 1e-6
    assert worst_q <= 1e-6 and worst_t <= 1e-6, (worst_q, worst_t)


def test_soft_nms_hand_case():
    """Two heavily overlapping boxes: the weaker one is decayed by exp(-iou^2/0.5) and dropped below threshold."""
    a = {"bbox": np.array([0., 0., 99., 99.]), "score": 0.9, "id": 0}
    b = {"bbox": np.array([0., 0., 99., 99.]), "score": 0.6, "id": 1}
    c = {"bbox": np.array([300., 300., 340., 340.]), "score": 0.5, "id": 2}
    boxes = [copy.deepcopy(b), copy.deepcopy(a), copy.deepcopy(c)]
    n = decode_ref.soft_nms(boxes, threshold=0.3)
    assert n == 2 and [d["id"] for d in boxes[:n]] == [0, 2]
    assert abs(boxes[0]["score"] - 0.9) < 1e-15


def test_nms_and_topk_semantics():
    heat = np.zeros((1, 6, 6), np.float32)
    heat[0, 2, 2] = 0.9
    heat[0, 2, 3] = 0.9           # plateau: both survive `hmax == heat`
    heat[0, 4, 4] = 0.5
    heat[0, 4, 5] = 0.4           # suppressed by its neighbour
    n = decode_ref.nms3x3(heat)
    assert n[0, 2, 2] == np.float32(0.9) and n[0, 2, 3] == np.float32(0.9) and n[0, 4, 5] == 0 and n[0, 4, 4] == 0.5
    sc, ind, ys, xs = decode_ref.topk_channel(n, 4)
    assert list(ind[0][:3]) == [14, 15, 28] and sc[0][3] == 0.0 and ind[0][3] == 0   # ties -> lowest index first


def test_moments_matches_reference_gpfit():
    from oracle.make_golden import gpfit_windows
    g = golden("gpfit_moments")
    for w, m, fit in zip(gpfit_windows(), g["moments"], g["fitgaussian"]):
        assert np.allclose(decode_ref.moments(w), m, rtol=0, atol=0)
        assert np.allclose(decode_ref.moments(w), fit, rtol=0, atol=1e-12)
