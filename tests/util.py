"""Shared helpers for the parity tests."""
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

# stated tolerances (BASELINE.json north_star / SURVEY.md 8d)
TOL_KP_PX = 1e-3        # keypoint pixel coordinates
TOL_QUAT = 1e-4         # sign-normalised quaternion
TOL_LOC_REL = 1e-4      # location, relative to |t|
# Network heads (stage B): max-abs <= 3e-4 * max|head| against the reference's fp32 CPU heads, on fixtures whose
# DCN offset convs have std 0.3.  (The graph amplifies fp32 rounding through ~50 layers and 16 deformable
# samplings: on these fixtures the reference's OWN fp32 CPU path is up to 6e-5 away from an fp64 evaluation of
# the same graph, and with offset std 1.5 on noise frames it is 16-23 % away, so SURVEY.md 8d's 1e-4 between two
# fp32 implementations is only meaningful relative to that floor.)  tests/test_gpu_net.py additionally requires
# the CUDA heads to be no further from the fp64 truth than 4x the reference's fp32 path + 3e-5.
TOL_HEAD_REL = 3e-4
# At 512 x 512 (the benched shape) the fp32 floor is higher: the reference's own fp32 CPU heads are 1.2e-4 .. 2.6e-4
# of max|head| away from the fp64 evaluation (64x more positions, 128-wide deformable sampling), so the bar between
# two fp32-equivalent implementations is 1e-3 there -- always together with the fp64-truth criterion
# (gpu-vs-fp64 <= 4 x reference-fp32-vs-fp64 + 3e-5).
TOL_HEAD_REL_512 = 1e-3


def golden(name):
    return np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False)


def net_case_inputs(g):
    """Regenerate the inputs of a net_*.npz fixture from its seeds (see oracle/make_golden.py)."""
    B, H, W, iseed, trk = int(g["batch"]), int(g["H"]), int(g["W"]), int(g["iseed"]), int(g["tracking"])
    rng = np.random.default_rng(iseed)
    x = rng.standard_normal((B, 3, H, W)).astype(np.float32)
    extra = {}
    if trk:
        extra["pre_img"] = rng.standard_normal((B, 3, H, W)).astype(np.float32)
        extra["pre_hm"] = rng.random((B, 1, H, W)).astype(np.float32)
        extra["pre_hm_hp"] = rng.random((B, 8, H, W)).astype(np.float32)
    return x, extra


def dcn_case_inputs(g):
    B, C, H, W, Co, seed, off_std = [g[k].item() for k in ("B", "C", "H", "W", "Co", "seed", "off_std")]
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((B, 18, H, W)) * off_std).astype(np.float32)
    mask = rng.random((B, 9, H, W)).astype(np.float32)
    w = (rng.standard_normal((Co, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    bias = rng.standard_normal(Co).astype(np.float32)
    return x, off, mask, w, bias


def decode_case_inputs(g):
    from centerpose_b200 import synth
    heads = dict(synth.TRACKING_HEADS if int(g["tracking"]) else synth.DEFAULT_HEADS)
    if "num_classes" in g.files:
        heads["hm"] = int(g["num_classes"])
    drop = tuple(int(v) for v in g["drop_joints"]) if "drop_joints" in g.files else ()
    hb, truths = synth.planted_batch(int(g["batch"]), n_obj=int(g["n_obj"]), seed=int(g["seed"]), heads=heads,
                                     disagree_px=float(g["disagree_px"]), drop_joints=drop)
    return hb, truths


DETS_KEYS = ("bboxes", "scores", "kps", "clses", "obj_scale", "obj_scale_uncertainty", "tracking", "tracking_hp",
             "kps_displacement_mean", "kps_displacement_std", "kps_heatmap_mean", "kps_heatmap_std",
             "kps_heatmap_height")


def compare_records(got, want, L, tol_px=TOL_KP_PX, tol_q=TOL_QUAT, check_pnp=True):
    """got / want: [n,192] pose records (same n).  Returns a dict of max errors and asserts the stated tolerances."""
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    err = {}
    if got.shape[0] == 0:
        return err

    def mx(a, n):
        return np.abs(got[:, a:a + n] - want[:, a:a + n]).max()
    err["score"] = mx(L.P_SCORE, 1)
    err["px"] = max(mx(L.P_BBOX, 4), mx(L.P_CT, 2), mx(L.P_KPS, 16), mx(L.P_KPS_DISP_MEAN, 16), mx(L.P_KPS_HM_MEAN, 16))
    err["std"] = max(mx(L.P_KPS_HM_STD, 16), mx(L.P_KPS_DISP_STD, 16))
    err["misc"] = max(mx(L.P_KPS_HM_HEIGHT, 8), mx(L.P_OBJ_SCALE, 6), mx(L.P_TRACKING, 18))
    assert err["score"] <= 2e-6, err
    assert err["px"] <= tol_px, err
    std_mag = max(np.abs(want[:, L.P_KPS_HM_STD:L.P_KPS_HM_STD + 16]).max(),
                  np.abs(want[:, L.P_KPS_DISP_STD:L.P_KPS_DISP_STD + 16]).max())
    assert err["std"] <= 5e-7 * std_mag + 1e-6, err          # fp32 products (incl. the -10000 * ratio * 0.32 sentinels)
    assert err["misc"] <= 1e-5, err
    if check_pnp:
        for i in range(got.shape[0]):
            ws = int(want[i, L.P_STATUS])
            gs = int(got[i, L.P_STATUS])
            if ws == -1:      # the reference only says "None" (z<0 / too few points / solver failure)
                assert gs in (L.PNP_BEHIND, L.PNP_FEW_POINTS, L.PNP_SOLVER_FAIL), (i, gs)
                continue
            assert gs == ws, (i, gs, ws)
            if ws in (L.PNP_OK, L.PNP_INVISIBLE):
                q1 = want[i, L.P_QUAT:L.P_QUAT + 4]
                q2 = got[i, L.P_QUAT:L.P_QUAT + 4]
                if np.dot(q1, q2) < 0:
                    q2 = -q2
                err["quat"] = max(err.get("quat", 0), np.abs(q1 - q2).max())
                t1 = want[i, L.P_LOCATION:L.P_LOCATION + 3]
                t2 = got[i, L.P_LOCATION:L.P_LOCATION + 3]
                err["loc_rel"] = max(err.get("loc_rel", 0), np.abs(t1 - t2).max() / np.linalg.norm(t1))
                err["proj_px"] = max(err.get("proj_px", 0), np.abs(
                    want[i, L.P_PROJ_CUBOID:L.P_PROJ_CUBOID + 16] - got[i, L.P_PROJ_CUBOID:L.P_PROJ_CUBOID + 16]).max())
                err["kps3d_rel"] = max(err.get("kps3d_rel", 0), np.abs(
                    want[i, L.P_KPS_3D_CAM:L.P_KPS_3D_CAM + 27] - got[i, L.P_KPS_3D_CAM:L.P_KPS_3D_CAM + 27]).max()
                    / np.linalg.norm(t1))
                err["kps_pnp"] = max(err.get("kps_pnp", 0), np.abs(
                    want[i, L.P_KPS_PNP:L.P_KPS_PNP + 18] - got[i, L.P_KPS_PNP:L.P_KPS_PNP + 18]).max())
        assert err.get("quat", 0) <= tol_q, err
        assert err.get("loc_rel", 0) <= TOL_LOC_REL, err
        assert err.get("proj_px", 0) <= 2e-3, err
        assert err.get("kps3d_rel", 0) <= TOL_LOC_REL, err
        assert err.get("kps_pnp", 0) <= 1e-5, err
    return err


def decode_case_geometry(g):
    """(c, s, scales, nms) of a decode_*.npz fixture; older fixtures are single-scale 512 x 512 frames with --nms."""
    if "c" in g.files:
        return (np.asarray(g["c"], np.float32), float(g["s"]), [float(v) for v in g["test_scales"]], bool(int(g["nms"])))
    return np.array([256., 256.], np.float32), 512.0, [1.0], True


def oracle_records(heads_b, prm, cam, width, height, c, s, L, scale=1):
    """Full oracle pipeline for one image -> (dets dict, [n,192] records)."""
    from oracle import decode_ref, pnp_ref
    import sys
    sys.path.insert(0, ROOT)
    from oracle.make_golden import result_to_record
    dets = decode_ref.decode(decode_ref.process_heads(heads_b), prm)
    pp = decode_ref.post_process(dets, c, s, heads_b["hm"].shape[1], heads_b["hm"].shape[2], scale=scale)
    for i, d in enumerate(pp):
        d["_k"] = i
    res = decode_ref.merge_outputs(pp, prm)
    recs = []
    for d in res:
        pts = pnp_ref.assemble_points(d, prm.rep_mode)
        st, _ = pnp_ref.pnp_shell(d, pts, cam, width, height, category=prm.category)
        d["_status"] = st
        recs.append(result_to_record(d, d["_k"]))
    return dets, (np.stack(recs) if recs else np.zeros((0, L.CP_POSE_RECORD)))


import contextlib
import os


@contextlib.contextmanager
def golden_threads():
    """The CPU thread count the reference ran with when it wrote the fixtures (oracle/make_golden.py GOLDEN_THREADS), for
    oracle computations that are compared with them."""
    import torch
    from oracle.make_golden import GOLDEN_THREADS
    old = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    try:
        yield
    finally:
        torch.set_num_threads(old)


@contextlib.contextmanager
def no_splitk():
    """The plan picks the split-K factor of the small-map convolutions from the batch size, so a frame's heads move by
    fp32 round-off (~1e-4 of their range) with the batch it sits in -- enough to flip a threshold in the tracker or to
    move a key point of a random-weight network by a pixel.  Tests that assert "batch of B == B single calls" hold the K
    partition fixed (CP_NO_SPLITK is read at every launch); tests/test_gpu_bench_parity.py bounds the effect itself."""
    old = os.environ.get("CP_NO_SPLITK")
    os.environ["CP_NO_SPLITK"] = "1"
    try:
        yield
    finally:
        if old is None:
            del os.environ["CP_NO_SPLITK"]
        else:
            os.environ["CP_NO_SPLITK"] = old
