"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.npz by running the
UNMODIFIED reference (through oracle/ref_shims.py) in the build container.

    python -m oracle.make_golden

The GPU box has no /root/reference, so the vectors are committed.  Inputs are
NOT stored: every input is regenerated bit-identically from the seed in the
fixture by `centerpose_b200.synth` (weights, planted heads) or
`numpy.random.default_rng` (images), which keeps the fixtures small.

Fixtures
  net_*.npz     head logits of the reference `DLASeg.forward` on seeded weights
  decode_*.npz  `object_pose_decode` (13 arrays) + post_process + merge_outputs +
                pnp_shell results of the reference on planted head tensors
                (torch==1.1.0 comparison semantics, see ref_shims.legacy_bool_arith)
  dcn_*.npz     the reference's own C++ CPU deformable-conv (oracle/_ref) outputs
  reference_opts.json, state_dict_keys.json
                the options `opts().parse / init` derives the way src/demo.py sets them up, and the
                state-dict keys / shapes of `create_model`, per model configuration
  gpfit_moments.npz
                `utils/gpfit.py` moments() and fitgaussian() on seeded 11 x 11 windows
  demo_frame_0.json
                the --debug 4 JSON the unmodified src/demo.py writes for tests/data/frame_0.png
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_shims          # noqa: E402
from centerpose_b200 import synth     # noqa: E402
from centerpose_b200 import _lib as L  # noqa: E402  (record layout constants only)

GOLD = os.path.join(ROOT, "tests", "golden")
# CPU threads of every reference run here.  oneDNN's fp32 convolutions sum in an order that depends on the thread count,
# and the random-weight graphs amplify that to ~1e-4 of max|head|, so the tests run the oracle with the same count
# (tests/util.py golden_threads) and hold it to the fixtures at the level of fp32 round-off.
GOLDEN_THREADS = 8

NET_CASES = [
    # name, arch, tracking, batch, H, W, weight seed, input seed
    ("net_dla34_b2_96x128", "dla_34", False, 2, 96, 128, 3, 101),
    ("net_dlav1_b1_64x64", "dlav1_34", False, 1, 64, 64, 4, 102),
    ("net_dla34track_b1_64x96", "dla_34", True, 1, 64, 96, 5, 103),
    # the benched shape (BASELINE.json configs[1]/[2]: 512 x 512, dla_34): feature maps 128 / 64 / 32 / 16 wide
    ("net_dla34_b1_512", "dla_34", False, 1, 512, 512, 12, 104),
]

DECODE_CASES = [
    # name, tracking heads, rep_mode, n_obj, disagree_px, batch, seed, category
    ("decode_rep1_3obj", False, 1, 3, 0.0, 2, 11, "chair"),
    ("decode_rep1_10obj_noisy", False, 1, 10, 1.5, 2, 21, "chair"),
    ("decode_rep0_3obj", False, 0, 3, 1.0, 1, 31, "cup"),
    ("decode_rep4_2obj", False, 4, 2, 0.5, 1, 41, "shoe"),
    ("decode_track_rep1_3obj", True, 1, 3, 1.0, 2, 51, "chair"),
    # rep_mode 4 with three keypoint peaks missing: kps carries the -10000 sentinel, 5 valid points -> cv2 SOLVEPNP_EPNP
    ("decode_rep4_5pts_epnp", False, 4, 2, 0.0, 1, 61, "shoe", (1, 4, 6)),
    # the same scene as decode_rep1_3obj evaluated by the UNMODIFIED reference on the torch of this image (>= 1.2), i.e.
    # WITHOUT ref_shims.legacy_bool_arith: `mask_2 == 7` is all-False there (cp_decode_params.modern_bool_semantics = 1)
    ("decode_rep1_3obj_modern_torch", False, 1, 3, 0.0, 2, 11, "chair", (), True),
    # opt.num_classes = 3: per-class top-K, then the K best of the 3 x K candidates (decode.py:52-68), `cls` in the results
    ("decode_cls3_rep1_6obj", False, 1, 6, 1.0, 2, 71, "chair", (), False, {"num_classes": 3}),
    # multi-scale testing, opt.test_scales = [0.75, 1]: merge_outputs keeps detections[0] (the 0.75 pass, coordinates divided
    # by 0.75 as float32) and forces the soft-NMS (object_pose.py:171-197); frame 512 x 512 resized to 384 x 384
    ("decode_scale075_rep1_3obj", False, 1, 3, 0.5, 2, 81, "chair", (), False, {"test_scales": [0.75, 1.0]}),
    # a single scale != 1 with --nms off: division only; rep_mode 0 feeds the divided `kps` to the PnP
    ("decode_scale125_rep0_nonms", False, 0, 4, 1.0, 1, 91, "cup", (), False, {"test_scales": [1.25], "nms": False}),
    # one frame each: five objects 2 px apart in their two keypoint estimates, the tracking heads, rep_mode 3
    ("decode_rep1_5obj", False, 1, 5, 2.0, 1, 77, "chair"),
    ("decode_track_rep1_2obj", True, 1, 2, 0.5, 1, 78, "chair"),
    ("decode_rep3_3obj", False, 3, 3, 1.0, 1, 79, "chair"),
]


def net_inputs(batch, H, W, seed, tracking):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((batch, 3, H, W)).astype(np.float32)
    extra = {}
    if tracking:
        extra["pre_img"] = rng.standard_normal((batch, 3, H, W)).astype(np.float32)
        extra["pre_hm"] = rng.random((batch, 1, H, W)).astype(np.float32)
        extra["pre_hm_hp"] = rng.random((batch, 8, H, W)).astype(np.float32)
    return x, extra


def make_net(only=None):
    import centerpose_b200 as cpb
    from lib.models.model import create_model as ref_create
    for name, arch, trk, B, H, W, wseed, iseed in NET_CASES:
        if only and name not in only:
            continue
        opt = ref_shims.make_opt(arch, tracking_task=trk)
        ours = cpb.create_model(opt.arch, opt.heads, opt.head_conv, cpb.default_opt(arch, tracking_task=trk))
        sd = synth.seeded_state_dict(ours, seed=wseed, offset_std=0.3)
        ref = ref_create(opt.arch, opt.heads, opt.head_conv, opt).eval()
        missing = ref.load_state_dict(sd, strict=True)
        x, extra = net_inputs(B, H, W, iseed, trk)
        with torch.no_grad():
            out = ref(torch.from_numpy(x), *[torch.from_numpy(extra[k]) if k in extra else None
                                             for k in ("pre_img", "pre_hm", "pre_hm_hp")])[-1]
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), arch=arch, tracking=int(trk), batch=B, H=H, W=W,
                            wseed=wseed, iseed=iseed, offset_std=0.3,
                            **{"head_" + k: v.numpy() for k, v in out.items()})
        print(name, {k: float(v.abs().max()) for k, v in out.items()}, missing)


def result_to_record(d, k_src=-1):
    r = np.zeros(L.CP_POSE_RECORD, np.float64)
    r[L.P_SCORE] = d["score"]
    r[L.P_CLS] = d["cls"]
    r[L.P_BBOX:L.P_BBOX + 4] = d["bbox"]
    r[L.P_CT:L.P_CT + 2] = d["ct"]
    r[L.P_KPS:L.P_KPS + 16] = d["kps"]
    r[L.P_KPS_DISP_MEAN:L.P_KPS_DISP_MEAN + 16] = d["kps_displacement_mean"]
    r[L.P_KPS_HM_MEAN:L.P_KPS_HM_MEAN + 16] = d["kps_heatmap_mean"]
    r[L.P_KPS_HM_STD:L.P_KPS_HM_STD + 16] = d["kps_heatmap_std"]
    r[L.P_KPS_HM_HEIGHT:L.P_KPS_HM_HEIGHT + 8] = d["kps_heatmap_height"]
    r[L.P_KPS_DISP_STD:L.P_KPS_DISP_STD + 16] = d["kps_displacement_std"]
    r[L.P_OBJ_SCALE:L.P_OBJ_SCALE + 3] = d["obj_scale"]
    r[L.P_OBJ_SCALE_UNC:L.P_OBJ_SCALE_UNC + 3] = d["obj_scale_uncertainty"]
    r[L.P_TRACKING:L.P_TRACKING + 2] = d["tracking"]
    r[L.P_TRACKING_HP:L.P_TRACKING_HP + 16] = d["tracking_hp"]
    st = d.get("_status", 0)
    r[L.P_STATUS] = st
    if "location" in d:
        r[L.P_LOCATION:L.P_LOCATION + 3] = d["location"]
        r[L.P_QUAT:L.P_QUAT + 4] = d["quaternion_xyzw"]
        r[L.P_PROJ_CUBOID:L.P_PROJ_CUBOID + 16] = np.asarray(d["projected_cuboid"]).reshape(-1)
        r[L.P_KPS_3D_CAM:L.P_KPS_3D_CAM + 27] = np.asarray(d["kps_3d_cam"]).reshape(-1)
        r[L.P_KPS_PNP:L.P_KPS_PNP + 18] = np.asarray(d["kps_pnp"]).reshape(-1)
    r[L.P_SRC_INDEX] = k_src
    return r


def reference_pipeline(heads_b, opt, cam, width, height, c, s, legacy=True, scale=1):
    """Runs the reference's process()-after-network, post_process, merge_outputs and the
    PnP loop of run() on one image's head tensors."""
    from lib.models.decode import object_pose_decode
    from lib.utils.post_process import object_pose_post_process
    from lib.detectors.object_pose import soft_nms_nvidia
    from lib.utils.pnp.cuboid_pnp_shell import pnp_shell
    T = {k: torch.from_numpy(v[None].copy()) for k, v in heads_b.items()}
    T["hm"] = T["hm"].sigmoid_()
    T["hm_hp"] = T["hm_hp"].sigmoid_()
    import contextlib
    with (ref_shims.legacy_bool_arith() if legacy else contextlib.nullcontext()):
        dets = object_pose_decode(
            T["hm"], T["hps"], wh=T["wh"], kps_displacement_std=T.get("hps_uncertainty"), obj_scale=T["scale"],
            obj_scale_uncertainty=T.get("scale_uncertainty"), reg=T["reg"], hm_hp=T["hm_hp"],
            hp_offset=T["hp_offset"], tracking=T.get("tracking"), tracking_hp=T.get("tracking_hp"), opt=opt,
            Inference=True)
    dets = {k: v.detach().cpu().numpy() for k, v in dets.items()}
    if scale != 1 or len(opt.test_scales) > 1:
        # the reference's own detector methods, unbound (they only read self.opt): post_process incl. the division by the
        # test scale (object_pose.py:167-182) and merge_outputs on [detections of scale 0] (:184-197)
        from lib.detectors.object_pose import ObjectPoseDetector as RefDet
        import types
        fake = types.SimpleNamespace(opt=opt)
        m = {"c": c, "s": s, "out_height": 128, "out_width": 128}
        pp = RefDet.post_process(fake, copy.deepcopy(dets), m, scale)
        for i, d in enumerate(pp):
            d["_k"] = i
        results = RefDet.merge_outputs(fake, [pp]) if any(d["score"] > opt.vis_thresh for d in pp) else np.array([])
    else:
        pp = object_pose_post_process(copy.deepcopy(dets), [c], [s], 128, 128, opt, Inference=True)[0]
        for i, d in enumerate(pp):
            d["_k"] = i
        results = np.array([d for d in pp if d["score"] > opt.vis_thresh])
        if opt.nms and len(results):
            keep = soft_nms_nvidia(results, Nt=0.5, method=2, threshold=opt.vis_thresh)
            results = results[keep]
    meta = {"camera_matrix": cam, "width": width, "height": height}
    recs = []
    for d in results:
        if opt.rep_mode in (0, 3, 4):
            pts = [(x[0], x[1]) for x in np.array(d["kps"]).reshape(-1, 2)]
        else:
            p1 = [(x[0], x[1]) for x in np.array(d["kps_displacement_mean"]).reshape(-1, 2)]
            p2 = [(x[0], x[1]) for x in np.array(d["kps_heatmap_mean"]).reshape(-1, 2)]
            pts = np.hstack((p1, p2)).reshape(-1, 2)
        ret = pnp_shell(opt, meta, d, pts, d["obj_scale"], OPENCV_RETURN=opt.show_axes)
        if ret is not None:
            d["_status"] = L.PNP_OK
        elif "location" in d:
            d["_status"] = L.PNP_INVISIBLE
        else:
            d["_status"] = -1       # reference: z<0 / too few points / solver failure (not distinguished)
        recs.append(result_to_record(d, d["_k"]))
    return dets, (np.stack(recs) if recs else np.zeros((0, L.CP_POSE_RECORD)))


def make_decode(only=None):
    for case in DECODE_CASES:
        name, trk, rep, nobj, dis, B, seed, cat = case[:8]
        drop = tuple(case[8]) if len(case) > 8 else ()
        modern = bool(case[9]) if len(case) > 9 else False
        extra = dict(case[10]) if len(case) > 10 else {}
        if only and name not in only:
            continue
        opt = ref_shims.make_opt("dla_34", tracking_task=trk, rep_mode=rep, c=cat)
        ncls = int(extra.get("num_classes", 1))
        scales = [float(v) for v in extra.get("test_scales", [1.0])]
        opt.num_classes = ncls
        opt.test_scales = scales
        opt.nms = bool(extra.get("nms", opt.nms))
        heads = dict(synth.TRACKING_HEADS if trk else synth.DEFAULT_HEADS)
        heads["hm"] = ncls
        hb, truths = synth.planted_batch(B, n_obj=nobj, seed=seed, heads=heads, disagree_px=dis, drop_joints=drop)
        cam = truths[0]["cam"]
        # base_detector.py:110-114 (fix_res): c = the centre of the RESIZED frame, s = max(height, width) of the original
        new = int(512 * scales[0])
        c = np.array([new / 2., new / 2.], np.float32)
        s = 512.0
        out = {"tracking": int(trk), "rep_mode": rep, "n_obj": nobj, "disagree_px": dis, "batch": B, "seed": seed,
               "category": cat, "vis_thresh": float(opt.vis_thresh), "cam": cam,
               "drop_joints": np.array(drop, np.int64), "modern_bool": int(modern), "num_classes": ncls,
               "test_scales": np.array(scales, np.float64), "nms": int(opt.nms), "c": c, "s": s}
        for b in range(B):
            dets, recs = reference_pipeline({k: v[b] for k, v in hb.items()}, opt, cam, 512, 512, c, s, legacy=not modern,
                                            scale=scales[0])
            for k, v in dets.items():
                out["dets%d_%s" % (b, k)] = v[0]
            out["records%d" % b] = recs
            print(name, b, "results", recs.shape[0], "status", recs[:, L.P_STATUS].tolist())
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)


def make_dcn():
    import ctypes
    so = os.path.join(HERE, "_ref", "libdcn_ref.so")
    if not os.path.exists(so):
        print("oracle/_ref/libdcn_ref.so missing (run `make -C oracle`); skipping dcn goldens")
        return
    lib = ctypes.CDLL(so)
    fp = ctypes.POINTER(ctypes.c_float)
    for name, B, C, H, W, Co, seed, off_std in [("dcn_small", 2, 16, 9, 11, 8, 7, 2.0),
                                               ("dcn_edge_big_offsets", 1, 32, 6, 5, 24, 8, 6.0)]:
        rng = np.random.default_rng(seed)
        x = rng.standard_normal((B, C, H, W)).astype(np.float32)
        off = (rng.standard_normal((B, 18, H, W)) * off_std).astype(np.float32)
        mask = rng.random((B, 9, H, W)).astype(np.float32)
        w = (rng.standard_normal((Co, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
        bias = rng.standard_normal(Co).astype(np.float32)
        out = np.zeros((B, Co, H, W), np.float32)
        lib.dcn_ref_forward(x.ctypes.data_as(fp), w.ctypes.data_as(fp), bias.ctypes.data_as(fp),
                            off.ctypes.data_as(fp), mask.ctypes.data_as(fp), out.ctypes.data_as(fp), B, C, H, W, Co)
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), B=B, C=C, H=H, W=W, Co=Co, seed=seed,
                            off_std=off_std, out=out)
        print(name, float(np.abs(out).max()))


DCN_BWD_CASES = [
    # name, B, C, H, W, Co, seed, offset std
    ("dcn_bwd_small", 2, 16, 9, 11, 8, 17, 2.0),
    ("dcn_bwd_edge_big_offsets", 1, 32, 6, 5, 24, 18, 6.0),
    ("dcn_bwd_64ch", 2, 64, 16, 16, 64, 19, 1.0),
]


def dcn_bwd_inputs(B, C, H, W, Co, seed, off_std):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((B, C, H, W)).astype(np.float32)
    off = (rng.standard_normal((B, 18, H, W)) * off_std).astype(np.float32)
    mask = rng.random((B, 9, H, W)).astype(np.float32)
    w = (rng.standard_normal((Co, C, 3, 3)) / np.sqrt(C * 9)).astype(np.float32)
    go = rng.standard_normal((B, Co, H, W)).astype(np.float32)
    return x, off, mask, w, go


def ref_dcn_backward(x, off, mask, w, go):
    """The reference's own C++ CPU backward (oracle/_ref, see oracle/dcn_ref_wrap.cpp)."""
    import ctypes
    lib = ctypes.CDLL(os.path.join(HERE, "_ref", "libdcn_ref.so"))
    fp = ctypes.POINTER(ctypes.c_float)
    B, C, H, W = x.shape
    Co = w.shape[0]
    out = {"grad_input": np.zeros_like(x), "grad_offset": np.zeros_like(off), "grad_mask": np.zeros_like(mask),
           "grad_weight": np.zeros_like(w), "grad_bias": np.zeros(Co, np.float32)}
    a = [np.ascontiguousarray(v) for v in (x, w, off, mask, go)]
    lib.dcn_ref_backward(*[v.ctypes.data_as(fp) for v in a], *[out[k].ctypes.data_as(fp) for k in
                         ("grad_input", "grad_offset", "grad_mask", "grad_weight", "grad_bias")], B, C, H, W, Co)
    return out


def make_dcn_bwd():
    so = os.path.join(HERE, "_ref", "libdcn_ref.so")
    if not os.path.exists(so):
        print("oracle/_ref/libdcn_ref.so missing (run `make -C oracle`); skipping dcn backward goldens")
        return
    for name, B, C, H, W, Co, seed, off_std in DCN_BWD_CASES:
        out = ref_dcn_backward(*dcn_bwd_inputs(B, C, H, W, Co, seed, off_std))
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), B=B, C=C, H=H, W=W, Co=Co, seed=seed, off_std=off_std, **out)
        print(name, {k: float(np.abs(v).max()) for k, v in out.items()})


# (arch, tracking task, rep_mode); state-dict keys are recorded for rep_mode 1
MODEL_CASES = [("dla_34", False, 1), ("dlav1_34", False, 1), ("dla_34", True, 1), ("dlav1_34", False, 0)]
OPT_FIELDS = ("K", "rep_mode", "vis_thresh", "nms", "use_pnp", "head_conv", "down_ratio", "mean", "std", "c", "input_h",
              "input_w", "num_classes", "test_scales", "fix_res", "hm_hp", "reg_offset", "reg_hp_offset", "tracking_task",
              "hps_uncertainty", "obj_scale_uncertainty", "balance_coefficient")


def model_key(arch, tracking):
    return "%s_%s" % (arch, "track" if tracking else "plain")


def make_reference_models():
    import json
    from lib.models.model import create_model as ref_create
    opts, keys = {}, {}
    for arch, trk, rep in MODEL_CASES:
        r = ref_shims.make_opt(arch, tracking_task=trk, rep_mode=rep)
        opts["%s_rep%d" % (model_key(arch, trk), rep)] = dict(heads=[[k, v] for k, v in r.heads.items()],
                                                              **{f: getattr(r, f) for f in OPT_FIELDS})
        if rep == 1:
            m = ref_create(r.arch, r.heads, r.head_conv, r)
            keys[model_key(arch, trk)] = [[k, list(v.shape)] for k, v in m.state_dict().items()]
    for name, d in (("reference_opts.json", opts), ("state_dict_keys.json", keys)):
        with open(os.path.join(GOLD, name), "w") as f:
            json.dump(d, f)
        print(name, list(d))


def gpfit_windows():
    """30 seeded 11 x 11 heat-map windows: a Gaussian bump off the pixel grid times uniform noise."""
    rng = np.random.default_rng(3)
    g = np.exp(-((np.arange(11)[:, None] - 5.3) ** 2 + (np.arange(11)[None] - 4.6) ** 2) / 6)
    return [rng.random((11, 11)) * g for _ in range(30)]


def make_gpfit():
    from lib.utils.gpfit import moments, fitgaussian
    ws = gpfit_windows()
    np.savez_compressed(os.path.join(GOLD, "gpfit_moments.npz"), moments=np.array([moments(w) for w in ws]),
                        fitgaussian=np.array([fitgaussian(w) for w in ws]))
    print("gpfit_moments", len(ws))


DEMO_FRAME = os.path.join(ROOT, "tests", "data", "frame_0.png")
# src/demo.py's camera matrix when --cam_intrinsic is not given
DEMO_CAMERA = np.array([[663.0287679036459, 0, 300.2775065104167], [0, 663.0287679036459, 395.00066121419275], [0, 0, 1]])


def demo_checkpoint(path):
    """Seeded dla_34 weights whose heat-map biases let a few centres pass vis_thresh on DEMO_FRAME, saved the way the
    reference saves checkpoints."""
    import cv2
    import centerpose_b200 as cpb
    from oracle import net_ref
    from oracle import preprocess_ref as pr
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    m.load_state_dict(synth.seeded_state_dict(m, seed=9, offset_std=0.3, head_gain=6.0))
    # the reference pre-process at 512 x 512 (cv2), then calibrate the two heat-map biases on the oracle heads
    x = torch.from_numpy(pr.pre_process(cv2.imread(DEMO_FRAME), 512, 512, opt.mean, opt.std))
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    synth.calibrate_head_bias(m, net_ref.forward(x, sd, opt.heads, "dla_34"), target=10)
    cpb.save_model(path, 1, m)
    return path


def make_demo():
    """The unmodified src/demo.py on the CPU (torch-1.1 comparison semantics, see DESIGN.md section 5)."""
    import json
    import runpy
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "ref") + "/"
        argv = ["--demo", DEMO_FRAME, "--arch", "dla_34", "--load_model", demo_checkpoint(os.path.join(tmp, "ck.pth")),
                "--debug", "4", "--c", "shoe", "--gpus", "-1", "--demo_save", out]
        saved_argv, saved_cwd = sys.argv, os.getcwd()
        sys.argv = ["demo.py"] + argv
        os.chdir(ref_shims.REF_SRC)
        try:
            with ref_shims.legacy_bool_arith():
                runpy.run_path(os.path.join(ref_shims.REF_SRC, "demo.py"), run_name="__main__")
        finally:
            sys.argv = saved_argv
            os.chdir(saved_cwd)
        j = json.load(open(os.path.join(out, "frame_0", "frame_0.json")))
    with open(os.path.join(GOLD, "demo_frame_0.json"), "w") as f:
        json.dump(j, f)
    print("demo_frame_0", len(j["objects"]), "objects")


if __name__ == "__main__":
    if not ref_shims.reference_available():
        raise SystemExit("reference tree not present: goldens can only be generated in the build container")
    ref_shims.install()
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(GOLDEN_THREADS)
    only = set(sys.argv[1:])
    if not only:
        make_dcn()
    if not only or "dcn_bwd" in only:
        make_dcn_bwd()
    make_net(only)
    if not only or any(n.startswith("decode_") for n in only):
        make_decode(only)
    if not only or "models" in only:
        make_reference_models()
    if not only or "gpfit" in only:
        make_gpfit()
    if not only or "demo" in only:
        make_demo()
