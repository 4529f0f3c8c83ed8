"""Drop-in proof (SURVEY.md rows a-12 / b / f-3): the flow of the reference's `src/demo.py` (demo.py:22-87:
`detector_factory[opt.task](opt)` from a checkpoint path, then `run(image path, meta_inp)` with `--debug 4`) on this
package's ObjectPoseDetector -- pre_process, result structures, dict_out, save_results -- must write the JSON file the
unmodified reference wrote for the same frame, checkpoint and arguments (tests/golden/demo_frame_0.json, recorded by
oracle/make_golden.py from the reference's own demo.py on the CPU).  The JSON is compared key by key.  Without a GPU the
two device stages (`DLASegB200.forward`, `cp_decode_pnp`) are replaced by the CPU oracle (test infrastructure) --
everything else is the product's host code.  `test_demo_flow_on_gpu` runs the same flow with the real engine on the
committed sample frames.
"""
import copy
import json
import os

import numpy as np
import pytest
import torch

import centerpose_b200 as cpb
from centerpose_b200 import _lib as L
from centerpose_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FRAME = os.path.join(ROOT, "tests", "data", "frame_0.png")
GOLD = os.path.join(ROOT, "tests", "golden")
OBJECT_KEYS = {"class", "ct", "bbox", "confidence", "kps_displacement_mean", "kps_heatmap_mean", "kps_heatmap_std",
               "kps_heatmap_height", "obj_scale", "location", "quaternion_xyzw", "kps_pnp", "kps_3d_cam"}


def _oracle_process(self, images, pre_images=None, pre_hms=None, pre_hm_hp=None, pre_inds=None, return_time=False, meta=None,
                    scale=1.0):
    """CPU stand-in for the two device stages of ObjectPoseDetector.process (network + fused decode / PnP)."""
    import time
    from centerpose_b200.detector import dets_to_dict
    from oracle import decode_ref, net_ref
    from tests.util import oracle_records
    sd = {k: v.detach().cpu() for k, v in self.model.state_dict().items()}
    heads = net_ref.forward(images.cpu(), sd, self.opt.heads, "dla_34")
    forward_time = time.time()
    prm = decode_ref.DecodeParams(rep_mode=self.opt.rep_mode, vis_thresh=self.opt.vis_thresh, category=self.opt.c,
                                  nms=self.opt.nms, num_scales=len(self.opt.test_scales))
    hb = {k: v[0].numpy() for k, v in heads.items()}
    s = meta["s"]
    s = float(s[0]) if isinstance(s, np.ndarray) and s.ndim else float(s)
    dets, recs = oracle_records(hb, prm, np.asarray(meta["camera_matrix"], np.float64), meta["width"], meta["height"],
                                np.asarray(meta["c"], np.float32), s, L, scale=scale)
    poses = np.zeros((1, self.opt.K, L.CP_POSE_RECORD), np.float32)
    poses[0, :recs.shape[0]] = recs
    self._last = (poses, np.array([recs.shape[0]], np.int32))
    self._last_dev = None
    output = {k: v.clone() for k, v in heads.items()}
    output["hm"] = output["hm"].sigmoid_()
    output["hm_hp"] = output["hm_hp"].sigmoid_()
    packed = np.zeros((1, self.opt.K, L.CP_DETS_RECORD), np.float32)
    d = dets_to_dict(packed)
    return (output, d, forward_time) if return_time else (output, d)


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    from oracle.make_golden import demo_checkpoint
    from tests.util import golden_threads
    with golden_threads():
        return demo_checkpoint(str(tmp_path_factory.mktemp("ckpt") / "chair_seeded.pth"))


class _RecordingDebugger(object):
    """Stands in for the reference's Debugger (drawing), which only exists inside the reference tree."""

    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        return lambda *a, **k: self.calls.append(name)


def test_demo_flow_matches_reference_json(checkpoint, tmp_path, monkeypatch):
    from oracle.make_golden import DEMO_CAMERA
    from tests.util import golden_threads
    ja = json.load(open(os.path.join(GOLD, "demo_frame_0.json")))
    opt = cpb.default_opt("dla_34", c="shoe", debug=4, load_model=checkpoint)
    opt.demo = FRAME
    opt.demo_save = str(tmp_path / "ours")
    dbg = _RecordingDebugger()
    monkeypatch.setattr(cpb.ObjectPoseDetector, "process", _oracle_process)
    monkeypatch.setattr(cpb.ObjectPoseDetector, "_to_device", lambda self, t: t)
    monkeypatch.setattr(cpb.ObjectPoseDetector, "_debugger", lambda self, debugger: dbg)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)      # run()'s timing stamps; no device here
    det = cpb.detector_factory[opt.task](opt)
    det.pause = False
    with golden_threads():
        det.run(FRAME, meta_inp={"camera_matrix": DEMO_CAMERA})
    jb = json.load(open(os.path.join(opt.demo_save, "frame_0", "frame_0.json")))
    # ---- same schema, same objects
    assert set(ja) == set(jb) == {"camera_data", "objects"}
    assert np.allclose(ja["camera_data"], jb["camera_data"])
    assert len(ja["objects"]) == len(jb["objects"]) >= 1, (len(ja["objects"]), len(jb["objects"]))
    for oa, ob in zip(ja["objects"], jb["objects"]):
        assert set(oa) == set(ob) == OBJECT_KEYS, (sorted(oa), sorted(ob))
        assert oa["class"] == ob["class"]
        for k in OBJECT_KEYS - {"class"}:
            a, b = np.asarray(oa[k], np.float64), np.asarray(ob[k], np.float64)
            assert a.shape == b.shape, k
            if k == "quaternion_xyzw" and np.dot(a, b) < 0:
                b = -b
            # The keypoints of a random-weight network are not a projected cuboid, so the PnP problem is far from
            # consistent and cv2's LM (the reference) and the restated LM (20-iteration cap, DESIGN.md section 4) stop
            # at slightly different points: the four PnP outputs get a loose bound here; on consistent keypoints the
            # two agree to 1e-6 (tests/test_pose_core_host.py, tests/test_oracle_decode.py).
            tol = {"quaternion_xyzw": 5e-2, "location": 5e-2, "kps_3d_cam": 5e-2, "kps_pnp": 5e-2, "confidence": 1e-5,
                   "kps_heatmap_height": 1e-5, "obj_scale": 1e-5}.get(k, 2e-3)      # pixels: fp32 records
            scale = max(1.0, np.abs(a).max()) if k in ("location", "kps_3d_cam", "kps_pnp") else 1.0
            assert np.abs(a - b).max() <= tol * scale, (k, float(np.abs(a - b).max()))
    # the frame is drawn and saved next to the JSON, as the reference does
    assert "save_all_imgs_demo" in dbg.calls


@pytest.mark.gpu
def test_demo_flow_on_gpu(cplib, tmp_path):
    """The demo flow (demo.py:22-87: Detector(opt) from a checkpoint path -> run(image path, meta_inp) per file ->
    --debug 4 JSON) with the real engine, on the committed sample frames."""
    opt = cpb.default_opt("dla_34", debug=4)
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    m.load_state_dict(synth.seeded_state_dict(m, seed=9, offset_std=0.3, head_gain=6.0))
    ck = str(tmp_path / "chair_seeded.pth")
    cpb.save_model(ck, 1, m)
    opt.load_model = ck
    opt.demo = os.path.join(ROOT, "tests", "data")
    opt.demo_save = str(tmp_path / "save")
    cam = np.array([[663.0287679036459, 0, 300.2775065104167], [0, 663.0287679036459, 395.00066121419275], [0, 0, 1]])
    det = cpb.detector_factory["object_pose"](opt)
    det.pause = False
    names = sorted(f for f in os.listdir(opt.demo) if f.endswith(".png"))
    for f in names:
        ret = det.run(os.path.join(opt.demo, f), meta_inp={"camera_matrix": cam})
        assert set(ret) == {"results", "boxes", "output", "tot", "load", "pre", "net", "dec", "post", "merge", "pnp", "track"}
        j = json.load(open(os.path.join(opt.demo_save, "data", os.path.splitext(f)[0] + ".json")))
        assert set(j) == {"camera_data", "objects"} and len(j["objects"]) == len(ret["boxes"])
        for o in j["objects"]:
            assert set(o) == OBJECT_KEYS
