"""create_model / load_model / save_model contract (models/model.py:26-105) and the drop-in installer."""
import json
import os
import sys

import pytest
import torch

import centerpose_b200 as cpb
from centerpose_b200 import synth
from tests.util import GOLD


@pytest.mark.parametrize("arch,trk,key,n", [("dla_34", False, "dla_34_plain", 416), ("dlav1_34", False, "dlav1_34_plain", 439),
                                           ("dla_34", True, "dla_34_track", 450)])
def test_state_dict_matches_reference(arch, trk, key, n):
    want = json.load(open(os.path.join(GOLD, "state_dict_keys.json")))[key]
    opt = cpb.default_opt(arch, tracking_task=trk)
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    got = [[k, list(v.shape)] for k, v in m.state_dict().items()]
    assert len(got) == n
    assert got == want          # same keys, same shapes, same order


def test_state_dict_matches_live_reference():
    """Same heads (names, channels, order) as the reference's options and the same state dict as its create_model."""
    ref = json.load(open(os.path.join(GOLD, "reference_opts.json")))
    keys = json.load(open(os.path.join(GOLD, "state_dict_keys.json")))
    for arch, trk in (("dla_34", False), ("dlav1_34", False), ("dla_34", True)):
        key = "%s_%s" % (arch, "track" if trk else "plain")
        opt = cpb.default_opt(arch, tracking_task=trk)
        assert [[k, v] for k, v in opt.heads.items()] == ref[key + "_rep1"]["heads"]
        m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
        assert [[k, list(v.shape)] for k, v in m.state_dict().items()] == keys[key]


def test_save_load_roundtrip(tmp_path, capsys):
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    sd = synth.seeded_state_dict(m, seed=9)
    m.load_state_dict(sd)
    path = str(tmp_path / "ckpt.pth")
    cpb.save_model(path, 7, m)
    ck = torch.load(path, weights_only=False)
    assert ck["epoch"] == 7 and set(ck["state_dict"]) == set(sd)
    # DataParallel-style prefix, a dropped key, a wrong-shape key and an unknown key (model.py:43-66)
    sd2 = {"module." + k: v for k, v in ck["state_dict"].items()}
    del sd2["module.hm.2.bias"]
    sd2["module.wh.2.weight"] = torch.zeros(5, 256, 1, 1)
    sd2["module.extra.weight"] = torch.zeros(3)
    torch.save({"epoch": 3, "state_dict": sd2}, path)
    m2 = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    keep_bias = m2.state_dict()["hm.2.bias"].clone()
    m2 = cpb.load_model(m2, path)
    out = capsys.readouterr().out
    assert "Skip loading parameter wh.2.weight" in out and "Drop parameter extra.weight" in out and "No param hm.2.bias" in out
    got = m2.state_dict()
    assert torch.equal(got["base.level2.tree1.conv1.weight"], sd["base.level2.tree1.conv1.weight"])
    assert torch.equal(got["hm.2.bias"], keep_bias)
    opt_ = torch.optim.Adam(m2.parameters(), lr=1e-3)
    cpb.save_model(path, 95, m2, opt_)
    m3, o3, ep = cpb.load_model(cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt), path, opt_, resume=True,
                                lr=1e-3, lr_step=[90, 120])
    assert ep == 95 and abs(o3.param_groups[0]["lr"] - 1e-4) < 1e-12


def test_unknown_arch_raises():
    with pytest.raises(KeyError):
        cpb.create_model("hourglass", {"hm": 1}, 256, None)
    with pytest.raises(ValueError):
        cpb.create_model("dla_60", {"hm": 1}, 256, None)


def test_dropin_registers_reference_module_names():
    from centerpose_b200 import dropin
    saved = {k: sys.modules.get(k) for k in ("lib.models.model", "lib.detectors.detector_factory", "_ext")}
    try:
        dropin.install()
        assert sys.modules["lib.models.model"].create_model is cpb.create_model
        assert sys.modules["lib.detectors.detector_factory"].detector_factory["object_pose"] is cpb.ObjectPoseDetector
        assert sys.modules["_ext"].dcn_v2_forward is cpb.dcn_v2_forward
        assert sys.modules["_ext"].dcn_v2_backward is cpb.dcn_v2_backward
        with pytest.raises(NotImplementedError):
            sys.modules["_ext"].dcn_v2_psroi_pooling_forward()
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_default_opt_matches_reference():
    """default_opt() vs the options the reference derives the way src/demo.py sets them up (oracle/make_golden.py)."""
    ref = json.load(open(os.path.join(GOLD, "reference_opts.json")))
    for arch, trk, rep in (("dla_34", False, 1), ("dla_34", True, 1), ("dlav1_34", False, 0)):
        r = ref["%s_%s_rep%d" % (arch, "track" if trk else "plain", rep)]
        o = cpb.default_opt(arch, tracking_task=trk, rep_mode=rep)
        for f in ("K", "rep_mode", "vis_thresh", "nms", "use_pnp", "head_conv", "down_ratio", "mean", "std", "c",
                  "input_h", "input_w", "num_classes", "test_scales", "fix_res", "hm_hp", "reg_offset",
                  "reg_hp_offset", "tracking_task", "hps_uncertainty", "obj_scale_uncertainty"):
            assert getattr(o, f) == r[f], f
        assert o.balance_coefficient == r["balance_coefficient"]


def test_seeded_weights_are_deterministic():
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    a = synth.seeded_state_dict(m, seed=3)
    b = synth.seeded_state_dict(cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt), seed=3)
    assert all(torch.equal(a[k], b[k]) for k in a)
    # pinned values: the fixtures in tests/golden were generated from exactly these weights
    assert abs(float(a["base.level0.0.weight"].flatten()[0]) - float(b["base.level0.0.weight"].flatten()[0])) == 0
    h1, _ = synth.planted_heads(3, seed=11)
    h2, _ = synth.planted_heads(3, seed=11)
    assert all((h1[k] == h2[k]).all() for k in h1)
