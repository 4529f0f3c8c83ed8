"""Parity on the configuration bench.py measures (VERDICT r01 item 1): 512 x 512, dla_34, the tensor-core plans
(`tf32x3` = the headline parity mode, `tf32` = the fast mode with its own bound), batch 1 and batch 32, and the
whole image -> pose chain against the CPU oracle chain `net_ref -> decode_ref -> pnp_ref` on the same uint8 frames.

At 512 x 512 the feature maps are 128 / 64 / 32 / 16 wide, i.e. the layers take the code paths the small fixtures
never reach: 32-channel slabs with 256-position tiles crossing image rows and images, `dcn_tma` 8 x 16 patches on
every DLAUp / IDAUp level, the fused heads epilogue, > 148 tiles per launch.
"""
import functools

import numpy as np
import pytest
import torch

import centerpose_b200 as cpb
from centerpose_b200 import _lib as L
from centerpose_b200 import synth
from tests.util import TOL_HEAD_REL_512, golden, net_case_inputs, oracle_records

pytestmark = pytest.mark.gpu

# Single-pass tf32 is a throughput option, not a parity mode: on the seeded random network at 512 x 512 the graph
# amplifies rounding ~2000x (the reference's own fp32 heads are 1e-4 from fp64), so tf32's 2^-11 operand rounding
# arrives at the heads as 0.14 - 0.22 of max|head| (measured, printed below).  The bound only guards against breakage.
TOL_512 = {"fp32": TOL_HEAD_REL_512, "tf32x3": TOL_HEAD_REL_512, "tf32": 0.5}


def _model(wseed, precision, offset_std=0.3, head_gain=1.0):
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    m.precision = precision
    sd = synth.seeded_state_dict(m, seed=wseed, offset_std=offset_std, head_gain=head_gain)
    m.load_state_dict(sd)
    return m.cuda().eval(), opt, sd


@functools.lru_cache(maxsize=None)
def _golden_512():
    g = golden("net_dla34_b1_512")
    x, _ = net_case_inputs(g)
    return g, x


@functools.lru_cache(maxsize=None)
def _truth_512():
    """fp64 CPU evaluation of the oracle graph on the golden's input (once per session, ~1 min)."""
    from oracle import net_ref
    g, x = _golden_512()
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    sd = synth.seeded_state_dict(m, seed=int(g["wseed"]), offset_std=float(g["offset_std"]))
    sd64 = {k: (v.double() if v.dtype.is_floating_point else v) for k, v in sd.items()}
    out = net_ref.forward(torch.from_numpy(x).double(), sd64, opt.heads, "dla_34")
    return {h: v.numpy() for h, v in out.items()}


@pytest.mark.parametrize("prec", ["tf32x3", "tf32", "fp32"])
def test_512_b1_matches_reference_golden(prec, cplib):
    """(i) batch 1, 512 x 512 vs the golden heads of the UNMODIFIED reference (oracle/make_golden.py) and, for the
    parity modes, vs the fp64 truth: the CUDA heads may be no further from fp64 than 4x the reference's own fp32 path."""
    g, x = _golden_512()
    m, opt, _ = _model(int(g["wseed"]), prec, float(g["offset_std"]))
    out = m(torch.from_numpy(x).cuda())[-1]
    truth = _truth_512() if prec != "tf32" else None
    for h in opt.heads:
        want = g["head_" + h]
        got = out[h].cpu().numpy()
        assert np.isfinite(got).all(), h
        mag = np.abs(want).max()
        e = np.abs(got - want).max() / mag
        msg = "512x512 b1 %-7s %-10s gpu-vs-ref %.2e" % (prec, h, e)
        if truth is not None:
            e_ref = np.abs(want.astype(np.float64) - truth[h]).max() / mag
            e_gpu = np.abs(got.astype(np.float64) - truth[h]).max() / mag
            msg += "  gpu-vs-fp64 %.2e  ref-fp32-vs-fp64 %.2e" % (e_gpu, e_ref)
            assert e_gpu <= 4.0 * e_ref + 3e-5, msg
        print(msg)
        assert e <= TOL_512[prec], msg


@pytest.mark.parametrize("prec", ["tf32x3", "tf32"])
def test_512_frame17_of_b32(prec, cplib):
    """(ii) frames are independent (SURVEY.md 8e): inside the benched batch of 32 a frame's heads do not depend on its
    neighbours or its slot (bit-identical when the same frame sits in slot 3 or 17 of two different batches); the same
    frame ALONE agrees to fp32 round-off only, because at batch 1 the plan deals the K loop of the small levels to
    several CTAs (split-K: a different, still fixed, summation order); and frame 17 matches the CPU oracle."""
    from oracle import net_ref
    m, opt, sd = _model(12, prec)
    frames = synth.synthetic_frames(32, 512, 512, seed=4242)
    x = torch.from_numpy(synth.normalize_frames(frames))
    full = m(x.cuda())[-1]
    perm = list(range(32))
    perm[3], perm[17] = perm[17], perm[3]
    other = torch.from_numpy(synth.normalize_frames(synth.synthetic_frames(32, 512, 512, seed=777)))
    other[3] = x[17]
    moved = m(other.cuda())[-1]
    again = m(x.cuda())[-1]
    one = m(x[17:18].contiguous().cuda())[-1]
    for h in opt.heads:
        assert torch.equal(full[h], again[h]), "the plan is not re-entrant: " + h
        assert torch.equal(full[h][17], moved[h][3]), "a frame's heads depend on its batch neighbours / slot: " + h
        d = (full[h][17:18] - one[h]).abs().max().item() / one[h].abs().max().item()
        # single-pass tf32: the truncating accumulator makes the result depend on the K partition at its own error level
        assert d <= (5e-4 if prec == "tf32x3" else 5e-2), "frame 17 of the batch vs the frame alone: %s %.2e" % (h, d)
    want = net_ref.forward(x[17:18], sd, opt.heads, "dla_34")
    for h in opt.heads:
        w = want[h].numpy()
        e = np.abs(full[h][17:18].cpu().numpy() - w).max() / np.abs(w).max()
        print("512x512 b32[17] %-7s %-10s gpu-vs-oracle %.2e" % (prec, h, e))
        assert e <= TOL_512[prec], (h, e)


@pytest.mark.parametrize("hw", [(512, 512), (256, 320)])
def test_split_k_partitions_agree(hw, cplib):
    """The plan picks the split-K factor of every small-map conv from the batch size (tiles vs SMs), so each batch size
    below runs a different K partition of levels 3-5 / the IDA nodes.  The same frame must come out the same to fp32
    round-off (the bound is a few times the reference's own fp32-vs-fp64 distance, see test_512_b1) whatever the
    partition, and bit-identically at every batch size once split-K is switched off (CP_NO_SPLITK=1)."""
    import os
    m, opt, sd = _model(12, "tf32x3")
    H, W = hw
    frames = synth.synthetic_frames(12, H, W, seed=99)
    x = torch.from_numpy(synth.normalize_frames(frames)).cuda()
    base = m(x[:1].contiguous())[-1]
    base = {h: base[h].clone() for h in opt.heads}
    worst = 0.0
    for B in (2, 3, 5, 12):
        got = m(x[:B].contiguous())[-1]
        for h in opt.heads:
            d = (got[h][:1] - base[h]).abs().max().item() / base[h].abs().max().item()
            worst = max(worst, d)
            assert d <= 5e-4, "batch %d vs batch 1, %s: %.2e" % (B, h, d)
    print("split-K partitions %dx%d: worst head difference %.2e" % (H, W, worst))
    os.environ["CP_NO_SPLITK"] = "1"
    try:
        one = m(x[:1].contiguous())[-1]
        one = {h: one[h].clone() for h in opt.heads}
        many = m(x[:5].contiguous())[-1]
        for h in opt.heads:
            assert torch.equal(many[h][:1], one[h]), "without split-K a frame must not depend on the batch size: " + h
            d = (one[h] - base[h]).abs().max().item() / base[h].abs().max().item()
            assert d <= 5e-4, "split-K vs serial K loop, %s: %.2e" % (h, d)
    finally:
        del os.environ["CP_NO_SPLITK"]


# ------------------------------------------------------------------------------------------- image -> pose
def _match(got, want):
    """Pairs (i_got, i_want) of records whose box centres agree to < 1 px (the top-K order may swap on score ties)."""
    pairs, used = [], set()
    for j in range(want.shape[0]):
        d = np.abs(got[:, L.P_CT:L.P_CT + 2] - want[j, L.P_CT:L.P_CT + 2]).max(axis=1) if got.shape[0] else np.zeros(0)
        cand = [i for i in np.argsort(d) if i not in used and d[i] < 1.0]
        if cand:
            used.add(cand[0])
            pairs.append((cand[0], j))
    return pairs


E2E_FRAMES = 6


@functools.lru_cache(maxsize=None)
def _e2e_oracle():
    """Calibrated weights + the oracle chain on E2E_FRAMES uint8 frames (CPU, once per session)."""
    from oracle import decode_ref, net_ref
    m, opt, _ = _model(0, "fp32", offset_std=0.3)
    frames = synth.synthetic_frames(E2E_FRAMES, 512, 512, seed=977)
    x = torch.from_numpy(synth.normalize_frames(frames))
    synth.calibrate_head_bias(m, m(x.cuda())[-1], target=4)       # setup: ~4 centre peaks per frame pass vis_thresh
    sd = {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}
    cam = synth.default_camera(512, 512)
    prm = decode_ref.DecodeParams(rep_mode=opt.rep_mode, vis_thresh=opt.vis_thresh, category=opt.c)
    c = np.array([256., 256.], np.float32)
    recs = []
    for b in range(E2E_FRAMES):
        heads = net_ref.forward(x[b:b + 1], sd, opt.heads, "dla_34")
        _, r = oracle_records({k: v[0].numpy() for k, v in heads.items()}, prm, cam, 512, 512, c, 512.0, L)
        recs.append(r)
    return sd, frames, cam, recs


# stated end-to-end bounds (image pixels / sign-normalised quaternion) for records that keep the same keypoint
# source (regressed vs heat-map peak) in both pipelines.  The network heads carry the fp32 floor of stage B
# (<= 1e-3 * max|head| at 512 x 512, i.e. up to ~0.03 map px = 0.12 image px on `hps`), so the stage-A bar of 1e-3 px
# does not transfer to image -> pose; the measured numbers are printed and recorded in DESIGN.md section 5.
E2E_BOUNDS = {"tf32x3": dict(score=2e-3, px=0.25, quat=5e-2, stable_frac=0.9),
              "tf32": dict(score=1.0, px=1e9, quat=2.0, stable_frac=0.0, match_all=False)}


@pytest.mark.parametrize("prec", ["tf32x3", "tf32"])
def test_image_to_pose_vs_oracle_chain(prec, cplib):
    """Same uint8 frames + calibrated weights: `run_batch()` records vs `net_ref -> decode_ref -> pnp_ref` records."""
    sd, frames, cam, want = _e2e_oracle()
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    m.precision = prec
    m.load_state_dict(sd)
    det = cpb.ObjectPoseDetector(opt, model=m)
    poses, n_valid = det.run_batch(frames, cam)
    bnd = E2E_BOUNDS[prec]
    n_want = n_got = n_pair = n_stable = 0
    worst = dict(score=0.0, px=0.0, quat=0.0, loc_rel=0.0)
    for b in range(E2E_FRAMES):
        got = poses[b, :n_valid[b]].astype(np.float64)
        w = want[b]
        # detections within 2e-3 of vis_thresh may legitimately fall on either side
        margin = np.abs(w[:, L.P_SCORE] - opt.vis_thresh) > 2e-3 if w.shape[0] else np.zeros(0, bool)
        n_want += int(margin.sum())
        n_got += got.shape[0]
        pairs = _match(got, w)
        n_pair += sum(1 for i, j in pairs if margin[j])
        for i, j in pairs:
            worst["score"] = max(worst["score"], abs(got[i, L.P_SCORE] - w[j, L.P_SCORE]))
            dk = np.abs(got[i, L.P_KPS:L.P_KPS + 16] - w[j, L.P_KPS:L.P_KPS + 16]).max()
            dh = np.abs(got[i, L.P_KPS_HM_MEAN:L.P_KPS_HM_MEAN + 16] - w[j, L.P_KPS_HM_MEAN:L.P_KPS_HM_MEAN + 16]).max()
            if max(dk, dh) > 2.0:          # a grouping gate flipped (regressed <-> heat-map peak): not a drift sample
                continue
            n_stable += 1
            dd = np.abs(got[i, L.P_KPS_DISP_MEAN:L.P_KPS_DISP_MEAN + 16] -
                        w[j, L.P_KPS_DISP_MEAN:L.P_KPS_DISP_MEAN + 16]).max()
            worst["px"] = max(worst["px"], dk, dh, dd, np.abs(got[i, L.P_BBOX:L.P_BBOX + 4] - w[j, L.P_BBOX:L.P_BBOX + 4]).max())
            if int(got[i, L.P_STATUS]) in (L.PNP_OK, L.PNP_INVISIBLE) and int(w[j, L.P_STATUS]) in (L.PNP_OK, L.PNP_INVISIBLE):
                q1, q2 = w[j, L.P_QUAT:L.P_QUAT + 4], got[i, L.P_QUAT:L.P_QUAT + 4]
                if np.dot(q1, q2) < 0:
                    q2 = -q2
                worst["quat"] = max(worst["quat"], np.abs(q1 - q2).max())
                t1, t2 = w[j, L.P_LOCATION:L.P_LOCATION + 3], got[i, L.P_LOCATION:L.P_LOCATION + 3]
                worst["loc_rel"] = max(worst["loc_rel"], np.abs(t1 - t2).max() / np.linalg.norm(t1))
    print("image->pose %s: oracle dets %d (away from the threshold), gpu dets %d, matched %d, same keypoint source %d; "
          "max drift: score %.2e, keypoints/boxes %.3e px, quaternion %.2e, location %.2e (relative)"
          % (prec, n_want, n_got, n_pair, n_stable, worst["score"], worst["px"], worst["quat"], worst["loc_rel"]))
    assert n_want > 0
    if bnd.get("match_all", True):
        assert n_pair == n_want, "a detection away from the score threshold is missing on the GPU path"
    assert n_stable >= bnd["stable_frac"] * n_pair
    assert worst["score"] <= bnd["score"]
    assert worst["px"] <= bnd["px"]
    assert worst["quat"] <= bnd["quat"]


def _with_env(name, value, fn):
    import os
    old = os.environ.get(name)
    os.environ[name] = value
    try:
        return fn()
    finally:
        if old is None:
            del os.environ[name]
        else:
            os.environ[name] = old


def test_pdl_and_mma_scheme_switches(cplib):
    """Programmatic dependent launch only reorders WHEN kernels start: heads with CP_PDL=1 and CP_NO_PDL=1 are
    bit-identical (batch 1 and batch 3).  The two-instruction 3-term product of the N <= 64 layers (hi | lo weight tiles as
    one operand) sums the same products in another order: against CP_NO_CAT=1 the heads move by fp32 round-off, which this
    graph amplifies ~2000x at 512 x 512 (measured 1.9e-4 / 6.5e-4 of max|head| on noise frames, the level of the split-K
    reordering; both forms are equally far from the fp64 truth, test_512_b1_matches_reference_golden prints 1.4 - 2.5e-4
    for either)."""
    m, opt, _ = _model(12, "tf32x3")
    for B in (1, 3):
        x = torch.from_numpy(synth.normalize_frames(synth.synthetic_frames(B, 512, 512, seed=77))).cuda()
        on = _with_env("CP_PDL", "1", lambda: {k: v.clone() for k, v in m(x)[-1].items()})
        off = _with_env("CP_NO_PDL", "1", lambda: {k: v.clone() for k, v in m(x)[-1].items()})
        for h in opt.heads:
            assert torch.equal(on[h], off[h]), (B, h)
        three = _with_env("CP_NO_CAT", "1", lambda: {k: v.clone() for k, v in m(x)[-1].items()})
        worst = max(float((on[h] - three[h]).abs().max() / three[h].abs().max()) for h in opt.heads)
        print("batch %d: two- vs three-instruction product, worst head %.2e of max|head|" % (B, worst))
        assert 0.0 < worst <= TOL_HEAD_REL_512, worst
