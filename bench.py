#!/usr/bin/env python
"""Benchmark of the CenterPose inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W            # this repo (CUDA path)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host CPU cores

One "step" = one pass of the hot path over one batch of synthetic 512x512
Objectron-shaped frames (BASELINE.json configs[2]: batch 32 per GPU, dla_34,
7 heads): pre-process -> DLA-34 + DCNv2 network -> heads -> decode ->
keypoint grouping -> soft-NMS -> PnP -> pose records (+ one all-gather of the
pose tensor when N > 1; frames shard over ranks, weak scaling).

Prints ONE JSON line (rank 0).  `value` is measured with the uint8 frames
already resident in HBM; `e2e` goes through the public serving API
(`centerpose_b200.BatchPipeline` over `ObjectPoseDetector.run_batch()`) with
pinned HOST frames: every step's H2D + D2H are inside the timed region, double
buffered against the compute of the neighbouring steps.  `roofline` is for the
dominant kernel (the heads' 3x3 implicit-GEMM launch), timed live with CUDA
events on the launching stream (cp_plan_profile); `cpu_baseline` is the CPU
oracle (a port of the reference algorithm, see oracle/) on a bounded sample.

The heat-map biases of the seeded weights are calibrated, before anything is
timed, on the reference graph in PyTorch (deterministic fp32, torchvision's
deform_conv2d for the DCNv2 layers), so every build sees the same weights and
inputs; bench.py therefore needs torchvision.  `--dump-outputs DIR` writes what
the last timed step returned, so two builds can be compared output for output.
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

# stdout carries exactly ONE JSON line: anything the host code prints while it sets up (the detector mirrors the
# reference's "Creating model..." message) goes to stderr
# (at the file-descriptor level: NCCL writes its version banner to fd 1 from C)
sys.stdout.flush()
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)
sys.stdout = sys.stderr

METRIC = "images/sec at 512x512 DLA-34 (dla_34 + DCNv2, 7 heads, decode + PnP)"
UNIT = "images/s"
GFLOP_PER_IMAGE = 85.11          # BASELINE.md section 2 (reference graph, 2*MAC)
HEAD_GAIN = 1.0
TARGET_OBJECTS = 4               # centre peaks per frame that pass vis_thresh after bias calibration (Objectron-like density)
N_ROTATE = 6                     # distinct input batches rotated through (6 x 25 MB uint8 + activations >> 126 MB L2)
DUMP_LIMIT = 64 << 20            # bytes written by --dump-outputs


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


def usable_cores():
    """Host threads this process may actually use: affinity mask and cgroup CPU quota, not just nproc."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(float(txt[0]) / float(txt[1]))))
            else:
                q = int(txt[0])
                if q > 0:
                    per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [s.strip() for s in out.strip().split(",")]
                if len(f) >= 7:
                    self.samples.append(f)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit())
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[3 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


@contextlib.contextmanager
def torch_graph_on_gpu(allow_tf32, deterministic=False):
    """The reference graph (oracle/net_ref.py: torch / cuDNN convolutions, BatchNorm, torchvision.ops.deform_conv2d for
    the DCNv2 layers -- the `_ext` stand-in of SURVEY.md Appendix E) on the GPU.  Yields the net_ref module."""
    from oracle import net_ref
    try:
        import torchvision
    except ImportError as e:
        raise RuntimeError("bench.py needs torchvision: its deform_conv2d runs the DCNv2 layers of the PyTorch reference "
                           "graph, which calibrates the benchmark's heat-map biases") from e
    cudnn = torch.backends.cudnn
    orig = net_ref.dcn_v2_forward_ref
    net_ref.dcn_v2_forward_ref = lambda a, off, mask, w, b: torchvision.ops.deform_conv2d(a, off, w, b, padding=1, mask=mask)
    old = (cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, cudnn.benchmark, cudnn.deterministic)
    cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = bool(allow_tf32)
    cudnn.benchmark, cudnn.deterministic = not deterministic, deterministic
    try:
        yield net_ref
    finally:
        net_ref.dcn_v2_forward_ref = orig
        cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, cudnn.benchmark, cudnn.deterministic = old


def calibrate_head_bias(model, sd, opt, x, target=TARGET_OBJECTS):
    """Setup only, outside any timed region: see centerpose_b200.synth.calibrate_head_bias.  The heads it reads come
    from the reference graph in PyTorch (fp32, deterministic cuDNN algorithms), not from this project's kernels, so the
    calibrated weights -- and with them every input of the timed steps -- are the same whichever build runs."""
    from centerpose_b200 import synth
    sdg = {k: v.to(x.device) for k, v in sd.items()}
    with torch_graph_on_gpu(allow_tf32=False, deterministic=True) as net_ref:
        heads = net_ref.forward(x, sdg, opt.heads, "dla_34")
    synth.calibrate_head_bias(model, heads, target)
    return model


def dump_outputs(out_dir, poses, n_valid):
    """Writes the pose records [frames, K, 192] and detection counts [frames] of one step as float32 .npy files.  The
    kernels leave the records past a frame's n_valid unwritten (they hold an earlier step's values), so those are
    zeroed: two builds compare on defined values only.  Above DUMP_LIMIT a fixed, seeded sample of frames is written;
    frame_index.npy names the frames kept."""
    poses = poses.cpu().numpy().copy()
    n_valid = n_valid.cpu().numpy()
    poses[np.arange(poses.shape[1])[None, :] >= n_valid[:, None]] = 0.0
    n = poses.shape[0]
    keep = min(n, (DUMP_LIMIT - 4096) // (poses[0].nbytes + 4 + 8))
    idx = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "poses.npy"), poses[idx])
    np.save(os.path.join(out_dir, "n_valid.npy"), n_valid[idx].astype(np.float32))
    np.save(os.path.join(out_dir, "frame_index.npy"), idx.astype(np.float64))


def cpu_reference_step(sd, opt, frames_u8, cam, budget_s=None, stages=None):
    """The reference algorithm (oracle port) for a few frames on the host: returns the number of images
    processed (stops early, after at least one frame, once `budget_s` seconds of wall clock are spent).
    `stages` (dict) accumulates the seconds per stage with the keys of the reference's run() stamps
    (base_detector.py:770-772): net, dec, post, merge, pnp."""
    t_begin = time.time()
    import centerpose_b200 as cpb  # noqa: F401
    from centerpose_b200 import synth
    from oracle import decode_ref, net_ref, pnp_ref
    n = frames_u8.shape[0]
    prm = decode_ref.DecodeParams(rep_mode=opt.rep_mode, vis_thresh=opt.vis_thresh, category=opt.c)
    c = np.array([256., 256.], np.float32)
    st = stages if stages is not None else {}
    for k in ("net", "dec", "post", "merge", "pnp"):
        st.setdefault(k, 0.0)
    for i in range(n):                                   # the reference's run() is one image per call
        t0 = time.time()
        x = torch.from_numpy(synth.normalize_frames(frames_u8[i:i + 1]))
        heads = net_ref.forward(x, sd, opt.heads, "dla_34")
        hb = {k: v[0].numpy() for k, v in heads.items()}
        t1 = time.time()
        dets = decode_ref.decode(decode_ref.process_heads(hb), prm)
        t2 = time.time()
        pp = decode_ref.post_process(dets, c, 512.0, hb["hm"].shape[1], hb["hm"].shape[2])
        t3 = time.time()
        res = decode_ref.merge_outputs(pp, prm)
        t4 = time.time()
        for d in res:
            pnp_ref.pnp_shell(d, pnp_ref.assemble_points(d, prm.rep_mode), cam, 512, 512, category=prm.category)
        t5 = time.time()
        for k, dt in (("net", t1 - t0), ("dec", t2 - t1), ("post", t3 - t2), ("merge", t4 - t3), ("pnp", t5 - t4)):
            st[k] += dt
        if budget_s is not None and time.time() - t_begin > budget_s:
            return i + 1
    return n


def gpu_torch_forward_ms(sd, opt, x, allow_tf32, reps=10):
    """BASELINE config 2 baseline leg: the reference graph on the GPU (torch_graph_on_gpu).
    Returns (ms per forward, heads)."""
    sdg = {k: v.to(x.device) for k, v in sd.items()}
    with torch_graph_on_gpu(allow_tf32) as net_ref, torch.no_grad():
        for _ in range(3):
            out = net_ref.forward(x, sdg, opt.heads, "dla_34")
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            out = net_ref.forward(x, sdg, opt.heads, "dla_34")
        e1.record()
        torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps, out


def extra_configs(args, det, eng32, sd, opt, cam, dev, ev_time):
    """BASELINE.json configs[0], [1] and [4] measured in the same run (single GPU, rank 0): extra keys of the JSON line."""
    import centerpose_b200 as cpb
    from centerpose_b200 import synth
    from centerpose_b200.engine import InferGraph, decode_params, make_meta
    out = {}
    prm = decode_params(opt)
    # ---- config 2: batch 1, dla_34, ours vs the reference graph in PyTorch on the same GPU, same input
    try:
        x1 = torch.from_numpy(synth.normalize_frames(synth.synthetic_frames(1, 512, 512, seed=99))).to(dev)
        meta1 = make_meta(1, np.array([256., 256.], np.float32), 512.0, 512, 512, cam).to(dev)
        eng1 = det.model.engine(1, 512, 512, dev)          # a batch-32 plan serves batch 1 too (same kernels)
        eager = ev_time(lambda: eng1.infer(x1, meta1, prm), reps=20)
        graph = InferGraph(eng1, 1, prm)
        graphed = ev_time(lambda: graph(x1, meta1), reps=20)
        fwd_only = ev_time(lambda: eng1.forward(x1), reps=20)
        ours = eng1.forward(x1)
        c2 = {"batch": 1, "ours_ms": eager, "ours_cuda_graph_ms": graphed, "ours_forward_only_ms": fwd_only,
              "what": "network + decode + soft-NMS + PnP for one 512 x 512 frame (CUDA events, mean of 20); the torch legs are the "
                      "NETWORK ONLY (the reference's decode / post-process / PnP run on the host: cpu_baseline)"}
        try:
            ms32, ref32 = gpu_torch_forward_ms(sd, opt, x1, allow_tf32=False)
            mstf, _ = gpu_torch_forward_ms(sd, opt, x1, allow_tf32=True)
            c2["torch_gpu_forward_ms"] = {"fp32": ms32, "tf32_allowed": mstf}
            c2["heads_max_abs_diff_vs_torch_fp32_rel"] = max(
                float((ours[h] - ref32[h]).abs().max() / ref32[h].abs().max()) for h in opt.heads)
            c2["speedup_forward_vs_torch_fp32"] = ms32 / fwd_only
        except Exception as e:                              # torchvision missing on the box, ...
            c2["torch_gpu_forward_ms"] = {"unavailable": repr(e)[:200]}
        out["config2"] = c2
        del graph
    except Exception as e:
        out["config2"] = {"error": repr(e)[:300]}
    # ---- config 5: CenterPoseTrack, batch = 8 video streams, two-frame network + decode + tracker step + heat-map rendering
    try:
        topt = cpb.default_opt("dla_34", tracking_task=True)
        tm = cpb.create_model(topt.arch, topt.heads, topt.head_conv, topt)
        tm.precision = args.precision
        tm.load_state_dict(synth.seeded_state_dict(tm, seed=0, offset_std=0.3, head_gain=HEAD_GAIN))
        tdet = cpb.ObjectPoseDetector(topt, model=tm)
        vids = [torch.from_numpy(synth.synthetic_frames(8, 512, 512, seed=500 + i)).to(dev) for i in range(4)]
        xcal = torch.from_numpy(synth.normalize_frames(synth.synthetic_frames(8, 512, 512, seed=500))).to(dev)
        teng = tdet.model.engine(8, 512, 512, dev)
        z1, z8 = torch.zeros((8, 1, 512, 512), device=dev), torch.zeros((8, 8, 512, 512), device=dev)
        synth.calibrate_head_bias(tdet.model, teng.forward(xcal, xcal, z1, z8), TARGET_OBJECTS)
        state = {"i": 0}

        def track_step():
            tdet.run_batch(vids[state["i"] % 4], cam, track=True, to_host=False)
            state["i"] += 1
        ms = ev_time(track_step, reps=12)
        _, nt = tdet.run_batch(vids[0], cam, track=True)
        out["config5"] = {"batch": 8, "pairs_per_s": 8 / (ms * 1e-3), "ms_per_step": ms, "tracks_per_stream": float(np.mean(nt)),
                          "what": "8 video streams: pre-process, render pre_hm / pre_hm_hp from the tracker state, two-frame "
                                  "dla_34 (3 stems, 11 heads / 71 ch), decode + PnP, tracker step (association, Kalman, scale pool, "
                                  "second PnP) -- all on the device, frames resident", "precision": args.precision}
        del tdet, tm
    except Exception as e:
        out["config5"] = {"error": repr(e)[:300]}
    # ---- config 1: one 512 x 512 image, dlav1_34 (DCN + convGRU + GroupNorm)
    try:
        vopt = cpb.default_opt("dlav1_34")
        vm = cpb.create_model(vopt.arch, vopt.heads, vopt.head_conv, vopt)
        vm.precision = args.precision
        vsd = synth.seeded_state_dict(vm, seed=0, offset_std=0.3, head_gain=HEAD_GAIN)
        vm.load_state_dict(vsd)
        vdet = cpb.ObjectPoseDetector(vopt, model=vm)
        fr = synth.synthetic_frames(1, 512, 512, seed=7)
        x1 = torch.from_numpy(synth.normalize_frames(fr)).to(dev)
        meta1 = make_meta(1, np.array([256., 256.], np.float32), 512.0, 512, 512, cam).to(dev)
        veng = vdet.model.engine(1, 512, 512, dev)
        ms = ev_time(lambda: veng.infer(x1, meta1, decode_params(vopt)), reps=10)
        c1 = {"arch": "dlav1_34", "batch": 1, "ours_ms": ms}
        if not args.no_cpu_baseline:
            from oracle import net_ref
            torch.set_num_threads(usable_cores())
            t0 = time.time()
            net_ref.forward(x1.cpu(), vsd, vopt.heads, "dlav1_34")
            c1["cpu_port_forward_s"] = time.time() - t0
            c1["cpu_cores"] = usable_cores()
        out["config1"] = c1
        del vdet, vm
    except Exception as e:
        out["config1"] = {"error": repr(e)[:300]}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import centerpose_b200 as cpb
    from centerpose_b200 import synth
    cores = usable_cores()
    torch.set_num_threads(cores)
    opt = cpb.default_opt("dla_34")
    m = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    sd = synth.seeded_state_dict(m, seed=0, offset_std=0.3, head_gain=HEAD_GAIN)
    cam = synth.default_camera(512, 512)
    per_step = args.ref_images
    frames = synth.synthetic_frames(per_step, 512, 512, seed=317)
    for _ in range(max(1, min(args.warmup, 1))):
        cpu_reference_step(sd, opt, frames[:1], cam)
    t0 = time.time()
    n = 0
    for _ in range(args.steps):
        n += cpu_reference_step(sd, opt, frames, cam)
    dt = time.time() - t0
    val = n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "batch=%d synthetic 512x512 frames, dla_34, host CPU" % per_step, "sample": per_step},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": "%d steps x %d frames, one frame per call like run()" % (args.steps, per_step)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), file=_REAL_STDOUT)
    _REAL_STDOUT.flush()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="frames per GPU per step")
    ap.add_argument("--ref-images", type=int, default=2, help="frames per step of the CPU reference arm")
    ap.add_argument("--cpu-sample", type=int, default=4, help="frames of the in-run cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--profile-ops", default="", help="write the per-op table (cp_plan_profile) to this path")
    ap.add_argument("--precision", default="tf32x3", choices=["fp32", "tf32x3", "bf16", "tf32"],
                    help="tf32x3 (default): tcgen05 3-term split, fp32-equivalent (meets the fp32 parity bar); fp32: CUDA-core "
                         "parity mode; tf32: tcgen05 single pass (cuDNN-default-like math); bf16: tcgen05 bf16 operands")
    ap.add_argument("--no-fast-mode", action="store_true", help="skip the extra single-pass tf32 measurement")
    ap.add_argument("--no-extra-configs", action="store_true",
                    help="skip the BASELINE.json configs 1 / 2 / 5 legs (batch-1 latency vs PyTorch-GPU, dlav1_34, tracking)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned (pose records, detection counts) to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if args.warmup < 3:
        args.warmup = 3

    import torch.distributed as dist
    import centerpose_b200 as cpb
    from centerpose_b200 import _lib as L
    from centerpose_b200 import synth
    from centerpose_b200.dist import PoseBuffer
    from centerpose_b200.engine import InferGraph, decode_params, make_meta, preprocess

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the hot path has no CPU fallback); "
                         "use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    B = args.batch

    opt = cpb.default_opt("dla_34")
    model = cpb.create_model(opt.arch, opt.heads, opt.head_conv, opt)
    model.precision = args.precision
    sd = synth.seeded_state_dict(model, seed=0, offset_std=0.3, head_gain=HEAD_GAIN)
    model.load_state_dict(sd)
    det = cpb.ObjectPoseDetector(opt, model=model)
    cam = synth.default_camera(512, 512)
    calib = torch.from_numpy(synth.normalize_frames(synth.synthetic_frames(B, 512, 512, seed=317 + 1000 * rank))).to(dev)
    calibrate_head_bias(det.model, sd, opt, calib)
    eng = det.model.engine(B, 512, 512, dev)            # with the calibrated weights
    sd = {k: v.detach().cpu() for k, v in det.model.state_dict().items()}
    del calib
    prm = decode_params(opt)
    meta = make_meta(B, np.array([256., 256.], np.float32), 512.0, 512, 512, cam).to(dev)

    # distinct frames per rank and per rotation slot
    host_frames = [torch.from_numpy(synth.synthetic_frames(B, 512, 512, seed=317 + 1000 * rank + i)).pin_memory()
                   for i in range(N_ROTATE)]
    dev_frames = [f.to(dev) for f in host_frames]
    x_buf = torch.empty((B, 3, 512, 512), dtype=torch.float32, device=dev)
    # ONE persistent buffer per rank: cp_infer writes the pose records + n_valid straight into the layout the all-gather
    # and the pinned device -> host copy use (centerpose_b200/dist.py); no packing kernel on the hot path
    pbuf = PoseBuffer(B, prm.K, dev, world=world)
    poses, n_valid = pbuf.poses, pbuf.n_valid

    def step_resident(i):
        preprocess(dev_frames[i % N_ROTATE], 512, 512, opt.mean, opt.std, out=x_buf)
        eng.infer(x_buf, meta, prm, poses=poses, n_valid=n_valid)
        return pbuf.all_gather()

    # end to end = the public serving API (centerpose_b200.BatchPipeline over ObjectPoseDetector.run_batch): every step
    # uploads ITS frames from pinned host memory, runs pre-process + network + decode + PnP + the all-gather, and reads
    # ITS records back into pinned host memory; double buffering hides the upload of step i+1 / the download of step i-1
    # behind the compute of step i, so a step's result is collected one submit later (the last one by drain()).
    pipe = cpb.BatchPipeline(det, B, 512, 512, cam, world=world, depth=2, to_host=(rank == 0))
    last_host = [None]

    def step_e2e(i):
        if pipe.in_flight == pipe.depth:
            last_host[0] = pipe.collect()
        pipe.submit(host_frames[i % N_ROTATE])
        return last_host[0]

    def drain_e2e():
        while pipe.in_flight:
            last_host[0] = pipe.collect()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, drain=None):
        for i in range(warmup):
            fn(i)
        if drain is not None:
            drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if drain is not None:
            drain()                                       # the last steps' records reach the host inside the timed region
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local)
    sampler.start()
    ms_res = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *pbuf.views(pbuf.gathered))
    clocks = sampler
    ms_e2e = timed(step_e2e, args.steps, args.warmup, drain=drain_e2e)
    sampler.stop_flag = True
    sampler.join(timeout=2)

    total_images = B * world * args.steps
    value = total_images / (ms_res / 1e3)
    e2e_value = total_images / (ms_e2e / 1e3)
    det_per_img = float(n_valid.float().mean().item())

    # ---- roofline of the dominant kernel, timed live (CUDA events between ops on the launching stream)
    peaks = load_peaks()
    ops = None
    for _ in range(3):
        ops = eng.profile(x_buf)
    tot_ms = sum(o["ms"] for o in ops)
    dom = max(ops, key=lambda o: o["ms"])
    reps = [eng.profile(x_buf) for _ in range(5)]
    dom_ms = float(np.mean([[o for o in r if o["name"] == dom["name"]][0]["ms"] for r in reps]))
    achieved = dom["flops"] / (dom_ms * 1e-3) / 1e12
    peak = peaks["bf16_tflops_sustained"]
    kname = {"fp32": "igemm_fp32_kernel<64,NHWC>", "tf32": "conv_tma_kernel<x1>", "tf32x3": "conv_tma_kernel<x3>"}.get(
        args.precision, "igemm_umma_kernel")
    traffic = None
    pipe_pct = None
    tpath = os.path.join(ROOT, "profiles", "r02_dominant_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_dominant_traffic.json")
    if os.path.exists(tpath):          # dram__bytes_read + dram__bytes_write of this launch, from the committed ncu capture
        tj = json.load(open(tpath))
        traffic = tj.get(kname + "@" + dom["name"])
        pipe_pct = tj.get("tensor_pipe_active_pct", {}).get(kname + "@" + dom["name"])
    mma_passes = 3 if args.precision == "tf32x3" else 1
    roofline = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic,
                "kernel": kname + " @ " + dom["name"],
                "tensor_work_tflops": achieved * mma_passes,     # tf32x3 issues 3 MMAs per algorithmic MAC
                "tensor_pipe_active_pct_ncu": pipe_pct,          # sm__pipe_tensor_cycles_active of the committed capture
                "ms_per_launch": dom_ms,
                "share_of_forward": dom_ms / tot_ms, "peak_source": peaks["source"] + " (cuBLAS bf16, sustained)",
                "algorithmic_flops_per_launch": dom["flops"],
                "network_tflops": GFLOP_PER_IMAGE * 1e9 * B / (tot_ms * 1e-3) / 1e12}
    if args.profile_ops and rank == 0:
        with open(args.profile_ops, "w") as f:
            f.write("name,kind,ms,gflop,mbytes,tflops,gbs\n")
            for o in ops:
                f.write("%s,%d,%.4f,%.3f,%.3f,%.2f,%.1f\n" % (o["name"], o["kind"], o["ms"], o["flops"] / 1e9,
                                                            o["bytes"] / 1e6, o["flops"] / max(o["ms"], 1e-6) / 1e9,
                                                            o["bytes"] / max(o["ms"], 1e-6) / 1e6))

    # ---- stage breakdown of one resident step (CUDA events, mean of 5)
    from centerpose_b200.engine import decode_pnp

    def ev_time(fn, reps=5):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    heads_out = eng.forward(x_buf)
    breakdown = {"preprocess": ev_time(lambda: preprocess(dev_frames[0], 512, 512, opt.mean, opt.std, out=x_buf)),
                 "forward": ev_time(lambda: eng.forward(x_buf)),
                 "decode_softnms_pnp": ev_time(lambda: decode_pnp(heads_out, meta, prm, want_dets=False))}

    # ---- HBM roofline of the decode / grouping / soft-NMS / PnP kernels (north_star).  Algorithmic bytes = SURVEY.md 8(d):
    # scan hm + hm_hp once (9 x 128^2 x 4 B), gathers at the K centres, the pose records written = 0.68 MB per image
    dec_bytes_img = (1 + 8) * 128 * 128 * 4 + prm.K * (2 + 16 + 2 + 3) * 4 + 8 * prm.K * 2 * 4 + prm.K * L.CP_POSE_RECORD * 4
    dec_bytes = dec_bytes_img * B
    dec_gbs = dec_bytes / (breakdown["decode_softnms_pnp"] * 1e-3) / 1e9
    heads1 = {k: v[:1].contiguous() for k, v in heads_out.items()}
    meta1 = meta[:1].contiguous()
    dec_b1_ms = ev_time(lambda: decode_pnp(heads1, meta1, prm, want_dets=False), reps=20)
    roofline_decode = {"bound": "hbm", "achieved": dec_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                       "frac": dec_gbs / peaks["hbm_gbs"], "traffic": None,
                       "kernel": "peaks_topk_kernel + group_pose_kernel", "algorithmic_bytes_per_step": dec_bytes,
                       "algorithmic_bytes_per_image": dec_bytes_img, "ms_per_step": breakdown["decode_softnms_pnp"],
                       "note": "SURVEY.md 8(d) bytes (0.68 MB / image); latency-bound: per-channel radix select + one warp "
                               "per object for the double-precision PnP"}
    decode_us_per_frame = {"b32": breakdown["decode_softnms_pnp"] * 1e3 / B, "b1": dec_b1_ms * 1e3,
                           "what": "sigmoid + NMS + top-K + grouping + affine + soft-NMS + PnP, CUDA events"}

    # ---- same step in the single-pass tf32 mode (what cuDNN does by default for fp32 convs on this class of GPU);
    # reported beside the headline, which stays on the fp32-equivalent mode
    fast_mode = None
    if args.precision == "tf32x3" and not args.no_fast_mode:
        model.precision = "tf32"
        eng_fast = det.model.engine(B, 512, 512, dev)
        eng_main = eng

        def step_fast(i):
            preprocess(dev_frames[i % N_ROTATE], 512, 512, opt.mean, opt.std, out=x_buf)
            eng_fast.infer(x_buf, meta, prm, poses=poses, n_valid=n_valid)
            return pbuf.all_gather()

        ms_fast = timed(step_fast, args.steps, args.warmup)
        fast_mode = {"precision": "tf32 (tcgen05 single pass)", "value": total_images / (ms_fast / 1e3), "unit": UNIT,
                     "ms_per_step": ms_fast / args.steps}
        model.precision = args.precision
        eng = eng_main
        del eng_fast

    extra = {}
    if rank == 0 and world == 1 and not args.no_extra_configs:
        extra = extra_configs(args, det, eng, sd, opt, cam, dev, ev_time)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = usable_cores()
        torch.set_num_threads(cores)
        fr = synth.synthetic_frames(args.cpu_sample, 512, 512, seed=317)
        cpu_reference_step(sd, opt, fr[:1], cam)
        t0 = time.time()
        stages = {}
        n = cpu_reference_step(sd, opt, fr, cam, budget_s=30.0, stages=stages)
        dt = time.time() - t0
        cpu_baseline = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": "%d frames of the same workload, one frame per call like run()" % n,
                        "stage_ms_per_image": {k: v / n * 1e3 for k, v in stages.items()}}

    if rank == 0:
        h2d = B * 512 * 512 * 3                          # uint8 frames (the per-frame meta of a fixed camera is uploaded once)
        d2h = pbuf.row * 4 * world                       # rank 0 reads the gathered records once (pinned)
        launches_per_step = eng.forward_launches + 2 + 1
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"fp32": "f32", "tf32x3": "tf32x3", "bf16": "bf16", "tf32": "tf32"}[args.precision], "data": "synthetic",
            "config": {"workload": "batch=%d synthetic 512x512 frames per GPU, dla_34 + DCNv2, 7 heads, K=100, rep_mode 1, "
                                   "decode + soft-NMS + PnP" % B,
                       "global_batch": B * world,
                       "precision": {"fp32": "fp32 CUDA-core implicit GEMM (parity mode)",
                                     "tf32x3": "tcgen05 kind::tf32 3-term split (fp32-equivalent parity mode)",
                                     "bf16": "tcgen05 kind::f16 bf16 operands, fp32 accumulate (fast mode)",
                                     "tf32": "tcgen05 kind::tf32 single pass, TMA-fed shifted-window convs (cuDNN-default-equivalent "
                                             "math); deformable / strided ops on the 3-term split kernel"}[args.precision],
                       "weights": "seeded random init; hm / hm_hp biases calibrated so ~%d peaks per frame pass the "
                                  "thresholds" % TARGET_OBJECTS,
                       "stage_b_bar": "network heads vs the reference: max-abs <= 3e-4 * max|head| on the small fixtures, 1e-3 at "
                                      "512 x 512 (SURVEY.md 8d says 1e-4; the reference's own fp32 heads are 1e-4 from fp64 "
                                      "there), always with gpu-vs-fp64 <= 4 x reference-vs-fp64 + 3e-5 (tests/util.py)",
                       "l2": "inputs rotate over %d distinct batches; per-step activations (~8 GB) exceed the 126 MB L2" % N_ROTATE,
                       "detections_per_image": det_per_img, "parallelism": "dp%d, 1 all-gather of pose records" % world},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": ms_e2e / args.steps},
            "gpu_launches": launches_per_step * args.steps,
            "clocks": clocks.summary(),
            "roofline": roofline,
            "roofline_decode": roofline_decode,
            "decode_us_per_frame": decode_us_per_frame,
            "config1": extra.get("config1"), "config2": extra.get("config2"), "config5": extra.get("config5"),
            "fast_mode": fast_mode,
            "stage_ms": breakdown,
            "cpu_baseline": cpu_baseline,
            "network_gflop_per_image": GFLOP_PER_IMAGE,
        }
        print(json.dumps(line), file=_REAL_STDOUT)
        _REAL_STDOUT.flush()
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
