#!/usr/bin/env python
"""bench.py -- VO frames/s of the DF-VO tracking hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|torch_gpu]
                    [--config vo|corr64|ransac10k|pairs64|parity] [--no-extras] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Default workload (`--config vo`, BASELINE.json configs[1]): KITTI-odometry-shaped stream of 376x1241 RGB frames, full hybrid
tracker per frame: monodepth2 depth + LiteFlowNet forward/backward flow + forward-backward consistency + local best-N
selection + 5x essential-matrix RANSAC with GRIC + pose recovery + scale recovery (PnP fallback when the E-model is
rejected).  One *step* = one VO frame.  With N GPUs every rank tracks its own sequence (weak scaling); weights are generated
on rank 0 and broadcast with NCCL.

There are no trained weights or KITTI frames offline: frames are seeded synthetic textures and both networks run with seeded
random-init weights (their cost is the real cost).  Random-weight flow has no consistent correspondences, so the tracker
stages (selection, RANSAC, scale, PnP) are fed analytic rigid-scene flow / depth of the same shapes, copied over the network
outputs on the device inside the timed region through the pipeline's official `inject=` hook; every kernel of the frame runs
every step.  The 8 distinct frames cycle the SURVEY 8d outlier fractions {0, 0.3, 0.6} (E-RANSAC stops after ~1 / ~28 / ~410
iterations) and contain one zero-translation frame (GRIC prefers the homography -> PnP fallback).

The object timed is `b200.pipeline.FramePipeline` itself (`step(frame) -> pose`): three network engines in flight and the tracker
split into its enqueue / read halves by default (`DFVO_INFLIGHT`, `DFVO_PIPELINED`, `DFVO_TRACKER_THREAD` select the other modes,
all with identical poses); `e2e.latency_ms` is the time from handing a frame to `step` until its pose comes back, and
`e2e.low_latency` / `e2e.in_order` report the two-engine same-step and the single-stream in-order pipelines next to it.

Output: ONE JSON line (rank 0).  `value` = frames/s with frames already in HBM; `e2e` = the same metric through the public API
(pinned host uint8 frames -> pose on the host) with H2D/D2H inside the timed region; `e2e_libs` = through the reference-API
mirror (`libs.deep_models.DeepModel.forward_depth/forward_flow`, `KeypointSampler`, `EssTracker`, `PnpTracker`) the way
libs/dfvo.py calls it; `roofline` = the tcgen05 convolution kernels against the measured bf16 peak (per-launch CUDA events on
an in-order stream); `cpu_baseline` = the CPU oracle port of the same frame timed on this box's cores; `precision_modes` = the
same pipeline in tf32 / fp32 mode; `gpu_library_baseline` = the reference graph through torch/cuDNN on the same GPU;
`extra_configs` = BASELINE configs[2] (correlation + consistency, HBM roofline) and configs[3] (RANSAC scoring, FP64 roofline).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "df-vo_b200"))

import numpy as np

H, W = 376, 1241
FEED_H, FEED_W = 192, 640
METRIC = "VO frames/sec on 376x1241 pairs"
WORKLOAD = "KITTI-odom seq-shape stream (376x1241), full hybrid tracker (depth+flow+E-RANSAC/PnP), 1 frame per step"
N_DISTINCT = 8                     # distinct synthetic frames cycled through the run
FRAME_MODES = ["normal"] * N_DISTINCT
FRAME_MODES[5] = "still"           # one PnP-fallback frame per cycle (GRIC prefers the homography)
FRAME_OUTLIERS = [0.0, 0.3, 0.6, 0.0, 0.3, 0.0, 0.6, 0.0]      # SURVEY 8d sweep, cycled
FP64_PEAK_TFLOPS = 40.0            # nominal B200 FP64 FMA peak (SURVEY 8d; no measured figure in MEASURED_PEAKS.json)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "torch_gpu"])
    ap.add_argument("--config", default="vo", choices=["vo", "corr64", "ransac10k", "pairs64", "parity"])
    ap.add_argument("--cpu-frames", type=int, default=3, help="frames of the CPU baseline sample")
    ap.add_argument("--no-extras", action="store_true", help="skip precision modes / library baseline / extra configs / e2e_libs")
    ap.add_argument("--diag-no-track", action="store_true",
                    help="DIAGNOSTIC, not a bench value: replace the tracker by an identity pose to see the networks-only ceiling of the pipeline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (the 4x4 float64 global pose) as DIR/pose.npy, "
                         "so that two builds can be compared output for output on the same seeded inputs")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.config != "vo" or a.diag_no_track):
        ap.error("--dump-outputs applies to the default workload (--impl b200 --config vo) only")
    return a


def dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------
# synthetic inputs (synthdata.py: seeded generators only, no arithmetic of the path)
# ------------------------------------------------------------------------------------------------
def make_inputs(seed):
    import synthdata as synth
    K = synth.kitti_intrinsics(H, W)
    frames = [synth.value_noise_image(H, W, seed * 100 + i) for i in range(N_DISTINCT)]
    analytic = [synth.frame_inputs(i, H, W, K, FRAME_MODES[i], FRAME_OUTLIERS[i]) for i in range(N_DISTINCT)]
    return K, frames, analytic


# ------------------------------------------------------------------------------------------------
# CPU baseline / --impl reference: the oracle port of one frame on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_frame(oracle_state, ref_img, cur_img, analytic, K):
    """One reference frame on the CPU (oracle restatement of dfvo.py:299-345 + 121-262): both networks in
    torch fp32, consistency map, then selection / E-tracker / scale (or PnP) on the analytic flow."""
    import torch
    from oracle import nets, vo
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    p_flow, p_enc, p_dec = oracle_state
    to_t = lambda im: torch.from_numpy(np.transpose(im / 255, (2, 0, 1))).unsqueeze(0).float()
    with torch.no_grad():
        nets.liteflow_inference_flow(p_flow, to_t(ref_img), to_t(cur_img))
        import PIL.Image as pil
        feed = np.transpose(np.asarray(pil.fromarray(cur_img).resize((FEED_W, FEED_H), pil.LANCZOS), np.float32) / 255, (2, 0, 1))[None]
        d = nets.monodepth2_inference_depth(p_enc, p_dec, torch.from_numpy(np.ascontiguousarray(feed)))[0, 0].numpy()
    vo.preprocess_depth(vo.resize_nearest(d, W, H), [[0.3, 1], [0, 1]], [0, 50])
    depth = vo.preprocess_depth(analytic["depth"], [[0.3, 1], [0, 1]], [0, 50])
    good, cells = vo.local_bestn_indices(analytic["diff"])
    pose = np.eye(4)
    if not good:
        return pose
    kp1, kp2 = vo.keypoints_from_indices(cells, analytic["fwd"], W)
    r = vo.compute_pose_2d2d(kp1, kp2, K)
    pose[:3, :3], pose[:3, 3:] = r["R"], r["t"]
    scale = -1
    if np.linalg.norm(r["t"]) != 0:
        scale = vo.find_scale_from_depth(kp1, kp2, np.linalg.inv(pose), depth, K)
        if scale != -1:
            pose[:3, 3] *= scale
    if np.linalg.norm(r["t"]) == 0 or scale == -1:
        pose = vo.compute_pose_3d2d(kp1, kp2, depth, K)[0]
    return pose


def cpu_baseline(n_frames, K, frames, analytic):
    import torch
    from oracle import nets, synth
    # all host threads it can usefully use: oneDNN/OpenMP convolutions stop scaling (and then collapse) well
    # before a 100+-core host is saturated, so the pool is capped; `cores` reports what was used
    cores = min(os.cpu_count() or 1, int(os.environ.get("DFVO_CPU_THREADS", "32")))
    torch.set_num_threads(cores)
    enc, dec = synth.monodepth2_weights(4869, FEED_H, FEED_W)
    state = (nets.to_torch(synth.liteflownet_weights()),
             {k: v for k, v in nets.to_torch(enc).items() if not isinstance(v, int)}, nets.to_torch(dec))
    np.random.seed(4869)
    poses = []
    cpu_frame(state, frames[0], frames[1], analytic[1], K)          # warm-up (thread pools, allocator)
    np.random.seed(4869)
    t0 = time.perf_counter()
    for i in range(1, n_frames + 1):
        poses.append(cpu_frame(state, frames[(i - 1) % N_DISTINCT], frames[i % N_DISTINCT], analytic[i % N_DISTINCT], K))
    dt = time.perf_counter() - t0
    return dict(value=n_frames / dt, unit="frames/s", cores=cores, kind="port",
                sample="%d frames of the same workload through oracle/ (torch-fp32 networks + cv2/sklearn solvers), %.1f s" % (n_frames, dt)), poses


# ------------------------------------------------------------------------------------------------
# clocks sampler (10 ms period: the timed region of the default run is ~0.3 s)
# ------------------------------------------------------------------------------------------------
class Clocks:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index
        self.t_begin = self.t_end = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
            t0 = time.time()
            while not self.rows and time.time() - t0 < 3.0:       # first sample before the timed region starts
                time.sleep(0.01)
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def mark(self, begin):
        if begin:
            self.t_begin = time.time()
        else:
            self.t_end = time.time()

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        time.sleep(0.05)
        self.proc.terminate()
        inside = [r for (t, r) in self.rows if self.t_begin is not None and self.t_begin - 0.02 <= t <= (self.t_end or t) + 0.02]
        rows = inside if inside else [r for (_, r) in self.rows]
        num = lambda v: v.replace(".", "", 1).isdigit()
        sm = [float(r[1]) for r in rows if len(r) > 8 and num(r[1])]
        mx = [float(r[2]) for r in rows if len(r) > 8 and num(r[2])]
        pw = [float(r[3]) for r in rows if len(r) > 8 and num(r[3])]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in rows if len(r) > 8 for i in range(4) if r[5 + i].lower().startswith("active")})
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=max(mx) if mx else None, reasons=reasons, samples=len(sm),
                    samples_in_timed_region=len(inside), power_w_max=max(pw) if pw else None)


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    K, frames, analytic = make_inputs(0)
    # `steps` bounded samples; each step = one frame of the same workload on all host threads
    n = max(1, min(args.steps, 6))
    base, _ = cpu_baseline(n, K, frames, analytic)
    line = dict(impl="reference", metric=METRIC, value=base["value"], unit="frames/s", n_gpus=args.gpus, steps=n, warmup=1,
                ms_per_step=1e3 / base["value"], higher_is_better=True, scaling="weak", vs_baseline=None, dtype="f32",
                data="synthetic", config=dict(workload=WORKLOAD, note="reference's CPU path = oracle port (the reference is pure "
                "Python + torch/cv2/sklearn; /root/reference does not travel to the GPU box)"),
                cpu_baseline=base, e2e=dict(value=base["value"], unit="frames/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
# library GPU baseline (SURVEY 8d last row / BASELINE.md 3.1): the reference graph through torch/cuDNN on this GPU
# ------------------------------------------------------------------------------------------------
def torch_gpu_baseline(frames, iters=8):
    """oracle/nets.py (the functional restatement of the reference modules) executed by torch on cuda: cuDNN convolutions,
    the correlation as 49 shifted multiply-reduce torch ops (the reference's own cupy kernel needs cupy; its kernel text lives
    under /root/reference, which does not travel).  Three settings: strict fp32, TF32 (torch's default for cuDNN convs), and
    bf16 autocast + channels_last.  A BASELINE measurement: nothing of the product runs here."""
    import torch
    import torch.nn.functional as F
    from oracle import nets, synth
    dev = torch.device("cuda")
    enc, dec = synth.monodepth2_weights(4869, FEED_H, FEED_W)
    cu = lambda d: {k: (v.to(dev) if hasattr(v, "to") else v) for k, v in nets.to_torch(d).items()}
    p_flow = cu(synth.liteflownet_weights())
    p_enc = {k: v for k, v in cu(enc).items() if not isinstance(v, int)}
    p_dec = cu(dec)
    to_t = lambda im: torch.from_numpy(np.transpose(im / 255, (2, 0, 1))).unsqueeze(0).float().to(dev)
    a, b = to_t(frames[0]), to_t(frames[1])
    feed = F.interpolate(b, (FEED_H, FEED_W), mode="bilinear", align_corners=False)

    def timed(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    out = {}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True

    class Bf16Convs:
        """torch.nn.functional with conv2d / conv_transpose2d running on bf16 channels_last operands (weights converted once),
        results returned as fp32: the same split as the product (bf16 conv operands, fp32 flows / coordinates)."""
        def __init__(self):
            self.cache = {}

        def __getattr__(self, k):
            return getattr(F, k)

        def _w(self, t):
            if t is None:
                return None
            c = self.cache.get(id(t))
            if c is None:
                c = t.to(torch.bfloat16)
                c = c.contiguous(memory_format=torch.channels_last) if c.dim() == 4 else c
                self.cache[id(t)] = c
            return c

        def conv2d(self, x, w, b=None, **kw):
            return F.conv2d(x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last), self._w(w), self._w(b), **kw).float()

        def conv_transpose2d(self, x, w, b=None, **kw):
            return F.conv_transpose2d(x.to(torch.bfloat16).contiguous(memory_format=torch.channels_last), self._w(w), self._w(b), **kw).float()

    try:
        with torch.no_grad(), torch.device(dev):
            for name, tf32, bf16 in (("fp32", False, False), ("tf32", True, False), ("bf16_convs_channels_last", True, True)):
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = tf32
                nets.F = Bf16Convs() if bf16 else F

                def flow():
                    return nets.liteflow_inference_flow(p_flow, a, b)

                def depth():
                    return nets.monodepth2_inference_depth(p_enc, p_dec, feed)
                ms_f, ms_d = timed(flow), timed(depth)
                out[name] = dict(flow_net_ms=ms_f, depth_net_ms=ms_d, networks_fps=1e3 / (ms_f + ms_d))
    finally:
        nets.F = F
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    out["what"] = ("reference graph (oracle/nets.py restatement of lite_flow_net.py:31-325, resnet_encoder.py:87-98, depth_decoder.py:50-65) "
                   "through torch %s / cuDNN on this GPU, networks only (no tracker); %d iterations after 3 warm-ups" % (torch.__version__, iters))
    return out


def run_torch_gpu(args):
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    import torch
    torch.cuda.set_device(local_rank)
    K, frames, analytic = make_inputs(0)
    base = torch_gpu_baseline(frames)
    best = max(v["networks_fps"] for v in base.values() if isinstance(v, dict))
    print(json.dumps(dict(impl="torch_gpu", metric=METRIC, value=best, unit="frames/s (networks only)", n_gpus=1, higher_is_better=True,
                          config=dict(workload=WORKLOAD), gpu_library_baseline=base)))


# ------------------------------------------------------------------------------------------------
# BASELINE configs[2]: 64 pairs through the correlation at the five level shapes + the consistency map (HBM roofline)
# ------------------------------------------------------------------------------------------------
CORR_LEVELS = [(6, 192, 11, 38, 1), (5, 128, 22, 76, 1), (4, 96, 44, 152, 1), (3, 64, 88, 304, 2), (2, 64, 176, 608, 2)]


def bench_corr64(rt, pairs=64, iters=5):
    """Times `dfvo_correlation_nhwc_bf16` (the kernel of the product path, on its own NHWC bf16 layout) for B = 2*pairs maps
    at each pyramid level, and `dfvo_fb_consistency` for `pairs` 376x1241 flow pairs.  Algorithmic bytes (SURVEY 8d, bytes
    *touched*, bf16 = half the fp32 figures): first operand at the sampled pixels + the (7s)^2-window union of the second
    operand (= the whole map) + the 49-channel output; consistency 20 B / pixel.  Inputs exceed the 126 MB L2 at levels 2-4;
    the small levels are timed L2-warm, as they run in the network."""
    import torch
    lib = rt.lib
    B = 2 * pairs
    hbm = float(peaks().get("hbm_gbs", 6650.0))
    rows, tot_bytes, tot_ms = [], 0.0, 0.0
    ev = lambda: torch.cuda.Event(enable_timing=True)
    for (L, C, h, w, s) in CORR_LEVELS:
        ho, wo = (h + s - 1) // s, (w + s - 1) // s
        a = torch.randn((B, h, w, C), device="cuda").to(torch.bfloat16)
        b = torch.randn((B, h, w, C), device="cuda").to(torch.bfloat16)
        o = torch.empty((B, ho, wo, 64), device="cuda", dtype=torch.bfloat16)
        call = lambda: lib.check(lib.dfvo_correlation_nhwc_bf16(ctypes.c_void_p(a.data_ptr()), ctypes.c_void_p(b.data_ptr()), ctypes.c_void_p(o.data_ptr()),
                                                                 B, C, C, h, w, s, 1, 0, rt.stream_ptr()))
        for _ in range(3):
            call()
        e0, e1 = ev(), ev()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(iters):
            call()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        nbytes = B * (ho * wo * C * 2 + h * w * C * 2 + ho * wo * 49 * 2)      # first @ sampled px, second (whole), output
        rows.append(dict(level=L, C=C, h=h, w=w, stride=s, ms=ms, algorithmic_mb=nbytes / 1e6, gbs=nbytes / ms / 1e6, frac_of_hbm=nbytes / ms / 1e6 / hbm))
        tot_bytes += nbytes; tot_ms += ms
        del a, b, o
    fwd = torch.randn((pairs, 2, H, W), device="cuda")
    bwd = -fwd
    diff = torch.empty((pairs, H, W), device="cuda")

    def fb():
        lib.check(lib.dfvo_fb_consistency_batch(ctypes.c_void_p(fwd.data_ptr()), ctypes.c_void_p(bwd.data_ptr()),
                                                ctypes.c_void_p(diff.data_ptr()), pairs, H, W, rt.stream_ptr()))
    fb()
    e0, e1 = ev(), ev()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fb()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    nb = pairs * H * W * 20
    fbrow = dict(ms=ms, algorithmic_mb=nb / 1e6, gbs=nb / ms / 1e6, frac_of_hbm=nb / ms / 1e6 / hbm, launches=1)
    tot_bytes += nb; tot_ms += ms
    return dict(workload="BASELINE configs[2]: %d pairs, correlation at the five level shapes (bf16 NHWC) + fwd-bwd consistency" % pairs,
                levels=rows, fb_consistency=fbrow, total_ms=tot_ms, total_algorithmic_gb=tot_bytes / 1e9, gbs=tot_bytes / tot_ms / 1e6,
                roofline=dict(bound="hbm", achieved=tot_bytes / tot_ms / 1e6, peak=hbm, unit="GB/s", frac=tot_bytes / tot_ms / 1e6 / hbm,
                              peak_source="MEASURED_PEAKS.json hbm_gbs" if "hbm_gbs" in peaks() else "fallback 6.65 TB/s"))


# ------------------------------------------------------------------------------------------------
# BASELINE configs[3]: Sampson scoring 10 000 x 2048 (FP64 roofline) + the full replayed E-RANSAC at {0, .3, .6} outliers
# ------------------------------------------------------------------------------------------------
def bench_ransac10k(rt, iters=10):
    import torch
    import synthdata as synth
    from b200 import tracking
    lib = rt.lib
    K = synth.kitti_intrinsics(H, W)
    cx, cy, fx, fy = K
    kp_ref, kp_cur, _ = synth.correspondences(seed=32, n=2048, outlier_frac=0.3)
    x1 = (kp_cur - [cx, cy]) / [fx, fy]
    x2 = (kp_ref - [cx, cy]) / [fx, fy]
    M, N = 10000, 2048
    # hypotheses: 5-point solutions of random minimal samples (first root of each) -- generated on the device, not timed
    rs = np.random.RandomState(0)
    ms_ = 6000
    sub = np.stack([rs.choice(N, 5, replace=False) for _ in range(ms_)])
    d1, d2 = rt.from_host(np.ascontiguousarray(x1[sub])), rt.from_host(np.ascontiguousarray(x2[sub]))
    dE, dn = rt.empty((ms_, 10, 9), np.float64), rt.empty((ms_,), np.int32)
    lib.check(lib.dfvo_five_point(d1.ptr, d2.ptr, ms_, dE.ptr, dn.ptr, rt.stream_ptr()))
    E, n = dE.numpy(), dn.numpy()
    models = np.concatenate([E[i, :n[i]] for i in range(ms_)])[:M]
    assert models.shape[0] == M, "not enough 5-point solutions for 10 000 hypotheses"
    dM, dx1, dx2 = rt.from_host(models), rt.from_host(x1), rt.from_host(x2)
    cnt = rt.empty((M,), np.int32)
    thr2 = (0.2 / fx) ** 2
    call = lambda: lib.check(lib.dfvo_score_hypotheses(dM.ptr, M, dx1.ptr, dx2.ptr, N, thr2, cnt.ptr, rt.stream_ptr()))
    for _ in range(3):
        call()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    flop = 33.0 * M * N
    out = dict(workload="BASELINE configs[3]: Sampson scoring of %d hypotheses x %d correspondences, FP64" % (M, N), scoring_ms=ms,
               algorithmic_gflop=flop / 1e9, evaluations_per_s=M * N / ms * 1e3,
               roofline=dict(bound="fp64", achieved=flop / ms / 1e9, peak=FP64_PEAK_TFLOPS, unit="TFLOP/s", frac=flop / ms / 1e9 / FP64_PEAK_TFLOPS,
                             peak_source="nominal B200 FP64 FMA peak (SURVEY 8d); FLOPs = 33 per (model, correspondence)"),
               inliers_max=int(cnt.numpy().max()))
    # the full replayed RANSAC (5 repeats + GRIC + homography vote + recoverPose) per outlier fraction
    eng = tracking.Engine(H, W, rt)
    full = {}
    for frac in (0.0, 0.3, 0.6):
        a, b, _ = synth.correspondences(seed=32, n=2000, outlier_frac=frac)
        da, db = rt.from_host(a), rt.from_host(b)
        ts = []
        for i in range(6):
            np.random.seed(4869)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = tracking.compute_pose_2d2d(eng, a, b, K, kp_ref_buf=da, kp_cur_buf=db)
            torch.cuda.synchronize()
            ts.append((time.perf_counter() - t0) * 1e3)
        full["%.1f" % frac] = dict(ms=float(np.median(ts[1:])), iterations=[int(v) for v in r["ransac_info"][:, 1]], inliers=int(r["inliers"].sum()),
                                   valid=bool(r["valid"]))
    out["full_ransac_ms_by_outlier_fraction"] = full
    return out


# ------------------------------------------------------------------------------------------------
# batched many-frames mode (north_star; BASELINE configs[2] sharding): 64 independent pairs split over the ranks
# ------------------------------------------------------------------------------------------------
def run_pairs64(args):
    import torch
    rank, local_rank, world = dist_env()
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from b200 import multi, native, runtime as rt_mod
    import synthdata as synth
    rt = rt_mod.CudaRuntime(local_rank)
    rt_mod.set_runtime(rt)
    total = 64
    flow_w = synth.liteflownet_weights()
    if world > 1:
        (flow_w,) = multi.broadcast_weights([flow_w], src=0, device=torch.device("cuda", local_rank))
    sh = multi.PairShard(total, rank, world)
    runner = multi.PairBatchRunner(rt, H, W, sh.count, flow_w, precision=native.PREC_BF16)
    # frames of pair p (global index sh.first + p): two distinct textures
    imgs = []
    for p in range(sh.count):
        g = sh.first + p
        imgs += [rt.from_host(synth.value_noise_image(H, W, 2000 + 2 * g)), rt.from_host(synth.value_noise_image(H, W, 2001 + 2 * g))]

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()
    warm = max(3, args.warmup if args.warmup < 6 else 3)
    for _ in range(warm):
        runner.forward(imgs)
    steps = max(1, min(args.steps, 10))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = rt.lib.dfvo_launch_count()
    barrier()
    e0.record()
    for _ in range(steps):
        stats = runner.forward(imgs)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = rt.lib.dfvo_launch_count() - l0
    if world > 1:
        ms = multi.max_over_ranks(ms, device=torch.device("cuda", local_rank))
    all_stats = multi.gather_pair_stats(stats, sh, world, device=torch.device("cuda", local_rank))
    if rank != 0:
        return
    line = dict(metric="image pairs/sec through LiteFlowNet fwd+bwd + consistency (batched many-frames mode)", value=total * steps / (ms / 1e3), unit="pairs/s",
                n_gpus=world, steps=steps, warmup=warm, ms_per_step=ms / steps, higher_is_better=True, scaling="strong", vs_baseline=None,
                dtype="bf16 tensor-core convs (fp32 accumulate)", data="synthetic frames + seeded random-init weights",
                config=dict(workload="64 independent 376x1241 image pairs, contiguous block of 64/N pairs per GPU, one batched forward per step; NCCL weight "
                            "broadcast + one all_gather of the per-pair consistency statistics", pairs_per_gpu=sh.count,
                            l2="activation working set of one rank (>0.5 GB per pair) exceeds the 126 MB L2"),
                gpu_launches=int(launches), pair_stats=dict(n=len(all_stats), mean_flow_diff_first=float(all_stats[0][0]), mean_flow_diff_last=float(all_stats[-1][0])))
    print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
# e2e through the reference-API mirror (what libs/dfvo.py would call per frame)
# ------------------------------------------------------------------------------------------------
def libs_e2e(rt, K, frames, d_fwd, d_bwd, d_diff, analytic, flow_w, enc, dec, n_steps, state):
    """dfvo.py:299-345 + 121-262 (hybrid, default configuration) against df-vo_b200/libs: DeepModel built from checkpoints on
    disk (torch.load path), forward_depth -> host depth (the driver resizes it with cv2 itself), forward_flow -> device-backed
    arrays, KeypointSampler, EssTracker (+ scale recovery), PnpTracker on fallback.  Analytic flow is copied over the network
    outputs on the device (as everywhere in this file); the depth the driver post-processes is the analytic one."""
    import torch
    from b200 import config, tracking
    for k in [k for k in sys.modules if k == "libs" or k.startswith("libs.")]:
        del sys.modules[k]
    from libs.deep_models.deep_models import DeepModel
    from libs.geometry.camera_modules import SE3, Intrinsics
    from libs.matching.keypoint_sampler import KeypointSampler
    from libs.tracker import EssTracker, PnpTracker
    tmp = tempfile.mkdtemp(prefix="dfvo_bench_")
    t = lambda d: {k: (torch.from_numpy(np.ascontiguousarray(v)) if isinstance(v, np.ndarray) else v) for k, v in d.items()}
    torch.save(t(flow_w), os.path.join(tmp, "lfn.pth"))
    os.makedirs(os.path.join(tmp, "depth"))
    torch.save(t(enc), os.path.join(tmp, "depth", "encoder.pth"))
    torch.save(t(dec), os.path.join(tmp, "depth", "depth.pth"))
    cfg = config.default_cfg(H, W)
    cfg.deep_flow.flow_net_weight = os.path.join(tmp, "lfn.pth")
    cfg.depth.deep_depth.pretrained_model = os.path.join(tmp, "depth")
    tracking._default_engine = None
    dm = DeepModel(cfg)
    dm.initialize_models()
    cam = Intrinsics(K)
    e_trk, p_trk, sampler = EssTracker(cfg, cam, None), PnpTracker(cfg, cam), KeypointSampler(cfg)
    ys = np.minimum(np.floor(np.arange(H) * (1.0 / (H / FEED_H))).astype(np.int64), FEED_H - 1)
    xs = np.minimum(np.floor(np.arange(W) * (1.0 / (W / FEED_W))).astype(np.int64), FEED_W - 1)
    crop = np.zeros((H, W)); crop[int(H * 0.3):H, 0:W] = 1
    ref, cur = {}, {}
    modes = {}

    def frame(fid):
        slot = fid % N_DISTINCT
        cur["id"], cur["img"] = fid, frames[slot]
        raw = dm.forward_depth(imgs=[cur["img"]])                      # D2H of the feed-size depth
        cur["raw_depth"] = raw[ys][:, xs]                               # cv2.resize(..., INTER_NEAREST) of the driver (dfvo.py:314-317)
        a = analytic[slot]["depth"]
        cur["depth"] = a * (crop * ((a < 50) * (a > 0)))                # preprocess_depth (utils.py:89-114) on the analytic depth
        pose = None
        if ref:
            flows = dm.forward_flow(cur, ref, forward_backward=True)
            flows[(ref["id"], fid)].dev.t.copy_(d_fwd[slot].t)
            flows[(fid, ref["id"])].dev.t.copy_(d_bwd[slot].t)
            flows[(ref["id"], fid, "diff")].dev.t.copy_(d_diff[slot].t)
            ref["flow"] = flows[(ref["id"], fid)].copy()
            cur["flow"] = flows[(fid, ref["id"])].copy()
            ref["flow_diff"] = flows[(ref["id"], fid, "diff")].copy()
            sel = sampler.kp_selection(cur, ref)
            pose = SE3()
            if sel["good_kp_found"]:
                sampler.update_kp_data(cur, ref, sel)
                out = e_trk.compute_pose_2d2d(ref["kp_best"], cur["kp_best"], True)
                E_pose, scale = out["pose"], -1
                pose.R = E_pose.R
                modes[fid] = "E"
                if np.linalg.norm(E_pose.t) != 0:
                    scale = e_trk.scale_recovery(cur, ref, E_pose, False)["scale"]
                    if scale != -1:
                        pose.t = E_pose.t * scale
                if np.linalg.norm(E_pose.t) == 0 or scale == -1:
                    pose = p_trk.compute_pose_3d2d(ref["kp_best"], cur["kp_best"], ref["depth"], True)["pose"]
                    modes[fid] = "PnP"
        for k in cur:
            ref[k] = cur[k]
        return pose

    for fid in range(3):
        frame(fid)
    torch.cuda.synchronize()
    state["h2d"] = state["d2h"] = 0
    t0 = time.perf_counter()
    for fid in range(3, 3 + n_steps):
        frame(fid)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    return dict(value=n_steps / dt, unit="frames/s", steps=n_steps, ms_per_step=dt / n_steps * 1e3, h2d_bytes_per_step=int(state["h2d"] / n_steps),
                d2h_bytes_per_step=int(state["d2h"] / n_steps), branches=sorted(set(modes.values())),
                what="libs.deep_models.DeepModel.forward_depth / forward_flow + KeypointSampler + EssTracker / PnpTracker called per frame like "
                     "libs/dfvo.py does (host frames in, host depth + device-backed flows out, one frame at a time, no overlap)")


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    rank, local_rank, world = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (there is no CPU fallback for --impl b200)"
    torch.cuda.set_device(local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from b200 import native, pipeline, runtime as rt_mod
    import synthdata as synth
    rt = rt_mod.CudaRuntime(local_rank)
    rt_mod.set_runtime(rt)
    lib = rt.lib
    extras = (not args.no_extras) and world == 1

    # ---- weights: rank 0 generates, NCCL broadcast to the others (the only collective of the path)
    enc, dec = synth.monodepth2_weights(4869, FEED_H, FEED_W)
    flow_w = synth.liteflownet_weights()
    if world > 1:
        from b200 import multi
        flow_w, enc, dec = multi.broadcast_weights([flow_w, enc, dec], src=0, device=torch.device("cuda", local_rank))

    K, frames, analytic = make_inputs(rank)
    overlap = os.environ.get("DFVO_OVERLAP", "1") != "0"
    # network engines in flight.  Measured (profiles/r02_pipeline_modes.json): 3 engines + pipelined tracker 446 fps at 11.2 ms latency,
    # 2 engines + tracker read in the same step 421 fps at 7.1 ms (reported as e2e.low_latency), 1 engine 362 fps
    inflight = int(os.environ.get("DFVO_INFLIGHT", "3")) if overlap else 1

    # device-resident copies of everything a step consumes
    d_frames = [rt.from_host(f) for f in frames]
    d_fwd = [rt.from_host(a["fwd"][None]) for a in analytic]
    d_bwd = [rt.from_host(a["bwd"][None]) for a in analytic]
    d_diff = [rt.from_host(a["diff"][None, :, :, 0]) for a in analytic]
    d_depth = [rt.from_host(a["depth"]) for a in analytic]
    pinned = [torch.from_numpy(f).pin_memory() for f in frames]
    state = dict(h2d=0, d2h=0)

    def inject(pipe, st):
        # analytic flow / depth over the (random-weight) network outputs: D2D, inside the timed region, on the frame's streams
        slot = st.id % N_DISTINCT
        if st.fwd is not None:
            st.fwd.t.copy_(d_fwd[slot].t); st.bwd.t.copy_(d_bwd[slot].t); st.diff.t.copy_(d_diff[slot].t)
        with pipe.depth_stream(st.id):                  # ordered after the depth network's own post-processing
            tmp = pipe._buf("dsrc%d" % pipe.slot(st.id), (H, W), np.float32)
            tmp.t.copy_(d_depth[slot].t)
            pipe.eng.depth_post(tmp, pipe.cfg.crop.depth_crop, 0.0, 50.0, st.raw_depth, st.depth)

    # count the bytes the host side moves per step
    up0, dn0 = rt_mod.Buf.upload, rt_mod.Buf.numpy

    def up(self, arr):
        state["h2d"] += int(arr.numel() * arr.element_size()) if torch.is_tensor(arr) else int(np.asarray(arr).nbytes)
        return up0(self, arr)

    def dn(self):
        a = dn0(self)
        state["d2h"] += int(a.nbytes)
        return a
    rt_mod.Buf.upload, rt_mod.Buf.numpy = up, dn
    fh0 = rt.from_host

    def from_host(arr):
        state["h2d"] += int(np.asarray(arr).nbytes)
        return fh0(arr)
    rt.from_host = from_host

    def barrier():
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
        torch.cuda.synchronize()

    def build_pipe(precision, overlap_, inflight_, pipelined_=None):
        np.random.seed(4869 + rank)
        if pipelined_ is None:
            pipelined_ = os.environ.get("DFVO_PIPELINED", "1") != "0"
        p = pipeline.FramePipeline(K, H, W, precision=precision, runtime=rt, overlap=overlap_, inflight=inflight_, inject=inject,
                                   tracker_thread=overlap_ and os.environ.get("DFVO_TRACKER_THREAD", "0") == "1",
                                   pipelined=overlap_ and pipelined_)
        p.load_weights(flow_w, enc, dec)
        return p

    def timed(pipe, n_steps, resident, clocks=None):
        """K steps of FramePipeline.step (the public API).  Returns (ms on the device, launches, mean host latency in ms from
        handing a frame to step() until its pose is returned)."""
        state["h2d"] = state["d2h"] = 0
        l0 = lib.dfvo_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        submit, lat = {}, []
        lag = pipe.lag
        barrier()
        if clocks:
            clocks.mark(True)
        e0.record()
        for _ in range(n_steps):
            fid = pipe.stage
            slot = fid % N_DISTINCT
            submit[fid] = time.perf_counter()
            pose = pipe.step(d_frames[slot] if resident else pinned[slot])
            if pose is not None and (fid - lag) in submit:
                lat.append(time.perf_counter() - submit[fid - lag])
        if pipe.overlap:                  # the closing event waits for all of the pipeline's streams
            cs = torch.cuda.current_stream()
            for sx in pipe.s_nets + pipe.s_depths + [pipe.s_trk]:
                cs.wait_stream(sx)
        e1.record()
        barrier()
        state["last_pose"] = pose
        if clocks:
            clocks.mark(False)
        ms = e0.elapsed_time(e1)
        if world > 1:
            from b200 import multi
            ms = multi.max_over_ranks(ms, device=torch.device("cuda", local_rank))
        return ms, lib.dfvo_launch_count() - l0, (float(np.mean(lat)) * 1e3 if lat else None)

    def warm(pipe, n):
        for _ in range(n + 1):
            fid = pipe.stage
            pipe.step(d_frames[fid % N_DISTINCT])

    # ---------------------------------------------------------------- headline: bf16, two engines in flight
    pipe = build_pipe(native.PREC_BF16, overlap, inflight)
    if args.diag_no_track:
        pipe.track = lambda cur, ref: np.eye(4)
        sys.stderr.write("bench.py: --diag-no-track: tracker replaced by an identity pose; the printed value is NOT the metric\n")
    # every network engine needs three forwards before it replays its CUDA graph (eager, capture, replay)
    warmup = max(3 * inflight + 1, args.warmup)
    warm(pipe, warmup)
    clocks = Clocks(local_rank)
    if rank == 0:
        clocks.start()
    ms, launches, _ = timed(pipe, args.steps, True, clocks if rank == 0 else None)
    clk = clocks.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        # the warm-up is longer than the pipeline's lag, so every timed step returns a pose
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "pose.npy"), np.asarray(state["last_pose"], np.float64))
    ms_e2e, _, lat_e2e = timed(pipe, args.steps, False)
    h2d, d2h = state["h2d"] / args.steps, state["d2h"] / args.steps
    pipe.flush()
    torch.cuda.synchronize()
    # tracker cost per branch / outlier fraction (host time of the tracker path of a frame, device waits included)
    by = {}
    for fid, m in pipe.modes.items():
        if m is None or fid not in pipe.track_ms:
            continue
        key = "%s@%.1f" % (m, FRAME_OUTLIERS[fid % N_DISTINCT])
        by.setdefault(key, []).append(pipe.track_ms[fid])
    tracker_ms = {k: float(np.median(v)) for k, v in sorted(by.items())}

    # ---------------------------------------------------------------- in-order variant (pose of frame t returned by step t)
    inorder = None
    if extras or world == 1:
        p1 = pipeline.FramePipeline(K, H, W, precision=native.PREC_BF16, runtime=rt, overlap=False, engine=pipe.eng, inject=inject)
        warm(p1, 3)
        n1 = max(10, args.steps // 2)
        ms1, _, _ = timed(p1, n1, False)
        inorder = dict(value=n1 / (ms1 / 1e3), unit="frames/s", latency_ms=ms1 / n1, what="FramePipeline(overlap=False): one stream, in order, host frames in, pose of "
                       "frame t returned by step t (latency = 1 step)")

    # ---------------------------------------------------------------- lower-latency overlapped variant: two engines, tracker read in the same step
    low_lat = None
    if extras and overlap:
        p2 = build_pipe(native.PREC_BF16, True, 2, False)
        warm(p2, 7)
        n2 = max(16, args.steps // 2)
        ms2, _, lat2 = timed(p2, n2, False)
        p2.flush()
        low_lat = dict(value=n2 / (ms2 / 1e3), unit="frames/s", latency_ms=lat2,
                       what="FramePipeline(overlap=True, inflight=2, pipelined=False): two network engines, step(t) returns the pose of frame t-2")
        del p2

    # ---------------------------------------------------------------- roofline of the dominant kernels (tcgen05 convs)
    # CUDA-event timing of every launch over a few steps, on an in-order single-stream pipeline sharing the built networks (in
    # the two-stream pipeline the tracker's and the depth network's kernels run beside the convolutions, which would be charged
    # to whichever launch they overlap)
    prof = pipeline.FramePipeline(K, H, W, precision=native.PREC_BF16, runtime=rt, overlap=False, engine=pipe.eng, inject=inject)
    warm(prof, 1)
    torch.cuda.synchronize()
    lib.dfvo_profile_enable(1)
    prof_steps = 5
    for _ in range(prof_steps):
        prof.step(d_frames[prof.stage % N_DISTINCT])
    torch.cuda.synchronize()
    tc_ms, tc_n, tc_fl = ctypes.c_double(), ctypes.c_longlong(), ctypes.c_double()
    lib.dfvo_profile_read(ctypes.byref(tc_ms), ctypes.byref(tc_n), ctypes.byref(tc_fl))
    lib.dfvo_profile_enable(0)

    # ---------------------------------------------------------------- other precision modes (same pipeline, same inputs)
    prec_modes = None
    if extras:
        prec_modes = {"bf16": dict(value=world * args.steps / (ms / 1e3), unit="frames/s")}
        for name, prec in (("tf32", native.PREC_TF32), ("fp32", native.PREC_FP32)):
            try:
                pm = build_pipe(prec, overlap, inflight)
                warm(pm, 3 * inflight + 1)
                n = max(8, args.steps // 4) if name == "tf32" else 8
                msm, _, _ = timed(pm, n, True)
                pm.flush()
                prec_modes[name] = dict(value=n / (msm / 1e3), unit="frames/s", steps=n)
                del pm
                torch.cuda.synchronize(); torch.cuda.empty_cache()
            except Exception as e:                              # a mode that cannot be built is reported, not hidden
                prec_modes[name] = dict(error=str(e)[:200])

    e2e_libs = None
    if extras:
        try:
            e2e_libs = libs_e2e(rt, K, frames, d_fwd, d_bwd, d_diff, analytic, flow_w, enc, dec, max(10, args.steps // 4), state)
        except Exception as e:
            e2e_libs = dict(error=str(e)[:300])
    extra_cfg = None
    if extras:
        extra_cfg = {}
        for name, fn in (("corr64", bench_corr64), ("ransac10k", bench_ransac10k)):
            try:
                extra_cfg[name] = fn(rt)
            except Exception as e:
                extra_cfg[name] = dict(error=str(e)[:300])
            torch.cuda.empty_cache()
    gpu_lib = None
    if extras:
        try:
            gpu_lib = torch_gpu_baseline(frames)
        except Exception as e:
            gpu_lib = dict(error=str(e)[:300])

    if rank != 0:
        return
    pk = peaks()
    peak_tf = float(pk.get("bf16_tflops_sustained", 1400.0))
    peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained" if "bf16_tflops_sustained" in pk else "fallback 1.4 PFLOP/s sustained (B200_PROFILING.md)"
    achieved = (tc_fl.value / 1e12) / (tc_ms.value / 1e3) if tc_ms.value > 0 else 0.0
    traffic, traffic_src = None, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "conv_tc_traffic.json")))
        traffic, traffic_src = tj["dram_bytes_per_frame"], "ncu dram__bytes_read.sum + dram__bytes_write.sum of the conv launches of one frame, " + tj.get("source", "profiles/ (round 1)")
    except Exception:
        pass
    if args.cpu_frames > 0 and world == 1:
        base, cpu_poses = cpu_baseline(args.cpu_frames, K, frames, analytic)
    else:
        base = None          # the CPU baseline is reported at N = 1 only (and skipped in ncu profiling runs)
    value = world * args.steps / (ms / 1e3)
    line = dict(
        metric=METRIC, value=value, unit="frames/s", n_gpus=world, steps=args.steps, warmup=warmup,
        ms_per_step=ms / args.steps, higher_is_better=True, scaling="weak", vs_baseline=None,
        dtype="bf16 tensor-core convs (fp32 accumulate) + fp32 flow/selection + fp64 pose solvers",
        data="synthetic frames + seeded random-init weights; tracker stages fed analytic rigid-scene flow/depth (see bench.py docstring)",
        config=dict(workload=WORKLOAD, image=[H, W], flow_net_input=[352, 1216], depth_feed=[FEED_H, FEED_W], keypoints=2000,
                    ransac_repeats=5, sequences_per_gpu=1, parallelism="1 sequence per GPU, NCCL weight broadcast only",
                    streams=("%d network engine(s) on their own streams, tracker %d frame(s) behind (%s); K steps = K frames inferred and K tracked"
                             % (inflight, pipe.lag, "its kernels enqueued in one step, its result read in the next" if pipe.pipelined else
                                "enqueued and read in the same step")) if overlap else "1 (in order)",
                    l2="per-frame activation working set (>1 GB written/read per frame) exceeds the 126 MB L2; no explicit flush",
                    frame_cycle=dict(modes=FRAME_MODES, outlier_fractions=FRAME_OUTLIERS), tracker_ms_by_branch_and_outliers=tracker_ms,
                    precision_modes=prec_modes),
        clocks=clk,
        e2e=dict(value=world * args.steps / (ms_e2e / 1e3), unit="frames/s", h2d_bytes_per_step=int(h2d), d2h_bytes_per_step=int(d2h),
                 ms_per_step=ms_e2e / args.steps, latency_ms=lat_e2e, api="FramePipeline.step(pinned uint8 frame) -> 4x4 pose on the host",
                 in_order=inorder, low_latency=low_lat),
        e2e_libs=e2e_libs,
        gpu_launches=int(launches),
        roofline=dict(kernel="k_conv_halo / k_conv_tc (tcgen05 implicit-GEMM conv, %d launches/frame)" % (tc_n.value // prof_steps), bound="tensor",
                      achieved=achieved, peak=peak_tf, unit="TFLOP/s", frac=achieved / peak_tf if peak_tf else None, traffic=traffic,
                      traffic_source=traffic_src, peak_source=peak_src, algorithmic_gflop_per_frame=tc_fl.value / prof_steps / 1e9,
                      kernel_ms_per_frame=tc_ms.value / prof_steps,
                      # share of the step of the pipeline the events were taken in (in order, one stream); the overlapped pipelines run
                      # the convolutions of up to three frames side by side, so their step is shorter than one frame's conv time
                      share_of_in_order_step=((tc_ms.value / prof_steps) / inorder["latency_ms"]) if inorder else None,
                      conv_ms_over_overlapped_step=(tc_ms.value / prof_steps) / (ms / args.steps)),
        cpu_baseline=base,
        gpu_library_baseline=gpu_lib,
        extra_configs=extra_cfg,
    )
    if args.diag_no_track:
        line = dict(diagnostic="--diag-no-track: networks-only ceiling of the pipeline, tracker replaced by an identity pose; NOT the metric",
                    frames_per_s=line["value"], e2e_frames_per_s=line["e2e"]["value"], ms_per_step=line["ms_per_step"])
    print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


def run_single_config(args):
    """--config corr64 | ransac10k | parity on one GPU: one JSON line with that configuration's numbers."""
    import torch
    rank, local_rank, world = dist_env()
    if rank != 0:
        return
    torch.cuda.set_device(local_rank)
    from b200 import runtime as rt_mod
    rt = rt_mod.CudaRuntime(local_rank)
    rt_mod.set_runtime(rt)
    if args.config == "corr64":
        r = bench_corr64(rt)
        line = dict(metric="GB/s of the correlation + consistency kernels, 64 pairs", value=r["gbs"], unit="GB/s", n_gpus=1, higher_is_better=True,
                    dtype="bf16", data="synthetic N(0,1) feature maps", config=dict(workload=r["workload"]), roofline=r["roofline"], detail=r)
    elif args.config == "ransac10k":
        r = bench_ransac10k(rt)
        line = dict(metric="Sampson evaluations/s, 10k hypotheses x 2048 correspondences", value=r["evaluations_per_s"], unit="evaluations/s", n_gpus=1,
                    higher_is_better=True, dtype="f64", data="synthetic correspondences (30 % outliers)", config=dict(workload=r["workload"]),
                    roofline=r["roofline"], detail=r)
    else:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import parity_cases as pc
        from b200 import tracking
        table = pc.measure_all(rt.lib, tracking.Engine(H, W, rt))
        line = dict(metric="precision-mode parity vs the CPU oracle at 376x1241 / 192x640", config=dict(workload="tests/parity_cases.py"), table=table)
    print(json.dumps(line))


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.impl == "torch_gpu":
        run_torch_gpu(a)
    elif a.config == "pairs64":
        run_pairs64(a)
    elif a.config != "vo":
        run_single_config(a)
    else:
        run_b200(a)
