#!/usr/bin/env python
"""bench.py -- 6-view scenes/sec of the RoadMapBCE training step on B200 (BASELINE.json config 2:
bf16 activations, batch 32 scenes per GPU, views 6x3x256x306, hidden 256 / latent 128).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]

One "step" = zero_grad + stitch/conv encoder/dense blocks/800x800 head + fused BCE/threat score +
backward + Adam on one batch of synthetic scenes; for N>1 the gradient exchange, the Adam update of each rank's
shard and the all-gather of the new weights are one kernel over NVLink peer memory (optim.FusedAdam).  `value` is timed
on the device with inputs resident in HBM; `e2e` goes through the reference-facing module call with
HOST (pinned) input buffers, H2D copies and a D2H read of the loss inside the timed region.
`--impl reference` times the CPU port of the reference path (oracle/scene_oracle.py: the same torch
CPU ops the reference executes; /root/reference itself is not present on the GPU box).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "6-view scenes/sec, RoadMapBCE train step (fwd + BCE/threat-score + bwd + Adam)"
UNIT = "scenes/s"
VIEW_H, VIEW_W, MAP = 256, 306, 800
HIDDEN, LATENT = 256, 128
FLOP_C2_PER_SCENE = 2.0 * 256 * 1836 * 32 * 288      # 8.663 GFLOP (SURVEY 8(d))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="roadmap", choices=["roadmap", "ae", "bb", "inference"],
                    help="roadmap = BASELINE config 2 (the metric's config); ae = config 3; bb = config 4; inference = config 5")
    ap.add_argument("--mode", default=None, choices=[None, "inference", "train"], help="--mode inference == --config inference")
    ap.add_argument("--parity-scenes", type=int, default=52, help="inference: scenes checked against the CPU oracle (0 = skip)")
    ap.add_argument("--batch", type=int, default=None, help="scenes per GPU per step (default: 32; ae: 64)")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--cpu-batch", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-defer-join", action="store_true", help="A/B: join the overlapped weight exchange inside step()")
    ap.add_argument("--multicast", default="auto", choices=["auto", "on", "off"],
                    help="A/B: NVLink multicast (multimem) vs peer loads in the sharded update; auto = peer loads")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float32 / "
                         "float64, at most 64 MB: larger tensors as a fixed seeded sample), to compare two builds")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.mode == "inference":
        a.config = "inference"
    if a.dump_outputs and (a.impl != "ours" or a.config == "inference"):
        ap.error("--dump-outputs covers the training step of --impl ours (configs roadmap, ae, bb)")
    if a.batch is None:
        a.batch = 64 if a.config == "ae" else (256 if a.config == "inference" else 32)
    return a


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi polled every 20 ms by a reader thread.  start() returns once the first sample has arrived (nvidia-smi
    takes ~1 s to come up, longer than the whole timed region); mark() / stop() bracket the timed region, and only the
    samples taken inside it are reported."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        import threading
        self.proc, self.lines, self.t0 = None, [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, bufsize=1)
        except Exception:  # noqa: BLE001
            self.proc = None
            return

        def reader():
            for line in self.proc.stdout:
                self.lines.append((time.perf_counter(), line))

        self.thread = threading.Thread(target=reader, daemon=True)
        self.thread.start()
        deadline = time.perf_counter() + 10.0
        while not self.lines and time.perf_counter() < deadline:
            time.sleep(0.01)

    def mark(self):
        self.t0 = time.perf_counter()

    def stop(self):
        t1 = time.perf_counter()
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.03)                      # let the sample that covers the end of the region arrive
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        t0 = self.t0 if self.t0 is not None else 0.0
        inside = [l for (t, l) in self.lines if t0 <= t <= t1 + 0.03]
        used = inside if inside else [l for (_, l) in self.lines[-3:]]
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in used:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm_v, mx_v = float(f[0]), float(f[1])
            except ValueError:
                continue
            sm.append(sm_v); mx.append(mx_v)
            try:
                pw.append(float(f[2]))          # "[N/A]" on boxes that do not report power
            except ValueError:
                pass
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "samples_in_timed_region": len(inside),
                "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference path
# ------------------------------------------------------------------------------------------------
def cpu_train_steps(batch: int, steps: int, warmup: int):
    """fwd + BCE + TS + backward + Adam of the reference path on the host cores (torch CPU ops =
    what the reference executes), B=`batch` scenes per step.  Returns (scenes/s, seconds/step)."""
    from oracle import scene_oracle as so
    torch.set_num_threads(os.cpu_count())
    params = so.init_roadmap_params(HIDDEN, LATENT, VIEW_H, VIEW_W)
    views, road = so.synthetic_scene_batch(batch, VIEW_H, VIEW_W)
    names = [k for k, v in params.items() if v.is_floating_point() and "running_" not in k]
    leaves = {k: params[k].clone().requires_grad_(True) for k in names}
    opt = torch.optim.Adam(list(leaves.values()), lr=1e-3)
    p = dict(params)
    p.update(leaves)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        out = so.run_step(p, views, road, training=True, seed=1234 + i)
        out["loss"].backward()
        opt.step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    sec = statistics.median(times)
    return batch / sec, sec


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(0, args.warmup)     # ~0.6 s per B=2 CPU step
    sps, sec = cpu_train_steps(args.cpu_batch, steps, warm)
    cores = os.cpu_count()
    line = {
        "impl": "reference", "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"RoadMapBCE train step, views 6x3x{VIEW_H}x{VIEW_W}, hidden {HIDDEN} latent {LATENT}, "
                               f"map {MAP}x{MAP}; CPU sample = {args.cpu_batch} scenes/step"},
        "cpu_baseline": {"value": sps, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{steps} steps of B={args.cpu_batch} scenes (fwd+BCE+TS+bwd+Adam), torch CPU ops, "
                                   f"{cores} threads"},
        "e2e": {"value": sps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def build_model(dtype: str, device):
    from driving_dirty_b200.synthetic import random_roadmap_model
    model = random_roadmap_model(HIDDEN, LATENT, VIEW_H, VIEW_W, dtype=dtype, device=device)
    model.frozen = False
    model.ae.unfreeze()
    model.train()
    return model


def time_kernel(fn, iters=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e-3


def dominant_kernel_roofline(batch: int, dtype: torch.dtype, pk, pk_src):
    """Times the c2-shaped conv kernels (32->32 3x3 over the 256x1836 mosaic: fwd, dgrad, wgrad) alone on the
    current stream with CUDA events.  Unfused, such a conv moves 128 B per pixel for 18,432 flop (144 flop/B, below
    this box's ridge of 243 flop/B), so the roof that bounds it is HBM: `roofline` reports the slowest of the three
    against the measured copy bandwidth, with ALGORITHMIC bytes per launch (activations in + out; dgrad also reads the
    ReLU mask) -- and the bf16 tensor fractions the north star asks about ride along in `all`."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    dev = torch.device("cuda")
    code = dtype_code(dtype)
    H, W = VIEW_H, 6 * VIEW_W
    x = torch.rand(batch, H, W, 32, device=dev).to(dtype)
    dy = (torch.rand(batch, H, W, 32, device=dev) - 0.5).to(dtype)
    out = torch.empty_like(x)
    w = torch.rand(32, 32, 3, 3, device=dev) * 0.1
    b = torch.zeros(32, device=dev)
    dw, db = torch.empty_like(w), torch.empty_like(b)
    n = int(_lib.load().dd_conv_wgrad_workspace_bytes())
    ws = torch.empty(n, dtype=torch.uint8, device=dev)
    st = stream_ptr()
    act = x.numel() * x.element_size()
    kernels = {
        "conv3x3_c32 fwd (c2)": (lambda: call("dd_conv3x3_c32_fwd", x.data_ptr(), w.data_ptr(), b.data_ptr(),
                                              out.data_ptr(), code, batch, H, W, 1, 0, st), 2 * act),
        "conv3x3_c32 dgrad (c2)": (lambda: call("dd_conv3x3_c32_dgrad", dy.data_ptr(), w.data_ptr(), x.data_ptr(),
                                                out.data_ptr(), code, batch, H, W, 1, 0, st), 3 * act),
        "conv3x3_c32 wgrad (c2)": (lambda: call("dd_conv3x3_c32_wgrad", x.data_ptr(), dy.data_ptr(), dw.data_ptr(),
                                                db.data_ptr(), ws.data_ptr(), n, code, batch, H, W, 1, 0, st), 2 * act),
    }
    traffic = {}
    try:        # dram__bytes_read + dram__bytes_write per launch from the committed ncu --set full capture of these kernels
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            traffic = json.load(f)
    except Exception:  # noqa: BLE001
        pass
    flops = FLOP_C2_PER_SCENE * batch
    rows = []
    for name, (fn, nbytes) in kernels.items():
        t = time_kernel(fn)
        rows.append({"kernel": name, "ms": t * 1e3, "gbs": nbytes / t / 1e9, "hbm_frac": nbytes / t / 1e9 / pk["hbm_gbs"],
                     "algorithmic_bytes_per_launch": nbytes, "tflops": flops / t / 1e12,
                     "tensor_frac": flops / t / 1e12 / pk["bf16_tflops"],
                     "dram_bytes_per_launch_ncu": traffic.get(name) if batch == 32 else None})
    worst = max(rows, key=lambda r: r["ms"])
    roof = {"bound": "hbm", "kernel": worst["kernel"], "achieved": worst["gbs"], "peak": pk["hbm_gbs"], "unit": "GB/s",
            "frac": worst["hbm_frac"], "traffic": worst["dram_bytes_per_launch_ncu"],
            "peak_source": pk_src + " (copy bandwidth; bf16 peak for tensor_frac: burst)",
            "algorithmic_bytes_per_launch": worst["algorithmic_bytes_per_launch"],
            "algorithmic_flops_per_launch": flops, "ms_per_launch": worst["ms"],
            "why_hbm": "unfused 32->32 3x3 conv in bf16 NHWC: 144 flop/B < ridge 243 flop/B", "all": rows}
    del x, dy, out
    torch.cuda.empty_cache()
    return roof


def hbm_kernel_rooflines(batch: int, pk):
    """Stitch and fused BCE/TS kernels against the measured HBM copy bandwidth."""
    from driving_dirty_b200 import ops
    dev = torch.device("cuda")
    views = torch.rand(batch, 6, 3, VIEW_H, VIEW_W, device=dev)
    t = time_kernel(lambda: ops.stitch(views))
    nbytes = 2 * views.numel() * 4
    rows = [{"kernel": "stitch f32", "ms": t * 1e3, "gbs": nbytes / t / 1e9, "frac": nbytes / t / 1e9 / pk["hbm_gbs"]}]
    logits = torch.randn(batch, MAP, MAP, device=dev) * 0.06
    target = (torch.rand(batch, MAP, MAP, device=dev) > 0.5).float()
    t = time_kernel(lambda: ops.bce_threat(logits, target, want_probs=False, want_binary=False))
    nbytes = 2 * logits.numel() * 4
    rows.append({"kernel": "bce+ts fwd (f32 target, sums only)", "ms": t * 1e3, "gbs": nbytes / t / 1e9,
                 "frac": nbytes / t / 1e9 / pk["hbm_gbs"]})
    t = time_kernel(lambda: ops.bce_threat(logits, target, want_probs=True, want_binary=True))
    nbytes = logits.numel() * 13          # logits + target + probs (f32) + binary map (u8)
    rows.append({"kernel": "bce+ts fwd (f32 target) + probs + binary map", "ms": t * 1e3, "gbs": nbytes / t / 1e9,
                 "frac": nbytes / t / 1e9 / pk["hbm_gbs"]})
    return rows


def verify_data_parallel_step(model, opt, step, views, road, world):
    """The N-GPU step checks itself (the sharded reduce + Adam + all-gather kernel runs nowhere else at this width):
    one more step from the current state, then (1) every parameter is bit-identical on all ranks (all-reduce MAX and
    MIN of each tensor), (2) the new head weight equals torch arithmetic for Adam applied to the all-reduced MEAN
    gradient, from the moments and weights saved before the step.  Collective on every rank; outside the timed region."""
    head = model.fc1.weight
    reg = opt._regions.get(id(head))
    if reg is None:
        return None
    st = opt.state[reg["key"]]
    t_before = int(st["step"])
    m0, v0 = opt._full_moments(reg)
    w0 = head.detach().clone().reshape(-1)
    torch.cuda.synchronize()
    dist.barrier()
    step(views, road)
    torch.cuda.synchronize()
    dist.barrier()
    g = head.grad.detach().clone().reshape(-1)          # this rank's gradient replica of the step just taken
    dist.all_reduce(g, op=dist.ReduceOp.SUM)
    g /= world
    lr, b1, b2, eps, wd = opt._hyper()
    tt = t_before + 1
    if wd:
        g = g + wd * w0
    m1 = m0 + (1 - b1) * (g - m0)
    v1 = b2 * v0 + (1 - b2) * g * g
    expect = w0 - (lr / (1 - b1 ** tt)) * (m1 / (v1.sqrt() / (1 - b2 ** tt) ** 0.5 + eps))
    got = head.detach().reshape(-1)
    err_w = float((got - expect).abs().max() / expect.abs().max())
    err_u = float((got - expect).abs().max() / (expect - w0).abs().max().clamp_min(1e-30))
    del m0, v0, m1, v1, g, expect
    worst = 0.0
    for p in model.parameters():
        hi, lo = p.detach().clone(), p.detach().clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        worst = max(worst, float((hi - lo).abs().max()))
        del hi, lo
    res = torch.tensor([worst, err_w, err_u], device=head.device, dtype=torch.float64)
    dist.all_reduce(res, op=dist.ReduceOp.MAX)
    worst, err_w, err_u = (float(x) for x in res)
    return {"replica_max_abs_diff": worst, "vs_single_rank_step_rel_err": err_w, "vs_single_rank_step_err_rel_to_update": err_u,
            "checked": "all parameters equal on all ranks after a step; head weight (81.9 M) vs torch Adam arithmetic on the "
                       "all-reduced mean gradient", "tolerance": 5e-6, "ok": worst == 0.0 and err_w < 5e-6}


# ------------------------------------------------------------------------------------------------
# workloads: BASELINE.json configs 2 (default, the metric's config), 3 and 4
# ------------------------------------------------------------------------------------------------
class Roadmap:
    """config 2: RoadMapBCE train step (roadmap_bce_v2.py:83-133), bf16, hidden 256 / latent 128."""
    key, metric = "roadmap", METRIC

    def __init__(self, args, dev, rank):
        from driving_dirty_b200.synthetic import scene_batch_bytes
        self.model = build_model(args.dtype, dev)
        # raw camera bytes (uint8, what the JPEG decoder yields): ToTensor's /255 (data_helper.py:109-114) is folded into
        # the first conv's loads, bit-identical to feeding bytes.float()/255 (test_raw_byte_front_end_on_the_model_path)
        views, road = scene_batch_bytes(args.batch, VIEW_H, VIEW_W, seed=20200506 + rank)
        self.host = [views.pin_memory(), road.pin_memory()]
        self.host_f32 = [(views.float() / 255).pin_memory(), self.host[1]]   # what the reference's dataloader hands over
        self.describe = (f"RoadMapBCE train step (BASELINE config 2), {args.batch} scenes/GPU/step, views 6x3x{VIEW_H}x{VIEW_W} as raw "
                         f"camera bytes (uint8; /255 folded into conv 1), hidden {HIDDEN} latent {LATENT}, map {MAP}x{MAP}, encoder unfrozen")

    def loss(self, dev_tensors):
        views, road = dev_tensors
        return self.model.training_step((views, None, road), 1)["loss"]


class AutoEncoder:
    """config 3: BasicAE self-supervised pretraining step (autoencoder.py:78-108): stitch + mask one view, encoder,
    decoder (2 dense blocks + 4 transposed convs), MSE."""
    key, metric = "ae", "6-view scenes/sec, BasicAE pretraining step (six-to-one task: fwd + MSE + bwd + Adam)"

    def __init__(self, args, dev, rank):
        from driving_dirty_b200.synthetic import random_ae_model, scene_batch
        self.model = random_ae_model(HIDDEN, LATENT, VIEW_H, VIEW_W, dtype=args.dtype, device=dev)
        self.model.train()
        views, _ = scene_batch(args.batch, VIEW_H, VIEW_W, map_hw=8, seed=20200506 + rank)
        self.host = [views.pin_memory()]
        self.host_f32 = None
        self.describe = (f"BasicAE train step (BASELINE config 3), {args.batch} scenes/GPU/step, views 6x3x{VIEW_H}x{VIEW_W} fp32, "
                         f"hidden {HIDDEN} latent {LATENT}, decoder to 3x{VIEW_H}x{VIEW_W}")

    def loss(self, dev_tensors):
        return self.model.training_step(dev_tensors[0], 1)["loss"]


class BoundingBox:
    """config 4: BBSpatialRoadMap step (spatial_w_rm.py:67-133): six strip convs + encoder convs (c3_only) + merging CNN
    (four dilated transposed convs to 400x400, k2 s2 to 800x800), probability-space BCE.  The box targets are rasterised
    ahead of time (the reference rasterises with PIL inside _run_step, :85-95: host work, not part of the device path)."""
    key, metric = "bb", "6-view scenes/sec, BBSpatialRoadMap train step (fwd + BCE + bwd + Adam)"

    def __init__(self, args, dev, rank):
        import numpy as np
        from driving_dirty_b200.synthetic import box_batch, random_bb_model, scene_batch
        from driving_dirty_b200.utils.bb_to_img import boxes_to_binary_map
        self.model = random_bb_model(HIDDEN, LATENT, dtype=args.dtype, device=dev)
        self.model.frozen = False
        self.model.ae.unfreeze()
        self.model.train()
        views, road = scene_batch(args.batch, VIEW_H, VIEW_W, seed=20200506 + rank)
        raster = torch.from_numpy(np.stack([boxes_to_binary_map(b).copy() for b in box_batch(args.batch, 20200507 + rank)])).float()
        self.host = [views.pin_memory(), road.pin_memory(), raster.pin_memory()]
        self.host_f32 = None
        self.describe = (f"BBSpatialRoadMap train step (BASELINE config 4), {args.batch} scenes/GPU/step, views 6x3x{VIEW_H}x{VIEW_W} fp32, "
                         f"road map + box raster {MAP}x{MAP}, hidden {HIDDEN} latent {LATENT}, encoder unfrozen")

    def loss(self, dev_tensors):
        views, road, raster = dev_tensors
        return self.model.training_step((views, raster, road), 1)["loss"]


WORKLOADS = {w.key: w for w in (Roadmap, AutoEncoder, BoundingBox)}

FLOP_CONVS_PER_SCENE = 11.641e9       # c1 + c2 + c3 forward (SURVEY 8(d))


def run_inference(args):
    """BASELINE config 5: ModelLoader.get_binary_road_map, batch sweep 1..256, bf16 tensor-core path and fp32 parity path,
    device-resident and end to end (pinned host bytes in, binary maps out); replicas only, no collective.  Parity on rank
    0 against the CPU oracle (oracle/scene_oracle.py, the reference's torch arithmetic) with identical dropout masks:
    flipped pixels in ppm, the largest |reference logit| among the flipped ones, and the rounded threat score in
    <= 26-scene chunks (the reference's fp32 sums are exact up to 26 scenes, SURVEY H5) against our integer counts."""
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from driving_dirty_b200 import _lib
    from driving_dirty_b200.model_loader import ModelLoader
    from driving_dirty_b200.synthetic import random_roadmap_model, scene_batch_bytes
    m16 = random_roadmap_model(HIDDEN, LATENT, VIEW_H, VIEW_W, dtype="bf16", device=dev)
    sd = {k: v.detach().clone() for k, v in m16.state_dict().items()}
    m32 = random_roadmap_model(HIDDEN, LATENT, VIEW_H, VIEW_W, dtype="fp32", device=dev, state_dict=sd)
    loaders = {"bf16": ModelLoader(m16, device=dev), "fp32": ModelLoader(m32, device=dev)}
    bmax = args.batch if args.batch else 256
    views_h, road_h = scene_batch_bytes(bmax, VIEW_H, VIEW_W, seed=20200506 + rank)
    views_h = views_h.pin_memory()
    views_d = views_h.to(dev)
    sizes = [b for b in (1, 2, 4, 8, 16, 32, 64, 128, 256) if b <= bmax]
    sampler = ClockSampler(local) if rank == 0 else None
    sweep, l0 = [], _lib.launch_count()
    if sampler:
        sampler.mark()
    for name, loader in loaders.items():
        for b in sizes:
            if name == "fp32" and b > 64:
                continue                                  # the fp32 SIMT parity path is not the throughput path
            iters = args.steps
            row = {"dtype": name, "batch": b}
            out_h = torch.empty(b, MAP, MAP, dtype=torch.uint8).pin_memory()
            for mode, src in (("resident", views_d[:b]), ("e2e", views_h[:b])):
                for _ in range(3):
                    out = loader.get_binary_road_map(src, as_bytes=(mode == "e2e"))
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    out = loader.get_binary_road_map(src, as_bytes=(mode == "e2e"))
                    if mode == "e2e":
                        out_h.copy_(out, non_blocking=False)   # the binary maps (bytes) back on the host, every call
                e1.record()
                torch.cuda.synchronize()
                sec = e0.elapsed_time(e1) * 1e-3 / iters
                row[mode + "_scenes_s"] = b / sec
                row[mode + "_ms"] = sec * 1e3
            sweep.append(row)
    clocks = sampler.stop() if sampler else None
    launches = _lib.launch_count() - l0
    best = max((r for r in sweep if r["dtype"] == "bf16"), key=lambda r: r["resident_scenes_s"])
    t = torch.tensor([best["resident_scenes_s"], max(r["e2e_scenes_s"] for r in sweep if r["dtype"] == "bf16")], device=dev,
                     dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)        # replicas only: the job's throughput is the sum over ranks
    if rank == 0:
        pk, pk_src = peaks()
        parity = inference_parity(loaders, sd, min(bmax, args.parity_scenes)) if args.parity_scenes > 0 else None
        line = {
            "metric": "6-view scenes/sec, ModelLoader.get_binary_road_map (inference)", "value": float(t[0]), "unit": UNIT,
            "n_gpus": world, "steps": args.steps, "warmup": 3, "ms_per_step": best["resident_ms"], "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": f"ModelLoader.get_binary_road_map (BASELINE config 5), batch sweep {sizes}, views 6x3x{VIEW_H}x{VIEW_W} raw "
                                   f"camera bytes, hidden {HIDDEN} latent {LATENT}, map {MAP}x{MAP}; value = best batch ({best['batch']}), "
                                   f"replicas only (sum over ranks); CUDA graph up to batch {loaders['bf16'].graph_max_batch}",
                       "batch_per_gpu": best["batch"], "parallelism": f"replicas x{world}",
                       "l2": "activations of the best batch exceed the 126 MB L2; small batches are L2 resident by nature"},
            "e2e": {"value": float(t[1]), "unit": UNIT, "h2d_bytes_per_step": best["batch"] * 6 * 3 * VIEW_H * VIEW_W,
                    "d2h_bytes_per_step": best["batch"] * MAP * MAP,
                    "note": "pinned host camera bytes copied in by ModelLoader every call, the uint8 binary maps copied back to pinned host memory"},
            "gpu_launches": int(launches), "clocks": clocks, "sweep": sweep,
            "conv_stack": {"tflops_at_best_batch": FLOP_CONVS_PER_SCENE * best["resident_scenes_s"] / 1e12,
                           "frac_of_bf16_peak": FLOP_CONVS_PER_SCENE * best["resident_scenes_s"] / 1e12 / pk["bf16_tflops"],
                           "peak_source": pk_src, "note": "c1+c2+c3 forward flops over the WHOLE call's time (convs, pool, FC, head, sigmoid)"},
            "parity_vs_oracle": parity,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def inference_parity(loaders, state_dict, n):
    """Binary maps of both paths against the oracle on n scenes with identical (CPU-generator) dropout masks."""
    from oracle import scene_oracle as so
    from tests.helpers import cpu_rng_dropout
    torch.set_num_threads(os.cpu_count())
    views, road = so.synthetic_scene_batch(n, VIEW_H, VIEW_W, seed=20200601)
    params = {k: v.detach().cpu() for k, v in state_dict.items()}
    res = {"scenes": n, "chunk": 26}
    ref_logits, ref_bin = [], []
    chunks = [(lo, min(lo + 26, n)) for lo in range(0, n, 26)]
    t0 = time.perf_counter()
    with torch.no_grad():
        for lo, hi in chunks:
            torch.manual_seed(4242 + lo)
            out = so.run_step(params, views[lo:hi], road[lo:hi], training=False)
            ref_logits.append(out["logits"])
            ref_bin.append(out["probs"].round())
    res["oracle_seconds"] = time.perf_counter() - t0
    for name, loader in loaders.items():
        old = loader.graph_max_batch
        loader.graph_max_batch = 0                        # the CPU-generator dropout patch cannot be graph-captured
        flips, worst, ts_err, ts_pairs = 0, 0.0, 0.0, []
        with cpu_rng_dropout(), torch.no_grad():
            for (lo, hi), rl, rb in zip(chunks, ref_logits, ref_bin):
                torch.manual_seed(4242 + lo)
                got = loader.get_binary_road_map(views[lo:hi].to(loader.device)).cpu()
                diff = got != rb
                flips += int(diff.sum())
                if diff.any():
                    worst = max(worst, float(rl[diff].abs().max()))
                t = road[lo:hi].float()
                tp, nt, nr = so.threat_score_counts(t, got)
                ours = tp / (nt + nr - tp)
                ref_ts = float(so.threat_score(t, rb))    # the reference's fp32 sums, exact for <= 26 scenes
                ts_pairs.append([ours, ref_ts])
                ts_err = max(ts_err, abs(ours - ref_ts))
        loader.graph_max_batch = old
        res[name] = {"flipped_ppm": flips / (n * MAP * MAP) * 1e6, "flipped_pixels": flips,
                     "max_abs_reference_logit_among_flipped": worst, "ts_rounded_max_abs_err_per_chunk": ts_err,
                     "ts_rounded_ours_vs_reference_first_chunk": ts_pairs[0]}
    res["min_abs_reference_logit"] = float(min(float(l.abs().min()) for l in ref_logits))
    res["note"] = ("random-init weights put the logits at ~N(0, 0.06^2), crowded around the threshold: the fp32 path may flip only "
                   "pixels whose reference logit is within ~1e-6 of it; the bf16 path flips those within bf16 rounding of the activations")
    return res


DUMP_MAX_BYTES = 64 << 20
DUMP_SAMPLE = 1 << 20          # elements written of a tensor larger than this


def step_outputs(model, loss):
    """What one training step hands its caller: the loss, the model state it leaves behind (parameters after the optimizer
    step, BatchNorm statistics) and, where the model keeps them (RoadMapBCE), the step's threat scores and binary map."""
    out = {"loss": loss}
    out.update(("state." + k, v) for k, v in model.state_dict().items())
    out.update(("metrics." + k, v) for k, v in (getattr(model, "last_metrics", None) or {}).items())
    return out


def dump_outputs(tensors, path):
    """Each tensor as <path>/<name>.npy: float32, or float64 for 64-bit floats and integers (exact counts).  A tensor of
    more than DUMP_SAMPLE elements is written flat as its elements at DUMP_SAMPLE indices drawn with a fixed seed, so two
    runs, or two builds, write the same positions."""
    import numpy as np
    arrays = {}
    for name, t in tensors.items():
        t = t.detach()
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        wide = t.dtype in (torch.float64, torch.int64, torch.int32)
        arrays[name] = t.to(torch.float64 if wide else torch.float32).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise SystemExit(f"bench.py: --dump-outputs would write {total} bytes (limit {DUMP_MAX_BYTES})")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from driving_dirty_b200 import _lib
    from driving_dirty_b200.optim import FusedAdam

    B = args.batch
    wl = WORKLOADS[args.config](args, dev, rank)
    model = wl.model
    params = [p for p in model.parameters() if p.requires_grad]
    # world 1: one fused launch per tensor; world N: the wide FC weights are reduced, updated and all-gathered by ONE kernel
    # over NVLink peer memory (optim.FusedAdam / csrc/adam.cu), launched from the backward pass; the small tensors share
    # one flat sharded bucket
    opt = FusedAdam(params, lr=1e-3, overlap_backward=True, defer_join=not args.no_defer_join,
                    multicast={"auto": None, "on": True, "off": False}[args.multicast])
    resident = [t.to(dev, non_blocking=True) for t in wl.host]

    def step(tensors):
        opt.zero_grad(set_to_none=True)
        loss = wl.loss(tensors)
        loss.backward()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing -------------------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None      # up and polling before the GPU work starts
    # >= 5 untimed steps: the first ones map the symmetric / multicast buffers and size the allocator's pools
    for _ in range(max(args.warmup, 5)):
        step(resident)
    barrier()
    if sampler:
        sampler.mark()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host = time.perf_counter()
    for _ in range(args.steps):
        loss = step(resident)
    opt.synchronize()        # the last step's weight exchange may still be running on the optimizer's side stream: time it too
    e1.record()
    host_ms = (time.perf_counter() - t_host) * 1e3 / args.steps      # host time to ENQUEUE a step (no device sync inside)
    barrier()
    launches = _lib.launch_count() - l0
    sec = e0.elapsed_time(e1) * 1e-3
    clocks = sampler.stop() if sampler else None
    final_loss = float(loss.detach())
    if args.dump_outputs and rank == 0:      # now: the end-to-end steps below train the model further
        dump_outputs(step_outputs(model, loss), args.dump_outputs)

    # ---- end to end: host buffers in, loss out, every step -------------------------------------
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    loss_h = torch.empty((), dtype=torch.float32).pin_memory()

    def e2e_time(host):
        bufs = [[torch.empty(t.shape, dtype=t.dtype, device=dev) for t in host] for _ in range(2)]

        def prefetch(i):
            with torch.cuda.stream(copy_stream):
                for d, h in zip(bufs[i], host):
                    d.copy_(h, non_blocking=True)
                ready[i].record(copy_stream)

        def e2e_loop(k):
            prefetch(0)
            for i in range(k):
                cur = i & 1
                torch.cuda.current_stream().wait_event(ready[cur])
                if i + 1 < k:
                    copy_stream.wait_stream(torch.cuda.current_stream())   # buffer (i+1)&1 was consumed by step i-1
                    prefetch((i + 1) & 1)
                l = step(bufs[cur])
                loss_h.copy_(l.detach(), non_blocking=False)               # D2H read of the step's result

        e2e_loop(2)
        barrier()
        e0.record()
        e2e_loop(args.steps)
        opt.synchronize()
        e1.record()
        barrier()
        return e0.elapsed_time(e1) * 1e-3

    sec_e2e = e2e_time(wl.host)
    sec_e2e_f32 = e2e_time(wl.host_f32) if wl.host_f32 is not None else 0.0

    t = torch.tensor([sec, sec_e2e, sec_e2e_f32], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec, sec_e2e, sec_e2e_f32 = float(t[0]), float(t[1]), float(t[2])
    verify = None
    if world > 1 and args.config == "roadmap":
        verify = verify_data_parallel_step(model, opt, lambda v, r: step([v, r]), resident[0], resident[1], world)
        if verify is not None and not verify["ok"]:
            raise SystemExit(f"bench.py: the data-parallel step failed its self-check: {json.dumps(verify)}")

    if rank == 0:
        pk, pk_src = peaks()
        adt = torch.bfloat16 if args.dtype == "bf16" else torch.float32
        torch.cuda.empty_cache()
        roof, hbm_rows, cpu = None, None, None
        if args.config == "roadmap":
            roof = dominant_kernel_roofline(B, adt, pk, pk_src)
            hbm_rows = hbm_kernel_rooflines(B, pk)
            if world == 1 and not args.no_cpu_baseline:
                sps, csec = cpu_train_steps(args.cpu_batch, 3, 1)
                cpu = {"value": sps, "unit": UNIT, "cores": os.cpu_count(), "kind": "port",
                       "sample": f"3 steps of B={args.cpu_batch} scenes (fwd+BCE+TS+bwd+Adam) through oracle/scene_oracle.py "
                                 f"(torch CPU ops: the arithmetic the reference executes; not the imported reference, which "
                                 f"does not travel to the GPU box), {os.cpu_count()} threads, {csec:.2f} s/step"}
        total = B * world * args.steps
        h2d = sum(t.numel() * t.element_size() for t in wl.host)
        line = {
            "metric": wl.metric, "value": total / sec, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 5), "ms_per_step": sec / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": args.dtype, "data": "synthetic",
            "config": {"workload": wl.describe + ", Adam (dd_adam_step" + (", sharded over NVLink peer memory" + (" + multicast" if opt.uses_multicast else "") if world > 1 else "") + ")",
                       "batch_per_gpu": B, "global_batch": B * world, "parallelism": f"dp{world}",
                       "l2": "activations (GBs per layer) and the FC weights exceed the 126 MB L2 many times over; no explicit flush"},
            "e2e": {"value": total / sec_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": sec_e2e / args.steps * 1e3,
                    "note": "pinned host inputs copied every step on a side stream (double-buffered), loss read back"},
            "gpu_launches": int(launches), "host_enqueue_ms_per_step": host_ms, "clocks": clocks, "roofline": roof, "hbm_kernels": hbm_rows,
            "cpu_baseline": cpu, "final_loss": final_loss,
        }
        if wl.host_f32 is not None:
            line["e2e_f32_views"] = {"value": total / sec_e2e_f32, "unit": UNIT,
                                     "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in wl.host_f32),
                                     "d2h_bytes_per_step": 4, "ms_per_step": sec_e2e_f32 / args.steps * 1e3,
                                     "note": "the same with fp32 host views (what the reference's ToTensor dataloader emits): 4x the view bytes"}
        if verify is not None:
            line["dp_self_check"] = verify
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.config == "inference":
        run_inference(a)
    else:
        run_ours(a)
