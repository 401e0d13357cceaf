"""The box model's training target, host raster against device raster, at the bench batch (32 scenes of
synthetic.box_batch):
  (a) utils/bb_to_img.boxes_to_binary_map per scene (Pillow, wall clock) against ops.boxes_to_map (host boxes in, device
      raster out, synchronised, wall clock), and dd_boxes_to_map alone on device inputs (CUDA events), with its output
      GB/s;
  (b) the config-4 training step (BBSpatialRoadMap, B = 32, bf16, FusedAdam as in bench.py) fed the dataloader's
      tuple-of-dicts target: once rasterised on the host (boxes_to_binary_map, tensor passed to the step) and once
      through the device rasteriser (dicts passed), alternating, in scenes/s;
  (c) the card's name, power limit and SM clock, read in the same run.
The two rasters are compared bit for bit."""
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from driving_dirty_b200 import ops  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402
from driving_dirty_b200.synthetic import box_batch, random_bb_model, scene_batch  # noqa: E402
from driving_dirty_b200.utils.bb_to_img import boxes_to_binary_map  # noqa: E402

B = int(os.environ.get("BATCH", 32))
KERNEL_ITERS = int(os.environ.get("KERNEL_ITERS", 200))
HOST_REPS = int(os.environ.get("HOST_REPS", 6))
STEPS, ROUNDS = int(os.environ.get("STEPS", 10)), int(os.environ.get("ROUNDS", 3))
MAP = 800


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                        "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def host_raster(boxes):
    return torch.from_numpy(np.stack([boxes_to_binary_map(b).copy() for b in boxes])).float()


def main():
    dev = torch.device("cuda", torch.cuda.current_device())
    print(f"GPU (name, power limit, SM clock, max SM clock): {gpu_info()}")
    boxes = box_batch(B, 20200507)
    n_boxes = sum(int(b.shape[0]) for b in boxes)
    out_bytes = B * MAP * MAP * 4
    print(f"batch: {B} scenes, {n_boxes} boxes (synthetic.box_batch), raster {B}x{MAP}x{MAP} fp32 = {out_bytes / 1e6:.1f} MB")

    # ---- (a) host path, end-to-end device path, kernel alone ---------------------------------------------------------
    ref = host_raster(boxes)
    dev_map = ops.boxes_to_map(boxes, dev)
    torch.cuda.synchronize()
    print(f"device raster equals host raster bit for bit: {torch.equal(dev_map.cpu(), ref)}")
    host_ms = []
    for _ in range(HOST_REPS):
        t = time.perf_counter()
        host_raster(boxes)
        host_ms.append((time.perf_counter() - t) * 1e3)
    e2e_ms = []
    for _ in range(HOST_REPS * 5):
        torch.cuda.synchronize()
        t = time.perf_counter()
        ops.boxes_to_map(boxes, dev)
        torch.cuda.synchronize()
        e2e_ms.append((time.perf_counter() - t) * 1e3)
    print(f"(a) host bb_to_img, {B} scenes: median {statistics.median(host_ms):.1f} ms "
          f"(min {min(host_ms):.1f}, max {max(host_ms):.1f}, {HOST_REPS} calls)")
    print(f"(a) ops.boxes_to_map, host boxes in, device raster out, synchronised: median {statistics.median(e2e_ms):.3f} ms "
          f"(min {min(e2e_ms):.3f}, max {max(e2e_ms):.3f}, {len(e2e_ms)} calls)")

    flat = torch.cat([b.reshape(-1, 8) for b in boxes]).to(dev)
    offsets = torch.tensor([0] + np.cumsum([b.shape[0] for b in boxes]).tolist(), dtype=torch.int32, device=dev)
    out = torch.empty(B, MAP, MAP, device=dev)
    st = stream_ptr()
    for _ in range(10):
        call("dd_boxes_to_map", flat.data_ptr(), 0, offsets.data_ptr(), B, out.data_ptr(), st)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(KERNEL_ITERS):
        call("dd_boxes_to_map", flat.data_ptr(), 0, offsets.data_ptr(), B, out.data_ptr(), st)
    e1.record()
    torch.cuda.synchronize()
    k_us = e0.elapsed_time(e1) * 1e3 / KERNEL_ITERS
    print(f"(a) box_raster_kernel alone (CUDA events, {KERNEL_ITERS} back-to-back launches, same output buffer): "
          f"{k_us:.2f} us, {out_bytes / (k_us * 1e-6) / 1e9:.0f} GB/s of output written")
    assert torch.equal(out.cpu(), ref)

    # ---- (b) config-4 training step, host raster vs device raster ---------------------------------------------------
    from driving_dirty_b200.optim import FusedAdam
    model = random_bb_model(256, 128, dtype="bf16", device=dev)
    model.frozen = False
    model.ae.unfreeze()
    model.train()
    params = [p for p in model.parameters() if p.requires_grad]
    opt = FusedAdam(params, lr=1e-3, overlap_backward=True)
    views, road = scene_batch(B, 256, 306, seed=20200506)
    views, road = views.to(dev), road.to(dev)
    dicts = tuple({"bounding_box": b} for b in boxes)

    def step(form):
        target = host_raster(boxes) if form == "host" else dicts
        opt.zero_grad(set_to_none=True)
        loss = model.training_step((views, target, road), 1)["loss"]
        loss.backward()
        opt.step()

    def timed(form):
        opt.synchronize()
        torch.cuda.synchronize()
        t = time.perf_counter()
        for _ in range(STEPS):
            step(form)
        opt.synchronize()
        torch.cuda.synchronize()
        return (time.perf_counter() - t) / STEPS

    for form in ("host", "device"):
        for _ in range(3):
            step(form)
    rates = {"host": [], "device": []}
    for r in range(ROUNDS):
        for form in (("host", "device") if r % 2 == 0 else ("device", "host")):
            rates[form].append(B / timed(form))
    for form in ("host", "device"):
        v = rates[form]
        print(f"(b) config-4 step, B={B} bf16, {form} raster: median {statistics.median(v):.0f} scenes/s "
              f"({', '.join(f'{x:.0f}' for x in v)}; {ROUNDS} rounds of {STEPS} steps, alternating, wall clock to a sync)")
    print(f"GPU after the run: {gpu_info()}")


if __name__ == "__main__":
    main()
