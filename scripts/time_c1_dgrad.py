"""The image gradient of the encoder's first conv (dd_conv_c1_dgrad) at the bench shape (B = 32 scenes, 256 x 1836 mosaic,
bf16 da1): the tensor-core kernel writing the views layout and the mosaic layout, the CUDA-core kernel, and the same
gradient through the existing generic conv engine (dd_conv2d_dgrad, Cin = 3) plus the layout passes it needs
(dd_nhwc_to_nchw_f32, dd_unstitch_f32).  CUDA events over ITERS launches per form, the forms alternating, ROUNDS rounds,
min over rounds; algorithmic bytes (da1 read once, dx written once) and GB/s against a torch copy measured in the same run.
da1 alone is 963 MB, far beyond the 126 MB L2, so no cache flush is needed between launches.  The forms' outputs are
compared.  Then the launch count of a bf16 RoadMapBCE training step without / with views that require grad, and the wall
time of a frozen-model attribution pass (RoadMapBCE, B = 32, bf16: forward + backward to the views)."""
import ctypes
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from driving_dirty_b200 import _lib  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402

ITERS, ROUNDS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 3))
B, H, W = 32, 256, 306
BF, F32 = _lib.DD_BF16, _lib.DD_F32


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm",
                        "--format=csv"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def event_ms(fn, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernels():
    dev = torch.device("cuda")
    Wm, st = 6 * W, stream_ptr()
    g = torch.Generator(device=dev).manual_seed(1)
    da1 = (torch.randn(B, H, Wm, 32, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    w1 = (torch.rand(32, 3, 3, 3, device=dev, generator=g) - 0.5) * 0.4
    views = lambda: torch.empty(B, 6, 3, H, W, device=dev)  # noqa: E731
    dx_tc, dx_tcm, dx_simt, dx_gen = views(), torch.empty(B, 3, H, Wm, device=dev), views(), views()
    desc = _lib.ConvDesc(B, 3, 32, H, Wm, H, Wm, 3, 3, 1, 1, 1, 1, 1, 1, 0)
    nws = int(_lib.load().dd_conv2d_workspace_bytes(ctypes.byref(desc)))
    ws = torch.empty(max(nws, 256), dtype=torch.uint8, device=dev)
    gen_nhwc = torch.empty(B, H, Wm, 3, dtype=torch.bfloat16, device=dev)
    gen_nchw = torch.empty(B, 3, H, Wm, device=dev)
    p = lambda t: t.data_ptr()  # noqa: E731

    def generic():
        call("dd_conv2d_dgrad", p(da1), p(w1), None, p(gen_nhwc), ctypes.byref(desc), BF, p(ws), nws, st)
        call("dd_nhwc_to_nchw_f32", p(gen_nhwc), BF, p(gen_nchw), B, 3, H, Wm, st)
        call("dd_unstitch_f32", p(gen_nchw), None, p(dx_gen), B, H, W, -1, st)

    forms = {
        "tensor cores, views layout": lambda: call("dd_conv_c1_dgrad", p(da1), BF, p(w1), p(dx_tc), 1, B, H, Wm, 2, st),
        "tensor cores, mosaic layout": lambda: call("dd_conv_c1_dgrad", p(da1), BF, p(w1), p(dx_tcm), 0, B, H, Wm, 2, st),
        "CUDA cores, views layout": lambda: call("dd_conv_c1_dgrad", p(da1), BF, p(w1), p(dx_simt), 1, B, H, Wm, 1, st),
        "generic engine + layout passes": generic,
    }
    for f in forms.values():
        f()
    torch.cuda.synchronize()
    ref = dx_simt.double()
    scale = float(ref.abs().max())
    unst = torch.empty_like(dx_tc)
    unst[:, [0, 1, 2, 5, 4, 3]] = dx_tcm.reshape(B, 3, H, 6, W).permute(0, 3, 1, 2, 4)
    print(f"views layout == unstitched mosaic layout (tensor cores): {'yes' if torch.equal(unst, dx_tc) else 'NO'}")
    print(f"max |difference| / max |dx| against the CUDA-core kernel (fp32 weights): tensor cores (bf16 weights) "
          f"{float((dx_tc.double() - ref).abs().max()) / scale:.1e}, generic engine (bf16 output) "
          f"{float((dx_gen.double() - ref).abs().max()) / scale:.1e}")

    src = torch.empty(1 << 30, dtype=torch.uint8, device=dev)
    dst = torch.empty_like(src)
    for _ in range(3):
        dst.copy_(src)
    copy_ms = min(event_ms(lambda: dst.copy_(src), ITERS) for _ in range(ROUNDS))
    roof = 2 * src.numel() / copy_ms * 1e-6
    print(f"copy bandwidth (torch copy of 1 GiB, read + write): {roof:.0f} GB/s")
    del src, dst

    nbytes = da1.numel() * 2 + dx_tc.numel() * 4
    print(f"B {B}, mosaic {H} x {Wm}; algorithmic bytes {nbytes / 1e9:.3f} GB (da1 bf16 read + dx fp32 written), "
          f"{2 * B * H * Wm * 32 * 3 * 9 / 1e9:.1f} GFLOP; {ITERS} launches per timing, {ROUNDS} rounds, forms alternating")
    times = {k: [] for k in forms}
    for _ in range(ROUNDS):
        for k, f in forms.items():
            times[k].append(event_ms(f, ITERS))
    for k in forms:
        t = min(times[k])
        print(f"  {k:31s} {t:.3f} ms (rounds {', '.join(f'{x:.3f}' for x in times[k])})  "
              f"{nbytes / t * 1e-6:.0f} GB/s = {nbytes / t * 1e-6 / roof:.0%} of copy")


def step_launches():
    from driving_dirty_b200.synthetic import random_roadmap_model, scene_batch
    model = random_roadmap_model(hidden=16, latent=8, view_h=16, view_w=20, map_size=800)
    model.frozen = False
    model.ae.unfreeze()
    views, road = scene_batch(3, 16, 20)
    counts = {}
    for req in (False, True):
        v = views.cuda().requires_grad_(req)
        n0 = _lib.launch_count()
        out = model.training_step((v, None, tuple(road.cuda().unbind(0))), 1)
        out["loss"].backward()
        torch.cuda.synchronize()
        counts[req] = _lib.launch_count() - n0
    print(f"library launches of a bf16 RoadMapBCE training step + backward: {counts[False]} without views.grad, "
          f"{counts[True]} with")


def attribution():
    from driving_dirty_b200.synthetic import random_roadmap_model, scene_batch
    model = random_roadmap_model(dtype="bf16")
    for q in model.parameters():
        q.requires_grad_(False)
    views, road = scene_batch(B)
    views, road = views.cuda(), road.cuda()

    def one():
        v = views.detach().requires_grad_()
        loss = model._run_step((v, None, road), 1, "train")[0]
        loss.backward()
        return v.grad

    for _ in range(3):
        one()
    torch.cuda.synchronize()
    ts = []
    for _ in range(ROUNDS):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(10):
            one()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) / 10 * 1e3)
    print(f"frozen-model attribution pass, RoadMapBCE B {B} bf16 fp32 views (forward + BCE + backward to the views): "
          f"{min(ts):.2f} ms (rounds {', '.join(f'{x:.2f}' for x in ts)}), peak memory "
          f"{torch.cuda.max_memory_allocated() / 2**30:.2f} GiB")


def main():
    print(f"GPU (nvidia-smi, same run):\n{gpu_info()}")
    kernels()
    step_launches()
    torch.cuda.reset_peak_memory_stats()
    attribution()


if __name__ == "__main__":
    main()
