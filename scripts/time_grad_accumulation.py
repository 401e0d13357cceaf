"""Gradient accumulation over micro-batches (optim.FusedAdam(accumulate_grad_batches=k)), timed on the GPU.

kernel: the last backward pass of a window on the two wide FC layers of the RoadMapBCE step at the bench shapes (B = 32):
        dd_linear_bwd_adam_acc against the three launches it replaces (dd_linear_dgrad + dd_linear_wgrad_acc +
        dd_adam_step).  CUDA events over ITERS launches per form, the forms alternating, ROUNDS rounds; the W / m / v / G
        arrays (0.96 GB for fc1, 0.33 GB for the head) are far larger than L2.  Outputs of one window compared bit for bit.
step:   the RoadMapBCE bf16 training step of bench.py (32-scene micro-batches, world size 1, overlap_backward=True) in
        windows of k in {1, 2, 4} micro-batches (loss / k, then step() and zero_grad()), the k alternating, ROUNDS rounds.
The card's name and power limit are read in the same run."""
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from driving_dirty_b200 import _lib  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402

ITERS, ROUNDS, WINDOWS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 3)), int(os.environ.get("WINDOWS", 8))
SHAPES = {"fc1": (32, 256, 940032, torch.bfloat16), "head": (32, 640000, 128, torch.float32)}   # B, N, K, dx dtype
LR, B1, B2, EPS, WD = 1e-3, 0.9, 0.999, 1e-8, 0.0


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def kernels():
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    for name, (B, N, K, dxt) in SHAPES.items():
        esz = torch.finfo(dxt).bits // 8
        x = torch.randn(B, K, device=dev, generator=g)
        dy = torch.randn(B, N, device=dev, generator=g) * 1e-3
        w0 = torch.randn(N, K, device=dev, generator=g) * 0.01
        m0 = torch.randn(N, K, device=dev, generator=g) * 1e-4
        v0 = torch.rand(N, K, device=dev, generator=g) * 1e-6
        g0 = torch.randn(N, K, device=dev, generator=g) * 1e-3        # the window's earlier passes
        n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
        ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
        forms = {f: dict(w=w0.clone(), m=m0.clone(), v=v0.clone(), G=g0.clone(), dx=torch.empty(B, K, dtype=dxt, device=dev),
                         db=torch.empty(N, device=dev), step=0) for f in ("unfused", "fused")}
        del w0, m0, v0, g0

        def run(form):
            s = forms[form]
            s["step"] += 1
            code = _lib.dtype_code(dxt)
            if form == "fused":
                call("dd_linear_bwd_adam_acc", dy.data_ptr(), x.data_ptr(), s["w"].data_ptr(), s["m"].data_ptr(),
                     s["v"].data_ptr(), s["G"].data_ptr(), s["dx"].data_ptr(), code, s["db"].data_ptr(), ws.data_ptr(), n_ws,
                     B, N, K, LR, B1, B2, EPS, WD, s["step"], stream_ptr())
            else:
                call("dd_linear_dgrad", dy.data_ptr(), s["w"].data_ptr(), s["dx"].data_ptr(), code, ws.data_ptr(), n_ws, B, N, K,
                     _lib.IMPL_TCGEN05, stream_ptr())
                call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), _lib.DD_F32, s["G"].data_ptr(), s["db"].data_ptr(),
                     B, N, K, _lib.IMPL_TCGEN05, 1, stream_ptr())
                call("dd_adam_step", s["w"].data_ptr(), s["G"].data_ptr(), s["m"].data_ptr(), s["v"].data_ptr(), N * K, LR, B1,
                     B2, EPS, WD, s["step"], 1.0, stream_ptr())

        run("unfused"); run("fused")
        torch.cuda.synchronize()
        same = {k: torch.equal(forms["unfused"][k], forms["fused"][k]) for k in ("dx", "db", "w", "m", "v")}
        print(f"{name}: B {B} N {N} K {K} dx {str(dxt).split('.')[-1]}; outputs of one last pass bit-identical: "
              + ", ".join(f"{k} {'yes' if v else 'NO'}" for k, v in same.items()), flush=True)
        # fused: W, m, v read + written (24 B), G read (4 B); unfused: dgrad reads W (4), wgrad_acc reads + writes G (8),
        # Adam reads W, G, m, v and writes W, m, v (28) = 40 B per parameter; plus x, dy, dx, db
        small = 4 * B * K + 4 * B * N + esz * B * K + 4 * N
        nbytes = {"unfused": 40 * N * K + small + 4 * B * N, "fused": 28 * N * K + small + 4 * B * N}
        times = {"unfused": [], "fused": []}
        for form in ("unfused", "fused"):
            for _ in range(3):
                run(form)
        for _ in range(ROUNDS):
            for form in ("unfused", "fused"):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(ITERS):
                    run(form)
                e1.record()
                torch.cuda.synchronize()
                times[form].append(e0.elapsed_time(e1) / ITERS)
        for form in ("unfused", "fused"):
            t = min(times[form])
            print(f"  {form:8s} {t:.3f} ms (rounds: {', '.join(f'{x:.3f}' for x in times[form])})  "
                  f"{nbytes[form] / 1e9:.2f} GB algorithmic -> {nbytes[form] / t * 1e-9:.2f} TB/s", flush=True)
        print(f"  saving {min(times['unfused']) - min(times['fused']):.3f} ms per window", flush=True)
        del forms
        torch.cuda.empty_cache()


def steps():
    import bench
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    wl = bench.Roadmap(SimpleNamespace(dtype="bf16", batch=32), dev, 0)
    params = [p for p in wl.model.parameters() if p.requires_grad]
    opt = FusedAdam(params, lr=1e-3, overlap_backward=True)
    resident = [t.to(dev, non_blocking=True) for t in wl.host]

    def window(k):
        opt.accumulate_grad_batches = k
        for _ in range(k):
            (wl.loss(resident) / k).backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    ks = (1, 2, 4)
    for k in ks:
        for _ in range(3):
            window(k)
    torch.cuda.synchronize()
    times = {k: [] for k in ks}
    for _ in range(ROUNDS):
        for k in ks:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(max(1, WINDOWS // k)):
                window(k)
            opt.synchronize()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1) / max(1, WINDOWS // k))
    print(f"step: {wl.describe}; world size 1, overlap_backward=True", flush=True)
    for k in ks:
        t = sorted(times[k])
        print(f"  k = {k}: {t[len(t) // 2]:.2f} ms per window, {t[len(t) // 2] / k:.2f} ms per 32-scene micro-batch "
              f"(windows: {', '.join(f'{x:.2f}' for x in times[k])} ms)", flush=True)


if __name__ == "__main__":
    print(f"GPU: {gpu_info()}", flush=True)
    what = sys.argv[1:] or ["kernels", "steps"]
    if "kernels" in what:
        kernels()
    if "steps" in what:
        steps()
