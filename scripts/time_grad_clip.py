"""Gradient clipping in optim.FusedAdam (gradient_clip_val), timed on the GPU.

sumsq: dd_grad_sumsq alone over gradients of the shapes of RoadMapBCE's trainable parameters (1.29 GB, far larger than L2),
       CUDA events over ITERS calls, ROUNDS rounds; bytes read over time against the read-only rate of
       profiles/r2_hbm_rw_probe.txt.
step:  the RoadMapBCE bf16 training step of bench.py (32-scene batches, world size 1, overlap_backward=True) in three forms
       that alternate within one run: no clipping (the wide weights step inside the backward pass), clipping inactive
       (a threshold far above the norm) and clipping active (a threshold far below it).  Both clipping forms take the
       unfused path: weight gradients written, then dd_grad_sumsq and one dd_adam_step_clipped per tensor.
The card's name and power limit are read in the same run."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from driving_dirty_b200 import _lib  # noqa: E402
from driving_dirty_b200._lib import call, stream_ptr  # noqa: E402

ITERS, ROUNDS, STEPS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 3)), int(os.environ.get("STEPS", 10))
HBM_READ_GBS = 6993.4            # profiles/r2_hbm_rw_probe.txt, best read-only grid


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def roadmap():
    import bench
    wl = bench.Roadmap(SimpleNamespace(dtype="bf16", batch=32), torch.device("cuda"), 0)
    return wl, [p for p in wl.model.parameters() if p.requires_grad]


def sumsq(params):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    grads = [torch.randn(p.shape, device=dev, generator=g) * 1e-3 for p in params]
    n = len(grads)
    nbytes = 4 * sum(t.numel() for t in grads)
    ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in grads])
    lens = (ctypes.c_longlong * n)(*[t.numel() for t in grads])
    ws = torch.zeros(int(_lib.load().dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
    out = torch.empty(4, device=dev)

    def run():
        call("dd_grad_sumsq", ptrs, lens, n, 1.0, out.data_ptr(), ws.data_ptr(), ws.numel(), stream_ptr())

    for _ in range(3):
        run()
    ref = torch.nn.utils.get_total_norm(grads)
    torch.cuda.synchronize()
    times = []
    for _ in range(ROUNDS):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(ITERS):
            run()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) / ITERS)
    t = min(times)
    print(f"dd_grad_sumsq: {n} tensors, {nbytes / 1e9:.3f} GB; norm {float(out[0]):.6e} (torch.nn.utils.get_total_norm "
          f"{float(ref):.6e})", flush=True)
    gbs = nbytes / (t * 1e-3) * 1e-9
    print(f"  {t:.3f} ms (rounds: {', '.join(f'{x:.3f}' for x in times)}) -> {gbs:.0f} GB/s, "
          f"{100 * gbs / HBM_READ_GBS:.0f} % of the {HBM_READ_GBS:.0f} GB/s read-only probe rate", flush=True)
    del grads
    torch.cuda.empty_cache()


def steps(wl, params):
    from driving_dirty_b200.optim import FusedAdam
    opt = FusedAdam(params, lr=1e-3, overlap_backward=True)
    resident = [t.to("cuda", non_blocking=True) for t in wl.host]
    forms = {"no clipping": 0.0, "clipping inactive": 1e30, "clipping active": 1e-6}

    def step(form):
        opt.gradient_clip_val = forms[form]
        wl.loss(resident).backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    for form in forms:
        for _ in range(3):
            step(form)
    torch.cuda.synchronize()
    times = {f: [] for f in forms}
    for _ in range(ROUNDS):
        for form in forms:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(STEPS):
                step(form)
            e1.record()
            torch.cuda.synchronize()
            times[form].append(e0.elapsed_time(e1) / STEPS)
    print(f"step: {wl.describe}; world size 1, overlap_backward=True", flush=True)
    for form in forms:
        t = sorted(times[form])
        print(f"  {form:18s} {t[len(t) // 2]:.2f} ms per step (rounds: {', '.join(f'{x:.2f}' for x in times[form])})",
              flush=True)
    opt.gradient_clip_val = 1e-6
    wl.loss(resident).backward()
    opt.step()
    print(f"  clipping active: last_grad_norm {float(opt.last_grad_norm):.4e}", flush=True)


if __name__ == "__main__":
    print(f"GPU: {gpu_info()}; {torch.cuda.device_count()} visible", flush=True)
    wl, params = roadmap()
    sumsq(params)
    steps(wl, params)
