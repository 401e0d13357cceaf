"""Gradient norms in optim.FusedAdam (track_grad_norm), timed on the GPU.  Off and on alternate within one run, ROUNDS rounds
each; the spread is the list of rounds.

kernel: dd_linear_bwd_adam against dd_linear_bwd_adam_sumsq (the same launch plus the fp64 sum of squares) at RoadMapBCE's
        two wide shapes (the head fc1 and the encoder fc1), B = 32, CUDA events over ITERS launches.
step:   the RoadMapBCE bf16 training step of bench.py (32-scene batches, world size 1, overlap_backward=True): tracking off,
        against tracking on with grad_norms() read on every step (every step a logging step).
N = 2:  with two GPUs, the sharded step with tracking on: a logging step (grad_norms() before step(), which waits for the
        side stream's overlapped updates) against a non-logging one; skipped with one GPU.
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

ITERS, ROUNDS, STEPS = int(os.environ.get("ITERS", 20)), int(os.environ.get("ROUNDS", 5)), int(os.environ.get("STEPS", 10))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    return q or torch.cuda.get_device_name()


def roadmap(batch=32):
    import bench
    return bench.Roadmap(SimpleNamespace(dtype="bf16", batch=batch), torch.device("cuda"), 0)


def _spread(ts):
    t = sorted(ts)
    return f"median {t[len(t) // 2]:.3f} ms (rounds: {', '.join(f'{x:.3f}' for x in ts)})"


def kernel(name, N, K, B=32):
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(2)
    x = torch.randn(B, K, device=dev, generator=g)
    dy = torch.randn(B, N, device=dev, generator=g)
    w = torch.randn(N, K, device=dev, generator=g) * 0.05
    m, v = torch.zeros_like(w), torch.zeros_like(w)
    dx = torch.empty(B, K, device=dev, dtype=torch.bfloat16)
    db = torch.empty(N, device=dev)
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    sws = torch.zeros(int(_lib.load().dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
    out = torch.empty(1, dtype=torch.float64, device=dev)
    head = (dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr())
    tail = (dx.data_ptr(), _lib.DD_BF16, db.data_ptr(), ws.data_ptr(), n_ws, B, N, K, 1e-4, 0.9, 0.999, 1e-8, 0.0, 1)

    def run(norm):
        if norm:
            call("dd_linear_bwd_adam_sumsq", *head, None, *tail, out.data_ptr(), sws.data_ptr(), sws.numel(), stream_ptr())
        else:
            call("dd_linear_bwd_adam", *head, *tail, stream_ptr())

    for norm in (False, True):
        for _ in range(3):
            run(norm)
    times = {False: [], True: []}
    for _ in range(ROUNDS):
        for norm in (False, True):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(ITERS):
                run(norm)
            e1.record()
            torch.cuda.synchronize()
            times[norm].append(e0.elapsed_time(e1) / ITERS)
    nbytes = 24 * N * K
    print(f"kernel {name} [{N} x {K}], B = {B} ({nbytes / 1e9:.2f} GB of W, m, v read and written):", flush=True)
    for norm, label in ((False, "dd_linear_bwd_adam      "), (True, "dd_linear_bwd_adam_sumsq")):
        t = sorted(times[norm])[ROUNDS // 2]
        print(f"  {label} {_spread(times[norm])} -> {nbytes / (t * 1e-3) * 1e-9:.0f} GB/s", flush=True)


def steps(wl):
    from driving_dirty_b200.optim import FusedAdam
    params = [p for p in wl.model.parameters() if p.requires_grad]
    opt = FusedAdam(params, lr=1e-3, overlap_backward=True)
    resident = [t.to("cuda", non_blocking=True) for t in wl.host]
    forms = {"tracking off": -1, "tracking on, grad_norms() every step": 2}

    def step(form):
        opt.track_grad_norm = forms[form]
        wl.loss(resident).backward()
        if forms[form] == 2:
            opt.grad_norms()
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
    print(f"step: {wl.describe}; world size 1, overlap_backward=True; {STEPS} steps per round", flush=True)
    for form in forms:
        print(f"  {form:38s} {_spread(times[form])}", flush=True)
    opt.track_grad_norm = 2
    wl.loss(resident).backward()
    got = opt.grad_norms()
    print(f"  total gradient norm of the last step: {float(got['total']):.6e} over {len(got) - 1} tensors", flush=True)


def _n2_worker(rank, world, port, q):
    import torch.distributed as dist
    from driving_dirty_b200.optim import FusedAdam
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        wl = roadmap()
        params = [p for p in wl.model.parameters() if p.requires_grad]
        opt = FusedAdam(params, lr=1e-3, overlap_backward=True, track_grad_norm=2)
        resident = [t.to("cuda", non_blocking=True) for t in wl.host]
        forms = ("non-logging step", "logging step (grad_norms() before step())")

        def step(form):
            wl.loss(resident).backward()
            if form == forms[1]:
                opt.grad_norms()
            opt.step()
            opt.zero_grad(set_to_none=True)

        for form in forms:
            for _ in range(3):
                step(form)
        torch.cuda.synchronize()
        times = {f: [] for f in forms}
        for _ in range(ROUNDS):
            for form in forms:
                dist.barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(STEPS):
                    step(form)
                opt.synchronize()
                e1.record()
                torch.cuda.synchronize()
                times[form].append(e0.elapsed_time(e1) / STEPS)
        if rank == 0:
            q.put([f"N = 2 (rank 0): {wl.describe}; overlap_backward=True, tracking on"] +
                  [f"  {form:42s} {_spread(times[form])}" for form in forms])
    finally:
        dist.destroy_process_group()


def n2():
    if torch.cuda.device_count() < 2:
        print("N = 2: not measured (one GPU visible)", flush=True)
        return
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_n2_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    lines = q.get(timeout=900)
    for p in procs:
        p.join(timeout=120)
    print("\n".join(lines), flush=True)


if __name__ == "__main__":
    print(f"GPU: {gpu_info()}; {torch.cuda.device_count()} visible", flush=True)
    wl = roadmap()
    shapes = {"head fc1.weight": tuple(wl.model.fc1.weight.shape),
              "encoder ae.encoder.fc1.fc1.weight": tuple(wl.model.ae.encoder.fc1.fc1.weight.shape)}
    for name, (N, K) in shapes.items():
        kernel(name, N, K)
    steps(wl)
    del wl
    torch.cuda.empty_cache()
    n2()
