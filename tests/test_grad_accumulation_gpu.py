"""Gradient accumulation over micro-batches on the wide linear layers: dd_linear_wgrad_acc against dd_linear_wgrad plus the
old gradient, dd_linear_bwd_adam_acc against the three unfused launches it replaces, and optim.FusedAdam with
accumulate_grad_batches = k against the same call sequence through autograd -- bit for bit -- and, on two GPUs, the
sharded form against torch.optim.Adam."""
import os

import pytest
import torch

from tests.helpers import build_roadmap_pair, cpu_rng_dropout
from tests.test_linear_bwd_adam_gpu import SENTINEL, _bands_intact, _guarded, _state_dicts_equal


@pytest.mark.gpu
@pytest.mark.parametrize("impl_name", ["SIMT", "TCGEN05"])
@pytest.mark.parametrize("B", [8, 32, 40, 64, 96])
@pytest.mark.parametrize("N,K", [(4100, 1028), (36, 131076)])     # ragged n and k tiles
@pytest.mark.parametrize("x_dtype", [torch.float32, torch.bfloat16])
def test_wgrad_acc_is_old_plus_wgrad(impl_name, B, N, K, x_dtype):
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    impl = getattr(_lib, "IMPL_" + impl_name)
    if impl == _lib.IMPL_TCGEN05 and x_dtype != torch.float32:
        pytest.skip("the tensor-core path reads fp32 x")
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(B + N)
    x = torch.randn(B, K, generator=g).to(dev, x_dtype)
    dy = torch.randn(B, N, generator=g).to(dev)
    old = torch.randn(N, K, generator=g).to(dev)
    d = torch.empty(N, K, device=dev)
    db_ref = torch.empty(N, device=dev)
    call("dd_linear_wgrad", dy.data_ptr(), x.data_ptr(), dtype_code(x_dtype), d.data_ptr(), db_ref.data_ptr(), B, N, K,
         impl, stream_ptr())
    buf, acc = _guarded(old)
    db = torch.full((N,), SENTINEL, device=dev)
    call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), dtype_code(x_dtype), acc.data_ptr(), db.data_ptr(), B, N, K,
         impl, 1, stream_ptr())
    torch.cuda.synchronize()
    assert _bands_intact(buf)
    assert torch.equal(acc, old + d), float((acc - (old + d)).abs().max())
    assert torch.equal(db, db_ref)                                # the bias gradient is overwritten
    # accumulate = 0 is dd_linear_wgrad
    call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), dtype_code(x_dtype), acc.data_ptr(), None, B, N, K, impl, 0,
         stream_ptr())
    torch.cuda.synchronize()
    assert torch.equal(acc, d)


def _run_window(fused, B, N, K, dx_dtype, windows=3, k=2, seed=4):
    """`windows` windows of k passes: the last pass of each either dd_linear_bwd_adam_acc, or dd_linear_dgrad +
    dd_linear_wgrad_acc + dd_adam_step; passes 1 .. k-1 dd_linear_dgrad + dd_linear_wgrad_acc."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(seed)
    wbuf, w = _guarded((torch.randn(N, K, generator=g) * 0.05).to(dev))
    mbuf, m = _guarded(torch.zeros(N, K, device=dev))
    vbuf, v = _guarded(torch.zeros(N, K, device=dev))
    gbuf, G = _guarded(torch.zeros(N, K, device=dev))
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    lr, b1, b2, eps, wd = 1e-2, 0.9, 0.999, 1e-8, 0.01
    out = []
    for t in range(1, windows + 1):
        for j in range(k):
            x = torch.randn(B, K, generator=g).to(dev)
            dy = torch.randn(B, N, generator=g).to(dev)
            db = torch.empty(N, device=dev)
            dxbuf, dx = _guarded(torch.zeros(B, K, dtype=dx_dtype or torch.float32, device=dev))
            dxp = dx.data_ptr() if dx_dtype is not None else None
            code = dtype_code(dx_dtype) if dx_dtype is not None else _lib.DD_F32
            if fused and j == k - 1:
                call("dd_linear_bwd_adam_acc", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(),
                     G.data_ptr(), dxp, code, db.data_ptr(), ws.data_ptr(), n_ws, B, N, K, lr, b1, b2, eps, wd, t,
                     stream_ptr())
            else:
                if dxp is not None:
                    call("dd_linear_dgrad", dy.data_ptr(), w.data_ptr(), dxp, code, ws.data_ptr(), n_ws, B, N, K,
                         _lib.IMPL_TCGEN05, stream_ptr())
                call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), _lib.DD_F32, G.data_ptr(), db.data_ptr(), B, N, K,
                     _lib.IMPL_TCGEN05, int(j > 0), stream_ptr())
                if j == k - 1:
                    call("dd_adam_step", w.data_ptr(), G.data_ptr(), m.data_ptr(), v.data_ptr(), N * K, lr, b1, b2, eps, wd,
                         t, 1.0, stream_ptr())
            torch.cuda.synchronize()
            assert _bands_intact(dxbuf)
            out.append((dx.clone() if dx_dtype is not None else None, db.clone()))
    assert all(_bands_intact(b) for b in (wbuf, mbuf, vbuf, gbuf))
    return w.clone(), m.clone(), v.clone(), out


@pytest.mark.gpu
@pytest.mark.parametrize("B,N,K,dx_dtype", [
    (32, 64, 65540, torch.float32),        # fc1-like: small N, long K (ragged last k tile), no split
    (32, 68, 65536, torch.bfloat16),       # ragged last n chunk, bf16 input gradient
    (32, 33000, 128, torch.float32),       # head-like: long N (ragged), K = 128, split input gradient
    (20, 32004, 132, torch.bfloat16),      # ragged K, split, B < 32
    (32, 64, 65540, None),                 # no input gradient
    (32, 33000, 128, None),
])
def test_bwd_adam_acc_matches_unfused_launches(B, N, K, dx_dtype):
    ref = _run_window(False, B, N, K, dx_dtype)
    got = _run_window(True, B, N, K, dx_dtype)
    for name, a, c in zip(("weight", "exp_avg", "exp_avg_sq"), ref[:3], got[:3]):
        assert torch.equal(a, c), (name, float((a - c).abs().max()))
    for (dx_r, db_r), (dx_g, db_g) in zip(ref[3], got[3]):
        assert torch.equal(db_r, db_g)
        if dx_dtype is not None:
            assert torch.equal(dx_r, dx_g), float((dx_r.float() - dx_g.float()).abs().max())


@pytest.mark.gpu
def test_bwd_adam_acc_rejects_what_it_cannot_run():
    from driving_dirty_b200._lib import call, last_error
    dev = torch.device("cuda")
    t = torch.zeros(64 * 65536 + 4, device=dev)
    p = t.data_ptr()
    args = lambda B, K, gp=p, w=p: (p, p, w, p, p, gp, None, 0, None, None, 0, B, 64, K, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1,  # noqa: E731
                                    None)
    with pytest.raises(RuntimeError, match="dd_status -1"):      # no partial gradient
        call("dd_linear_bwd_adam_acc", *args(32, 65536, gp=None))
    with pytest.raises(RuntimeError, match="dd_status -1"):      # B > 32
        call("dd_linear_bwd_adam_acc", *args(33, 65536))
    with pytest.raises(RuntimeError, match="dd_status -2"):      # too narrow for the tensor-core path
        call("dd_linear_bwd_adam_acc", *args(32, 1024))
    with pytest.raises(RuntimeError, match="dd_status -4"):      # misaligned partial gradient
        call("dd_linear_bwd_adam_acc", *args(32, 65536, gp=p + 4))
    assert "grad_partial" in last_error()
    with pytest.raises(RuntimeError, match="dd_status -2"):      # accumulating more than 128 rows
        call("dd_linear_wgrad_acc", p, p, 0, p, None, 129, 64, 1024, 1, 1, None)


def _linear_windows(overlap, B, k, plan):
    """FusedAdam(accumulate_grad_batches=k) on one wide tensor-core linear layer; plan = passes per window."""
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(9)
    N, K = 4096, 1028
    w = torch.nn.Parameter((torch.randn(N, K, generator=g) * 0.05).to(dev))
    b = torch.nn.Parameter((torch.randn(N, generator=g) * 0.05).to(dev))
    opt = FusedAdam([w, b], lr=1e-2, weight_decay=0.01, overlap_backward=overlap, accumulate_grad_batches=k)
    grads = []
    for passes in plan:
        opt.zero_grad()
        for _ in range(passes):
            x = torch.randn(B, K, generator=g).to(dev).requires_grad_(True)
            gy = torch.randn(B, N, generator=g).to(dev) / k
            ops.linear(x, w, b, impl=_lib.IMPL_TCGEN05).backward(gy)
            grads.append((w.grad is None, x.grad.clone()))
        opt.step()
    return w.detach().clone(), b.detach().clone(), opt.state_dict(), grads


@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 40])
@pytest.mark.parametrize("k,plan", [(2, [2, 2, 1]), (3, [3, 2, 3])])     # a partial window: step after j < k passes
def test_fused_adam_accumulation_world_one(B, k, plan):
    """overlap_backward=True with a window of k passes gives the results of overlap_backward=False (autograd adds the
    gradients): weights, x.grad and the optimizer state, bit for bit.  B = 32: the last pass of a full window steps inside
    the backward pass (no gradient tensor); B = 40: the window adds up in the gradient buffer and step() steps from it."""
    ref, got = _linear_windows(False, B, k, plan), _linear_windows(True, B, k, plan)
    assert all(not none for none, _ in ref[3])
    assert all(none for none, _ in got[3])                      # the wide weight never shows a gradient tensor
    for (_, a), (_, c) in zip(ref[3], got[3]):
        assert torch.equal(a, c)
    assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
    _state_dicts_equal(ref[2], got[2])


@pytest.mark.gpu
def test_fused_adam_accumulation_refuses_pass_k_plus_one():
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    w = torch.nn.Parameter(torch.randn(4096, 1028, device=dev) * 0.05)
    opt = FusedAdam([w], lr=1e-2, overlap_backward=True, accumulate_grad_batches=2)
    x = torch.randn(32, 1028, device=dev)
    for _ in range(2):
        ops.linear(x, w, impl=_lib.IMPL_TCGEN05).sum().backward()
    with pytest.raises(RuntimeError, match="accumulate_grad_batches=2"):
        ops.linear(x, w, impl=_lib.IMPL_TCGEN05).sum().backward()
    opt.step()
    ops.linear(x, w, impl=_lib.IMPL_TCGEN05).sum().backward()    # a new window


@pytest.mark.gpu
def test_fused_adam_k1_launches_unchanged():
    """accumulate_grad_batches = 1: a backward pass launches exactly what dd_linear_bwd_adam launches for it (the fused
    kernel, its split fold and the bias column sum), as before the flag existed."""
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200._lib import call, stream_ptr
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    N, K, B = 4096, 1028, 32
    w = torch.nn.Parameter(torch.randn(N, K, device=dev) * 0.05)
    b = torch.nn.Parameter(torch.zeros(N, device=dev))
    FusedAdam([w, b], lr=1e-2, overlap_backward=True)
    x = torch.randn(B, K, device=dev, requires_grad=True)
    y = ops.linear(x, w, b, impl=_lib.IMPL_TCGEN05)
    gy = torch.randn_like(y)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    y.backward(gy)
    torch.cuda.synchronize()
    n_backward = _lib.launch_count() - n0
    assert w.grad is None
    m, v, dx, db = torch.zeros_like(w), torch.zeros_like(w), torch.empty_like(x), torch.empty_like(b)
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    n0 = _lib.launch_count()
    call("dd_linear_bwd_adam", gy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(), dx.data_ptr(),
         _lib.DD_F32, db.data_ptr(), ws.data_ptr(), n_ws, B, N, K, 1e-2, 0.9, 0.999, 1e-8, 0.0, 1, stream_ptr())
    assert n_backward == _lib.launch_count() - n0


@pytest.mark.gpu
def test_roadmap_accumulated_windows_with_the_update_in_backward():
    """RoadMapBCE on the bf16 tensor-core path, two windows of k = 2 micro-batches in a Lightning-style loop (loss / k):
    model and optimizer state as with the update in step() and autograd's accumulation."""
    from driving_dirty_b200.optim import FusedAdam
    k = 2
    res = []
    for overlap in (False, True):
        model, _, views, road = build_roadmap_pair(batch=4, hidden=16, latent=8, view_h=16, view_w=20, dtype="bf16",
                                                   device="cuda:0")
        model.frozen = False
        model.ae.unfreeze()
        opt = FusedAdam([p for p in model.parameters() if p.requires_grad], lr=1e-3, overlap_backward=overlap,
                        accumulate_grad_batches=k)
        batch = (tuple(views.cuda().unbind(0)), None, tuple(road.cuda().unbind(0)))
        head = model.fc1.weight
        for i in range(2 * k):
            with cpu_rng_dropout():
                torch.manual_seed(7 + i)
                loss = model._run_step(batch, 1, "train")[0]
                (loss / k).backward()
            assert (head.grad is None) == overlap
            if i % k == k - 1:
                opt.step()
                opt.zero_grad()
        torch.cuda.synchronize()
        res.append(({kk: v.detach().clone() for kk, v in model.state_dict().items()}, opt.state_dict()))
    (sd0, o0), (sd1, o1) = res
    assert sd0.keys() == sd1.keys()
    for kk in sd0:
        assert torch.equal(sd0[kk], sd1[kk]), kk
    _state_dicts_equal(o0, o1)


@pytest.mark.gpu
def test_make_adam_passes_the_factor():
    from types import SimpleNamespace
    from driving_dirty_b200.optim import FusedAdam, make_adam
    model = torch.nn.Linear(8, 4).cuda()
    model.hparams = SimpleNamespace(accumulate_grad_batches={0: 1, 3: 4})
    model.current_epoch = 5
    opt = make_adam(model, 1e-3)
    assert isinstance(opt, FusedAdam) and opt._factor() == 4


# ------------------------------------------------------------------------------------------------
# two GPUs: the sharded form with k = 2 (fp32 CUDA-core kernels, B = 40: two 32-row chunks per accumulating pass)
# ------------------------------------------------------------------------------------------------
def _sharded_worker(rank, world, port, overlap, out):
    import torch.distributed as dist
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    from tests.test_optim import _reference_adam
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        k, windows, N, K, B = 2, 2, 2048, 1024, 40
        g = torch.Generator().manual_seed(12)
        w0, b0 = torch.randn(N, K, generator=g) * 0.05, torch.randn(N, generator=g) * 0.05
        xs = [[[torch.randn(B, K, generator=g) for _ in range(world)] for _ in range(k)] for _ in range(windows)]
        gys = [[[torch.randn(B, N, generator=g) / k for _ in range(world)] for _ in range(k)] for _ in range(windows)]
        w = torch.nn.Parameter(w0.clone().to(dev))
        b = torch.nn.Parameter(b0.clone().to(dev))
        opt = FusedAdam([w, b], lr=1e-2, overlap_backward=overlap, accumulate_grad_batches=k)
        for t in range(windows):
            opt.zero_grad()
            for j in range(k):
                ops.linear(xs[t][j][rank].to(dev), w, b, impl=_lib.IMPL_SIMT).backward(gys[t][j][rank].to(dev))
            opt.step()
        opt.synchronize()
        torch.cuda.synchronize()
        # reference: Adam on the rank mean of the per-rank window sums
        steps = []
        for t in range(windows):
            gw = sum(sum(gys[t][j][r].t() @ xs[t][j][r] for j in range(k)) for r in range(world)) / world
            gb = sum(sum(gys[t][j][r].sum(0) for j in range(k)) for r in range(world)) / world
            steps.append([gw, gb])
        ref = _reference_adam([w0, b0], steps, lr=1e-2)
        ew = float((w.detach().cpu() - ref[0]).abs().max() / ref[0].abs().max())
        eb = float((b.detach().cpu() - ref[1]).abs().max() / ref[1].abs().max())
        gathered = [torch.empty_like(w.data) for _ in range(world)]
        dist.all_gather(gathered, w.data.contiguous())
        same = all(torch.equal(gathered[0], x) for x in gathered)
        if rank == 0:
            with open(out, "w") as f:
                f.write(f"{ew} {eb} {int(same)}")
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
def test_fused_adam_sharded_accumulation_two_gpus(tmp_path, overlap):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from tests.test_optim import _free_port
    out = str(tmp_path / "res.txt")
    mp.spawn(_sharded_worker, args=(2, _free_port(), overlap, out), nprocs=2, join=True)
    ew, eb, same = open(out).read().split()
    assert float(ew) < 5e-6 and float(eb) < 5e-6 and same == "1", (ew, eb, same)
