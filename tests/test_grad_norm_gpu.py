"""Gradient norms (FusedAdam's track_grad_norm, Lightning's grad_norm) on the GPU: the fused backward + Adam kernel's sum of
squares against an fp64 sum of the gradient the unfused kernels write, bit-identical updates with tracking on and off,
dd_grad_sumsq_each against float64, FusedAdam's grad_norms() in the fused, stored-gradient and clipping forms, the modules'
grad_norm(), and on two GPUs the rank mean's norms, the same bits on both ranks."""
import os

import pytest
import torch

from tests.helpers import build_roadmap_pair, cpu_rng_dropout
from tests.test_grad_clip_gpu import _ragged


def _rel(a, b):
    a, b = float(a), float(b)
    return abs(a - b) / max(abs(b), 1e-30)


# ------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------
def _bwd_adam(N, K, B, acc, sumsq, seed=3):
    """One fused backward + Adam launch (plain or accumulating) from seeded inputs; with sumsq the _sumsq entry point."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, K, generator=g).to(dev)
    dy = torch.randn(B, N, generator=g).to(dev)
    w = (torch.randn(N, K, generator=g) * 0.05).to(dev)
    m = (torch.randn(N, K, generator=g) * 0.01).to(dev)
    v = torch.rand(N, K, generator=g).to(dev) * 1e-3
    G = torch.randn(N, K, generator=g).to(dev) if acc else None
    dx = torch.empty(B, K, device=dev)
    db = torch.empty(N, device=dev)
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    hyper = (1e-2, 0.9, 0.999, 1e-8, 0.01, 3)
    common = (dx.data_ptr(), _lib.DD_F32, db.data_ptr(), ws.data_ptr(), n_ws, B, N, K, *hyper)
    out = torch.full((1,), -1.0, dtype=torch.float64, device=dev)
    if sumsq:
        sws = torch.zeros(int(_lib.load().dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
        call("dd_linear_bwd_adam_sumsq", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(),
             G.data_ptr() if acc else None, *common, out.data_ptr(), sws.data_ptr(), sws.numel(), stream_ptr())
    elif acc:
        call("dd_linear_bwd_adam_acc", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(), G.data_ptr(),
             *common, stream_ptr())
    else:
        call("dd_linear_bwd_adam", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(), *common,
             stream_ptr())
    # the gradient the step applied, from the unfused weight-gradient kernel (bit for bit the fused kernel's)
    d = torch.empty(N, K, device=dev)
    call("dd_linear_wgrad", dy.data_ptr(), x.data_ptr(), _lib.DD_F32, d.data_ptr(), None, B, N, K, _lib.IMPL_TCGEN05,
         stream_ptr())
    torch.cuda.synchronize()
    applied = d + G if acc else d
    return (w, m, v, dx, db), out, applied


@pytest.mark.gpu
@pytest.mark.parametrize("acc", [False, True])
@pytest.mark.parametrize("N,K", [(4096, 1028), (4100, 1028), (1036, 4100)])    # ragged n chunks and k tiles
@pytest.mark.parametrize("B", [7, 32])
def test_bwd_adam_sumsq_kernel(acc, N, K, B):
    ref, _, applied = _bwd_adam(N, K, B, acc, sumsq=False)
    got, out, _ = _bwd_adam(N, K, B, acc, sumsq=True)
    for a, b in zip(ref, got):                                     # W, m, v, dx, db: the same bits
        assert torch.equal(a, b)
    want = float((applied.double() ** 2).sum())
    assert _rel(out, want) < 1e-6, (float(out), want)
    _, out2, _ = _bwd_adam(N, K, B, acc, sumsq=True)
    assert torch.equal(out, out2)                                  # deterministic


@pytest.mark.gpu
@pytest.mark.parametrize("N,K,where", [(4100, 1028, "x"), (1036, 4100, "dy")])
def test_bwd_adam_sumsq_counts_no_padding(N, K, where):
    """Tile padding is masked, not assumed zero: an infinite x element makes its real gradient column infinite, and the
    padded rows of a ragged N would hold 0 * inf = NaN (an infinite dy element does the same to the padded columns of a
    ragged K).  The sum must be +inf, the sum over the real elements, not NaN."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(4)
    B = 8
    x = torch.randn(B, K, generator=g).to(dev)
    dy = torch.randn(B, N, generator=g).to(dev)
    (x if where == "x" else dy)[3, 5] = float("inf")
    w, m, v = torch.zeros(N, K, device=dev), torch.zeros(N, K, device=dev), torch.zeros(N, K, device=dev)
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    sws = torch.zeros(int(_lib.load().dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
    out = torch.zeros(1, dtype=torch.float64, device=dev)
    call("dd_linear_bwd_adam_sumsq", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(), None, None,
         _lib.DD_F32, None, ws.data_ptr(), n_ws, B, N, K, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, out.data_ptr(), sws.data_ptr(),
         sws.numel(), stream_ptr())
    torch.cuda.synchronize()
    assert float(out) == float("inf"), float(out)


@pytest.mark.gpu
@pytest.mark.parametrize("count", [1, 6, 70])                      # 70: two launches
def test_grad_sumsq_each_ragged(count):
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, stream_ptr
    import ctypes
    _, ts = _ragged(count, count=count)
    outs = torch.full((count,), -1.0, dtype=torch.float64, device="cuda")
    ws = torch.zeros(int(_lib.load().dd_grad_sumsq_each_workspace_bytes()), dtype=torch.uint8, device="cuda")
    res = []
    for _ in range(2):
        call("dd_grad_sumsq_each", (ctypes.c_void_p * count)(*[t.data_ptr() for t in ts]),
             (ctypes.c_longlong * count)(*[t.numel() for t in ts]),
             (ctypes.c_void_p * count)(*[outs[i].data_ptr() for i in range(count)]), count, ws.data_ptr(), ws.numel(),
             stream_ptr())
        res.append(outs.clone())
    torch.cuda.synchronize()
    assert torch.equal(res[0], res[1])
    for t, o in zip(ts, res[0].tolist()):
        want = float((t.double() ** 2).sum())
        assert (o == 0.0 and want == 0.0) or _rel(o, want) < 1e-12, (o, want)


# ------------------------------------------------------------------------------------------------
# FusedAdam: fused forms, stored gradients, clipping
# ------------------------------------------------------------------------------------------------
SHAPES = [(4096, 1028), (4100, 1036)]          # a wide layer and a ragged one (N % 32, K % 128 != 0)


def _run(overlap, k, track, clip=None, windows=2, B=32, seed=5, sync_check=False):
    """Two wide tensor-core layers (+ bias, + a small tensor) trained `windows` windows of k passes; returns the final
    tensors, optimizer state, the x gradients, and per window (norms, fp64 norms of the stored gradients)."""
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(seed)
    ws_ = [torch.nn.Parameter((torch.randn(n, kk, generator=g) * 0.05).to(dev)) for n, kk in SHAPES]
    bs = [torch.nn.Parameter((torch.randn(n, generator=g) * 0.05).to(dev)) for n, _ in SHAPES]
    s = torch.nn.Parameter(torch.randn(37, generator=g).to(dev))
    params = ws_ + bs + [s]
    extra = {"gradient_clip_val": clip} if clip else {}
    opt = FusedAdam(params, lr=1e-2, weight_decay=0.01, overlap_backward=overlap, accumulate_grad_batches=k,
                    track_grad_norm=2 if track else -1, **extra)
    norms, stored, xgrads = [], [], []
    for t in range(windows):
        opt.zero_grad()
        for j in range(k):
            loss = 0
            for (n, kk), w, b in zip(SHAPES, ws_, bs):
                x = torch.randn(B, kk, generator=g).to(dev).requires_grad_(True)
                gy = torch.randn(B, n, generator=g).to(dev)
                y = ops.linear(x, w, b, impl=_lib.IMPL_TCGEN05)
                loss = loss + (y * gy).sum() / k
                xgrads.append(x)
            loss = loss + (s * s).sum() / k
            if sync_check:
                torch.cuda.set_sync_debug_mode("error")
            try:
                loss.backward()
                if track:
                    got = opt.grad_norms() if j == k - 1 else None
            finally:
                torch.cuda.set_sync_debug_mode(0)
        stored.append({id(p): float(torch.linalg.vector_norm(p.grad.double())) for p in params if p.grad is not None})
        if sync_check:
            torch.cuda.set_sync_debug_mode("error")
        try:
            opt.step()
            after = opt.grad_norms() if track else None
        finally:
            torch.cuda.set_sync_debug_mode(0)
        if track:
            norms.append(({id(p): v.clone() for p, v in got.items() if not isinstance(p, str)}, got["total"].clone(),
                          {id(p): v.clone() for p, v in after.items() if not isinstance(p, str)}))
    torch.cuda.synchronize()
    xg = [x.grad.clone() for x in xgrads]
    return params, [p.detach().clone() for p in params], opt.state_dict(), xg, norms, stored, opt


def _same_state(a, b):
    for i in a["state"]:
        for key in ("exp_avg", "exp_avg_sq"):
            assert torch.equal(a["state"][i][key], b["state"][i][key]), (i, key)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 3])
def test_fused_forms_norms_and_bit_identity(k):
    """overlap_backward=True: tracking leaves W, m, v, dx and db bit-identical; every norm and the total are within 1e-6
    of fp64 norms of the gradient the unfused path stores (overlap_backward=False, autograd accumulation); before and
    after step() the same; two runs give the same bits."""
    p_off, t_off, s_off, xg_off, _, _, _ = _run(True, k, track=False)
    params, t_on, s_on, xg_on, norms, _, _ = _run(True, k, track=True)
    for a, b in zip(t_off, t_on):
        assert torch.equal(a, b)
    _same_state(s_off, s_on)
    for a, b in zip(xg_off, xg_on):
        assert torch.equal(a, b)
    ref_params, _, _, _, _, stored, _ = _run(False, k, track=False)
    for (before, total, after), want in zip(norms, stored):
        assert len(before) == len(params)
        tot = 0.0
        for p, q in zip(params, ref_params):
            assert _rel(before[id(p)], want[id(q)]) < 1e-6, (tuple(p.shape), float(before[id(p)]), want[id(q)])
            assert torch.equal(before[id(p)], after[id(p)])
            tot += want[id(q)] ** 2
        assert _rel(total, tot ** 0.5) < 1e-6
    _, _, _, _, norms2, _, _ = _run(True, k, track=True)
    for (a, ta, _), (b, tb, _) in zip(norms, norms2):
        assert torch.equal(ta, tb) and all(torch.equal(a[i], b[j]) for i, j in zip(a, b))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2])
def test_stored_gradient_norms_without_host_sync(k):
    """overlap_backward=False: the norms of p.grad (autograd's accumulation) within 1e-6, no host sync in backward,
    grad_norms() or step(), and the same updates as without tracking."""
    params, t_on, s_on, _, norms, stored, _ = _run(False, k, track=True, sync_check=True)
    _, t_off, s_off, _, _, _, _ = _run(False, k, track=False)
    for a, b in zip(t_off, t_on):
        assert torch.equal(a, b)
    _same_state(s_off, s_on)
    for (before, total, _), want in zip(norms, stored):
        for p in params:
            assert _rel(before[id(p)], want[id(p)]) < 1e-6
        assert _rel(total, sum(v * v for v in want.values()) ** 0.5) < 1e-6


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
def test_clipping_with_tracking(overlap):
    """gradient_clip_val + tracking: the weights of the clip-only run bit for bit, and the tracked total within 1e-6 of
    last_grad_norm (the clip's own dd_grad_sumsq, unchanged)."""
    params, t_both, _, _, norms, _, opt = _run(overlap, 2, track=True, clip=100.0, windows=1)
    _, t_clip1, _, _, _, _, opt1 = _run(overlap, 2, track=False, clip=100.0, windows=1)
    for a, b in zip(t_clip1, t_both):
        assert torch.equal(a, b)
    (before, total, _), = norms
    assert _rel(total, opt.last_grad_norm) < 1e-6 and torch.equal(opt.last_grad_norm, opt1.last_grad_norm)
    ref_params, _, _, _, _, stored, _ = _run(False, 2, track=False, clip=100.0, windows=1)   # autograd's .grad
    for p, q in zip(params, ref_params):
        assert _rel(before[id(p)], stored[0][id(q)]) < 1e-6


# ------------------------------------------------------------------------------------------------
# the modules' grad_norm()
# ------------------------------------------------------------------------------------------------
def _roadmap_step(opt_factory):
    from types import SimpleNamespace
    model, _, views, road = build_roadmap_pair(batch=4, hidden=16, latent=8, view_h=16, view_w=20, dtype="bf16",
                                               device="cuda:0")
    model.frozen = False
    model.ae.unfreeze()
    model.hparams = SimpleNamespace(**{**vars(model.hparams), "track_grad_norm": 2})
    opt = opt_factory(model)
    batch = (tuple(views.cuda().unbind(0)), None, tuple(road.cuda().unbind(0)))
    with cpu_rng_dropout():
        torch.manual_seed(7)
        loss = model._run_step(batch, 1, "train")[0]
        loss.backward()
    out = model.grad_norm(2)
    stored = {n: float(torch.linalg.vector_norm(p.grad.double())) for n, p in model.named_parameters()
              if p.grad is not None}
    opt.step()
    torch.cuda.synchronize()
    return model, out, stored


@pytest.mark.gpu
def test_roadmap_grad_norm_hook():
    from driving_dirty_b200.optim import FusedAdam, attach_optimizer, make_adam
    model, out, stored = _roadmap_step(lambda m: make_adam(m, 1e-3))
    assert isinstance(model._dd_optimizer, FusedAdam) and model._dd_optimizer.track_grad_norm == 2
    names = [n for n, p in model.named_parameters() if p.requires_grad]
    assert set(out) == {f"grad_2_norm_{n}" for n in names} | {"grad_2_norm_total"}
    for wide in ("fc1.weight", "ae.encoder.fc1.fc1.weight"):
        assert f"grad_2_norm_{wide}" in out
    for n in names:
        v = out[f"grad_2_norm_{n}"]
        assert v.is_cuda and v.dtype == torch.float32 and v.dim() == 0
        assert _rel(v, stored[n]) < 1e-6, n

    def fused(m):
        opt = FusedAdam([p for p in m.parameters() if p.requires_grad], lr=1e-3, overlap_backward=True, track_grad_norm=2)
        attach_optimizer(m, opt)
        return opt
    model2, out2, stored2 = _roadmap_step(fused)
    assert model2.fc1.weight.grad is None                          # stepped inside the backward pass
    assert set(out2) == set(out)
    for n in names:
        assert _rel(out2[f"grad_2_norm_{n}"], stored[n]) < 1e-6, n
    # --optimizer torch: the base class's numbers
    model3, out3, _ = _roadmap_step(lambda m: (setattr(m.hparams, "optimizer", "torch"), make_adam(m, 1e-3))[1])
    assert all(isinstance(v, float) for v in out3.values())


# ------------------------------------------------------------------------------------------------
# two GPUs: the rank mean's norms, identical on both ranks
# ------------------------------------------------------------------------------------------------
def _dist_worker(rank, world, port, k, frozen, out, wide=True):
    import torch.distributed as dist
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        N, K, B = 2048, 1028, 32
        res = []
        for track in (False, True):
            g = torch.Generator().manual_seed(12)
            w = torch.nn.Parameter((torch.randn(N, K, generator=g) * 0.05).to(dev))
            b = torch.nn.Parameter((torch.randn(N, generator=g) * 0.05).to(dev))
            s = torch.nn.Parameter(torch.randn(37, generator=g).to(dev))
            f = torch.nn.Parameter(torch.randn(5, generator=g).to(dev))      # frozen in the replicated form
            opt = FusedAdam([w, b, s, f], lr=1e-2, overlap_backward=True, accumulate_grad_batches=k,
                            track_grad_norm=2 if track else -1, shard_min_numel=(1 << 20) if wide else (1 << 40))
            norms, means = [], []
            for t in range(3):
                opt.zero_grad()
                gw = gb = gs = gf = 0
                for j in range(k):
                    xs = [torch.randn(B, K, generator=g) for _ in range(world)]
                    gys = [torch.randn(B, N, generator=g) / k for _ in range(world)]
                    ops.linear(xs[rank].to(dev), w, b, impl=_lib.IMPL_TCGEN05).backward(gys[rank].to(dev))
                    c = torch.randn(world, 37, generator=g)
                    (s * c[rank].to(dev)).sum().backward()
                    if not frozen:
                        cf = torch.randn(world, 5, generator=g)
                        (f * cf[rank].to(dev)).sum().backward()
                        gf = gf + cf.double().mean(0)
                    gw = gw + sum((gys[r].t() @ xs[r]).double() for r in range(world)) / world
                    gb = gb + sum(gys[r].sum(0).double() for r in range(world)) / world
                    gs = gs + c.double().mean(0)
                if track:
                    got = opt.grad_norms()
                    norms.append(torch.stack([got[w], got[b], got[s], got["total"]] + ([got[f]] if not frozen else [])))
                want = [gw.norm(), gb.norm(), gs.norm()] + ([gf.norm()] if not frozen else [])
                means.append(torch.stack(want))
                opt.step()
            opt.synchronize()
            torch.cuda.synchronize()
            res.append(([t.detach().clone() for t in (w, b, s, f)], norms, means))
        (w_off, _, _), (w_on, norms, means) = res
        same_w = all(torch.equal(a, c) for a, c in zip(w_off, w_on))
        allnorm = torch.stack(norms)
        gathered = [torch.empty_like(allnorm) for _ in range(world)]
        dist.all_gather(gathered, allnorm)
        same_bits = all(torch.equal(gathered[0], x) for x in gathered)
        err = 0.0
        for nrm, want in zip(norms, means):
            got = nrm.double().cpu()
            parts = torch.cat([got[:3], got[4:]])
            err = max(err, float(((parts - want) / want).abs().max()))
            err = max(err, abs(float(got[3]) - float(want.norm())) / float(want.norm()))
        if rank == 0:
            with open(out, "w") as fh:
                fh.write(f"{int(same_w)} {int(same_bits)} {err}")
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("frozen", [False, True])
@pytest.mark.parametrize("wide", [True, False])       # False: every tensor in the flat bucket, no wide weight
def test_rank_mean_norms_two_gpus(tmp_path, k, frozen, wide):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    from tests.test_optim import _free_port
    out = str(tmp_path / "res.txt")
    mp.spawn(_dist_worker, args=(2, _free_port(), k, frozen, out, wide), nprocs=2, join=True)
    same_w, same_bits, err = open(out).read().split()
    assert same_w == "1" and same_bits == "1" and float(err) < 1e-6, (same_w, same_bits, err)
