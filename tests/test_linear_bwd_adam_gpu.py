"""dd_linear_bwd_adam (the backward pass of a wide linear layer with the Adam step of its weight folded in) against the
unfused launches it replaces: dd_linear_dgrad + dd_linear_wgrad + dd_adam_step, bit for bit, over several steps with
weight decay; and optim.FusedAdam(overlap_backward=True) at world size 1 against overlap_backward=False."""
import pytest
import torch

from tests.helpers import build_roadmap_pair, cpu_rng_dropout

PAD = 64                 # sentinel elements on each side of every buffer (keeps the 16-byte alignment)
SENTINEL = -12345.0


def _guarded(t):
    """(buffer with sentinel bands, view of t's shape inside it)."""
    buf = torch.full((t.numel() + 2 * PAD,), SENTINEL, dtype=t.dtype, device=t.device)
    inner = buf[PAD:PAD + t.numel()].view_as(t)
    inner.copy_(t)
    return buf, inner


def _bands_intact(buf):
    return bool((buf[:PAD] == SENTINEL).all()) and bool((buf[-PAD:] == SENTINEL).all())


def _run(fused, B, N, K, dx_dtype, steps, seed=3):
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(seed)
    w0 = (torch.randn(N, K, generator=g) * 0.05).to(dev)
    wbuf, w = _guarded(w0)
    mbuf, m = _guarded(torch.zeros(N, K, device=dev))
    vbuf, v = _guarded(torch.zeros(N, K, device=dev))
    n_ws = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    ws = torch.empty(n_ws, dtype=torch.uint8, device=dev)
    lr, b1, b2, eps, wd = 1e-2, 0.9, 0.999, 1e-8, 0.01
    out = []
    for t in range(1, steps + 1):
        x = torch.randn(B, K, generator=g).to(dev)
        dy = torch.randn(B, N, generator=g).to(dev)
        db = torch.empty(N, device=dev)
        dxbuf, dx = _guarded(torch.zeros(B, K, dtype=dx_dtype or torch.float32, device=dev))
        dxp = dx.data_ptr() if dx_dtype is not None else None
        code = dtype_code(dx_dtype) if dx_dtype is not None else _lib.DD_F32
        if fused:
            call("dd_linear_bwd_adam", dy.data_ptr(), x.data_ptr(), w.data_ptr(), m.data_ptr(), v.data_ptr(), dxp, code,
                 db.data_ptr(), ws.data_ptr(), n_ws, B, N, K, lr, b1, b2, eps, wd, t, stream_ptr())
        else:
            if dxp is not None:
                call("dd_linear_dgrad", dy.data_ptr(), w.data_ptr(), dxp, code, ws.data_ptr(), n_ws, B, N, K,
                     _lib.IMPL_TCGEN05, stream_ptr())
            dw = torch.empty(N, K, device=dev)
            call("dd_linear_wgrad", dy.data_ptr(), x.data_ptr(), _lib.DD_F32, dw.data_ptr(), db.data_ptr(), B, N, K,
                 _lib.IMPL_TCGEN05, stream_ptr())
            call("dd_adam_step", w.data_ptr(), dw.data_ptr(), m.data_ptr(), v.data_ptr(), N * K, lr, b1, b2, eps, wd, t, 1.0,
                 stream_ptr())
        torch.cuda.synchronize()
        assert _bands_intact(dxbuf)
        out.append((dx.clone() if dx_dtype is not None else None, db.clone()))
    assert _bands_intact(wbuf) and _bands_intact(mbuf) and _bands_intact(vbuf)
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
def test_bwd_adam_matches_unfused_launches(B, N, K, dx_dtype):
    ref = _run(False, B, N, K, dx_dtype, steps=3)
    got = _run(True, B, N, K, dx_dtype, steps=3)
    for name, a, c in zip(("weight", "exp_avg", "exp_avg_sq"), ref[:3], got[:3]):
        assert torch.equal(a, c), (name, float((a - c).abs().max()))
    for (dx_r, db_r), (dx_g, db_g) in zip(ref[3], got[3]):
        assert torch.equal(db_r, db_g)
        if dx_dtype is not None:
            assert torch.equal(dx_r, dx_g), float((dx_r.float() - dx_g.float()).abs().max())


@pytest.mark.gpu
def test_bwd_adam_rejects_what_it_cannot_run():
    from driving_dirty_b200._lib import call
    dev = torch.device("cuda")
    t = torch.zeros(64 * 65536, device=dev)
    with pytest.raises(RuntimeError):     # B > 32
        call("dd_linear_bwd_adam", t.data_ptr(), t.data_ptr(), t.data_ptr(), t.data_ptr(), t.data_ptr(), None, 0, None,
             None, 0, 33, 64, 65536, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, None)
    with pytest.raises(RuntimeError):     # too narrow for the tensor-core path
        call("dd_linear_bwd_adam", t.data_ptr(), t.data_ptr(), t.data_ptr(), t.data_ptr(), t.data_ptr(), None, 0, None,
             None, 0, 32, 64, 1024, 1e-3, 0.9, 0.999, 1e-8, 0.0, 1, None)


def _linear_steps(overlap, B, steps=3):
    from driving_dirty_b200 import _lib, ops
    from driving_dirty_b200.optim import FusedAdam
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(8)
    N, K = 4096, 1028
    w = torch.nn.Parameter((torch.randn(N, K, generator=g) * 0.05).to(dev))
    b = torch.nn.Parameter((torch.randn(N, generator=g) * 0.05).to(dev))
    opt = FusedAdam([w, b], lr=1e-2, weight_decay=0.01, overlap_backward=overlap)
    grads = []
    for _ in range(steps):
        x = torch.randn(B, K, generator=g).to(dev).requires_grad_(True)
        gy = torch.randn(B, N, generator=g).to(dev)
        opt.zero_grad()
        ops.linear(x, w, b, impl=_lib.IMPL_TCGEN05).backward(gy)
        grads.append((w.grad is None, x.grad.clone()))
        opt.step()
    return w.detach().clone(), b.detach().clone(), opt.state_dict(), grads


@pytest.mark.gpu
@pytest.mark.parametrize("B", [32, 40])
def test_fused_adam_overlap_backward_world_one(B):
    """B = 32: the weight is stepped inside backward (no gradient tensor); B = 40: the stored-gradient fallback.  Both give
    the results of overlap_backward=False."""
    ref, got = _linear_steps(False, B), _linear_steps(True, B)
    assert all(not none for none, _ in ref[3])
    assert all(none == (B <= 32) for none, _ in got[3])
    for (_, a), (_, c) in zip(ref[3], got[3]):
        assert torch.equal(a, c)
    assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
    _state_dicts_equal(ref[2], got[2])


def _state_dicts_equal(a, c):
    assert a["param_groups"] == c["param_groups"]
    assert a["state"].keys() == c["state"].keys()
    for k in a["state"]:
        for f in ("step", "exp_avg", "exp_avg_sq"):
            assert torch.equal(a["state"][k][f], c["state"][k][f]), (k, f)


@pytest.mark.gpu
def test_roadmap_train_steps_with_the_update_in_backward():
    """RoadMapBCE on the bf16 tensor-core path (its 640,000-wide head streams through dd_linear_bwd_adam), two training
    steps: model and optimizer state as with the update in step()."""
    from driving_dirty_b200.optim import FusedAdam
    res = []
    for overlap in (False, True):
        model, _, views, road = build_roadmap_pair(batch=4, hidden=16, latent=8, view_h=16, view_w=20, dtype="bf16",
                                                   device="cuda:0")
        model.frozen = False
        model.ae.unfreeze()
        opt = FusedAdam([p for p in model.parameters() if p.requires_grad], lr=1e-3, overlap_backward=overlap)
        batch = (tuple(views.cuda().unbind(0)), None, tuple(road.cuda().unbind(0)))
        head = model.fc1.weight
        for i in range(2):
            opt.zero_grad()
            with cpu_rng_dropout():
                torch.manual_seed(7 + i)
                loss = model._run_step(batch, 1, "train")[0]
                loss.backward()
            assert (head.grad is None) == overlap
            opt.step()
        torch.cuda.synchronize()
        res.append(({k: v.detach().clone() for k, v in model.state_dict().items()}, opt.state_dict()))
    (sd0, o0), (sd1, o1) = res
    assert sd0.keys() == sd1.keys()
    for k in sd0:
        assert torch.equal(sd0[k], sd1[k]), k
    _state_dicts_equal(o0, o1)
