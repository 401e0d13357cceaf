"""Gradient clipping by the global L2 norm in optim.FusedAdam (gradient_clip_val, Lightning's flag): dd_grad_sumsq against
float64 NumPy and torch.nn.utils.get_total_norm, its clip coefficient against torch's formula bit for bit, and FusedAdam
against clip_grad_norm_ + torch.optim.Adam -- with the update inside the backward pass or not, with accumulation windows,
with and without weight decay -- and, when clipping does not bite, against FusedAdam without clipping bit for bit."""
import ctypes
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from tests.helpers import build_roadmap_pair, cpu_rng_dropout
from tests.test_linear_bwd_adam_gpu import PAD, _bands_intact, _guarded, _state_dicts_equal


def _sumsq(tensors, max_norm):
    """dd_grad_sumsq -> (guarded output buffer, norm, coefficient, fp64 sum of squares)."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, stream_ptr
    assert PAD % 2 == 0                                         # the fp64 sum at out + 2 stays 8-byte aligned
    dev = torch.device("cuda")
    ws = torch.zeros(int(_lib.load().dd_grad_sumsq_workspace_bytes()), dtype=torch.uint8, device=dev)
    buf, out = _guarded(torch.zeros(4, device=dev))
    n = len(tensors)
    call("dd_grad_sumsq", (ctypes.c_void_p * n)(*[t.data_ptr() for t in tensors]),
         (ctypes.c_longlong * n)(*[t.numel() for t in tensors]), n, float(max_norm), out.data_ptr(), ws.data_ptr(),
         ws.numel(), stream_ptr())
    torch.cuda.synchronize()
    return buf, out[0].clone(), out[1].clone(), float(out[2:].clone().view(torch.float64))


def _ragged(seed, count=6):
    """Tensors of lengths 0, 1, 3, 4, 5, 2^20 + 3 (and more when count > 6), each starting 0..3 elements past a 16-byte
    boundary, inside sentinel-banded buffers."""
    g = torch.Generator().manual_seed(seed)
    lens = [0, 1, 3, 4, 5, (1 << 20) + 3] + [int(x) for x in torch.randint(0, 5000, (max(count - 6, 0),), generator=g)]
    bufs, views = [], []
    for i, n in enumerate(lens[:count]):
        shift = i % 4
        buf = torch.full((n + shift + 2 * PAD,), -7.0, device="cuda")
        v = buf[PAD + shift: PAD + shift + n]
        v.copy_(torch.randn(n, generator=g).cuda() * (1 + i % 3))
        bufs.append((buf, shift, n))
        views.append(v)
    return bufs, views


@pytest.mark.gpu
@pytest.mark.parametrize("count", [6, 150])          # 150: three launches of up to 64 tensors each
def test_grad_sumsq_ragged_lists(count):
    from driving_dirty_b200 import _lib  # noqa: F401
    bufs, views = _ragged(count, count)
    out_buf, norm, coef, sumsq = _sumsq(views, 1.0)
    ref = float(sum(np.square(v.cpu().numpy().astype(np.float64)).sum() for v in views))
    assert abs(sumsq - ref) <= 1e-12 * ref, (sumsq, ref)
    tn = torch.nn.utils.get_total_norm(views)
    assert abs(float(norm) - float(tn)) <= 2e-6 * float(tn)
    assert _bands_intact(out_buf)
    for buf, shift, n in bufs:                                  # the inputs are only read
        assert bool((buf[:PAD + shift] == -7.0).all()) and bool((buf[PAD + shift + n:] == -7.0).all())
    again = _sumsq(views, 1.0)
    assert torch.equal(again[1], norm) and torch.equal(again[2], coef) and again[3] == sumsq


@pytest.mark.gpu
def test_grad_sumsq_empty_list():
    _, norm, coef, sumsq = _sumsq([], 1.0)
    assert float(norm) == 0.0 and sumsq == 0.0 and float(coef) == 1.0


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["below", "equal", "above", "zeros", "inf", "nan"])
def test_clip_coefficient_is_torchs_formula(case):
    g = torch.Generator().manual_seed(3)
    ts = [torch.randn(n, generator=g).cuda() for n in (1000, 37, 4096)]
    if case == "zeros":
        ts = [t.zero_() for t in ts]
    if case == "inf":
        ts[1][5] = float("inf")
    if case == "nan":
        ts[2][7] = float("nan")
    true_norm = float(torch.nn.utils.get_total_norm(ts))
    max_norm = {"below": 0.5 * true_norm, "above": 2.0 * true_norm}.get(case, true_norm if np.isfinite(true_norm) else 1.0)
    if case == "zeros":
        max_norm = 1.0
    _, norm, coef, _ = _sumsq(ts, max_norm)
    want = torch.clamp(max_norm / (norm + 1e-6), max=1.0)      # torch's clip_grad_norm_ on the kernel's norm
    assert torch.equal(coef.view(torch.int32), want.view(torch.int32)), (float(coef), float(want))
    if case == "inf":
        assert float(norm) == float("inf") and float(coef) == 0.0
    if case == "nan":
        assert np.isnan(float(norm)) and np.isnan(float(coef))
    if case == "above":
        assert float(coef) == 1.0
    if case == "below":
        assert float(coef) < 1.0


# ------------------------------------------------------------------------------------------------
# FusedAdam(gradient_clip_val) against clip_grad_norm_ + torch.optim.Adam
# ------------------------------------------------------------------------------------------------
N, K, B = 4096, 1028, 32
SCALES = [1.0, 0.01, 3.0, 0.05]           # per-window gradient scale: clipping bites in some windows, not in others
CLIP = 1000.0                             # the wide weight's gradient norm is ~1e4 at scale 1


def _problem(seed=11):
    g = torch.Generator().manual_seed(seed)
    w0 = torch.randn(N, K, generator=g) * 0.05
    b0 = torch.randn(N, generator=g) * 0.05
    s0 = torch.randn(37, generator=g)
    data = [[(torch.randn(B, K, generator=g), torch.randn(B, N, generator=g), torch.randn(37, generator=g))
             for _ in range(2)] for _ in SCALES]
    return (w0, b0, s0), data


def _loss_backward(w, b, s, x, gy, gs, scale, k):
    from driving_dirty_b200 import _lib, ops
    y = ops.linear(x.cuda(), w, b, impl=_lib.IMPL_TCGEN05)
    ((y * gy.cuda()).sum() * (scale / k) + (s * s * gs.cuda()).sum() * (scale / k)).backward()


def _fused_run(init, data, clip, overlap, k, wd, **kw):
    from driving_dirty_b200.optim import FusedAdam
    w, b, s = [torch.nn.Parameter(t.clone().cuda()) for t in init]
    extra = {} if clip is None else {"gradient_clip_val": clip}
    opt = FusedAdam([{"params": [w, b]}, {"params": [s]}], lr=1e-2, weight_decay=wd, overlap_backward=overlap,
                    accumulate_grad_batches=k, **extra, **kw)
    norms = []
    for scale, window in zip(SCALES, data):
        opt.zero_grad()
        for j in range(k):
            _loss_backward(w, b, s, *window[j], scale, k)
        opt.step()
        norms.append(None if opt.last_grad_norm is None else opt.last_grad_norm.clone())
    torch.cuda.synchronize()
    return [t.detach().clone() for t in (w, b, s)], opt.state_dict(), norms


def _torch_run(init, data, clip, k, wd):
    w, b, s = [torch.nn.Parameter(t.clone().cuda()) for t in init]
    opt = torch.optim.Adam([{"params": [w, b]}, {"params": [s]}], lr=1e-2, weight_decay=wd)
    norms, clipped = [], []
    for scale, window in zip(SCALES, data):
        opt.zero_grad()
        for j in range(k):
            _loss_backward(w, b, s, *window[j], scale, k)
        norms.append(torch.nn.utils.clip_grad_norm_([w, b, s], clip))
        clipped.append(float(norms[-1]) > clip)
        opt.step()
    torch.cuda.synchronize()
    return [t.detach().clone() for t in (w, b, s)], opt.state_dict(), norms, clipped


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("k", [1, 2])
@pytest.mark.parametrize("wd", [0.0, 0.01])
def test_fused_adam_clipping_matches_torch(overlap, k, wd):
    init, data = _problem()
    clip = CLIP
    ref_w, ref_sd, ref_norms, clipped = _torch_run(init, data, clip, k, wd)
    assert any(clipped) and not all(clipped), clipped
    got_w, got_sd, got_norms = _fused_run(init, data, clip, overlap, k, wd)
    for a, c in zip(got_norms, ref_norms):
        assert abs(float(a) - float(c)) <= 2e-6 * float(c), (float(a), float(c))
    # Deliberately looser than 1e-6 relative for the moments.  exp_avg: the coefficient carries torch's fp32 norm error
    # (<= 2e-6).  exp_avg_sq besides: FusedAdam forms 1 - beta2 in fp32 (dd_adam_step, unchanged by clipping), torch
    # rounds the double 1 - beta2 to fp32 -- 1.3e-5 apart at beta2 = 0.999, with or without clipping
    for i in ref_sd["state"]:
        for f, tol in (("exp_avg", 5e-6), ("exp_avg_sq", 3e-5)):
            r, x = ref_sd["state"][i][f], got_sd["state"][i][f]
            assert float((x - r).abs().max()) <= tol * float(r.abs().max()), (i, f)
    for a, c in zip(got_w, ref_w):
        assert float((a - c).abs().max()) <= 1e-5 * float(c.abs().max()) + 1e-7


@pytest.mark.gpu
@pytest.mark.parametrize("overlap", [False, True])
@pytest.mark.parametrize("k", [1, 2])
def test_inactive_clipping_is_bit_identical(overlap, k):
    """With a threshold far above the norm the coefficient is exactly 1: weights and moments are those of FusedAdam
    without clipping, bit for bit (with overlap_backward=True that one steps inside the backward pass)."""
    init, data = _problem()
    ref_w, ref_sd, _ = _fused_run(init, data, None, overlap, k, 0.01)
    got_w, got_sd, norms = _fused_run(init, data, 1e30, overlap, k, 0.01)
    assert all(n is not None and n.dim() == 0 and n.dtype == torch.float32 and n.is_cuda for n in norms)
    for a, c in zip(got_w, ref_w):
        assert torch.equal(a, c)
    _state_dicts_equal(ref_sd, got_sd)


@pytest.mark.gpu
def test_clipping_off_launches_unchanged():
    """gradient_clip_val = 0 or None launches what FusedAdam without the argument launches, in backward and in step();
    clipping on adds dd_grad_sumsq's launch to step()."""
    from driving_dirty_b200 import _lib
    from driving_dirty_b200.optim import FusedAdam
    init, data = _problem()

    def count(**kw):
        w, b, s = [torch.nn.Parameter(t.clone().cuda()) for t in init]
        opt = FusedAdam([w, b, s], lr=1e-2, overlap_backward=True, **kw)
        torch.cuda.synchronize()
        n0 = _lib.launch_count()
        _loss_backward(w, b, s, *data[0][0], 1.0, 1)
        torch.cuda.synchronize()
        n1 = _lib.launch_count()
        stepped_in_backward = w.grad is None
        opt.step()
        torch.cuda.synchronize()
        return n1 - n0, _lib.launch_count() - n1, stepped_in_backward, opt.last_grad_norm is None

    base = count()
    assert base[2] and base[3]
    assert count(gradient_clip_val=0) == base and count(gradient_clip_val=None) == base
    on = count(gradient_clip_val=1.0)
    assert not on[2] and not on[3]                              # the wide weight's step left the backward pass


@pytest.mark.gpu
def test_bad_values_rejected():
    from driving_dirty_b200.optim import FusedAdam
    w = torch.nn.Parameter(torch.zeros(8, device="cuda"))
    for bad in (-1.0, float("inf"), float("nan"), "1", True):
        with pytest.raises(ValueError, match="gradient_clip_val"):
            FusedAdam([w], gradient_clip_val=bad)


@pytest.mark.gpu
def test_roadmap_configure_optimizers_clips():
    """RoadMapBCE on the bf16 tensor-core path through configure_optimizers with hparams.gradient_clip_val, three steps:
    the norms, and the model and moments after the first step, agree with torch's clip_grad_norm_ followed by FusedAdam
    without clipping."""
    from driving_dirty_b200.optim import FusedAdam
    res = []
    for mode in ("fused", "torch_clip"):
        model, _, views, road = build_roadmap_pair(batch=4, hidden=16, latent=8, view_h=16, view_w=20, dtype="bf16",
                                                   device="cuda:0")
        model.frozen = False
        model.ae.unfreeze()
        clip = 0.05
        if mode == "fused":
            model.hparams.gradient_clip_val = clip
            opt = model.configure_optimizers()[0][0]
            assert isinstance(opt, FusedAdam) and opt.gradient_clip_val == clip
        else:
            opt = model.configure_optimizers()[0][0]
            assert isinstance(opt, FusedAdam) and not opt.gradient_clip_val
        params = [p for p in model.parameters() if p.requires_grad]
        batch = (tuple(views.cuda().unbind(0)), None, tuple(road.cuda().unbind(0)))
        norms = []
        for i in range(3):
            with cpu_rng_dropout():
                torch.manual_seed(7 + i)
                model._run_step(batch, 1, "train")[0].backward()
            if i == 0:
                exact = float(sum((p.grad.double() ** 2).sum() for p in params if p.grad is not None) ** 0.5)
            if mode == "torch_clip":
                norms.append(float(torch.nn.utils.clip_grad_norm_(params, clip)))
            opt.step()
            if mode == "fused":
                norms.append(float(opt.last_grad_norm))
            opt.zero_grad()
            if i == 0:
                torch.cuda.synchronize()
                first = ({kk: v.detach().clone() for kk, v in model.state_dict().items()}, opt.state_dict())
        torch.cuda.synchronize()
        res.append((*first, norms))
    (sd0, o0, n0), (sd1, o1, n1) = res
    assert all(n > clip for n in n1), n1                       # clipping bit in every step
    # the first step's gradients are the same in both runs: the kernel's norm against a float64 one, and torch's fp32
    # norm (its own error is a few 1e-6 here), and the state after that step.  Later steps start from weights clipped with
    # coefficients a few 1e-6 apart, which Adam's normalised update and the bf16 forward spread: their norms agree loosely.
    assert abs(n0[0] - exact) <= 1e-6 * exact, (n0[0], exact)
    assert abs(n0[0] - n1[0]) <= 1e-5 * n1[0], (n0[0], n1[0])
    for a, c in zip(n0[1:], n1[1:]):
        assert abs(a - c) <= 1e-2 * c, (a, c)
    for kk in sd0:
        if sd0[kk].is_floating_point():
            r = sd1[kk].float()
            assert float((sd0[kk].float() - r).abs().max()) <= 1e-5 * float(r.abs().max()) + 1e-7, kk
    for i in o1["state"]:
        for f in ("exp_avg", "exp_avg_sq"):
            r, x = o1["state"][i][f], o0["state"][i][f]
            assert float((x - r).abs().max()) <= 1e-4 * float(r.abs().max()) + 1e-30, (i, f)


@pytest.mark.gpu
def test_make_adam_passes_gradient_clip_val():
    from driving_dirty_b200.optim import FusedAdam, make_adam
    model = torch.nn.Linear(8, 4).cuda()
    model.hparams = SimpleNamespace(gradient_clip_val=0.5)
    opt = make_adam(model, 1e-3)
    assert isinstance(opt, FusedAdam) and opt.gradient_clip_val == 0.5
    model.hparams = SimpleNamespace()
    assert make_adam(model, 1e-3).gradient_clip_val == 0.0
