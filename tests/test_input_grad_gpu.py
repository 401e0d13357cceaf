"""Gradients to the camera views: the c1 image-gradient kernel (dd_conv_c1_dgrad), the differentiable stitch / stitch-mask /
view extraction, and views.grad through RoadMapBCE, BasicAE and BBSpatialRoadMap against torch autograd through the
reference's own expressions.  Pure data movement is compared bit for bit."""
import contextlib

import numpy as np
import pytest
import torch

from oracle import scene_oracle as so
from tests.helpers import build_roadmap_pair, cpu_rng_dropout, rel_max_err

pytestmark = pytest.mark.gpu

ORDER = [0, 1, 2, 5, 4, 3]
IMPL_AUTO, IMPL_SIMT, IMPL_TCGEN05 = 0, 1, 2


# ----------------------------------------------------------------------------- differentiable restatements -----
def ref_stitch(views):
    """wide_stitch_six_images (roadmap_bce_v2.py:53-64) as the reference writes it: differentiable."""
    b, _, c, h, _ = views.shape
    return views[:, ORDER].permute(0, 2, 3, 1, 4).reshape(b, c, h, -1)


def ref_six_to_one(views, slot):
    """six_to_one_task (autoencoder.py:53-73) with the slot drawn: clone, take the slot's block, zero it."""
    x = ref_stitch(views).clone()
    w = views.shape[-1]
    y = x[:, :, :, slot * w:(slot + 1) * w].clone()
    x[:, :, :, slot * w:(slot + 1) * w] = 0.0
    return x, y


def ref_view_transform(views, view, mode):
    """SpatialMappingCNN's camera transforms (spatial_bb/components.py:34-62): rot90 / flip."""
    img = views[:, view]
    if mode == 1:
        return torch.rot90(img, 1, [2, 3])
    if mode == 2:
        return torch.rot90(img, 1, [3, 2])
    if mode == 3:
        return torch.flip(img, [2, 3])
    return img


@contextlib.contextmanager
def differentiable_oracle():
    """The oracle restates the stitch and the camera transforms in numpy, which drops the autograd graph; for views.grad
    it runs with the restatements above in their place (test_restatements_equal_the_oracle checks they agree)."""
    saved = so.stitch, so.view_transform
    so.stitch, so.view_transform = ref_stitch, ref_view_transform
    try:
        yield
    finally:
        so.stitch, so.view_transform = saved


@pytest.fixture(scope="module")
def lib():
    from driving_dirty_b200 import _lib
    assert torch.cuda.is_available()
    return _lib


def test_restatements_equal_the_oracle():
    views = torch.rand(2, 6, 3, 5, 7)
    assert torch.equal(ref_stitch(views), so.stitch(views))
    for slot in range(6):
        x, y = ref_six_to_one(views, slot)
        xo, yo = so.six_to_one(views, slot)
        assert torch.equal(x, xo) and torch.equal(y, yo)
    for mode in range(4):
        assert torch.equal(ref_view_transform(views, 2, mode).contiguous(), so.view_transform(views, 2, mode))


# ----------------------------------------------------------------------------- the c1 image gradient -----------
def _c1_dgrad(lib, da1, w1, views, impl, B, H, Wm):
    shape = (B, 6, 3, H, Wm // 6) if views else (B, 3, H, Wm)
    dx = torch.full(shape, float("nan"), device="cuda")
    code = 1 if da1.dtype == torch.bfloat16 else 0
    lib.call("dd_conv_c1_dgrad", da1.data_ptr(), code, w1.data_ptr(), dx.data_ptr(), int(views), B, H, Wm, impl,
             lib.stream_ptr())
    return dx


@pytest.mark.parametrize("B,H,Wv", [(1, 5, 7), (3, 37, 35), (2, 70, 23), (2, 256, 306)])
@pytest.mark.parametrize("dtype,impl", [(torch.float32, IMPL_AUTO), (torch.bfloat16, IMPL_AUTO),
                                        (torch.bfloat16, IMPL_TCGEN05), (torch.bfloat16, IMPL_SIMT)])
def test_c1_dgrad_against_conv2d_input(lib, B, H, Wv, dtype, impl):
    """Both layouts against torch.nn.grad.conv2d_input on the same operands (the tensor-core form reads w1 as bf16) within
    1e-5 of max|ref|; the views layout is the inverse stitch of the mosaic layout, bit for bit.  The ragged shapes put
    128-pixel strips across view boundaries and the image edge; 70 rows span two 64-row work items."""
    Wm = 6 * Wv
    g = torch.Generator().manual_seed(B * 1000 + H + Wv)
    da1 = (torch.rand(B, H, Wm, 32, generator=g) - 0.5).to(dtype)
    w1 = torch.rand(32, 3, 3, 3, generator=g) - 0.5
    tc = dtype == torch.bfloat16 and impl != IMPL_SIMT
    w_ref = w1.bfloat16().double() if tc else w1.double()
    ref = torch.nn.grad.conv2d_input((B, 3, H, Wm), w_ref, da1.double().permute(0, 3, 1, 2), padding=1)
    da1_d, w1_d = da1.cuda(), w1.cuda()
    mosaic = _c1_dgrad(lib, da1_d, w1_d, False, impl, B, H, Wm)
    views = _c1_dgrad(lib, da1_d, w1_d, True, impl, B, H, Wm)
    torch.cuda.synchronize()
    err = rel_max_err(mosaic, ref)
    assert err < 1e-5, err
    unstitched = torch.empty_like(views)
    unstitched[:, ORDER] = mosaic.reshape(B, 3, H, 6, Wv).permute(0, 3, 1, 2, 4)
    assert torch.equal(views, unstitched)


def test_c1_dgrad_guard_bands_and_errors(lib):
    """The tensor-core form stays inside its output (sentinel bands before and after, both layouts, ragged shape); raw
    bytes are refused, misalignment is reported, B = 0 enqueues nothing."""
    GUARD = 4096
    B, H, Wv = 3, 37, 35
    Wm = 6 * Wv
    da1 = (torch.rand(B, H, Wm, 32, device="cuda") - 0.5).bfloat16()
    w1 = torch.rand(32, 3, 3, 3, device="cuda")
    st = lib.stream_ptr()
    for views in (0, 1):
        n = B * 3 * H * Wm
        raw = torch.full((n + 2 * GUARD,), 7.0, device="cuda")
        out = raw[GUARD:GUARD + n]
        lib.call("dd_conv_c1_dgrad", da1.data_ptr(), 1, w1.data_ptr(), out.data_ptr(), views, B, H, Wm, IMPL_TCGEN05, st)
        torch.cuda.synchronize()
        assert bool((raw[:GUARD] == 7).all()) and bool((raw[GUARD + n:] == 7).all()), "wrote outside its output"
    l = lib.load()
    dx = torch.empty(B, 3, H, Wm, device="cuda")
    assert l.dd_conv_c1_dgrad(da1.data_ptr(), 1, w1.data_ptr(), dx.data_ptr(), 2, B, H, Wm, 0, st) == -2     # DD_IN_U8
    assert l.dd_conv_c1_dgrad(da1.data_ptr(), 1, w1.data_ptr(), dx.data_ptr(), 3, B, H, Wm, 0, st) == -2
    for impl in (IMPL_AUTO, IMPL_SIMT):
        assert l.dd_conv_c1_dgrad(da1.data_ptr() + 2, 1, w1.data_ptr(), dx.data_ptr(), 0, B, H, Wm, impl, st) == -4
    assert l.dd_conv_c1_dgrad(da1.data_ptr(), 1, w1.data_ptr(), dx.data_ptr(), 1, B, H, Wm + 1, 0, st) == -1
    assert l.dd_conv_c1_dgrad(None, 1, None, None, 0, B, H, Wm, 0, st) == -1
    n0 = lib.launch_count()
    assert l.dd_conv_c1_dgrad(None, 1, None, None, 1, 0, H, Wm, 0, st) == 0
    assert lib.launch_count() == n0


# ----------------------------------------------------------------------------- data-movement gradients -----------
@pytest.mark.parametrize("B,H,W", [(1, 4, 6), (2, 5, 7), (2, 256, 306)])
def test_stitch_gradients_bit_exact(B, H, W):
    from driving_dirty_b200 import ops
    g = torch.Generator().manual_seed(H * W)
    views = torch.rand(B, 6, 3, H, W, generator=g)
    gm = torch.randn(B, 3, H, 6 * W, generator=g)
    gy = torch.randn(B, 3, H, W, generator=g)
    v = views.cuda().requires_grad_()
    m = ops.stitch(v)
    (m * gm.cuda()).sum().backward()
    r = views.clone().requires_grad_()
    (ref_stitch(r) * gm).sum().backward()
    assert torch.equal(m.detach().cpu(), ref_stitch(views)) and torch.equal(v.grad.cpu(), r.grad)
    # the collate_fn tuple form reaches the same leaf
    v.grad = None
    (ops.stitch(tuple(v.unbind(0))) * gm.cuda()).sum().backward()
    assert torch.equal(v.grad.cpu(), r.grad)
    for slot in range(6):
        v = views.cuda().requires_grad_()
        x, y = ops.stitch_mask(v, slot)
        ((x * gm.cuda()).sum() + (y * gy.cuda()).sum()).backward()
        r = views.clone().requires_grad_()
        xr, yr = ref_six_to_one(r, slot)
        ((xr * gm).sum() + (yr * gy).sum()).backward()
        assert torch.equal(x.detach().cpu(), xr.detach()) and torch.equal(y.detach().cpu(), yr.detach())
        assert torch.equal(v.grad.cpu(), r.grad), slot
    # only y used (x's gradient materialised as zeros)
    v = views.cuda().requires_grad_()
    (ops.stitch_mask(v, 4)[1] * gy.cuda()).sum().backward()
    r = views.clone().requires_grad_()
    (ref_six_to_one(r, 4)[1] * gy).sum().backward()
    assert torch.equal(v.grad.cpu(), r.grad)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_view_extraction_gradients_bit_exact(dtype):
    from driving_dirty_b200 import ops
    from driving_dirty_b200.bounding_box_model.spatial_bb.components import _STRIPS
    B, H, W = 2, 9, 13
    g = torch.Generator().manual_seed(5)
    views = torch.rand(B, 6, 3, H, W, generator=g)
    specs = [(cam, mode) for _, cam, mode, _ in _STRIPS]
    grads = [torch.randn(B, *((W, H) if m in (1, 2) else (H, W)), 3, generator=g).to(dtype) for _, m in specs]
    v = views.cuda().requires_grad_()
    outs = ops.view_extract_all(v, specs, dtype)
    sum((o.float() * gg.cuda().float()).sum() for o, gg in zip(outs, grads)).backward()
    r = views.clone().requires_grad_()
    refs = [ref_view_transform(r, cam, mode).permute(0, 2, 3, 1) for cam, mode in specs]
    sum((o * gg.float()).sum() for o, gg in zip(refs, grads)).backward()
    for o, ro in zip(outs, refs):
        assert torch.equal(o.cpu(), ro.detach().to(dtype))
    assert torch.equal(v.grad.cpu(), r.grad)
    # one camera: the other five views get zeros
    v = views.cuda().requires_grad_()
    (ops.view_extract(v, 4, 1, dtype).float() * grads[2].cuda().float()).sum().backward()
    r = views.clone().requires_grad_()
    (ref_view_transform(r, 4, 1).permute(0, 2, 3, 1) * grads[2].float()).sum().backward()
    assert torch.equal(v.grad.cpu(), r.grad)
    with pytest.raises(ValueError):
        ops.view_extract_all(v, [(1, 0), (1, 2)])


# ----------------------------------------------------------------------------- RoadMapBCE end to end ---------------
def _roadmap_views_grad(g, dtype, tuple_form):
    model, params, views, road = build_roadmap_pair(g["batch"], g["hidden"], g["latent"], g["view_h"], g["view_w"],
                                                    dtype=dtype, seed_w=g["seed_w"], seed_x=g["seed_x"])
    v = views.cuda().requires_grad_()
    batch = (tuple(v.unbind(0)) if tuple_form else v, None, tuple(road.cuda().unbind(0)))
    with cpu_rng_dropout():
        torch.manual_seed(g["seed_fwd"])
        out = model.training_step(batch, 1)
        out["loss"].backward()
        r = views.clone().requires_grad_()
        rnd = dict(act_dtype=torch.bfloat16, weight_dtype=torch.bfloat16) if dtype == "bf16" else {}
        with differentiable_oracle():
            so.train_step_grads(params, r, road, seed=g["seed_fwd"], **rnd)
    return v.grad.cpu(), r.grad


@pytest.mark.parametrize("tuple_form", [False, True])
@pytest.mark.parametrize("name", ["roadmap_small", "roadmap_odd"])
def test_roadmap_views_grad_fp32(golden, name, tuple_form):
    got, ref = _roadmap_views_grad(golden(name), "fp32", tuple_form)
    err = rel_max_err(got, ref)
    print(name, "views.grad rel-max", err)
    assert err < 1e-5, err


@pytest.mark.parametrize("tuple_form", [False, True])
@pytest.mark.parametrize("name", ["roadmap_small", "roadmap_odd"])
def test_roadmap_views_grad_bf16(golden, name, tuple_form):
    got, ref = _roadmap_views_grad(golden(name), "bf16", tuple_form)
    frob = float((got.double() - ref.double()).norm() / ref.double().norm())
    print(name, "bf16 views.grad rel-frobenius", frob)
    assert frob < 2e-2, frob


def _frozen_pair_run(model, views, road, requires):
    for p in model.parameters():
        p.requires_grad_(requires)
        p.grad = None
    v = views.cuda().requires_grad_()
    batch = (v, None, tuple(road.cuda().unbind(0)))
    with cpu_rng_dropout():
        torch.manual_seed(3)
        loss = model._run_step(batch, 1, "train")[0]
        loss.backward()
    return v.grad


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
def test_frozen_model_views_grad(dtype):
    """A frozen model under attribution: the same views.grad, bit for bit, as with every parameter requiring grad; no
    parameter gets a .grad; on the sign-word path the stack does not keep a1 / a2."""
    model, params, views, road = build_roadmap_pair(3, 16, 8, 16, 20, dtype=dtype)
    a = _frozen_pair_run(model, views, road, True)
    assert all(p.grad is not None for p in model.parameters() if p.requires_grad)
    b = _frozen_pair_run(model, views, road, False)
    assert torch.equal(a, b)
    assert all(p.grad is None for p in model.parameters())
    enc = model.ae.encoder
    feats = enc._stack(views.cuda().requires_grad_())
    saved = feats.grad_fn.saved_tensors          # (inp, w1, w2, w3, a1, a2, a3, bits1, bits2)
    if dtype == "bf16":
        assert saved[0] is None and saved[4] is None and saved[5] is None and saved[7] is not None
    else:
        assert saved[4] is not None and saved[5] is not None


def test_frozen_backward_launches_no_weight_gradient_kernel():
    from torch.profiler import ProfilerActivity, profile
    model, params, views, road = build_roadmap_pair(3, 16, 8, 16, 20, dtype="bf16")
    for p in model.parameters():
        p.requires_grad_(False)
    v = views.cuda().requires_grad_()
    with cpu_rng_dropout():
        torch.manual_seed(3)
        loss = model._run_step((v, None, tuple(road.cuda().unbind(0))), 1, "train")[0]
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            loss.backward()
            torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    # the c1 image gradient ran on the tensor cores (MODE 2 of the stride-1 kernel)
    assert any("s1_tc_kernel<2" in n or "s1_tc_kernelILi2E" in n for n in names), names
    bad = [n for n in names if "wgrad" in n or "bwd_adam" in n]
    assert not bad, bad
    assert v.grad is not None


def test_training_step_launches_one_kernel_more_with_views_grad(lib):
    """bf16 training step (all weights trainable): views that require grad add exactly the c1 image gradient."""
    model, params, views, road = build_roadmap_pair(3, 16, 8, 16, 20, dtype="bf16")
    counts = []
    for req in (False, True, False):
        for p in model.parameters():
            p.grad = None
        v = views.cuda().requires_grad_(req)
        with cpu_rng_dropout():
            torch.manual_seed(3)
            n0 = lib.launch_count()
            out = model.training_step((v, None, tuple(road.cuda().unbind(0))), 1)
            out["loss"].backward()
            torch.cuda.synchronize()
            counts.append(lib.launch_count() - n0)
        assert (v.grad is not None) == req
    print("launches per step without / with views.grad:", counts[0], counts[1])
    assert counts[0] == counts[2] and counts[1] == counts[0] + 1


# ----------------------------------------------------------------------------- the other models -----------------
def test_basic_ae_views_grad_fp32(golden):
    from driving_dirty_b200.autoencoder.autoencoder import BasicAE, default_hparams
    g = golden("ae_small")
    hp = default_hparams(hidden_dim=g["hidden"], latent_dim=g["latent"], input_width=6 * g["view_w"],
                         input_height=g["view_h"], output_width=g["view_w"], output_height=g["view_h"])
    ae = BasicAE(hp)
    ae.load_state_dict(g["state_dict"])
    ae = ae.cuda().train()
    views, _ = so.synthetic_scene_batch(g["batch"], g["view_h"], g["view_w"], map_hw=8, seed=777)
    v = views.cuda().requires_grad_()
    with cpu_rng_dropout():
        np.random.seed(4321)
        torch.manual_seed(99)
        loss = ae._run_step(v, 0, "train")
        loss.backward()
        p = {k: t.clone() for k, t in g["state_dict"].items()}
        r = views.clone().requires_grad_()
        with differentiable_oracle():
            ref = so.ae_run_step(p, r, g["slot"], True, (ae.decoder.deconv_dim_h, ae.decoder.deconv_dim_w), seed=99)
        ref["loss"].backward()
    lref = float(ref["loss"].detach())
    assert abs(float(loss.detach()) - lref) < 1e-5 * max(1.0, lref)
    err = rel_max_err(v.grad, r.grad)
    print("ae views.grad rel-max", err)
    # B = 3 batch-statistics BatchNorm amplifies fp32 summation-order noise (see test_ae_train_step_fp32_against_golden)
    assert err < 5e-4, err


def test_bb_views_and_road_map_grad_fp32(golden):
    """views.grad from both branches (the encoder's c1 image gradient and the six camera extractions) and rm.grad at full
    geometry, under one fixed random upstream gradient on the predicted occupancy map.  Measured against the oracle run in
    float64 (the exact gradient to fp32 precision): these gradients are sums of strongly cancelling terms, so the fp32
    oracle itself is 5e-3 to 7e-3 of max|exact| away from them (on the B200, with the merging CNN's backward that predates
    this test carrying rm.grad as far off as views.grad); the product must be no farther from the exact gradient than
    twice the fp32 reference's own error."""
    from tests.test_modules_gpu import _bb_batch, _bb_model
    g = golden("bb_full_b1")
    model, params = _bb_model(g)
    model.ae.unfreeze()
    views, road, _ = _bb_batch(g)
    v = views.cuda().requires_grad_()
    rm = road.cuda().float().unsqueeze(1).requires_grad_()
    pred = model(v, rm)
    up = torch.randn(pred.shape, generator=torch.Generator().manual_seed(17))
    (pred * up.cuda()).sum().backward()

    def oracle(dtype):
        p = {k: (t.to(dtype) if t.is_floating_point() else t) for k, t in params.items()}
        r = views.detach().to(dtype).clone().requires_grad_()
        rmr = road.detach().to(dtype).unsqueeze(1).clone().requires_grad_()
        with differentiable_oracle():
            pr = so.bb_forward(p, r, rmr)
        (pr * up.to(dtype)).sum().backward()
        return pr, r.grad, rmr.grad

    pr32, gv32, grm32 = oracle(torch.float32)
    pr64, gv64, grm64 = oracle(torch.float64)
    assert rel_max_err(pred, pr64) < 1e-5
    errs = {}
    for name, got, ref32, exact in (("views", v.grad, gv32, gv64), ("rm", rm.grad, grm32, grm64)):
        errs[name] = (rel_max_err(got, exact), rel_max_err(ref32, exact))
        print(f"bb {name}.grad rel-max against float64: product {errs[name][0]:.2e}, fp32 oracle {errs[name][1]:.2e}")
    for name, (ours, ref) in errs.items():
        assert ours < max(2 * ref, 1e-5), (name, ours, ref)
