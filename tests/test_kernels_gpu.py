"""Kernel-level parity: every C-ABI entry point against the CPU oracle on the same seeded inputs.
Bit-exact for index / byte / count work; fp32 within 1e-5 and bf16 within 1e-2 of max|ref|."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import scene_oracle as so
from tests.helpers import rel_max_err

pytestmark = pytest.mark.gpu

FP32_TOL = 1e-5
BF16_TOL = 1e-2


@pytest.fixture(scope="module")
def dd():
    from driving_dirty_b200 import _lib, ops
    assert torch.cuda.is_available()
    _lib.load()
    return ops


def nhwc(x_nchw, dtype):
    return x_nchw.permute(0, 2, 3, 1).contiguous().to(dtype).cuda()


def to_nchw(x_nhwc):
    return x_nhwc.float().permute(0, 3, 1, 2).contiguous().cpu()


def q(x, dtype):
    """round-trip through the storage dtype so the oracle sees what the kernel reads"""
    return x.to(dtype).float()


def init_from(mod, g):
    """torch's default Conv2d / ConvTranspose2d initialisation (uniform in +-1/sqrt(fan_in)) drawn from the test's own
    generator: with the global RNG the layer would depend on which tests ran before it in the same process."""
    bound = mod.weight[0].numel() ** -0.5
    with torch.no_grad():
        for t in (mod.weight, mod.bias):
            t.copy_((torch.rand(t.shape, generator=g) * 2 - 1) * bound)


# ------------------------------------------------------------------------------- stitch ------
@pytest.mark.parametrize("B,H,W", [(1, 4, 6), (3, 16, 20), (2, 5, 7), (2, 256, 306)])
def test_stitch_bit_exact(dd, B, H, W):
    views, _ = so.synthetic_scene_batch(B, H, W, map_hw=4, seed=11)
    ref = so.stitch(views)
    out = dd.stitch(views.cuda())
    assert torch.equal(out.cpu(), ref)
    # tuple input (collate_fn form), zero-copy and copying variants
    vc = views.cuda()
    assert torch.equal(dd.stitch(tuple(vc.unbind(0))).cpu(), ref)
    assert torch.equal(dd.stitch(tuple(t.clone() for t in vc.unbind(0))).cpu(), ref)


@pytest.mark.parametrize("slot", [0, 2, 4, 5])
def test_stitch_mask_bit_exact(dd, slot):
    views, _ = so.synthetic_scene_batch(2, 16, 20, map_hw=4, seed=12)
    xr, yr = so.six_to_one(views, slot)
    x, y = dd.stitch_mask(views.cuda(), slot)
    assert torch.equal(x.cpu(), xr) and torch.equal(y.cpu(), yr)


def test_stitch_u8_matches_to_tensor(dd):
    g = torch.Generator().manual_seed(1)
    u8 = torch.randint(0, 256, (2, 6, 3, 9, 10), dtype=torch.uint8, generator=g)
    ref = so.stitch(u8.float() / 255)
    assert torch.equal(dd.stitch_u8(u8.cuda()).cpu(), ref)


def test_stitch_empty_batch(dd):
    out = dd.stitch(torch.zeros(0, 6, 3, 4, 6, device="cuda"))
    assert out.shape == (0, 3, 4, 36)


# ------------------------------------------------------------------------------- convs -------
def _conv_inputs(B, H, W, seed, cin=32):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, cin, H, W, generator=g)
    w = (torch.rand(32, cin, 3, 3, generator=g) * 2 - 1) / (cin * 9) ** 0.5
    b = (torch.rand(32, generator=g) * 2 - 1) * 0.1
    return x, w, b


def _call_conv_fwd(dd, x, w, b, dtype, stride, impl=1):
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    B, _, H, W = x.shape
    xin = nhwc(x, dtype)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    out = torch.empty(B, Ho, Wo, 32, dtype=dtype, device="cuda")
    wc, bc = w.cuda(), b.cuda()
    call("dd_conv3x3_c32_fwd", xin.data_ptr(), wc.data_ptr(), bc.data_ptr(), out.data_ptr(), dtype_code(dtype),
         B, H, W, stride, impl, stream_ptr())
    return to_nchw(out)


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
@pytest.mark.parametrize("B,H,W,stride", [(2, 16, 120, 1), (2, 16, 120, 2), (1, 10, 84, 2), (1, 9, 35, 1),
                                           (1, 7, 33, 2), (1, 64, 200, 1)])
def test_conv3x3_fwd_simt(dd, dtype, tol, B, H, W, stride):
    x, w, b = _conv_inputs(B, H, W, seed=20 + H)
    ref = F.relu(F.conv2d(q(x, dtype), w, b, stride=stride, padding=1))
    out = _call_conv_fwd(dd, x, w, b, dtype, stride)
    assert rel_max_err(out, ref) < tol


TC_SHAPES = [(2, 16, 120, 1), (2, 16, 120, 2), (1, 10, 84, 2), (1, 9, 35, 1), (1, 7, 33, 2), (1, 64, 200, 1),
             (1, 70, 300, 2), (2, 256, 1836, 1), (2, 256, 1836, 2), (1, 40, 129, 1), (1, 33, 257, 2)]


@pytest.mark.parametrize("B,H,W,stride", TC_SHAPES)
def test_conv3x3_fwd_tcgen05(dd, B, H, W, stride):
    """tcgen05/TMEM implicit-GEMM forward (bf16 operands, fp32 accumulate) against the oracle conv on
    the same bf16-rounded inputs and weights; the full-size cases run 240 work items over 148 CTAs
    (persistent loop, slab-ring and accumulator-ring wrap-around)."""
    x, w, b = _conv_inputs(B, H, W, seed=20 + H)
    ref = F.relu(F.conv2d(q(x, torch.bfloat16), q(w, torch.bfloat16), b, stride=stride, padding=1))
    out = _call_conv_fwd(dd, x, w, b, torch.bfloat16, stride, impl=2)
    assert rel_max_err(out, ref) < 5e-3      # one bf16 rounding of the output
    simt = _call_conv_fwd(dd, x, w, b, torch.bfloat16, stride, impl=1)
    assert rel_max_err(out, simt) < BF16_TOL


@pytest.mark.parametrize("B,H,W,stride", [(2, 16, 120, 1), (1, 9, 35, 1), (1, 64, 200, 1), (2, 256, 1836, 1),
                                           (1, 40, 129, 1), (2, 16, 120, 2), (1, 9, 35, 2), (1, 10, 84, 2),
                                           (1, 64, 515, 2), (2, 256, 1836, 2), (1, 33, 258, 2)])
def test_conv3x3_dgrad_tcgen05(dd, B, H, W, stride):
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    dtype = torch.bfloat16
    x, w, b = _conv_inputs(B, H, W, seed=40 + H)
    x = F.relu(x)
    xq = q(x, dtype).requires_grad_(True)
    y = F.conv2d(xq, q(w, dtype), None, stride=stride, padding=1)
    g = torch.Generator().manual_seed(5)
    dy = q(torch.randn(y.shape, generator=g), dtype)
    y.backward(dy)
    dx_ref = xq.grad * (xq.detach() > 0)
    xin, dyin = nhwc(x, dtype), nhwc(dy, dtype)
    dx = torch.empty_like(xin)
    wc = w.cuda()
    call("dd_conv3x3_c32_dgrad", dyin.data_ptr(), wc.data_ptr(), xin.data_ptr(), dx.data_ptr(), dtype_code(dtype),
         B, H, W, stride, 2, stream_ptr())
    assert rel_max_err(to_nchw(dx), dx_ref) < 5e-3
    call("dd_conv3x3_c32_dgrad", dyin.data_ptr(), wc.data_ptr(), None, dx.data_ptr(), dtype_code(dtype),
         B, H, W, stride, 2, stream_ptr())
    assert rel_max_err(to_nchw(dx), xq.grad) < 5e-3


@pytest.mark.parametrize("B,H,W,stride", [(2, 16, 120, 1), (1, 9, 35, 1), (1, 64, 200, 1), (2, 256, 1836, 1),
                                           (1, 40, 129, 1), (3, 5, 131, 1), (2, 16, 120, 2), (1, 9, 35, 2),
                                           (1, 10, 84, 2), (1, 64, 515, 2), (2, 256, 1836, 2), (3, 5, 131, 2)])
def test_conv3x3_wgrad_tcgen05(dd, B, H, W, stride):
    """tcgen05 weight gradient (pixels as the contraction axis, MN-major operands) against autograd on
    the same bf16-rounded x / dy; fp32 accumulation, deterministic ordered reduction."""
    from driving_dirty_b200._lib import call, dtype_code, load, stream_ptr
    dtype = torch.bfloat16
    x, w, b = _conv_inputs(B, H, W, seed=40 + H)
    xq = q(F.relu(x), dtype)
    wq, bq = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = F.conv2d(xq, wq, bq, stride=stride, padding=1)
    g = torch.Generator().manual_seed(5)
    dy = q(torch.randn(y.shape, generator=g), dtype)
    y.backward(dy)
    n = int(load().dd_conv_wgrad_workspace_bytes())
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    xin, dyin = nhwc(xq, dtype), nhwc(dy, dtype)
    outs = []
    for _ in range(2):
        dw, db = torch.empty(32, 32, 3, 3, device="cuda"), torch.empty(32, device="cuda")
        call("dd_conv3x3_c32_wgrad", xin.data_ptr(), dyin.data_ptr(), dw.data_ptr(), db.data_ptr(), ws.data_ptr(), n,
             dtype_code(dtype), B, H, W, stride, 2, stream_ptr())
        outs.append((dw.clone(), db.clone()))
    assert rel_max_err(outs[0][0], wq.grad) < 2e-4
    assert rel_max_err(outs[0][1], bq.grad) < 2e-4
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1])   # run-to-run identical


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
@pytest.mark.parametrize("B,H,W,stride", [(2, 16, 120, 1), (2, 16, 120, 2), (1, 10, 84, 2), (1, 9, 35, 1),
                                           (1, 7, 33, 2), (1, 9, 35, 2)])
def test_conv3x3_dgrad_wgrad_simt(dd, dtype, tol, B, H, W, stride):
    from driving_dirty_b200._lib import call, dtype_code, load, stream_ptr
    x, w, b = _conv_inputs(B, H, W, seed=40 + H)
    x = F.relu(x)                      # the layer input is a post-ReLU activation
    xq = q(x, dtype).requires_grad_(True)
    wq = w.clone().requires_grad_(True)
    bq = b.clone().requires_grad_(True)
    y = F.conv2d(xq, wq, bq, stride=stride, padding=1)
    g = torch.Generator().manual_seed(5)
    dy = q(torch.randn(y.shape, generator=g), dtype)
    y.backward(dy)
    dx_ref = xq.grad * (xq.detach() > 0)          # mask by the input activation (previous ReLU)
    code, st = dtype_code(dtype), stream_ptr()
    xin, dyin = nhwc(x, dtype), nhwc(dy, dtype)
    dx = torch.empty_like(xin)
    wc = w.cuda()
    call("dd_conv3x3_c32_dgrad", dyin.data_ptr(), wc.data_ptr(), xin.data_ptr(), dx.data_ptr(), code, B, H, W,
         stride, 1, st)
    assert rel_max_err(to_nchw(dx), dx_ref) < tol
    # no-mask variant
    call("dd_conv3x3_c32_dgrad", dyin.data_ptr(), wc.data_ptr(), None, dx.data_ptr(), code, B, H, W, stride, 1, st)
    assert rel_max_err(to_nchw(dx), xq.grad) < tol
    n = int(load().dd_conv_wgrad_workspace_bytes())
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    dw, db = torch.empty(32, 32, 3, 3, device="cuda"), torch.empty(32, device="cuda")
    call("dd_conv3x3_c32_wgrad", xin.data_ptr(), dyin.data_ptr(), dw.data_ptr(), db.data_ptr(), ws.data_ptr(), n,
         code, B, H, W, stride, 1, st)
    assert rel_max_err(dw, wq.grad) < tol
    assert rel_max_err(db, bq.grad) < tol


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
@pytest.mark.parametrize("B,H,W", [(2, 16, 20), (1, 10, 14), (1, 33, 7), (2, 40, 50)])
@pytest.mark.parametrize("impl", [1, 2])
def test_conv_c1_fwd_and_wgrad(dd, dtype, tol, B, H, W, impl):
    if impl == 2 and dtype == torch.float32:
        pytest.skip("tcgen05 conv is bf16 only")
    from driving_dirty_b200._lib import call, dtype_code, load, stream_ptr
    views, _ = so.synthetic_scene_batch(B, H, W, map_hw=4, seed=31)
    _, w, b = _conv_inputs(1, 4, 4, seed=32, cin=3)
    mosaic = so.stitch(views)
    wq, bq = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = F.relu(F.conv2d(mosaic, wq, bq, padding=1))
    code, st = dtype_code(dtype), stream_ptr()
    Wm = 6 * W
    wc, bc = w.cuda(), b.cuda()
    outs = []
    for is_views, src in ((1, views.cuda()), (0, mosaic.cuda())):
        out = torch.empty(B, H, Wm, 32, dtype=dtype, device="cuda")
        call("dd_conv_c1_fwd", src.data_ptr(), is_views, wc.data_ptr(), bc.data_ptr(), out.data_ptr(), code, B, H, Wm,
             impl, st)
        assert rel_max_err(to_nchw(out), y) < tol
        outs.append(out)
    assert torch.equal(outs[0], outs[1])     # folding the stitch changes nothing
    g = torch.Generator().manual_seed(6)
    dy = q(torch.randn(y.shape, generator=g), dtype) * (y.detach() > 0)
    y.backward(dy)
    n = int(load().dd_conv_wgrad_workspace_bytes())
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    dyin = nhwc(dy, dtype)
    for is_views, src in ((1, views.cuda()), (0, mosaic.cuda())):
        dw, db = torch.empty(32, 3, 3, 3, device="cuda"), torch.empty(32, device="cuda")
        call("dd_conv_c1_wgrad", src.data_ptr(), is_views, dyin.data_ptr(), code, dw.data_ptr(), db.data_ptr(),
             ws.data_ptr(), n, B, H, Wm, impl, st)
        assert rel_max_err(dw, wq.grad) < tol
        assert rel_max_err(db, bq.grad) < tol


@pytest.mark.parametrize("B,H,W", [(2, 16, 20), (1, 33, 7), (2, 70, 50), (2, 256, 306)])
def test_conv_c1_tcgen05_raw_bytes_and_full_size(dd, B, H, W):
    """The u8 front-end (data_helper.py:109-114 ToTensor folded into c1's loads, DD_IN_U8): forward and weight gradient
    from raw camera bytes are BIT-IDENTICAL to the same kernels fed ``bytes.float() / 255`` -- and the fp32 forms agree
    with autograd, here also at the full 256 x 1836 mosaic (several row segments and column strips per CTA)."""
    from driving_dirty_b200._lib import call, dtype_code, load, stream_ptr
    g = torch.Generator().manual_seed(33)
    raw = torch.randint(0, 256, (B, 6, 3, H, W), dtype=torch.uint8, generator=g)
    views = raw.float() / 255                               # what ToTensor hands the reference
    _, w, b = _conv_inputs(1, 4, 4, seed=32, cin=3)
    mosaic = so.stitch(views)
    wq, bq = w.clone().requires_grad_(True), b.clone().requires_grad_(True)
    y = F.relu(F.conv2d(mosaic, wq, bq, padding=1))
    dtype, Wm, st = torch.bfloat16, 6 * W, stream_ptr()
    code = dtype_code(dtype)
    wc, bc = w.cuda(), b.cuda()
    outs = []
    for flags, src in ((1, views.cuda()), (3, raw.cuda()), (2, so.stitch(raw).cuda())):
        out = torch.empty(B, H, Wm, 32, dtype=dtype, device="cuda")
        call("dd_conv_c1_fwd", src.data_ptr(), flags, wc.data_ptr(), bc.data_ptr(), out.data_ptr(), code, B, H, Wm, 2, st)
        outs.append(out)
    assert rel_max_err(to_nchw(outs[0]), y) < BF16_TOL
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    dy = q(torch.randn(y.shape, generator=g), dtype) * (y.detach() > 0)
    y.backward(dy)
    n = int(load().dd_conv_wgrad_workspace_bytes())
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    dyin = nhwc(dy, dtype)
    res = []
    for flags, src in ((1, views.cuda()), (3, raw.cuda()), (2, so.stitch(raw).cuda()), (3, raw.cuda())):
        dw, db = torch.empty(32, 3, 3, 3, device="cuda"), torch.empty(32, device="cuda")
        call("dd_conv_c1_wgrad", src.data_ptr(), flags, dyin.data_ptr(), code, dw.data_ptr(), db.data_ptr(),
             ws.data_ptr(), n, B, H, Wm, 2, st)
        res.append((dw.clone(), db.clone()))
    assert rel_max_err(res[0][0], wq.grad) < BF16_TOL and rel_max_err(res[0][1], bq.grad) < 2e-4
    for dw, db in res[1:]:
        assert torch.equal(dw, res[0][0]) and torch.equal(db, res[0][1])      # same bits from bytes, run to run
    # the fp32 parity path refuses raw bytes instead of misreading them
    with pytest.raises(RuntimeError):
        call("dd_conv_c1_fwd", raw.cuda().data_ptr(), 3, wc.data_ptr(), bc.data_ptr(),
             torch.empty(B, H, Wm, 32, device="cuda").data_ptr(), dtype_code(torch.float32), B, H, Wm, 0, st)


@pytest.mark.parametrize("B,H,W", [(2, 16, 20), (1, 33, 7), (2, 70, 50), (1, 1, 22), (3, 130, 43), (2, 256, 306)])
def test_encoder_c1c2_fused_bit_identical(dd, B, H, W):
    """dd_encoder_c1c2_fused_fwd (inference: the first activation never leaves the SM) against the two-kernel tensor-core
    path it replaces: BIT-IDENTICAL a2 (a1 is rounded to bf16 at the same point and the MMAs see the same operands in the
    same order), for views, raw bytes and a mosaic, ragged strips (Wm % 126 != 0), short / single rows and several row
    segments; and within bf16 tolerance of the fp32 reference convs (components.py:41-43)."""
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    g = torch.Generator().manual_seed(35 + H)
    raw = torch.randint(0, 256, (B, 6, 3, H, W), dtype=torch.uint8, generator=g)
    views = raw.float() / 255
    _, w1, b1 = _conv_inputs(1, 4, 4, seed=36, cin=3)
    _, w2, b2 = _conv_inputs(1, 4, 4, seed=37)
    Wm, st, code = 6 * W, stream_ptr(), dtype_code(torch.bfloat16)
    w1c, b1c, w2c, b2c = w1.cuda(), b1.cuda(), w2.cuda(), b2.cuda()
    vd = views.cuda()
    a1 = torch.empty(B, H, Wm, 32, dtype=torch.bfloat16, device="cuda")
    a2 = torch.empty_like(a1)
    call("dd_conv_c1_fwd", vd.data_ptr(), 1, w1c.data_ptr(), b1c.data_ptr(), a1.data_ptr(), code, B, H, Wm, 2, st)
    call("dd_conv3x3_c32_fwd", a1.data_ptr(), w2c.data_ptr(), b2c.data_ptr(), a2.data_ptr(), code, B, H, Wm, 1, 2, st)
    ref = F.relu(F.conv2d(F.relu(F.conv2d(so.stitch(views), w1, b1, padding=1)), w2, b2, padding=1))
    assert rel_max_err(to_nchw(a2), ref) < BF16_TOL
    for flags, src in ((1, vd), (3, raw.cuda()), (2, so.stitch(raw).cuda()), (0, so.stitch(views).cuda())):
        fused = torch.full_like(a2, float("nan"))
        call("dd_encoder_c1c2_fused_fwd", src.data_ptr(), flags, w1c.data_ptr(), b1c.data_ptr(), w2c.data_ptr(), b2c.data_ptr(),
             fused.data_ptr(), B, H, Wm, st)
        assert torch.equal(fused.view(torch.int16), a2.view(torch.int16)), f"flags {flags}"


# ------------------------------------------------------------------------------- pool --------
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,H,W", [(2, 8, 60), (2, 5, 42), (1, 3, 7), (1, 128, 918)])
def test_pool4_fwd_bwd_exact(dd, dtype, B, H, W):
    from driving_dirty_b200._lib import call, dtype_code, stream_ptr
    g = torch.Generator().manual_seed(50)
    a3 = q(F.relu(torch.randn(B, 32, H, W, generator=g)), dtype)
    ref = so.pool4_flat(a3)
    code, st = dtype_code(dtype), stream_ptr()
    a3d = nhwc(a3, dtype)
    n_out = (32 * H * W) // 4
    pooled = torch.empty(B, n_out, dtype=dtype, device="cuda")
    call("dd_pool4_fwd", a3d.data_ptr(), pooled.data_ptr(), code, B, H, W, st)
    assert torch.equal(pooled.float().cpu(), ref)          # max of stored values: exact in any dtype
    pooled32 = torch.empty(B, n_out, dtype=torch.float32, device="cuda")      # the inference path's fp32 features
    call("dd_pool4_fwd_f32", a3d.data_ptr(), pooled32.data_ptr(), code, B, H, W, st)
    assert torch.equal(pooled32.cpu(), ref)
    # backward: route to the FIRST max, times relu'(a3)
    a3r = a3.clone().requires_grad_(True)
    p = F.max_pool1d(F.relu(a3r).reshape(B, -1).unsqueeze(1), 4).squeeze(1)
    dp = q(torch.randn(p.shape, generator=g), dtype)
    p.backward(dp)
    da3 = torch.empty_like(a3d)
    dpd = dp.to(dtype).cuda()
    call("dd_pool4_bwd", a3d.data_ptr(), dpd.data_ptr(), da3.data_ptr(), code, B, H, W, st)
    assert torch.equal(to_nchw(da3), a3r.grad)


def test_layout_round_trip(dd):
    from driving_dirty_b200._lib import call, stream_ptr
    x = torch.randn(2, 32, 5, 7)
    xd = x.cuda()
    nh = torch.empty(2, 5, 7, 32, device="cuda")
    call("dd_nchw_f32_to_nhwc", xd.data_ptr(), nh.data_ptr(), 0, 2, 32, 5, 7, stream_ptr())
    assert torch.equal(nh.cpu(), x.permute(0, 2, 3, 1).contiguous())
    back = torch.empty_like(xd)
    call("dd_nhwc_to_nchw_f32", nh.data_ptr(), 0, back.data_ptr(), 2, 32, 5, 7, stream_ptr())
    assert torch.equal(back.cpu(), x)


# ------------------------------------------------------------------------------- linear ------
@pytest.mark.parametrize("xdtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, FP32_TOL)])
@pytest.mark.parametrize("B,N,K", [(3, 16, 3840), (32, 256, 8192), (5, 5000, 8), (32, 4096, 128), (2, 24, 1680),
                                    (40, 64, 1024), (1, 7, 12), (8, 130, 2052)])
def test_linear_fwd_dgrad_wgrad(dd, xdtype, tol, B, N, K):
    g = torch.Generator().manual_seed(60 + B)
    x = q(torch.randn(B, K, generator=g), xdtype).requires_grad_(True)
    w = ((torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5).requires_grad_(True)
    b = ((torch.rand(N, generator=g) * 2 - 1) * 0.1).requires_grad_(True)
    y = F.linear(x, w, b)
    dy = torch.randn(B, N, generator=g)
    y.backward(dy)
    xd = x.detach().to(xdtype).cuda().requires_grad_(True)
    wd = w.detach().cuda().requires_grad_(True)
    bd = b.detach().cuda().requires_grad_(True)
    yd = dd.linear(xd, wd, bd, impl=1)
    assert rel_max_err(yd, y) < tol
    yd.backward(dy.cuda())
    # dx is stored in the activation dtype
    assert rel_max_err(xd.grad, x.grad) < (tol if xdtype == torch.float32 else BF16_TOL)
    assert rel_max_err(wd.grad, w.grad) < tol
    assert rel_max_err(bd.grad, b.grad) < tol


TF32_TOL = 2e-3   # tf32 operands (10-bit mantissa) on the weight-streaming tensor-core path


@pytest.mark.parametrize("xdtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("B,N,K", [(32, 256, 16384 + 64), (5, 1028, 4100), (32, 66000, 128), (3, 640000, 8),
                                    (32, 16, 300000), (40, 4096, 1024), (32, 256, 940032)])
def test_linear_tcgen05_fwd_dgrad_wgrad(dd, xdtype, B, N, K):
    """TMA-fed tcgen05 (tf32) weight-streaming kernels against torch's fp32 CPU linear and autograd."""
    g = torch.Generator().manual_seed(61 + B)
    x = q(torch.randn(B, K, generator=g), xdtype).requires_grad_(True)
    w = ((torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5).requires_grad_(True)
    b = ((torch.rand(N, generator=g) * 2 - 1) * 0.1).requires_grad_(True)
    y = F.linear(x, w, b)
    dy = torch.randn(B, N, generator=g)
    y.backward(dy)
    xd = x.detach().to(xdtype).cuda().requires_grad_(True)
    wd = w.detach().cuda().requires_grad_(True)
    bd = b.detach().cuda().requires_grad_(True)
    yd = dd.linear(xd, wd, bd, impl=2)
    assert rel_max_err(yd, y) < TF32_TOL
    yd.backward(dy.cuda())
    assert rel_max_err(xd.grad, x.grad) < (TF32_TOL if xdtype == torch.float32 else BF16_TOL)
    assert rel_max_err(wd.grad, w.grad) < TF32_TOL
    assert rel_max_err(bd.grad, b.grad) < FP32_TOL
    # deterministic: the split reductions are ordered
    xd2 = x.detach().to(xdtype).cuda().requires_grad_(True)
    yd2 = dd.linear(xd2, wd, bd, impl=2)
    assert torch.equal(yd2, yd)


@pytest.mark.parametrize("B", [33, 64, 100, 128, 200, 256, 300])
@pytest.mark.parametrize("N,K", [(256, 32768 + 96), (33000, 128), (1028, 4100)])
def test_linear_tcgen05_fwd_wide_batch(dd, B, N, K):
    """Inference batches: up to 256 rows share ONE pass over the weights (MMA N = 64 / 128 / 256); more are chunked by 256.
    Same values as the 32-row passes of the training step to tf32 accuracy, deterministic."""
    g = torch.Generator().manual_seed(67 + B)
    x = torch.randn(B, K, generator=g)
    w = (torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5
    b = (torch.rand(N, generator=g) * 2 - 1) * 0.1
    y = F.linear(x, w, b)
    with torch.no_grad():
        yd = dd.linear(x.cuda(), w.cuda(), b.cuda(), impl=2)
        assert rel_max_err(yd, y) < TF32_TOL
        assert torch.equal(dd.linear(x.cuda(), w.cuda(), b.cuda(), impl=2), yd)
        # rows do not mix: any 32-row slice run on its own gives the same bits (same k order, same split plan per tile)
        y32 = dd.linear(x[:32].cuda(), w.cuda(), b.cuda(), impl=2)
        assert rel_max_err(yd[:32], y32) < 1e-6


# ------------------------------------------------------------------------------- loss / TS ---
def _ref_loss_bundle(logits, target):
    probs = torch.sigmoid(logits)
    return dict(loss=F.binary_cross_entropy_with_logits(logits.view(logits.shape[0], -1),
                                                        target.view(target.shape[0], -1)),
                probs=probs, binary=probs.round(), ts=so.threat_score(target, probs),
                ts_r=so.threat_score(target, probs.round()))


@pytest.mark.parametrize("shape", [(2, 800, 800), (3, 37, 41), (1, 1, 5), (26, 800, 800)])
@pytest.mark.parametrize("u8", [False, True])
def test_bce_threat_forward_backward(dd, shape, u8):
    g = torch.Generator().manual_seed(70)
    logits = torch.randn(shape, generator=g) * 0.06          # the scale random-init logits have
    flat = logits.view(-1)
    flat[:: 97] = 0.0
    flat[1:: 89] *= 1e-6                                      # crowd the binarise threshold
    target_b = torch.rand(shape, generator=g) > 0.5
    target = target_b.float()
    ref = _ref_loss_bundle(logits, target)
    ld = logits.cuda().requires_grad_(True)
    loss, probs, binary, stats, counts = dd.bce_threat(ld, target_b.cuda() if u8 else target.cuda())
    assert abs(float(loss) - float(ref["loss"])) < 1e-6 * max(1.0, abs(float(ref["loss"])))
    assert rel_max_err(probs, ref["probs"]) < 3e-7                       # IEEE sigmoid: a last place or two of 0.5
    assert torch.equal(binary.cpu().float(), ref["binary"])             # bit-exact binarisation
    # forward()'s contract (roadmap_bce_v2.py:72,81,140): rounding the RETURNED probabilities gives the binary map
    assert torch.equal(probs.round(), binary.float())
    assert torch.equal(probs.cpu().round(), ref["probs"].round())
    tp, nt, nr = so.threat_score_counts(target, ref["binary"])
    assert counts.cpu().tolist() == [nt, nr, tp, logits.numel()]        # exact integer counts
    assert float(stats[2]) == float(ref["ts_r"])                        # bit-exact rounded TS (<= 26 scenes)
    assert abs(float(stats[1]) - float(ref["ts"])) < 2e-6
    lr = logits.clone().requires_grad_(True)
    F.binary_cross_entropy_with_logits(lr.view(shape[0], -1), target.view(shape[0], -1)).backward()
    (loss * 1.0).backward()
    assert rel_max_err(ld.grad, lr.grad) < 1e-6
    assert rel_max_err(ld.grad, so.bce_with_logits_grad(logits, target)) < 1e-6


def test_binarise_exhaustive_sweep(dd, golden):
    """Every fp32 in [2^-27, 2^-20): the kernel's binary map equals the reference's
    sigmoid().round() (goldens: first 1 at bits 0x33C00001), plus the edge cases."""
    gold = golden("binarise")
    bits = np.arange(gold["sweep_lo"], gold["sweep_hi"], dtype=np.uint32)
    n = (len(bits) // 4) * 4
    x = torch.from_numpy(bits[:n].view(np.float32).copy())
    probs, binary = dd.sigmoid_binary(x.cuda())
    assert torch.equal(probs.round(), binary.float())                    # over the whole sweep, on the device
    assert torch.equal(probs.cpu().round(), torch.sigmoid(x).round())    # and against the reference's own arithmetic
    got = binary.cpu()
    first = int(torch.nonzero(got).flatten()[0])
    assert int(bits[first]) == gold["first_one_bits"]
    assert bool((got[first:] == 1).all()) and bool((got[:first] == 0).all())
    e = gold["edge_x"]
    e = torch.cat([e, e[:2]])[:16]
    p, b = dd.sigmoid_binary(e.cuda())
    assert torch.equal(p.round(), b.float())
    assert torch.equal(b.cpu().float()[:14], gold["edge_round"])
    assert rel_max_err(p.cpu()[:12], gold["edge_sigmoid"][:12]) < 1e-6
    # negatives never binarise to 1
    _, bn = dd.sigmoid_binary((-x[: 1 << 20]).cuda())
    assert int(bn.sum()) == 0


def test_bce_threat_soft_target(dd):
    """compute_ts_road_map (helper.py:74-77) sums VALUES: a soft (augmented) target must give the reference's score,
    for the soft and for the rounded prediction."""
    g = torch.Generator().manual_seed(71)
    logits = torch.randn(3, 64, 64, generator=g)
    target = torch.rand(3, 64, 64, generator=g)
    loss, probs, binary, stats, counts = dd.bce_threat(logits.cuda(), target.cuda())
    p = torch.sigmoid(logits)
    assert abs(float(stats[1]) - float(so.threat_score(target, p))) < 2e-6
    assert abs(float(stats[2]) - float(so.threat_score(target, p.round()))) < 2e-6
    assert abs(float(loss) - float(F.binary_cross_entropy_with_logits(logits, target))) < 1e-6


def test_threat_score_and_mse(dd):
    g = torch.Generator().manual_seed(80)
    a, b = torch.rand(3, 100, 100, generator=g), (torch.rand(3, 100, 100, generator=g) > 0.5).float()
    assert abs(float(dd.threat_score(a.cuda(), b.cuda())) - float(so.threat_score(a, b))) < 1e-6
    z = torch.zeros(4, 4)
    assert torch.isnan(dd.threat_score(z.cuda(), z.cuda()))             # 0/0 like the reference
    y, yh = torch.randn(2, 3, 16, 20, generator=g), torch.randn(2, 3, 16, 20, generator=g)
    yhd = yh.cuda().requires_grad_(True)
    yhr = yh.clone().requires_grad_(True)
    lr = F.mse_loss(y, yhr)
    lr.backward()
    ld = dd.mse_loss(y.cuda(), yhd)
    ld.backward()
    assert abs(float(ld) - float(lr)) < 1e-6 and rel_max_err(yhd.grad, yhr.grad) < 1e-6


# ------------------------------------------------------------------------------- generic conv --
# one case per layer TYPE of the decoder (components.py:70-73) and of the bounding-box CNNs
# (spatial_bb/components.py:18-26,129-139), at reduced spatial size
GENERIC_LAYERS = {
    "dc1_convT_64_32_k3p1": dict(t=True, cin=64, cout=32, k=3, s=1, p=1, d=1, hw=(9, 11)),
    "dc3_convT_32_32_k2s2": dict(t=True, cin=32, cout=32, k=2, s=2, p=0, d=1, hw=(8, 10)),
    "dc4_convT_32_3_k1": dict(t=True, cin=32, cout=3, k=1, s=1, p=0, d=1, hw=(16, 20)),
    "strip_conv_3_32_1x50_s32": dict(t=False, cin=3, cout=32, k=(1, 50), s=(3, 2), p=0, d=1, hw=(20, 70)),
    "strip_conv_3_32_52x1_s32_p1": dict(t=False, cin=3, cout=32, k=(52, 1), s=(3, 2), p=1, d=1, hw=(64, 18)),
    "out_conv_32_32_k3_valid": dict(t=False, cin=32, cout=32, k=3, s=1, p=0, d=1, hw=(12, 13)),
    "rm_conv2_32_32_k3_d3": dict(t=False, cin=32, cout=32, k=3, s=1, p=0, d=3, hw=(14, 15)),
    "ss_conv_32_32_1x24_s17": dict(t=False, cin=32, cout=32, k=(1, 24), s=(1, 7), p=0, d=1, hw=(5, 66)),
    "rm_conv1_1_32_k7s3d3p1": dict(t=False, cin=1, cout=32, k=7, s=3, p=1, d=3, hw=(40, 43)),
    "up_conv1_convT_96_64_k7d7": dict(t=True, cin=96, cout=64, k=7, s=1, p=0, d=7, hw=(6, 7)),
    "up_conv4_convT_16_8_k7d3": dict(t=True, cin=16, cout=8, k=7, s=1, p=0, d=3, hw=(9, 8)),
    "up_conv5_convT_8_1_k2s2": dict(t=True, cin=8, cout=1, k=2, s=2, p=0, d=1, hw=(10, 11)),
}


@pytest.mark.parametrize("dtype,tol", [(torch.float32, FP32_TOL), (torch.bfloat16, BF16_TOL)])
@pytest.mark.parametrize("layer", sorted(GENERIC_LAYERS))
@pytest.mark.parametrize("relu", [False, True])
def test_conv2d_generic_fwd_dgrad_wgrad(dd, layer, dtype, tol, relu):
    """dd_conv2d_fwd / dgrad / wgrad against torch's CPU conv2d / conv_transpose2d and autograd."""
    L = GENERIC_LAYERS[layer]
    B = 2
    g = torch.Generator().manual_seed(sum(map(ord, layer)))
    mod_cls = torch.nn.ConvTranspose2d if L["t"] else torch.nn.Conv2d
    mod = mod_cls(L["cin"], L["cout"], kernel_size=L["k"], stride=L["s"], padding=L["p"], dilation=L["d"])
    init_from(mod, g)
    with torch.no_grad():
        # bf16 path: the tensor-core layers read their weights as bf16 operands; give the reference the same operands, or
        # outputs within rounding of zero flip their ReLU mask and the comparison measures the flips, not the kernel
        mod.weight.copy_(q(mod.weight, dtype))
    x = q(torch.randn(B, L["cin"], *L["hw"], generator=g), dtype).requires_grad_(True)
    y = mod(x)
    if relu:
        y = F.relu(y)
    dy = q(torch.randn(y.shape, generator=g), dtype)
    y.backward(dy)
    # device
    m2 = mod_cls(L["cin"], L["cout"], kernel_size=L["k"], stride=L["s"], padding=L["p"], dilation=L["d"]).cuda()
    m2.load_state_dict(mod.state_dict())
    xd = nhwc(x.detach(), dtype).requires_grad_(True)
    yd = dd.conv2d_nhwc(xd, m2, relu=relu)
    assert tuple(yd.shape) == (B, y.shape[2], y.shape[3], L["cout"])
    assert rel_max_err(to_nchw(yd.detach()), y) < tol
    yd.backward(nhwc(dy, dtype))
    assert rel_max_err(to_nchw(xd.grad), x.grad) < tol
    assert rel_max_err(m2.weight.grad, mod.weight.grad) < tol
    assert rel_max_err(m2.bias.grad, mod.bias.grad) < tol


TC_LAYERS = {
    # name: (transposed, cin, cout, k, pad, dil, (H, W), batch) -- every (gathered, produced) channel pair the tcgen05
    # implicit-GEMM kernel is instantiated for, at sizes with several column strips, row groups and residue classes
    "up_conv1_96_64_k7d7": (True, 96, 64, 7, 0, 7, (20, 150), 2),
    "up_conv2_64_32_k7d7": (True, 64, 32, 7, 0, 7, (30, 140), 2),
    "up_conv3_32_16_k7d7": (True, 32, 16, 7, 0, 7, (33, 100), 1),
    "up_conv4_16_8_k7d3": (True, 16, 8, 7, 0, 3, (37, 140), 2),     # all three passes through zero-padded 32-channel pixels
    "dc1_64_32_k3p1": (True, 64, 32, 3, 1, 1, (40, 153), 2),
    "dc2_32_32_k3p1": (True, 32, 32, 3, 1, 1, (128, 153), 1),
    "out_conv_32_32_k3": (False, 32, 32, 3, 0, 1, (50, 258), 2),
    "rm_conv2_32_32_k3d3": (False, 32, 32, 3, 0, 3, (41, 262), 1),
}


@pytest.mark.parametrize("layer", sorted(TC_LAYERS))
def test_conv2d_tcgen05_layers(dd, layer):
    """The tcgen05 implicit-GEMM path of dd_conv2d_fwd / dd_conv2d_dgrad (csrc/conv_dil_tc.cu: residue-class row groups, taps
    scattered over N, weight slabs streamed by TMA) against torch's CPU conv2d / conv_transpose2d and autograd on the same
    bf16-rounded operands: forward with bias + ReLU, input gradient with the ReLU mask of the layer input."""
    import ctypes
    from driving_dirty_b200 import _lib
    t, cin, cout, k, p, d, hw, B = TC_LAYERS[layer]
    dtype = torch.bfloat16
    g = torch.Generator().manual_seed(sum(map(ord, layer)))
    mod_cls = torch.nn.ConvTranspose2d if t else torch.nn.Conv2d
    mod = mod_cls(cin, cout, kernel_size=k, stride=1, padding=p, dilation=d)
    init_from(mod, g)
    with torch.no_grad():
        mod.weight.copy_(q(mod.weight, dtype))            # the kernel reads the weights as bf16 operands
    x = q(F.relu(torch.randn(B, cin, *hw, generator=g)), dtype).requires_grad_(True)
    y = F.relu(mod(x))
    dy = q(torch.randn(y.shape, generator=g), dtype)
    y.backward(dy)
    m2 = mod_cls(cin, cout, kernel_size=k, stride=1, padding=p, dilation=d).cuda()
    m2.load_state_dict(mod.state_dict())
    desc = _lib.ConvDesc(B, cin, cout, hw[0], hw[1], y.shape[2], y.shape[3], k, k, 1, 1, p, p, d, d, int(t))
    assert _lib.load().dd_conv2d_tc_supported(ctypes.byref(desc), 1, 0) == 1
    # tensors with 16 (up_conv_3's output) or 8 / 16 channels (up_conv_4) are below the kernels' 32-channel pixels: they are
    # zero-padded to 32 channels first, an 8-channel result is narrowed afterwards (conv_generic.cu, chan_pad32_kernel)
    assert _lib.load().dd_conv2d_tc_supported(ctypes.byref(desc), 1, 1) == 1
    assert _lib.load().dd_conv2d_tc_supported(ctypes.byref(desc), 1, 2) == 1
    assert _lib.load().dd_conv2d_tc_supported(ctypes.byref(desc), 0, 0) == 0          # fp32 stays on the CUDA-core parity engine
    xd = nhwc(x.detach(), dtype).requires_grad_(True)
    yd = dd.conv2d_nhwc(xd, m2, relu=True)
    assert tuple(yd.shape) == (B, y.shape[2], y.shape[3], cout)
    assert rel_max_err(to_nchw(yd.detach()), y) < 1e-2
    yd.backward(nhwc(dy, dtype))
    assert rel_max_err(to_nchw(xd.grad), x.grad) < 1e-2
    assert rel_max_err(m2.weight.grad, mod.weight.grad) < 1e-2
    # the ReLU mask of the layer input, fused into the input-gradient epilogue (dd_conv2d_dgrad's x_mask)
    st, code = _lib.stream_ptr(), 1
    n = int(_lib.load().dd_conv2d_workspace_bytes(ctypes.byref(desc)))
    ws = torch.empty(n, dtype=torch.uint8, device="cuda")
    dym = (nhwc(dy, dtype).float() * (yd.detach().float() > 0)).to(dtype)
    dxm = torch.empty_like(xd)
    _lib.call("dd_conv2d_dgrad", dym.data_ptr(), m2.weight.detach().float().contiguous().data_ptr(), xd.detach().data_ptr(),
              dxm.data_ptr(), ctypes.byref(desc), code, ws.data_ptr(), n, st)
    assert rel_max_err(to_nchw(dxm), x.grad * (x.detach() > 0)) < 1e-2


def test_relu_mask_ragged_tail(dd):
    from driving_dirty_b200._lib import call, stream_ptr
    g = torch.randn(1003, device="cuda")
    a = torch.randn(1003, device="cuda")
    out = torch.empty_like(g)
    call("dd_relu_mask", g.data_ptr(), a.data_ptr(), out.data_ptr(), 0, 1003, stream_ptr())
    assert torch.equal(out, g * (a > 0))


# ------------------------------------------------------------------------------- boxes -------
@pytest.mark.parametrize("n1,n2,seed", [(7, 9, 0), (20, 20, 1), (1, 5, 2), (33, 3, 3)])
def test_ats_bounding_boxes_matches_the_reference_loop(dd, n1, n2, seed):
    """compute_ats_bounding_boxes (helper.py:33-72) on the device against the line-by-line restatement (Python pair loop,
    float64 polygon stand-in for shapely): IoU matrix to 1e-6, the score bit for bit (integer counts and the reference's
    float32 arithmetic)."""
    import math
    from driving_dirty_b200.utils.helper import compute_ats_bounding_boxes
    g = torch.Generator().manual_seed(100 + seed)

    def boxes(n, jitter):
        c = torch.rand(n, 2, generator=g) * 16 - 8
        ang = torch.rand(n, generator=g) * math.pi
        out = []
        for k in range(n):
            cs, sn = math.cos(float(ang[k])), math.sin(float(ang[k]))
            pts = [(2.3, 1.0), (2.3, -1.0), (-2.3, 1.0), (-2.3, -1.0)]
            out.append(torch.tensor([[float(c[k, 0]) + cs * x - sn * y for x, y in pts],
                                     [float(c[k, 1]) + sn * x + cs * y for x, y in pts]]))
        return torch.stack(out) + jitter
    b2 = boxes(n2, 0.0)
    b1 = torch.cat([b2[: min(n1, n2) // 2] + 0.05 * torch.randn(min(n1, n2) // 2, 2, 4, generator=g),      # near matches
                    boxes(n1 - min(n1, n2) // 2, 0.0)])
    ref, ref_iou = so.compute_ats_bounding_boxes(b1, b2)
    got, iou = compute_ats_bounding_boxes(b1.cuda(), b2.cuda(), return_iou=True)
    assert float((iou.cpu() - ref_iou).abs().max()) < 1e-6
    assert float(got) == float(ref)
    # identical sets: every threshold counts every box (the reference's float32 weighted mean lands an ulp under 1)
    assert float(compute_ats_bounding_boxes(b2.cuda(), b2.cuda())) == float(so.compute_ats_bounding_boxes(b2, b2)[0])


# ------------------------------------------------------------------------------- guard bands -
def test_kernels_stay_inside_their_output_buffers(dd):
    """compute-sanitizer is closed on this GPU pool (profiles/r2_sanitizer_closed.txt), so the out-of-bounds check is our own:
    every output of the tensor-core kernels sits between two guard bands of a sentinel pattern (ragged shapes: partial
    column strips, odd row counts, residue classes of different length) and the bands must come back untouched."""
    import ctypes
    from driving_dirty_b200 import _lib
    from driving_dirty_b200._lib import call, stream_ptr
    st = stream_ptr()
    GUARD = 4096
    bands = []

    def guarded(shape, dtype):
        n = int(np.prod(shape))
        raw = torch.full((n + 2 * GUARD,), 7.0, device="cuda").to(dtype) if dtype != torch.uint8 else \
            torch.full((n + 2 * GUARD,), 7, dtype=torch.uint8, device="cuda")
        bands.append((raw, n))
        return raw[GUARD: GUARD + n].view(shape)

    B, H, W = 2, 37, 205
    H3, W3 = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    x = torch.rand(B, H, W, 32, device="cuda").bfloat16()
    dy = (torch.rand(B, H, W, 32, device="cuda") - 0.5).bfloat16()
    dy3 = (torch.rand(B, H3, W3, 32, device="cuda") - 0.5).bfloat16()
    w, b = torch.rand(32, 32, 3, 3, device="cuda") * 0.1, torch.zeros(32, device="cuda")
    n = int(_lib.load().dd_conv_wgrad_workspace_bytes())
    ws = guarded((n,), torch.uint8)
    o1, o2 = guarded((B, H, W, 32), torch.bfloat16), guarded((B, H3, W3, 32), torch.bfloat16)
    call("dd_conv3x3_c32_fwd", x.data_ptr(), w.data_ptr(), b.data_ptr(), o1.data_ptr(), 1, B, H, W, 1, 2, st)
    call("dd_conv3x3_c32_fwd", x.data_ptr(), w.data_ptr(), b.data_ptr(), o2.data_ptr(), 1, B, H, W, 2, 2, st)
    o3, o4 = guarded((B, H, W, 32), torch.bfloat16), guarded((B, H, W, 32), torch.bfloat16)
    call("dd_conv3x3_c32_dgrad", dy.data_ptr(), w.data_ptr(), x.data_ptr(), o3.data_ptr(), 1, B, H, W, 1, 2, st)
    call("dd_conv3x3_c32_dgrad", dy3.data_ptr(), w.data_ptr(), x.data_ptr(), o4.data_ptr(), 1, B, H, W, 2, 2, st)
    for stride, g in ((1, dy), (2, dy3)):
        dw, db = guarded((32, 32, 3, 3), torch.float32), guarded((32,), torch.float32)
        call("dd_conv3x3_c32_wgrad", x.data_ptr(), g.data_ptr(), dw.data_ptr(), db.data_ptr(), ws.data_ptr(), n, 1, B, H, W, stride, 2, st)
    views = torch.rand(B, 6, 3, 37, 35, device="cuda")          # mosaic 37 x 210
    a1 = guarded((B, 37, 210, 32), torch.bfloat16)
    w1 = torch.rand(32, 3, 3, 3, device="cuda")
    call("dd_conv_c1_fwd", views.data_ptr(), 1, w1.data_ptr(), b.data_ptr(), a1.data_ptr(), 1, B, 37, 210, 2, st)
    dw1, db1 = guarded((32, 3, 3, 3), torch.float32), guarded((32,), torch.float32)
    dya = (torch.rand(B, 37, 210, 32, device="cuda") - 0.5).bfloat16()
    call("dd_conv_c1_wgrad", views.data_ptr(), 1, dya.data_ptr(), 1, dw1.data_ptr(), db1.data_ptr(), ws.data_ptr(), n, B, 37, 210, 2, st)
    # wide dilated layers: forward, input gradient, weight gradient
    for (t, cin, cout, k, p, d, hw) in ((1, 96, 64, 7, 0, 7, (9, 23)), (1, 64, 32, 7, 0, 7, (11, 150)), (0, 32, 32, 3, 0, 3, (19, 140))):
        Hi, Wi = hw
        Ho = Hi + d * (k - 1) if t else Hi - d * (k - 1)
        Wo = Wi + d * (k - 1) if t else Wi - d * (k - 1)
        desc = _lib.ConvDesc(B, cin, cout, Hi, Wi, Ho, Wo, k, k, 1, 1, p, p, d, d, t)
        xin = torch.rand(B, Hi, Wi, cin, device="cuda").bfloat16()
        g = (torch.rand(B, Ho, Wo, cout, device="cuda") - 0.5).bfloat16()
        wt = torch.rand((cin, cout, k, k) if t else (cout, cin, k, k), device="cuda") * 0.05
        bb = torch.zeros(cout, device="cuda")
        nn_ = int(_lib.load().dd_conv2d_workspace_bytes(ctypes.byref(desc)))
        ws2 = guarded((nn_,), torch.uint8)
        y = guarded((B, Ho, Wo, cout), torch.bfloat16)
        call("dd_conv2d_fwd", xin.data_ptr(), wt.data_ptr(), bb.data_ptr(), y.data_ptr(), ctypes.byref(desc), 1, 1, ws2.data_ptr(), nn_, st)
        dxo = guarded((B, Hi, Wi, cin), torch.bfloat16)
        call("dd_conv2d_dgrad", g.data_ptr(), wt.data_ptr(), xin.data_ptr(), dxo.data_ptr(), ctypes.byref(desc), 1, ws2.data_ptr(), nn_, st)
        dwo, dbo = guarded(tuple(wt.shape), torch.float32), guarded((cout,), torch.float32)
        call("dd_conv2d_wgrad", xin.data_ptr(), g.data_ptr(), dwo.data_ptr(), dbo.data_ptr(), ctypes.byref(desc), 1, ws2.data_ptr(), nn_, st)
    torch.cuda.synchronize()
    for raw, nel in bands:
        lo, hi = raw[:GUARD].float(), raw[GUARD + nel:].float()
        assert bool((lo == 7).all()) and bool((hi == 7).all()), "a kernel wrote outside its output buffer"
