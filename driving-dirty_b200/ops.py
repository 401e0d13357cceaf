"""Host-side operators over the C ABI (include/dd_b200.h): thin wrappers and the
``torch.autograd.Function``s the drop-in modules are built from.

PyTorch is plumbing here -- it owns device memory, streams and the autograd tape; every byte
of arithmetic on the scene path is done by libdd_b200.so.  There is no CPU path: tensors that
are not CUDA tensors raise.
"""
from __future__ import annotations

from typing import Sequence

import torch

from . import _lib
from ._lib import DD_BF16, DD_F32, IMPL_AUTO, call, dtype_code, stream_ptr

VIEW_ORDER = (0, 1, 2, 5, 4, 3)


def _require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("driving-dirty_b200 runs on CUDA (sm_100a) only; got a CPU tensor. "
                               "There is no CPU fallback on this path.")


def _c(t: torch.Tensor) -> torch.Tensor:
    return t if t.is_contiguous() else t.contiguous()


class _Workspaces:
    """Per-device scratch buffers (owned by torch's allocator, handed to the library per call)."""

    def __init__(self):
        self._bufs = {}

    def get(self, key: str, nbytes: int, device, zero: bool = False) -> torch.Tensor:
        k = (key, device.index)
        buf = self._bufs.get(k)
        if buf is None or buf.numel() < nbytes:
            buf = (torch.zeros if zero else torch.empty)(max(nbytes, 256), dtype=torch.uint8, device=device)
            self._bufs[k] = buf
        return buf


_ws = _Workspaces()


# --------------------------------------------------------------------------------------------
# input handling / stitch
# --------------------------------------------------------------------------------------------
def as_view_batch(sample, keep_bytes=False) -> torch.Tensor:
    """tuple/list of B [6,3,H,W] tensors (what collate_fn yields) or a [B,6,3,H,W] tensor ->
    contiguous [B,6,3,H,W] fp32 CUDA tensor, without a copy when the tuple is ``batch.unbind(0)``.  uint8 raw camera
    bytes are taken as they come off the JPEG decoder: ToTensor's /255 (data_helper.py:109-114) runs here on the device
    (``dd_u8_to_f32``, bit-identical to ``x.float() / 255``), so only a quarter of the bytes cross PCIe.  ``keep_bytes``:
    hand the uint8 batch on as it is (``encoder_conv_stack`` converts, or reads the bytes inside its fused inference kernel)."""
    if torch.is_tensor(sample):
        x = sample
    else:
        sample = tuple(sample)
        first = sample[0]
        base = first._base
        zero_copy = (base is not None and base.dim() == 5 and base.is_contiguous() and base.shape[0] == len(sample)
                     and all(s._base is base and s.storage_offset() == base.storage_offset() + i * first.numel()
                             and s.is_contiguous() for i, s in enumerate(sample)))
        x = base if zero_copy else torch.stack(sample, dim=0)
    _require_cuda(x)
    if x.dim() != 5 or x.shape[1] != 6 or x.shape[2] != 3:
        raise RuntimeError(f"expected views of shape [B,6,3,H,W], got {tuple(x.shape)}")
    if x.dtype == torch.uint8:
        return _c(x) if keep_bytes else bytes_to_float(x)
    if x.dtype != torch.float32:
        x = x.float()
    return _c(x)


def bytes_to_float(x_u8: torch.Tensor) -> torch.Tensor:
    """torchvision ToTensor's scaling on the device: uint8 -> float32 / 255 (any shape), bit-identical."""
    _require_cuda(x_u8)
    x_u8 = _c(x_u8)
    out = torch.empty(x_u8.shape, dtype=torch.float32, device=x_u8.device)
    call("dd_u8_to_f32", x_u8.data_ptr(), out.data_ptr(), x_u8.numel(), stream_ptr())
    return out


class _Stitch(torch.autograd.Function):
    """wide_stitch_six_images on fp32 views; backward: the inverse permutation (dd_unstitch_f32)."""

    @staticmethod
    def forward(ctx, views):
        B, _, _, H, W = views.shape
        out = torch.empty(B, 3, H, 6 * W, dtype=torch.float32, device=views.device)
        call("dd_stitch_f32", views.data_ptr(), out.data_ptr(), B, H, W, stream_ptr())
        return out

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        B, _, H, Wm = g.shape
        d = torch.empty(B, 6, 3, H, Wm // 6, dtype=torch.float32, device=g.device)
        call("dd_unstitch_f32", g.data_ptr(), None, d.data_ptr(), B, H, Wm // 6, -1, stream_ptr())
        return d


def stitch(views: torch.Tensor) -> torch.Tensor:
    """wide_stitch_six_images (roadmap_bce_v2.py:53-64): [B,6,3,H,W] -> [B,3,H,6W] (raw bytes: with ToTensor's /255).
    Differentiable for float views: the mosaic's gradient goes back to the views."""
    if torch.is_tensor(views) and views.dtype == torch.uint8:
        return stitch_u8(views)
    return _Stitch.apply(as_view_batch(views))


def stitch_u8(views_u8: torch.Tensor) -> torch.Tensor:
    """uint8 camera bytes [B,6,3,H,W] -> fp32 mosaic with the ToTensor /255 folded in."""
    _require_cuda(views_u8)
    views_u8 = _c(views_u8)
    B, _, _, H, W = views_u8.shape
    out = torch.empty(B, 3, H, 6 * W, dtype=torch.float32, device=views_u8.device)
    call("dd_stitch_u8", views_u8.data_ptr(), out.data_ptr(), B, H, W, stream_ptr())
    return out


class _StitchMask(torch.autograd.Function):
    """six_to_one_task on fp32 views.  Backward: the zeroed block of x passes no gradient, the slot's view takes y's."""

    @staticmethod
    def forward(ctx, views, slot):
        B, _, _, H, W = views.shape
        x = torch.empty(B, 3, H, 6 * W, dtype=torch.float32, device=views.device)
        y = torch.empty(B, 3, H, W, dtype=torch.float32, device=views.device)
        call("dd_stitch_mask_f32", views.data_ptr(), x.data_ptr(), y.data_ptr(), B, H, W, slot, stream_ptr())
        ctx.slot = slot
        return x, y

    @staticmethod
    def backward(ctx, gx, gy):
        gx, gy = _c(gx), _c(gy)
        B, _, H, W = gy.shape
        d = torch.empty(B, 6, 3, H, W, dtype=torch.float32, device=gx.device)
        call("dd_unstitch_f32", gx.data_ptr(), gy.data_ptr(), d.data_ptr(), B, H, W, ctx.slot, stream_ptr())
        return d, None


def stitch_mask(views: torch.Tensor, slot: int):
    """six_to_one_task (autoencoder.py:53-73) for an already drawn slot: (x, y), both differentiable in the views."""
    return _StitchMask.apply(as_view_batch(views), int(slot))


# --------------------------------------------------------------------------------------------
# encoder conv stack (c1 -> c2 -> c3 [-> flat max-pool]) as ONE autograd node
# --------------------------------------------------------------------------------------------
# On the bf16 tensor-core training path the c2 / c3 input gradients take the ReLU masks of a1 / a2 as sign words (4 bytes
# per pixel, written by the c1 / c2 forward kernels) instead of re-reading the 64-byte activations; the gradients are
# bit-identical either way.  False selects the activation-mask form (kept so that the two can be compared in one process).
RELU_MASK_BITS = True


def _conv_ws(device):
    n = int(_lib.load().dd_conv_wgrad_workspace_bytes())
    return _ws.get("conv_wgrad", n, device), n


class EncoderConvStack(torch.autograd.Function):
    """relu(c1) -> relu(c2) -> relu(c3, stride 2) -> view(B,-1) -> max_pool1d(4)
    (components.py:41-47).  ``inp`` is the views batch [B,6,3,H,W] (stitch folded into c1's loads)
    or a mosaic / NCHW image [B,3,H,Wm].  Activations are NHWC in ``act_dtype``.  Returns the
    pooled features [B, 8*H3*W3] (act_dtype; fp32 copies of the same values when nothing requires grad) or, with ``c3_only``, the c3 activation as NCHW fp32
    (components.py:44-45; ``c3_only == 2``: as the NHWC activation itself).

    An fp32 ``inp`` that requires grad gets the image gradient of c1 (dd_conv_c1_dgrad), in its own layout: views or
    mosaic.  When no conv weight requires grad (a frozen model under attribution) the backward runs the input-gradient
    chain alone, and on the sign-word path a1 / a2 are not kept: that chain reads only a3 and the sign words."""

    @staticmethod
    def forward(ctx, inp, w1, b1, w2, b2, w3, b3, act_dtype, c3_only, impl):
        _require_cuda(inp, w1, w2, w3)
        inp = _c(inp)
        inference = not any(ctx.needs_input_grad)
        want_dw = any(ctx.needs_input_grad[1:7])
        tensor_core = act_dtype == torch.bfloat16 and impl != _lib.IMPL_SIMT
        fused_front = inference and tensor_core
        if inp.dtype == torch.uint8 and not tensor_core:
            # raw camera bytes on the fp32 parity path: ToTensor's /255 as a pass of its own (dd_u8_to_f32).  The tensor-core
            # kernels (c1 forward, c1 weight gradient, the fused inference front) read the bytes themselves (DD_IN_U8,
            # bit-identical, tested): their converter warps issue all loads of a row before the first table look-up, so
            # bytes cost them nothing (0.29 / 0.25 ms either way, profiles/r2_kernel_times.txt) and the pass (0.07 ms, 200 MB) goes
            inp = bytes_to_float(inp)
        is_views = inp.dim() == 5
        if is_views:
            B, _, _, H, W = inp.shape
            Wm = 6 * W
        else:
            B, _, H, Wm = inp.shape
        dev, code, st = inp.device, dtype_code(act_dtype), stream_ptr()
        H3, W3 = (H - 1) // 2 + 1, (Wm - 1) // 2 + 1
        w1, b1, w2, b2, w3, b3 = (_c(t.detach().float()) for t in (w1, b1, w2, b2, w3, b3))
        in_flags = (_lib.IN_VIEWS if is_views else 0) | (_lib.IN_U8 if inp.dtype == torch.uint8 else 0)
        bits1 = bits2 = None
        if fused_front:
            # no backward pass will ask for the first activation: c1 -> c2 in one kernel, a1 stays in shared memory / TMEM
            # (same bits as the two kernels below)
            a1 = None
            a2 = torch.empty(B, H, Wm, 32, dtype=act_dtype, device=dev)
            call("dd_encoder_c1c2_fused_fwd", inp.data_ptr(), in_flags, w1.data_ptr(), b1.data_ptr(), w2.data_ptr(),
                 b2.data_ptr(), a2.data_ptr(), B, H, Wm, st)
        elif tensor_core and RELU_MASK_BITS:
            # training: a1 / a2 are kept for the weight gradients, their ReLU masks as sign words for the input gradients
            a1 = torch.empty(B, H, Wm, 32, dtype=act_dtype, device=dev)
            bits1 = torch.empty(B, H, Wm, dtype=torch.int32, device=dev)
            call("dd_conv_c1_fwd_bits", inp.data_ptr(), in_flags, w1.data_ptr(), b1.data_ptr(), a1.data_ptr(),
                 bits1.data_ptr(), code, B, H, Wm, impl, st)
            a2 = torch.empty_like(a1)
            bits2 = torch.empty_like(bits1)
            call("dd_conv3x3_c32_fwd_bits", a1.data_ptr(), w2.data_ptr(), b2.data_ptr(), a2.data_ptr(), bits2.data_ptr(),
                 code, B, H, Wm, 1, impl, st)
        else:
            a1 = torch.empty(B, H, Wm, 32, dtype=act_dtype, device=dev)
            call("dd_conv_c1_fwd", inp.data_ptr(), in_flags, w1.data_ptr(), b1.data_ptr(), a1.data_ptr(), code,
                 B, H, Wm, impl, st)
            a2 = torch.empty_like(a1)
            call("dd_conv3x3_c32_fwd", a1.data_ptr(), w2.data_ptr(), b2.data_ptr(), a2.data_ptr(), code, B, H, Wm, 1,
                 impl, st)
        a3 = torch.empty(B, H3, W3, 32, dtype=act_dtype, device=dev)
        call("dd_conv3x3_c32_fwd", a2.data_ptr(), w3.data_ptr(), b3.data_ptr(), a3.data_ptr(), code, B, H, Wm, 2,
             impl, st)
        if c3_only == 2:
            out = a3               # the NHWC activation itself, for the bounding-box CNNs
        elif c3_only:
            out = torch.empty(B, 32, H3, W3, dtype=torch.float32, device=dev)
            call("dd_nhwc_to_nchw_f32", a3.data_ptr(), code, out.data_ptr(), B, 32, H3, W3, st)
        elif inference:
            # inference: fp32 features (exactly the bf16 maxima) -- the tf32 linear that follows reads them as they are
            out = torch.empty(B, 8 * H3 * W3, dtype=torch.float32, device=dev)
            call("dd_pool4_fwd_f32", a3.data_ptr(), out.data_ptr(), code, B, H3, W3, st)
        else:
            out = torch.empty(B, 8 * H3 * W3, dtype=act_dtype, device=dev)
            call("dd_pool4_fwd", a3.data_ptr(), out.data_ptr(), code, B, H3, W3, st)
        ctx.geom = (B, H, Wm, H3, W3, in_flags, code, c3_only, impl, act_dtype)
        if not inference:
            keep = want_dw or bits1 is None     # the activation-mask form reads a1 / a2 as the ReLU masks
            ctx.save_for_backward(inp if want_dw else None, w1, w2, w3, a1 if keep else None, a2 if keep else None, a3,
                                  bits1, bits2)
        return out

    @staticmethod
    def backward(ctx, g):
        inp, w1, w2, w3, a1, a2, a3, bits1, bits2 = ctx.saved_tensors
        B, H, Wm, H3, W3, in_flags, code, c3_only, impl, act_dtype = ctx.geom
        want_dx, want_dw = ctx.needs_input_grad[0], any(ctx.needs_input_grad[1:7])
        dw1 = db1 = dw2 = db2 = dw3 = db3 = dx = None
        dev, st = g.device, stream_ptr()
        ws, ws_n = _conv_ws(dev)
        da3 = torch.empty_like(a3)
        if c3_only == 2:
            g = _c(g.to(act_dtype))
            call("dd_relu_mask", g.data_ptr(), a3.data_ptr(), da3.data_ptr(), code, da3.numel(), st)
        elif c3_only:
            g = _c(g.float())
            call("dd_nchw_f32_to_nhwc", g.data_ptr(), da3.data_ptr(), code, B, 32, H3, W3, st)
            call("dd_relu_mask", da3.data_ptr(), a3.data_ptr(), da3.data_ptr(), code, da3.numel(), st)
        else:
            g = _c(g.to(act_dtype))
            call("dd_pool4_bwd", a3.data_ptr(), g.data_ptr(), da3.data_ptr(), code, B, H3, W3, st)
        f32 = dict(dtype=torch.float32, device=dev)
        if want_dw:
            dw3, db3 = torch.empty(32, 32, 3, 3, **f32), torch.empty(32, **f32)
            call("dd_conv3x3_c32_wgrad", a2.data_ptr(), da3.data_ptr(), dw3.data_ptr(), db3.data_ptr(), ws.data_ptr(),
                 ws_n, code, B, H, Wm, 2, impl, st)
        da2 = torch.empty(B, H, Wm, 32, dtype=act_dtype, device=dev)     # (a1 / a2 are not kept for a frozen stack)
        if bits2 is not None:
            call("dd_conv3x3_c32_dgrad_bits", da3.data_ptr(), w3.data_ptr(), bits2.data_ptr(), da2.data_ptr(), code, B, H,
                 Wm, 2, impl, st)
        else:
            call("dd_conv3x3_c32_dgrad", da3.data_ptr(), w3.data_ptr(), a2.data_ptr(), da2.data_ptr(), code, B, H, Wm, 2,
                 impl, st)
        del da3
        if want_dw:
            dw2, db2 = torch.empty(32, 32, 3, 3, **f32), torch.empty(32, **f32)
            call("dd_conv3x3_c32_wgrad", a1.data_ptr(), da2.data_ptr(), dw2.data_ptr(), db2.data_ptr(), ws.data_ptr(),
                 ws_n, code, B, H, Wm, 1, impl, st)
        da1 = torch.empty(B, H, Wm, 32, dtype=act_dtype, device=dev)
        if bits1 is not None:
            call("dd_conv3x3_c32_dgrad_bits", da2.data_ptr(), w2.data_ptr(), bits1.data_ptr(), da1.data_ptr(), code, B, H,
                 Wm, 1, impl, st)
        else:
            call("dd_conv3x3_c32_dgrad", da2.data_ptr(), w2.data_ptr(), a1.data_ptr(), da1.data_ptr(), code, B, H, Wm, 1,
                 impl, st)
        del da2
        if want_dw:
            dw1, db1 = torch.empty(32, 3, 3, 3, **f32), torch.empty(32, **f32)
            call("dd_conv_c1_wgrad", inp.data_ptr(), in_flags, da1.data_ptr(), code, dw1.data_ptr(), db1.data_ptr(),
                 ws.data_ptr(), ws_n, B, H, Wm, impl, st)
        if want_dx:
            views = in_flags & _lib.IN_VIEWS
            dx = torch.empty((B, 6, 3, H, Wm // 6) if views else (B, 3, H, Wm), **f32)
            call("dd_conv_c1_dgrad", da1.data_ptr(), code, w1.data_ptr(), dx.data_ptr(), views, B, H, Wm, impl, st)
        return dx, dw1, db1, dw2, db2, dw3, db3, None, None, None


def encoder_conv_stack(inp, c1, c2, c3, act_dtype=torch.float32, c3_only=False, impl=IMPL_AUTO):
    return EncoderConvStack.apply(inp, c1.weight, c1.bias, c2.weight, c2.bias, c3.weight, c3.bias, act_dtype,
                                  int(c3_only), int(impl))


# --------------------------------------------------------------------------------------------
# skinny linear
# --------------------------------------------------------------------------------------------
def _linear_ws(B, N, K, device):
    n = int(_lib.load().dd_linear_workspace_bytes(B, N, K))
    return _ws.get("linear", n, device), n


class SkinnyLinear(torch.autograd.Function):
    """y = x W^T + b for a small batch and a very wide K or N (nn.Linear at components.py:105,
    roadmap_bce_v2.py:75).  x: [B,K] fp32 or bf16; W [N,K], b [N], y [B,N] fp32.
    ``impl``: IMPL_SIMT = fp32 CUDA-core kernels (1e-5 parity); IMPL_TCGEN05 = TMA + tcgen05 tf32
    weight-streaming kernels (x is read as fp32)."""

    @staticmethod
    def forward(ctx, x, w, b, impl, grad_buffer=None, grad_ready=None, fused_update=None, grad_begin=None):
        _require_cuda(x, w)
        ctx.grad_buffer, ctx.grad_ready, ctx.fused_update, ctx.grad_begin = grad_buffer, grad_ready, fused_update, grad_begin
        x, wd = _c(x), _c(w.detach())
        if wd.dtype != torch.float32:
            wd = wd.float()
        B, K = x.shape
        N = wd.shape[0]
        ctx.x_dtype = x.dtype
        if impl == _lib.IMPL_TCGEN05 and x.dtype != torch.float32:
            x = x.float()          # the tf32 path streams fp32 operands through TMA
        y = torch.empty(B, N, dtype=torch.float32, device=x.device)
        ws, n = _linear_ws(B, N, K, x.device)
        bias_ptr = _c(b.detach().float()).data_ptr() if b is not None else None
        call("dd_linear_fwd", x.data_ptr(), dtype_code(x.dtype), wd.data_ptr(), bias_ptr, y.data_ptr(),
             ws.data_ptr(), n, B, N, K, impl, stream_ptr())
        ctx.save_for_backward(x, wd)
        ctx.has_bias = b is not None
        ctx.impl = impl
        return y

    @staticmethod
    def backward(ctx, dy):
        x, w = ctx.saved_tensors
        B, K = x.shape
        N = w.shape[0]
        dy = _c(dy.float())
        st = stream_ptr()
        dx = dw = db = None
        fusable = ctx.impl == _lib.IMPL_TCGEN05 and B <= 32 and x.dtype == torch.float32
        if ctx.needs_input_grad[1] and ctx.fused_update is not None and ctx.fused_update.takes(fusable):
            # optim.FusedAdam (world size 1) folds this weight's Adam step into the backward pass: one kernel computes the
            # input gradient from the old weight and updates the weight and its moments in place; the weight gradient never
            # exists in HBM (dd_linear_bwd_adam).  With gradient accumulation it takes every pass of a window: the earlier
            # ones add into its gradient buffer, the last one steps from it (dd_linear_bwd_adam_acc)
            dx = torch.empty(B, K, dtype=ctx.x_dtype, device=x.device) if ctx.needs_input_grad[0] else None
            ws, n = _linear_ws(B, N, K, x.device)
            db = torch.empty(N, dtype=torch.float32, device=x.device) if ctx.has_bias else None
            ctx.fused_update(dy, x, w, dx, db, ws, n, fusable, ctx.impl)
            return dx, None, db, None, None, None, None, None
        if ctx.needs_input_grad[0]:
            dx = torch.empty(B, K, dtype=ctx.x_dtype, device=x.device)
            ws, n = _linear_ws(B, N, K, x.device)
            call("dd_linear_dgrad", dy.data_ptr(), w.data_ptr(), dx.data_ptr(), dtype_code(ctx.x_dtype), ws.data_ptr(), n,
                 B, N, K, ctx.impl, st)
        if ctx.needs_input_grad[1]:
            # a parameter claimed by optim.FusedAdam's sharded update owns a persistent (peer-mapped) gradient
            # buffer: the kernel writes there and autograd gets no tensor to clone or accumulate
            direct = ctx.grad_buffer is not None
            dw = ctx.grad_buffer if direct else torch.empty_like(w)
            db = torch.empty(N, dtype=torch.float32, device=x.device) if ctx.has_bias else None
            # ... which the passes after the first of a gradient-accumulation window add to (FusedAdam's grad_begin)
            if direct and ctx.grad_begin is not None and ctx.grad_begin():
                call("dd_linear_wgrad_acc", dy.data_ptr(), x.data_ptr(), dtype_code(x.dtype), dw.data_ptr(),
                     db.data_ptr() if db is not None else None, B, N, K, ctx.impl, 1, st)
            else:
                call("dd_linear_wgrad", dy.data_ptr(), x.data_ptr(), dtype_code(x.dtype), dw.data_ptr(),
                     db.data_ptr() if db is not None else None, B, N, K, ctx.impl, st)
            if direct:
                dw = None
                if ctx.grad_ready is not None:
                    ctx.grad_ready()
        elif ctx.has_bias and ctx.needs_input_grad[2]:
            db = dy.sum(0)
        return dx, dw, db, None, None, None, None, None


def linear(x, weight, bias=None, impl=IMPL_AUTO, allow_tf32=False):
    """IMPL_AUTO: the tensor-core (tf32) kernels when the caller is on the reduced-precision path
    (bf16 activations, or ``allow_tf32``) and the layer is wide enough to stream; else fp32 CUDA cores."""
    impl = int(impl)
    if impl == IMPL_AUTO:
        B, K = x.shape
        fast = (x.dtype == torch.bfloat16 or allow_tf32) and x.is_cuda and \
            bool(_lib.load().dd_linear_tc_supported(B, weight.shape[0], K))
        impl = _lib.IMPL_TCGEN05 if fast else _lib.IMPL_SIMT
    ev = getattr(weight, "_dd_ready_event", None)
    if ev is not None:                 # optim.FusedAdam: this weight's last update may still be landing (side stream)
        torch.cuda.current_stream().wait_event(ev)
        weight._dd_ready_event = None
    buf = getattr(weight, "_dd_grad_buffer", None)
    if buf is not None and not (buf.shape == weight.shape and buf.dtype == torch.float32 and buf.is_contiguous()):
        raise RuntimeError("linear: weight._dd_grad_buffer does not match the weight")
    return SkinnyLinear.apply(x, weight, bias, impl, buf, getattr(weight, "_dd_grad_ready", None) if buf is not None else None,
                              getattr(weight, "_dd_fused_update", None) if torch.is_grad_enabled() else None,
                              getattr(weight, "_dd_grad_begin", None) if buf is not None else None)


# --------------------------------------------------------------------------------------------
# sigmoid + BCE + threat score + binarise
# --------------------------------------------------------------------------------------------
def _bce_ws(device):
    n = int(_lib.load().dd_bce_ts_workspace_bytes())
    return _ws.get("bce_ts", n, device, zero=True), n


class BceThreat(torch.autograd.Function):
    """One pass: mean BCE-with-logits (roadmap_bce_v2.py:103-106), probs = sigmoid (:81),
    binary = probs.round() (:140), TS(target, probs) and TS(target, binary) (helper.py:74-77).
    Returns (loss, probs, binary_u8, stats[4], counts[4]); only ``loss`` is differentiable."""

    @staticmethod
    def forward(ctx, logits, target, want_probs, want_binary):
        _require_cuda(logits, target)
        logits = _c(logits)
        if logits.dtype != torch.float32:
            raise RuntimeError("roadmap logits must be fp32")
        target = _c(target)
        is_u8 = target.dtype in (torch.uint8, torch.bool)
        if not is_u8 and target.dtype != torch.float32:
            target = target.float()
        n = logits.numel()
        if target.numel() != n:
            raise RuntimeError(f"target has {target.numel()} elements, logits {n}")
        dev = logits.device
        probs = torch.empty_like(logits) if want_probs else None
        binary = torch.empty(logits.shape, dtype=torch.uint8, device=dev) if want_binary else None
        stats = torch.empty(4, dtype=torch.float32, device=dev)
        counts = torch.empty(4, dtype=torch.int64, device=dev)
        ws, wn = _bce_ws(dev)
        call("dd_bce_ts_fwd", logits.data_ptr(), target.data_ptr(), int(is_u8),
             probs.data_ptr() if want_probs else None, binary.data_ptr() if want_binary else None,
             stats.data_ptr(), counts.data_ptr(), ws.data_ptr(), wn, n, stream_ptr())
        ctx.save_for_backward(logits, target)
        ctx.is_u8 = is_u8
        loss = stats[0].clone()
        outs = (loss, probs, binary, stats, counts)
        ctx.mark_non_differentiable(*[t for t in outs[1:] if t is not None])
        return outs

    @staticmethod
    def backward(ctx, g_loss, *unused):
        logits, target = ctx.saved_tensors
        dlogits = torch.empty_like(logits)
        g = _c(g_loss.float().reshape(1))
        call("dd_bce_bwd", logits.data_ptr(), target.data_ptr(), int(ctx.is_u8), g.data_ptr(), dlogits.data_ptr(),
             logits.numel(), stream_ptr())
        return dlogits, None, None, None


def bce_threat(logits, target, want_probs=True, want_binary=True):
    return BceThreat.apply(logits, target, bool(want_probs), bool(want_binary))


class _SigmoidBinary(torch.autograd.Function):
    """forward()'s ``torch.sigmoid(y)`` (roadmap_bce_v2.py:81) plus the binarised map, through the
    same kernel without a target (statistics discarded)."""

    @staticmethod
    def forward(ctx, logits):
        logits = _c(logits)
        dev = logits.device
        probs = torch.empty_like(logits)
        binary = torch.empty(logits.shape, dtype=torch.uint8, device=dev)
        stats = torch.empty(4, dtype=torch.float32, device=dev)
        counts = torch.empty(4, dtype=torch.int64, device=dev)
        ws, wn = _bce_ws(dev)
        # no target: the kernel reads none (statistics are computed against an all-zero map and discarded)
        call("dd_bce_ts_fwd", logits.data_ptr(), None, 0, probs.data_ptr(), binary.data_ptr(),
             stats.data_ptr(), counts.data_ptr(), ws.data_ptr(), wn, logits.numel(), stream_ptr())
        ctx.save_for_backward(probs)
        ctx.mark_non_differentiable(binary)
        return probs, binary

    @staticmethod
    def backward(ctx, g, _):
        (p,) = ctx.saved_tensors
        return g * p * (1.0 - p)


def sigmoid_binary(logits):
    return _SigmoidBinary.apply(logits)


def binary_map(logits: torch.Tensor) -> torch.Tensor:
    """``sigmoid(logits).round()`` (roadmap_bce_v2.py:81,140) as a uint8 map, without materialising the probabilities:
    the inference front-end's last pass reads the logits once and writes one byte per pixel."""
    _require_cuda(logits)
    logits = _c(logits)
    dev = logits.device
    binary = torch.empty(logits.shape, dtype=torch.uint8, device=dev)
    stats = torch.empty(4, dtype=torch.float32, device=dev)
    counts = torch.empty(4, dtype=torch.int64, device=dev)
    ws, wn = _bce_ws(dev)
    call("dd_bce_ts_fwd", logits.data_ptr(), None, 0, None, binary.data_ptr(), stats.data_ptr(), counts.data_ptr(),
         ws.data_ptr(), wn, logits.numel(), stream_ptr())
    return binary


def threat_score(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """compute_ts_road_map (helper.py:74-77) for two maps of any float values -> 0-dim tensor."""
    _require_cuda(a, b)
    a, b = _c(a.float()), _c(b.float())
    if a.numel() != b.numel():
        raise RuntimeError("threat_score: maps differ in size")
    out = torch.empty(1, dtype=torch.float32, device=a.device)
    ws, wn = _bce_ws(a.device)
    call("dd_threat_score_f32", a.data_ptr(), b.data_ptr(), out.data_ptr(), ws.data_ptr(), wn, a.numel(), stream_ptr())
    return out[0]


class MseLoss(torch.autograd.Function):
    """F.mse_loss(y, y_hat) (autoencoder.py:91), mean over all elements."""

    @staticmethod
    def forward(ctx, y, y_hat):
        _require_cuda(y, y_hat)
        y, y_hat = _c(y.float()), _c(y_hat.float())
        out = torch.empty(1, dtype=torch.float32, device=y.device)
        ws, wn = _bce_ws(y.device)
        call("dd_mse_fwd", y.data_ptr(), y_hat.data_ptr(), out.data_ptr(), ws.data_ptr(), wn, y.numel(), stream_ptr())
        ctx.save_for_backward(y, y_hat)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        y, y_hat = ctx.saved_tensors
        d = torch.empty_like(y_hat)
        gg = _c(g.float().reshape(1))
        call("dd_mse_bwd", y.data_ptr(), y_hat.data_ptr(), gg.data_ptr(), d.data_ptr(), y.numel(), stream_ptr())
        return (-d if ctx.needs_input_grad[0] else None), d


def mse_loss(y, y_hat):
    return MseLoss.apply(y, y_hat)


# --------------------------------------------------------------------------------------------
# generic conv / transposed conv on NHWC activations (decoder, bounding-box CNNs)
# --------------------------------------------------------------------------------------------
def _pair(v):
    return (int(v), int(v)) if not isinstance(v, (tuple, list)) else (int(v[0]), int(v[1]))


def conv_out_size(hi, k, s, p, d, transposed, output_padding=0):
    if transposed:
        return (hi - 1) * s - 2 * p + d * (k - 1) + output_padding + 1
    return (hi + 2 * p - d * (k - 1) - 1) // s + 1


def _conv_desc(B, Cin, Cout, Hi, Wi, Ho, Wo, k, s, p, d, transposed):
    return _lib.ConvDesc(B, Cin, Cout, Hi, Wi, Ho, Wo, k[0], k[1], s[0], s[1], p[0], p[1], d[0], d[1], int(transposed))


def _conv2d_ws(desc, device):
    import ctypes
    n = int(_lib.load().dd_conv2d_workspace_bytes(ctypes.byref(desc)))
    return _ws.get("conv2d", n, device), n


class LayoutToNHWC(torch.autograd.Function):
    """NCHW fp32 (API edge) -> NHWC activation of ``dtype``."""

    @staticmethod
    def forward(ctx, x, dtype):
        _require_cuda(x)
        x = _c(x.float())
        B, Cn, H, W = x.shape
        out = torch.empty(B, H, W, Cn, dtype=dtype, device=x.device)
        call("dd_nchw_f32_to_nhwc", x.data_ptr(), out.data_ptr(), dtype_code(dtype), B, Cn, H, W, stream_ptr())
        return out

    @staticmethod
    def backward(ctx, g):
        g = _c(g)
        B, H, W, Cn = g.shape
        out = torch.empty(B, Cn, H, W, dtype=torch.float32, device=g.device)
        call("dd_nhwc_to_nchw_f32", g.data_ptr(), dtype_code(g.dtype), out.data_ptr(), B, Cn, H, W, stream_ptr())
        return out, None


class LayoutToNCHW(torch.autograd.Function):
    """NHWC activation -> NCHW fp32 (API edge)."""

    @staticmethod
    def forward(ctx, x):
        _require_cuda(x)
        x = _c(x)
        ctx.dtype = x.dtype
        B, H, W, Cn = x.shape
        out = torch.empty(B, Cn, H, W, dtype=torch.float32, device=x.device)
        call("dd_nhwc_to_nchw_f32", x.data_ptr(), dtype_code(x.dtype), out.data_ptr(), B, Cn, H, W, stream_ptr())
        return out

    @staticmethod
    def backward(ctx, g):
        g = _c(g.float())
        B, Cn, H, W = g.shape
        out = torch.empty(B, H, W, Cn, dtype=ctx.dtype, device=g.device)
        call("dd_nchw_f32_to_nhwc", g.data_ptr(), out.data_ptr(), dtype_code(ctx.dtype), B, Cn, H, W, stream_ptr())
        return out


def to_nhwc(x, dtype=torch.float32):
    return LayoutToNHWC.apply(x, dtype)


def to_nchw(x):
    return LayoutToNCHW.apply(x)


class Conv2dNHWC(torch.autograd.Function):
    """nn.Conv2d / nn.ConvTranspose2d (+ bias, + optional ReLU) on an NHWC activation [B,H,W,Cin] of
    fp32 or bf16; weight / bias fp32 in torch layout.  geom = (kernel, stride, padding, dilation,
    transposed, output_padding), pairs like torch's; act 0 none / 1 ReLU / 2 sigmoid."""

    @staticmethod
    def forward(ctx, x, weight, bias, geom, act):
        import ctypes
        _require_cuda(x, weight)
        k, s, p, d, transposed, opad = geom
        x = _c(x)
        w = _c(weight.detach().float())
        B, Hi, Wi, Cin = x.shape
        Cout = w.shape[1] if transposed else w.shape[0]
        if (w.shape[0] if transposed else w.shape[1]) != Cin:
            raise RuntimeError(f"conv2d: input has {Cin} channels, weight {tuple(w.shape)}")
        Ho = conv_out_size(Hi, k[0], s[0], p[0], d[0], transposed, opad[0])
        Wo = conv_out_size(Wi, k[1], s[1], p[1], d[1], transposed, opad[1])
        desc = _conv_desc(B, Cin, Cout, Hi, Wi, Ho, Wo, k, s, p, d, transposed)
        y = torch.empty(B, Ho, Wo, Cout, dtype=x.dtype, device=x.device)
        ws, n = _conv2d_ws(desc, x.device)
        bptr = _c(bias.detach().float()).data_ptr() if bias is not None else None
        call("dd_conv2d_fwd", x.data_ptr(), w.data_ptr(), bptr, y.data_ptr(), ctypes.byref(desc), dtype_code(x.dtype),
             int(act), ws.data_ptr(), n, stream_ptr())
        ctx.desc, ctx.act, ctx.has_bias = desc, int(act), bias is not None
        ctx.save_for_backward(x, w, y if act else None)
        return y

    @staticmethod
    def backward(ctx, dy):
        import ctypes
        x, w, y = ctx.saved_tensors
        desc, st, code = ctx.desc, stream_ptr(), dtype_code(x.dtype)
        dy = _c(dy.to(x.dtype))
        if ctx.act:
            dym = torch.empty_like(dy)
            call("dd_relu_mask" if ctx.act == 1 else "dd_sigmoid_bwd", dy.data_ptr(), y.data_ptr(), dym.data_ptr(), code,
                 dy.numel(), st)
            dy = dym
        ws, n = _conv2d_ws(desc, x.device)
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = torch.empty_like(x)
            call("dd_conv2d_dgrad", dy.data_ptr(), w.data_ptr(), None, dx.data_ptr(), ctypes.byref(desc), code,
                 ws.data_ptr(), n, st)
        if ctx.needs_input_grad[1]:
            dw = torch.empty_like(w)
            db = torch.empty(desc.Cout, dtype=torch.float32, device=x.device) if ctx.has_bias else None
            call("dd_conv2d_wgrad", x.data_ptr(), dy.data_ptr(), dw.data_ptr(), db.data_ptr() if db is not None else None,
                 ctypes.byref(desc), code, ws.data_ptr(), n, st)
        return dx, dw, db, None, None, None


ACT_NONE, ACT_RELU, ACT_SIGMOID = 0, 1, 2


def conv2d_nhwc(x, module, relu=False, act=None):
    """Apply an nn.Conv2d / nn.ConvTranspose2d parameter container to an NHWC activation
    (act: ACT_NONE / ACT_RELU / ACT_SIGMOID fused after the bias; ``relu=True`` = ACT_RELU)."""
    transposed = isinstance(module, torch.nn.ConvTranspose2d)
    geom = (_pair(module.kernel_size), _pair(module.stride), _pair(module.padding), _pair(module.dilation), transposed,
            _pair(module.output_padding) if transposed else (0, 0))
    if module.groups != 1:
        raise RuntimeError("conv2d_nhwc: grouped convolutions are not part of the scene pipeline")
    return Conv2dNHWC.apply(x, module.weight, module.bias, geom, int(act) if act is not None else int(bool(relu)))


def decoder_deconv_stack(x, dc1, dc2, dc3, dc4, act_dtype=torch.float32):
    """Decoder transposed-conv stack (components.py:88-92): x [B,64,h,w] NCHW fp32 ->
    relu(dc1) -> relu(dc2) -> relu(dc3, k2 s2) -> dc4 (1x1) -> [B,3,2h,2w] NCHW fp32."""
    a = to_nhwc(x, act_dtype)
    a = conv2d_nhwc(a, dc1, relu=True)
    a = conv2d_nhwc(a, dc2, relu=True)
    a = conv2d_nhwc(a, dc3, relu=True)
    a = conv2d_nhwc(a, dc4, relu=False)
    return to_nchw(a)


# --------------------------------------------------------------------------------------------
# bounding-box model plumbing: camera extraction, tiling / concatenation, prob-space BCE
# --------------------------------------------------------------------------------------------
class ViewExtract(torch.autograd.Function):
    """Cameras of every scene as NHWC images, ``specs`` = ((view, mode), ...) with each view at most once.  Backward writes
    ONE views-shaped gradient: every extracted view's slice by dd_view_extract_bwd, the others zero."""

    @staticmethod
    def forward(ctx, views, specs, dtype):
        B, _, _, H, W = views.shape
        outs = []
        for view, mode in specs:
            Ho, Wo = (W, H) if mode in (1, 2) else (H, W)
            out = torch.empty(B, Ho, Wo, 3, dtype=dtype, device=views.device)
            call("dd_view_extract", views.data_ptr(), out.data_ptr(), dtype_code(dtype), B, H, W, view, mode, stream_ptr())
            outs.append(out)
        ctx.specs, ctx.shape = specs, tuple(views.shape)
        return tuple(outs)

    @staticmethod
    def backward(ctx, *grads):
        B, _, _, H, W = ctx.shape
        every_view = len(ctx.specs) == 6
        d = (torch.empty if every_view else torch.zeros)(ctx.shape, dtype=torch.float32, device=grads[0].device)
        for (view, mode), g in zip(ctx.specs, grads):
            g = _c(g)
            call("dd_view_extract_bwd", g.data_ptr(), dtype_code(g.dtype), d.data_ptr(), B, H, W, view, mode, stream_ptr())
        return d, None, None


def view_extract_all(views, specs, dtype=torch.float32):
    """The cameras ``specs`` = ((view, mode), ...) of every scene as NHWC images with SpatialMappingCNN's rot90 / flip
    folded in (spatial_bb/components.py:34-62); mode 0 as is, 1 rot90(1,[2,3]), 2 rot90(1,[3,2]), 3 flip([2,3]).
    Differentiable in the views; each view may be extracted once."""
    views = as_view_batch(views)
    specs = tuple((int(v), int(m)) for v, m in specs)
    if len({v for v, _ in specs}) != len(specs):
        raise ValueError(f"view_extract_all: a view is extracted more than once in {specs}")
    return ViewExtract.apply(views, specs, dtype)


def view_extract(views, view: int, mode: int, dtype=torch.float32):
    """One camera of every scene as an NHWC image (see view_extract_all)."""
    return view_extract_all(views, ((view, mode),), dtype)[0]


class TileNHWC(torch.autograd.Function):
    """torch.cat of NHWC blocks into one tensor [B,H,W,C]: ``offsets[i] = (oy, ox, oc)`` of block i.
    Backward hands every block its window of the gradient."""

    @staticmethod
    def forward(ctx, shape, offsets, *blocks):
        B, H, W, Cn = shape
        first = blocks[0]
        out = torch.empty(B, H, W, Cn, dtype=first.dtype, device=first.device)
        st, code = stream_ptr(), dtype_code(first.dtype)
        ctx.meta = (shape, offsets, [tuple(b.shape) for b in blocks], first.dtype)
        for blk, (oy, ox, oc) in zip(blocks, offsets):
            blk = _c(blk)
            _, h, w, c = blk.shape
            call("dd_nhwc_place", blk.data_ptr(), out.data_ptr(), code, B, h, w, c, H, W, Cn, oy, ox, oc, 0, st)
        return out

    @staticmethod
    def backward(ctx, g):
        (B, H, W, Cn), offsets, shapes, dtype = ctx.meta
        g = _c(g.to(dtype))
        st, code = stream_ptr(), dtype_code(dtype)
        grads = []
        for (oy, ox, oc), shp in zip(offsets, shapes):
            d = torch.empty(shp, dtype=dtype, device=g.device)
            call("dd_nhwc_place", d.data_ptr(), g.data_ptr(), code, B, shp[1], shp[2], shp[3], H, W, Cn, oy, ox, oc, 1, st)
            grads.append(d)
        return (None, None, *grads)


def tile_nhwc(shape, offsets, blocks):
    return TileNHWC.apply(tuple(shape), tuple(offsets), *blocks)


def _bce_prob_ws(device):
    n = int(_lib.load().dd_bce_prob_workspace_bytes())
    return _ws.get("bce_prob", n, device, zero=True), n


class BceProb(torch.autograd.Function):
    """F.binary_cross_entropy(pred, target) on probabilities, mean (spatial_w_rm.py:131)."""

    @staticmethod
    def forward(ctx, pred, target):
        _require_cuda(pred, target)
        pred, target = _c(pred.float()), _c(target.float())
        if pred.numel() != target.numel():
            raise RuntimeError("bce_prob: prediction and target differ in size")
        out = torch.empty(1, dtype=torch.float32, device=pred.device)
        ws, n = _bce_prob_ws(pred.device)
        call("dd_bce_prob_fwd", pred.data_ptr(), target.data_ptr(), out.data_ptr(), ws.data_ptr(), n, pred.numel(), stream_ptr())
        ctx.save_for_backward(pred, target)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        pred, target = ctx.saved_tensors
        d = torch.empty_like(pred)
        gg = _c(g.float().reshape(1))
        call("dd_bce_prob_bwd", pred.data_ptr(), target.data_ptr(), gg.data_ptr(), d.data_ptr(), pred.numel(), stream_ptr())
        return d, None


def bce_prob(pred, target):
    return BceProb.apply(pred, target)


# --------------------------------------------------------------------------------------------
# training target of the box model: boxes_to_binary_map (utils/bb_to_img.py:5-21) on the device
MAP_SIZE = 800


class _BoxStaging:
    """Per-device ring of two staging slots for ``boxes_to_map``'s inputs (offsets, then boxes), so host boxes cross in
    one asynchronous copy.  A slot is (pinned host buffer, device buffer, event); the event is recorded after the kernel
    that reads the slot's device buffer.  Before a slot is reused, waiting on its event guarantees that the copy out of
    the pinned buffer and the kernel reading the device buffer have both finished, whichever stream they ran on.  With
    two slots the host waits for the call before last, not the last one, so it can run a step ahead of the device.
    Buffers grow to the next power of two, so slowly growing batches do not re-pin memory on every call."""

    SLOTS = 2

    def __init__(self):
        self._rings = {}

    def get(self, nbytes: int, device):
        ring = self._rings.setdefault(device.index, {"next": 0, "slots": [None] * self.SLOTS})
        i = ring["next"]
        ring["next"] = (i + 1) % self.SLOTS
        slot = ring["slots"][i]
        if slot is None or slot[0].numel() < nbytes:
            if slot is not None:
                slot[2].synchronize()                        # the old buffers' last copy and reader have finished
            n = 1 << max(12, (nbytes - 1).bit_length())
            slot = (torch.empty(n, dtype=torch.uint8).pin_memory(), torch.empty(n, dtype=torch.uint8, device=device),
                    torch.cuda.Event())
            ring["slots"][i] = slot
        return slot


_box_staging = _BoxStaging()


def boxes_to_map(boxes: Sequence[torch.Tensor], device) -> torch.Tensor:
    """The dataloader's per-scene boxes ([N,2,4]: metres; rows x / y; columns fl, fr, bl, br; N may be 0), all float32 or
    all float64, on the host or on ``device`` -> float32 [B,800,800] of 0./1. on ``device``: exactly
    ``boxes_to_binary_map`` of each scene (the reference's Pillow fill, arithmetic in the boxes' own dtype).
    Host boxes travel with their offsets through reused pinned buffers (_BoxStaging) in one asynchronous copy."""
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("boxes_to_map runs on CUDA (sm_100a) only; there is no CPU fallback on this path.")
    if device.index is None:
        device = torch.device("cuda", torch.cuda.current_device())
    boxes = list(boxes)
    dtypes = set()
    for b in boxes:
        if not torch.is_tensor(b) or b.dim() != 3 or tuple(b.shape[1:]) != (2, 4):
            raise ValueError(f"boxes_to_map: every scene's boxes must have shape [N,2,4], got "
                             f"{tuple(b.shape) if torch.is_tensor(b) else type(b).__name__}")
        if b.dtype not in (torch.float32, torch.float64):
            raise ValueError(f"boxes_to_map: boxes dtype must be float32 or float64, got {b.dtype}")
        dtypes.add(b.dtype)
    if len(dtypes) > 1:
        raise ValueError("boxes_to_map: the batch mixes float32 and float64 boxes (dtype); the fill's arithmetic "
                         "differs per dtype, so convert them explicitly")
    B = len(boxes)
    out = torch.empty(B, MAP_SIZE, MAP_SIZE, dtype=torch.float32, device=device)
    if B == 0:
        return out
    dtype = dtypes.pop()
    counts = [int(b.shape[0]) for b in boxes]
    offsets = [0]
    for c in counts:
        offsets.append(offsets[-1] + c)
    total = offsets[-1]
    on_device = all(b.is_cuda and b.device == device for b in boxes)
    box_at = (4 * (B + 1) + 15) // 16 * 16
    nbytes = box_at + (0 if on_device else total * 8 * dtype.itemsize)
    with torch.cuda.device(device):
        host, dev, done = _box_staging.get(nbytes, device)
        done.synchronize()                                   # this slot's last copy and kernel have finished
        host[:4 * (B + 1)].view(torch.int32).copy_(torch.tensor(offsets, dtype=torch.int32))
        if not on_device and total:
            torch.cat([b.detach().reshape(-1, 8).cpu() for b in boxes],
                      out=host[box_at:nbytes].view(dtype).view(total, 8))
        cur = torch.cuda.current_stream(device)
        dev[:nbytes].copy_(host[:nbytes], non_blocking=True)
        if on_device and total:
            src = _c(torch.cat([b.detach().reshape(-1, 8) for b in boxes]))
        else:
            src = dev[box_at:]
        call("dd_boxes_to_map", src.data_ptr(), int(dtype == torch.float64), dev.data_ptr(), B, out.data_ptr(),
             cur.cuda_stream)
        done.record(cur)
        if on_device and total:
            src.record_stream(cur)
    return out
