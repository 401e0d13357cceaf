"""ReLU sign words (include/dd_b200.h, dd_*_bits): the c1 / c2 forward kernels store, beside a1 / a2, one uint32 per pixel
whose bit c is (stored bf16 activation of channel c) > 0, and the c2 / c3 input gradients read those words instead of the
64-byte activations.  Everything here is bit for bit: the activations against the plain forward, the words against the
activations they describe, the input gradients against the activation-mask form, the encoder's weight gradients with the
switch on and off."""
import pytest
import torch

from oracle import scene_oracle as so

pytestmark = pytest.mark.gpu

GUARD = 16                        # sentinel words on each side of a sign-word buffer (keeps the 8-byte alignment)
SENTINEL = 0x5A5A5A5A
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def lib():
    from driving_dirty_b200 import _lib
    assert torch.cuda.is_available()
    return _lib


def pack(act):
    """[B,H,W,32] bf16 -> the sign words as int64 in [0, 2^32): bit c = act[..., c] > 0"""
    shifts = torch.arange(32, device=act.device, dtype=torch.int64)
    return ((act > 0).to(torch.int64) << shifts).sum(-1)


def words(t):
    return t.to(torch.int64) & 0xFFFFFFFF


class Guarded:
    """int32 sign-word buffer of `n` words, pre-filled with a sentinel, with sentinel guard bands before and after"""

    def __init__(self, shape):
        self.shape = shape
        n = 1
        for s in shape:
            n *= s
        self.n = n
        self.buf = torch.full((n + 2 * GUARD,), SENTINEL, dtype=torch.int32, device="cuda")

    def ptr(self):
        return self.buf[GUARD:].data_ptr()

    def bits(self):
        return self.buf[GUARD:GUARD + self.n].view(self.shape)

    def guards_intact(self):
        return bool((self.buf[:GUARD] == SENTINEL).all()) and bool((self.buf[GUARD + self.n:] == SENTINEL).all())


def conv_params(cin, seed, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    bound = (cin * 9) ** -0.5
    w = (torch.rand(32, cin, 3, 3, generator=g) * 2 - 1) * bound * scale
    b = (torch.rand(32, generator=g) * 2 - 1) * bound
    return w.cuda(), b.cuda()


def relu_act(B, H, W, seed):
    """a post-ReLU bf16 activation with many zeros, some of them -0"""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, H, W, 32, generator=g).clamp_min(0)
    x[torch.rand(B, H, W, 32, generator=g) < 0.1] = -0.0
    return x.to(BF16).cuda()


# ------------------------------------------------------------------------------- forward ------
C1_CASES = [  # (B, H, W, flags, source); views: Wm = 6W, mosaics: any Wm (odd included)
    (1, 16, 20, 1, "views"), (2, 33, 7, 3, "views"), (3, 70, 50, 1, "views"), (2, 37, 211, 0, "mosaic"),
    (1, 65, 129, 2, "mosaic"), (2, 256, 306, 3, "views"),
]


def c1_source(B, H, W, flags, kind, seed):
    g = torch.Generator().manual_seed(seed)
    shape = (B, 6, 3, H, W) if kind == "views" else (B, 3, H, W)
    raw = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g)
    src = raw if flags & 2 else raw.float() / 255
    return src.cuda(), (6 * W if kind == "views" else W)


@pytest.mark.parametrize("B,H,W,flags,kind", C1_CASES)
def test_c1_fwd_bits(lib, B, H, W, flags, kind):
    src, Wm = c1_source(B, H, W, flags, kind, seed=H + W)
    w, b = conv_params(3, seed=H)
    st = lib.stream_ptr()
    ref = torch.empty(B, H, Wm, 32, dtype=BF16, device="cuda")
    lib.call("dd_conv_c1_fwd", src.data_ptr(), flags, w.data_ptr(), b.data_ptr(), ref.data_ptr(), lib.DD_BF16, B, H, Wm, 2, st)
    out = torch.full_like(ref, float("nan"))
    bits = Guarded((B, H, Wm))
    lib.call("dd_conv_c1_fwd_bits", src.data_ptr(), flags, w.data_ptr(), b.data_ptr(), out.data_ptr(), bits.ptr(),
             lib.DD_BF16, B, H, Wm, 0, st)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    assert torch.equal(words(bits.bits()), pack(ref))
    assert bits.guards_intact()


C2_CASES = [(1, 16, 20), (2, 33, 7), (3, 70, 131), (2, 65, 129), (1, 64, 256), (2, 256, 1836)]


@pytest.mark.parametrize("B,H,W", C2_CASES)
def test_c2_fwd_bits(lib, B, H, W):
    x = relu_act(B, H, W, seed=W)
    w, b = conv_params(32, seed=H)
    st = lib.stream_ptr()
    ref = torch.empty_like(x)
    lib.call("dd_conv3x3_c32_fwd", x.data_ptr(), w.data_ptr(), b.data_ptr(), ref.data_ptr(), lib.DD_BF16, B, H, W, 1, 2, st)
    out = torch.full_like(x, float("nan"))
    bits = Guarded((B, H, W))
    lib.call("dd_conv3x3_c32_fwd_bits", x.data_ptr(), w.data_ptr(), b.data_ptr(), out.data_ptr(), bits.ptr(), lib.DD_BF16,
             B, H, W, 1, 0, st)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))
    assert torch.equal(words(bits.bits()), pack(ref))
    assert bits.guards_intact()


# +0, -0, positive below half of bf16's smallest subnormal (rounds to +0), exactly half of it (ties to even: +0), bf16's
# smallest subnormal, bf16's smallest normal, +1, -1
EDGE_BIAS = [0.0, -0.0, 2.0 ** -136, 2.0 ** -134, 2.0 ** -133, 2.0 ** -126, 1.0, -1.0]


def test_sign_words_at_the_rounding_edge(lib):
    """zero weights: every output is relu(bias) rounded to bf16, so the bias pins the words' rounding edge"""
    B, H, W = 1, 5, 20
    st = lib.stream_ptr()
    bias = torch.tensor(EDGE_BIAS * 4, dtype=torch.float32, device="cuda")
    src, Wm = c1_source(B, H, W, 1, "views", seed=3)
    w1 = torch.zeros(32, 3, 3, 3, device="cuda")
    a1 = torch.empty(B, H, Wm, 32, dtype=BF16, device="cuda")
    bits1 = Guarded((B, H, Wm))
    lib.call("dd_conv_c1_fwd_bits", src.data_ptr(), 1, w1.data_ptr(), bias.data_ptr(), a1.data_ptr(), bits1.ptr(),
             lib.DD_BF16, B, H, Wm, 2, st)
    x = relu_act(B, H, Wm, seed=4)
    w2 = torch.zeros(32, 32, 3, 3, device="cuda")
    a2 = torch.empty_like(x)
    bits2 = Guarded((B, H, Wm))
    lib.call("dd_conv3x3_c32_fwd_bits", x.data_ptr(), w2.data_ptr(), bias.data_ptr(), a2.data_ptr(), bits2.ptr(),
             lib.DD_BF16, B, H, Wm, 1, 2, st)
    torch.cuda.synchronize()
    for act, bits in ((a1, bits1), (a2, bits2)):
        assert torch.equal(words(bits.bits()), pack(act)) and bits.guards_intact()
        expect = sum(1 << c for c in range(32) if torch.tensor(EDGE_BIAS[c % 8]).relu().to(BF16) > 0)
        assert bool((words(bits.bits()) == expect).all())


# ------------------------------------------------------------------------------- input gradient ------
DGRAD_CASES = [(1, 16, 20), (2, 33, 7), (3, 70, 131), (2, 65, 129), (1, 31, 257), (2, 256, 1836)]


@pytest.mark.parametrize("stride", [1, 2])
@pytest.mark.parametrize("B,H,W", DGRAD_CASES)
def test_dgrad_bits_equals_activation_mask(lib, B, H, W, stride):
    x = relu_act(B, H, W, seed=H * 7 + W)
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    g = torch.Generator().manual_seed(W)
    dy = torch.randn(B, Ho, Wo, 32, generator=g).to(BF16).cuda()
    w, _ = conv_params(32, seed=W)
    bits = pack(x).to(torch.int32)        # wraps to the same 32 bits
    st = lib.stream_ptr()
    ref = torch.empty_like(x)
    lib.call("dd_conv3x3_c32_dgrad", dy.data_ptr(), w.data_ptr(), x.data_ptr(), ref.data_ptr(), lib.DD_BF16, B, H, W, stride,
             2, st)
    out = torch.full_like(x, float("nan"))
    lib.call("dd_conv3x3_c32_dgrad_bits", dy.data_ptr(), w.data_ptr(), bits.data_ptr(), out.data_ptr(), lib.DD_BF16, B, H, W,
             stride, 0, st)
    torch.cuda.synchronize()
    assert torch.equal(out.view(torch.int16), ref.view(torch.int16))


# ------------------------------------------------------------------------------- whole encoder ------
@pytest.mark.parametrize("B,H,W", [(2, 40, 50), (1, 256, 306)])
@pytest.mark.parametrize("as_bytes", [False, True])
def test_encoder_stack_bits_switch(lib, B, H, W, as_bytes):
    from driving_dirty_b200 import ops
    torch.manual_seed(11)
    convs = [torch.nn.Conv2d(3, 32, 3, padding=1), torch.nn.Conv2d(32, 32, 3, padding=1),
             torch.nn.Conv2d(32, 32, 3, stride=2, padding=1)]
    c1, c2, c3 = (c.cuda() for c in convs)
    views, _ = so.synthetic_scene_batch(B, H, W, map_hw=4, seed=12)
    inp = (views * 255).round().to(torch.uint8).cuda() if as_bytes else views.cuda()
    params = [c1.weight, c1.bias, c2.weight, c2.bias, c3.weight, c3.bias]
    res = {}
    saved = ops.RELU_MASK_BITS
    try:
        for on in (True, False):
            ops.RELU_MASK_BITS = on
            out = ops.encoder_conv_stack(inp, c1, c2, c3, act_dtype=BF16)
            gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(13)).to(out.dtype).cuda()
            grads = torch.autograd.grad(out, params, gout)
            res[on] = (out.detach().clone(), [t.clone() for t in grads])
    finally:
        ops.RELU_MASK_BITS = saved
    assert torch.equal(res[True][0].view(torch.int16), res[False][0].view(torch.int16))
    for a, b in zip(res[True][1], res[False][1]):
        assert torch.equal(a.view(torch.int32), b.view(torch.int32))


# ------------------------------------------------------------------------------- errors ------
def test_bits_entry_points_reject_bad_calls(lib):
    L = lib.load()
    B, H, W = 1, 8, 12
    st = lib.stream_ptr()
    views = torch.rand(B, 6, 3, H, W, device="cuda")
    x = relu_act(B, H, 6 * W, seed=1)
    w1, b = conv_params(3, seed=1)
    w2, _ = conv_params(32, seed=2)
    out = torch.full_like(x, 7.0)
    bits = torch.full((B * H * 6 * W + 2,), SENTINEL, dtype=torch.int32, device="cuda")
    Wm = 6 * W
    p = lambda t: t.data_ptr()  # noqa: E731
    c1 = lambda o, bp, dt, impl: L.dd_conv_c1_fwd_bits(p(views), 1, p(w1), p(b), o, bp, dt, B, H, Wm, impl, st)  # noqa: E731
    fw = lambda i, o, bp, dt, s, impl: L.dd_conv3x3_c32_fwd_bits(i, p(w2), p(b), o, bp, dt, B, H, Wm, s, impl, st)  # noqa: E731
    dg = lambda d, bp, o, dt, s, impl: L.dd_conv3x3_c32_dgrad_bits(d, p(w2), bp, o, dt, B, H, Wm, s, impl, st)  # noqa: E731
    cases = [
        (lambda: c1(p(out), p(bits), lib.DD_F32, 0), -2, "tensor-core"),
        (lambda: c1(p(out), p(bits), lib.DD_BF16, lib.IMPL_SIMT), -2, "tensor-core"),
        (lambda: c1(p(out), None, lib.DD_BF16, 0), -1, "null"),
        (lambda: c1(p(out), p(bits) + 4, lib.DD_BF16, 0), -4, "aligned"),
        (lambda: fw(p(x), p(out), p(bits), lib.DD_F32, 1, 0), -2, "tensor-core"),
        (lambda: fw(p(x), p(out), p(bits), lib.DD_BF16, 1, lib.IMPL_SIMT), -2, "tensor-core"),
        (lambda: fw(p(x), p(out), p(bits), lib.DD_BF16, 2, 0), -2, "stride"),
        (lambda: fw(p(x), p(out), None, lib.DD_BF16, 1, 0), -1, "null"),
        (lambda: fw(p(x), p(out), p(bits) + 4, lib.DD_BF16, 1, 0), -4, "aligned"),
        (lambda: dg(p(x), p(bits), p(out), lib.DD_F32, 2, 0), -2, "tensor-core"),
        (lambda: dg(p(x), p(bits), p(out), lib.DD_BF16, 1, lib.IMPL_SIMT), -2, "tensor-core"),
        (lambda: dg(p(x), None, p(out), lib.DD_BF16, 1, 0), -1, "null"),
        (lambda: dg(None, p(bits), p(out), lib.DD_BF16, 2, 0), -1, "null"),
        (lambda: dg(p(x), p(bits) + 4, p(out), lib.DD_BF16, 2, 0), -4, "aligned"),
        (lambda: dg(p(x), p(bits), p(out), lib.DD_BF16, 3, 0), -2, "stride"),
    ]
    for i, (fn, code, word) in enumerate(cases):
        assert fn() == code, f"case {i}"
        assert word in lib.last_error(), f"case {i}: {lib.last_error()}"
    torch.cuda.synchronize()
    assert bool((out == 7.0).all()) and bool((bits == SENTINEL).all())      # nothing was written
