"""Which engine runs each pass of a generic conv layer (csrc/conv_generic.cu, tc_plan), checked on the host: the choice,
the workspace size and the argument checks that return before any launch depend only on the descriptor and the dtype, so
they are compared here, without a device, with a restatement of the rules and with sizes pinned from earlier builds."""
import ctypes
import itertools

import pytest

from driving_dirty_b200 import _lib, ops
from tests.test_kernels_gpu import GENERIC_LAYERS, TC_LAYERS

DD_ERR_BAD_ARG, DD_ERR_WORKSPACE = -1, -3

# (gathered, produced) channel pairs of the tcgen05 implicit-GEMM kernel (conv_dil_tc.cu) and the channel counts of its
# weight-gradient kernel (conv_dil_wgrad_tc.cu)
DIL_PAIRS = {(96, 64), (64, 32), (32, 16), (32, 32), (64, 96), (32, 64)}
WGRAD_K, WGRAD_N = {32, 64, 96}, {32, 64}


def pad32(c):
    return 32 if c in (8, 16) else c


def tc_expected(d, dtype, pass_):
    """pass 0 forward, 1 input gradient, 2 weight gradient"""
    if not (dtype == _lib.DD_BF16 and d.sh == d.sw == 1 and d.kh == d.kw and d.dh == d.dw and d.ph == d.pw):
        return False
    taps_ok = d.kh in (3, 7) and 1 <= d.dh <= 7
    if pass_ == 0:      # gathered x: 8 / 16 channels padded to 32; produced y: 8 channels computed as 16, then narrowed
        return taps_ok and (pad32(d.Cin), 16 if d.Cout == 8 else d.Cout) in DIL_PAIRS
    if pass_ == 1:      # gathered dy: 8 / 16 channels padded to 32; produced dx as it is
        return taps_ok and (pad32(d.Cout), d.Cin) in DIL_PAIRS
    return taps_ok and pad32(d.Cin) in WGRAD_K and pad32(d.Cout) in WGRAD_N      # x and dy: 8 / 16 channels padded to 32


def desc(B, cin, cout, hw, k, s=1, p=0, d=1, transposed=False):
    k, s, p, d = ops._pair(k), ops._pair(s), ops._pair(p), ops._pair(d)
    ho = ops.conv_out_size(hw[0], k[0], s[0], p[0], d[0], transposed)
    wo = ops.conv_out_size(hw[1], k[1], s[1], p[1], d[1], transposed)
    return ops._conv_desc(B, cin, cout, hw[0], hw[1], ho, wo, k, s, p, d, transposed)


def test_tc_supported_follows_the_rules():
    lib = _lib.load()
    chans = (1, 3, 8, 16, 32, 64, 96)
    kernels = (1, 2, 3, 7, (1, 50), (52, 1), (1, 24), (3, 7))
    strides = (1, 2, (1, 2), (3, 2))
    dilations = (1, 3, 7, (3, 1))
    pads = (0, 1, (1, 0))
    taken = [0, 0, 0]
    for cin, cout, k, s, dil, p, t in itertools.product(chans, chans, kernels, strides, dilations, pads, (False, True)):
        dsc = desc(2, cin, cout, (400, 410), k, s, p, dil, t)
        for dtype, pass_ in itertools.product((_lib.DD_F32, _lib.DD_BF16), (0, 1, 2)):
            want = tc_expected(dsc, dtype, pass_)
            got = lib.dd_conv2d_tc_supported(ctypes.byref(dsc), dtype, pass_)
            assert got == int(want), (cin, cout, k, s, dil, p, t, dtype, pass_)
            taken[pass_] += want
    assert all(taken), taken
    assert lib.dd_conv2d_tc_supported(None, _lib.DD_BF16, 0) == 0
    bad = desc(2, 0, 32, (40, 40), 3, 1, 1, 1, True)
    assert all(lib.dd_conv2d_tc_supported(ctypes.byref(bad), _lib.DD_BF16, q) == 0 for q in (0, 1, 2))


# every generic conv layer of the bench's ae (B = 64) and bb (B = 32) steps:
# name: (transposed, cin, cout, kernel, stride, pad, dilation, input (H, W), batch)
MODEL_LAYERS = {
    "Decoder.dc1": (True, 64, 32, 3, 1, 1, 1, (128, 153), 64),
    "Decoder.dc2": (True, 32, 32, 3, 1, 1, 1, (128, 153), 64),
    "Decoder.dc3": (True, 32, 32, 2, 2, 0, 1, (128, 153), 64),
    "Decoder.dc4": (True, 32, 3, 1, 1, 0, 1, (256, 306), 64),
    "SpatialMappingCNN.f_conv": (False, 3, 32, (52, 1), (3, 2), 1, 1, (306, 256), 32),      # b_conv alike
    "SpatialMappingCNN.fl_conv": (False, 3, 32, (1, 50), (3, 2), 0, 1, (256, 306), 32),     # fr / bl / br_conv alike
    "SpatialMappingCNN.out_conv": (False, 32, 32, 3, 1, 0, 1, (258, 258), 32),
    "RoadMapBoxesMergingCNN.ss_conv": (False, 32, 32, (1, 24), (1, 7), 0, 1, (128, 918), 32),
    "RoadMapBoxesMergingCNN.ss_deconv": (True, 32, 32, 2, 2, 0, 1, (128, 128), 32),
    "RoadMapBoxesMergingCNN.rm_conv_1": (False, 1, 32, 7, 3, 1, 3, (800, 800), 32),
    "RoadMapBoxesMergingCNN.rm_conv_2": (False, 32, 32, 3, 1, 0, 3, (262, 262), 32),
    "RoadMapBoxesMergingCNN.up_conv_1": (True, 96, 64, 7, 1, 0, 7, (256, 256), 32),
    "RoadMapBoxesMergingCNN.up_conv_2": (True, 64, 32, 7, 1, 0, 7, (298, 298), 32),
    "RoadMapBoxesMergingCNN.up_conv_3": (True, 32, 16, 7, 1, 0, 7, (340, 340), 32),
    "RoadMapBoxesMergingCNN.up_conv_4": (True, 16, 8, 7, 1, 0, 3, (382, 382), 32),
    "RoadMapBoxesMergingCNN.up_conv_5": (True, 8, 1, 2, 2, 0, 1, (400, 400), 32),
}


def all_layers():
    out = {}
    for name, (t, cin, cout, k, s, p, d, hw, B) in MODEL_LAYERS.items():
        out[name] = desc(B, cin, cout, hw, k, s, p, d, t)
    for name, L in GENERIC_LAYERS.items():
        out["GENERIC_LAYERS." + name] = desc(2, L["cin"], L["cout"], L["hw"], L["k"], L["s"], L["p"], L["d"], L["t"])
    for name, (t, cin, cout, k, p, d, hw, B) in TC_LAYERS.items():
        out["TC_LAYERS." + name] = desc(B, cin, cout, hw, k, 1, p, d, t)
    return out


# dd_conv2d_workspace_bytes of each layer above
WORKSPACE_BYTES = {
    "Decoder.dc1": 38874112,
    "Decoder.dc2": 38874112,
    "Decoder.dc3": 38874112,
    "Decoder.dc4": 38805504,
    "GENERIC_LAYERS.dc1_convT_64_32_k3p1": 38874112,
    "GENERIC_LAYERS.dc3_convT_32_32_k2s2": 38874112,
    "GENERIC_LAYERS.dc4_convT_32_3_k1": 38805504,
    "GENERIC_LAYERS.out_conv_32_32_k3_valid": 38874112,
    "GENERIC_LAYERS.rm_conv1_1_32_k7s3d3p1": 38874112,
    "GENERIC_LAYERS.rm_conv2_32_32_k3_d3": 38874112,
    "GENERIC_LAYERS.ss_conv_32_32_1x24_s17": 38874112,
    "GENERIC_LAYERS.strip_conv_3_32_1x50_s32": 38874112,
    "GENERIC_LAYERS.strip_conv_3_32_52x1_s32_p1": 38874112,
    "GENERIC_LAYERS.up_conv1_convT_96_64_k7d7": 38949888,
    "GENERIC_LAYERS.up_conv4_convT_16_8_k7d3": 38919936,
    "GENERIC_LAYERS.up_conv5_convT_8_1_k2s2": 38800384,
    "RoadMapBoxesMergingCNN.rm_conv_1": 38874112,
    "RoadMapBoxesMergingCNN.rm_conv_2": 38874112,
    "RoadMapBoxesMergingCNN.ss_conv": 38874112,
    "RoadMapBoxesMergingCNN.ss_deconv": 38874112,
    "RoadMapBoxesMergingCNN.up_conv_1": 38949888,
    "RoadMapBoxesMergingCNN.up_conv_2": 38874112,
    "RoadMapBoxesMergingCNN.up_conv_3": 337691648,
    "RoadMapBoxesMergingCNN.up_conv_4": 665353216,
    "RoadMapBoxesMergingCNN.up_conv_5": 38800384,
    "SpatialMappingCNN.f_conv": 38874112,
    "SpatialMappingCNN.fl_conv": 38874112,
    "SpatialMappingCNN.out_conv": 38874112,
    "TC_LAYERS.dc1_64_32_k3p1": 38874112,
    "TC_LAYERS.dc2_32_32_k3p1": 38874112,
    "TC_LAYERS.out_conv_32_32_k3": 38874112,
    "TC_LAYERS.rm_conv2_32_32_k3d3": 38874112,
    "TC_LAYERS.up_conv1_96_64_k7d7": 38949888,
    "TC_LAYERS.up_conv2_64_32_k7d7": 38874112,
    "TC_LAYERS.up_conv3_32_16_k7d7": 39520896,
    "TC_LAYERS.up_conv4_16_8_k7d3": 40596224,
}


@pytest.mark.parametrize("name", sorted(all_layers()))
def test_workspace_bytes_are_pinned(name):
    dsc = all_layers()[name]
    assert _lib.load().dd_conv2d_workspace_bytes(ctypes.byref(dsc)) == WORKSPACE_BYTES[name]


def test_checks_before_any_launch():
    """Argument and workspace errors come back before anything is enqueued (no device is touched)."""
    lib = _lib.load()
    P = 1 << 20                          # never dereferenced: every call below returns before a launch
    bf16 = _lib.DD_BF16

    def fwd(d, ws, act=0):
        return lib.dd_conv2d_fwd(P, P, P, P, ctypes.byref(d), bf16, act, P, ws, None)

    def dgrad(d, ws):
        return lib.dd_conv2d_dgrad(P, P, None, P, ctypes.byref(d), bf16, P, ws, None)

    def wgrad(d, ws):
        return lib.dd_conv2d_wgrad(P, P, P, P, ctypes.byref(d), bf16, P, ws, None)

    layers = all_layers()
    plain = layers["RoadMapBoxesMergingCNN.up_conv_1"]          # tensor cores as it is
    padded = layers["RoadMapBoxesMergingCNN.up_conv_4"]         # tensor cores through 32-channel copies, every pass
    generic = layers["RoadMapBoxesMergingCNN.rm_conv_1"]        # CUDA cores
    for d in (plain, padded, generic):
        n = lib.dd_conv2d_workspace_bytes(ctypes.byref(d))
        bad = ops._conv_desc(d.B, 0, d.Cout, d.Hi, d.Wi, d.Ho, d.Wo, (d.kh, d.kw), (d.sh, d.sw), (d.ph, d.pw),
                             (d.dh, d.dw), d.transposed)
        assert fwd(bad, n) == dgrad(bad, n) == wgrad(bad, n) == DD_ERR_BAD_ARG
        assert fwd(d, n, act=3) == DD_ERR_BAD_ARG
        assert fwd(d, 0) == dgrad(d, 0) == wgrad(d, 0) == DD_ERR_WORKSPACE
        assert wgrad(d, n - 1) == DD_ERR_WORKSPACE
        empty = ops._conv_desc(0, d.Cin, d.Cout, d.Hi, d.Wi, d.Ho, d.Wo, (d.kh, d.kw), (d.sh, d.sw), (d.ph, d.pw),
                               (d.dh, d.dw), d.transposed)
        assert fwd(empty, 0) == dgrad(empty, 0) == 0 and wgrad(empty, n) == DD_ERR_BAD_ARG
        assert lib.dd_conv2d_fwd(None, P, P, P, ctypes.byref(d), bf16, 0, P, n, None) == DD_ERR_BAD_ARG
    # the zero-padded passes need the whole workspace, copies included
    n = lib.dd_conv2d_workspace_bytes(ctypes.byref(padded))
    assert fwd(padded, n - 1) == dgrad(padded, n - 1) == DD_ERR_WORKSPACE
