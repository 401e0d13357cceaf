"""SpatialMappingCNN / BoxesMergingCNN / RoadMapBoxesMergingCNN with the reference's constructor
order, attribute names and state_dict keys (src/bounding_box_model/spatial_bb/components.py),
running on libdd_b200.so.  The nn.Conv2d / nn.ConvTranspose2d submodules are parameter containers;
``forward`` keeps the reference's NCHW fp32 signature, ``forward_nhwc`` is the internal path that
stays in the library's NHWC layout between layers."""
import torch
from torch import nn

from ... import ops
from ...autoencoder.components import resolve_dtype

# (layer, camera index, transform, canvas cell (row, col)): components.py:34-73.
# transform 0 as is, 1 rot90(1,[2,3]), 2 rot90(1,[3,2]), 3 flip([2,3])
_STRIPS = (("bl_conv", 3, 0, (0, 0)), ("fl_conv", 0, 0, (0, 1)), ("b_conv", 4, 1, (1, 0)), ("f_conv", 1, 2, (1, 1)),
           ("br_conv", 5, 3, (2, 0)), ("fr_conv", 2, 3, (2, 1)))


class SpatialMappingCNN(nn.Module):
    """Six strip convs on the plain / rotated / flipped cameras, tiled 3 x 2 into a square canvas,
    then a 3x3 valid conv: [B,6,3,256,306] -> [B,32,256,256] (components.py:6-77)."""

    def __init__(self, compute_dtype="fp32"):
        super().__init__()
        self.f_conv = nn.Conv2d(3, 32, kernel_size=(52, 1), stride=(3, 2), padding=(1))
        self.fl_conv = nn.Conv2d(3, 32, kernel_size=(1, 50), stride=(3, 2))
        self.fr_conv = nn.Conv2d(3, 32, kernel_size=(1, 50), stride=(3, 2))
        self.b_conv = nn.Conv2d(3, 32, kernel_size=(52, 1), stride=(3, 2), padding=(1))
        self.bl_conv = nn.Conv2d(3, 32, kernel_size=(1, 50), stride=(3, 2))
        self.br_conv = nn.Conv2d(3, 32, kernel_size=(1, 50), stride=(3, 2))
        self.out_conv = nn.Conv2d(32, 32, kernel_size=(3, 3))
        self.compute_dtype = resolve_dtype(compute_dtype)

    def forward_nhwc(self, x):
        views = ops.as_view_batch(x)
        cells, offsets = [], []
        imgs = ops.view_extract_all(views, [(cam, mode) for _, cam, mode, _ in _STRIPS], self.compute_dtype)
        for (name, cam, mode, (r, c)), img in zip(_STRIPS, imgs):
            cells.append((r, c, ops.conv2d_nhwc(img, getattr(self, name), relu=True)))
        hs = [max(t.shape[1] for rr, _, t in cells if rr == r) for r in range(3)]
        w0 = max(t.shape[2] for _, cc, t in cells if cc == 0)
        for r, c, t in cells:       # torch.cat needs equal heights per row and equal row widths
            assert t.shape[1] == hs[r] and (c == 1 or t.shape[2] == w0), "view size does not tile into a canvas"
        H = sum(hs)
        W = w0 + cells[1][2].shape[2]
        blocks = [t for _, _, t in cells]
        offsets = [(sum(hs[:r]), 0 if c == 0 else w0, 0) for r, c, _ in cells]
        canvas = ops.tile_nhwc((views.shape[0], H, W, 32), offsets, blocks)
        return ops.conv2d_nhwc(canvas, self.out_conv, relu=True)

    def forward(self, x):
        return ops.to_nchw(self.forward_nhwc(x))


class _MergingBase(nn.Module):
    def _ssr_branch(self, ssr):
        ssr = ops.conv2d_nhwc(ssr, self.ss_conv, relu=True)
        return ops.conv2d_nhwc(ssr, self.ss_deconv, relu=True)

    @staticmethod
    def _concat(blocks):
        B, H, W, _ = blocks[0].shape
        offs, oc = [], 0
        for b in blocks:
            offs.append((0, 0, oc))
            oc += b.shape[3]
        return ops.tile_nhwc((B, H, W, oc), offs, blocks)


class BoxesMergingCNN(_MergingBase):
    """No-roadmap variant (components.py:80-119)."""

    def __init__(self, compute_dtype="fp32"):
        super().__init__()
        self.ss_conv = nn.Conv2d(32, 32, kernel_size=(1, 24), stride=(1, 7))
        self.ss_deconv = nn.ConvTranspose2d(32, 32, kernel_size=2, stride=2)
        self.up_conv_1 = nn.ConvTranspose2d(64, 32, kernel_size=8, stride=1, dilation=8)
        self.up_conv_2 = nn.ConvTranspose2d(32, 16, kernel_size=8, stride=1, dilation=8)
        self.up_conv_3 = nn.ConvTranspose2d(16, 8, kernel_size=6, stride=1, dilation=6, output_padding=2)
        self.up_conv_4 = nn.ConvTranspose2d(8, 1, kernel_size=2, stride=2)
        self.compute_dtype = resolve_dtype(compute_dtype)

    def forward_nhwc(self, ssr, spatial_map):
        x = self._concat([self._ssr_branch(ssr), spatial_map])
        x = ops.conv2d_nhwc(x, self.up_conv_1, relu=True)
        x = ops.conv2d_nhwc(x, self.up_conv_2, relu=True)
        x = ops.conv2d_nhwc(x, self.up_conv_3, relu=True)
        return ops.conv2d_nhwc(x, self.up_conv_4, act=ops.ACT_SIGMOID)

    def forward(self, ssr, spatial_map):
        out = self.forward_nhwc(ops.to_nhwc(ssr, self.compute_dtype), ops.to_nhwc(spatial_map, self.compute_dtype))
        return ops.to_nchw(out)


class RoadMapBoxesMergingCNN(_MergingBase):
    """ssr [B,32,128,918], spatial map [B,32,256,256], road map [B,1,800,800] -> probabilities
    [B,1,800,800] (components.py:122-170): 96 channels at 256x256, four dilated transposed convs
    up to 400x400, a k2 s2 transposed conv to 800x800, sigmoid."""

    def __init__(self, compute_dtype="fp32"):
        super().__init__()
        self.ss_conv = nn.Conv2d(32, 32, kernel_size=(1, 24), stride=(1, 7))
        self.ss_deconv = nn.ConvTranspose2d(32, 32, kernel_size=2, stride=2)
        self.rm_conv_1 = nn.Conv2d(1, 32, kernel_size=7, stride=3, dilation=3, padding=1)
        self.rm_conv_2 = nn.Conv2d(32, 32, kernel_size=3, stride=1, dilation=3)
        self.up_conv_1 = nn.ConvTranspose2d(96, 64, kernel_size=7, stride=1, dilation=7)
        self.up_conv_2 = nn.ConvTranspose2d(64, 32, kernel_size=7, stride=1, dilation=7)
        self.up_conv_3 = nn.ConvTranspose2d(32, 16, kernel_size=7, stride=1, dilation=7)
        self.up_conv_4 = nn.ConvTranspose2d(16, 8, kernel_size=7, stride=1, dilation=3)
        self.up_conv_5 = nn.ConvTranspose2d(8, 1, kernel_size=2, stride=2)
        self.compute_dtype = resolve_dtype(compute_dtype)

    def forward_nhwc(self, ssr, spatial_map, rm):
        """All three inputs NHWC in the compute dtype; returns NHWC probabilities [B,800,800,1]."""
        ssr = self._ssr_branch(ssr)
        rm = ops.conv2d_nhwc(rm, self.rm_conv_1, relu=True)
        rm = ops.conv2d_nhwc(rm, self.rm_conv_2, relu=True)
        x = self._concat([ssr, spatial_map, rm])
        x = ops.conv2d_nhwc(x, self.up_conv_1, relu=True)
        x = ops.conv2d_nhwc(x, self.up_conv_2, relu=True)
        x = ops.conv2d_nhwc(x, self.up_conv_3, relu=True)
        x = ops.conv2d_nhwc(x, self.up_conv_4, relu=True)
        return ops.conv2d_nhwc(x, self.up_conv_5, act=ops.ACT_SIGMOID)

    def forward(self, ssr, spatial_map, rm):
        dt = self.compute_dtype
        out = self.forward_nhwc(ops.to_nhwc(ssr, dt), ops.to_nhwc(spatial_map, dt), ops.to_nhwc(rm, dt))
        return ops.to_nchw(out)
