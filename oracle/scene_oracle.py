"""CPU oracle for the six-camera scene pipeline -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
import this module.  The product package (driving-dirty_b200/) never imports it and fails
loudly when its CUDA library is missing.

What it is: a restatement of the reference's algorithm for the hot path as plain functions
over a flat ``params`` dict (keys = the reference's state_dict keys).  The reference is a
Python/PyTorch program whose arithmetic is torch's CPU ops, so the floating-point pieces are
restated with the same torch CPU primitives (conv2d, linear, batch_norm, ...) composed by
hand; the byte/index pieces (stitch, flat max-pool, binarise, threat-score counts) are
restated in numpy integer/index arithmetic and, again, in C (oracle/scene_oracle.c).

Parity pinning: the reference ships no tests or golden vectors (SURVEY.md section 4).  The
oracle is pinned against outputs of the UNMODIFIED reference modules imported from
/root/reference in the build container (oracle/make_golden.py, dependency shims under
oracle/shims/); those outputs are committed under tests/golden/ and tests/test_oracle.py
checks the oracle against them bit-for-bit.

Every function cites the reference lines it follows (paths relative to /root/reference/src).
"""
from __future__ import annotations

import numpy as np
import torch
import torch.nn.functional as F

VIEW_ORDER = (0, 1, 2, 5, 4, 3)  # roadmap_bce_v2.py:58, autoencoder.py:55, spatial_w_rm.py:58
# intra-op threads of torch's CPU ops when the golden files were written: conv / linear split their reductions by
# thread count, so a bit-for-bit comparison with those files has to run with the same count on any machine
GOLDEN_THREADS = 8
BINARISE_THRESHOLD_BITS = 0x33C00000  # sigmoid(x).round()==1  <=>  x > 1.5*2**-24 (see binarise)


# ----------------------------------------------------------------------------------------
# A1 / A2: stitch
# ----------------------------------------------------------------------------------------
def stitch(views: torch.Tensor) -> torch.Tensor:
    """mosaic[b,c,h,j*W+w] = views[b,VIEW_ORDER[j],c,h,w].

    roadmap_bce_v2.py:53-64 (wide_stitch_six_images): stack, x[:, [0,1,2,5,4,3]],
    permute(0,2,3,1,4).reshape(b,c,h,-1).  Restated as an explicit index gather in numpy.
    """
    v = views.detach().cpu().numpy()
    b, n, c, h, w = v.shape
    assert n == 6
    out = np.empty((b, c, h, 6 * w), dtype=v.dtype)
    for j, src in enumerate(VIEW_ORDER):
        out[:, :, :, j * w:(j + 1) * w] = v[:, src]
    return torch.from_numpy(out).to(views.device)      # (device kept: tests also run this restatement on cuda tensors)


def six_to_one(views: torch.Tensor, target_slot: int):
    """autoencoder.py:53-73 (six_to_one_task) with the host RNG draw made explicit.

    The reference draws ``target_slot = np.random.randint(0, 5)`` (slot 5 never chosen),
    clones mosaic[..., 306t:306t+306] as y and zeroes that block of x.  The slot width is the
    view width (306 in the reference; parametrised here for reduced-geometry tests).
    """
    x = stitch(views).clone()
    w = views.shape[-1]
    s, e = target_slot * w, (target_slot + 1) * w
    y = x[:, :, :, s:e].clone()
    x[:, :, :, s:e] = 0.0
    return x, y


# ----------------------------------------------------------------------------------------
# A3 / A4 / A5: encoder convs and the flat max-pool
# ----------------------------------------------------------------------------------------
class _StoreAs(torch.autograd.Function):
    """Emulates a tensor being STORED in a narrower dtype on both passes: forward rounds the
    activation to ``dtype``, backward rounds the gradient arriving at it.  Used only for the
    like-for-like check of the bf16 activation-storage path (the fp32 oracle never calls it)."""

    @staticmethod
    def forward(ctx, x, dtype):
        ctx.dtype = dtype
        return x.to(dtype).float()

    @staticmethod
    def backward(ctx, g):
        return g.to(ctx.dtype).float(), None


def _store(x, dtype):
    return x if dtype is None or dtype == torch.float32 else _StoreAs.apply(x, dtype)


def _weight_as(w, dtype):
    """Operand rounding of a weight (tensor-core path reads conv weights as bf16); gradients pass
    straight through to the fp32 master weight."""
    if dtype is None or dtype == torch.float32:
        return w
    return w + (w.detach().to(dtype).float() - w.detach())


def encoder_convs(p: dict, x: torch.Tensor, prefix: str = "ae.encoder.", act_dtype=None, weight_dtype=None):
    """components.py:41-43: relu(c1), relu(c2), relu(c3 stride 2), all 3x3 pad 1.
    ``act_dtype`` / ``weight_dtype`` (default None = the reference's fp32) emulate the storage
    rounding points of the bf16 path: a1, a2, a3 and their gradients; the conv weights and the
    input image as tensor-core operands."""
    if weight_dtype is not None and weight_dtype != torch.float32:
        x = x.to(weight_dtype).float()     # the tensor-core c1 reads the image as bf16 operands too
    a1 = _store(F.relu(F.conv2d(x, _weight_as(p[prefix + "c1.weight"], weight_dtype), p[prefix + "c1.bias"],
                                padding=1)), act_dtype)
    a2 = _store(F.relu(F.conv2d(a1, _weight_as(p[prefix + "c2.weight"], weight_dtype), p[prefix + "c2.bias"],
                                padding=1)), act_dtype)
    a3 = _store(F.relu(F.conv2d(a2, _weight_as(p[prefix + "c3.weight"], weight_dtype), p[prefix + "c3.bias"],
                                stride=2, padding=1)), act_dtype)
    return a1, a2, a3


def pool4_flat(a3: torch.Tensor) -> torch.Tensor:
    """components.py:46-47: view(B,-1) then max_pool1d(kernel_size=4) over the NCHW-flat index.

    numpy restatement: reshape to [B, n/4, 4] and take the max; the trailing n%4 elements are
    dropped exactly as max_pool1d (floor mode) drops them.
    """
    v = a3.detach().cpu().numpy().reshape(a3.shape[0], -1)
    n = v.shape[1] // 4
    return torch.from_numpy(v[:, :n * 4].reshape(v.shape[0], n, 4).max(axis=2).copy())


def pool4_flat_argmax(a3: torch.Tensor) -> np.ndarray:
    """First-max index inside each window (torch's max_pool backward routes to the first max)."""
    v = a3.detach().cpu().numpy().reshape(a3.shape[0], -1)
    n = v.shape[1] // 4
    return v[:, :n * 4].reshape(v.shape[0], n, 4).argmax(axis=2).astype(np.uint8)


# ----------------------------------------------------------------------------------------
# A6 / A7: DenseBlock with the always-on dropout
# ----------------------------------------------------------------------------------------
def dense_block(p: dict, prefix: str, x: torch.Tensor, training: bool, drop_p: float = 0.2,
                momentum: float = 0.1, eps: float = 1e-5) -> torch.Tensor:
    """components.py:104-109: Linear -> BatchNorm1d -> ReLU -> F.dropout(x, p) (training=True
    default: NEVER disabled, SURVEY D5).  BatchNorm uses batch statistics and updates the
    running buffers in ``p`` in place when ``training`` (i.e. after unfreeze()).
    """
    y = F.linear(x, p[prefix + "fc1.weight"], p[prefix + "fc1.bias"])
    y = F.batch_norm(y, p[prefix + "fc_bn.running_mean"], p[prefix + "fc_bn.running_var"],
                     p[prefix + "fc_bn.weight"], p[prefix + "fc_bn.bias"],
                     training=training, momentum=momentum, eps=eps)
    if training and (prefix + "fc_bn.num_batches_tracked") in p:
        p[prefix + "fc_bn.num_batches_tracked"] += 1
    y = F.relu(y)
    return F.dropout(y, drop_p)  # consumes the global torch RNG exactly like the reference


def encoder_forward(p: dict, x: torch.Tensor, training: bool, prefix: str = "ae.encoder.",
                    c3_only: bool = False, act_dtype=None, weight_dtype=None) -> torch.Tensor:
    """components.py:40-52 (Encoder.forward)."""
    _, _, a3 = encoder_convs(p, x, prefix, act_dtype, weight_dtype)
    if c3_only:  # components.py:44-45
        return a3
    # components.py:46-47.  F.max_pool1d (not amax) so that autograd routes the gradient to the
    # FIRST maximum of each window like the reference; pool4_flat() above is the index-level
    # restatement and tests check the two agree.
    pooled = F.max_pool1d(a3.reshape(a3.shape[0], -1).unsqueeze(1), kernel_size=4).squeeze(1)
    pooled = _store(pooled, act_dtype)   # no-op on the values; rounds d(pooled) on the way back
    h = dense_block(p, prefix + "fc1.", pooled, training)
    h = dense_block(p, prefix + "fc2.", h, training)
    return F.linear(h, p[prefix + "fc_z_out.weight"], p[prefix + "fc_z_out.bias"])


# ----------------------------------------------------------------------------------------
# A8-A11: roadmap head, loss, binarise, threat score
# ----------------------------------------------------------------------------------------
def roadmap_forward(p: dict, views, training: bool, map_hw: int = 800, act_dtype=None, weight_dtype=None):
    """roadmap_bce_v2.py:66-81: stitch -> encoder -> Linear(latent, 800*800) -> reshape;
    returns (logits, sigmoid(logits)).  ``views`` may be a [B,6,3,H,W] tensor or the
    collate_fn tuple of [6,3,H,W] tensors (roadmap_bce_v2.py:55 stacks it)."""
    if not torch.is_tensor(views):
        views = torch.stack(tuple(views), dim=0)
    x = stitch(views)
    z = encoder_forward(p, x, training, act_dtype=act_dtype, weight_dtype=weight_dtype)
    y = F.linear(z, p["fc1.weight"], p["fc1.bias"]).reshape(z.shape[0], map_hw, map_hw)
    return y, torch.sigmoid(y)


def bce_with_logits_mean(logits: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """roadmap_bce_v2.py:103-106: F.binary_cross_entropy_with_logits on [B, H*W] views, mean
    over B*H*W.  Elementwise form: (1-t)*x + max(-x,0) + log1p(exp(-|x|)); float64 sum."""
    x = logits.detach().double().reshape(-1)
    t = target.detach().double().reshape(-1)
    per = (1.0 - t) * x + torch.clamp(-x, min=0.0) + torch.log1p(torch.exp(-x.abs()))
    return (per.sum() / x.numel()).float()


def bce_with_logits_grad(logits: torch.Tensor, target: torch.Tensor) -> torch.Tensor:
    """d(mean BCE)/d logits = (sigmoid(x) - t) / numel  (SURVEY A9)."""
    return (torch.sigmoid(logits) - target) / logits.numel()


def binarise(probs_or_logits: torch.Tensor, from_logits: bool = False) -> torch.Tensor:
    """roadmap_bce_v2.py:140 / :115: ``probs.round()`` (round-half-even of the fp32 sigmoid).

    From logits this equals ``x > 1.5 * 2**-24`` bit-for-bit: an exhaustive sweep of every
    fp32 in [2**-27, 2**-20) through torch's CPU sigmoid (tests/test_oracle.py repeats it)
    shows sigmoid(x).round() flips 0 -> 1 exactly between 0x33C00000 and 0x33C00001 and is
    monotone either side; sigmoid(0)=0.5 rounds (half to even) to 0.
    """
    if from_logits:
        thr = np.uint32(BINARISE_THRESHOLD_BITS).view(np.float32)
        return (probs_or_logits > float(thr)).to(torch.float32)
    return probs_or_logits.round()


def threat_score(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """helper.py:74-77: tp = (a*b).sum(); tp*1.0 / (a.sum() + b.sum() - tp), fp32, pooled
    over the whole batch.  Restated with torch fp32 sums (same reduction as the reference)."""
    tp = (a * b).sum()
    return tp * 1.0 / (a.sum() + b.sum() - tp)


def threat_score_counts(target01: torch.Tensor, pred01: torch.Tensor):
    """Integer restatement for 0/1 maps: returns (tp, n_target, n_pred) as python ints.
    TS = tp / (n_target + n_pred - tp).  Exact for any batch size (the reference's fp32 sums
    are exact only while every partial < 2**24, i.e. <= 26 scenes -- SURVEY H5)."""
    t = target01.detach().cpu().numpy().astype(np.int64).reshape(-1)
    r = pred01.detach().cpu().numpy().astype(np.int64).reshape(-1)
    return int((t * r).sum()), int(t.sum()), int(r.sum())


def run_step(p: dict, views, road_image, training: bool, seed: int | None = None, act_dtype=None,
             weight_dtype=None):
    """roadmap_bce_v2.py:83-108 (_run_step) + :135-143 (validation_step metrics).

    Returns dict(loss, logits, probs, ts, ts_rounded).  ``seed`` re-seeds the torch RNG just
    before the forward so that the always-on dropout mask is reproducible (SURVEY D5).
    """
    if not torch.is_tensor(road_image):
        road_image = torch.stack(tuple(road_image), dim=0)
    target = road_image.float()  # :87
    if seed is not None:
        torch.manual_seed(seed)
    logits, probs = roadmap_forward(p, views, training, map_hw=target.shape[-1], act_dtype=act_dtype,
                                    weight_dtype=weight_dtype)
    b = target.shape[0]
    loss = F.binary_cross_entropy_with_logits(logits.view(b, -1), target.view(b, -1))  # :106
    return dict(loss=loss, logits=logits, probs=probs, target=target,
                ts=threat_score(target, probs), ts_rounded=threat_score(target, probs.round()))


def train_step_grads(p: dict, views, road_image, seed: int, names=None, act_dtype=None, weight_dtype=None):
    """fwd + BCE + backward through the restated path with torch autograd on CPU (what
    loss.backward() does in the reference after unfreeze(), roadmap_bce_v2.py:125-133).
    Returns (out dict, {name: grad})."""
    names = names or [k for k, v in p.items() if v.is_floating_point()
                      and not k.endswith(("running_mean", "running_var"))]
    q = dict(p)
    for k in names:
        q[k] = p[k].detach().clone().requires_grad_(True)
    for k in p:
        if k.endswith(("running_mean", "running_var", "num_batches_tracked")):
            q[k] = p[k].clone()
    out = run_step(q, views, road_image, training=True, seed=seed, act_dtype=act_dtype, weight_dtype=weight_dtype)
    out["loss"].backward()
    return out, {k: q[k].grad for k in names}


# ----------------------------------------------------------------------------------------
# A13 / A14: AE decoder and MSE (config 3)
# ----------------------------------------------------------------------------------------
def decoder_forward(p: dict, z: torch.Tensor, training: bool, hw, prefix: str = "decoder."):
    """components.py:85-93 (Decoder.forward); hw = (deconv_dim_h, deconv_dim_w)."""
    x = dense_block(p, prefix + "fc1.", z, training)
    x = dense_block(p, prefix + "fc2.", x, training)
    x = x.view(x.size(0), 64, hw[0], hw[1])
    x = F.relu(F.conv_transpose2d(x, p[prefix + "dc1.weight"], p[prefix + "dc1.bias"], padding=1))
    x = F.relu(F.conv_transpose2d(x, p[prefix + "dc2.weight"], p[prefix + "dc2.bias"], padding=1))
    x = F.relu(F.conv_transpose2d(x, p[prefix + "dc3.weight"], p[prefix + "dc3.bias"], stride=2))
    return F.conv_transpose2d(x, p[prefix + "dc4.weight"], p[prefix + "dc4.bias"])


def ae_run_step(p: dict, views: torch.Tensor, target_slot: int, training: bool, hw,
                seed: int | None = None):
    """autoencoder.py:78-93: six_to_one_task -> encoder -> decoder -> F.mse_loss(y, y_hat)."""
    x, y = six_to_one(views, target_slot)
    if seed is not None:
        torch.manual_seed(seed)
    z = encoder_forward(p, x, training, prefix="encoder.")
    y_hat = decoder_forward(p, z, training, hw)
    return dict(loss=F.mse_loss(y, y_hat), x=x, y=y, z=z, y_hat=y_hat)


# ----------------------------------------------------------------------------------------
# A15-A17: bounding-box model with roadmap input (config 4)
# ----------------------------------------------------------------------------------------
def view_transform(views: torch.Tensor, view: int, mode: int) -> torch.Tensor:
    """One camera of the batch as an image [B,3,H',W'], restated as explicit index maps (numpy):
    mode 0: as is; 1: torch.rot90(x, 1, [2,3]) -> out[i,j] = x[j, W-1-i]; 2: torch.rot90(x, 1, [3,2])
    -> out[i,j] = x[H-1-j, i]; 3: torch.flip(x, [2,3]) -> out[i,j] = x[H-1-i, W-1-j]
    (spatial_bb/components.py:34-62)."""
    v = views[:, view].detach().cpu().numpy()
    if mode == 0:
        out = v
    elif mode == 1:
        out = np.transpose(v, (0, 1, 3, 2))[:, :, ::-1, :]
    elif mode == 2:
        out = np.transpose(v, (0, 1, 3, 2))[:, :, :, ::-1]
    else:
        out = v[:, :, ::-1, ::-1]
    return torch.from_numpy(np.ascontiguousarray(out))


# (name, camera index, transform mode) in the order the strips are computed; canvas cell (row, col)
BB_STRIPS = (("bl_conv", 3, 0, (0, 0)), ("fl_conv", 0, 0, (0, 1)), ("b_conv", 4, 1, (1, 0)), ("f_conv", 1, 2, (1, 1)),
             ("br_conv", 5, 3, (2, 0)), ("fr_conv", 2, 3, (2, 1)))


def spatial_mapping_forward(p: dict, views: torch.Tensor, prefix: str = "space_map_cnn.") -> torch.Tensor:
    """spatial_bb/components.py:28-77 (SpatialMappingCNN.forward): six strip convs (+ReLU) on the
    plain / rotated / flipped cameras, tiled 3 x 2 into a square canvas, 3x3 valid conv + ReLU."""
    cells = {}
    for name, cam, mode, cell in BB_STRIPS:
        img = view_transform(views, cam, mode)
        pad = 1 if name in ("f_conv", "b_conv") else 0          # :18,22 (padding=(1))
        cells[cell] = F.relu(F.conv2d(img, p[prefix + name + ".weight"], p[prefix + name + ".bias"], stride=(3, 2),
                                      padding=pad))
    rows = [torch.cat([cells[(r, 0)], cells[(r, 1)]], dim=3) for r in range(3)]
    canvas = torch.cat(rows, dim=2)
    return F.relu(F.conv2d(canvas, p[prefix + "out_conv.weight"], p[prefix + "out_conv.bias"]))


def merging_forward(p: dict, ssr, spatial_map, rm, prefix: str = "box_merge.") -> torch.Tensor:
    """spatial_bb/components.py:141-170 (RoadMapBoxesMergingCNN.forward) -> probabilities [B,1,800,800]."""
    w = lambda n: p[prefix + n + ".weight"]  # noqa: E731
    b = lambda n: p[prefix + n + ".bias"]    # noqa: E731
    ssr = F.relu(F.conv2d(ssr, w("ss_conv"), b("ss_conv"), stride=(1, 7)))
    ssr = F.relu(F.conv_transpose2d(ssr, w("ss_deconv"), b("ss_deconv"), stride=2))
    rm = F.relu(F.conv2d(rm, w("rm_conv_1"), b("rm_conv_1"), stride=3, dilation=3, padding=1))
    rm = F.relu(F.conv2d(rm, w("rm_conv_2"), b("rm_conv_2"), dilation=3))
    x = torch.cat([ssr, spatial_map, rm], dim=1)
    x = F.relu(F.conv_transpose2d(x, w("up_conv_1"), b("up_conv_1"), dilation=7))
    x = F.relu(F.conv_transpose2d(x, w("up_conv_2"), b("up_conv_2"), dilation=7))
    x = F.relu(F.conv_transpose2d(x, w("up_conv_3"), b("up_conv_3"), dilation=7))
    x = F.relu(F.conv_transpose2d(x, w("up_conv_4"), b("up_conv_4"), dilation=3))
    return torch.sigmoid(F.conv_transpose2d(x, w("up_conv_5"), b("up_conv_5"), stride=2))


def bb_forward(p: dict, views: torch.Tensor, rm: torch.Tensor) -> torch.Tensor:
    """spatial_w_rm.py:67-83 (BBSpatialRoadMap.forward): views [B,6,3,H,W], rm [B,1,800,800] -> [B,800,800]."""
    space_rep = spatial_mapping_forward(p, views)
    _, _, ssr = encoder_convs(p, stitch(views))            # encoder with c3_only (spatial_w_rm.py:47)
    return merging_forward(p, ssr, space_rep, rm).squeeze(1)


def bb_run_step(p: dict, views, road_image, target_bb_img, mse_loss: bool = False):
    """spatial_w_rm.py:97-133 with the rasterised box target passed in (bb_to_img.py is host-side
    label preparation): prob-space BCE (torch clamps each log at -100) or MSE."""
    rm = road_image.float().unsqueeze(1)
    pred = bb_forward(p, views, rm)
    b = pred.shape[0]
    pv, tv = pred.reshape(b, -1), target_bb_img.float().reshape(b, -1)
    loss = F.mse_loss(pv, tv) if mse_loss else F.binary_cross_entropy(pv, tv)
    return dict(loss=loss, pred=pred)


def boxes_to_binary_map(boxes: torch.Tensor) -> np.ndarray:
    """utils/bb_to_img.py:5-21 restated: boxes [N,2,4] (metres; rows x/y; cols fl, fr, bl, br) ->
    800x800 map; polygon corner order fl, fr, br, bl; pixel = metre*10 + 400; vertical flip."""
    from PIL import Image, ImageDraw
    x = boxes.cpu().numpy()
    img = Image.fromarray(np.zeros((800, 800)))
    draw = ImageDraw.Draw(img)
    for i in range(x.shape[0]):
        box = np.stack([x[i][:, 0], x[i][:, 1], x[i][:, 3], x[i][:, 2]]) * 10 + 400
        draw.polygon(list(box.flatten()), fill=1)
    return np.flip(np.asarray(img), 0)


def synthetic_boxes(batch: int, seed: int = 20200507):
    """5-20 axis-aligned 4.6 m x 2 m boxes per scene, centres U(-30, 30) m (SURVEY 8(d))."""
    g = torch.Generator().manual_seed(seed)
    out = []
    for _ in range(batch):
        n = int(torch.randint(5, 21, (1,), generator=g))
        c = torch.rand(n, 2, generator=g) * 60 - 30
        dx, dy = 2.3, 1.0
        xs = torch.stack([c[:, 0] + dx, c[:, 0] + dx, c[:, 0] - dx, c[:, 0] - dx], dim=1)
        ys = torch.stack([c[:, 1] + dy, c[:, 1] - dy, c[:, 1] + dy, c[:, 1] - dy], dim=1)
        out.append(torch.stack([xs, ys], dim=1))
    return out


def init_bb_params(hidden: int, latent: int, view_h: int = 256, view_w: int = 306, seed: int = 20200505) -> dict:
    """Random-init BBSpatialRoadMap parameters keyed like its state_dict: the AE encoder (through
    init_roadmap_params' generator, prefix ae.encoder.), then SpatialMappingCNN and
    RoadMapBoxesMergingCNN layers built by torch's own constructors (default init) in the
    reference's order (spatial_bb/components.py:16-26,127-139) under torch.manual_seed(seed)."""
    from torch import nn
    p = {k: v for k, v in init_roadmap_params(hidden, latent, view_h, view_w, map_hw=8, seed=seed).items()
         if k.startswith("ae.encoder.")}
    state = torch.random.get_rng_state()
    torch.manual_seed(seed)
    space = [("f_conv", nn.Conv2d(3, 32, (52, 1), (3, 2), 1)), ("fl_conv", nn.Conv2d(3, 32, (1, 50), (3, 2))),
             ("fr_conv", nn.Conv2d(3, 32, (1, 50), (3, 2))), ("b_conv", nn.Conv2d(3, 32, (52, 1), (3, 2), 1)),
             ("bl_conv", nn.Conv2d(3, 32, (1, 50), (3, 2))), ("br_conv", nn.Conv2d(3, 32, (1, 50), (3, 2))),
             ("out_conv", nn.Conv2d(32, 32, 3))]
    merge = [("ss_conv", nn.Conv2d(32, 32, (1, 24), (1, 7))), ("ss_deconv", nn.ConvTranspose2d(32, 32, 2, 2)),
             ("rm_conv_1", nn.Conv2d(1, 32, 7, 3, 1, 3)), ("rm_conv_2", nn.Conv2d(32, 32, 3, 1, 0, 3)),
             ("up_conv_1", nn.ConvTranspose2d(96, 64, 7, 1, dilation=7)), ("up_conv_2", nn.ConvTranspose2d(64, 32, 7, 1, dilation=7)),
             ("up_conv_3", nn.ConvTranspose2d(32, 16, 7, 1, dilation=7)), ("up_conv_4", nn.ConvTranspose2d(16, 8, 7, 1, dilation=3)),
             ("up_conv_5", nn.ConvTranspose2d(8, 1, 2, 2))]
    torch.random.set_rng_state(state)
    for prefix, layers in (("space_map_cnn.", space), ("box_merge.", merge)):
        for name, m in layers:
            p[prefix + name + ".weight"] = m.weight.detach().clone()
            p[prefix + name + ".bias"] = m.bias.detach().clone()
    return p


def strided_sample(t: torch.Tensor, n: int = 4096) -> torch.Tensor:
    """n evenly spaced elements of the flattened tensor (integer index arithmetic); how the
    golden files keep a checkable slice of tensors too large to commit."""
    f = t.detach().reshape(-1)
    idx = (torch.arange(n, dtype=torch.int64) * (f.numel() - 1)) // max(n - 1, 1)
    return f[idx.to(f.device)].clone()


# ----------------------------------------------------------------------------------------
# synthetic inputs / weights shared by tests, smoke() and bench.py (SURVEY 8(d))
# ----------------------------------------------------------------------------------------
def min_abs_preactivation(p: dict, views: torch.Tensor, prefix: str = "ae.encoder.") -> float:
    """Smallest |pre-activation| over the three encoder convs.  An fp32 implementation that sums in
    a different order can flip relu'(x) for |x| ~ 1e-7, which moves every upstream gradient by a
    whole pixel's contribution; golden train cases are chosen so that this value is > 2e-6 and the
    1e-5 gradient contract is testable (make_golden.py searches the input seed)."""
    x = stitch(views)
    m = float("inf")
    strides = {"c1": 1, "c2": 1, "c3": 2}
    for name in ("c1", "c2", "c3"):
        pre = F.conv2d(x, p[prefix + name + ".weight"], p[prefix + name + ".bias"], stride=strides[name], padding=1)
        m = min(m, float(pre.abs().min()))
        x = F.relu(pre)
    return m


def synthetic_scene_batch(batch: int, view_h: int = 256, view_w: int = 306, map_hw: int = 800,
                          seed: int = 20200505):
    g = torch.Generator().manual_seed(seed)
    views = torch.rand(batch, 6, 3, view_h, view_w, generator=g)
    road = torch.rand(batch, map_hw, map_hw, generator=g) > 0.5
    return views, road


def init_roadmap_params(hidden: int, latent: int, view_h: int, view_w: int, map_hw: int = 800,
                        seed: int = 20200505) -> dict:
    """Random-init parameters with the reference's shapes and torch default initialisers
    (nn.Conv2d / nn.Linear kaiming-uniform(a=sqrt(5)), BatchNorm1d ones/zeros), keyed like
    RoadMapBCE.state_dict() after ``self.ae.decoder = None`` (roadmap_bce_v2.py:43-50)."""
    g = torch.Generator().manual_seed(seed)

    def uni(shape, fan_in):
        bound = 1.0 / fan_in ** 0.5
        return (torch.rand(shape, generator=g) * 2 - 1) * bound

    mh, mw = view_h, 6 * view_w
    h3, w3 = (mh - 1) // 2 + 1, (mw - 1) // 2 + 1
    pooled = (32 * h3 * w3) // 4
    p = {}
    e = "ae.encoder."
    p[e + "c1.weight"], p[e + "c1.bias"] = uni((32, 3, 3, 3), 27), uni((32,), 27)
    p[e + "c2.weight"], p[e + "c2.bias"] = uni((32, 32, 3, 3), 288), uni((32,), 288)
    p[e + "c3.weight"], p[e + "c3.bias"] = uni((32, 32, 3, 3), 288), uni((32,), 288)
    for name, (i, o) in (("fc1.", (pooled, hidden)), ("fc2.", (hidden, hidden))):
        p[e + name + "fc1.weight"], p[e + name + "fc1.bias"] = uni((o, i), i), uni((o,), i)
        p[e + name + "fc_bn.weight"], p[e + name + "fc_bn.bias"] = torch.ones(o), torch.zeros(o)
        p[e + name + "fc_bn.running_mean"] = torch.zeros(o)
        p[e + name + "fc_bn.running_var"] = torch.ones(o)
        p[e + name + "fc_bn.num_batches_tracked"] = torch.tensor(0)
    p[e + "fc_z_out.weight"], p[e + "fc_z_out.bias"] = uni((latent, hidden), hidden), uni((latent,), hidden)
    p["fc1.weight"], p["fc1.bias"] = uni((map_hw * map_hw, latent), latent), uni((map_hw * map_hw,), latent)
    return p


# ----------------------------------------------------------------------------------------
# 8(f)3: compute_ats_bounding_boxes (helper.py:33-72) with a stand-in for shapely's polygons
# ----------------------------------------------------------------------------------------
def _hull(points):
    """Convex hull (counter-clockwise, no collinear points) of a few 2-D points -- what
    ``Polygon(torch.t(box)).convex_hull`` (helper.py:80-81) yields for a box's four corners.  shapely (GEOS, unpinned in
    requirements.txt) is not installable here: this is a pure-Python float64 stand-in, pinned by analytic cases in
    tests/test_oracle.py rather than by shapely itself."""
    pts = sorted(set((float(x), float(y)) for x, y in points))
    if len(pts) < 3:
        return pts

    def cross(o, a, b):
        return (a[0] - o[0]) * (b[1] - o[1]) - (a[1] - o[1]) * (b[0] - o[0])

    lower, upper = [], []
    for p in pts:
        while len(lower) >= 2 and cross(lower[-2], lower[-1], p) <= 0:
            lower.pop()
        lower.append(p)
    for p in reversed(pts):
        while len(upper) >= 2 and cross(upper[-2], upper[-1], p) <= 0:
            upper.pop()
        upper.append(p)
    return lower[:-1] + upper[:-1]


def _poly_area(poly):
    return 0.5 * abs(sum(poly[i][0] * poly[(i + 1) % len(poly)][1] - poly[(i + 1) % len(poly)][0] * poly[i][1]
                         for i in range(len(poly)))) if len(poly) >= 3 else 0.0


def _clip(subject, clip):
    """Sutherland-Hodgman: the part of convex ``subject`` inside convex counter-clockwise ``clip``."""
    out = list(subject)
    for i in range(len(clip)):
        a, b = clip[i], clip[(i + 1) % len(clip)]
        side = lambda p: (b[0] - a[0]) * (p[1] - a[1]) - (b[1] - a[1]) * (p[0] - a[0])  # noqa: E731
        inp, out = out, []
        for k in range(len(inp)):
            p, q = inp[k], inp[(k + 1) % len(inp)]
            sp, sq = side(p), side(q)
            if sp >= 0:
                out.append(p)
            if (sp > 0 > sq) or (sp < 0 < sq):
                t = sp / (sp - sq)
                out.append((p[0] + t * (q[0] - p[0]), p[1] + t * (q[1] - p[1])))
        if not out:
            break
    return out


def compute_iou(box1: torch.Tensor, box2: torch.Tensor) -> float:
    """helper.py:79-83: intersection area / union area of the two corner sets' convex hulls."""
    a, b = _hull(torch.t(box1).tolist()), _hull(torch.t(box2).tolist())
    inter = _poly_area(_clip(a, b)) if len(a) >= 3 and len(b) >= 3 else 0.0
    return inter / (_poly_area(a) + _poly_area(b) - inter)


def compute_ats_bounding_boxes(boxes1: torch.Tensor, boxes2: torch.Tensor):
    """helper.py:33-72 line by line (torch ops kept: they fix the float32 rounding of the score); returns
    (average_threat_score 0-dim float32 tensor, iou_matrix)."""
    num_boxes1, num_boxes2 = boxes1.size(0), boxes2.size(0)
    b1_max_x, b1_min_x = boxes1[:, 0].max(dim=1)[0], boxes1[:, 0].min(dim=1)[0]
    b1_max_y, b1_min_y = boxes1[:, 1].max(dim=1)[0], boxes1[:, 1].min(dim=1)[0]
    b2_max_x, b2_min_x = boxes2[:, 0].max(dim=1)[0], boxes2[:, 0].min(dim=1)[0]
    b2_max_y, b2_min_y = boxes2[:, 1].max(dim=1)[0], boxes2[:, 1].min(dim=1)[0]
    cond = ((b1_max_x.unsqueeze(1) > b2_min_x.unsqueeze(0)) * (b1_min_x.unsqueeze(1) < b2_max_x.unsqueeze(0)) *
            (b1_max_y.unsqueeze(1) > b2_min_y.unsqueeze(0)) * (b1_min_y.unsqueeze(1) < b2_max_y.unsqueeze(0)))
    iou_matrix = torch.zeros(num_boxes1, num_boxes2)
    for i in range(num_boxes1):
        for j in range(num_boxes2):
            if cond[i][j]:
                iou_matrix[i][j] = compute_iou(boxes1[i], boxes2[j])
    iou_max = iou_matrix.max(dim=0)[0]
    total_threat_score, total_weight = 0, 0
    for threshold in [0.5, 0.6, 0.7, 0.8, 0.9]:
        tp = (iou_max > threshold).sum()
        threat_score = tp * 1.0 / (num_boxes1 + num_boxes2 - tp)
        total_threat_score += 1.0 / threshold * threat_score
        total_weight += 1.0 / threshold
    return total_threat_score / total_weight, iou_matrix
