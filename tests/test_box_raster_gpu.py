"""ops.boxes_to_map (csrc/boxes.cu box_raster_kernel) against the reference's host rasteriser,
utils/bb_to_img.boxes_to_binary_map (Pillow's polygon fill), bit for bit: the golden target of
bb_full_b1.pt, then families of boxes chosen to reach every rule of the fill (box_raster.cuh).

Each family packs many small boxes into one scene, so tens of thousands of polygons are checked
without tens of thousands of Pillow images; the fill of a scene is the union of its boxes' fills
either way."""
import hashlib
import math

import numpy as np
import pytest
import torch

from oracle import scene_oracle as so

SIZE, SCALE, OFFSET = 800, 10.0, 400.0


def to_metres(px):
    """pixel coordinates (float64 array) -> metres, the inverse of pixel = metre * 10 + 400"""
    return (np.asarray(px, dtype=np.float64) - OFFSET) / SCALE


def quads_to_boxes(q):
    """q [N,4,2] pixel corners in drawing order (fl, fr, br, bl) -> boxes [N,2,4] in metres, columns fl, fr, bl, br"""
    q = np.asarray(q, dtype=np.float64)
    cols = q[:, [0, 1, 3, 2], :]                         # fl, fr, bl, br
    return torch.from_numpy(to_metres(cols).transpose(0, 2, 1).copy())


def rects(c, w, h, theta):
    """rotated rectangles (pixel space): centres c [N,2], widths, heights, angles -> corners [N,4,2] in loop order"""
    dx = np.stack([-w, w, w, -w], 1) / 2
    dy = np.stack([h, h, -h, -h], 1) / 2
    ct, st = np.cos(theta)[:, None], np.sin(theta)[:, None]
    return np.stack([c[:, None, 0] + ct * dx - st * dy, c[:, None, 1] + st * dx + ct * dy], -1)


def grid_centres(n, cell, rng, jitter=0.0):
    k = SIZE // cell
    idx = rng.permutation(k * k)[:n]
    c = np.stack([idx % k, idx // k], 1) * cell + cell / 2.0
    return c + (rng.random((n, 2)) - 0.5) * jitter


def family_scenes():
    """name -> list of float64 box tensors [N,2,4] (metres)"""
    rng = np.random.default_rng(20261021)
    fam = {}
    n = 1000
    c = grid_centres(n, 25, rng, 4.0)
    fam["axis_aligned"] = [quads_to_boxes(rects(c, rng.random(n) * 20 + 0.3, rng.random(n) * 20 + 0.3, np.zeros(n)))]
    fam["rotated"] = [quads_to_boxes(rects(grid_centres(n, 25, rng, 4.0), rng.random(n) * 20 + 0.3,
                                           rng.random(n) * 20 + 0.3, rng.random(n) * 2 * math.pi)) for _ in range(3)]
    # corners on integers and half-integers (in pixels) and next to them
    fam["integer_and_half"] = [quads_to_boxes(np.round(grid_centres(n, 25, rng))[:, None, :]
                                              + rng.integers(-16, 17, size=(n, 4, 2)) * 0.5)]
    # off the map on every side, partly and wholly, including negative pixel coordinates
    m = 600
    side = rng.integers(0, 4, m)
    along = rng.random(m) * (SIZE + 40) - 20
    across = rng.random(m) * 60 - 30                   # -30 .. 30 px from the border
    cx = np.where(side == 0, across, np.where(side == 1, SIZE + across, along))
    cy = np.where(side == 2, across, np.where(side == 3, SIZE + across, along))
    fam["off_map"] = [quads_to_boxes(rects(np.stack([cx, cy], 1), rng.random(m) * 30 + 1, rng.random(m) * 30 + 1,
                                           rng.random(m) * 2 * math.pi))]
    # degenerate: zero width, zero height, a single point, collinear corners
    c = grid_centres(n, 25, rng, 6.0)
    w, h, t = rng.random(n) * 18, rng.random(n) * 18, rng.random(n) * 2 * math.pi
    kind = np.arange(n) % 4
    q = rects(c, np.where(kind == 0, 0.0, w), np.where(kind == 1, 0.0, h), np.where(kind < 2, np.where(
        np.arange(n) % 8 < 4, 0.0, t), t))
    q[kind == 2] = c[kind == 2][:, None, :]
    s = rng.random((n, 4, 1)) * 2 - 1
    line = c[:, None, :] + s * np.stack([np.cos(t), np.sin(t)], 1)[:, None, :] * 10
    q[kind == 3] = line[kind == 3]
    fam["degenerate"] = [quads_to_boxes(q)]
    # bow-ties: the dataset's column order fl, fr, bl, br drawn as it is
    q = rects(grid_centres(n, 25, rng, 4.0), rng.random(n) * 20 + 1, rng.random(n) * 20 + 1, rng.random(n) * math.pi)
    fam["bow_tie"] = [quads_to_boxes(q[:, [0, 1, 3, 2]])]
    fam["sub_pixel"] = [quads_to_boxes(rects(grid_centres(n, 25, rng, 10.0), rng.random(n) * 1.2,
                                             rng.random(n) * 1.2, rng.random(n) * math.pi))]
    fam["whole_map"] = [quads_to_boxes(rects(np.array([[400.0, 400.0]]), np.array([900.0]), np.array([900.0]),
                                             np.zeros(1))),
                        quads_to_boxes(rects(np.array([[400.0, 400.0]]), np.array([1200.0]), np.array([1200.0]),
                                             np.array([0.3])))]
    m = 300
    fam["overlapping"] = [quads_to_boxes(rects(rng.random((m, 2)) * 700 + 50, rng.random(m) * 80 + 5,
                                               rng.random(m) * 80 + 5, rng.random(m) * math.pi))]
    fam["ragged"] = [quads_to_boxes(rects(rng.random((k, 2)) * 860 - 30, rng.random(k) * 50 + 1,
                                          rng.random(k) * 30 + 1, rng.random(k) * math.pi)) for k in (0, 1, 7, 130, 333, 0, 45)]
    fam["pillow_triangle"] = [quads_to_boxes(np.array([[[2, 2], [15, 5], [4, 14], [4, 14]]], np.float64)
                                             + np.array([300.0, 500.0]))]
    return fam


def ulp_scenes(dtype):
    """corners one ulp (of the box dtype, in metres) below, on and above pixel coordinates k and k + 1/2"""
    rng = np.random.default_rng(7)
    npdt = np.float32 if dtype == torch.float32 else np.float64
    n = 1000
    base = np.round(grid_centres(n, 25, rng))[:, None, :] + rng.integers(-16, 17, size=(n, 4, 2)) * 0.5
    m = to_metres(base[:, [0, 1, 3, 2], :]).astype(npdt)
    step = rng.integers(-1, 2, size=m.shape)
    m = np.where(step > 0, np.nextafter(m, npdt(np.inf)), np.where(step < 0, np.nextafter(m, npdt(-np.inf)), m))
    return [torch.from_numpy(np.ascontiguousarray(m.transpose(0, 2, 1)))]


def host_maps(scenes):
    from driving_dirty_b200.utils.bb_to_img import boxes_to_binary_map
    return torch.from_numpy(np.stack([boxes_to_binary_map(s).astype(np.float32) for s in scenes]))


def first_difference(got, ref):
    d = (got != ref).nonzero()
    return None if d.numel() == 0 else (tuple(d[0].tolist()), int((got != ref).sum()))


# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_golden_target(golden):
    from driving_dirty_b200 import ops
    g = golden("bb_full_b1")
    t = ops.boxes_to_map(so.synthetic_boxes(g["batch"]), "cuda")
    assert t.shape == (g["batch"], SIZE, SIZE) and t.dtype == torch.float32 and t.is_cuda
    t = t.cpu()
    assert int(t.sum()) == g["target_ones"]
    assert hashlib.sha256(t.reshape(g["batch"], -1).contiguous().numpy().tobytes()).hexdigest() == g["target_sha"]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64], ids=["f32", "f64"])
@pytest.mark.parametrize("family", sorted(family_scenes()) + ["ulp"])
def test_matches_pillow(family, dtype):
    from driving_dirty_b200 import ops
    scenes = ulp_scenes(dtype) if family == "ulp" else [s.to(dtype) for s in family_scenes()[family]]
    got = ops.boxes_to_map(scenes, "cuda").cpu()
    ref = host_maps(scenes)
    assert got.shape == ref.shape
    assert torch.equal(got, ref), first_difference(got, ref)


@pytest.mark.gpu
@pytest.mark.xfail(strict=True, reason="known difference (box_raster.cuh header): a quad that visits the same vertex "
                                       "twice (v1 == v3) differs from Pillow by one pixel at that vertex")
def test_retraced_vertex_matches_pillow():
    from driving_dirty_b200 import ops
    scenes = [quads_to_boxes(np.array([[[491, 160], [481, 162], [490, 167], [481, 162]]], np.float64))]
    got = ops.boxes_to_map(scenes, "cuda").cpu()
    ref = host_maps(scenes)
    assert torch.equal(got, ref), first_difference(got, ref)


@pytest.mark.gpu
def test_empty_batch_and_empty_scenes():
    from driving_dirty_b200 import ops
    assert ops.boxes_to_map([], "cuda").shape == (0, SIZE, SIZE)
    out = ops.boxes_to_map([torch.zeros(0, 2, 4), torch.zeros(0, 2, 4)], "cuda")
    assert out.shape == (2, SIZE, SIZE) and int(out.count_nonzero()) == 0


@pytest.mark.gpu
def test_stays_inside_its_output_buffer():
    """the map sits between two guard bands of a sentinel; the kernel writes every element of the map and nothing else"""
    from driving_dirty_b200._lib import call, stream_ptr
    GUARD = 4096
    scenes = family_scenes()["ragged"] + family_scenes()["off_map"]
    B = len(scenes)
    raw = torch.full((B * SIZE * SIZE + 2 * GUARD,), 7.0, device="cuda")
    out = raw[GUARD: GUARD + B * SIZE * SIZE]
    boxes = torch.cat([s.float() for s in scenes]).cuda()
    offsets = torch.tensor([0] + np.cumsum([s.shape[0] for s in scenes]).tolist(), dtype=torch.int32, device="cuda")
    call("dd_boxes_to_map", boxes.data_ptr(), 0, offsets.data_ptr(), B, out.data_ptr(), stream_ptr())
    torch.cuda.synchronize()
    assert bool((raw[:GUARD] == 7).all()) and bool((raw[GUARD + B * SIZE * SIZE:] == 7).all())
    assert torch.equal(out.view(B, SIZE, SIZE).cpu(), host_maps([s.float() for s in scenes]))


@pytest.mark.gpu
def test_host_pinned_pageable_and_device_inputs_agree():
    """host tensors, pinned or not, are packed into the staging buffer; device tensors are concatenated on the device"""
    from driving_dirty_b200 import ops
    scenes = family_scenes()["ragged"]
    ref = host_maps(scenes)
    pageable = ops.boxes_to_map(scenes, "cuda")
    pinned = ops.boxes_to_map([s.pin_memory() for s in scenes], "cuda")
    device = ops.boxes_to_map([s.cuda() for s in scenes], "cuda")
    for t in (pageable, pinned, device):
        assert torch.equal(t.cpu(), ref)


@pytest.mark.gpu
def test_back_to_back_calls_keep_their_results():
    """the staging slots are reused in turn and grow when a batch needs more room: later calls with other boxes (more
    calls than there are slots, growing batches, device inputs in between) must not change an earlier call's map"""
    from driving_dirty_b200 import ops
    fam = family_scenes()
    batches = [fam["ragged"][:3], fam["rotated"], [s.cuda() for s in fam["off_map"]], fam["overlapping"] * 3,
               fam["ragged"][:3], fam["rotated"] + fam["overlapping"]]
    maps = [ops.boxes_to_map(b, "cuda") for b in batches]
    for b, m in zip(batches, maps):
        assert torch.equal(m.cpu(), host_maps([s.cpu() for s in b]))
    assert torch.equal(maps[0], maps[4])


@pytest.mark.gpu
def test_run_step_dict_targets_match_host_raster(golden):
    """BBSpatialRoadMap._run_step fed the dataloader's dicts (device raster) against the same step fed the host raster"""
    from argparse import Namespace
    import os
    import tempfile
    from driving_dirty_b200.autoencoder.autoencoder import BasicAE, default_hparams
    from driving_dirty_b200.bounding_box_model.spatial_bb.spatial_w_rm import BBSpatialRoadMap
    from driving_dirty_b200.lightning_compat import save_checkpoint
    from driving_dirty_b200.utils.bb_to_img import boxes_to_binary_map
    g = golden("bb_full_b1")
    hp = default_hparams(hidden_dim=g["hidden"], latent_dim=g["latent"])
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ae.ckpt")
        save_checkpoint(BasicAE(hp), path)
        model = BBSpatialRoadMap(Namespace(pretrained_path=path, learning_rate=1e-3, batch_size=2,
                                           output_img_freq=10 ** 9, unfreeze_epoch_no=0, link="", mse_loss=False,
                                           compute_dtype="fp32"))
    model.load_state_dict(so.init_bb_params(g["hidden"], g["latent"]), strict=True)
    model = model.cuda()
    views, road = so.synthetic_scene_batch(2, 256, 306, seed=g["seed_x"])
    boxes = so.synthetic_boxes(2, seed=11) + []
    boxes[1] = torch.cat([boxes[1], family_scenes()["rotated"][0][:50].float()])
    dicts = tuple({"bounding_box": b} for b in boxes)
    raster = torch.from_numpy(np.stack([boxes_to_binary_map(b).copy() for b in boxes]))
    sample, rd = tuple(views.cuda().unbind(0)), tuple(road.cuda().unbind(0))
    with torch.no_grad():
        loss_d, tgt_d, pred_d = model._run_step((sample, dicts, rd), 1, "valid")
        loss_h, tgt_h, pred_h = model._run_step((sample, raster, rd), 1, "valid")
    assert torch.equal(tgt_d, tgt_h)
    assert torch.equal(loss_d, loss_h) and torch.equal(pred_d, pred_h)


@pytest.mark.gpu
def test_bad_inputs_raise():
    from driving_dirty_b200 import ops
    with pytest.raises(ValueError, match="dtype"):
        ops.boxes_to_map([torch.zeros(1, 2, 4), torch.zeros(1, 2, 4, dtype=torch.float64)], "cuda")
    with pytest.raises(ValueError, match="shape"):
        ops.boxes_to_map([torch.zeros(3, 4, 2)], "cuda")
    with pytest.raises(ValueError, match="shape"):
        ops.boxes_to_map([torch.zeros(2, 4)], "cuda")
    with pytest.raises(ValueError, match="dtype"):
        ops.boxes_to_map([torch.zeros(1, 2, 4, dtype=torch.int32)], "cuda")


@pytest.mark.gpu
def test_abi_argument_errors():
    from driving_dirty_b200 import _lib
    lib = _lib.load()
    out = torch.empty(SIZE * SIZE, device="cuda")
    boxes = torch.zeros(8, device="cuda")
    offs = torch.zeros(2, dtype=torch.int32, device="cuda")
    st = _lib.stream_ptr()
    assert lib.dd_boxes_to_map(boxes.data_ptr(), 0, offs.data_ptr(), -1, out.data_ptr(), st) == -1
    assert "B" in _lib.last_error()
    assert lib.dd_boxes_to_map(None, 0, offs.data_ptr(), 1, out.data_ptr(), st) == -1
    assert "null" in _lib.last_error()
    assert lib.dd_boxes_to_map(boxes.data_ptr(), 0, None, 1, out.data_ptr(), st) == -1
    assert lib.dd_boxes_to_map(boxes.data_ptr(), 0, offs.data_ptr(), 1, None, st) == -1
    assert lib.dd_boxes_to_map(None, 0, None, 0, None, st) == 0
    assert lib.dd_boxes_to_map(boxes.data_ptr(), 0, offs.data_ptr(), 1, out.data_ptr() + 4, st) == -4
