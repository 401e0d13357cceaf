"""The oracle (oracle/scene_oracle.py) against outputs of the unmodified reference
(tests/golden/*.pt, written by oracle/make_golden.py in the build container).  CPU only."""
import hashlib

import numpy as np
import pytest
import torch

from oracle import scene_oracle as so


@pytest.fixture(autouse=True)
def golden_thread_count():
    """The goldens are compared bit for bit: run torch's CPU ops with the thread count they were written with."""
    n = torch.get_num_threads()
    torch.set_num_threads(so.GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def sha(t):
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def _case(golden, name):
    g = golden(name)
    p = so.init_roadmap_params(g["hidden"], g["latent"], g["view_h"], g["view_w"], seed=g["seed_w"])
    views, road = so.synthetic_scene_batch(g["batch"], g["view_h"], g["view_w"], seed=g["seed_x"])
    return g, p, views, road


@pytest.mark.parametrize("name", ["roadmap_small", "roadmap_odd"])
def test_params_reproduce(golden, name):
    g, p, _, _ = _case(golden, name)
    for k, h in g["params_sha"].items():
        assert sha(p[k]) == h, k
    for k, v in g["params_small"].items():
        assert torch.equal(p[k], v)


@pytest.mark.parametrize("name", ["roadmap_small", "roadmap_odd"])
def test_eval_pass_bit_exact(golden, name):
    g, p, views, road = _case(golden, name)
    e = g["eval"]
    assert sha(so.stitch(views)) == e["mosaic_sha"]
    with torch.no_grad():
        out = so.run_step(p, tuple(views.unbind(0)), tuple(road.unbind(0)), training=False, seed=g["seed_fwd"])
    assert sha(out["logits"]) == e["logits_sha"]
    assert torch.equal(so.strided_sample(out["logits"]), e["logits_sample"])
    assert torch.equal(so.strided_sample(out["probs"]), e["probs_sample"])
    assert torch.equal(out["loss"], e["loss"])
    assert torch.equal(out["ts"], e["ts"])
    assert torch.equal(out["ts_rounded"], e["ts_rounded"])
    binary = so.binarise(out["probs"])
    assert sha(binary.to(torch.uint8)) == e["binary_sha"]
    assert int(binary.sum()) == e["binary_ones"]
    # the threshold form and the integer TS restatement agree with the reference too
    assert torch.equal(so.binarise(out["logits"], from_logits=True), binary)
    tp, nt, nr = so.threat_score_counts(out["target"], binary)
    assert np.float32(tp) / np.float32(nt + nr - tp) == e["ts_rounded"].numpy()
    # float64 BCE restatement within fp32 rounding of torch's
    assert abs(float(so.bce_with_logits_mean(out["logits"], out["target"])) - float(e["loss"])) < 2e-7


@pytest.mark.parametrize("name", ["roadmap_small", "roadmap_odd"])
def test_train_pass_bit_exact(golden, name):
    g, p, views, road = _case(golden, name)
    t = g["train"]
    out, grads = so.train_step_grads(p, tuple(views.unbind(0)), tuple(road.unbind(0)), seed=g["seed_fwd"])
    assert torch.equal(out["loss"].detach(), t["loss"])
    assert sha(out["logits"]) == t["logits_sha"]
    for k, h in t["grad_sha"].items():
        assert sha(grads[k]) == h, k
    # analytic BCE gradient restatement
    gl = so.bce_with_logits_grad(out["logits"].detach(), out["target"])
    assert gl.shape == out["logits"].shape


def test_pool_restatement_matches_torch():
    torch.manual_seed(0)
    a3 = torch.relu(torch.randn(2, 32, 5, 42))
    ref = torch.nn.functional.max_pool1d(a3.view(2, -1).unsqueeze(1), 4).squeeze(1)
    assert torch.equal(so.pool4_flat(a3), ref)
    # ragged: 3*7*5 = 105 elements -> 26 windows, 1 element dropped
    a = torch.randn(1, 3, 7, 5)
    ref = torch.nn.functional.max_pool1d(a.view(1, -1).unsqueeze(1), 4).squeeze(1)
    assert torch.equal(so.pool4_flat(a), ref)
    arg = so.pool4_flat_argmax(torch.zeros(1, 1, 2, 4))
    assert (arg == 0).all()  # ties -> first


def test_binarise_threshold_exhaustive(golden):
    g = golden("binarise")
    assert g["first_one_bits"] == so.BINARISE_THRESHOLD_BITS + 1
    bits = np.arange(g["sweep_lo"], g["sweep_hi"], dtype=np.uint32)
    x = torch.from_numpy(bits.view(np.float32).copy())
    assert torch.equal(so.binarise(x, from_logits=True), torch.sigmoid(x).round())
    assert torch.equal(so.binarise(g["edge_x"], from_logits=True), g["edge_round"])
    assert torch.equal(so.binarise(-x[::7], from_logits=True), torch.zeros_like(x[::7]))


def test_ae_small(golden):
    g = golden("ae_small")
    p = g["state_dict"]
    views, _ = so.synthetic_scene_batch(g["batch"], g["view_h"], g["view_w"], map_hw=8, seed=777)
    out = so.ae_run_step({k: v.clone() for k, v in p.items()}, views, g["slot"], True, g["hw"], seed=99)
    assert torch.equal(out["z"], g["z"])
    assert torch.equal(out["y_hat"], g["y_hat"])
    assert torch.equal(out["loss"], g["loss"])


def test_ae_stitch_full(golden):
    g = golden("ae_stitch_full")
    views, _ = so.synthetic_scene_batch(g["batch"], 256, 306, map_hw=8, seed=777)
    x, y = so.six_to_one(views, g["slot"])
    assert sha(x) == g["x_sha"] and sha(y) == g["y_sha"]


@pytest.mark.slow
def test_full_size_eval(golden):
    """BASELINE config 1 (B=2, 6x3x256x306, hidden 256 / latent 128) -- about 20 s of CPU."""
    g, p, views, road = _case(golden, "roadmap_full_b2")
    e = g["eval"]
    assert sha(so.stitch(views)) == e["mosaic_sha"]
    with torch.no_grad():
        out = so.run_step(p, tuple(views.unbind(0)), tuple(road.unbind(0)), training=False, seed=g["seed_fwd"])
    assert sha(out["logits"]) == e["logits_sha"]
    assert torch.equal(out["loss"], e["loss"])
    assert torch.equal(out["ts_rounded"], e["ts_rounded"])
    assert sha(so.binarise(out["logits"], from_logits=True).to(torch.uint8)) == e["binary_sha"]


def _bb_inputs(g):
    import numpy as np
    p = so.init_bb_params(g["hidden"], g["latent"])
    views, road = so.synthetic_scene_batch(g["batch"], 256, 306, seed=g["seed_x"])
    boxes = so.synthetic_boxes(g["batch"])
    target = torch.from_numpy(np.stack([so.boxes_to_binary_map(b).copy() for b in boxes])).float()
    return p, views, road, target


@pytest.mark.slow
def test_bb_full_b1(golden):
    """Bounding-box model with roadmap input (config 4), full geometry, B=1: the oracle's restatement
    against the unmodified reference's _run_step (loss, prediction sample, every gradient)."""
    g = golden("bb_full_b1")
    p, views, road, target = _bb_inputs(g)
    for k, v in p.items():
        assert sha(v) == g["params_sha"][k], k
    assert int(target.sum()) == g["target_ones"] and sha(target.reshape(g["batch"], -1)) == g["target_sha"]
    q = {k: v.clone().requires_grad_(k in g["grad_norm"]) for k, v in p.items()}
    out = so.bb_run_step(q, views, road, target)
    assert torch.equal(out["loss"].detach(), g["loss"])
    assert torch.equal(so.strided_sample(out["pred"]), g["pred_sample"])
    out["loss"].backward()
    for k in g["grad_norm"]:
        assert torch.equal(so.strided_sample(q[k].grad, 512), g["grad_sample"][k]), k


def test_box_iou_stand_in_on_analytic_cases():
    """The shapely stand-in of compute_iou (helper.py:79-83) against cases with a closed form; corners in the dataset's
    order fl, fr, bl, br (a bow-tie as a ring, hence the reference's convex_hull)."""
    def box(cx, cy, dx, dy, ang=0.0):
        import math
        c, s = math.cos(ang), math.sin(ang)
        pts = [(dx, dy), (dx, -dy), (-dx, dy), (-dx, -dy)]
        xs = [cx + c * x - s * y for x, y in pts]
        ys = [cy + s * x + c * y for x, y in pts]
        return torch.tensor([xs, ys], dtype=torch.float32)
    a = box(0, 0, 2, 1)
    assert abs(so.compute_iou(a, a) - 1.0) < 1e-12
    assert abs(so.compute_iou(a, box(2, 0, 2, 1)) - (4.0 / 12.0)) < 1e-6          # half overlap: 4 / (8 + 8 - 4)
    assert abs(so.compute_iou(a, box(1, 1, 2, 1)) - (3.0 / 13.0)) < 1e-6
    assert so.compute_iou(a, box(10, 0, 2, 1)) == 0.0
    sq, diamond = box(0, 0, 1, 1), box(0, 0, 1, 1, ang=0.7853981633974483)        # unit square vs the same rotated 45 deg
    inter = 8 * (2 ** 0.5 - 1)                                                    # regular octagon of inradius 1
    assert abs(so.compute_iou(sq, diamond) - inter / (8 - inter)) < 1e-6
    # score: identical sets -> every box matches at every threshold -> tp = n, ts = n / (2n - n) = 1
    boxes = torch.stack([box(3 * i, 0, 1, 1) for i in range(4)])
    ats, iou = so.compute_ats_bounding_boxes(boxes, boxes)
    assert abs(float(ats) - 1.0) < 1e-6 and torch.allclose(torch.diagonal(iou), torch.ones(4))
    ats0, _ = so.compute_ats_bounding_boxes(boxes, boxes + 100.0)
    assert float(ats0) == 0.0
