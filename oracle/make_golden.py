"""Generate tests/golden/*.pt from the UNMODIFIED reference -- TEST INFRASTRUCTURE.

Runs only in the build container, where /root/reference exists:

    python oracle/make_golden.py

It imports the reference's own modules (src.autoencoder.autoencoder.BasicAE,
src.roadmap_model.roadmap_bce_v2.RoadMapBCE, src.utils.helper.compute_ts_road_map) from
/root/reference with the dependency stand-ins in oracle/shims/ (pytorch_lightning, test_tube,
shapely, matplotlib are not installed and there is no network), drives them on seeded
synthetic inputs, and stores inputs (or their seeds), weights (or their seeds) and the
reference's outputs.  tests/test_oracle.py then checks oracle/scene_oracle.py against these
files; tests on the GPU box check the CUDA path against the same files.  Nothing at test,
smoke or bench time reads /root/reference.
"""
from __future__ import annotations

import hashlib
import os
import sys
import tempfile
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "shims"))
sys.path.insert(0, "/root/reference")
sys.path.insert(0, ROOT)

from oracle import scene_oracle as so  # noqa: E402

from src.autoencoder.autoencoder import BasicAE  # noqa: E402
from src.roadmap_model.roadmap_bce_v2 import RoadMapBCE  # noqa: E402
from src.utils.helper import compute_ts_road_map  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def sha(t: torch.Tensor) -> str:
    return hashlib.sha256(np.ascontiguousarray(t.detach().cpu().numpy()).tobytes()).hexdigest()


def sample(t: torch.Tensor, n: int = 4096) -> torch.Tensor:
    return so.strided_sample(t, n)


def build_reference_roadmap(params: dict, hidden: int, latent: int, view_h: int, view_w: int):
    """Fabricate the AE checkpoint RoadMapBCE.__init__ demands (roadmap_bce_v2.py:43) and load
    ``params`` into the reference model."""
    ns = Namespace(hidden_dim=hidden, latent_dim=latent, input_width=6 * view_w, input_height=view_h,
                   output_width=view_w, output_height=view_h, in_channels=3, batch_size=4,
                   learning_rate=1e-3, output_img_freq=10 ** 9, link="/nonexistent")
    ae = BasicAE(ns)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ae.ckpt")
        torch.save({"state_dict": ae.state_dict(), "hparams": vars(ns)}, path)
        del ae
        model = RoadMapBCE(Namespace(pretrained_path=path, learning_rate=1e-3, batch_size=4,
                                     output_img_freq=10 ** 9, unfreeze_epoch_no=0, link="/nonexistent"))
    missing = model.load_state_dict({k: v.clone() for k, v in params.items()}, strict=True)
    assert not missing.missing_keys and not missing.unexpected_keys
    return model


def roadmap_case(name: str, batch: int, hidden: int, latent: int, view_h: int, view_w: int,
                 with_grads: bool, store_params: bool):
    seed_w, seed_x, seed_fwd = 20200505, 20200506, 1234
    params = so.init_roadmap_params(hidden, latent, view_h, view_w, seed=seed_w)
    views, road = so.synthetic_scene_batch(batch, view_h, view_w, seed=seed_x)
    if store_params:
        # small train cases: pick the first input seed with no conv pre-activation within 2e-6 of the
        # ReLU threshold (see scene_oracle.min_abs_preactivation)
        while so.min_abs_preactivation(params, views) < 2e-6:
            seed_x += 1
            views, road = so.synthetic_scene_batch(batch, view_h, view_w, seed=seed_x)
    model = build_reference_roadmap(params, hidden, latent, view_h, view_w)
    sample_t = tuple(views.unbind(0))   # what collate_fn hands the module (helper.py:22-23)
    road_t = tuple(road.unbind(0))
    gold = dict(name=name, batch=batch, hidden=hidden, latent=latent, view_h=view_h, view_w=view_w,
                seed_w=seed_w, seed_x=seed_x, seed_fwd=seed_fwd,
                min_abs_preactivation=so.min_abs_preactivation(params, views))

    # ---- frozen / eval pass (validation_step, roadmap_bce_v2.py:135-143) -------------------
    with torch.no_grad():
        mosaic = model.wide_stitch_six_images(sample_t)
        torch.manual_seed(seed_fwd)
        loss, target_rm, logits, probs = model._run_step((sample_t, None, road_t), 1, "valid")
        ts = compute_ts_road_map(target_rm, probs)
        ts_r = compute_ts_road_map(target_rm, probs.round())
    gold["eval"] = dict(mosaic_sha=sha(mosaic), mosaic_sample=sample(mosaic),
                        loss=loss.clone(), ts=ts.clone(), ts_rounded=ts_r.clone(),
                        logits_sha=sha(logits), logits_sample=sample(logits),
                        probs_sample=sample(probs),
                        binary_sha=sha(probs.round().to(torch.uint8)),
                        binary_ones=int(probs.round().sum().item()),
                        logits_absmax=float(logits.abs().max()))
    if store_params:
        gold["eval"]["logits_b0_strided"] = logits[0, ::8, ::8].clone()

    # ---- unfrozen training pass (training_step, :125-133) ---------------------------------
    if with_grads:
        model.current_epoch = 0
        model.zero_grad()
        if model.frozen:                       # the reference's own unfreeze logic (:127-129)
            model.frozen = False
            model.ae.unfreeze()
        torch.manual_seed(seed_fwd)
        loss, _, logits, probs = model._run_step((sample_t, None, road_t), 1, "train")
        loss.backward()
        grads = {k: v.grad.clone() for k, v in model.named_parameters()}
        tr = dict(loss=loss.detach().clone(), logits_sample=sample(logits), logits_sha=sha(logits),
                  grad_sha={k: sha(g) for k, g in grads.items()},
                  grad_norm={k: float(g.double().norm()) for k, g in grads.items()},
                  grad_sample={k: sample(g, 2048) for k, g in grads.items()},
                  bn_after={k: v.clone() for k, v in model.state_dict().items()
                            if "running_" in k or "num_batches" in k})
        if store_params:
            tr["grads_small"] = {k: g for k, g in grads.items() if g.numel() <= 70000}
        gold["train"] = tr

    if store_params:
        gold["params_small"] = {k: v.clone() for k, v in params.items() if v.numel() <= 70000}
        gold["params_sha"] = {k: sha(v) for k, v in params.items()}
    torch.save(gold, os.path.join(GOLD, name + ".pt"))
    print(name, "loss", float(gold["eval"]["loss"]), "ts_r", float(gold["eval"]["ts_rounded"]),
          "ones", gold["eval"]["binary_ones"])


def ae_case(name: str, batch: int, hidden: int, latent: int, view_h: int, view_w: int):
    ns = Namespace(hidden_dim=hidden, latent_dim=latent, input_width=6 * view_w, input_height=view_h,
                   output_width=view_w, output_height=view_h, in_channels=3, batch_size=batch,
                   learning_rate=1e-3, output_img_freq=10 ** 9, link="/nonexistent")
    torch.manual_seed(20200505)
    ae = BasicAE(ns)
    views, _ = so.synthetic_scene_batch(batch, view_h, view_w, map_hw=8, seed=777)
    # six_to_one_task hard-codes the 306-pixel slot (autoencoder.py:61-62): only exercise it at
    # full width; at reduced geometry call it for the stitch and redo the mask by hand below.
    np.random.seed(4321)
    slot = int(np.random.randint(0, 5))
    gold = dict(name=name, batch=batch, hidden=hidden, latent=latent, view_h=view_h, view_w=view_w,
                slot=slot, hw=(ae.decoder.deconv_dim_h, ae.decoder.deconv_dim_w))
    if view_w == 306:
        np.random.seed(4321)
        x, y = ae.six_to_one_task(views.clone())
        gold["x_sha"], gold["y_sha"] = sha(x), sha(y)
        gold["x_sample"], gold["y_sample"] = sample(x), sample(y)
    else:
        gold["state_dict"] = {k: v.clone() for k, v in ae.state_dict().items()}
        x, y = so.six_to_one(views, slot)
        ae.train()
        torch.manual_seed(99)
        z = ae.encoder(x)
        y_hat = ae(z)
        loss = torch.nn.functional.mse_loss(y, y_hat)
        loss.backward()
        gold.update(z=z.detach().clone(), y_hat=y_hat.detach().clone(), loss=loss.detach().clone(),
                    grad_norm={k: float(v.grad.double().norm()) for k, v in ae.named_parameters()},
                    grad_sample={k: sample(v.grad, 512) for k, v in ae.named_parameters()})
    torch.save(gold, os.path.join(GOLD, name + ".pt"))
    print(name, "slot", slot, "loss", float(gold.get("loss", float("nan"))))


def bb_case(name: str, batch: int, hidden: int, latent: int):
    """BBSpatialRoadMap (spatial_w_rm.py) at full geometry (the merging CNN only fits 256x306 views
    and 800x800 maps).  The module imports boxes_to_binary_map from src.utils.helper, where it
    does not exist (SURVEY D6): inject the real one from src.utils.bb_to_img before the import --
    a test-time patch of the module namespace, no reference file is edited."""
    import src.utils.helper as ref_helper
    import src.utils.bb_to_img as ref_bb
    ref_helper.boxes_to_binary_map = ref_bb.boxes_to_binary_map
    from src.bounding_box_model.spatial_bb.spatial_w_rm import BBSpatialRoadMap

    params = so.init_bb_params(hidden, latent)
    ns = Namespace(hidden_dim=hidden, latent_dim=latent, input_width=6 * 306, input_height=256, output_width=306,
                   output_height=256, in_channels=3, batch_size=batch, learning_rate=1e-3, output_img_freq=10 ** 9,
                   link="/nonexistent")
    ae = BasicAE(ns)
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "ae.ckpt")
        torch.save({"state_dict": ae.state_dict(), "hparams": vars(ns)}, path)
        del ae
        torch.manual_seed(20200505)
        model = BBSpatialRoadMap(Namespace(pretrained_path=path, learning_rate=1e-3, batch_size=batch,
                                           output_img_freq=10 ** 9, unfreeze_epoch_no=0, link="/nonexistent",
                                           mse_loss=False))
    sd = model.state_dict()
    assert all(k in sd and sd[k].shape == v.shape for k, v in params.items())
    missing = model.load_state_dict({k: v.clone() for k, v in params.items()}, strict=False)
    assert not missing.unexpected_keys
    views, road = so.synthetic_scene_batch(batch, 256, 306, seed=20200508)
    boxes = so.synthetic_boxes(batch)
    target = tuple({"bounding_box": b} for b in boxes)
    model.logger = None
    model.frozen = False
    model.ae.unfreeze()
    model.train()
    batch_t = (tuple(views.unbind(0)), target, tuple(road.unbind(0)))
    loss, tgt, pred = model._run_step(batch_t, 1, "train")
    loss.backward()
    grads = {k: v.grad for k, v in model.named_parameters() if v.grad is not None}
    # the oracle's restatement of the rasteriser and of the whole step
    tgt_o = torch.from_numpy(np.stack([so.boxes_to_binary_map(b).copy() for b in boxes])).float()
    assert torch.equal(tgt_o.reshape(batch, -1), tgt)
    gold = dict(name=name, batch=batch, hidden=hidden, latent=latent, seed_x=20200508,
                loss=loss.detach().clone(), pred_sample=sample(pred), pred_absmax=float(pred.abs().max()),
                target_ones=int(tgt.sum()), target_sha=sha(tgt),
                params_sha={k: sha(v) for k, v in params.items()},
                grad_norm={k: float(v.double().norm()) for k, v in grads.items()},
                grad_sample={k: sample(v, 512) for k, v in grads.items()})
    torch.save(gold, os.path.join(GOLD, name + ".pt"))
    print(name, "loss", float(loss), "target ones", gold["target_ones"], "grads", len(grads))


def binarise_case():
    """Exhaustive fp32 sweep around 0 through the reference's own sigmoid().round() (:140)."""
    lo = np.float32(2.0 ** -27).view(np.uint32)
    hi = np.float32(2.0 ** -20).view(np.uint32)
    bits = np.arange(lo, hi, dtype=np.uint32)
    x = torch.from_numpy(bits.view(np.float32).copy())
    r = torch.sigmoid(x).round()
    first = int(torch.nonzero(r == 1).flatten()[0])
    assert bool((r[first:] == 1).all()) and bool((r[:first] == 0).all())
    edge = torch.tensor([0.0, -0.0, -1e-30, 1e-30, -2.0 ** -20, 2.0 ** -20, 20.0, -20.0, 88.0, -88.0,
                         -104.0, 104.0, float("inf"), float("-inf")])
    gold = dict(first_one_bits=int(bits[first]), sweep_lo=int(lo), sweep_hi=int(hi),
                edge_x=edge, edge_round=torch.sigmoid(edge).round(), edge_sigmoid=torch.sigmoid(edge))
    torch.save(gold, os.path.join(GOLD, "binarise.pt"))
    print("binarise first-one bits", hex(gold["first_one_bits"]))


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    torch.set_num_threads(so.GOLDEN_THREADS)
    if len(sys.argv) > 1 and sys.argv[1] == "bb":
        bb_case("bb_full_b1", batch=1, hidden=8, latent=8)
        sys.exit(0)
    binarise_case()
    roadmap_case("roadmap_small", batch=4, hidden=16, latent=8, view_h=16, view_w=20,
                 with_grads=True, store_params=True)
    roadmap_case("roadmap_odd", batch=5, hidden=24, latent=8, view_h=10, view_w=14,
                 with_grads=True, store_params=True)
    ae_case("ae_small", batch=3, hidden=16, latent=8, view_h=16, view_w=20)
    ae_case("ae_stitch_full", batch=2, hidden=8, latent=8, view_h=256, view_w=306)
    roadmap_case("roadmap_full_b2", batch=2, hidden=256, latent=128, view_h=256, view_w=306,
                 with_grads=True, store_params=False)
