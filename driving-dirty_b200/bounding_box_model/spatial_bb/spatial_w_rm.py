"""BBSpatialRoadMap: six views + the road map -> 800x800 object-occupancy probabilities
(src/bounding_box_model/spatial_bb/spatial_w_rm.py) on the B200 kernels.  Hook names, return
structures and state_dict keys (``ae.encoder.*``, ``space_map_cnn.*``, ``box_merge.*``) are the
reference's."""
import random
from argparse import ArgumentParser

import numpy as np
import torch

from ... import ops
from ...autoencoder.autoencoder import BasicAE
from ...autoencoder.components import resolve_dtype
from ...lightning_compat import FusedGradNorm, LightningModule
from .components import RoadMapBoxesMergingCNN, SpatialMappingCNN

random.seed(20200505)
np.random.seed(20200505)
torch.manual_seed(20200505)


class BBSpatialRoadMap(FusedGradNorm, LightningModule):
    def __init__(self, hparams):
        super().__init__()
        self.hparams = hparams
        self.output_dim = 800 * 800
        dtype = resolve_dtype(getattr(hparams, "compute_dtype", "fp32"))

        # pretrained feature extractor: the AE checkpoint, frozen, conv stack only (:44-49)
        self.ae = BasicAE.load_from_checkpoint(self.hparams.pretrained_path)
        self.ae.encoder.compute_dtype = dtype
        self.frozen = True
        self.ae.freeze()
        self.ae.encoder.c3_only = True
        self.ae.decoder = None

        self.space_map_cnn = SpatialMappingCNN(dtype)
        self.box_merge = RoadMapBoxesMergingCNN(dtype)
        self.compute_dtype = dtype

    def wide_stitch_six_images(self, x):
        """[B,6,3,H,W] -> [B,3,H,6W], views ordered [0,1,2,5,4,3] (:54-65)."""
        return ops.stitch(x)

    def forward(self, x, rm):
        """x [B,6,3,256,306], rm [B,1,800,800] -> [B,800,800] probabilities (:67-83)."""
        views = ops.as_view_batch(x)
        space_rep = self.space_map_cnn.forward_nhwc(views)
        enc = self.ae.encoder
        ssr = ops.encoder_conv_stack(views, enc.c1, enc.c2, enc.c3, act_dtype=enc.compute_dtype, c3_only=2, impl=enc.impl)
        rm_nhwc = ops.to_nhwc(rm, self.compute_dtype)                 # one channel: a cast, no reordering
        yhat = self.box_merge.forward_nhwc(ssr, space_rep, rm_nhwc)   # [B,800,800,1]
        return yhat.float().reshape(yhat.shape[0], yhat.shape[1], yhat.shape[2])

    def bb_coord_to_map(self, target):
        """tuple of B dicts with 'bounding_box' [N,2,4] -> [B,800,800] raster (:85-95) on the model's device: the
        reference's boxes_to_binary_map per scene, bit for bit, rasterised by the device kernel (ops.boxes_to_map)."""
        return ops.boxes_to_map([s["bounding_box"] for s in target], next(self.parameters()).device)

    def _run_step(self, batch, batch_idx, step_name):
        sample, target, road_image = batch
        sample = ops.as_view_batch(sample)
        # `target`: the dataloader's tuple of dicts (rasterised here, on the device, :85-95), or -- an
        # extension for loaders that rasterise ahead of time -- the [B,800,800] raster itself
        target_bb_img = (target if torch.is_tensor(target) else self.bb_coord_to_map(target)).to(device=sample.device,
                                                                                              dtype=torch.float32)
        rm = (road_image if torch.is_tensor(road_image) else torch.stack(tuple(road_image), dim=0)).float().unsqueeze(1)
        pred_bb_img = self(sample, rm)
        if batch_idx % self.hparams.output_img_freq == 0 and self.logger is not None:
            self._log_rm_images(sample[0], target_bb_img[0], pred_bb_img[0], step_name)
        batch_size = target_bb_img.size(0)
        target_bb_img = target_bb_img.view(batch_size, -1)
        pred_bb_img = pred_bb_img.view(batch_size, -1)
        if getattr(self.hparams, "mse_loss", False):
            loss = ops.mse_loss(pred_bb_img, target_bb_img)       # F.mse_loss(pred, target), :129
        else:
            loss = ops.bce_prob(pred_bb_img, target_bb_img)       # F.binary_cross_entropy, :131
        return loss, target_bb_img, pred_bb_img

    def _log_rm_images(self, x, target, pred, step_name, limit=1):
        import torchvision
        exp, step = self.logger.experiment, getattr(self.trainer, "global_step", 0)
        exp.add_image(f"{step_name}_input_images", torchvision.utils.make_grid(x), step)
        exp.add_image(f"{step_name}_target_bbs", torchvision.utils.make_grid(target), step)
        exp.add_image(f"{step_name}_pred_bbs", torchvision.utils.make_grid(pred), step)

    def training_step(self, batch, batch_idx):
        if self.current_epoch >= self.hparams.unfreeze_epoch_no and self.frozen:
            self.frozen = False
            self.ae.unfreeze()
        train_loss, _, _ = self._run_step(batch, batch_idx, step_name="train")
        return {"loss": train_loss, "log": {"train_loss": train_loss}}

    def validation_step(self, batch, batch_idx):
        val_loss, _, _ = self._run_step(batch, batch_idx, step_name="valid")
        return {"val_loss": val_loss}

    def validation_epoch_end(self, outputs):
        avg_val_loss = torch.stack([x["val_loss"] for x in outputs]).mean()
        return {"val_loss": avg_val_loss, "log": {"avg_val_loss": avg_val_loss}}

    def configure_optimizers(self):
        from ...optim import make_adam
        return make_adam(self, self.hparams.learning_rate)

    @staticmethod
    def add_model_specific_args(parent_parser):
        parser = ArgumentParser(parents=[parent_parser], add_help=False)
        parser.add_argument("--learning_rate", type=float, default=0.001)
        parser.add_argument("--batch_size", type=int, default=16)
        parser.add_argument("--link", type=str, default="/scratch/ab8690/DLSP20Dataset/data")
        parser.add_argument("--pretrained_path", type=str, required=True)
        parser.add_argument("--output_img_freq", type=int, default=500)
        parser.add_argument("--unfreeze_epoch_no", type=int, default=0)
        parser.add_argument("--mse_loss", default=False, action="store_true")
        parser.add_argument("--compute_dtype", type=str, default="fp32", choices=["fp32", "bf16"])
        return parser
