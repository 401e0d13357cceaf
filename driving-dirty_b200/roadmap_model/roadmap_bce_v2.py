"""RoadMapBCE: six views -> 800x800 bird's-eye road map, BCE-with-logits loss and threat score
(src/roadmap_model/roadmap_bce_v2.py) on the B200 kernels.  Hook names, return structures and
state_dict keys (``ae.encoder.*``, ``fc1.*``) are the reference's."""
import random
from argparse import ArgumentParser

import numpy as np
import torch
from torch import nn

from .. import ops
from .._lib import IMPL_AUTO
from ..autoencoder.autoencoder import BasicAE
from ..autoencoder.components import resolve_dtype
from ..lightning_compat import FusedGradNorm, LightningModule
from ..utils.helper import compute_ts_road_map  # noqa: F401  (re-exported like the reference)

random.seed(20200505)
np.random.seed(20200505)
torch.manual_seed(20200505)


class RoadMapBCE(FusedGradNorm, LightningModule):
    def __init__(self, hparams):
        super().__init__()
        self.hparams = hparams
        self.map_size = getattr(hparams, "map_size", 800)   # the reference hard-codes 800 (:30,79)
        self.output_dim = self.map_size * self.map_size

        # pretrained feature extractor: the AE checkpoint, frozen, decoder dropped (:43-47)
        self.ae = BasicAE.load_from_checkpoint(self.hparams.pretrained_path)
        if hasattr(hparams, "compute_dtype"):
            self.ae.encoder.compute_dtype = resolve_dtype(hparams.compute_dtype)
        self.frozen = True
        self.ae.freeze()
        self.ae.decoder = None

        self.fc1 = nn.Linear(self.ae.latent_dim, self.output_dim)   # :50
        self.impl = IMPL_AUTO

    # ------------------------------------------------------------------ forward pieces ------
    def wide_stitch_six_images(self, sample):
        """tuple of B [6,3,H,W] (or a [B,6,3,H,W] tensor) -> [B,3,H,6W], views ordered
        [0,1,2,5,4,3] (:53-64)."""
        return ops.stitch(sample)

    def _head(self, z):
        y = ops.linear(z, self.fc1.weight, self.fc1.bias, self.impl,
                       allow_tf32=self.ae.encoder.compute_dtype == torch.bfloat16)
        return y.reshape(y.size(0), self.map_size, self.map_size)

    def _logits(self, x):
        return self._head(self.ae.encoder.forward_views(x))          # stitch folded into the first conv

    def forward(self, x):
        """Returns ``(logits, sigmoid(logits))`` like the reference (:66-81)."""
        y = self._logits(x)
        probs, _ = ops.sigmoid_binary(y)
        return y, probs

    def _run_step(self, batch, batch_idx, step_name):
        """(:83-108) returns (loss, target_rm, logits, probs); BCE, sigmoid and both threat-score
        sums come out of one fused pass, kept on ``self.last_metrics`` for validation_step."""
        sample, target, road_image = batch
        target_rm = (road_image if torch.is_tensor(road_image) else torch.stack(tuple(road_image), dim=0)).float()
        logits = self._logits(sample)
        if batch_idx % self.hparams.output_img_freq == 0 and self.logger is not None:
            self._log_rm_images(self.wide_stitch_six_images(sample), target_rm, torch.sigmoid(logits), step_name)
        loss, probs, binary, stats, counts = ops.bce_threat(logits, target_rm, want_probs=True, want_binary=True)
        self.last_metrics = {"ts": stats[1], "ts_rounded": stats[2], "counts": counts, "binary": binary}
        return loss, target_rm, logits, probs

    def _log_rm_images(self, x, target_rm, pred_rm, step_name, limit=1):
        import torchvision
        x, target_rm, pred_rm = x[:limit], target_rm[:limit], pred_rm[:limit].round()
        exp, step = self.logger.experiment, getattr(self.trainer, "global_step", 0)
        exp.add_image(f"{step_name}_input_images", torchvision.utils.make_grid(x), step)
        exp.add_image(f"{step_name}_target_roadmaps", torchvision.utils.make_grid(target_rm), step)
        exp.add_image(f"{step_name}_pred_roadmaps", torchvision.utils.make_grid(pred_rm), step)

    # ------------------------------------------------------------------ Lightning hooks -----
    def training_step(self, batch, batch_idx):
        if self.current_epoch >= self.hparams.unfreeze_epoch_no and self.frozen:   # :127-129
            self.frozen = False
            self.ae.unfreeze()
        train_loss, _, _, _ = self._run_step(batch, batch_idx, step_name="train")
        return {"loss": train_loss, "log": {"train_loss": train_loss}}

    def validation_step(self, batch, batch_idx):
        val_loss, target_rm, pred_rm, pred_logit_rm = self._run_step(batch, batch_idx, step_name="valid")
        # compute_ts_road_map(target, probs) and (target, probs.round()) (:139-140) were accumulated
        # by the fused loss kernel in the same pass
        m = self.last_metrics
        return {"val_loss": val_loss, "val_ts_rounded": m["ts_rounded"], "val_ts": m["ts"]}

    def validation_epoch_end(self, outputs):
        avg_val_loss = torch.stack([x["val_loss"] for x in outputs]).mean()
        avg_val_ts = torch.stack([x["val_ts"] for x in outputs]).mean()
        avg_val_ts_rounded = torch.stack([x["val_ts_rounded"] for x in outputs]).mean()
        logs = {"avg_val_loss": avg_val_loss, "avg_val_ts_rounded": avg_val_ts_rounded, "avg_val_ts": avg_val_ts}
        return {"val_loss": avg_val_loss, "log": logs}

    def configure_optimizers(self):
        from ..optim import make_adam
        optimizer = make_adam(self, self.hparams.learning_rate)       # :155 (FusedAdam unless --optimizer torch)
        scheduler = torch.optim.lr_scheduler.ReduceLROnPlateau(optimizer, patience=10)
        return [optimizer], [scheduler]

    @staticmethod
    def add_model_specific_args(parent_parser):
        parser = ArgumentParser(parents=[parent_parser], add_help=False)
        parser.add_argument("--learning_rate", type=float, default=1e-3)
        parser.add_argument("--unfreeze_epoch_no", type=int, default=0)
        parser.add_argument("--batch_size", type=int, default=16)
        parser.add_argument("--link", type=str, default="/scratch/ab8690/DLSP20Dataset/data")
        parser.add_argument("--pretrained_path", type=str, required=True)
        parser.add_argument("--output_img_freq", type=int, default=500)
        parser.add_argument("--compute_dtype", type=str, default="fp32", choices=["fp32", "bf16"])
        parser.add_argument("--optimizer", type=str, default="fused", choices=["fused", "torch"])
        return parser
