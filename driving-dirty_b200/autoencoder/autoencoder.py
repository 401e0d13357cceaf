"""BasicAE: the self-supervised six-to-one autoencoder (src/autoencoder/autoencoder.py) on the
B200 kernels.  Same hparams, attributes, methods and state_dict keys as the reference."""
import random
from argparse import ArgumentParser, Namespace

import numpy as np
import torch

from .. import ops
from ..lightning_compat import FusedGradNorm, LightningModule
from .components import Decoder, Encoder, resolve_dtype

# the reference seeds at import time (autoencoder.py:16-18); kept so that scripts which rely on
# that reproducibility see the same streams
random.seed(20200505)
np.random.seed(20200505)
torch.manual_seed(20200505)


class BasicAE(FusedGradNorm, LightningModule):
    def __init__(self, hparams=None):
        super().__init__()
        self.__check_hparams(hparams)
        self.hparams = hparams
        self.encoder = self.init_encoder(self.hidden_dim, self.latent_dim, self.in_channels, self.input_height,
                                         self.input_width)
        self.decoder = self.init_decoder(self.hidden_dim, self.latent_dim, self.in_channels, self.output_height,
                                         self.output_width)

    def __check_hparams(self, hparams):  # autoencoder.py:32-43 (defaults included)
        g = lambda name, default: getattr(hparams, name) if hasattr(hparams, name) else default  # noqa: E731
        self.hidden_dim = g("hidden_dim", 128)
        self.latent_dim = g("latent_dim", 128)
        self.input_width = g("input_width", 306 * 6)
        self.input_height = g("input_height", 256)
        self.output_width = g("output_width", 306)
        self.output_height = g("output_height", 256)
        self.batch_size = g("batch_size", 16)
        self.in_channels = g("in_channels", 3)
        # new, optional: storage type of the conv activations ("fp32" parity path | "bf16")
        self.compute_dtype = resolve_dtype(g("compute_dtype", "fp32"))

    def init_encoder(self, hidden_dim, latent_dim, in_channels, input_height, input_width):
        return Encoder(hidden_dim, latent_dim, in_channels, input_height, input_width, self.compute_dtype)

    def init_decoder(self, hidden_dim, latent_dim, in_channels, output_height, output_width):
        return Decoder(hidden_dim, latent_dim, in_channels, output_height, output_width, self.compute_dtype)

    def six_to_one_task(self, x):
        """autoencoder.py:53-73: stitch, draw ``np.random.randint(0, 5)`` (host RNG, one slot per
        batch, slot 5 never drawn), y = the slot's block, x with that block zeroed.  The slot width
        is the view width (306 in the reference, which hard-codes it)."""
        target_img_index = np.random.randint(0, 5)
        x, y = ops.stitch_mask(x, target_img_index)
        assert x.size(-1) == 6 * y.size(-1)
        return x, y

    def forward(self, z):
        return self.decoder(z)

    def _run_step(self, batch, batch_idx, step_name):
        x, y = self.six_to_one_task(batch)
        z = self.encoder(x)
        y_hat = self(z)
        return ops.mse_loss(y, y_hat)  # F.mse_loss(y, y_hat), autoencoder.py:91

    def training_step(self, batch, batch_idx):
        train_loss = self._run_step(batch, batch_idx, step_name="train")
        return {"loss": train_loss, "log": {"train_loss": train_loss}}

    def validation_step(self, batch, batch_idx):
        return {"val_loss": self._run_step(batch, batch_idx, step_name="valid")}

    def validation_epoch_end(self, outputs):
        avg_val_loss = torch.stack([x["val_loss"] for x in outputs]).mean()
        return {"val_loss": avg_val_loss, "log": {"avg_val_loss": avg_val_loss}}

    def configure_optimizers(self):
        from ..optim import make_adam
        return make_adam(self, self.hparams.learning_rate)

    @staticmethod
    def add_model_specific_args(parent_parser):
        parser = ArgumentParser(parents=[parent_parser], add_help=False)
        parser.add_argument("--hidden_dim", type=int, default=256)
        parser.add_argument("--latent_dim", type=int, default=128)
        parser.add_argument("--learning_rate", type=float, default=0.001)
        parser.add_argument("--batch_size", type=int, default=16)
        parser.add_argument("--input_width", type=int, default=306 * 6)
        parser.add_argument("--input_height", type=int, default=256)
        parser.add_argument("--output_width", type=int, default=306)
        parser.add_argument("--output_height", type=int, default=256)
        parser.add_argument("--in_channels", type=int, default=3)
        parser.add_argument("--link", type=str, default="/scratch/ab8690/DLSP20Dataset/data")
        parser.add_argument("--output_img_freq", type=int, default=500)
        parser.add_argument("--compute_dtype", type=str, default="fp32", choices=["fp32", "bf16"])
        return parser


def default_hparams(**over):
    """Namespace with the reference's CLI defaults (autoencoder.py:161-182)."""
    d = dict(hidden_dim=256, latent_dim=128, learning_rate=1e-3, batch_size=16, input_width=306 * 6,
             input_height=256, output_width=306, output_height=256, in_channels=3, link="", output_img_freq=500,
             compute_dtype="fp32")
    d.update(over)
    return Namespace(**d)
