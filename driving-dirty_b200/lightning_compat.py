"""LightningModule base for the drop-in task modules.

The reference subclasses pytorch_lightning.LightningModule (0.7.5, requirements.txt:3) and uses
four things from it on this path: ``freeze`` / ``unfreeze`` (roadmap_bce_v2.py:46,129),
``load_from_checkpoint`` (:43) and ``current_epoch`` (:127).  When pytorch-lightning is installed
the real class is used; otherwise this minimal base supplies those four with PL 0.7.5 semantics,
so the modules work as plain nn.Modules driven by any loop.
"""
from argparse import Namespace

import torch
from torch import nn

try:  # pragma: no cover - not installed in the build image
    from pytorch_lightning import LightningModule as _PLModule  # type: ignore
    HAVE_LIGHTNING = True
except Exception:  # noqa: BLE001
    _PLModule = None
    HAVE_LIGHTNING = False


class _MinimalLightningModule(nn.Module):
    def __init__(self, *args, **kwargs):
        super().__init__()
        self.current_epoch = 0
        self.global_step = 0
        self.logger = None
        self.trainer = None

    def freeze(self):
        for p in self.parameters():
            p.requires_grad = False
        self.eval()

    def unfreeze(self):
        for p in self.parameters():
            p.requires_grad = True
        self.train()

    def grad_norm(self, norm_type):
        """PL 0.7.5's GradInformation.grad_norm: the norm of every parameter's .grad (rounded host floats) and their total."""
        results, total_norm = {}, 0
        for name, p in self.named_parameters():
            if p.requires_grad and p.grad is not None:
                param_norm = p.grad.data.norm(norm_type)
                total_norm += param_norm ** norm_type
                results[f"grad_{norm_type}_norm_{name}"] = round(float(param_norm ** (1 / norm_type)), 3)
        results[f"grad_{norm_type}_norm_total"] = round(float(total_norm ** (1. / norm_type)), 3)
        return results

    @classmethod
    def load_from_checkpoint(cls, checkpoint_path, map_location=None, **kwargs):
        ckpt = torch.load(checkpoint_path, map_location=map_location or "cpu", weights_only=False)
        hparams = ckpt.get("hparams", ckpt.get("hyper_parameters", {}))
        if not isinstance(hparams, Namespace):
            hparams = Namespace(**hparams)
        model = cls(hparams)
        model.load_state_dict(ckpt["state_dict"])
        return model


LightningModule = _PLModule if HAVE_LIGHTNING else _MinimalLightningModule


class FusedGradNorm:
    """``grad_norm(norm_type)``, the hook behind Lightning's ``track_grad_norm``, for modules whose optimizer
    (``optim.attach_optimizer``) may be a FusedAdam: the wide weights' gradients never reach ``.grad`` there, and at world
    size N ``.grad`` is this rank's replica.  With a FusedAdam that tracks this norm the values are its ``grad_norms()``
    -- the gradients its step applies, the rank mean at world size N -- as device tensors (no rounding, no host copy);
    otherwise the base class answers, as before."""

    def grad_norm(self, norm_type):
        from .optim import FusedAdam
        opt = getattr(self, "_dd_optimizer", None)
        tracked = (isinstance(opt, FusedAdam) and opt.track_grad_norm == 2 and not isinstance(norm_type, bool)
                   and isinstance(norm_type, (int, float)) and norm_type == 2)
        if not tracked:
            return super().grad_norm(norm_type)
        norms = opt.grad_norms()
        by_id = {id(k): v for k, v in norms.items() if not isinstance(k, str)}
        out = {f"grad_{norm_type}_norm_{name}": by_id[id(p)] for name, p in self.named_parameters() if id(p) in by_id}
        out[f"grad_{norm_type}_norm_total"] = norms["total"]
        return out


def save_checkpoint(module, path):
    """Write the ``{'state_dict', 'hparams'}`` file load_from_checkpoint reads (PL 0.7.5 layout)."""
    hp = getattr(module, "hparams", None)
    # clones: a parameter adopted by optim.FusedAdam's sharded form lives inside one large symmetric buffer, and
    # torch.save writes a tensor's whole storage
    sd = {k: v.detach().clone() for k, v in module.state_dict().items()}
    torch.save({"state_dict": sd, "hparams": vars(hp) if isinstance(hp, Namespace) else dict(hp or {})}, path)
