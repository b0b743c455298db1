"""``PseudoSpeakerVAE`` -- drop-in for the LightningModule of ps_vae/lightning.py:10-214.

Same ``**hparams`` constructor, attributes (``model``, ``classifier``, ``consistency_classifier``, ``multilabel``,
``accuracy``, ``kl_loss_weight``, ``classifier_loss_weight``, ``consitency_loss_weight`` (sic), ``use_cos_loss``),
methods (``forward``, ``decode``, ``training_step``, ``validation_step``, ``configure_optimizers``,
``load_vae_from_checkpoint``), metric names and state-dict keys.  It subclasses ``pytorch_lightning.LightningModule``
when that package is importable and a small stand-in with the same surface otherwise (it is not installed in the
build image, SURVEY F9/H7).

What changes underneath: ``training_step`` makes ONE call into the CUDA library that runs the forward, all loss
terms, and the whole backward (lightning.py:67-131 + ``loss.backward()``), and returns a loss tensor whose
``.backward()`` merely hands the already-computed flat gradients to autograd (so Lightning's automatic
optimisation, gradient accumulation and DDP hooks keep working); ``configure_optimizers`` returns ``FusedAdam``
(one vectorised pass) with the stock ``CosineAnnealingLR``.

Extra hparams (additive): ``precision`` ('fp32' parity mode / 'bf16' tensor-core mode), and ``model`` accepts
``hidden_dim`` / ``num_hidden_layers``.  ``consistency_classifier_ckpt`` (lightning.py:44-52) loads the frozen
``EmbeddingClassifier`` whose cross entropy on ``x_hat`` joins the loss inside the same fused call.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import _lib as L
from .embedding_classifier import EmbeddingClassifier
from .engine import HotPath
from .latent_classifier import LatentClassifier
from .model import VAEModel
from .optim import FusedAdam

from ._compat import HAVE_LIGHTNING, _Accuracy, _Base  # noqa: F401  (Lightning base class or its stand-in)


class PseudoSpeakerVAE(_Base):
    def __init__(self, **hparams):
        super().__init__()
        self.save_hyperparameters()

        self.model = VAEModel(**hparams["model"])

        if hparams.get("vae_checkpoint", None):
            print(f"Using VAE checkpoint {hparams['vae_checkpoint']}")
            self.load_vae_from_checkpoint(hparams["vae_checkpoint"])

        if hparams.get("freeze_vae", False):
            print("Freezing VAE")
            for param in self.model.parameters():
                param.requires_grad = False

        if "classifier" in hparams:
            classifier_hparams = hparams["classifier"]
            clf_kwargs = {k: v for k, v in classifier_hparams.items() if k != "label_classes"}
            self.classifier = LatentClassifier(**clf_kwargs)
            if isinstance(classifier_hparams["num_classes"], int):
                self.multilabel = False
                self.accuracy = _Accuracy(task="multiclass", num_classes=classifier_hparams["num_classes"])
            else:
                # the reference reads classifier_hparams['label_classes'] here and then passes the same dict to
                # LatentClassifier, which rejects it (SURVEY F10); both spellings are accepted
                self.multilabel = True
                classes = classifier_hparams.get("label_classes", classifier_hparams["num_classes"])
                self.accuracy = nn.ModuleDict({name: _Accuracy(task="multiclass", num_classes=c) for name, c in classes.items()})
        else:
            self.classifier = None

        if "consistency_classifier_ckpt" in hparams:
            # lightning.py:44-52: a frozen EmbeddingClassifier in eval mode; its CE on x_hat joins the loss (lightning.py:100-108)
            self.consistency_classifier = EmbeddingClassifier.load_from_checkpoint(hparams["consistency_classifier_ckpt"])
            for param in self.consistency_classifier.parameters():
                param.requires_grad = False
            self.consistency_classifier.eval()
        else:
            self.consistency_classifier = None

        self.kl_loss_weight = hparams.get("kl_loss_weight", 1.0)
        self.classifier_loss_weight = hparams.get("classifier_loss_weight", 1.0)
        self.consitency_loss_weight = hparams.get("consistency_loss_weight", 1.0)
        self.use_cos_loss = hparams.get("use_cos_loss", False)

        precision = hparams.get("precision", hparams["model"].get("precision", "fp32"))
        hot = HotPath(self.model, self.classifier, precision)
        object.__setattr__(self, "_hot", hot)
        self.model._adopt(hot)

    # ---- reference surface ---------------------------------------------------------------------------
    @property
    def hot_path(self) -> HotPath:
        return self._hot

    def forward(self, x: torch.Tensor, eps: Optional[torch.Tensor] = None) -> tuple:
        return self._hot.forward(x, eps)

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        return self._hot.decode(z)

    def _shared_step(self, batch, prefix: str, compute_grads: bool, eps: Optional[torch.Tensor], **log_kw) -> dict:
        x, y = batch
        cons = self.consistency_classifier
        if cons is not None and isinstance(y, dict):
            # the reference calls cross_entropy(y_hat_consistency, y) with the batch's y (lightning.py:102): a single label tensor
            raise ValueError("the consistency classifier needs single-label targets (a tensor), got a dict of labels")
        cons_y = y if cons is not None else None
        if self.classifier is None:
            y = None
        hot = self._hot
        train_vae = any(p.requires_grad for p in self.model.parameters())
        need_grads = compute_grads and torch.is_grad_enabled() and (train_vae or self.classifier is not None)
        # freeze_vae (the second stage of a two-stage run): the classifier scope skips the whole VAE backward
        losses, gflat, _ = hot.step(x, y, eps, kl_weight=self.kl_loss_weight, clf_weight=self.classifier_loss_weight,
                                    use_cos_loss=self.use_cos_loss, compute_grads=need_grads, consistency=cons, consistency_y=cons_y,
                                    consistency_weight=self.consitency_loss_weight, grad_scope=hot.train_scope() if need_grads else "all")
        if self.classifier is not None:
            if not self.multilabel:
                self.log(f"{prefix}_classifier_acc", losses[L.LOSS_ACC_HEAD0], sync_dist=True)
                self.log(f"{prefix}_classifier_loss", losses[L.LOSS_CLF], sync_dist=True)
            else:
                running = 0
                for h, name in enumerate(hot.head_names):
                    running = running + losses[L.LOSS_CLF_HEAD0 + h]      # the reference logs the running sum (lightning.py:88-93)
                    self.log(f"{prefix}_classifier_acc_{name}", losses[L.LOSS_ACC_HEAD0 + h], sync_dist=True)
                    self.log(f"{prefix}_classifier_loss_{name}", running, sync_dist=True)
        if cons is not None:
            self.log(f"{prefix}_consistency", losses[L.LOSS_CONS_ACC], sync_dist=True)          # lightning.py:105-106 / 167-168
            self.log(f"{prefix}_consistency_loss", losses[L.LOSS_CONS], sync_dist=True)
        self.log(f"{prefix}_loss", losses[L.LOSS_TOTAL], sync_dist=True, **log_kw)
        self.log(f"{prefix}_recon_loss", losses[L.LOSS_RECON], sync_dist=True, **log_kw)
        self.log(f"{prefix}_kl_loss", losses[L.LOSS_KL], sync_dist=True, **log_kw)
        total = hot.loss_with_grad(losses, gflat) if need_grads else losses[L.LOSS_TOTAL].clone()
        return {"loss": total}

    def training_step(self, batch: tuple, batch_idx: int, eps: Optional[torch.Tensor] = None) -> dict:
        """lightning.py:67-131.  ``eps`` (optional) injects the reparameterisation noise (parity tests)."""
        return self._shared_step(batch, "train", True, eps)

    def validation_step(self, batch: tuple, batch_idx: int, eps: Optional[torch.Tensor] = None) -> dict:
        """lightning.py:133-197: identical math, ``val_`` names, no gradients."""
        return self._shared_step(batch, "val", False, eps, batch_size=batch[0].size(0))

    def load_vae_from_checkpoint(self, checkpoint_path):
        checkpoint = torch.load(checkpoint_path, map_location=self.device, weights_only=False)
        vae_state_dict = {k.replace("model.", ""): v for k, v in checkpoint["state_dict"].items() if k.startswith("model.")}
        self.model.load_state_dict(vae_state_dict)

    def configure_optimizers(self):
        # the frozen consistency classifier never receives a gradient (lightning.py:48-49): torch's Adam skips it, the fused pass leaves it out
        in_arena = {id(p) for p in self._hot.parameters()}
        params = [p for p in self.parameters() if id(p) in in_arena]
        optimizer = FusedAdam(params, **self.hparams["optimizer"], arena=self._hot.arena)
        scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, **self.hparams["scheduler"])
        return {
            "optimizer": optimizer,
            "lr_scheduler": {"scheduler": scheduler, "interval": "epoch", "frequency": 1},
        }
