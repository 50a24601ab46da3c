"""SEModel — Lightning-free mirror of ``baseline_code/d_model.py::SEModel`` (reference d_model.py:12-113): selector
``cfg.se_model == "bsrnn"`` -> ``BSRNN_SE(**cfg.model_configs)`` under the attribute ``se_model`` (so checkpoint keys are
``se_model.bsrnn.bsrnn.*``), TypeError for anything else (reference :19-23); ``forward_step`` / ``training_step`` /
``validation_step`` / ``configure_optimizers`` keep the reference's names and meaning, with the optimizer replaced by
the fused flat-buffer step of training.SETrainer."""
from __future__ import annotations

import torch
import torch.nn as nn

from .bsrnn import BSRNN_SE


class SEModel(nn.Module):
    def __init__(self, cfg, precision=None):
        super().__init__()
        self.cfg = cfg
        if cfg.se_model == "bsrnn":
            self.se_model = BSRNN_SE(**cfg.model_configs, precision=precision)
        else:
            self.se_model = None
            raise TypeError

    @torch.no_grad()
    def forward(self, noisy_speech, speech_length, fs):
        return self.se_model(noisy_speech, speech_length, fs)

    # ------------------------------------------------------------------------------------------------ training
    def configure_optimizers(self, process_group=None, precision=None, cuda_graph=None):
        """AdamW(lr, eps=adam_epsilon, weight_decay) + StepLR(lr_step_size epochs, lr_gamma) + clip 0.5
        [d_model.py:102-113, train_se.py:78] as one SETrainer (flat parameters, one allreduce, fused update).
        precision None reads ``cfg.train_precision`` (default "fp32": the f32 kernels); cuda_graph None replays the
        step as a CUDA graph exactly when the BLSTM blocks run on tensor cores ("fp16" / "bf16")."""
        from .training import SETrainer
        cfg = self.cfg
        if precision is None:
            precision = getattr(cfg, "train_precision", "fp32")
        if cuda_graph is None:
            cuda_graph = precision != "fp32"
        self.trainer_ = SETrainer(self.se_model, lr=cfg.learning_rate, weight_decay=cfg.weight_decay,
                                  eps=cfg.adam_epsilon, gradient_clip=cfg.gradient_clip, process_group=process_group,
                                  precision=precision, cuda_graph=cuda_graph)
        self.epoch_ = 0
        return self.trainer_

    def forward_step(self, batch, batch_idx=0, stage="train"):
        """(clean (B,1,T), noisy (B,1,T), fs, lengths) -> loss   [d_model.py:61-89]; logs land in self.logged."""
        clean, noisy, fs, lengths = batch
        assert clean.shape[1] == 1 and noisy.shape[1] == 1                   # d_model.py:66
        if not hasattr(self, "trainer_"):
            self.configure_optimizers()
        loss, sisnr = self.trainer_.loss(noisy, clean, lengths, fs)
        self.logged = {f"{stage}_loss": float(loss.detach()), f"{stage}_sisnr": float(sisnr),
                       f"{stage}_sisnr_{int(fs)}": float(sisnr)}
        return loss

    def training_step(self, batch, batch_idx=0):
        """One full optimisation step (forward, loss, backward, allreduce, clip, AdamW); returns the loss."""
        clean, noisy, fs, lengths = batch
        if not hasattr(self, "trainer_"):
            self.configure_optimizers()
        loss, sisnr = self.trainer_.step(noisy, clean, lengths, fs)
        self.logged = {"train_loss": float(loss), "train_sisnr": float(sisnr), "Grad_norm": self.trainer_.grad_norm()}
        return loss

    @torch.no_grad()
    def validation_step(self, batch, batch_idx=0):
        return self.forward_step(batch, batch_idx, stage="val")

    def on_train_epoch_end(self):
        """StepLR(step_size=lr_step_size, gamma=lr_gamma) [d_model.py:110-111]."""
        self.epoch_ += 1
        if self.epoch_ % max(1, int(self.cfg.lr_step_size)) == 0:
            self.trainer_.set_lr(self.trainer_.lr * self.cfg.lr_gamma)

    @classmethod
    def load_from_checkpoint(cls, ckpt_path, map_location="cuda", precision=None):
        """Reads a Lightning-style .ckpt (``state_dict`` + ``hyper_parameters['cfg']``) or a raw state_dict
        (reference train_se.py:55-60 accepts both for init_from)."""
        from .checkpoint import load_checkpoint, model_kind
        sd, cfg, _ = load_checkpoint(ckpt_path)
        if model_kind(sd) != "se":
            raise KeyError("not an SEModel checkpoint (no se_model.* keys)")      # inference.py:30-33 falls back on this
        if cfg is None:
            from .config import Config
            n = sd["se_model.bsrnn.bsrnn.fc_time.0.bias"].numel()
            layers = 1 + max(int(k.split(".")[4]) for k in sd if k.startswith("se_model.bsrnn.bsrnn.fc_time."))
            cfg = Config(se_model="bsrnn", model_configs={"num_channel": n, "num_layer": layers})
        model = cls(cfg, precision=precision)
        model.load_state_dict(sd)
        return model.to(map_location)
