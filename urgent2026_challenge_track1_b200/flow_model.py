"""FlowSEModel — the inference-side mirror of ``baseline_code/flow_model.py::FlowSEModel`` (reference
flow_model.py:17-249) without the Lightning dependency: same constructor (``cfg``), same ``dnn.*`` state_dict keys,
same ``enhance(y, fs, speech_length, N=15)``, ``forward(x, t, y) = -dnn(cat[x, y], t)``, ``speech_to_feature`` /
``feature_to_speech``, and the EMA swap at ``eval()`` / ``train()`` (reference :98-112).

``enhance`` runs the fused sampler: STFT (+ exponent compression) kernel -> prior -> N x [network kernels + fused
Euler update on the (B,T,F,2) layout, band_split_y hoisted] -> inverse compression + iSTFT kernel.
"""
from __future__ import annotations

import warnings

import torch
import torch.nn as nn

from . import _lib as L
from . import runtime as R
from .bsrnn_flowse import BSRNN
from .ema import ExponentialMovingAverage
from .odes import FLOWMATCHING
from .sampling import euler_schedule, get_white_box_solver


class FlowSEModel(nn.Module):
    DEFAULT_FS = 48000

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        self.ode = FLOWMATCHING(sigma_min=cfg.sigma_min, sigma_max=cfg.sigma_max)
        self.n_fft, self.hop_length = cfg.n_fft, cfg.hop_length
        self.spec_transform_type = cfg.spec_transform_type
        self.spec_abs_exponent, self.spec_factor = cfg.spec_abs_exponent, cfg.spec_factor
        if self.spec_transform_type not in ("exponent", None, "none"):
            raise NotImplementedError(f"spec_transform_type={self.spec_transform_type!r}")
        self.dnn = BSRNN(input_dim=cfg.n_fft // 2 + 1, num_spk=1, num_layer=cfg.num_layer, target_fs=48000,
                         causal=False, num_channel=cfg.bsrnn_hidden)
        self.lr, self.ema_decay = cfg.learning_rate, cfg.ema_decay
        self.ema = ExponentialMovingAverage(self.parameters(), decay=self.ema_decay)
        self._error_loading_ema = False
        self.t_eps, self.T_rev = cfg.t_eps, cfg.T_rev
        self.ode.T_rev = cfg.T_rev
        self.loss_type = cfg.loss_type

    @classmethod
    def load_from_checkpoint(cls, ckpt_path, map_location="cuda"):
        """Lightning-style .ckpt -> FlowSEModel: ``hyper_parameters['cfg']`` builds the module, ``state_dict`` fills
        it, ``on_load_checkpoint`` restores the EMA shadow weights that ``eval()`` swaps in (flow_model.py:87-112)."""
        from .checkpoint import load_checkpoint, model_kind
        sd, cfg, ckpt = load_checkpoint(ckpt_path)
        if model_kind(sd) != "flowse":
            raise KeyError("not a FlowSEModel checkpoint (no dnn.* keys)")
        if cfg is None:
            raise KeyError("FlowSEModel checkpoint without hyper_parameters['cfg']")
        model = cls(cfg)
        model.load_state_dict(sd)
        model.on_load_checkpoint(ckpt)
        return model.to(map_location)

    # ---- checkpoint hooks (Lightning names kept so a trainer can call them) ---------------------------------
    def on_load_checkpoint(self, checkpoint):
        ema = checkpoint.get("ema", None)
        if ema is not None:
            self.ema.load_state_dict(ema)
        else:
            self._error_loading_ema = True
            warnings.warn("EMA state_dict not found in checkpoint!")

    def on_save_checkpoint(self, checkpoint):
        checkpoint["ema"] = self.ema.state_dict()

    def train(self, mode=True, no_ema=False):
        res = super().train(mode)
        R.invalidate_packed()                      # the EMA swap below rewrites every parameter in place
        if not self._error_loading_ema:
            if mode is False and not no_ema:
                self.ema.store(self.parameters())
                self.ema.copy_to(self.parameters())
            elif self.ema.collected_params is not None:
                self.ema.restore(self.parameters())
        return res

    def eval(self, no_ema=False):
        return self.train(False, no_ema=no_ema)

    def _apply(self, fn, *args, **kwargs):
        """The EMA shadow (and any stored copy) follows the module through .to() / .cuda() / .float() -- the reference
        overrides only ``to`` (flow_model.py:114-117: Lightning moves modules with .to); nn.Module routes all of them
        through ``_apply``."""
        res = super()._apply(fn, *args, **kwargs)
        ema = self.__dict__.get("ema")
        if ema is not None:
            ema.shadow_params = [fn(s) for s in ema.shadow_params]
            if ema.collected_params is not None:
                ema.collected_params = [fn(c) for c in ema.collected_params]
        return res

    # ---- features ---------------------------------------------------------------------------------------------
    def _dims(self, fs):
        return R.stft_dims(int(fs), self.n_fft, self.hop_length, self.DEFAULT_FS)

    def _encode(self, speech, fs, speech_length):
        """(B,L) -> compressed spectrum in the kernel layout (B,T,F,2)."""
        dev = self.dnn.condition_fc.weight.device
        wav = speech.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()
        lens = R.device_lengths(speech_length, dev)
        n_fft, hop = self._dims(fs)
        tr = 1 if self.spec_transform_type == "exponent" else 0
        return R.stft(wav, lens, n_fft, hop, tr, float(self.spec_abs_exponent), float(self.spec_factor))

    def speech_to_feature(self, speech, fs, speech_length):
        """-> complex (B,1,F,T) like the reference (flow_model.py:134-140)."""
        spec = self._encode(speech, fs, speech_length)
        return torch.view_as_complex(spec).permute(0, 2, 1).unsqueeze(1)

    def feature_to_speech(self, feature, fs, speech_length):
        """complex (B,1,F,T) -> (B, max len); decoder hard-codes the 'exponent' transform (flow_model.py:39)."""
        spec = torch.view_as_real(feature.squeeze(1).permute(0, 2, 1).contiguous()).contiguous()
        n_fft, hop = self._dims(fs)
        L_out = int(torch.as_tensor(speech_length).max())
        wav, _ = R.istft(spec, None, None, L_out, n_fft, hop, want_spec=False, transform=1,
                         exponent=float(self.spec_abs_exponent), factor=float(self.spec_factor))
        return wav

    # ---- training (reference flow_model.py:149-187, :211-231) -------------------------------------------------
    def forward_step(self, batch, t=None, z=None):
        """(clean (B,1,T), noisy (B,1,T), fs, lengths) -> flow-matching loss (differentiable; training.py)."""
        from .training import flowse_forward_step
        clean, noisy, fs, lengths = batch
        assert clean.shape[1] == 1                                               # flow_model.py:153
        return flowse_forward_step(self, noisy, clean, lengths, int(fs), t=t, z=z)[0]

    def configure_optimizers(self, process_group=None, precision=None, cuda_graph=False):
        """AdamW(lr, eps=adam_epsilon, weight_decay) [flow_model.py:238-249] + EMA [:84] as one FlowSETrainer.
        precision: "fp32" (f32 recurrence kernels) or "fp16" / "bf16" (the BLSTM blocks on tensor cores); None reads
        ``cfg.train_precision`` (default "fp32").  cuda_graph: replay forward + loss + backward as one CUDA graph."""
        from .training import FlowSETrainer
        cfg = self.cfg
        if precision is None:
            precision = getattr(cfg, "train_precision", "fp32")
        self.trainer_ = FlowSETrainer(self, weight_decay=getattr(cfg, "weight_decay", 1e-6),
                                      eps=getattr(cfg, "adam_epsilon", 1e-8),
                                      gradient_clip=getattr(cfg, "gradient_clip", 0.5), process_group=process_group,
                                      precision=precision, cuda_graph=cuda_graph)
        return self.trainer_

    def training_step(self, batch, batch_idx=0):
        clean, noisy, fs, lengths = batch
        if not hasattr(self, "trainer_"):
            self.configure_optimizers()
        loss, _ = self.trainer_.step(noisy, clean, lengths, fs)
        self.logged = {"train_loss": float(loss)}
        return loss

    # ---- network ----------------------------------------------------------------------------------------------
    @torch.no_grad()
    def forward(self, x, t, y):
        """vector field: -dnn(cat[x, y], t)   (reference flow_model.py:203-209); complex (B,1,F,T) in and out."""
        return -self.dnn(torch.cat([x, y], dim=1), t)

    @torch.no_grad()
    def enhance(self, y, fs, speech_length, N=15, z=None, solver="euler_fused"):
        """Reference flow_model.py:189-200.  ``z``: optional prior noise, complex (B,1,F,T) (drawn with
        torch.randn_like on that shape otherwise, which is what odes.py:88 does).  ``solver``: "euler_fused"
        (default, kernel layout throughout) or any ODEsolverRegistry name for the literal reference loop."""
        L.require_device()
        Y = self._encode(y, fs, speech_length)                                   # (B,T,F,2)
        B, T, F, _ = Y.shape
        dev = Y.device
        if solver != "euler_fused":
            Yc = torch.view_as_complex(Y).permute(0, 2, 1).unsqueeze(1)
            sampler = get_white_box_solver(solver, self.ode, self, Yc, T_rev=self.T_rev, t_eps=self.t_eps, N=N)
            sample, _ = sampler()
            return self.feature_to_speech(sample, fs, speech_length)
        if z is None:
            z = torch.randn_like(torch.view_as_complex(Y).permute(0, 2, 1).unsqueeze(1))
        z_btf = torch.view_as_real(z.to(dev).squeeze(1).permute(0, 2, 1).contiguous()).contiguous()
        st = L.stream_ptr()
        x = torch.empty_like(Y)
        sigma1 = float(self.ode._std(torch.ones(1))[0])
        L.call("bsrnn_axpy_complex", x.data_ptr(), Y.data_ptr(), z_btf.data_ptr(), sigma1, B * T * F, st)   # odes.py:84-91
        zz, plan = self.dnn.embed_y(Y)                                            # loop-invariant band_split_y(y)
        ts, steps = euler_schedule(self.T_rev, self.t_eps, N)
        for i in range(N):
            t = torch.full((B,), float(ts[i]), dtype=torch.float32, device=dev)
            m, r = self.dnn.mask_resid(x, zz, plan, t)
            # x + VF*dt with VF = -(m x + r), dt = -step  ->  x + step*(m x + r)      (odesolvers.py:76-81)
            L.call("bsrnn_euler_step", x.data_ptr(), m.data_ptr(), r.data_ptr(), float(steps[i]), B * T * F, st)
        n_fft, hop = self._dims(fs)
        L_out = int(torch.as_tensor(speech_length).max())
        wav, _ = R.istft(x, None, None, L_out, n_fft, hop, want_spec=False, transform=1,
                         exponent=float(self.spec_abs_exponent), factor=float(self.spec_factor))
        return wav
