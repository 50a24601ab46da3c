"""Lightning-format ``.ckpt`` reader / writer (SURVEY.md §8f.3) so checkpoints move both ways between this package and
the reference: ``state_dict`` + ``hyper_parameters['cfg']`` (+ ``ema`` for FlowSE, flow_model.py:87-96), the layout
``L.Trainer``'s ModelCheckpoint writes and ``SEModel/FlowSEModel.load_from_checkpoint`` read (reference
inference.py:30-33, train_se.py:55-60,67-72).

The reference pickles its ``Config`` object by class reference ``baseline_code.config.Config`` (config.py:6).  To
read such a file without the reference installed -- and to write files the reference can read -- an alias module
``baseline_code.config`` exposing a ``Config`` with the same attribute-bag behaviour is registered in ``sys.modules``
when (and only when) the real one is not importable."""
from __future__ import annotations

import importlib
import sys
import types

import torch

from .config import Config

LIGHTNING_VERSION = "2.5.2"          # reference pin (setup.py:17); informational only


def _reference_config_class():
    """``baseline_code.config.Config``: the real class when the reference is importable, else an alias of ours."""
    try:
        return importlib.import_module("baseline_code.config").Config
    except Exception:
        pass
    pkg = sys.modules.get("baseline_code")
    if pkg is None:
        pkg = types.ModuleType("baseline_code")
        pkg.__path__ = []                                   # a package, so ``baseline_code.config`` resolves
        sys.modules["baseline_code"] = pkg
    mod = types.ModuleType("baseline_code.config")
    alias = type("Config", (Config,), {"__module__": "baseline_code.config", "__qualname__": "Config"})
    mod.Config = alias
    sys.modules["baseline_code.config"] = mod
    pkg.config = mod
    return alias


def to_reference_config(cfg):
    """Our Config (or any attribute bag) -> an instance that pickles as ``baseline_code.config.Config``."""
    cls = _reference_config_class()
    out = cls.__new__(cls)
    out.__dict__.update(vars(cfg))
    return out


def from_reference_config(obj):
    """Pickled reference Config (or a dict) -> our Config carrying the same attributes."""
    if obj is None:
        return None
    return Config(**(dict(obj) if isinstance(obj, dict) else vars(obj)))


def save_checkpoint(path, model, cfg, *, global_step=0, epoch=0, ema=None, optimizer_states=None, lr_schedulers=None,
                    extra=None):
    """Writes the dict Lightning's ModelCheckpoint writes.  ``model``: SEModel / FlowSEModel (keys ``se_model.*`` /
    ``dnn.*``).  ``ema``: torch_ema-style state_dict (FlowSEModel.on_save_checkpoint, flow_model.py:95-96).  ``extra``:
    further top-level keys (the training loop's ``b200_trainer`` state)."""
    sd = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
    ckpt = {"epoch": int(epoch), "global_step": int(global_step), "pytorch-lightning_version": LIGHTNING_VERSION,
            "state_dict": sd, "loops": {}, "callbacks": {}, "optimizer_states": optimizer_states or [],
            "lr_schedulers": lr_schedulers or [], "hparams_name": "cfg",
            "hyper_parameters": {"cfg": to_reference_config(cfg)}}
    if ema is None and hasattr(model, "on_save_checkpoint") and hasattr(model, "ema"):
        model.on_save_checkpoint(ckpt)
    elif ema is not None:
        ckpt["ema"] = ema
    if "ema" in ckpt:
        e = dict(ckpt["ema"])
        for k in ("shadow_params", "collected_params"):
            if e.get(k) is not None:
                e[k] = [t.detach().cpu().clone() for t in e[k]]
        ckpt["ema"] = e
    ckpt.update(extra or {})
    torch.save(ckpt, path)
    return path


def load_checkpoint(path):
    """-> (state_dict, cfg or None, raw checkpoint dict).  Accepts a Lightning .ckpt or a bare state_dict file."""
    _reference_config_class()                                # make the pickled Config resolvable
    ckpt = torch.load(path, map_location="cpu", weights_only=False)
    if isinstance(ckpt, dict) and "state_dict" in ckpt:
        cfg = from_reference_config((ckpt.get("hyper_parameters") or {}).get("cfg"))
        return ckpt["state_dict"], cfg, ckpt
    return ckpt, None, {}


def model_kind(state_dict):
    """'se' for SEModel checkpoints (``se_model.*`` keys), 'flowse' for FlowSEModel ones (``dnn.*``)."""
    if any(k.startswith("se_model.") for k in state_dict):
        return "se"
    if any(k.startswith("dnn.") for k in state_dict):
        return "flowse"
    raise ValueError("neither an SEModel (se_model.*) nor a FlowSEModel (dnn.*) checkpoint")
