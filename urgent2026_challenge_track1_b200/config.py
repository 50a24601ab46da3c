"""Config — same schema and flag behaviour as ``baseline_code/config.py`` (reference config.py:6-73): defaults become
--flags of the default's type, YAML keys overwrite/extend attributes without validation, train_tag := YAML basename."""
from __future__ import annotations

import argparse
import os

import yaml

_DEFAULTS = dict(
    learning_rate=1e-3, batch_size=2, weight_decay=1e-6, adam_epsilon=1e-8, num_worker=4, num_train_epochs=150,
    device="cuda", num_gpu=1, train_version=0, train_tag="run_0", train_name="baseline", val_check_interval=50000,
    save_top_k=3, resume=True, seed=1996, gradient_clip=0.5, lr_step_size=1, lr_gamma=0.85, train_set_path="none",
    train_set_dynamic_mixing=True, valid_set_path="none", init_from="none", max_duration=96000, use_high_pass=True,
    se_model="bsrnn", config_file="none", model_configs=None)


class Config:
    def __init__(self, **kwargs):
        for k, v in _DEFAULTS.items():
            setattr(self, k, v)
        for k, v in kwargs.items():
            setattr(self, k, v)

    def read_yaml(self):
        if self.config_file != "none":
            with open(self.config_file, "r", encoding="utf-8") as f:
                for k, v in yaml.safe_load(f.read()).items():
                    setattr(self, k, v)
            self.train_tag = os.path.basename(self.config_file).replace(".yaml", "")

    def __repr__(self):
        return f"Config({vars(self)})"


def _str2bool(v):
    if isinstance(v, bool):
        return v
    if v.lower() in ("yes", "true", "t", "y", "1"):
        return True
    if v.lower() in ("no", "false", "f", "n", "0"):
        return False
    raise argparse.ArgumentTypeError("Boolean value expected.")


# keys of this package that have no reference default: a flag sets them, and without the flag (or the YAML key) the
# attribute stays absent, so every getattr(cfg, key, default) keeps its default
_OPTIONAL_FLAGS = dict(train_precision=str, max_steps=int)


def config_parser(argv=None):
    parser = argparse.ArgumentParser()
    for name, default in vars(Config()).items():
        parser.add_argument(f"--{name}", type=_str2bool if isinstance(default, bool) else type(default), default=default)
    for name, typ in _OPTIONAL_FLAGS.items():
        parser.add_argument(f"--{name}", type=typ, default=argparse.SUPPRESS)
    return parser.parse_args(argv)
