"""train_se — entry point mirroring ``baseline_code/train_se.py`` (reference train_se.py:37-84) for both models it
selects by ``model_type`` (:50-53): the discriminative BSRNN (``se``, default) and BSRNN-FlowSE (``flowse``).
``--config_file conf/models/BSRNN_baseline.yaml`` plus every Config field as a flag; one process per GPU
under torchrun (the reference lets Lightning spawn them), gradients averaged with ONE NCCL allreduce of the flat
buffer per step; ``init_from`` accepts a raw or Lightning-style state_dict (:55-60); checkpoints are written in the
reference's layout ``{"state_dict": ..., "hyper_parameters": {"cfg": cfg}}``.

FlowSE (``model_type: flowse``) trains with the flow-matching loss, AdamW and the EMA fused into the optimizer tail, the
forward + loss + backward replayed as one CUDA graph.  Its BLSTM blocks run at the precision of the YAML key
``train_precision`` (default ``fp16``: tensor cores, f32 master weights; ``fp32``: the f32 recurrence kernels).  Its
checkpoints carry the EMA weights under ``ema`` (flow_model.py:87-96), so FlowSEModel.load_from_checkpoint and
inference.py read them as they read the reference's.

The reference's data pipeline (dataset.py, dynamic mixing, simulation/) is out of scope (SURVEY.md §2 row 9): pass
``--data synthetic`` (default) for random (clean, noisy) pairs of the dataset contract — (clean (B,1,T), noisy (B,1,T),
fs int32 scalar, lengths (B,) int32), one fs per batch (dataset.py:417,441) — or plug any iterator yielding that
contract into ``fit()``.
"""
from __future__ import annotations

import os
import sys

import torch

from .config import Config, config_parser
from .d_model import SEModel

RATES = (8000, 16000, 22050, 24000, 32000, 44100, 48000)


def synthetic_batches(cfg, rank, world, steps, device):
    """Rank-strided stream of synthetic batches (the sampler shards by sorted_indices[rank::world], dataset.py:361)."""
    g = torch.Generator().manual_seed(cfg.seed + rank)
    for i in range(steps):
        fs = RATES[(i * world + rank) % len(RATES)] if getattr(cfg, "mixed_rates", False) else 48000
        n = int(cfg.max_duration)                                   # max_duration is in SAMPLES (dataset.py:144-147)
        clean = 0.05 * torch.randn(cfg.batch_size, 1, n, generator=g)
        noisy = clean + 0.03 * torch.randn(cfg.batch_size, 1, n, generator=g)
        lens = torch.full((cfg.batch_size,), n, dtype=torch.int32)
        yield clean.to(device), noisy.to(device), torch.tensor(fs, dtype=torch.int32), lens


def fit(model: SEModel, batches, cfg, rank=0, log_every=10, out_dir=None):
    trainer = model.configure_optimizers()
    last = None
    for step, batch in enumerate(batches):
        last = model.training_step(batch, step)
        if rank == 0 and step % log_every == 0:
            print(f"step {step}: " + " ".join(f"{k}={v:.4g}" for k, v in model.logged.items()), flush=True)
    if out_dir and rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        torch.save({"state_dict": model.state_dict(), "hyper_parameters": {"cfg": cfg}, "global_step": trainer.step_count},
                   os.path.join(out_dir, f"last-step{trainer.step_count:06d}.ckpt"))
    return last


def fit_flowse(model, batches, cfg, rank=0, log_every=10, out_dir=None):
    """FlowSEModel training loop: FlowSETrainer steps (fp16 tensor-core blocks by default, CUDA-graph replay); at the
    end rank 0 writes ``last-step<N>.ckpt`` with the EMA state (``trainer.sync_ema()`` first)."""
    from .checkpoint import save_checkpoint
    trainer = model.configure_optimizers(precision=getattr(cfg, "train_precision", "fp16"), cuda_graph=True)
    last = None
    for step, (clean, noisy, fs, lengths) in enumerate(batches):
        last, _ = trainer.step(noisy, clean, lengths, fs)
        if rank == 0 and step % log_every == 0:
            print(f"step {step}: train_loss={float(last):.4g}", flush=True)
    if out_dir and rank == 0:
        trainer.sync_ema()
        os.makedirs(out_dir, exist_ok=True)
        save_checkpoint(os.path.join(out_dir, f"last-step{trainer.step_count:06d}.ckpt"), model, cfg,
                        global_step=trainer.step_count, ema=model.ema.state_dict())
    return last


def main(argv=None):
    import torch.distributed as dist
    args = config_parser(argv)
    cfg = Config(**vars(args))
    cfg.read_yaml()
    if cfg.model_configs is None:
        cfg.model_configs = {"num_channel": 196, "num_layer": 6}
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.manual_seed(cfg.seed)
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    flowse = getattr(cfg, "model_type", "se") == "flowse"
    if flowse:
        from .flow_model import FlowSEModel
        model = FlowSEModel(cfg)
    else:
        model = SEModel(cfg, precision="fp32")
    if cfg.init_from != "none":
        sd = torch.load(cfg.init_from, map_location="cpu", weights_only=False)
        model.load_state_dict(sd.get("state_dict", sd))
    model.to(dev)
    if world > 1:                                                    # DDP broadcasts rank 0's parameters at wrap time
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    steps = int(getattr(cfg, "max_steps", 20))
    out_dir = os.path.join("exp", cfg.train_tag, cfg.train_name, f"version_{cfg.train_version}", "checkpoints")
    (fit_flowse if flowse else fit)(model, synthetic_batches(cfg, rank, world, steps, dev), cfg, rank,
                                    out_dir=out_dir if getattr(cfg, "save", False) else None)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main(sys.argv[1:])
