"""train_se — entry point mirroring ``baseline_code/train_se.py`` (reference train_se.py:37-84) for both models it
selects by ``model_type`` (:50-53): the discriminative BSRNN (``se``, default) and BSRNN-FlowSE (``flowse``).
``--config_file conf/models/BSRNN_baseline.yaml`` plus every Config field as a flag; one process per GPU
under torchrun (the reference lets Lightning spawn them), gradients averaged with ONE NCCL allreduce of the flat
buffer per step; ``init_from`` accepts a raw or Lightning-style state_dict (:55-60); checkpoints are written in the
reference's layout ``{"state_dict": ..., "hyper_parameters": {"cfg": cfg}}``.

The YAML key ``train_precision`` picks the BLSTM precision: ``fp16`` runs the blocks on tensor cores (f32 master
weights) and replays forward + loss + backward as one CUDA graph, ``fp32`` runs the f32 recurrence kernels.  SE defaults
to ``fp32`` with host launches when the key is absent (``fp16`` is the recommended setting); FlowSE defaults to ``fp16``.
FlowSE trains with the flow-matching loss, AdamW and the EMA fused into the optimizer tail; its checkpoints carry the EMA
weights under ``ema`` (flow_model.py:87-96), so FlowSEModel.load_from_checkpoint and inference.py read them as they read
the reference's.

Data.  With ``train_set_path`` a directory of pre-simulated pairs (``wav.scp`` noisy, ``spk1.scp`` clean; data.py), the
run loops ``num_train_epochs`` epochs over it (``max_steps``, when set, caps the global step), in same-rate,
length-bucketed batches of ``batch_size`` cropped to ``max_duration`` samples, read by ``num_worker`` DataLoader workers.
``valid_set_path`` adds a validation pass every ``val_check_interval`` global steps and at the end; rank 0 keeps the best
``save_top_k`` checkpoints by ``val_loss`` under ``exp/<train_tag>/<train_name>/version_<v>/checkpoints/``, named
``best_epoch=EE-step=SSSSSS-val_loss=V.VVV.ckpt``, with the optimizer state under ``b200_trainer``; ``resume: true``
continues from the newest of them.  StepLR (``lr_step_size`` epochs, ``lr_gamma``) runs at each epoch end.  With
``train_set_dynamic_mixing: true`` the training set is a dynamic-mixing set instead (``speech.scp``, ``noise.scp``,
optional ``rir.scp``; mixing.py): the workers read speech, noise and RIRs, and mixing.simulate makes a new noisy / clean
pair per utterance and epoch on the GPU, with the parameters of the optional ``dynamic_mixing:`` YAML mapping; validation
stays a pre-simulated set.  With ``train_set_path: none`` the run trains ``max_steps``
steps on synthetic (clean, noisy) pairs of the dataset contract -- (clean (B,1,T), noisy (B,1,T), fs int32 scalar,
lengths (B,) int32), one fs per batch (dataset.py:417,441) -- and ``save: true`` writes ``last-step<N>.ckpt``.
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


def _configure(model, cfg, flowse):
    if flowse:
        return model.configure_optimizers(precision=getattr(cfg, "train_precision", "fp16"), cuda_graph=True)
    return model.configure_optimizers()


def fit_flowse(model, batches, cfg, rank=0, log_every=10, out_dir=None):
    """FlowSEModel training loop: FlowSETrainer steps (fp16 tensor-core blocks by default, CUDA-graph replay); at the
    end rank 0 writes ``last-step<N>.ckpt`` with the EMA state (``trainer.sync_ema()`` first)."""
    from .checkpoint import save_checkpoint
    trainer = _configure(model, cfg, True)
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


# ------------------------------------------------------------------------------------------------ corpus training
def val_reduce(records, rates, device, flowse=False):
    """records: (loss, sisnr, B, fs) of this rank's validation batches.  ONE all-reduce of (sum loss*B, sum B, sum
    SI-SNR*B, per-rate SI-SNR*B and B) -> means over the utterances of all ranks: what one process computes over the
    same batches.  SE logs val_loss, val_sisnr and val_sisnr_<fs> (d_model.py:84-87), FlowSE val_loss."""
    import torch.distributed as dist
    sums = torch.zeros(3 + 2 * len(rates), dtype=torch.float64, device=device)
    for loss, sisnr, B, fs in records:
        j = 3 + 2 * rates.index(int(fs))
        sums[0] += loss.double() * B
        sums[1] += B
        sums[2] += sisnr.double() * B
        sums[j] += sisnr.double() * B
        sums[j + 1] += B
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    v = sums.tolist()
    out = {"val_loss": v[0] / max(v[1], 1)}
    if not flowse:
        out["val_sisnr"] = v[2] / max(v[1], 1)
        for i, fs in enumerate(rates):
            if v[4 + 2 * i] > 0:
                out[f"val_sisnr_{fs}"] = v[3 + 2 * i] / v[4 + 2 * i]
    return out


def validate(model, trainer, corpus, cfg, rank, world, dev, flowse):
    """One pass over this rank's validation batches (rank-strided) with the no-grad loss path, reduced by val_reduce.
    FlowSE draws t and z from a generator re-seeded at every pass, so that passes compare."""
    from . import data as D
    from .training import flowse_forward_step
    g = torch.Generator(device=dev).manual_seed(int(cfg.seed))
    batches = D.valid_batches(corpus, cfg.batch_size, int(cfg.max_duration), rank, world)
    loader = D.make_loader(corpus, batches, int(cfg.max_duration), False, cfg.num_worker)
    records = []
    with torch.no_grad():
        for clean, noisy, fs, lens in D.prefetch_to_device(loader, dev):
            B, fs = clean.shape[0], int(fs)
            if flowse:
                n_fft, hop = model._dims(fs)
                t = torch.clamp((1 - torch.rand(B, generator=g, device=dev)) * (model.T_rev - model.t_eps) + model.t_eps,
                                max=model.T_rev)
                z = torch.randn(B, 1 + clean.shape[-1] // hop, n_fft // 2 + 1, dtype=torch.complex64, generator=g, device=dev)
                loss, _ = flowse_forward_step(model, noisy, clean, lens, fs, t=t, z=z, blstm_fn=trainer.block_fn)
                sisnr = torch.zeros((), device=dev)
            else:
                loss, sisnr = trainer.loss(noisy, clean, lens, fs)
            records.append((loss, sisnr, B, fs))
    return val_reduce(records, sorted(set(corpus.rates)), dev, flowse)


def fit_corpus(model, cfg, rank, world, dev, flowse, out_dir, log_every=10):
    """Epochs over the set of ``train_set_path`` (pre-simulated pairs, or dynamic mixing) with periodic validation, top-k
    checkpoints and resume.
    -> {"global_step", "epoch", "val": [logged dicts with "step" and "epoch"], "checkpoints": [paths kept]}."""
    import warnings
    from . import data as D
    from . import runtime as R
    from .checkpoint import load_checkpoint, save_checkpoint
    from . import mixing as M
    mixing = bool(cfg.train_set_dynamic_mixing)
    if mixing and not M.is_mix_set(cfg.train_set_path):
        raise NotImplementedError(f"{cfg.train_set_path}: dynamic mixing reads a set of speech.scp + noise.scp (+ optional "
                                  "rir.scp); a pre-simulated set (wav.scp + spk1.scp) needs train_set_dynamic_mixing: false")
    mix_params = M.mix_params(cfg) if mixing else None
    if rank == 0 and getattr(cfg, "use_high_pass", False):
        print(f"note: use_high_pass is not applied by {'dynamic mixing' if mixing else 'the pre-simulated corpus loader'}",
              flush=True)
    max_len = int(cfg.max_duration)
    train = M.MixCorpus(cfg.train_set_path) if mixing else D.PairCorpus(cfg.train_set_path)
    valid = D.PairCorpus(cfg.valid_set_path) if cfg.valid_set_path != "none" else None
    trainer = _configure(model, cfg, flowse)
    epoch, global_step, skip, last_val = 0, 0, 0, -1
    ckpt_path = D.newest_checkpoint(out_dir) if cfg.resume else None
    if ckpt_path is not None:
        sd, _, raw = load_checkpoint(ckpt_path)
        model.load_state_dict(sd)
        R.invalidate_packed()
        state = raw.get("b200_trainer")
        if state is None:
            warnings.warn(f"{ckpt_path} has no b200_trainer state: weights restored, optimizer state starts afresh")
            if flowse and raw.get("ema") is not None:
                model.on_load_checkpoint(raw)
                trainer.load_ema_from_model()
        else:
            trainer.load_state_dict(state)
            epoch, global_step, skip = int(state["epoch"]), int(state["global_step"]), int(state["batches_in_epoch"])
            last_val = global_step                       # the checkpoint was written by the validation at that step
        if rank == 0:
            print(f"resumed from {ckpt_path}: epoch {epoch}, step {global_step}", flush=True)
    model.epoch_ = epoch
    topk = D.TopK(out_dir, cfg.save_top_k) if rank == 0 else None
    max_steps = getattr(cfg, "max_steps", None)
    history = {"val": [], "global_step": global_step}

    def run_validation(done_in_epoch, label_epoch):
        """label_epoch: the epoch the file name and ``epoch`` carry (the last one trained); the trainer state keeps the
        position to resume from (epoch, batches consumed in it)."""
        if flowse:                                 # validate the EMA weights the checkpoint ships, as eval() does
            trainer.sync_ema()
            model.eval()
        try:
            logged = validate(model, trainer, valid, cfg, rank, world, dev, flowse)
        finally:
            if flowse:
                model.train()
                model.ema.collected_params = None
        logged.update(step=global_step, epoch=label_epoch)
        history["val"].append(logged)
        if rank == 0:
            print(f"val step {global_step}: " + " ".join(f"{k}={v!r}" for k, v in logged.items()
                                                         if k not in ("step", "epoch")), flush=True)
            state = dict(trainer.state_dict(), epoch=epoch, global_step=global_step, batches_in_epoch=done_in_epoch)

            def save(path):
                save_checkpoint(path, model, cfg, global_step=global_step, epoch=label_epoch,
                                ema=model.ema.state_dict() if flowse else None, extra={"b200_trainer": state})
            topk.update(logged["val_loss"], label_epoch, global_step, save)

    done = skip
    stop = bool(max_steps) and global_step >= int(max_steps)
    while epoch < int(cfg.num_train_epochs) and not stop:
        batches, dropped = D.train_batches(train, cfg.batch_size, max_len, rank, world, epoch, cfg.seed)
        if rank == 0 and skip == 0:
            print(f"epoch {epoch}: {len(batches)} batches per rank, {dropped} utterances dropped (uneven tail)", flush=True)
        if mixing:
            loader = M.make_loader(train, batches[skip:], max_len, mix_params, cfg.num_worker, cfg.seed, epoch)
        else:
            loader = D.make_loader(train, batches[skip:], max_len, True, cfg.num_worker, seed=cfg.seed, epoch=epoch)
        done = skip
        for batch in D.prefetch_to_device(loader, dev):
            clean, noisy, fs, lens = M.simulate(batch, dev) if mixing else batch
            loss, _ = trainer.step(noisy, clean, lens, fs)
            done += 1
            global_step += 1
            if rank == 0 and global_step % log_every == 0:
                print(f"step {global_step}: train_loss={float(loss):.4g}", flush=True)
            if valid is not None and global_step % max(1, int(cfg.val_check_interval)) == 0:
                run_validation(done, epoch)
                last_val = global_step
            if max_steps and global_step >= int(max_steps):
                stop = True
                break
        skip = 0
        if not stop:
            model.on_train_epoch_end()
            epoch += 1
    if valid is not None and last_val != global_step:
        if stop:
            run_validation(done, epoch)
        else:                                      # every epoch ran: name the file after the last one
            run_validation(0, max(epoch - 1, 0))
    history.update(global_step=global_step, epoch=epoch,
                   checkpoints=[p for _, p in topk.kept] if topk is not None else [])
    return history


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
    corpus = cfg.train_set_path != "none"
    if cfg.init_from != "none":
        sd = torch.load(cfg.init_from, map_location="cpu", weights_only=False)
        model.load_state_dict(sd.get("state_dict", sd))
    model.to(dev)
    if world > 1:                                                    # DDP broadcasts rank 0's parameters at wrap time
        for p in model.parameters():
            dist.broadcast(p.data, 0)
    out_dir = os.path.join("exp", cfg.train_tag, cfg.train_name, f"version_{cfg.train_version}", "checkpoints")
    result = None
    if corpus:
        result = fit_corpus(model, cfg, rank, world, dev, flowse, out_dir)
    else:
        steps = int(getattr(cfg, "max_steps", 20))
        (fit_flowse if flowse else fit)(model, synthetic_batches(cfg, rank, world, steps, dev), cfg, rank,
                                        out_dir=out_dir if getattr(cfg, "save", False) else None)
    if world > 1:
        dist.destroy_process_group()
    return result


if __name__ == "__main__":
    main(sys.argv[1:])
