"""Batched inference front-end — mirrors ``baseline_code/inference.py`` (reference inference.py:26-112: same flags,
same scp in / ``inf.scp`` + ``wav/<uid>.wav`` out, ``SEModel`` first with the ``FlowSEModel`` fallback (:30-33,
:54-58), peak-normalise to 0.9 (:60), PCM-16 WAV (:62)) but groups utterances into (fs, length) buckets and runs them
as batches, sharded over ranks when launched under torchrun (SURVEY.md §8f.1).

Parity with the reference's batch-1 loop: by default only utterances of EQUAL length share a batch, so every output
equals the batch-1 output (``--max_pad_ratio`` > 0 allows right-zero-padded batches, whose outputs then depend on the
padding like the training collate's do, SURVEY.md §8g.1).  Audio is read lazily, one batch at a time: only the WAV
headers are touched up front.  WAV I/O uses scipy.io.wavfile (soundfile is not a dependency of this package)."""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch

from .d_model import SEModel
from .data import _probe_wav, _read_wav, read_scp
from .flow_model import FlowSEModel
from .pipeline import StreamedEnhancer
from .sharding import shard_utterances


def _write_wav(path, x, sr):
    from scipy.io import wavfile
    wavfile.write(path, sr, np.clip(np.round(x * 32767.0), -32768, 32767).astype(np.int16))


def load_model(ckpt_path, device, precision=None):
    """inference.py:30-33: try SEModel, fall back to FlowSEModel; ``eval()`` swaps the FlowSE EMA weights in (:34)."""
    try:
        model = SEModel.load_from_checkpoint(ckpt_path, map_location=device, precision=precision)
    except KeyError:
        model = FlowSEModel.load_from_checkpoint(ckpt_path, map_location=device)
    return model.eval()


def _peak_normalise(y):
    return y / y.abs().max().clamp_min(1e-12) * 0.9                              # inference.py:60


def main(args):
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    dev = torch.device(args.device, int(os.environ.get("LOCAL_RANK", 0))) if args.device == "cuda" else torch.device(args.device)
    model = load_model(args.ckpt_path, dev, args.precision)
    utts = read_scp(args.input_scp)
    os.makedirs(os.path.join(args.output_dir, "wav"), exist_ok=True)
    meta = [_probe_wav(p) for _, p in utts]
    batches = shard_utterances([n for n, _ in meta], [sr for _, sr in meta], rank, world, args.max_batch,
                               args.max_pad_ratio)

    def host_batches():
        for fs, idx in batches:                                                 # audio is read here, batch by batch
            lens = torch.tensor([meta[i][0] for i in idx], dtype=torch.int32)
            batch = torch.zeros(len(idx), int(lens.max()), dtype=torch.float32).pin_memory()
            for row, i in enumerate(idx):
                batch[row, : lens[row]] = torch.from_numpy(_read_wav(utts[i][1])[0])   # right zero-pad (dataset.py:404-441)
            yield batch, lens, fs

    with open(os.path.join(args.output_dir, f"inf.{rank}.scp" if world > 1 else "inf.scp"), "w") as f:
        def emit(idx, enhanced, lens, fs):
            for row, i in enumerate(idx):
                y = _peak_normalise(enhanced[row, : lens[row]].clone())
                out = os.path.join(args.output_dir, "wav", f"{utts[i][0]}.wav")
                _write_wav(out, y.numpy(), fs)
                print(f"{utts[i][0]} {out}", file=f)

        if isinstance(model, SEModel):
            # H2D of the next batch and D2H of the previous one overlap the current batch's kernels
            for (fs, idx), (enhanced, lens, _) in zip(batches, StreamedEnhancer(model.se_model).run(host_batches())):
                emit(idx, enhanced, lens, fs)
        else:                                                                   # FlowSEModel.enhance (inference.py:58)
            for (fs, idx), (batch, lens, _) in zip(batches, host_batches()):
                enhanced = model.enhance(batch.to(dev, non_blocking=True), fs, lens, N=args.nfe)
                emit(idx, enhanced.cpu(), lens, fs)
    print("done")


def build_parser():
    p = argparse.ArgumentParser()
    p.add_argument("--input_scp", type=str, required=True)
    p.add_argument("--output_dir", type=str, default="./tmp/se")
    p.add_argument("--ckpt_path", type=str, default="./tmp/se")
    p.add_argument("--device", type=str, default="cuda")
    p.add_argument("--precision", type=str, default=None)
    p.add_argument("--max_batch", type=int, default=64)
    p.add_argument("--max_pad_ratio", type=float, default=0.0,
                   help="0 = batch only equal-length utterances (bit-for-bit the batch-1 result of each)")
    p.add_argument("--nfe", type=int, default=15, help="FlowSE Euler steps (flow_model.py:189 default)")
    return p


if __name__ == "__main__":
    main(build_parser().parse_args())
