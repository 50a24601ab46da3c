"""Score enhanced speech against its clean reference on the GPU: ESTOI and SDR, the intrusive metrics of the reference's
``evaluation_metrics/calculate_intrusive_se_metrics.py`` that can be restated (metrics.py, csrc/metrics.cu).

    python -m urgent2026_challenge_track1_b200.evaluate --ref_scp clean.scp --inf_scp <out>/inf.scp --output_dir <dir>

Both lists hold ``uid path`` lines.  Utterances are paired by uid in the order of ``--inf_scp``; a uid missing from
``--ref_scp``, or a pair whose rate or length differs, is an error that names the uid, raised before any audio is read.
WAVs are read like inference.py reads them (first channel, PCM scaled by 1/32768), one same-rate batch at a time.

Written to ``--output_dir``, following the reference's ``<METRIC>.scp`` + ``RESULTS.txt`` convention (this layout has
not been compared file for file with the reference's evaluation scripts):
    ESTOI.scp    ``uid value`` per utterance, in --inf_scp order
    SDR.scp      the same for SDR (dB)
    RESULTS.txt  ``ESTOI: 0.1234`` and ``SDR: 12.3456``: the nanmean over the utterances, 4 decimals

PESQ is not offered: its ITU-T P.862 implementation cannot be restated here.  The scores differ from pystoi /
fast_bss_eval in a few degenerate cases (all-zero signals, too-short input, an extremely ill-conditioned reference); see
the docstring of metrics.py.
"""
from __future__ import annotations

import argparse
import os

import numpy as np
import torch

from . import metrics as MET
from .data import _probe_wav, _read_wav, read_scp
from .sharding import shard_utterances


def pair_scps(ref_scp, inf_scp):
    """-> [(uid, ref_path, inf_path, n_samples, fs)] in inf_scp order, from the WAV headers only."""
    refs = dict(read_scp(ref_scp))
    pairs = []
    for uid, inf_path in read_scp(inf_scp):
        if uid not in refs:
            raise ValueError(f"uid {uid!r} of {inf_scp} is not in {ref_scp}")
        (n_r, fs_r), (n_i, fs_i) = _probe_wav(refs[uid]), _probe_wav(inf_path)
        if fs_r != fs_i:
            raise ValueError(f"uid {uid!r}: the reference is {fs_r} Hz, the estimate {fs_i} Hz")
        if n_r != n_i:
            raise ValueError(f"uid {uid!r}: the reference has {n_r} samples, the estimate {n_i}")
        pairs.append((uid, refs[uid], inf_path, n_r, fs_r))
    return pairs


def score(pairs, device, max_batch=64):
    """-> (estoi, sdr) float64 arrays in the order of pairs."""
    est = np.full(len(pairs), np.nan)
    sdr = np.full(len(pairs), np.nan)
    # scores do not depend on padding, so any length mix may share a batch
    batches = shard_utterances([p[3] for p in pairs], [p[4] for p in pairs], 0, 1, max_batch, max_pad_ratio=1.0)
    for fs, idx in batches:
        lens = torch.tensor([pairs[i][3] for i in idx], dtype=torch.int32)
        T = int(lens.max())
        ref = torch.zeros(len(idx), T, dtype=torch.float32)
        inf = torch.zeros(len(idx), T, dtype=torch.float32)
        for row, i in enumerate(idx):
            for dst, path in ((ref, pairs[i][1]), (inf, pairs[i][2])):
                x, sr = _read_wav(path)
                if sr != fs or x.shape[0] != pairs[i][3]:
                    raise ValueError(f"uid {pairs[i][0]!r}: {path} changed since the lists were read")
                dst[row, : x.shape[0]] = torch.from_numpy(x)
        ref, inf = ref.to(device), inf.to(device)
        lens_d = lens.to(device)
        e = MET.estoi(ref, inf, lens_d, fs).cpu().numpy()
        s = MET.sdr(ref, inf, lens_d).cpu().numpy()
        est[idx], sdr[idx] = e, s
    return est, sdr


def main(args):
    pairs = pair_scps(args.ref_scp, args.inf_scp)
    dev = torch.device(args.device)
    est, sdr = score(pairs, dev, args.max_batch)
    os.makedirs(args.output_dir, exist_ok=True)
    for name, vals in (("ESTOI", est), ("SDR", sdr)):
        with open(os.path.join(args.output_dir, f"{name}.scp"), "w") as f:
            for (uid, *_), v in zip(pairs, vals):
                print(f"{uid} {float(v)!r}", file=f)
    with open(os.path.join(args.output_dir, "RESULTS.txt"), "w") as f:
        for name, vals in (("ESTOI", est), ("SDR", sdr)):
            m = float(np.nanmean(vals)) if len(vals) and not np.isnan(vals).all() else float("nan")
            print(f"{name}: {m:.4f}", file=f)
    print(open(os.path.join(args.output_dir, "RESULTS.txt")).read(), end="")


def build_parser():
    p = argparse.ArgumentParser(description="ESTOI and SDR of enhanced speech against its reference, on the GPU")
    p.add_argument("--ref_scp", type=str, required=True, help="clean references: uid path")
    p.add_argument("--inf_scp", type=str, required=True, help="estimates to score, e.g. inference.py's inf.scp")
    p.add_argument("--output_dir", type=str, required=True)
    p.add_argument("--device", type=str, default="cuda")
    p.add_argument("--max_batch", type=int, default=64)
    return p


if __name__ == "__main__":
    main(build_parser().parse_args())
