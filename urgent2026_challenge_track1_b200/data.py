"""Corpus reader, sampler and collate of the training loop: pre-simulated (noisy, clean) pairs listed in Kaldi-style scp
files, served in the dataset contract of SURVEY.md §2 row 9 -- (clean (B,1,T), noisy (B,1,T), fs int32 scalar,
lengths (B,) int32), one fs per batch (reference dataset.py:404-441).

A set is a directory holding ``wav.scp`` (noisy input) and ``spk1.scp`` (clean target), one ``uid path`` per line, the
same uids in both, in any order.  Audio is WAV as ``scipy.io.wavfile`` reads it; only the headers are read when a set is
opened, the samples batch by batch in the DataLoader workers (which never touch CUDA).

Batches follow the reference's GroupedBatchSampler (dataset.py:338-401): one sample rate per batch, utterances sorted by
(fs, length) and cut into batches of ``batch_size`` within each rate, the batch order shuffled per epoch from
``seed + epoch``, rank r taking batches r, r + world, ...  Every rank must take the same number of training steps (one
gradient allreduce per step), so the batches that do not divide evenly over the ranks are dropped for that epoch.
"""
from __future__ import annotations

import glob
import os
import re
import zlib

import numpy as np
import torch


# ------------------------------------------------------------------------------------------------ WAV + scp
def _to_float(x):
    if x.dtype.kind == "i":
        x = x.astype(np.float32) / float(np.iinfo(x.dtype).max + 1)
    elif x.dtype.kind == "u":
        x = (x.astype(np.float32) - 128.0) / 128.0
    if x.ndim > 1:
        x = x[:, 0]
    return np.ascontiguousarray(x, dtype=np.float32)


def _read_wav(path):
    from scipy.io import wavfile
    sr, x = wavfile.read(path)
    return _to_float(x), int(sr)


def _probe_wav(path):
    """(n_samples, sample_rate) from the header only (memory-mapped read: no sample is touched)."""
    from scipy.io import wavfile
    sr, x = wavfile.read(path, mmap=True)
    return int(x.shape[0]), int(sr)


def read_scp(path):
    utts = []
    with open(path) as f:
        for line in f:
            if line.strip():
                uid, wav = line.strip().split()
                utts.append((uid, wav))
    return utts


class PairCorpus:
    """A set of pre-simulated pairs: ``uids``, ``lengths`` and ``rates`` from the WAV headers (sorted by uid), and the
    noisy / clean paths of each uid.  Raises with the name of the missing file or the offending uid."""

    def __init__(self, root):
        lists = {}
        for name in ("wav.scp", "spk1.scp"):
            path = os.path.join(root, name)
            if not os.path.isfile(path):
                raise FileNotFoundError(f"{root}: missing {name} (a set holds wav.scp = noisy and spk1.scp = clean)")
            entries = read_scp(path)
            d = dict(entries)
            if len(d) != len(entries):
                seen = set()
                dup = next(u for u, _ in entries if u in seen or seen.add(u))
                raise ValueError(f"{path}: uid {dup!r} listed twice")
            lists[name] = d
        noisy, clean = lists["wav.scp"], lists["spk1.scp"]
        for a, b, an, bn in ((noisy, clean, "wav.scp", "spk1.scp"), (clean, noisy, "spk1.scp", "wav.scp")):
            extra = sorted(set(a) - set(b))
            if extra:
                raise ValueError(f"{root}: uid {extra[0]!r} is in {an} but not in {bn}")
        self.root = root
        self.uids = sorted(noisy)
        self.noisy = [noisy[u] for u in self.uids]
        self.clean = [clean[u] for u in self.uids]
        self.lengths, self.rates = [], []
        for u, pn, pc in zip(self.uids, self.noisy, self.clean):
            (nn, rn), (nc, rc) = _probe(u, pn), _probe(u, pc)
            if rn != rc:
                raise ValueError(f"uid {u!r}: noisy is {rn} Hz, clean is {rc} Hz")
            if nn != nc:
                raise ValueError(f"uid {u!r}: noisy has {nn} samples, clean has {nc}")
            self.lengths.append(nn)
            self.rates.append(rn)

    def __len__(self):
        return len(self.uids)


def _probe(uid, path):
    try:
        return _probe_wav(path)
    except Exception as e:                                  # scipy raises ValueError / OSError for non-WAV data
        raise ValueError(f"uid {uid!r}: cannot read {path} as WAV ({e})") from e


# ------------------------------------------------------------------------------------------------ crop
def crop_offset(seed, epoch, uid, n, max_len):
    """Start of the training window of an utterance of n > max_len samples: a function of (seed, epoch, uid) only, so a
    resumed run crops the same way.  crc32, not hash(): Python salts str hashes per process."""
    rng = np.random.default_rng([int(seed) & 0xFFFFFFFF, int(epoch), zlib.crc32(uid.encode())])
    return int(rng.integers(0, n - max_len + 1))


# ------------------------------------------------------------------------------------------------ sampler
def _batches_by_rate(corpus, batch_size, max_len):
    """Utterances sorted by (fs, cropped length, index), cut into batches of batch_size within each rate."""
    order = sorted(range(len(corpus)), key=lambda i: (corpus.rates[i], min(corpus.lengths[i], max_len), i))
    out, cur = [], []
    for i in order:
        if cur and (len(cur) == batch_size or corpus.rates[cur[0]] != corpus.rates[i]):
            out.append(cur)
            cur = []
        cur.append(i)
    if cur:
        out.append(cur)
    return out


def train_batches(corpus, batch_size, max_len, rank, world, epoch, seed):
    """-> (batches of this rank for this epoch, number of utterances dropped).  Every rank gets len(all) // world
    batches; the shuffled order's tail that does not divide evenly is dropped (a different one every epoch)."""
    allb = _batches_by_rate(corpus, batch_size, max_len)
    g = torch.Generator().manual_seed(int(seed) + int(epoch))
    perm = torch.randperm(len(allb), generator=g).tolist()
    keep = (len(allb) // world) * world
    dropped = sum(len(allb[j]) for j in perm[keep:])
    return [allb[j] for j in perm[rank:keep:world]], dropped


def valid_batches(corpus, batch_size, max_len, rank, world):
    """Validation batches of this rank: formed like the training ones, not shuffled, rank-strided, nothing dropped (the
    validation reduction is one collective after the pass, so the ranks may run different numbers of batches)."""
    return _batches_by_rate(corpus, batch_size, max_len)[rank::world]


# ------------------------------------------------------------------------------------------------ collate + loading
def collate(corpus, idx, max_len, train, seed=0, epoch=0):
    """Reads the pairs of one batch and right-zero-pads them to its longest (cropped) utterance (dataset.py:404-441).
    Training crops an utterance longer than max_len to a window at crop_offset(); validation keeps its first max_len
    samples.  -> (clean (B,1,T), noisy (B,1,T), fs int32 scalar, lengths (B,) int32), all on the CPU."""
    fs = corpus.rates[idx[0]]
    lens = [min(corpus.lengths[i], max_len) for i in idx]
    T = max(lens)
    clean = torch.zeros(len(idx), 1, T, dtype=torch.float32)
    noisy = torch.zeros(len(idx), 1, T, dtype=torch.float32)
    for row, i in enumerate(idx):
        n = corpus.lengths[i]
        off = crop_offset(seed, epoch, corpus.uids[i], n, max_len) if (train and n > max_len) else 0
        for dst, path in ((noisy, corpus.noisy[i]), (clean, corpus.clean[i])):
            x, sr = _read_wav(path)
            if sr != fs or x.shape[0] != n:
                raise ValueError(f"uid {corpus.uids[i]!r}: {path} changed since the set was opened")
            dst[row, 0, : lens[row]] = torch.from_numpy(x[off: off + lens[row]])
    return clean, noisy, torch.tensor(fs, dtype=torch.int32), torch.tensor(lens, dtype=torch.int32)


class BatchDataset(torch.utils.data.Dataset):
    """One item = one collated batch (DataLoader with batch_size=None): the workers read and pad, nothing else."""

    def __init__(self, corpus, batches, max_len, train, seed=0, epoch=0):
        self.corpus, self.batches, self.max_len, self.train, self.seed, self.epoch = corpus, batches, max_len, train, seed, epoch

    def __len__(self):
        return len(self.batches)

    def __getitem__(self, i):
        return collate(self.corpus, self.batches[i], self.max_len, self.train, self.seed, self.epoch)


def make_loader(corpus, batches, max_len, train, num_workers, seed=0, epoch=0):
    return torch.utils.data.DataLoader(BatchDataset(corpus, batches, max_len, train, seed, epoch), batch_size=None,
                                       shuffle=False, num_workers=int(num_workers), pin_memory=torch.cuda.is_available())


def prefetch_to_device(batches, device):
    """Copies the leading tensors of batch i+1 (all but the last two entries: clean / noisy of a pair batch, the signals
    of a mixing batch) to the device on a side stream while the caller works on batch i (the pattern of
    pipeline.StreamedEnhancer).  The last two entries (fs and lengths, or fs and the mixing parameters) stay on the host:
    the caller reads them there."""
    copy = torch.cuda.Stream(device)
    cur = torch.cuda.current_stream(device)

    def submit(b):
        *lead, fs, tail = b
        with torch.cuda.stream(copy):
            copy.wait_stream(cur)               # blocks the allocator may hand out could still be read by queued work
            lead = [t.to(device, non_blocking=True) for t in lead]
            ev = torch.cuda.Event()
            ev.record(copy)
        return (*lead, fs, tail), ev

    pending = None
    for b in batches:
        nxt = submit(b)
        if pending is not None:
            yield _ready(pending, cur)
        pending = nxt
    if pending is not None:
        yield _ready(pending, cur)


def _ready(pending, cur):
    b, ev = pending
    cur.wait_event(ev)
    for t in b[:-2]:
        t.record_stream(cur)
    return b


# ------------------------------------------------------------------------------------------------ checkpoint files
_VAL_LOSS = re.compile(r"val_loss=([-+0-9.eE]+|nan|inf)\.ckpt$")


def checkpoint_name(epoch, step, val_loss):
    """Lightning's rendering of ``filename="best_{epoch:02d}-{step:06d}-{val_loss:.3f}"`` (reference train_se.py)."""
    return f"best_epoch={int(epoch):02d}-step={int(step):06d}-val_loss={float(val_loss):.3f}.ckpt"


def newest_checkpoint(dirpath):
    """The newest ``*-val_loss*.ckpt`` of dirpath by mtime (reference train_se.py:67-72), or None."""
    files = glob.glob(os.path.join(dirpath, "*-val_loss*.ckpt"))
    return max(files, key=os.path.getmtime) if files else None


class TopK:
    """The best save_top_k checkpoints by val_loss (mode min) in dirpath, files that fall out deleted.  Files already
    there (a resumed run) take part.  save_top_k = -1 keeps every file, 0 none."""

    def __init__(self, dirpath, k):
        self.dir, self.k = dirpath, int(k)
        self.kept = []                                                  # (val_loss, path)
        for p in glob.glob(os.path.join(dirpath, "best_*-val_loss=*.ckpt")):
            m = _VAL_LOSS.search(os.path.basename(p))
            if m:
                self.kept.append((float(m.group(1)), p))

    def update(self, val_loss, epoch, step, save):
        """save(path) writes the checkpoint; called only when val_loss enters the top k.  -> the path or None."""
        val_loss = float(val_loss)
        if self.k == 0 or not np.isfinite(val_loss):
            return None
        if self.k > 0 and len(self.kept) >= self.k and val_loss >= max(v for v, _ in self.kept):
            return None
        os.makedirs(self.dir, exist_ok=True)
        path = os.path.join(self.dir, checkpoint_name(epoch, step, val_loss))
        save(path)
        self.kept = [(v, p) for v, p in self.kept if p != path] + [(val_loss, path)]
        if self.k > 0:
            self.kept.sort(key=lambda e: e[0])
            for _, p in self.kept[self.k:]:
                if os.path.exists(p):
                    os.remove(p)
            self.kept = self.kept[: self.k]
        return path
