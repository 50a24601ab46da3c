"""Corpus reader, crop, sampler, collate, validation reduction, checkpoint bookkeeping and trainer state of the
corpus-fed training loop (data.py, train_se.py, training.SETrainer), on small WAV sets written into tmp_path."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest
import torch

from conftest import ROOT
from urgent2026_challenge_track1_b200 import data as D
from urgent2026_challenge_track1_b200.synth import synth_pair

RATES = (8000, 16000, 48000)


def _wav(path, x, fs):
    from scipy.io import wavfile
    wavfile.write(str(path), fs, np.asarray(x, dtype=np.float32))


def make_set(root, n_per_rate=5, rates=RATES, seed=0):
    """n_per_rate utterances per rate, ragged lengths between 0.25 s and 0.6 s; the scp lines in shuffled order."""
    root.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(seed)
    lines_n, lines_c, meta = [], [], {}
    for fs in rates:
        for i in range(n_per_rate):
            uid = f"u{fs}_{i}"
            n = int(rng.integers(fs // 4, fs * 6 // 10))
            clean, noisy = synth_pair(1, n, fs, seed=seed * 1000 + i + fs)
            _wav(root / f"{uid}_n.wav", noisy[0].numpy(), fs)
            _wav(root / f"{uid}_c.wav", clean[0].numpy(), fs)
            lines_n.append(f"{uid} {root / f'{uid}_n.wav'}")
            lines_c.append(f"{uid} {root / f'{uid}_c.wav'}")
            meta[uid] = (n, fs)
    rng.shuffle(lines_n)
    rng.shuffle(lines_c)
    (root / "wav.scp").write_text("\n".join(lines_n) + "\n")
    (root / "spk1.scp").write_text("\n".join(lines_c) + "\n")
    return meta


@pytest.fixture(scope="module")
def corpus(tmp_path_factory):
    root = tmp_path_factory.mktemp("set")
    meta = make_set(root)
    return D.PairCorpus(str(root)), meta


def test_reader_reads_headers(corpus):
    c, meta = corpus
    assert sorted(c.uids) == sorted(meta)
    for u, n, fs in zip(c.uids, c.lengths, c.rates):
        assert (n, fs) == meta[u]


def test_reader_errors(tmp_path):
    root = tmp_path / "s"
    make_set(root, n_per_rate=2, rates=(16000,))
    os.rename(root / "spk1.scp", root / "spk1.bak")
    with pytest.raises(FileNotFoundError, match="spk1.scp"):
        D.PairCorpus(str(root))
    lines = (root / "spk1.bak").read_text().splitlines()
    (root / "spk1.scp").write_text("\n".join(lines[:1]) + "\n")             # one uid in wav.scp only
    missing = [l.split()[0] for l in (root / "wav.scp").read_text().splitlines() if l.split()[0] != lines[0].split()[0]][0]
    with pytest.raises(ValueError, match=missing):
        D.PairCorpus(str(root))
    (root / "spk1.scp").write_text("\n".join(lines) + "\n")
    D.PairCorpus(str(root))
    uid, cpath = lines[0].split()
    x, _ = D._read_wav(cpath)
    _wav(cpath, x, 8000)                                                      # rate mismatch inside the pair
    with pytest.raises(ValueError, match=f"{uid}.*Hz"):
        D.PairCorpus(str(root))
    _wav(cpath, x[:-10], 16000)                                               # length mismatch
    with pytest.raises(ValueError, match=f"{uid}.*samples"):
        D.PairCorpus(str(root))
    with open(cpath, "wb") as f:                                              # not a WAV file
        f.write(b"this is not a RIFF file" * 10)
    with pytest.raises(ValueError, match=f"{uid}.*WAV"):
        D.PairCorpus(str(root))


def test_crops_are_deterministic_and_shared_by_the_pair(corpus):
    c, _ = corpus
    max_len = 3000
    long = [i for i in range(len(c)) if c.lengths[i] > max_len]
    assert long
    for i in long:
        u, n = c.uids[i], c.lengths[i]
        o = D.crop_offset(7, 3, u, n, max_len)
        assert o == D.crop_offset(7, 3, u, n, max_len) and 0 <= o <= n - max_len
    offs = {(e, c.uids[i]): D.crop_offset(7, e, c.uids[i], c.lengths[i], max_len) for e in range(3) for i in long}
    assert len(set(offs.values())) > 1
    for i in long:
        clean, noisy, fs, lens = D.collate(c, [i], max_len, train=True, seed=7, epoch=2)
        o = D.crop_offset(7, 2, c.uids[i], c.lengths[i], max_len)
        xn, _ = D._read_wav(c.noisy[i])
        xc, _ = D._read_wav(c.clean[i])
        assert clean.shape == (1, 1, max_len) and int(lens[0]) == max_len
        assert torch.equal(noisy[0, 0], torch.from_numpy(xn[o:o + max_len]))
        assert torch.equal(clean[0, 0], torch.from_numpy(xc[o:o + max_len]))
        vc, vn, _, _ = D.collate(c, [i], max_len, train=False)                # validation: cut at the start
        assert torch.equal(vn[0, 0], torch.from_numpy(xn[:max_len]))


def test_batches_have_one_rate_and_collate_zero_pads(corpus):
    c, _ = corpus
    max_len = 6000
    batches, dropped = D.train_batches(c, 2, max_len, 0, 1, 0, 1)
    assert dropped == 0 and sorted(i for b in batches for i in b) == list(range(len(c)))
    for idx in batches:
        assert len({c.rates[i] for i in idx}) == 1
        clean, noisy, fs, lens = D.collate(c, idx, max_len, train=True, seed=1, epoch=0)
        assert fs.dtype == torch.int32 and fs.dim() == 0 and int(fs) == c.rates[idx[0]]
        assert lens.dtype == torch.int32 and lens.tolist() == [min(c.lengths[i], max_len) for i in idx]
        assert clean.shape == noisy.shape == (len(idx), 1, int(lens.max()))
        for row in range(len(idx)):
            assert float(noisy[row, 0, lens[row]:].abs().sum()) == 0.0 and float(clean[row, 0, lens[row]:].abs().sum()) == 0.0
            assert float(noisy[row, 0, : lens[row]].abs().sum()) > 0.0
    # shuffled per epoch from seed + epoch
    assert D.train_batches(c, 2, max_len, 0, 1, 0, 1)[0] == batches
    assert D.train_batches(c, 2, max_len, 0, 1, 1, 1)[0] != batches


@pytest.mark.parametrize("world", [1, 2, 3])
def test_ranks_take_equal_disjoint_shares(corpus, world):
    c, _ = corpus
    for epoch in range(3):
        per_rank = [D.train_batches(c, 2, 6000, r, world, epoch, 5) for r in range(world)]
        counts = {len(b) for b, _ in per_rank}
        assert len(counts) == 1
        drops = {d for _, d in per_rank}
        assert len(drops) == 1
        sets = [set(i for b in bs for i in b) for bs, _ in per_rank]
        assert sum(len(s) for s in sets) == len(set().union(*sets))          # disjoint
        assert len(set().union(*sets)) + drops.pop() == len(c)
    vb = [D.valid_batches(c, 2, 6000, r, world) for r in range(world)]
    assert sorted(i for bs in vb for b in bs for i in b) == list(range(len(c)))


_VAL_WORKER = r'''
import os, sys, json, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from urgent2026_challenge_track1_b200.train_se import val_reduce
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
recs = [(torch.tensor(0.1 + 0.37 * i, dtype=torch.float32), torch.tensor(3.0 - 0.9 * i), 1 + i % 3, (8000, 16000, 48000)[i % 3])
        for i in range(7)]
out = val_reduce(recs[rank::world], [8000, 16000, 48000], torch.device("cpu"))
json.dump(out, open(os.path.join(sys.argv[2], f"val{rank}.json"), "w"))
dist.destroy_process_group()
'''


def test_validation_reduction_over_two_gloo_ranks_equals_one_process(tmp_path):
    from urgent2026_challenge_track1_b200.train_se import val_reduce
    script = tmp_path / "worker.py"
    script.write_text(_VAL_WORKER)
    import socket
    with socket.socket() as sk:                                                # a free port, not a fixed one
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(tmp_path)], env=dict(env, RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    import json
    got = [json.load(open(tmp_path / f"val{r}.json")) for r in range(2)]
    recs = [(torch.tensor(0.1 + 0.37 * i, dtype=torch.float32), torch.tensor(3.0 - 0.9 * i), 1 + i % 3, (8000, 16000, 48000)[i % 3])
            for i in range(7)]
    one = val_reduce(recs, [8000, 16000, 48000], torch.device("cpu"))
    w = [1 + i % 3 for i in range(7)]
    assert abs(one["val_loss"] - sum(float(r[0]) * b for r, b in zip(recs, w)) / sum(w)) < 1e-12
    assert set(one) == {"val_loss", "val_sisnr", "val_sisnr_8000", "val_sisnr_16000", "val_sisnr_48000"}
    for g in got:
        assert g.keys() == one.keys()
        assert all(abs(g[k] - one[k]) <= 1e-12 * max(1.0, abs(one[k])) for k in one)


def test_top_k_and_resume_file_selection(tmp_path):
    assert D.checkpoint_name(0, 500, 0.1234) == "best_epoch=00-step=000500-val_loss=0.123.ckpt"
    d = tmp_path / "ck"
    saved = []
    topk = D.TopK(str(d), 2)

    def save(p):
        open(p, "w").write("x")
        saved.append(p)
    for step, v in [(1, 0.5), (2, 0.4), (3, 0.6), (4, 0.3), (5, 0.45)]:
        topk.update(v, 0, step, save)
        time.sleep(0.01)
    left = sorted(os.listdir(d))
    assert left == ["best_epoch=00-step=000002-val_loss=0.400.ckpt", "best_epoch=00-step=000004-val_loss=0.300.ckpt"]
    assert len(saved) == 3                                            # 0.6 and 0.45 never entered the top 2
    assert D.newest_checkpoint(str(d)) == str(d / "best_epoch=00-step=000004-val_loss=0.300.ckpt")
    (d / "last.ckpt").write_text("x")                                  # not matched by *-val_loss*.ckpt
    other = d / "epoch=1-val_loss=0.9.ckpt"
    other.write_text("x")
    assert D.newest_checkpoint(str(d)) == str(other)
    again = D.TopK(str(d), 2)                                          # a resumed run picks the kept files up
    assert sorted(v for v, _ in again.kept) == [0.3, 0.4]
    assert again.update(0.35, 1, 6, save) and not (d / "best_epoch=00-step=000002-val_loss=0.400.ckpt").exists()
    assert D.newest_checkpoint(str(tmp_path / "none")) is None


def test_trainer_state_dict_round_trips_bit_exactly():
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.training import SETrainer
    torch.manual_seed(0)
    a = SETrainer(BSRNN_SE(16, 1), lr=3e-4, ema_decay=0.99)
    for t in (a.exp_avg, a.exp_avg_sq, a.ema, a.stats):
        t.copy_(torch.randn(t.shape, dtype=t.dtype))
    a.set_lr(1.2345e-4)
    st = a.state_dict()
    b =SETrainer(BSRNN_SE(16, 1), lr=1e-3, ema_decay=0.99)
    b.load_state_dict(st)
    for name in ("exp_avg", "exp_avg_sq", "ema", "stats"):
        assert torch.equal(getattr(a, name), getattr(b, name)), name
    assert b.lr == a.lr
    with pytest.raises(ValueError):
        SETrainer(BSRNN_SE(16, 2)).load_state_dict(st)


def test_dynamic_mixing_with_a_real_set_is_not_built(corpus):
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.train_se import fit_corpus
    c, _ = corpus
    cfg = Config(train_set_path=c.root, train_set_dynamic_mixing=True)
    with pytest.raises(NotImplementedError, match="train_set_dynamic_mixing: false"):
        fit_corpus(None, cfg, 0, 1, None, False, "unused")


def test_optional_flags_stay_absent_unless_given():
    from urgent2026_challenge_track1_b200.config import Config, config_parser
    cfg = Config(**vars(config_parser([])))
    assert not hasattr(cfg, "train_precision") and not hasattr(cfg, "max_steps")
    cfg = Config(**vars(config_parser(["--train_precision", "fp16", "--max_steps", "7"])))
    assert cfg.train_precision == "fp16" and cfg.max_steps == 7
