"""Corpus-fed training on the GPU: ragged batches through one captured graph, train_se end to end on a WAV set
(validation, top-k checkpoints, the inference CLI on a kept checkpoint), resume, and the FlowSE corpus run."""
import os

import pytest
import torch
import yaml

from conftest import rel_l2
from oracle import restated as R
from test_corpus_cpu import make_set

pytestmark = pytest.mark.gpu


def _tiny_se(width=32, layers=1):
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    torch.manual_seed(0)
    return BSRNN_SE(num_channel=width, num_layer=layers, precision="fp32").cuda()


def test_ragged_batches_replay_one_graph():
    """Batches of one shape with different lengths replay ONE captured graph (lengths are device data of the graph); each
    replay matches an eager step on the same batch, including a batch whose second utterance is half the padded width
    with non-zero samples beyond its length (they must be masked, not read)."""
    from urgent2026_challenge_track1_b200.training import SETrainer
    fs, n = 16000, 8000
    x, clean = R.synth_noisy(2, n, fs, seed=1), R.synth_noisy(2, n, fs, seed=7)
    noisy, cl = x.cuda().view(2, 1, -1), clean.cuda().view(2, 1, -1)
    batches = [(noisy, cl, torch.tensor([n, n - 517], dtype=torch.int32)),
               (noisy * 1.1, cl, torch.tensor([n, n // 2], dtype=torch.int32)),
               (noisy * 0.9, cl, torch.tensor([n - 300, n], dtype=torch.int32)),
               (noisy, cl, torch.tensor([n, n // 2], dtype=torch.int32))]
    outs = []
    for graph in (False, True):
        tr = SETrainer(_tiny_se(), lr=1e-3, precision="fp16", cuda_graph=graph)
        losses = [float(tr.step(nb, cb, lb, fs)[0]) for nb, cb, lb in batches]
        outs.append((losses, tr.flat.flat.clone(), tr))
    (l0, p0, _), (l1, p1, tg) = outs
    print("eager", l0, "graph", l1)
    assert tg.captures == 1 and len(tg._graphs) == 1
    assert all(abs(a - b) / abs(a) < 1e-3 for a, b in zip(l0, l1))
    assert rel_l2(p1.cpu(), p0.cpu()) < 3e-4
    # the masked frames matter: the same batch with the full length gives another loss
    te = SETrainer(_tiny_se(), lr=0.0, precision="fp16")
    with torch.no_grad():
        a = float(te.loss(noisy * 1.1, cl, torch.tensor([n, n // 2]), fs)[0])
        b = float(te.loss(noisy * 1.1, cl, torch.tensor([n, n]), fs)[0])
    assert abs(a - b) / abs(b) > 1e-4
    with pytest.raises(ValueError, match="padded"):
        tg.step(noisy, cl, torch.tensor([n - 1, n - 2], dtype=torch.int32), fs)


def _write_yaml(tmp_path, name, **over):
    cfg = dict(model_configs={"num_channel": 32, "num_layer": 1}, train_precision="fp16", train_set_dynamic_mixing=False,
               num_worker=2, seed=11, learning_rate=1e-3)
    cfg.update(over)
    p = tmp_path / f"{name}.yaml"
    p.write_text(yaml.safe_dump(cfg))
    return str(p)


def _run(tmp_path, monkeypatch, yml, *flags):
    from urgent2026_challenge_track1_b200 import train_se
    monkeypatch.chdir(tmp_path)
    return train_se.main(["--config_file", yml, *flags])


@pytest.fixture(scope="module")
def sets(tmp_path_factory):
    root = tmp_path_factory.mktemp("corpus")
    make_set(root / "train", n_per_rate=5, seed=0)
    make_set(root / "valid", n_per_rate=2, seed=1)
    return str(root / "train"), str(root / "valid")


def test_train_se_corpus_end_to_end(tmp_path, monkeypatch, sets):
    from urgent2026_challenge_track1_b200 import data as D
    from urgent2026_challenge_track1_b200 import inference as I
    from urgent2026_challenge_track1_b200.d_model import SEModel
    train, valid = sets
    yml = _write_yaml(tmp_path, "se_tiny")
    hist = _run(tmp_path, monkeypatch, yml, "--train_set_path", train, "--valid_set_path", valid, "--val_check_interval", "2",
                "--save_top_k", "2", "--batch_size", "2", "--max_duration", "8000", "--num_train_epochs", "1",
                "--train_precision", "fp16")
    ck_dir = tmp_path / "exp" / "se_tiny" / "baseline" / "version_0" / "checkpoints"
    files = sorted(os.listdir(ck_dir))
    print(files, [(v["step"], v["val_loss"]) for v in hist["val"]])
    assert hist["global_step"] == 9 and len(hist["val"]) == 5                 # steps 2, 4, 6, 8 and the end (9)
    assert 1 <= len(files) <= 2 and all(f.startswith("best_") and "-val_loss=" in f for f in files)
    by_step = {v["step"]: v for v in hist["val"]}
    best = sorted(v["val_loss"] for v in hist["val"])[:2]
    kept = {int(f.split("step=")[1].split("-")[0]): f for f in files}
    assert sorted(by_step[s]["val_loss"] for s in kept) == best
    assert all(k in by_step[s] for s in kept for k in ("val_sisnr", "val_sisnr_8000", "val_sisnr_16000", "val_sisnr_48000"))
    # the logged val_loss is the utterance-weighted mean of SEModel.forward_step(stage="val") over the same batches
    step, fname = sorted(kept.items())[0]
    ckpt = str(ck_dir / fname)
    m = SEModel.load_from_checkpoint(ckpt, map_location="cuda")
    corpus = D.PairCorpus(valid)
    tot, cnt = 0.0, 0
    for idx in D.valid_batches(corpus, 2, 8000, 0, 1):
        clean, noisy, fs, lens = D.collate(corpus, idx, 8000, train=False)
        loss = m.validation_step((clean.cuda(), noisy.cuda(), fs, lens))
        tot += float(loss) * len(idx)
        cnt += len(idx)
    assert abs(tot / cnt - by_step[step]["val_loss"]) <= 1e-6 * abs(tot / cnt), (tot / cnt, by_step[step]["val_loss"])
    raw = torch.load(ckpt, map_location="cpu", weights_only=False)
    assert raw["global_step"] == step and set(raw["b200_trainer"]) >= {"exp_avg", "exp_avg_sq", "stats", "lr", "epoch",
                                                                        "global_step", "batches_in_epoch"}
    # the kept checkpoint enhances a WAV through the inference CLI
    model = I.load_model(ckpt, torch.device("cuda"))
    assert isinstance(model, SEModel)
    wav = os.path.join(train, "u16000_0_n.wav")
    (tmp_path / "in.scp").write_text(f"utt {wav}\n")
    I.main(I.build_parser().parse_args(["--input_scp", str(tmp_path / "in.scp"), "--output_dir", str(tmp_path / "out"),
                                        "--ckpt_path", ckpt]))
    y, sr = I._read_wav(str(tmp_path / "out" / "wav" / "utt.wav"))
    x, sr0 = I._read_wav(wav)
    assert sr == sr0 == 16000 and len(y) == len(x) and abs(abs(y).max() - 0.9) < 1e-3


def test_train_se_corpus_resume(tmp_path, monkeypatch):
    """6 steps uninterrupted against 3 steps + resume + 3 more, on a set of 4 batches per epoch: the resume lands mid-epoch
    and the resumed part crosses an epoch end with its StepLR.  Counters, lr and position agree exactly.  The graphed step is
    not bitwise reproducible (atomic accumulations), so the moments and parameters are compared against the spread of a
    second uninterrupted run: a resume must stay within a few times that spread (and within 3e-4 when the spread is below
    it), far below how much the same 3 steps move them."""
    root = tmp_path / "set"
    make_set(root, n_per_rate=4, rates=(16000, 48000), seed=3)
    yml = _write_yaml(tmp_path, "se_resume")
    common = ["--train_set_path", str(root), "--valid_set_path", str(root), "--val_check_interval", "3", "--save_top_k", "-1",
              "--batch_size", "2", "--max_duration", "8000", "--num_train_epochs", "3", "--lr_gamma", "0.5"]
    _run(tmp_path, monkeypatch, yml, *common, "--train_name", "full", "--max_steps", "6")
    _run(tmp_path, monkeypatch, yml, *common, "--train_name", "twin", "--max_steps", "6")
    _run(tmp_path, monkeypatch, yml, *common, "--train_name", "split", "--max_steps", "3")
    h = _run(tmp_path, monkeypatch, yml, *common, "--train_name", "split", "--max_steps", "6")
    assert h["global_step"] == 6 and [v["step"] for v in h["val"]] == [6]
    base = tmp_path / "exp" / "se_resume"

    def ck(name, step):
        d = base / name / "version_0" / "checkpoints"
        f = [x for x in os.listdir(d) if f"step={step:06d}" in x]
        assert len(f) == 1, os.listdir(d)
        return torch.load(d / f[0], map_location="cpu", weights_only=False)

    def params(c):
        return torch.cat([v.flatten().double() for v in c["state_dict"].values()])
    a3, b3, a6, b6, t6 = ck("full", 3), ck("split", 3), ck("full", 6), ck("split", 6), ck("twin", 6)
    for x, y, pos in ((a3, b3, (0, 3, 3)), (a6, b6, (1, 6, 2))):
        sx, sy = x["b200_trainer"], y["b200_trainer"]
        assert (sx["epoch"], sx["global_step"], sx["batches_in_epoch"]) == (sy["epoch"], sy["global_step"], sy["batches_in_epoch"]) == pos
        assert torch.equal(sx["stats"][2:4], sy["stats"][2:4]) and sx["lr"] == sy["lr"]
    assert a3["b200_trainer"]["lr"] == 1e-3 and a6["b200_trainer"]["lr"] == 1e-3 * 0.5
    spread = {k: rel_l2(t6["b200_trainer"][k], a6["b200_trainer"][k]) for k in ("exp_avg", "exp_avg_sq")}
    spread["params"] = rel_l2(params(t6), params(a6))
    resumed = {k: rel_l2(b6["b200_trainer"][k], a6["b200_trainer"][k]) for k in ("exp_avg", "exp_avg_sq")}
    resumed["params"] = rel_l2(params(b6), params(a6))
    # floors: 5x the spread of two uninterrupted runs measured on a B200 (exp_avg 2.2e-3, exp_avg_sq 8.3e-4, params 3.2e-4)
    bound = {k: max(floor, 4 * spread[k]) for k, floor in (("exp_avg", 1e-2), ("exp_avg_sq", 4e-3), ("params", 1.5e-3))}
    moved = rel_l2(a6["b200_trainer"]["exp_avg"], a3["b200_trainer"]["exp_avg"])   # what losing the moments would cost
    print("run-to-run spread", spread, "resumed vs uninterrupted", resumed, "bound", bound, "exp_avg over 3 steps", moved)
    for k in resumed:
        assert resumed[k] <= bound[k], (k, resumed, bound)
    assert moved > 10 * bound["exp_avg"]


def test_train_se_corpus_flowse(tmp_path, monkeypatch, sets):
    import types
    import warnings
    from oracle import ref_loader
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    train, valid = sets
    cfg = dict(vars(ref_loader.flowse_config(types.SimpleNamespace(Config=Config), num_layer=1)))
    cfg = {k: v for k, v in cfg.items() if k not in ("config_file", "train_tag", "model_configs")}
    cfg.update(model_type="flowse", train_set_dynamic_mixing=False, num_worker=1, train_set_path=train, valid_set_path=valid,
               max_steps=3, val_check_interval=2, batch_size=2, max_duration=8000)       # YAML keys win over flags
    yml = tmp_path / "flowse_tiny.yaml"
    yml.write_text(yaml.safe_dump(cfg))
    hist = _run(tmp_path, monkeypatch, str(yml))
    assert hist["global_step"] == 3 and [v["step"] for v in hist["val"]] == [2, 3]
    d = tmp_path / "exp" / "flowse_tiny" / "baseline" / "version_0" / "checkpoints"
    files = sorted(os.listdir(d))
    assert files
    raw = torch.load(d / files[0], map_location="cpu", weights_only=False)
    assert "ema" in raw and "b200_trainer" in raw and raw["b200_trainer"]["ema"] is not None
    with warnings.catch_warnings():
        warnings.simplefilter("error")
        FlowSEModel.load_from_checkpoint(str(d / files[0]), map_location="cuda")
    # val_loss is computed on the EMA weights (what eval() swaps in and the checkpoint ships), not the live ones
    from urgent2026_challenge_track1_b200 import data as D
    from urgent2026_challenge_track1_b200.checkpoint import load_checkpoint
    from urgent2026_challenge_track1_b200.train_se import validate
    last = [f for f in files if "step=000003" in f][0]
    _, ccfg, raw = load_checkpoint(str(d / last))
    fm = FlowSEModel.load_from_checkpoint(str(d / last), map_location="cuda")
    tr = fm.configure_optimizers(precision="fp16", cuda_graph=True)
    tr.load_state_dict(raw["b200_trainer"])
    dev = torch.device("cuda")
    tr.sync_ema()
    fm.eval()
    on_ema = validate(fm, tr, D.PairCorpus(valid), ccfg, 0, 1, dev, True)["val_loss"]
    fm.train()
    on_live = validate(fm, tr, D.PairCorpus(valid), ccfg, 0, 1, dev, True)["val_loss"]
    logged = [v for v in hist["val"] if v["step"] == 3][0]["val_loss"]
    print("FlowSE val_loss logged", logged, "EMA", on_ema, "live", on_live)
    assert abs(on_ema - logged) <= 1e-5 * abs(logged) and abs(on_live - logged) > 1e-4 * abs(logged)
    # a checkpoint without b200_trainer (as the reference writes) restores its EMA into the flat buffer
    fm2 = FlowSEModel.load_from_checkpoint(str(d / last), map_location="cuda")
    tr2 = fm2.configure_optimizers(precision="fp16", cuda_graph=True)
    tr2.load_ema_from_model()
    assert torch.equal(tr2.ema.cpu(), raw["b200_trainer"]["ema"]) and int(tr2.stats[3]) == raw["ema"]["num_updates"] == 3
