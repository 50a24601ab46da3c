"""GPU tests of BSRNN-FlowSE training at the published width (N = 384, H = 768): the tensor-core BLSTM block with the fused
and the step-wise forward, the whole flow-matching forward step against the f64 oracle, CUDA-graph replay, the published
config, the train_se command line with its checkpoint, and two data-parallel ranks."""
import copy
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from conftest import rel_l2
from oracle import restated as R
from oracle import ref_loader

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cfg(**over):
    from urgent2026_challenge_track1_b200.config import Config
    return ref_loader.flowse_config(types.SimpleNamespace(Config=Config), **over)


def _block_run(x, wgt, rnn, fc, axis):
    from urgent2026_challenge_track1_b200.training_tc import blstm_block_tc
    rnn, fc = copy.deepcopy(rnn).cuda(), copy.deepcopy(fc).cuda()
    xg = x.float().cuda().requires_grad_(True)
    out = blstm_block_tc(xg, rnn, fc, axis)
    (out * wgt.float().cuda()).sum().backward()
    grads = {f"rnn.{n}": p.grad.cpu().double() for n, p in rnn.named_parameters()}
    grads.update({f"fc.{n}": p.grad.cpu().double() for n, p in fc.named_parameters()})
    return out.detach().cpu().double(), xg.grad.cpu().double(), grads


# (axis, B, T, K): one sequence tile with 9 steps; 3 tiles (odd) with R = 300; one step over 2 tiles with R = 130; 48 steps
@pytest.mark.parametrize("axis,B,T,K", [("time", 2, 9, 5), ("freq", 3, 100, 4), ("time", 1, 1, 130), ("freq", 2, 3, 48)])
def test_blstm_block_n384_fused_and_stepwise_vs_torch(axis, B, T, K, monkeypatch):
    """training_tc.BLSTMBlockTC at N = 384 / H = 768 with the fused forward (bsrnn_blstm_fused768_train_tc) and the
    step-wise one, against nn.LSTM + nn.Linear under torch autograd in f64, and against each other."""
    from urgent2026_challenge_track1_b200 import _lib as L, training_tc as TT
    N, H = 384, 768
    torch.manual_seed(0)
    rnn = torch.nn.LSTM(N, H, batch_first=True, bidirectional=True)
    fc = torch.nn.Linear(2 * H, N)
    x = torch.randn(B, T, K, N, dtype=torch.float64) * 0.8
    wgt = torch.randn(B, T, K, N, dtype=torch.float64) * 3e-3
    ref_rnn, ref_fc = copy.deepcopy(rnn).double(), copy.deepcopy(fc).double()
    xr = x.clone().requires_grad_(True)
    if axis == "time":
        yr = ref_rnn(xr.permute(0, 2, 1, 3).reshape(B * K, T, N))[0].reshape(B, K, T, 2 * H).permute(0, 2, 1, 3)
    else:
        yr = ref_rnn(xr.reshape(B * T, K, N))[0].reshape(B, T, K, 2 * H)
    outr = ref_fc(yr)
    (outr * wgt).sum().backward()
    ref_g = {f"rnn.{n}": p.grad for n, p in ref_rnn.named_parameters()}
    ref_g.update({f"fc.{n}": p.grad for n, p in ref_fc.named_parameters()})
    calls = []
    orig_call = L.call
    monkeypatch.setattr(L, "call", lambda name, *a: (calls.append(name), orig_call(name, *a))[1])
    res = {}
    for fused in (True, False):
        monkeypatch.setattr(TT, "FUSED_TRAIN", fused)
        calls.clear()
        res[fused] = out, dx, grads = _block_run(x, wgt, rnn, fc, axis)
        assert ("bsrnn_blstm_fused768_train_tc" in calls) == fused and ("bsrnn_blstm_train_fwd_tc" in calls) != fused
        e_out, e_dx = rel_l2(out, outr.detach()), rel_l2(dx, xr.grad)
        e_w = {n: rel_l2(g, ref_g[n]) for n, g in grads.items()}
        print(f"block N=384 {'fused' if fused else 'steps'} {axis} B={B} T={T} K={K}: out {e_out:.2e} dx {e_dx:.2e} "
              f"worst dW {max(e_w.values()):.2e}")
        assert e_out < 3e-3 and e_dx < 1e-2, (e_out, e_dx)
        assert max(e_w.values()) < 1e-2, e_w
    (o1, d1, g1), (o0, d0, g0) = res[True], res[False]
    assert rel_l2(o1, o0) < 3e-3 and rel_l2(d1, d0) < 1e-2
    assert max(rel_l2(g1[n], g0[n]) for n in g0) < 1e-2


def _oracle_loss(fm, clean, noisy, lens, fs, t, z, layers):
    sd = {k: v.detach().clone().double().requires_grad_(v.dtype.is_floating_point and not k.endswith(".W"))
          for k, v in fm.state_dict().items()}
    x0, _ = R.stft_encode(clean.double(), lens, fs, 1536, 384, 48000, "exponent", 0.667, 0.065)      # (B,T,F)
    y, _ = R.stft_encode(noisy.double(), lens, fs, 1536, 384, 48000, "exponent", 0.667, 0.065)
    std = ((1 - t) * 0.05 + t * 0.5).double()[:, None, None]
    xt = (1 - t.double())[:, None, None] * x0 + t.double()[:, None, None] * y + std * z
    cond = (0.5 - 0.05) * z + (y - x0)
    to_bft = lambda a: a.permute(0, 2, 1).unsqueeze(1)                                                  # (B,1,F,T)
    vf = -R.flow_bsrnn_forward(sd, torch.cat([to_bft(xt), to_bft(y)], dim=1), t.double(), 769, num_layer=layers)
    loss = R.flow_matching_loss(vf, to_bft(cond))
    loss.backward()
    return loss, sd


@pytest.mark.parametrize("fs", (16000, 48000))
def test_flowse_forward_step_n384_tensorcore_matches_oracle(fs):
    """flowse_forward_step at bsrnn_hidden = 384 (2 layers, ragged lengths, t and z passed in) with the BLSTM blocks on
    tensor cores: loss and every parameter gradient against the f64 oracle; 16-bit bars."""
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    from urgent2026_challenge_track1_b200.training import block_tc, flowse_forward_step
    torch.manual_seed(0)
    fm = FlowSEModel(_cfg(num_layer=2))
    n = fs // 8
    clean, noisy = R.synth_noisy(2, n, fs, seed=7), R.synth_noisy(2, n, fs, seed=1)
    lens = torch.tensor([n, n - 211])
    t = torch.tensor([0.83, 0.27])
    n_fft, hop = 1536 * fs // 48000, 384 * fs // 48000
    z = torch.randn(2, 1 + n // hop, n_fft // 2 + 1, dtype=torch.complex128, generator=torch.Generator().manual_seed(3))
    ref_loss, sd = _oracle_loss(fm, clean, noisy, lens, fs, t, z, 2)
    fm = fm.cuda()
    loss, _ = flowse_forward_step(fm, noisy.cuda(), clean.cuda(), lens, fs, t=t, z=z.to(torch.complex64), blstm_fn=block_tc)
    loss.backward()
    worst, num, den = 0.0, 0.0, 0.0
    for k, p in fm.named_parameters():
        g_ref = sd[k].grad
        if g_ref is None or float(g_ref.abs().max()) == 0.0:
            continue
        d = p.grad.cpu().double() - g_ref
        num += float((d ** 2).sum()); den += float((g_ref ** 2).sum())
        worst = max(worst, rel_l2(p.grad.cpu().double(), g_ref))
    e_loss = abs(float(loss) - float(ref_loss)) / float(ref_loss)
    print(f"FlowSE N=384 fs={fs}: loss {float(loss):.4f} vs {float(ref_loss):.4f} ({e_loss:.1e}); all-parameter gradient "
          f"rel_l2 {(num / den) ** 0.5:.2e}, worst tensor {worst:.2e}")
    assert e_loss < 5e-3
    assert (num / den) ** 0.5 < 1e-2 and worst < 5e-2


def _batch(fs, n, B=2, seed=0):
    clean, noisy = R.synth_noisy(B, n, fs, seed=seed + 7), R.synth_noisy(B, n, fs, seed=seed + 1)
    return clean.view(B, 1, -1).cuda(), noisy.view(B, 1, -1).cuda(), torch.tensor(fs, dtype=torch.int32), torch.tensor([n] * B)


def _fixed_draws(fs, n, B, seed=5):
    n_fft, hop = 1536 * fs // 48000, 384 * fs // 48000
    g = torch.Generator().manual_seed(seed)
    t = (0.03 + 0.97 * torch.rand(B, generator=g)).cuda()
    z = torch.randn(B, 1 + n // hop, n_fft // 2 + 1, dtype=torch.complex64, generator=g).cuda()
    return t, z


def _fix_tz(tr, t, z):
    from urgent2026_challenge_track1_b200.training import flowse_forward_step
    tr.loss_fn = lambda m, noisy, clean, lengths, fs, blstm_fn=None: flowse_forward_step(m, noisy, clean, lengths, fs, t=t, z=z,
                                                                                          blstm_fn=blstm_fn)


def test_flowse_graphed_step_matches_eager():
    """FlowSETrainer(fp16, cuda_graph=True) at N = 384 replays the same loss and parameter trajectory as host launches
    with (t, z) fixed; with the trainer's own draws, replays on one batch draw t and z afresh."""
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    fs, n = 16000, 8000
    t, z = _fixed_draws(fs, n, 2)
    outs = []
    for graph in (False, True):
        torch.manual_seed(0)
        fm = FlowSEModel(_cfg(num_layer=1, learning_rate=1e-3)).cuda()
        tr = fm.configure_optimizers(precision="fp16", cuda_graph=graph)
        _fix_tz(tr, t, z)
        clean, noisy, fsd, lens = _batch(fs, n)
        losses = [float(tr.step(noisy * (1 + 0.1 * i), clean, lens, fsd)[0]) for i in range(4)]
        outs.append((losses, tr.flat.flat.clone(), tr.step_count))
    (l0, p0, n0), (l1, p1, n1) = outs
    print("eager", l0, "graph", l1)
    assert n0 == n1 == 4
    assert all(abs(a - b) / abs(a) < 1e-3 for a, b in zip(l0, l1))
    assert rel_l2(p1.cpu(), p0.cpu()) < 3e-4
    torch.manual_seed(0)
    fm = FlowSEModel(_cfg(num_layer=1, learning_rate=0.0)).cuda()
    tr = fm.configure_optimizers(precision="fp16", cuda_graph=True)
    clean, noisy, fsd, lens = _batch(fs, n)
    drawn = [float(tr.step(noisy, clean, lens, fsd)[0]) for _ in range(4)]
    assert len(tr._graphs) == 1 and all(np.isfinite(drawn))
    assert len(set(drawn)) == 4, drawn                      # replays of one graph on one batch at lr 0: new (t, z) each


def test_flowse_published_config_fp16_graph_trains():
    """The published config (N = 384, 6 layers, 103 M parameters), B = 2 x 1 s at 48 kHz, fp16 + CUDA graph, 5 steps with
    fixed (t, z): losses finite and falling, the optimizer and EMA counters advance, and the synced EMA weights enhance
    differently from the live ones."""
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    fs, n = 48000, 48000
    torch.manual_seed(0)
    fm = FlowSEModel(_cfg()).cuda()
    assert sum(p.numel() for p in fm.parameters()) == 103245488
    tr = fm.configure_optimizers(precision="fp16", cuda_graph=True)
    t, z = _fixed_draws(fs, n, 2)
    _fix_tz(tr, t, z)
    clean, noisy, fsd, lens = _batch(fs, n)
    losses = [float(tr.step(noisy, clean, lens, fsd)[0]) for _ in range(5)]
    print("published config losses", losses)
    assert all(np.isfinite(losses)) and losses[-1] < losses[0], losses
    assert tr.step_count == 5
    tr.sync_ema()
    assert fm.ema.num_updates == 5
    y, ln = noisy.view(2, -1), torch.tensor([n, n])
    zz = lambda: torch.randn(2, 1, 769, 1 + n // 384, dtype=torch.complex64, generator=torch.Generator().manual_seed(0))
    live = fm.train().enhance(y, fs, ln, N=2, z=zz())
    ema_out = fm.eval().enhance(y, fs, ln, N=2, z=zz())
    assert torch.isfinite(ema_out).all() and torch.isfinite(live).all()
    assert rel_l2(ema_out.cpu(), live.cpu()) > 1e-6


def test_train_se_cli_flowse_checkpoint_and_inference(tmp_path):
    """python -m ...train_se with model_type: flowse trains, writes a reference-layout checkpoint with the EMA, and
    inference.py enhances with it."""
    import yaml
    from urgent2026_challenge_track1_b200 import inference as I
    cfg = dict(vars(_cfg()))
    cfg.update(model_type="flowse", bsrnn_hidden=384, num_layer=1, max_steps=3, save=True, batch_size=2, max_duration=24000)
    cfg = {k: v for k, v in cfg.items() if k not in ("config_file", "train_tag", "model_configs")}
    yml = tmp_path / "flowse_tiny.yaml"
    yml.write_text(yaml.safe_dump(cfg))
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "urgent2026_challenge_track1_b200.train_se", "--config_file", str(yml)],
                       cwd=tmp_path, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    ck_dir = tmp_path / "exp" / "flowse_tiny" / "baseline" / "version_0" / "checkpoints"
    ckpt = ck_dir / "last-step000003.ckpt"
    assert ckpt.exists(), os.listdir(ck_dir)
    from urgent2026_challenge_track1_b200.checkpoint import load_checkpoint
    sd, c, raw = load_checkpoint(str(ckpt))
    assert any(k.startswith("dnn.") for k in sd) and c.model_type == "flowse" and c.bsrnn_hidden == 384
    assert "state_dict" in raw and raw["hyper_parameters"]["cfg"] is not None
    assert raw["ema"]["num_updates"] == 3 and len(raw["ema"]["shadow_params"]) > 0
    import warnings
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    with warnings.catch_warnings():
        warnings.simplefilter("error")                 # no "EMA state_dict not found"
        FlowSEModel.load_from_checkpoint(str(ckpt), map_location="cuda")
    from urgent2026_challenge_track1_b200.synth import synth_noisy
    lines = []
    for i, (fs, n) in enumerate([(16000, 6000), (48000, 12000)]):
        p = str(tmp_path / f"in_{i}.wav")
        I._write_wav(p, synth_noisy(1, n, fs, seed=100 + i)[0].numpy(), fs)
        lines.append(f"utt{i} {p}")
    (tmp_path / "wav.scp").write_text("\n".join(lines) + "\n")
    out_dir = str(tmp_path / "out")
    r = subprocess.run([sys.executable, "-m", "urgent2026_challenge_track1_b200.inference", "--input_scp", str(tmp_path / "wav.scp"),
                        "--output_dir", out_dir, "--ckpt_path", str(ckpt), "--nfe", "2"], cwd=tmp_path, env=env,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    listed = dict(l.split() for l in open(os.path.join(out_dir, "inf.scp")).read().strip().splitlines())
    assert set(listed) == {"utt0", "utt1"}
    for i, (fs, n) in enumerate([(16000, 6000), (48000, 12000)]):
        y, sr = I._read_wav(listed[f"utt{i}"])
        assert sr == fs and len(y) == n and np.isfinite(y).all() and abs(np.abs(y).max() - 0.9) < 1e-3


_DDP_WORKER = r'''
import os, sys, types, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from oracle import ref_loader
from urgent2026_challenge_track1_b200.config import Config
from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
from urgent2026_challenge_track1_b200.train_se import synthetic_batches
rank = int(os.environ["RANK"])
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
cfg = ref_loader.flowse_config(types.SimpleNamespace(Config=Config), num_layer=1, batch_size=2, max_duration=24000, seed=3)
torch.manual_seed(100 + rank)                 # different initial weights per rank: the broadcast must align them
fm = FlowSEModel(cfg).to(dev)
for p in fm.parameters():
    dist.broadcast(p.data, 0)
tr = fm.configure_optimizers(precision="fp16", cuda_graph=True)
for clean, noisy, fs, lens in synthetic_batches(cfg, rank, 2, 2, dev):
    tr.step(noisy, clean, lens, fs)
tr.sync_ema()
torch.save({"flat": tr.flat.flat.cpu(), "ema": [s.cpu() for s in fm.ema.shadow_params], "steps": tr.step_count},
           os.path.join(sys.argv[2], f"rank{rank}.pt"))
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_flowse_two_ranks_stay_identical(tmp_path):
    """Two NCCL ranks, 2 fp16 + graph steps on different data: one flat-buffer allreduce per step keeps the parameters and
    the EMA bit-identical across ranks."""
    script = tmp_path / "worker.py"
    script.write_text(_DDP_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29741", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(tmp_path)], env=dict(env, RANK=str(r), LOCAL_RANK=str(r)),
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=900)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    a, b = (torch.load(tmp_path / f"rank{r}.pt") for r in range(2))
    assert a["steps"] == b["steps"] == 2
    assert torch.equal(a["flat"], b["flat"])
    assert all(torch.equal(x, y) for x, y in zip(a["ema"], b["ema"]))
