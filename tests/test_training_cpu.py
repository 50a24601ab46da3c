"""CPU tests of the training-side host logic: the loss restatement against the oracle and the golden loss fixture,
the flat parameter/gradient buffers, and the one-bucket gradient allreduce over 2 gloo ranks with rank-dependent unused
parameters (the reference's ddp_find_unused_parameters_true case, train_se.py:82)."""
import os
import sys

import pytest
import torch

from conftest import golden, rel_l2
from oracle import restated as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_losses_match_oracle_and_golden():
    from urgent2026_challenge_track1_b200.losses import multires_l1_spec_loss_reference as multires_l1_spec_loss, si_snr_loss
    g = golden("losses.npz")
    tgt, est = torch.from_numpy(g["target"]), torch.from_numpy(g["estimate"])
    mine = multires_l1_spec_loss(tgt, est)
    assert torch.allclose(mine, torch.from_numpy(g["mr_l1"]), rtol=1e-5, atol=1e-3)      # verbatim-reference output
    assert torch.allclose(mine, R.multires_l1_spec_loss(tgt, est), rtol=1e-6)
    assert torch.allclose(si_snr_loss(tgt, est), torch.from_numpy(g["sisnr"]), rtol=1e-5, atol=1e-5)
    # gradients agree with the oracle's
    e1, e2 = est.clone().requires_grad_(True), est.clone().requires_grad_(True)
    multires_l1_spec_loss(tgt, e1).mean().backward()
    R.multires_l1_spec_loss(tgt, e2).mean().backward()
    assert rel_l2(e1.grad, e2.grad) < 1e-5


def test_flat_params_alias_module_parameters():
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.training import FlatParams
    m = BSRNN_SE(16, 1)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    fp = FlatParams(m)
    assert fp.numel == sum(p.numel() for p in m.parameters())
    assert all(torch.equal(before[k], v) for k, v in m.state_dict().items())     # values survive the re-pointing
    p = m.bsrnn.bsrnn.fc_time[0].weight
    fp.flat.mul_(2.0)                                                            # the flat buffer IS the parameters
    assert torch.equal(p, before["bsrnn.bsrnn.fc_time.0.weight"] * 2)
    (p.sum() * 3).backward()                                                     # autograd accumulates into the flat grad
    fp.gather_grads()
    off = fp.offsets[[id(q) for q in fp.params].index(id(p))]
    assert torch.equal(fp.grad[off:off + p.numel()], torch.full((p.numel(),), 3.0))
    fp.zero_grad()
    assert float(fp.grad.abs().sum()) == 0.0 and p.grad.data_ptr() == fp.grad[off:off + 1].data_ptr()


_WORKER = r'''
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from urgent2026_challenge_track1_b200 import BSRNN_SE
from urgent2026_challenge_track1_b200.training import SETrainer
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dist.init_process_group("gloo", rank=rank, world_size=world)
torch.manual_seed(0)
m = BSRNN_SE(16, 1)
tr = SETrainer(m)
core = m.bsrnn.bsrnn
tr.flat.zero_grad()
# rank 0 "saw a 16 kHz batch": bands >= 27 get no gradient; rank 1 touches every band
used = range(27) if rank == 0 else range(len(core.band_split.fc))
loss = sum((core.band_split.fc[k].weight * (rank + 1)).sum() for k in used) + core.fc_time[0].weight.sum() * (rank + 1)
loss.backward()
tr.flat.gather_grads()
w = tr.allreduce_gradients()
g_lo = core.band_split.fc[0].weight.grad.flatten()[0].item()       # both ranks: 1 + 2
g_hi = core.band_split.fc[30].weight.grad.flatten()[0].item()      # rank 1 only: 0 + 2
g_fc = core.fc_time[0].weight.grad.flatten()[0].item()
ok = w == 2 and g_lo == 3.0 and g_hi == 2.0 and g_fc == 3.0
print(f"rank {rank} world {w} grads {g_lo} {g_hi} {g_fc} {'OK' if ok else 'FAIL'}")
dist.destroy_process_group()
sys.exit(0 if ok else 1)
'''


def test_flat_gradient_allreduce_two_gloo_ranks(tmp_path):
    import subprocess
    script = tmp_path / "worker.py"
    script.write_text(_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29731", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, str(script), ROOT], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True) for r in range(2)]
    outs = [p.communicate(timeout=240)[0] for p in procs]
    assert all(p.returncode == 0 for p in procs), outs
    assert all("OK" in o for o in outs), outs


@pytest.mark.parametrize("fs", [48000, 16000, 44100])
def test_batched_band_ops_equal_the_per_band_loops(fs):
    """training.band_split_batched / mask_decoder_batched (one gather + batched GEMMs over zero-padded bands) against the
    per-band loops that mirror the reference modules: outputs and every parameter gradient, in f64, incl. truncated bands."""
    from urgent2026_challenge_track1_b200 import BSRNN_SE, runtime as RT, training as TR
    torch.manual_seed(0)
    m = BSRNN_SE(num_channel=16, num_layer=1, precision="fp32").double()
    core = m.bsrnn.bsrnn
    n_fft, hop = RT.stft_dims(fs, m.N_FFT, m.HOP, m.DEFAULT_FS)
    Fb = n_fft // 2 + 1
    plan = RT.BandPlan.make(core.band_split.subbands, Fb)
    spec = torch.randn(2, 7, Fb, 2, dtype=torch.float64)
    for p in m.parameters():
        p.data = p.data + 0.1 * torch.randn_like(p)

    def run(bsf, mdf):
        for p in m.parameters():
            p.grad = None
        skip = bsf(core.band_split, spec, plan)
        mc, rc = mdf(core.mask_decoder, skip, plan, Fb)
        ((mc.abs() ** 2).sum() + (rc.real * 1.3 + rc.imag * 0.7).sum() + 0.01 * (skip ** 2).sum()).backward()
        return skip.detach(), mc.detach(), rc.detach(), {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}

    a = run(TR.band_split_diff, TR.mask_decoder_diff)
    b = run(TR.band_split_batched, TR.mask_decoder_batched)
    rel = lambda x, y: float((x - y).abs().max() / (y.abs().max() + 1e-30))
    assert rel(b[0], a[0]) < 1e-12 and rel(b[1], a[1]) < 1e-12 and rel(b[2], a[2]) < 1e-12
    assert set(a[3]) == set(b[3])                       # bands the spectrum does not reach get no gradient in either
    assert max(rel(b[3][n], a[3][n]) for n in a[3]) < 1e-11

