"""CPU tests of the host-side logic: band plans, STFT sizes, state_dict layout (against the golden fixtures, i.e. the
reference's own key names), config / registry behaviour, KB8 packing, multi-rank sharding (gloo, world_size 2)."""
import os
import sys

import pytest
import torch

from conftest import golden, golden_sd
from oracle import restated as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_band_plan_matches_reference_table():
    from urgent2026_challenge_track1_b200.runtime import BandPlan, subbands_for, stft_dims
    want = {8000: (81, 20), 16000: (161, 27), 22050: (221, 28), 24000: (241, 29), 32000: (321, 31), 44100: (442, 34),
            48000: (481, 34)}                                                      # SURVEY.md §8a
    for fs, (F, K) in want.items():
        n_fft, hop = stft_dims(fs, 960, 480)
        assert (n_fft, hop) == R.stft_dims(fs, 960, 480) and n_fft // 2 + 1 == F
        plan = BandPlan.make(subbands_for(481), F)
        assert plan.K == K and sum(plan.width) == F
    plan = BandPlan.make(subbands_for(481), 161)
    assert plan.width[-1] == 20 and plan.subbands[plan.K - 1] == 40               # 20 real + 20 padded bins @16 kHz
    assert BandPlan.make(subbands_for(769), 769).K == 48
    with pytest.raises(NotImplementedError):
        subbands_for(513)


def test_state_dict_layout_is_the_references():
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    g = golden("bsrnn_se_n16_l2.npz")
    m = BSRNN_SE(16, 2)
    ref = golden_sd(g)
    assert set(m.state_dict()) == set(ref)
    assert all(m.state_dict()[k].shape == ref[k].shape for k in ref)
    m.load_state_dict(ref)
    full = BSRNN_SE(196, 6)
    assert sum(p.numel() for p in full.parameters()) == 37_800_844 and len(full.state_dict()) == 688   # SURVEY §8b
    g = golden("flowse_n16_l1.npz")
    cfg = Config(model_type="flowse", ema_decay=0.999, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0,
                 loss_type="mse", n_fft=1536, hop_length=384, spec_transform_type="exponent", spec_abs_exponent=0.667,
                 spec_factor=0.065, bsrnn_hidden=16, num_layer=1)
    fm = FlowSEModel(cfg)
    ref = golden_sd(g)
    assert set(fm.state_dict()) == set(ref)
    fm.load_state_dict(ref)
    assert fm.dnn.t_cond[0].W.requires_grad is False


def test_param_counts_are_the_published_ones():
    """Our modules carry the parameter counts the reference publishes, conf/models/BSRNN_baseline.yaml:30-32:
    'Parameters: 36.01795196533203 M' @48k, '32.0456657409668 M' @16k (unit 2**20, GroupNorm affine parameters not
    counted), and the BSRNN_flowse.yaml model's 103 245 488 parameters."""
    import types
    from oracle import ref_loader
    from urgent2026_challenge_track1_b200 import BSRNN_SE
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    b = BSRNN_SE(num_channel=196, num_layer=6).bsrnn.bsrnn
    gn = {n for n, mod in b.named_modules() if isinstance(mod, torch.nn.GroupNorm)}
    beyond_27 = lambda name: name.split(".")[0] in ("band_split", "mask_decoder") and int(name.split(".")[2]) >= 27
    counted = [(n, p.numel()) for n, p in b.named_parameters() if n.rsplit(".", 1)[0] not in gn]
    assert sum(c for _, c in counted) / 2 ** 20 == pytest.approx(36.01795196533203, abs=1e-9)
    # @16 kHz only K'=27 bands of band_split / mask_decoder are touched
    assert sum(c for n, c in counted if not beyond_27(n)) / 2 ** 20 == pytest.approx(32.0456657409668, abs=1e-9)
    cfg = ref_loader.flowse_config(types.SimpleNamespace(Config=Config))
    assert sum(p.numel() for p in FlowSEModel(cfg).parameters()) == 103_245_488


def test_flowse_eval_swaps_ema_weights():
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    cfg = Config(model_type="flowse", ema_decay=0.5, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0,
                 loss_type="mse", n_fft=1536, hop_length=384, spec_transform_type="exponent", spec_abs_exponent=0.667,
                 spec_factor=0.065, bsrnn_hidden=16, num_layer=1)
    fm = FlowSEModel(cfg)
    p = fm.dnn.condition_fc.bias
    before = p.detach().clone()
    with torch.no_grad():
        p.add_(1.0)
    fm.ema.update(fm.parameters())
    fm.eval()                                   # reference flow_model.py:98-109: EMA weights swapped in place
    assert not torch.allclose(p, before + 1.0)
    fm.train()
    assert torch.allclose(p, before + 1.0)
    ck = {}
    fm.on_save_checkpoint(ck)
    assert set(ck["ema"]) == {"decay", "num_updates", "shadow_params", "collected_params"}


def test_config_yaml_and_flags(tmp_path):
    from urgent2026_challenge_track1_b200.config import Config, config_parser
    y = tmp_path / "BSRNN_baseline.yaml"
    y.write_text("batch_size: 4\nse_model: bsrnn\nmodel_configs:\n  num_channel: 196\n  num_layer: 6\nnew_key: 7\n")
    args = config_parser(["--config_file", str(y), "--resume", "no", "--learning_rate", "2e-3"])
    cfg = Config(**vars(args))
    cfg.read_yaml()
    assert cfg.batch_size == 4 and cfg.model_configs == {"num_channel": 196, "num_layer": 6} and cfg.new_key == 7
    assert cfg.train_tag == "BSRNN_baseline" and cfg.resume is False and cfg.learning_rate == 2e-3


def test_semodel_selector():
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.d_model import SEModel
    m = SEModel(Config(se_model="bsrnn", model_configs={"num_channel": 16, "num_layer": 1}))
    assert all(k.startswith("se_model.bsrnn.bsrnn.") for k in m.state_dict())
    with pytest.raises(TypeError):
        SEModel(Config(se_model="tfgridnet", model_configs={}))


def test_euler_schedule_and_registry():
    from urgent2026_challenge_track1_b200.sampling import ODEsolverRegistry, euler_schedule
    ts, steps = euler_schedule(1.0, 0.03, 15)
    rts, rsteps = R.euler_schedule(1.0, 0.03, 15)
    assert torch.equal(ts, rts) and torch.equal(steps, rsteps)
    with pytest.raises(ValueError):
        ODEsolverRegistry.get_by_name("nope")


def test_kb8_roundtrip_and_lstm_pack():
    from urgent2026_challenge_track1_b200 import runtime_tc as tc
    w = torch.randn(300, 196)
    t = tc.to_kb8(w, 208, 26)
    assert t.shape == (2, 26, 208, 8) and torch.equal(tc.from_kb8(t, 300, 196), w.half().float())
    rnn = torch.nn.LSTM(196, 392, batch_first=True, bidirectional=True)
    p = tc.pack_lstm_tc(rnn)
    assert p["wih"].shape == (16, 26, 208, 8) and p["whh"].shape == (2, 8, 50, 208, 8)
    # packed column c = 4*u + gate of CTA q is LSTM row gate*H + 49*q + u
    q, u, gate = 3, 17, 2
    row = tc.from_kb8(p["whh"][0, q][None], 208, 392)[4 * u + gate]
    assert torch.equal(row, rnn.weight_hh_l0[gate * 392 + 49 * q + u].half().float())
    with pytest.raises(NotImplementedError):
        tc.pack_lstm_tc(torch.nn.LSTM(16, 32, batch_first=True, bidirectional=True))


def test_fused_layer_weight_packs_and_geometry_choice():
    """Weight packs of the fused BLSTM layer kernel (csrc/lstm_fused.cu) for the three group geometries and the FlowSE
    width: every packed row is the LSTM row of (gate, unit) it claims to be, the bias rides in operand column N, the i/f/o
    rows are pre-halved; the geometry heuristic picks the small-batch groups for few tiles and the 10-group split where 9
    groups divide the tile pairs badly."""
    from urgent2026_challenge_track1_b200 import runtime_tc as tc, runtime_tc_steps as ts
    torch.manual_seed(0)
    rnn = torch.nn.LSTM(196, 392, batch_first=True, bidirectional=True)
    p = tc.pack_lstm_tc(rnn)
    H, N, kc_in = 392, 196, 26
    bsum = (rnn.bias_ih_l0_reverse + rnn.bias_hh_l0_reverse).detach()
    for geo, (P, U) in {8: (8, 49), 7: (7, 56), 14: (14, 28)}.items():
        wf = tc.fused_weights(p, geo).float()                        # [dir][pair][half][76][rows/2][8]
        BH = wf.shape[4]
        assert wf.shape[:4] == (2, P, 2, kc_in + 50) and BH == (208 if geo == 8 else 4 * U) // 2
        q, u, gate, d = P - 2, U - 3, 1, 1                           # a forget-gate row of the reverse direction
        c = 4 * u + gate
        e, r = divmod(c, BH)
        row = wf[d, q, e, :, r, :].reshape(-1)                       # K = 208 + 400
        src = gate * H + U * q + u
        assert torch.equal(row[:N], (0.5 * rnn.weight_ih_l0_reverse[src]).half().float())
        assert torch.equal(row[N], (0.5 * bsum[src]).half().float()) and float(row[N + 1: kc_in * 8].abs().max()) == 0
        assert torch.equal(row[kc_in * 8: kc_in * 8 + H], (0.5 * rnn.weight_hh_l0_reverse[src]).half().float())
        g_row = wf[0, 0, 0, :, 2, :].reshape(-1)                     # c = 2: cell gate of unit 0, not halved
        assert torch.equal(g_row[:N], rnn.weight_ih_l0[2 * H].half().float())
    rnn768 = torch.nn.LSTM(384, 768, batch_first=True, bidirectional=True)
    w768 = ts.pack_lstm_fused768(rnn768)
    assert w768["wfused"].shape == (2, 24, 2, 146, 64, 8) and w768["kc_fused"] == 50 and w768["one_col"] == 384
    row = w768["wfused"][0, 5, 1, :, 3, :].float().reshape(-1)       # pair 5, second half: c = 67 -> unit 16, gate 3
    src = 3 * 768 + 32 * 5 + 16
    assert torch.equal(row[400: 400 + 768], (0.5 * rnn768.weight_hh_l0[src]).half().float())
    # geometry choice (48 kHz: tiles = ceil(34 B / 128) on the time axis, ceil(1001 B / 128) on the band axis)
    assert [tc.fused_geometry(t) for t in (1, 3, 5, 6)] == [14, 14, 14, 14]
    assert tc.fused_geometry(17) == 7 and tc.fused_geometry(501) == 7 and tc.fused_geometry(9) == 8


def test_band_split_and_mask_decoder_tensorcore_packs():
    """Host side of the round-2 small-kernel work: the tensor-core BandSplit pack (one 208-row weight tile per band, K
    padded to 16, offsets of the grouped launch) and the mask-decoder pack with each family's GroupNorm affine folded into
    its first Conv1d: W (z*gamma + beta) + b == (W diag(gamma)) z + (W beta + b), bias in operand column N."""
    from urgent2026_challenge_track1_b200 import BSRNN_SE, runtime_tc as tc
    torch.manual_seed(0)
    m = BSRNN_SE(num_channel=196, num_layer=1, precision="fp16")
    for p in m.parameters():
        p.data.add_(0.05 * torch.randn_like(p))
    core = m.bsrnn.bsrnn
    bs = tc.pack_band_split_tc(core.band_split)
    K = len(core.band_split.subbands)
    assert bs["BN"] == 208 and bs["bias"].shape == (K, 208) and len(bs["kcs"]) == K
    assert all(kc == ((2 * s + 15) // 16) * 2 for kc, s in zip(bs["kcs"], core.band_split.subbands))
    k = 26                                                               # a 40-bin band: 80 channels -> 10 k-cores
    kc = bs["kcs"][k]
    w = tc.from_kb8(bs["w"][bs["w_off"][k]: bs["w_off"][k] + kc * 208 * 8].view(1, kc, 208, 8), 196, 2 * core.band_split.subbands[k])
    assert torch.equal(w, core.band_split.fc[k].weight[:, :, 0].half().float())
    assert bs["w_off"][k + 1] - bs["w_off"][k] == kc * 208 * 8 and float(bs["bias"][k, 196:].abs().max()) == 0
    md = tc.pack_mask_decoder_tc(core.mask_decoder)
    for name in ("mlp_mask", "mlp_residual"):
        p = md[name]
        assert p["one_col"] == 196 and p["shared_norm"] and p["kc1"] == 26 and p["kc2"] == 98 and p["nt1"] == 4
        mlp = getattr(core.mask_decoder, name)[k]
        W, b = mlp[1].weight[:, :, 0].double(), mlp[1].bias.double()
        gamma, beta = mlp[0].weight.double(), mlp[0].bias.double()
        packed = tc.from_kb8(p["w1"][k], 4 * 196, 208).double()          # (784, 208): columns [0,196) weights, 196 bias
        assert float((packed[:, :196] - W * gamma[None, :]).abs().max()) < 2e-3 * float((W * gamma[None, :]).abs().max())
        assert float((packed[:, 196] - (b + W @ beta)).abs().max()) < 2e-3 * float((b + W @ beta).abs().max())
        assert float(packed[:, 197:].abs().max()) == 0
        z = torch.randn(5, 196, dtype=torch.float64)                     # the identity the fold relies on, on the packed operands
        ref = (z * gamma + beta) @ W.t() + b
        got = torch.cat([z, torch.ones(5, 1, dtype=torch.float64), torch.zeros(5, 11, dtype=torch.float64)], 1) @ packed.t()
        assert float((got - ref).abs().max()) < 5e-3 * float(ref.abs().max())


def _shard_worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, ROOT)
    from urgent2026_challenge_track1_b200.sharding import shard_utterances, gather_max_ms
    lengths = [480000, 120000, 480000, 96000, 240000, 240000, 64000]
    fss = [48000, 16000, 48000, 16000, 48000, 48000, 8000]
    mine = shard_utterances(lengths, fss, rank, world)
    ms = gather_max_ms(10.0 + rank)
    flat = sorted(i for _, idx in mine for i in idx)
    gathered = [None] * world
    dist.all_gather_object(gathered, flat)
    if rank == 0:
        out.put((gathered, ms, [fs for fs, _ in mine]))
    dist.destroy_process_group()


def test_utterance_sharding_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 200
    procs = [ctx.Process(target=_shard_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    gathered, ms, _ = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert sorted(gathered[0] + gathered[1]) == list(range(7))            # every utterance exactly once
    assert not set(gathered[0]) & set(gathered[1])
    assert ms == 11.0                                                      # max over ranks


def test_equal_length_batches_and_batch_split():
    """Default batching never pads (the reference is batch-1, inference.py:48-64): only equal-length utterances share
    a batch; a pad ratio relaxes that.  shard_batch is the contiguous 64/G split of BASELINE config 2."""
    from urgent2026_challenge_track1_b200.sharding import shard_utterances, shard_batch
    lengths = [1000, 900, 1000, 1000, 500, 900, 1000]
    fss = [16000] * 6 + [8000]
    got = shard_utterances(lengths, fss, 0, 1, max_batch=2)
    assert sorted(i for _, idx in got for i in idx) == list(range(7))
    for fs, idx in got:
        assert len(idx) <= 2 and len({lengths[i] for i in idx}) == 1 and len({fss[i] for i in idx}) == 1
    padded = shard_utterances(lengths, fss, 0, 1, max_batch=8, max_pad_ratio=0.15)
    assert [sorted(idx) for fs, idx in padded if fs == 16000] == [[0, 1, 2, 3, 5], [4]]
    for world in (1, 2, 3, 8):
        parts = [shard_batch(64, r, world) for r in range(world)]
        assert sum(c for _, c in parts) == 64 and parts[0][0] == 0
        assert all(parts[i][0] + parts[i][1] == parts[i + 1][0] for i in range(world - 1))
        assert max(c for _, c in parts) - min(c for _, c in parts) <= 1


def test_packed_cache_invalidation_paths():
    """ADVICE r1 (high): writers torch's version counter does not see -- the fused optimizer kernel and p.data.copy_ --
    must invalidate packed weights; the EMA swap must bump versions.  (Pure host logic: counts rebuilds.)"""
    from urgent2026_challenge_track1_b200 import runtime as R
    from urgent2026_challenge_track1_b200.ema import ExponentialMovingAverage
    lin = torch.nn.Linear(4, 4)
    builds = []
    cache = R.PackedCache(lin, lambda m: builds.append(1) or m.weight.detach().clone())
    cache.get(); cache.get()
    assert len(builds) == 1
    lin.weight.data.mul_(2.0)                            # invisible to _version ...
    cache.get()
    assert len(builds) == 1
    R.invalidate_packed()                                # ... so raw writers declare it
    assert torch.equal(cache.get(), lin.weight) and len(builds) == 2
    ema = ExponentialMovingAverage(lin.parameters(), decay=0.5)
    with torch.no_grad():
        lin.weight.add_(1.0)
    ema.update(lin.parameters())
    cache.get()
    n = len(builds)
    v0 = lin.weight._version
    ema.store(lin.parameters()); ema.copy_to(lin.parameters())
    assert lin.weight._version > v0 and torch.equal(cache.get(), lin.weight) and len(builds) == n + 1
    ema.restore(lin.parameters())
    assert torch.equal(cache.get(), lin.weight) and len(builds) == n + 2


def test_untouched_parameter_ranges():
    from urgent2026_challenge_track1_b200.training import FlatParams
    m = torch.nn.ModuleList([torch.nn.Linear(3, 2) for _ in range(4)])      # 8 params: (6, 2) x 4 = 32 elements
    fp = FlatParams(m)
    assert fp.untouched_ranges() == [[0, 32]]
    out = m[0](torch.ones(1, 3)).sum() + m[3](torch.ones(1, 3)).sum()
    out.backward()
    assert fp.untouched_ranges() == [[8, 24]]                                 # m[1], m[2] merged into one range
    assert float(fp.grad[:8].abs().sum()) > 0 and float(fp.grad[8:24].abs().sum()) == 0
    fp.zero_grad()
    assert fp.untouched_ranges() == [[0, 32]]


def _flow_cfg(**kw):
    from urgent2026_challenge_track1_b200.config import Config
    base = dict(model_type="flowse", ema_decay=0.999, sigma_max=0.5, sigma_min=0.05, t_eps=0.03, T_rev=1.0,
                loss_type="mse", loss_abs_exponent=0.5, n_fft=1536, hop_length=384, spec_transform_type="exponent",
                spec_abs_exponent=0.667, spec_factor=0.065, bsrnn_hidden=16, num_layer=1, learning_rate=1e-4)
    base.update(kw)
    return Config(**base)


def test_lightning_checkpoint_roundtrip(tmp_path):
    """Write a Lightning-format .ckpt (state_dict + pickled baseline_code.config.Config + ema) and read it back through
    the same-flags loaders; SEModel loader refuses a FlowSE file so inference.py's fallback (inference.py:30-33) works."""
    from urgent2026_challenge_track1_b200.checkpoint import save_checkpoint, load_checkpoint, model_kind
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.d_model import SEModel
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    cfg = Config(se_model="bsrnn", model_configs={"num_channel": 16, "num_layer": 1}, learning_rate=3e-4)
    m = SEModel(cfg)
    p = save_checkpoint(str(tmp_path / "se.ckpt"), m, cfg, global_step=123, epoch=4)
    sd, cfg2, raw = load_checkpoint(p)
    assert type(raw["hyper_parameters"]["cfg"]).__module__ == "baseline_code.config"     # what the reference unpickles
    assert raw["global_step"] == 123 and model_kind(sd) == "se" and cfg2.model_configs == cfg.model_configs
    m2 = SEModel.load_from_checkpoint(p, map_location="cpu")
    assert all(torch.equal(v, m2.state_dict()[k]) for k, v in m.state_dict().items())
    fcfg = _flow_cfg()
    fm = FlowSEModel(fcfg)
    with torch.no_grad():
        fm.dnn.condition_fc.bias.add_(1.0)
    fm.ema.update(fm.parameters())
    fp = save_checkpoint(str(tmp_path / "flow.ckpt"), fm, fcfg)
    with pytest.raises(KeyError):
        SEModel.load_from_checkpoint(fp, map_location="cpu")
    fm2 = FlowSEModel.load_from_checkpoint(fp, map_location="cpu")
    assert fm2.ema.num_updates == 1 and not fm2._error_loading_ema
    assert all(torch.equal(a, b) for a, b in zip(fm.ema.shadow_params, fm2.ema.shadow_params))
    live = fm2.dnn.condition_fc.bias.detach().clone()
    fm2.eval()                                                                  # EMA weights swapped in (flow_model.py:98-109)
    assert not torch.equal(fm2.dnn.condition_fc.bias, live)


@pytest.mark.reference
def test_checkpoints_interchange_with_the_verbatim_reference(tmp_path, ref_ns):
    """Our .ckpt loads into the reference's own SEModel / FlowSEModel classes (real Config class unpickled) and a
    checkpoint written from the reference's modules loads into ours."""
    from urgent2026_challenge_track1_b200.checkpoint import save_checkpoint, load_checkpoint
    from urgent2026_challenge_track1_b200.config import Config
    from urgent2026_challenge_track1_b200.d_model import SEModel
    from urgent2026_challenge_track1_b200.flow_model import FlowSEModel
    cfg = Config(se_model="bsrnn", model_configs={"num_channel": 16, "num_layer": 1})
    m = SEModel(cfg)
    p = save_checkpoint(str(tmp_path / "se.ckpt"), m, cfg)
    raw = torch.load(p, map_location="cpu", weights_only=False)
    rcfg = raw["hyper_parameters"]["cfg"]
    assert isinstance(rcfg, ref_ns.Config)
    rm = ref_ns.SEModel(rcfg)
    rm.load_state_dict(raw["state_dict"], strict=True)
    # reference -> ours (FlowSE incl. EMA)
    from oracle import ref_loader
    rfm = ref_ns.FlowSEModel(ref_loader.flowse_config(ref_ns, bsrnn_hidden=16, num_layer=1))
    ck = {"state_dict": rfm.state_dict(), "hyper_parameters": {"cfg": rfm.cfg}, "epoch": 0, "global_step": 0}
    rfm.on_save_checkpoint(ck)
    torch.save(ck, str(tmp_path / "ref_flow.ckpt"))
    fm = FlowSEModel.load_from_checkpoint(str(tmp_path / "ref_flow.ckpt"), map_location="cpu")
    assert all(torch.equal(v, fm.state_dict()[k]) for k, v in rfm.state_dict().items())
    sd, cfg2, _ = load_checkpoint(str(tmp_path / "ref_flow.ckpt"))
    assert cfg2.bsrnn_hidden == 16 and cfg2.n_fft == 1536
