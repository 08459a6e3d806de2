"""Pins oracle/denoiser_oracle.py (the fp32 restatement the GPU tests compare against) against the golden fixtures that
oracle/gen_golden.py produced from the reference's OWN modules.  CPU only."""
import torch

from conftest import load_golden
from oracle import denoiser_oracle as do
from oracle import synth


def _cfg(d):
    return do.DenoiserConfig(inflated_layers=tuple(range(d["num_layers"])), **d)


def test_schedule_known_answers():
    host = load_golden("host_logic.pt")
    for n, (ts, ds) in host["schedule"].items():
        ots, ods = do.flow_schedule(n)
        assert torch.equal(ots, ts) and torch.equal(ods, ds)
    ts, ds = do.flow_schedule(4)
    # SURVEY Appendix B (values printed by the reference's SchedulerFlow)
    assert torch.allclose(ts, torch.tensor([1000.0, 900.3590698, 751.1210938, 502.9850769, 8.9285717]), atol=1e-4)
    assert abs(float(ds.sum()) - 0.9910714626) < 1e-6


def test_noise_stream_order():
    host = load_golden("host_logic.pt")
    g = torch.Generator().manual_seed(44)
    n = do.flow_noise([2048, 64], 1, 16, g)
    assert torch.equal(n[0, :2, :4, :8], host["noise_seed44_head"])
    assert abs(float(n[0, 0, 0, 0]) - (-0.0826127529)) < 1e-7


def test_chunk_from_partitions():
    host = load_golden("host_logic.pt")
    for args, ref in host["chunk_from"].items():
        got = do.chunk_from(*args)
        assert len(got) == len(ref)
        for a, b in zip(got, ref):
            assert torch.equal(a, b), args
    assert len(do.chunk_from(0, 256, 16, 15)) == 17 and len(do.chunk_from(0, 32, 16, 15)) == 3


def test_rope_and_cfg_and_bank():
    host = load_golden("host_logic.pt")
    cos, sin = do.rotary_tables(128, torch.arange(16.0))
    assert torch.equal(cos, host["rope_cos"]) and torch.equal(sin, host["rope_sin"])
    x = host["rope_apply_in"]
    out = do.apply_rotary(x, cos[:5][None].expand(2, -1, -1), sin[:5][None].expand(2, -1, -1))
    assert torch.allclose(out, host["rope_apply_out"], atol=1e-6)
    assert torch.allclose(do.cfg_aggregate(host["cfg_in"], [7.5], 2), host["cfg_out"], atol=1e-5)
    bank = do.LatentBank(empty_dims=(4, 2))
    bank.update(torch.tensor([3.0]), torch.ones(1, 4, 2))
    lat, msk = bank.get(torch.tensor([2.0, 3.0, 4.0]), add_batch_dim=True)
    assert torch.equal(lat, host["bank_get"][0]) and torch.equal(msk, host["bank_get"][1])


def test_tiny_denoiser_forward_and_denoise_match_reference_outputs():
    g = load_golden("denoiser_tiny.pt")
    cfg = _cfg(g["config"])
    model = do.OracleDenoiser(synth.make_state_dict(cfg, g["seed"]), cfg)
    lat, ctx, fs, mask = synth.make_inputs(1, 3, 31, 64, 9, 128, seed=g["input_seed"])
    h, c, m, f = do.cfg_batch(lat, ctx, mask, fs, ((0, 1), (1, 1)))
    out, _ = model.forward(h, c, f, g["t"], m)
    assert (out - g["forward_out"]).abs().max() < 2e-5
    den = do.flow_denoise(model, lat, ctx, mask, fs, num_inference_steps=4, guidance_scales=[7.5])
    assert (den - g["denoise4_out"]).abs().max() < 2e-4
    assert torch.equal(den[0, 0], lat[0, 0])  # observed frame untouched
    cfg2 = do.DenoiserConfig(inflated_layers=(0, 2, 4), **g["config"])
    model2 = do.OracleDenoiser(synth.make_state_dict(cfg2, g["seed"]), cfg2)
    out2, _ = model2.forward(h, c, f, g["t"], None)
    assert (out2 - g["forward_out_partial_inflate_nomask"]).abs().max() < 2e-5


def test_wide3_forward_matches_reference_output():
    g = load_golden("denoiser_wide3.pt")
    cfg = _cfg(g["config"])
    model = do.OracleDenoiser(synth.make_state_dict(cfg, g["seed"]), cfg)
    lat, ctx, fs, mask = synth.make_inputs(1, 2, 255, 64, 257, 1024, seed=g["input_seed"])
    h, c, m, f = do.cfg_batch(lat, ctx, mask, fs, ((0, 1), (1, 1)))
    out, _ = model.forward(h, c, f, g["t"], m)
    assert (out - g["forward_out"]).abs().max() < 5e-5


def test_stage2_decoder_and_chamfer_match_reference_outputs():
    """The test-side Stage-II decoder (latents -> vertex displacements) and the Chamfer metric restatement reproduce the
    reference's ActionMeshAutoencoder.forward and actionbench/chamfer.py outputs stored in the fixture."""
    from oracle import autoencoder_oracle as ao

    g = load_golden("autoencoder_tiny.pt")
    cfg = ao.AutoencoderConfig(**g["config"])
    sd = ao.make_autoencoder_state_dict(cfg, g["seed"])
    out = ao.autoencoder_forward(sd, cfg, g["latent"], g["framestep"], g["source_alpha"], g["target_alphas"], g["query"])
    assert out.shape == g["displacement"].shape and (out - g["displacement"]).abs().max() < 1e-5
    assert abs(ao.chamfer_score(g["chamfer_a"], g["chamfer_b"], n=300) - g["chamfer_n300"]) < 1e-12
    assert abs(ao.chamfer_score(g["chamfer_a"], g["chamfer_b"], n=0) - g["chamfer_all"]) < 1e-12
    assert ao.chamfer_score(g["chamfer_a"], g["chamfer_a"], n=0) == 0.0


def test_oracle_matches_live_reference_modules():
    """The reference's ActionMeshDenoiser forward on a batch of 2 with an observed frame and no CFG batch, its state-dict
    key names (SURVEY A.1) and its chunk_from over a grid of window starts, as stored by oracle/gen_golden.py."""
    g = load_golden("denoiser_small3.pt")
    d = g["config"]
    cfg = do.DenoiserConfig(inflated_layers=(0, 1, 2), **d)
    sd = synth.make_state_dict(cfg, g["seed"])
    assert sorted(sd) == g["state_dict_keys"]
    lat, ctx, fs, mask = synth.make_inputs(2, 4, 7, 64, 5, 64, seed=g["input_seed"], observed=(1,))
    out, _ = do.OracleDenoiser(sd, cfg).forward(lat, ctx, fs, g["t"], mask)
    assert (out - g["forward_out"]).abs().max() < 2e-5
    assert len(g["chunk_from"]) == 24
    for (start, total), a in g["chunk_from"].items():
        b = do.chunk_from(start, total, 16, 15)
        assert len(a) == len(b) and all(torch.equal(x, y) for x, y in zip(a, b)), (start, total)
