"""Stage 0 (TripoSG DiT + rectified-flow sampler) on the CPU: the oracle restatement and the host-side mirrors against
the fixtures written by the reference's own TripoSGDiTModel / RectifiedFlowScheduler (tests/golden/triposg_tiny.pt,
tests/golden/triposg_schedules.pt, oracle/gen_golden.py)."""
import pytest
import torch

from conftest import load_golden
from oracle import denoiser_oracle as do
from oracle import synth
from oracle import triposg_oracle as tro


class _TinyCfg:
    in_channels, num_layers, num_attention_heads, width, mlp_ratio, cross_attention_dim = 64, 5, 2, 256, 4.0, 128


def _setup():
    g = load_golden("triposg_tiny.pt")
    cfg = do.DenoiserConfig(inflated_layers=(), **g["config"])
    return g, cfg, synth.make_state_dict(_TinyCfg(), g["seed"])


def test_oracle_matches_reference_triposg_forward_and_loop():
    g, cfg, sd = _setup()
    emb2 = torch.cat([torch.zeros_like(g["image_embeds"]), g["image_embeds"]])
    out = tro.dit_forward(sd, cfg, torch.cat([g["x0"], g["x0"]]), g["t"], emb2)
    assert float((out - g["forward_out"]).abs().max()) < 1e-4
    lat = tro.stage0_denoise(sd, cfg, g["image_embeds"], g["x0"], num_inference_steps=4, guidance_scale=2.0, shift=g["shift"])
    assert float((lat - g["denoise4_cfg2_out"]).abs().max()) < 1e-4
    ts, sig = tro.rectified_flow_sigmas(4, shift=g["shift"])
    assert torch.equal(ts, g["timesteps"]) and torch.equal(sig, g["sigmas"])


def test_key_remap_covers_the_reference_state_dict():
    from actionmesh_b200.stage0 import remap_triposg_state_dict

    g, cfg, sd = _setup()
    mapped = remap_triposg_state_dict({k: 0 for k in g["state_dict_keys"]})          # the reference's own key names
    assert set(mapped) == set(sd)                                                     # == the ActionMeshDenoiser key set
    assert set(tro.remap_state_dict({k: 0 for k in g["state_dict_keys"]})) == set(sd)


def test_scheduler_mirror_matches_reference_values():
    from actionmesh_b200.stage0 import B200RectifiedFlowScheduler, _Stage0Flow

    g, _, _ = _setup()
    s = B200RectifiedFlowScheduler(num_train_timesteps=1000, shift=g["shift"])
    s.set_timesteps(4)
    assert torch.equal(s.timesteps, g["timesteps"]) and torch.equal(s.sigmas, g["sigmas"])
    x = torch.randn(1, 5, 3)
    v = torch.randn(1, 5, 3)
    y = x
    for i, t in enumerate(s.timesteps):
        y = s.step(v, t, y, return_dict=False)[0]
        assert s.step_index == i + 1
    assert torch.allclose(y, x + float(g["sigmas"][0]) * v, atol=1e-6)                # the steps sum to sigma_0 - 0
    with pytest.raises(ValueError):
        s.step(v, 3, x)
    ts, ds = _Stage0Flow(num_inference_steps=4, shift=g["shift"], is_additive=True).get_schedule()
    assert torch.equal(ts[:-1], g["timesteps"]) and torch.allclose(ds, g["sigmas"][:-1] - g["sigmas"][1:])


def test_live_reference_scheduler_matches_mirror():
    """Against RectifiedFlowScheduler.set_timesteps of the reference's TripoSG (tests/golden/triposg_schedules.pt)."""
    from actionmesh_b200.stage0 import B200RectifiedFlowScheduler

    ref = load_golden("triposg_schedules.pt")
    assert sorted(ref) == [(7, 2.5), (50, 1.0), (100, 3.0)]
    for (n, shift), (ref_timesteps, ref_sigmas) in ref.items():
        ours = B200RectifiedFlowScheduler(num_train_timesteps=1000, shift=shift)
        ours.set_timesteps(n)
        assert torch.equal(ours.timesteps, ref_timesteps) and torch.equal(ours.sigmas, ref_sigmas)
