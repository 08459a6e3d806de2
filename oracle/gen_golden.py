"""TEST INFRASTRUCTURE ONLY — regenerate tests/golden/* from the reference's OWN modules (needs the reference checkout).

    python -m oracle.gen_golden

Runs facebookresearch/actionmesh's unmodified `ActionMeshDenoiser`, `SchedulerFlow`, `ClassifierFreeGuidance`,
`chunk_from`, `compute_rotary_embeddings`, `LatentBank` (imported from /root/reference on top of oracle/diffusers_shim.py)
on seeded inputs and stores inputs + outputs.  Weights are NOT stored: they are re-derived from (config, seed) by
oracle/synth.py, and loaded into the reference module with strict=True (which also pins the state-dict key names).
"""
from __future__ import annotations

import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import reference_loader, synth  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

TINY = dict(num_layers=5, num_attention_heads=2, width=256, cross_attention_dim=128, in_channels=64, mlp_ratio=4.0)


class TINY_CFG:
    """Attribute view of TINY for oracle/synth.py."""
    in_channels, num_layers, num_attention_heads, width, mlp_ratio, cross_attention_dim = 64, 5, 2, 256, 4.0, 128


MULTI_SEEDS = [(1234, 5), (11, 21), (12, 22), (13, 23), (14, 24), (15, 25), (16, 26), (17, 27)]
WIDE = dict(num_layers=3, num_attention_heads=16, width=2048, cross_attention_dim=1024, in_channels=64, mlp_ratio=4.0)


def _model(ns, cfgd, seed):
    m = ns.ActionMeshDenoiser(inflated_layers=tuple(range(cfgd["num_layers"])), **cfgd).eval()
    sd = synth.make_state_dict(m, seed)
    m.load_state_dict(sd, strict=True)
    return m


def main():
    ns = reference_loader.load()
    os.makedirs(GOLD, exist_ok=True)
    torch.set_grad_enabled(False)

    # ---- known answers for host logic (SURVEY Appendix B)
    host = {"schedule": {}, "chunk_from": {}}
    for n in (4, 15, 30):
        ts, ds = ns.SchedulerFlow(num_inference_steps=n, shift=3.0).get_schedule()
        host["schedule"][n] = (ts, ds)
    g = torch.Generator().manual_seed(44)
    noise = ns.SchedulerFlow(num_inference_steps=4).get_noise([2048, 64], 1, 16, "cpu", g)
    host["noise_seed44_head"] = noise[0, :2, :4, :8].clone()
    host["noise_seed44_stats"] = (float(noise.mean()), float(noise.std()))
    for args in ((0, 16, 16, 15), (0, 31, 16, 15), (0, 32, 16, 15), (0, 256, 16, 15), (5, 31, 16, 15), (30, 31, 16, 15),
                 (7, 16, 16, 15), (20, 47, 16, 15), (0, 8, 16, 15)):
        host["chunk_from"][args] = ns.chunk_from(*args)
    cos, sin = ns.compute_rotary_embeddings(128, torch.arange(16.0))
    host["rope_cos"], host["rope_sin"] = cos, sin
    x = torch.randn(2, 3, 5, 128, generator=torch.Generator().manual_seed(1))
    host["rope_apply_in"] = x
    host["rope_apply_out"] = ns.apply_rotary_embedding(x, cos[:5], sin[:5])
    cf = ns.ClassifierFreeGuidance(guidance_at_inference=[[0, 1], [1, 1]], guidance_scales=[7.5])
    p = torch.randn(2, 3, 4, 8, generator=torch.Generator().manual_seed(2))
    host["cfg_in"] = p.clone()
    host["cfg_out"] = cf.aggregate_cfg(p.clone())
    bank = ns.LatentBank(empty_dims=(4, 2))
    bank.update(torch.tensor([3.0]), torch.ones(1, 4, 2))
    lat, msk = bank.get(torch.tensor([2.0, 3.0, 4.0]), "cpu", add_batch_dim=True)
    host["bank_get"] = (lat, msk)
    torch.save(host, os.path.join(GOLD, "host_logic.pt"))

    # ---- Stage-II time bookkeeping (reference embeddings.py:156-242, imported unchanged)
    E = ns.embeddings
    s2 = {"n_subdivisions": {(a, b, l): E.get_n_subdivisions(a, b, l) for a, b, l in ((0, 15, 1), (0.0, 15.0, 2), (3, 18, 3), (5.0, 5.0, 1))},
          "interp": {}, "scaling": {}}
    for name, ts in (("w16", torch.arange(16.0)[None]), ("w16_off", torch.arange(15.0, 31.0)[None]), ("w5", torch.tensor([[2.0, 3.0, 4.0, 5.0, 6.0]]))):
        for lvl in (1, 2):
            for df in (False, True):
                s2["interp"][(name, lvl, df)] = E.interpolate_timesteps(ts, subsampling_level=lvl, device="cpu", drop_first=df)
        t_min, t_range = E.get_scaling(ts)
        s2["scaling"][name] = (ts, t_min, t_range, E.apply_scaling(ts[:, 0], t_min, t_range), E.apply_scaling(ts, t_min, t_range))
    torch.save(s2, os.path.join(GOLD, "stage2_host_logic.pt"))

    # ---- tiny denoiser: forward + 4-step CFG denoise through the reference scheduler
    m = _model(ns, TINY, 1234)
    lat, ctx, fs, mask = synth.make_inputs(1, 3, 31, 64, 9, 128, seed=5)
    cfg_b = ns.ClassifierFreeGuidance(guidance_at_inference=[[0, 1], [1, 1]], guidance_scales=[7.5])
    h_in, c_in, m_in, f_in = cfg_b.cfg_at_inference(lat, ctx, mask, fs)
    t = torch.tensor([751.1210938, 751.1210938])
    out, _ = m.forward(hidden_states=h_in, context=c_in, framestep=f_in, diffusion_time=t, mask=m_in)
    sch = ns.SchedulerFlow(num_inference_steps=4, shift=3.0, is_additive=True)
    den = sch.denoise(m, cfg_b, lat.clone(), ctx, device="cpu", mask=mask, framestep=fs)
    # non-inflated variant (per-frame self-attention) and no-mask variant
    m2 = ns.ActionMeshDenoiser(inflated_layers=(0, 2, 4), **TINY).eval()
    m2.load_state_dict(synth.make_state_dict(m2, 1234), strict=True)
    out2, _ = m2.forward(hidden_states=h_in, context=c_in, framestep=f_in, diffusion_time=t, mask=None)
    torch.save({"config": TINY, "seed": 1234, "input_seed": 5, "forward_out": out, "denoise4_out": den,
                "forward_out_partial_inflate_nomask": out2, "t": t},
               os.path.join(GOLD, "denoiser_tiny.pt"))

    # ---- the same 4-step trajectory under the reference's OWN mixed-precision recipe (pipeline.py:671 wraps the stages in
    # torch.autocast(bf16)); run here with device_type="cpu" (same autocast op policy: linear/matmul/SDPA in bf16,
    # layer_norm in fp32).  Yardstick for "how far is a bf16 path allowed to be from the fp32 path" in the Chamfer test.
    with torch.autocast(device_type="cpu", dtype=torch.bfloat16):
        den_ac = sch.denoise(m, cfg_b, lat.clone(), ctx, device="cpu", mask=mask, framestep=fs)
    torch.save({"config": TINY, "seed": 1234, "input_seed": 5, "denoise4_out_autocast_bf16": den_ac.float(),
                "rel_err_vs_fp32": float((den_ac.float()[0, 1:] - den[0, 1:]).norm() / den[0, 1:].norm())},
               os.path.join(GOLD, "denoiser_tiny_autocast.pt"))

    # ---- the same pair of trajectories (fp32 and the reference's bf16 autocast recipe) for 8 (weight seed, input seed)
    # draws: tests/test_chamfer_gpu.py compares the B200 path's Chamfer with the reference-autocast Chamfer in the MEAN
    multi = {"config": TINY, "pairs": []}
    for ws, isd in MULTI_SEEDS:
        mm = _model(ns, TINY, ws)
        lat_m, ctx_m, fs_m, mask_m = synth.make_inputs(1, 3, 31, 64, 9, 128, seed=isd)
        d32 = sch.denoise(mm, cfg_b, lat_m.clone(), ctx_m, device="cpu", mask=mask_m, framestep=fs_m)
        with torch.autocast(device_type="cpu", dtype=torch.bfloat16):
            dac = sch.denoise(mm, cfg_b, lat_m.clone(), ctx_m, device="cpu", mask=mask_m, framestep=fs_m)
        multi["pairs"].append({"seed": ws, "input_seed": isd, "denoise4_out": d32[0, 1:].clone(),
                               "denoise4_out_autocast_bf16": dac.float()[0, 1:].clone()})
    torch.save(multi, os.path.join(GOLD, "denoiser_tiny_multiseed.pt"))

    # ---- full-width 3-layer model (covers the skip block at D=2048, 16 heads, F=8192, Dc=1024)
    mw = _model(ns, WIDE, 77)
    lat, ctx, fs, mask = synth.make_inputs(1, 2, 255, 64, 257, 1024, seed=6)
    h_in, c_in, m_in, f_in = cfg_b.cfg_at_inference(lat, ctx, mask, fs)
    t = torch.tensor([502.9850769, 502.9850769])
    outw, _ = mw.forward(hidden_states=h_in, context=c_in, framestep=f_in, diffusion_time=t, mask=m_in)
    torch.save({"config": WIDE, "seed": 77, "input_seed": 6, "forward_out": outw, "t": t},
               os.path.join(GOLD, "denoiser_wide3.pt"))
    # ---- Stage-II decoder (test-side only: turns latents into vertices for the Chamfer metric) + ActionBench Chamfer
    import importlib.util

    from actionmesh.model.temporal_autoencoder import ActionMeshAutoencoder
    from oracle import autoencoder_oracle as ao

    acfg = dict(width=256, num_layers=2, num_attention_heads=2)
    ae = ActionMeshAutoencoder(verbose=False, **acfg).eval()
    ae.load_state_dict(ao.make_autoencoder_state_dict(ao.AutoencoderConfig(**acfg), 4321), strict=True)
    gg = torch.Generator().manual_seed(0)
    lat = torch.randn(1, 3, 7, 64, generator=gg)
    fsx = torch.tensor([[2.0, 3.0, 4.0]])
    sa, ta = torch.tensor([0.0]), torch.tensor([[0.0, 0.5, 1.0]])
    qv = torch.rand(1, 50, 6, generator=gg) * 2 - 1
    disp = ae.forward(lat, fsx, sa, ta, qv)
    spec = importlib.util.spec_from_file_location("ref_chamfer", os.path.join(reference_loader.REFERENCE_ROOT, "actionbench", "chamfer.py"))
    ch = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ch)
    pa, pb = torch.rand(500, 3, generator=gg).numpy(), torch.rand(600, 3, generator=gg).numpy()
    torch.save({"config": acfg, "seed": 4321, "latent": lat, "framestep": fsx, "source_alpha": sa, "target_alphas": ta,
                "query": qv, "displacement": disp, "chamfer_a": pa, "chamfer_b": pb,
                "chamfer_n300": ch.compute_chamfer_score(pa, pb, n=300), "chamfer_all": ch.compute_chamfer_score(pa, pb, n=0)},
               os.path.join(GOLD, "autoencoder_tiny.pt"))

    # ---- Stage 0: the vendored TripoSG DiT + RectifiedFlowScheduler (third_party/TripoSG, imported unchanged), tiny width:
    # one forward and a 4-step CFG-2.0 denoising loop as TripoSGPipeline.__call__ drives them (pipeline_triposg.py:243-294)
    tns = reference_loader.load_triposg()
    tri = tns.TripoSGDiTModel(num_attention_heads=2, width=256, in_channels=64, num_layers=5, cross_attention_dim=128).eval()
    tsd = synth.make_state_dict(TINY_CFG(), 4242)
    from oracle import triposg_oracle as tro

    inv = tro.remap_state_dict({k: k for k in tri.state_dict()})  # ActionMesh key name -> TripoSG key name
    tri.load_state_dict({inv[k]: v for k, v in tsd.items()}, strict=True)
    gg = torch.Generator().manual_seed(31)
    x0 = torch.randn(1, 31, 64, generator=gg)
    emb = torch.randn(1, 9, 128, generator=gg)
    tt = torch.tensor([750.0, 750.0])
    fwd = tri(torch.cat([x0, x0]), tt, encoder_hidden_states=torch.cat([torch.zeros_like(emb), emb]), return_dict=False)[0]
    sched = tns.RectifiedFlowScheduler(num_train_timesteps=1000, shift=3.0)
    sched.set_timesteps(4)
    lat = x0.clone()
    for t in sched.timesteps:
        pred = tri(torch.cat([lat, lat]), t.expand(2), encoder_hidden_states=torch.cat([torch.zeros_like(emb), emb]),
                   return_dict=False)[0]
        unc, img = pred.chunk(2)
        lat = sched.step(unc + 2.0 * (img - unc), t, lat, return_dict=False)[0]
    torch.save({"config": TINY, "seed": 4242, "x0": x0, "image_embeds": emb, "t": tt, "forward_out": fwd, "shift": 3.0,
                "timesteps": sched.timesteps.clone(), "sigmas": sched.sigmas.clone(), "denoise4_cfg2_out": lat,
                "state_dict_keys": sorted(tri.state_dict().keys())}, os.path.join(GOLD, "triposg_tiny.pt"))

    reference_outputs(ns, tns)
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))


def _key_paths(node, prefix=""):
    out = []
    for k, v in node.items():
        out.append(prefix + k)
        if isinstance(v, dict):
            out += _key_paths(v, prefix + k + ".")
    return out


def reference_outputs(ns, tns):
    """Fixtures for the tests that compare against the reference's shipped YAML configs, its ImagePreprocessor, a small
    ActionMeshDenoiser forward + chunk_from, and TripoSG's RectifiedFlowScheduler schedules."""
    import importlib.util
    import json

    import numpy as np
    from PIL import Image

    from actionmesh_b200.config import load_config

    # ---- YAML configs, through the project's own loader: the key tree and the values the B200 presets must keep
    cdir = os.path.join(reference_loader.REFERENCE_ROOT, "actionmesh", "configs")
    ref, fast = load_config("actionmesh.yaml", cdir), load_config("actionmesh_fast.yaml", cdir)
    top = ("stage_0_steps", "face_decimation", "floaters_threshold", "stage_1_steps", "anchor_idx", "sliding_window_denoiser",
           "subsampling_level", "sliding_window_autoencoder")
    conf = {"key_paths": sorted(_key_paths(ref)),
            "values": {k: ref[k] for k in top},
            "model_blocks": {b: {k: v for k, v in ref.model[b].items() if k != "_target_"} for b in ("scheduler", "cf_guidance")},
            "fast": {"stage_1_steps": fast.stage_1_steps, "scheduler.num_inference_steps": fast.model.scheduler.num_inference_steps}}
    with open(os.path.join(GOLD, "reference_config.json"), "w") as f:
        json.dump(conf, f, indent=1, sort_keys=True)
        f.write("\n")

    # ---- ImagePreprocessor.process_images (loaded by file path) on the seeded RGBA frames
    spec = importlib.util.spec_from_file_location(
        "ref_image_processor", os.path.join(reference_loader.REFERENCE_ROOT, "actionmesh", "preprocessing", "image_processor.py"))
    ip = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ip)
    frames = [Image.fromarray(f, "RGBA") for f in synth.make_rgba_frames()]
    outs = {}
    for ind in (False, True):
        done = ip.ImagePreprocessor(independent_cropping=ind, padding_ratio=0.1).process_images(frames)
        outs.update({f"independent{int(ind)}_frame{i}": np.asarray(im) for i, im in enumerate(done)})
    np.savez_compressed(os.path.join(GOLD, "frame_preprocess.npz"), **outs)

    # ---- a 3-layer ActionMeshDenoiser forward (batch of 2, frame 1 observed, no CFG batch); the chunk_from grid
    d = dict(num_layers=3, num_attention_heads=2, width=256, cross_attention_dim=64, in_channels=64, mlp_ratio=2.0)
    m = ns.ActionMeshDenoiser(inflated_layers=(0, 1, 2), **d).eval()
    m.load_state_dict(synth.make_state_dict(m, 9), strict=True)
    lat, ctx, fs, mask = synth.make_inputs(2, 4, 7, 64, 5, 64, seed=11, observed=(1,))
    t = torch.tensor([300.0, 300.0])
    with torch.no_grad():
        out, _ = m.forward(hidden_states=lat, context=ctx, framestep=fs, diffusion_time=t, mask=mask)
    chunks = {(start, total): ns.chunk_from(start, total, 16, 15)
              for total in (16, 17, 31, 32, 47, 64) for start in (0, 3, total // 2, total - 1)}
    torch.save({"config": d, "seed": 9, "input_seed": 11, "t": t, "forward_out": out,
                "state_dict_keys": sorted(m.state_dict().keys()), "chunk_from": chunks},
               os.path.join(GOLD, "denoiser_small3.pt"))

    # ---- TripoSG RectifiedFlowScheduler.set_timesteps
    sch = {}
    for n, shift in ((50, 1.0), (100, 3.0), (7, 2.5)):
        s = tns.RectifiedFlowScheduler(num_train_timesteps=1000, shift=shift)
        s.set_timesteps(n)
        sch[(n, shift)] = (s.timesteps.clone(), s.sigmas.clone())
    torch.save(sch, os.path.join(GOLD, "triposg_schedules.pt"))


if __name__ == "__main__":
    main()
