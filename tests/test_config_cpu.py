"""Seam 3 + seam 4 plumbing on the CPU (no GPU, no arithmetic): the shipped `actionmesh_b200*.yaml` load through the same
mechanism the reference uses (hydra when installed, else the loader fallback in actionmesh_b200/config.py), every
`_target_` string resolves to a class with the constructor arguments the YAML passes, the fast preset inherits through
`defaults:`, `${...}` interpolations resolve, and ActionMeshB200Pipeline keeps the reference's constructor / __call__
signature (actionmesh/pipeline.py:47-53,602-613) and override plumbing (:637-648)."""
import inspect
import json
import os

import pytest
import torch

from actionmesh_b200 import AmbError
from actionmesh_b200.config import DEFAULT_CONFIG_DIR, get_target, instantiate, load_config


def test_default_yaml_resolves_and_instantiates():
    cfg = load_config("actionmesh_b200.yaml", DEFAULT_CONFIG_DIR)
    assert cfg.stage_1_steps == 30 and cfg.stage_0_steps == 100 and list(cfg.guidance_scales) == [7.5]
    assert list(cfg.denoiser_latent_shape) == [2048, 64]                       # ${model.temporal_3D_denoiser....}
    assert cfg.model.scheduler.num_inference_steps == 30                       # ${stage_1_steps}
    sch = instantiate(cfg.model.scheduler, _convert_="partial")()             # _partial_ then call, like pipeline.py:103-110
    cf = instantiate(cfg.model.cf_guidance, _convert_="partial")()
    from actionmesh_b200.guidance import ClassifierFreeGuidance
    from actionmesh_b200.scheduler import B200SchedulerFlow

    assert isinstance(sch, B200SchedulerFlow) and (sch.num_inference_steps, sch.shift, sch.is_additive) == (30, 3.0, True)
    assert isinstance(cf, ClassifierFreeGuidance) and cf.branches() == [(0, 1), (1, 1)] and list(cf.guidance_scales) == [7.5]
    ts, ds = sch.get_schedule()
    assert ts.shape == (31,) and ds.shape == (30,)
    # model targets: constructed from the YAML's keyword arguments (weights come later through from_pretrained / load_state_dict)
    den = instantiate(cfg.model.temporal_3D_denoiser, _convert_="partial")()
    assert den.config.num_layers == 21 and den.config.width == 2048 and den.config.head_dim == 128
    vae = instantiate(cfg.model.temporal_3D_vae, _convert_="partial")()
    assert vae.config.width == 1024 and vae.config.num_layers == 16
    for key in ("temporal_3D_denoiser", "temporal_3D_vae", "image_encoder"):
        cls = get_target(cfg.model[key]["_target_"])
        assert hasattr(cls, "to") and hasattr(cls, "eval")
    # the encoder refuses a checkpoint path that is not a local directory (no silent fall-back)
    with pytest.raises(AmbError):
        instantiate(cfg.model.image_encoder, _convert_="partial")()
    enc = instantiate(cfg.model.image_encoder, pretrained_dino_feature_extractor=None, pretrained_dino_model=None)()
    assert hasattr(enc, "encode_images")


def test_fast_preset_inherits_and_overrides():
    cfg = load_config("actionmesh_b200_fast.yaml", DEFAULT_CONFIG_DIR)
    assert cfg.stage_1_steps == 15 and cfg.stage_0_steps == 50
    assert cfg.model.scheduler.num_inference_steps == 15 and cfg.model.image_to_3D_denoiser.num_inference_steps == 50
    assert cfg.model.scheduler["_target_"] == "actionmesh_b200.scheduler.B200SchedulerFlow"      # inherited block
    cfg2 = load_config("actionmesh_b200.yaml", DEFAULT_CONFIG_DIR, updates={"stage_1_steps": 4, "guidance_scales": [3.0]})
    assert cfg2.model.scheduler.num_inference_steps == 4 and list(cfg2.model.cf_guidance.guidance_scales) == [3.0]


def test_yaml_keeps_the_reference_keys(golden_dir):
    """Same key tree as the reference's YAML (only `_target_` values differ), checked with the same loader.  The
    reference side (actionmesh.yaml / actionmesh_fast.yaml loaded by load_config) is stored by oracle/gen_golden.py."""
    with open(os.path.join(golden_dir, "reference_config.json")) as f:
        ref = json.load(f)
    ours = load_config("actionmesh_b200.yaml", DEFAULT_CONFIG_DIR)

    def keys(node, prefix=""):
        out = set()
        for k, v in node.items():
            out.add(prefix + k)
            if isinstance(v, dict):
                out |= keys(v, prefix + k + ".")
        return out

    missing = set(ref["key_paths"]) - keys(ours) - {"model.temporal_3D_denoiser.clear_autocast"}  # autocast-cache knob has no meaning here
    assert not missing, missing
    assert sorted(ref["values"]) == ["anchor_idx", "face_decimation", "floaters_threshold", "sliding_window_autoencoder",
                                     "sliding_window_denoiser", "stage_0_steps", "stage_1_steps", "subsampling_level"]
    for k, v in ref["values"].items():
        assert ours[k] == v, k
    for blk in ("scheduler", "cf_guidance"):
        assert ref["model_blocks"][blk]
        for k, v in ref["model_blocks"][blk].items():
            assert ours.model[blk][k] == v, (blk, k)
    assert ref["fast"] == {"stage_1_steps": 15, "scheduler.num_inference_steps": 15}   # the loader handles `defaults:`


def test_pipeline_signature_and_override_plumbing():
    from actionmesh_b200.pipeline import ActionMeshB200Pipeline, ActionMeshInput

    sig = inspect.signature(ActionMeshB200Pipeline.__call__)
    assert list(sig.parameters)[1:] == ["input", "seed", "stage_0_steps", "face_decimation", "floaters_threshold",
                                        "stage_1_steps", "guidance_scales", "anchor_idx"]     # pipeline.py:602-613
    assert sig.parameters["seed"].default == 44
    init = inspect.signature(ActionMeshB200Pipeline.__init__)
    assert list(init.parameters)[1:5] == ["config_name", "config_dir", "dtype", "lazy_loading"]  # pipeline.py:47-53
    pipe = ActionMeshB200Pipeline("actionmesh_b200.yaml", lazy_loading=True)
    assert pipe._denoiser_latent_shape == (2048, 64) and pipe.scheduler.num_inference_steps == 30
    with pytest.raises(AmbError):
        pipe.to("cpu")
    frames = [object()] * 16
    inp = ActionMeshInput(frames, torch.arange(16, dtype=torch.float32))
    with pytest.raises(AssertionError):
        ActionMeshInput(frames[:8], torch.arange(8, dtype=torch.float32))               # video_input.py:40-43
    # overrides mutate the live objects before any stage runs; Stage 0 is an injected component
    with pytest.raises(AmbError, match="Stage 0"):
        pipe(inp, seed=1, stage_0_steps=7, face_decimation=123, floaters_threshold=0.5, stage_1_steps=9,
             guidance_scales=[2.0], anchor_idx=3)
    assert pipe.scheduler.num_inference_steps == 9 and pipe.cf_guidance.guidance_scales == [2.0]
    assert pipe.mesh_process.face_decimation == 123 and pipe.mesh_process.floaters_threshold == 0.5
    assert pipe.cfg.anchor_idx == 3 and pipe.cfg.model.image_to_3D_denoiser.num_inference_steps == 7
