"""TEST INFRASTRUCTURE ONLY.  Import the reference's OWN hot-path modules unchanged from a checkout of
facebookresearch/actionmesh (path in $ACTIONMESH_REFERENCE).

Used only by gen_golden.py, which stores the outputs of these modules under tests/golden/; the tests read those
fixtures and never need the checkout.
"""
from __future__ import annotations

import os
import sys
import types

REFERENCE_ROOT = os.environ.get("ACTIONMESH_REFERENCE", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "actionmesh"))


def load():
    """Returns a namespace with the reference classes/functions on the hot path."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REFERENCE_ROOT}")
    from . import diffusers_shim

    diffusers_shim.install()
    if "trimesh" not in sys.modules:  # storage.py:13 imports trimesh only for MeshBank typing
        try:
            import trimesh  # noqa: F401
        except Exception:  # noqa: BLE001
            tm = types.ModuleType("trimesh")
            tm.Trimesh = type("Trimesh", (), {})
            tm._AMB_SHIM = True
            sys.modules["trimesh"] = tm
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import torch

    # AttentionProcessor.__init__ checks torch.backends.cuda.flash_sdp_enabled(); True on CPU builds too.
    from actionmesh.model.temporal_denoiser import ActionMeshDenoiser
    from actionmesh.model.utils.attention_processor import AttentionProcessor
    from actionmesh.model.utils.block import FlowMatchingBlock
    from actionmesh.model.utils import embeddings as ref_embeddings
    from actionmesh.model.utils.rotary_embedding import apply_rotary_embedding, compute_rotary_embeddings
    from actionmesh.model.utils.storage import LatentBank
    from actionmesh.model.utils.timesteps import chunk_from
    from actionmesh.scheduler.guidance import ClassifierFreeGuidance
    from actionmesh.scheduler.scheduler import SchedulerFlow

    ns = types.SimpleNamespace(
        ActionMeshDenoiser=ActionMeshDenoiser, AttentionProcessor=AttentionProcessor,
        FlowMatchingBlock=FlowMatchingBlock, apply_rotary_embedding=apply_rotary_embedding,
        compute_rotary_embeddings=compute_rotary_embeddings, LatentBank=LatentBank, chunk_from=chunk_from,
        ClassifierFreeGuidance=ClassifierFreeGuidance, SchedulerFlow=SchedulerFlow, torch=torch,
        embeddings=ref_embeddings,
    )
    return ns


def load_triposg():
    """The vendored TripoSG Stage-0 denoiser and scheduler (third_party/TripoSG @ fc5c409), imported unchanged."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REFERENCE_ROOT}")
    from . import diffusers_shim

    diffusers_shim.install()
    root = os.path.join(REFERENCE_ROOT, "third_party", "TripoSG")
    if root not in sys.path:
        sys.path.insert(0, root)
    from triposg.models.transformers.triposg_transformer import TripoSGDiTModel
    from triposg.schedulers.scheduling_rectified_flow import RectifiedFlowScheduler

    return types.SimpleNamespace(TripoSGDiTModel=TripoSGDiTModel, RectifiedFlowScheduler=RectifiedFlowScheduler)
