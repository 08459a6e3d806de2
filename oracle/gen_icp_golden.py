"""TEST INFRASTRUCTURE ONLY.  Writes tests/golden/icp_small.pt from the reference's OWN actionbench/icp.py and
actionbench/benchmark.py, imported unchanged on top of pytorch3d_shim (CPU, fp32; a few minutes on an 8-core host).

    python -m oracle.gen_icp_golden            # reference checkout in $ACTIONMESH_REFERENCE

Contents:
  - icp_pred (1000, 3), icp_gt (1000, 3): a ground-truth cloud and a rotated, anisotropically scaled, translated and
    noised copy of it;
  - r_init (24, 3, 3): actionbench's canonical_rotation_matrices();
  - trace (200, 24): the per-iteration, per-start Chamfer losses of gradient_icp(icp_pred, icp_gt, lr=0.01, n_iter=200);
    best_loss / best_start: the best the reference kept (the strict-< first-minimum rule of icp.py:99-106, applied to the
    trace); best_matrix (1, 4, 4): the composed transform it returned; icp_aligned: that transform applied to icp_pred;
  - spc_input / spc_output: sample_point_cloud on a small (2, 50, 3) sequence, n_pts=20, seed=44;
  - e2e_gt (3, 2000, 3), e2e_pred (3, 2000, 3), e2e_pred_sync (3, 2000, 3): the inputs of compute_chamfer_3d_4d, with
    sample_meshes patched to return e2e_pred (synchronized=False) or e2e_pred_sync (True); e2e_cd: (cd_3d, cd_4d,
    cd_motion) for is_4D=True, n_pts_icp=1000, n_pts_chamfer=2000, seed=44.
"""
from __future__ import annotations

import math
import os
import sys

import torch

from . import pytorch3d_shim
from .reference_loader import REFERENCE_ROOT, available

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "icp_small.pt")


def load_actionbench():
    """(icp, benchmark) modules of the reference checkout, on the shim."""
    if not available():
        raise RuntimeError(f"reference checkout not found at {REFERENCE_ROOT}")
    pytorch3d_shim.install()
    path = os.path.join(REFERENCE_ROOT, "actionbench")
    if path not in sys.path:
        sys.path.insert(0, path)
    import benchmark
    import icp

    return icp, benchmark


def _rot(axis, deg):
    a = math.radians(deg)
    c, s = math.cos(a), math.sin(a)
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    R = torch.eye(3, dtype=torch.float64)
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


def shape(n: int, g: torch.Generator, phase: float = 0.0) -> torch.Tensor:
    """An asymmetric cloud: an ellipsoid shell with an off-centre bump whose position moves with `phase`."""
    u = torch.randn(n, 3, generator=g, dtype=torch.float64)
    u = u / u.norm(dim=1, keepdim=True)
    pts = u * torch.tensor([0.5, 0.3, 0.2], dtype=torch.float64)
    k = n // 4
    pts[:k] = pts[:k] * 0.4 + torch.tensor([0.45, 0.2 + 0.1 * phase, 0.05], dtype=torch.float64)
    return pts


def misalign(gt: torch.Tensor, g: torch.Generator, noise: float = 0.005) -> torch.Tensor:
    """pred such that (s * pred) @ R + T ~ gt for a rotation off every canonical start, anisotropic s and some T."""
    R = _rot(2, 25.0) @ _rot(0, -15.0) @ _rot(1, 100.0)
    s = torch.tensor([1.1, 0.9, 1.05], dtype=torch.float64)
    T = torch.tensor([0.1, -0.05, 0.08], dtype=torch.float64)
    pred = ((gt - T) @ R.T) / s
    return pred + noise * torch.randn(pred.shape, generator=g, dtype=torch.float64)


def best_from_trace(trace: torch.Tensor):
    """icp.py:99-106: first index of each iteration's minimum, kept only when strictly below the running best."""
    best, start = float("inf"), -1
    for it in range(trace.shape[0]):
        m, i = trace[it].min(0)
        if m.item() < best:
            best, start = m.item(), int(i)
    return best, start


def run_reference_icp(icp, pred, gt, n_iter):
    pytorch3d_shim.LOSS_TRACE.clear()
    tf = icp.gradient_icp(pc_pred=pred, pc_gt=gt, lr=0.01, n_iter=n_iter)
    return tf, torch.stack(pytorch3d_shim.LOSS_TRACE)


def main() -> None:
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    icp, benchmark = load_actionbench()
    g = torch.Generator().manual_seed(1234)
    gt = shape(1000, g).float()
    pred = misalign(gt.double(), g).float()
    out = {"icp_pred": pred, "icp_gt": gt, "r_init": icp.canonical_rotation_matrices()}
    tf, trace = run_reference_icp(icp, pred, gt, 200)
    out["trace"] = trace
    out["best_loss"], out["best_start"] = best_from_trace(trace)
    out["best_matrix"] = tf.get_matrix()
    out["icp_aligned"] = tf.transform_points(pred)
    print("icp: best", out["best_loss"], "start", out["best_start"], flush=True)

    spc_in = torch.arange(2 * 50 * 3, dtype=torch.float32).reshape(2, 50, 3)
    out["spc_input"] = spc_in
    out["spc_output"] = benchmark.sample_point_cloud(spc_in, n_pts=20, seed=44)

    T = 3
    e2e_gt = torch.stack([shape(2000, g, phase=k) for k in range(T)]).float()
    e2e_pred = torch.stack([misalign(shape(2000, g, phase=k), g) for k in range(T)]).float()
    sync_base = shape(2000, g)
    e2e_pred_sync = torch.stack([misalign(sync_base, g) for _ in range(T)]).float()
    out["e2e_gt"], out["e2e_pred"], out["e2e_pred_sync"] = e2e_gt, e2e_pred, e2e_pred_sync
    benchmark.sample_meshes = lambda meshes, n_pts, synchronized, seed: (e2e_pred_sync if synchronized else e2e_pred).clone()
    benchmark.tqdm = lambda it, **_: it
    cd = benchmark.compute_chamfer_3d_4d(e2e_gt, [None] * T, "cpu", is_4D=True, n_pts_icp=1000, n_pts_chamfer=2000,
                                         seed=44)
    out["e2e_cd"] = tuple(float(v) for v in cd)
    print("e2e:", out["e2e_cd"], flush=True)
    torch.save(out, OUT)
    print("wrote", OUT)


if __name__ == "__main__":
    main()
