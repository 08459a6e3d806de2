"""ActionBench metrics on the GPU — SURVEY 8(f) rank 4 (reference actionbench/chamfer.py, icp.py, benchmark.py).

Same functions, arguments, subsampling (numpy RandomState(seed) / (seed + 1) permutations) and return values as
`compute_chamfer_score` (chamfer.py:12-53) and `compute_motion_chamfer_score` (:56-89); the KD-tree nearest-neighbour queries
run as a brute-force CUDA search (amb_nearest_neighbors).  Distances are fp32 (the KD-tree works in fp64): the scores agree to
~1e-6 relative, see tests/test_evaluation_gpu.py.

`gradient_icp` (icp.py:53-112) runs its 24-start Adam loop entirely on the device (amb_gradient_icp), batched over frames,
and `compute_chamfer_3d_4d` (benchmark.py:67-153) scores a clip with it.  Mesh surface sampling is not part of this
package: the caller passes its own `sample_meshes(meshes, n_pts, synchronized, seed)`."""
from __future__ import annotations

import numpy as np
import torch

from . import ops
from ._lib import AmbError


def _cuda_points(x, device) -> torch.Tensor:
    t = torch.as_tensor(np.asarray(x) if not torch.is_tensor(x) else x)
    return t.to(device=device, dtype=torch.float32).contiguous()


def compute_chamfer_score(pred, gt, n: int = 10_000, seed: int = 44, device="cuda") -> float:
    """Symmetric Chamfer distance between two point clouds (chamfer.py:12-53)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise AmbError("actionmesh_b200.evaluation runs on CUDA only")
    rng_pred = np.random.RandomState(seed=seed)
    rng_gt = np.random.RandomState(seed=seed + 1)
    idx_pred = rng_pred.permutation(len(pred))[:n] if 0 < n < len(pred) else np.arange(len(pred))
    idx_gt = rng_gt.permutation(len(gt))[:n] if 0 < n < len(gt) else np.arange(len(gt))
    with torch.cuda.device(dev):
        p, g = _cuda_points(pred, dev), _cuda_points(gt, dev)
        d1, _ = ops.nearest_neighbors(g[torch.from_numpy(idx_gt).to(dev)], p, want_index=False)     # gt -> pred
        d2, _ = ops.nearest_neighbors(p[torch.from_numpy(idx_pred).to(dev)], g, want_index=False)   # pred -> gt
        return float(d1.double().mean() + d2.double().mean())


def compute_motion_chamfer_score(preds, gts, device="cuda") -> float:
    """Motion Chamfer distance over a sequence: correspondences from frame 0, distances over all frames (chamfer.py:56-89)."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise AmbError("actionmesh_b200.evaluation runs on CUDA only")
    with torch.cuda.device(dev):
        p, g = _cuda_points(preds, dev), _cuda_points(gts, dev)
        assert p.shape[0] == g.shape[0], "Mismatching number of timesteps"
        _, i_gt_to_pred = ops.nearest_neighbors(g[0], p[0])
        _, i_pred_to_gt = ops.nearest_neighbors(p[0], g[0])
        d1 = (p[:, i_gt_to_pred.long()] - g).double().norm(dim=-1).mean(dim=0)
        d2 = (g[:, i_pred_to_gt.long()] - p).double().norm(dim=-1).mean(dim=0)
        return float(d1.mean() + d2.mean())


# ---- gradient ICP (actionbench/icp.py) and the clip metrics (actionbench/benchmark.py) ---------------------------------
def _axis_angle_rotation(axis: str, angle: torch.Tensor) -> torch.Tensor:
    cos, sin = torch.cos(angle), torch.sin(angle)
    one, zero = torch.ones_like(angle), torch.zeros_like(angle)
    if axis == "X":
        flat = (one, zero, zero, zero, cos, -sin, zero, sin, cos)
    elif axis == "Y":
        flat = (cos, zero, sin, zero, one, zero, -sin, zero, cos)
    else:
        flat = (cos, -sin, zero, sin, cos, zero, zero, zero, one)
    return torch.stack(flat, -1).reshape(angle.shape + (3, 3))


def canonical_rotation_matrices() -> torch.Tensor:
    """The 24 axis-aligned start rotations of icp.py:18-49, (24, 3, 3) fp32 on the host, built with the op order of
    pytorch3d's euler_angles_to_matrix(..., "XYZ") so the table is bit-identical to the reference's."""
    deg_to_rad = torch.pi / 180
    azim = torch.tensor([0] * 4 + [90] * 4 + [180] * 4 + [270] * 4 + [0] * 4 + [90] * 4, dtype=torch.float32) * deg_to_rad
    elev = torch.tensor([0] * 16 + [90] * 2 + [-90] * 2 + [90] * 2 + [-90] * 2, dtype=torch.float32) * deg_to_rad
    roll = torch.tensor([0, 90, 180, 270] * 4 + [0, 90] * 4, dtype=torch.float32) * deg_to_rad
    mats = [_axis_angle_rotation(c, e) for c, e in zip("XYZ", (azim, elev, roll))]
    return torch.matmul(torch.matmul(mats[0], mats[1]), mats[2])


class IcpTransform:
    """Per-problem x -> (x * s) @ R + T: the part of pytorch3d's Transform3d that benchmark.py uses (`transform_points`,
    `stack`).  R (F, 3, 3), T (F, 3), s (F, 3) on the device; `loss` / `start` hold the best Chamfer loss and the start that
    reached it (F,), when the transform came from gradient_icp."""

    def __init__(self, R: torch.Tensor, T: torch.Tensor, s: torch.Tensor, loss=None, start=None):
        self.R, self.T, self.s, self.loss, self.start = R, T, s, loss, start

    def __len__(self) -> int:
        return self.R.shape[0]

    def __getitem__(self, k: int) -> "IcpTransform":
        sl = slice(k, k + 1)
        pick = lambda t: None if t is None else t[sl]  # noqa: E731
        return IcpTransform(self.R[sl], self.T[sl], self.s[sl], pick(self.loss), pick(self.start))

    def stack(self, *others: "IcpTransform") -> "IcpTransform":
        parts = (self,) + others
        cat = lambda name: None if any(getattr(p, name) is None for p in parts) else torch.cat([getattr(p, name) for p in parts])  # noqa: E731
        return IcpTransform(cat("R"), cat("T"), cat("s"), cat("loss"), cat("start"))

    def transform_points(self, points: torch.Tensor) -> torch.Tensor:
        """(N, 3) or (B, N, 3) points; a single transform applies to every batch entry, otherwise B must equal len(self)."""
        if points.dim() == 2:
            return self.transform_points(points[None])[0]
        F, B = len(self), points.shape[0]
        R, T, s = self.R, self.T, self.s
        if F == 1 and B != 1:
            R, T, s = R.expand(B, 3, 3), T.expand(B, 3), s.expand(B, 3)
        elif F != B:
            raise AmbError(f"transform_points: {F} transforms for a batch of {B} point sets")
        with torch.cuda.device(points.device):
            return ops.transform_points(points, R, T, s)


def gradient_icp_batched(pc_pred: torch.Tensor, pc_gt: torch.Tensor, lr: float = 0.01, n_iter: int = 200) -> IcpTransform:
    """gradient_icp for F independent problems at once: pc_pred (F, P, 3), pc_gt (F, Q, 3) CUDA tensors.  Problem f's
    result is bit-identical to gradient_icp(pc_pred[f], pc_gt[f])."""
    if not (torch.is_tensor(pc_pred) and pc_pred.is_cuda and torch.is_tensor(pc_gt) and pc_gt.is_cuda):
        raise AmbError("actionmesh_b200.evaluation runs on CUDA only")
    dev = pc_pred.device
    with torch.cuda.device(dev):
        r_init = canonical_rotation_matrices().to(dev)
        R, T, s, loss, start, _ = ops.gradient_icp(pc_pred.float(), pc_gt.to(dev, torch.float32), r_init, lr=lr, n_iter=n_iter)
    return IcpTransform(R, T, s, loss, start)


def gradient_icp(pc_pred: torch.Tensor, pc_gt: torch.Tensor, lr: float = 0.01, n_iter: int = 200) -> IcpTransform:
    """Rigid + anisotropic-scale transform aligning pc_pred (P, 3) to pc_gt (Q, 3) (icp.py:53-112): 24 canonical starts,
    n_iter Adam steps each on the Chamfer loss, the best start kept as the reference keeps it."""
    return gradient_icp_batched(pc_pred[None], pc_gt[None], lr=lr, n_iter=n_iter)


def sample_point_cloud(point_cloud: torch.Tensor, n_pts: int, seed: int = 44) -> torch.Tensor:
    """(T, N, C) -> (T, n_pts, C) with one numpy RandomState(seed) permutation for all frames (sample_point_cloud.py)."""
    n_src = point_cloud.shape[1]
    if n_src <= n_pts:
        return point_cloud
    idx = torch.from_numpy(np.random.RandomState(seed=seed).permutation(n_src)[:n_pts]).long()
    return point_cloud[:, idx.to(point_cloud.device)]


def compute_chamfer_3d_4d(gt_pc, pred_meshes, device, is_4D: bool = False, n_pts_icp: int = 10_000,
                          n_pts_chamfer: int = 100_000, seed: int = 44, *, sample_meshes) -> tuple[float, float, float]:
    """(cd_3d, cd_4d, cd_motion) of benchmark.py:67-153: Chamfer after per-frame ICP, after the frame-0 ("unified") ICP,
    and the motion Chamfer after the unified ICP (0.0 unless is_4D).  `sample_meshes(meshes, n_pts, synchronized, seed)`
    returns (T, n_pts, 3) surface samples of the T predicted meshes.  The per-frame ICPs run as one batched call; the
    unified ICP has exactly the inputs of frame 0's, and the loop is deterministic and batch-independent, so it is
    problem 0 of that call."""
    dev = torch.device(device)
    if dev.type != "cuda":
        raise AmbError("actionmesh_b200.evaluation runs on CUDA only")
    n_ts = len(pred_meshes)
    pred_pc = torch.as_tensor(sample_meshes(pred_meshes, n_pts=n_pts_chamfer, synchronized=False, seed=seed))
    gt_pc = torch.as_tensor(gt_pc)
    pred_pc_icp = sample_point_cloud(pred_pc, n_pts=n_pts_icp, seed=seed)
    gt_pc_icp = sample_point_cloud(gt_pc, n_pts=n_pts_icp, seed=seed)
    with torch.cuda.device(dev):
        pred_pc = _cuda_points(pred_pc, dev)
        gt_pc = _cuda_points(gt_pc, dev)
        icp_3d = gradient_icp_batched(_cuda_points(pred_pc_icp, dev), _cuda_points(gt_pc_icp, dev), lr=0.01, n_iter=200)
        icp_u4d = icp_3d[0]
        aligned_3d = icp_3d.transform_points(pred_pc)
        aligned_u4d = icp_u4d.transform_points(pred_pc)
        cd_3d = np.mean([compute_chamfer_score(gt=gt_pc[k], pred=aligned_3d[k], device=dev) for k in range(n_ts)])
        cd_4d = np.mean([compute_chamfer_score(gt=gt_pc[k], pred=aligned_u4d[k], device=dev) for k in range(n_ts)])
        cd_motion = 0.0
        if is_4D:
            pred_pc_4d = _cuda_points(torch.as_tensor(sample_meshes(pred_meshes, n_pts=n_pts_chamfer, synchronized=True,
                                                                    seed=seed)), dev)
            cd_motion = compute_motion_chamfer_score(preds=icp_u4d.transform_points(pred_pc_4d), gts=gt_pc, device=dev)
    return cd_3d, cd_4d, cd_motion
