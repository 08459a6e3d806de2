"""TEST INFRASTRUCTURE ONLY.  A CPU/GPU torch restatement of the pytorch3d pieces that actionbench/icp.py and
actionbench/benchmark.py import, so the reference's OWN icp.py / benchmark.py run unchanged where pytorch3d and trimesh
are absent (modelled on diffusers_shim.py).

Restated (pytorch3d 0.7 semantics, not pinned against pytorch3d itself, which is not a dependency):
  - transforms.euler_angles_to_matrix, transforms.rotation_6d_to_matrix;
  - loss.chamfer_distance with batch_reduction=None and the default point mean of squared nearest-neighbour distances
    (both directions summed).  Nearest neighbours use exact coordinate differences; torch.cdist is avoided on purpose,
    it switches to the |x|^2 - 2 x.y + |y|^2 expansion above 25 points;
  - transforms.transform3d: Scale / Rotate / Translate / compose / stack / transform_points (row-vector convention).
Also registered: stub `trimesh` and `sample_mesh` modules (mesh sampling is injected by the caller).

Every chamfer_distance call appends its detached per-batch loss to LOSS_TRACE, so a caller can read the per-iteration
losses of gradient_icp."""
from __future__ import annotations

import sys
import types

import torch
import torch.nn.functional as F

LOSS_TRACE: list = []


# ---- transforms -------------------------------------------------------------------------------------------------------
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


def euler_angles_to_matrix(euler_angles: torch.Tensor, convention: str) -> torch.Tensor:
    mats = [_axis_angle_rotation(c, e) for c, e in zip(convention, torch.unbind(euler_angles, -1))]
    return torch.matmul(torch.matmul(mats[0], mats[1]), mats[2])


def rotation_6d_to_matrix(d6: torch.Tensor) -> torch.Tensor:
    a1, a2 = d6[..., :3], d6[..., 3:]
    b1 = F.normalize(a1, dim=-1)
    b2 = a2 - (b1 * a2).sum(-1, keepdim=True) * b1
    b2 = F.normalize(b2, dim=-1)
    b3 = torch.cross(b1, b2, dim=-1)
    return torch.stack((b1, b2, b3), dim=-2)


class Transform3d:
    def __init__(self, matrix: torch.Tensor | None = None, dtype=torch.float32, device="cpu"):
        self._matrix = torch.eye(4, dtype=dtype, device=device)[None] if matrix is None else matrix
        self._transforms: list = []

    def get_matrix(self) -> torch.Tensor:
        m = self._matrix.clone()
        for other in self._transforms:
            m = _broadcast_bmm(m, other.get_matrix())
        return m

    def compose(self, *others) -> "Transform3d":
        out = Transform3d(self._matrix.clone())
        out._transforms = self._transforms[:] + list(others)
        return out

    def stack(self, *others) -> "Transform3d":
        return Transform3d(torch.cat([self.get_matrix()] + [o.get_matrix() for o in others], dim=0))

    def transform_points(self, points: torch.Tensor, eps: float | None = None) -> torch.Tensor:
        pts = points[None] if points.dim() == 2 else points
        homog = torch.cat([pts, torch.ones_like(pts[..., :1])], dim=-1)
        out = _broadcast_bmm(homog, self.get_matrix())
        denom = out[..., 3:]
        if eps is not None:
            denom = denom.sign() * torch.clamp(denom.abs(), eps)
        out = out[..., :3] / denom
        return out[0] if points.dim() == 2 else out


def _broadcast_bmm(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    if a.shape[0] != b.shape[0]:
        if a.shape[0] == 1:
            a = a.expand(b.shape[0], -1, -1)
        elif b.shape[0] == 1:
            b = b.expand(a.shape[0], -1, -1)
        else:
            raise ValueError("batch sizes of the transform and the points differ")
    return a.bmm(b)


class Scale(Transform3d):
    def __init__(self, x: torch.Tensor):
        s = x if x.dim() == 2 else x[None]
        m = torch.eye(4, dtype=s.dtype, device=s.device).repeat(s.shape[0], 1, 1)
        m[:, 0, 0], m[:, 1, 1], m[:, 2, 2] = s[:, 0], s[:, 1], s[:, 2]
        super().__init__(m)


class Rotate(Transform3d):
    def __init__(self, R: torch.Tensor):
        R = R if R.dim() == 3 else R[None]
        m = torch.eye(4, dtype=R.dtype, device=R.device).repeat(R.shape[0], 1, 1)
        m[:, :3, :3] = R
        super().__init__(m)


class Translate(Transform3d):
    def __init__(self, x: torch.Tensor):
        t = x if x.dim() == 2 else x[None]
        m = torch.eye(4, dtype=t.dtype, device=t.device).repeat(t.shape[0], 1, 1)
        m[:, 3, :3] = t
        super().__init__(m)


# ---- loss -------------------------------------------------------------------------------------------------------------
def nearest_index(x: torch.Tensor, y: torch.Tensor, chunk: int = 512) -> torch.Tensor:
    """(B, P, 3), (B, Q, 3) -> (B, P) index of each x's nearest y (exact squared differences; first index on ties)."""
    out = []
    for c0 in range(0, x.shape[1], chunk):
        xc = x[:, c0:c0 + chunk]
        d = (xc[..., 0, None] - y[:, None, :, 0]) ** 2
        d += (xc[..., 1, None] - y[:, None, :, 1]) ** 2
        d += (xc[..., 2, None] - y[:, None, :, 2]) ** 2
        out.append(d.argmin(-1))
    return torch.cat(out, dim=1)


def chamfer_distance(x: torch.Tensor, y: torch.Tensor, batch_reduction=None, **_):
    assert batch_reduction is None
    with torch.no_grad():
        ix = nearest_index(x.detach(), y.detach())
        iy = nearest_index(y.detach(), x.detach())
    y_nn = torch.gather(y, 1, ix[..., None].expand(-1, -1, 3))
    x_nn = torch.gather(x, 1, iy[..., None].expand(-1, -1, 3))
    loss = ((x - y_nn) ** 2).sum(-1).mean(1) + ((y - x_nn) ** 2).sum(-1).mean(1)
    LOSS_TRACE.append(loss.detach().clone())
    return loss, None


# ---- module registration ----------------------------------------------------------------------------------------------
def install() -> None:
    """Register the stand-ins under the module names actionbench imports."""
    def mod(name):
        m = types.ModuleType(name)
        m._AMB_SHIM = True
        sys.modules[name] = m
        return m

    p3 = mod("pytorch3d")
    loss = mod("pytorch3d.loss")
    tr = mod("pytorch3d.transforms")
    t3 = mod("pytorch3d.transforms.transform3d")
    p3.loss, p3.transforms, tr.transform3d = loss, tr, t3
    loss.chamfer_distance = chamfer_distance
    tr.euler_angles_to_matrix, tr.rotation_6d_to_matrix = euler_angles_to_matrix, rotation_6d_to_matrix
    t3.Transform3d, t3.Scale, t3.Rotate, t3.Translate = Transform3d, Scale, Rotate, Translate
    if "trimesh" not in sys.modules:
        mod("trimesh").Trimesh = type("Trimesh", (), {})
    sm = mod("sample_mesh")

    def sample_meshes(meshes, n_pts, synchronized, seed):
        raise RuntimeError("mesh sampling is not restated; patch benchmark.sample_meshes")

    sm.sample_meshes = sample_meshes
