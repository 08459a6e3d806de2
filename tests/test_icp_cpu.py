"""Gradient ICP host side, no GPU: the golden fixture against the reference's own icp.py (live when a reference checkout
is present), the start-rotation table, the point-cloud subsampling, the Adam tables, and argument validation of the
new C-ABI entry points (fake non-null pointers: validation must stop before any launch)."""
import ctypes as C

import pytest
import torch

from conftest import load_golden
from oracle import reference_loader


def test_canonical_rotation_matrices_bit_equal_to_reference():
    from actionmesh_b200.evaluation import canonical_rotation_matrices

    g = load_golden("icp_small.pt")
    R = canonical_rotation_matrices()
    assert R.dtype == torch.float32 and R.shape == (24, 3, 3)
    assert torch.equal(R, g["r_init"])


def test_sample_point_cloud_matches_reference():
    from actionmesh_b200.evaluation import sample_point_cloud

    g = load_golden("icp_small.pt")
    assert torch.equal(sample_point_cloud(g["spc_input"], n_pts=20, seed=44), g["spc_output"])
    small = g["spc_input"][:, :10]
    assert sample_point_cloud(small, n_pts=20, seed=44) is small   # fewer points than asked: returned unchanged


def test_adam_tables_match_torch_formula():
    from actionmesh_b200.ops import adam_tables

    step, bc2 = adam_tables(0.01, 200)
    assert step.dtype == bc2.dtype == torch.float32 and step.shape == bc2.shape == (200,)
    for t in (1, 2, 50, 200):
        assert float(step[t - 1]) == float(torch.tensor(0.01 / (1 - 0.9 ** t), dtype=torch.float32))
        assert float(bc2[t - 1]) == float(torch.tensor((1 - 0.999 ** t) ** 0.5, dtype=torch.float32))
    # the same scalars torch.optim.Adam uses: one step of a scalar parameter from m = v = 0 moves it by -lr * sign(g)
    p = torch.nn.Parameter(torch.tensor([1.0]))
    opt = torch.optim.Adam([p], lr=0.01)
    p.grad = torch.tensor([0.3])
    opt.step()
    m, v = 0.1 * 0.3, 0.001 * 0.3 ** 2
    want = torch.tensor(1.0) - step[0] * (torch.tensor(m) / (torch.tensor(v).sqrt() / bc2[0] + 1e-8))
    assert abs(float(p.detach()) - float(want)) < 1e-7


def test_golden_trace_is_consistent():
    """The stored best loss / start follow from the stored trace by the reference's rule, and the trace decreases."""
    from oracle.gen_icp_golden import best_from_trace

    g = load_golden("icp_small.pt")
    assert g["trace"].shape == (200, 24)
    assert best_from_trace(g["trace"]) == (g["best_loss"], g["best_start"])
    assert g["best_loss"] < 0.05 * float(g["trace"][0].min())


@pytest.mark.skipif(not reference_loader.available(), reason="reference checkout not present")
def test_shim_driven_reference_reproduces_golden():
    """The reference's own gradient_icp on the shim reproduces the fixture's first iterations and start table."""
    from oracle import gen_icp_golden as gen

    icp, benchmark = gen.load_actionbench()
    g = load_golden("icp_small.pt")
    assert torch.equal(icp.canonical_rotation_matrices(), g["r_init"])
    _, trace = gen.run_reference_icp(icp, g["icp_pred"], g["icp_gt"], 5)
    assert torch.allclose(trace, g["trace"][:5], rtol=1e-6, atol=0)
    assert torch.equal(benchmark.sample_point_cloud(g["spc_input"], n_pts=20, seed=44), g["spc_output"])


def test_icp_entry_points_validate_arguments(amb_lib):
    P = 16
    err = lambda: amb_lib.amb_last_error().decode()
    nb = C.c_size_t()
    assert amb_lib.amb_icp_workspace_bytes(1, 100, 100, None) < 0 and "null pointer" in err()
    assert amb_lib.amb_icp_workspace_bytes(1, 0, 100, C.byref(nb)) < 0 and "bad counts" in err()
    assert amb_lib.amb_icp_workspace_bytes(2, 100, 120, C.byref(nb)) == 0 and nb.value > 0
    need = nb.value
    # chamfer_grad: null pointers, empty clouds, too small a workspace
    assert amb_lib.amb_icp_chamfer_grad(None, P, 2, 100, 120, P, P, P, need, P, P, None) < 0 and "null pointer" in err()
    assert amb_lib.amb_icp_chamfer_grad(P, P, 2, 100, 120, P, None, P, need, P, P, None) < 0 and "null pointer" in err()
    assert amb_lib.amb_icp_chamfer_grad(P, P, 2, 0, 120, P, P, P, need, P, P, None) < 0 and "empty cloud" in err()
    assert amb_lib.amb_icp_chamfer_grad(P, P, 0, 100, 120, P, P, P, need, P, P, None) < 0 and "empty cloud" in err()
    assert amb_lib.amb_icp_chamfer_grad(P, P, 2, 100, 120, P, P, P, need - 4, P, P, None) < 0 and "workspace" in err()
    # gradient_icp: the same checks plus the iteration count and the tables
    args = lambda **kw: [kw.get("pred", P), P, kw.get("F", 2), kw.get("np", 100), kw.get("ng", 120), P, kw.get("it", 200),
                         kw.get("tab", P), P, P, kw.get("ws", need), P, P, P, P, P, None, None]
    assert amb_lib.amb_gradient_icp(*args(pred=None)) < 0 and "null pointer" in err()
    assert amb_lib.amb_gradient_icp(*args(tab=None)) < 0 and "null pointer" in err()
    assert amb_lib.amb_gradient_icp(*args(ng=0)) < 0 and "empty cloud" in err()
    assert amb_lib.amb_gradient_icp(*args(np=-3)) < 0 and "empty cloud" in err()
    assert amb_lib.amb_gradient_icp(*args(it=0)) < 0 and "n_iter" in err()
    assert amb_lib.amb_gradient_icp(*args(ws=16)) < 0 and "workspace" in err()
    # transform_points
    assert amb_lib.amb_transform_points(None, 1, 10, P, P, P, P, None) < 0 and "null pointer" in err()
    assert amb_lib.amb_transform_points(P, -1, 10, P, P, P, P, None) < 0 and "bad counts" in err()
    assert amb_lib.amb_transform_points(P, 0, 10, P, P, P, P, None) == 0      # no work: no launch


def test_icp_transform_and_ops_refuse_cpu_tensors():
    from actionmesh_b200 import AmbError, evaluation, ops

    x = torch.zeros(1, 10, 3)
    with pytest.raises(AmbError):
        evaluation.gradient_icp(x[0], x[0])
    with pytest.raises(AmbError):
        ops.gradient_icp(x, x, evaluation.canonical_rotation_matrices())
    with pytest.raises(AmbError):
        ops.transform_points(x, torch.eye(3)[None], torch.zeros(1, 3), torch.ones(1, 3))
    with pytest.raises(AmbError):
        evaluation.compute_chamfer_3d_4d(x, [None], "cpu", sample_meshes=lambda *a, **k: x)
