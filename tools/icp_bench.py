"""Gradient ICP timing on one GPU; prints one JSON line.

    python tools/icp_bench.py [--runs 5] [--baseline-iters 200]

- gradient_icp at P = 10 000 prediction and ground-truth points x 24 starts x 200 iterations: ms per call (CUDA events,
  median of --runs after a warm-up call), nearest-neighbour pair evaluations per second (2 directions x 24 x P x P per
  iteration), and that rate over the card's fp32 issue rate (148 SMs x 128 lanes x max SM clock) times the
  instructions one pair costs in the search loop (FP32_INSTR_PER_PAIR, counted in `cuobjdump -sass` of icp_search_kernel);
- one clip: the F = 16 batched ICP, and compute_chamfer_3d_4d at T = 16 with 100 000 / 10 000 points from a seeded
  synthetic sampler (s per clip);
- baseline: one gradient_icp through a torch restatement of the reference loop on the same GPU (chunked exact Chamfer
  from oracle/pytorch3d_shim.py, autograd, torch.optim.Adam, a host sync per iteration).  It is labelled as the torch
  restatement: pytorch3d itself is not installed.
The card's name, power limit and clocks are read with nvidia-smi in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from actionmesh_b200 import ops  # noqa: E402
from actionmesh_b200.evaluation import canonical_rotation_matrices, compute_chamfer_3d_4d  # noqa: E402

# Per pair and query in the inner loop: 3 FADD (differences), FMUL + 2 FFMA (squared distance), FSETP + 2 SEL (running
# minimum and its index).  Shared-memory loads are amortised over the 6 (pred->gt) or 4 (gt->pred) queries a thread holds.
FP32_INSTR_PER_PAIR = 9


def gpu_info() -> dict:
    q = "name,power.limit,clocks.max.sm,clocks.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, plim, cmax, ccur = [v.strip() for v in out.split(",")]
        return {"gpu": name, "power_limit": plim, "sm_clock_max": cmax, "sm_clock_now": ccur}
    except Exception as exc:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(), "nvidia_smi_error": str(exc)}


def shape(n: int, g: torch.Generator, phase: float = 0.0) -> torch.Tensor:
    u = torch.randn(n, 3, generator=g)
    u = u / u.norm(dim=1, keepdim=True)
    pts = u * torch.tensor([0.5, 0.3, 0.2])
    k = n // 4
    pts[:k] = pts[:k] * 0.4 + torch.tensor([0.45, 0.2 + 0.1 * phase, 0.05])
    return pts


def misalign(x: torch.Tensor, g: torch.Generator) -> torch.Tensor:
    c, s = 0.9063, 0.4226  # 25 degrees about z
    R = torch.tensor([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])
    return ((x - torch.tensor([0.1, -0.05, 0.08])) @ R.T) / torch.tensor([1.1, 0.9, 1.05]) + 0.003 * torch.randn(x.shape, generator=g)


def timed(fn, runs: int) -> list[float]:
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(runs):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return ms


def median(v):
    v = sorted(v)
    return v[len(v) // 2]


def torch_restatement_icp(pred, gt, r_init, n_iter):
    """icp.py:75-106 on the restated pytorch3d pieces, as the reference runs it (per-iteration .item())."""
    from oracle import pytorch3d_shim as p3

    n = r_init.shape[0]
    pp, gg = pred[None].expand(n, -1, -1), gt[None].expand(n, -1, -1)
    T = torch.nn.Parameter(torch.zeros(n, 3, device=pred.device))
    r6 = torch.nn.Parameter(torch.tensor([[1.0, 0, 0, 0, 1, 0]], device=pred.device).repeat(n, 1))
    s = torch.nn.Parameter(torch.ones(n, 3, device=pred.device))
    opt = torch.optim.Adam([T, r6, s], lr=0.01)
    best = float("inf")
    for _ in range(n_iter):
        opt.zero_grad()
        R = r_init @ p3.rotation_6d_to_matrix(r6)
        loss = p3.chamfer_distance(s[:, None] * pp @ R + T[:, None], gg)[0]
        loss.mean().backward()
        opt.step()
        m, _ = loss.detach().min(0)
        best = min(best, m.item())
    p3.LOSS_TRACE.clear()
    return best


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--points", type=int, default=10_000)
    ap.add_argument("--baseline-iters", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("icp_bench needs a CUDA device")
    dev = torch.device("cuda")
    res = gpu_info()
    g = torch.Generator().manual_seed(0)
    P = args.points
    r_init = canonical_rotation_matrices().to(dev)

    # one gradient_icp call at the reference's n_pts_icp
    gt1 = shape(P, g)
    pred1 = misalign(gt1, g)
    gt1, pred1 = gt1.to(dev), pred1.to(dev)
    ms = timed(lambda: ops.gradient_icp(pred1[None], gt1[None], r_init), args.runs)
    pairs = 2 * 24 * P * P * 200
    pair_rate = pairs / (median(ms) / 1e3)
    res.update({"icp_points": P, "icp_ms_per_call": median(ms), "icp_ms_runs": ms, "pairs_per_call": pairs,
                "pair_evals_per_s": pair_rate, "fp32_instr_per_pair_assumed": FP32_INSTR_PER_PAIR})
    try:
        clk_mhz = float(res["sm_clock_max"].split()[0])
        issue = torch.cuda.get_device_properties(dev).multi_processor_count * 128 * clk_mhz * 1e6
        res["fp32_issue_share_of_peak"] = pair_rate * FP32_INSTR_PER_PAIR / issue
    except (KeyError, ValueError):
        res["fp32_issue_share_of_peak"] = None

    # one clip: 16 frames
    Tn = 16
    gt_clip = torch.stack([shape(P, g, phase=k / 4) for k in range(Tn)]).to(dev)
    pred_clip = torch.stack([misalign(shape(P, g, phase=k / 4), g) for k in range(Tn)]).to(dev)
    ms16 = timed(lambda: ops.gradient_icp(pred_clip, gt_clip, r_init), max(3, args.runs // 2))
    res.update({"clip_frames": Tn, "clip_icp_s": median(ms16) / 1e3, "clip_icp_s_runs": [m / 1e3 for m in ms16]})

    n_chamfer = 100_000
    gt_full = torch.stack([shape(n_chamfer, g, phase=k / 4) for k in range(Tn)])
    pred_full = torch.stack([misalign(shape(n_chamfer, g, phase=k / 4), g) for k in range(Tn)])
    pred_sync = torch.stack([misalign(shape(n_chamfer, torch.Generator().manual_seed(9)), g) for _ in range(Tn)])

    def sampler(meshes, n_pts, synchronized, seed):
        return pred_sync if synchronized else pred_full

    def clip():
        return compute_chamfer_3d_4d(gt_full, [None] * Tn, "cuda", is_4D=True, n_pts_icp=P, n_pts_chamfer=n_chamfer,
                                     seed=44, sample_meshes=sampler)

    clip()
    wall = []
    for _ in range(max(3, args.runs // 2)):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        scores = clip()
        torch.cuda.synchronize()
        wall.append(time.perf_counter() - t0)
    res.update({"clip_chamfer_3d_4d_s": median(wall), "clip_chamfer_3d_4d_s_runs": wall,
                "clip_scores": [float(v) for v in scores]})

    # baseline: the torch restatement of the reference loop, one call
    if args.baseline_iters > 0:
        torch_restatement_icp(pred1, gt1, r_init, 2)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        torch_restatement_icp(pred1, gt1, r_init, args.baseline_iters)
        torch.cuda.synchronize()
        t = time.perf_counter() - t0
        res.update({"torch_restatement_iters": args.baseline_iters, "torch_restatement_ms_per_call": t * 1e3 * 200 / args.baseline_iters,
                    "speedup_vs_torch_restatement": t * 1e3 * 200 / args.baseline_iters / median(ms)})
    res.update(gpu_info() | {"after": True})
    print(json.dumps(res))


if __name__ == "__main__":
    main()
