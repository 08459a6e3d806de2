"""TEST INFRASTRUCTURE ONLY — deterministic synthetic weights/inputs shared by the golden generator, the tests and bench.

No checkpoints exist offline (SURVEY 8(c)), so parity work uses seeded random weights with the reference's state-dict
key names (SURVEY A.1).  Values are rounded to bf16-representable fp32 so the fp32 oracle and the bf16-weight CUDA path
consume IDENTICAL weights (differences are then activation rounding only).  Drawn from a CPU torch.Generator in a fixed
order => reproducible on any box with the same torch build.
"""
from __future__ import annotations

import math

import torch


def _bf16r(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16).to(torch.float32)


def make_state_dict(cfg, seed: int = 1234, residual_scale: float | None = None, device="cpu") -> dict:
    """cfg: any object with in_channels, num_layers, num_attention_heads, width, mlp_ratio, cross_attention_dim.
    `device="cuda"` draws from a CUDA generator (the 1.44 B-parameter default config is generated on the GPU in the
    full-depth parity test; the values differ from the CPU stream but both sides of a test always share one dict)."""
    g = torch.Generator(device=device).manual_seed(seed)
    D, C, Dc = cfg.width, cfg.in_channels, cfg.cross_attention_dim
    F_ = int(D * cfg.mlp_ratio)
    dh = D // cfg.num_attention_heads
    rs = residual_scale if residual_scale is not None else 1.0 / math.sqrt(cfg.num_layers)

    def lin(out_f, in_f, scale=1.0):
        b = 1.0 / math.sqrt(in_f)
        return _bf16r((torch.rand(out_f, in_f, generator=g, device=device) * 2 - 1) * b * scale)

    def vec(n, lo, hi):
        return _bf16r(torch.rand(n, generator=g, device=device) * (hi - lo) + lo)

    sd = {}
    sd["time_proj.linear_1.weight"], sd["time_proj.linear_1.bias"] = lin(4 * D, D), vec(4 * D, -0.02, 0.02)
    sd["time_proj.linear_2.weight"], sd["time_proj.linear_2.bias"] = lin(D, 4 * D), vec(D, -0.02, 0.02)
    sd["proj_in.weight"], sd["proj_in.bias"] = lin(D, C), vec(D, -0.1, 0.1)
    for i in range(cfg.num_layers):
        p = f"blocks.{i}."
        if i > cfg.num_layers // 2:
            sd[p + "linear_skip.weight"], sd[p + "linear_skip.bias"] = lin(D, 2 * D), vec(D, -0.02, 0.02)
            sd[p + "norm_skip.weight"], sd[p + "norm_skip.bias"] = vec(D, 0.8, 1.2), vec(D, -0.1, 0.1)
        for n in ("norm_s_attn", "norm_x_attn", "norm_ff"):
            sd[p + n + ".weight"], sd[p + n + ".bias"] = vec(D, 0.8, 1.2), vec(D, -0.1, 0.1)
        for a, kd in (("s_attn", D), ("x_attn", Dc)):
            sd[p + a + ".to_q.weight"] = lin(D, D)
            sd[p + a + ".to_k.weight"] = lin(D, kd)
            sd[p + a + ".to_v.weight"] = lin(D, kd)
            sd[p + a + ".norm_q.weight"] = vec(dh, 0.8, 1.2)
            sd[p + a + ".norm_k.weight"] = vec(dh, 0.8, 1.2)
            sd[p + a + ".to_out.0.weight"], sd[p + a + ".to_out.0.bias"] = lin(D, D, rs), vec(D, -0.02, 0.02)
        sd[p + "ff.net.0.proj.weight"], sd[p + "ff.net.0.proj.bias"] = lin(F_, D), vec(F_, -0.02, 0.02)
        sd[p + "ff.net.2.weight"], sd[p + "ff.net.2.bias"] = lin(D, F_, rs), vec(D, -0.02, 0.02)
    sd["norm_out.weight"], sd["norm_out.bias"] = vec(D, 0.8, 1.2), vec(D, -0.1, 0.1)
    sd["proj_out.weight"], sd["proj_out.bias"] = lin(C, D), vec(C, -0.02, 0.02)
    return sd


def make_inputs(B: int, T: int, N: int, C: int, S: int, Dc: int, seed: int = 5, observed=(0,)):
    """Seeded latents / context / framestep / mask for one window (batch B before CFG)."""
    g = torch.Generator(device="cpu").manual_seed(seed)
    latents = torch.randn(B, T, N, C, generator=g)
    context = torch.randn(B, T, S, Dc, generator=g)
    framestep = torch.arange(T, dtype=torch.float32)[None].repeat(B, 1) + 3.0  # centred by the model
    mask = torch.zeros(B, T)
    for o in observed:
        mask[:, o] = 1.0
    return latents, context, framestep, mask


def make_rgba_frames(n: int = 5, H: int = 96, W: int = 128, seed: int = 3):
    """Seeded (H, W, 4) uint8 frames: random RGB under a moving disc of alpha with a soft (partially transparent) edge."""
    import numpy as np

    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        img = rng.integers(0, 256, (H, W, 4), dtype=np.uint8)
        yy, xx = np.mgrid[0:H, 0:W]
        cy, cx, r = H // 2 + 3 * i - 4, W // 2 - 2 * i, 20 + 2 * i
        d = np.sqrt((yy - cy) ** 2 + (xx - cx) ** 2)
        img[..., 3] = np.clip((r + 6 - d) * 40, 0, 255).astype(np.uint8)
        out.append(img)
    return out
