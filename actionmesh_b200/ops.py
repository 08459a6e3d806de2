"""Torch-tensor front door to the C ABI (device pointers + the current CUDA stream; torch is only plumbing here).

Every function launches hand-written sm_100a kernels from libactionmesh_b200.so; nothing here computes with torch ops.
A global launch counter (`launch_count`) lets bench.py report how many of OUR kernels ran in the timed region.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib

launch_count = 0

# Optional per-kernel CUDA-event timing (bench.py's roofline legs): when `event_log` is a list, launches whose `tag` is
# in `event_tags` append (tag, start_event, end_event, meta) recorded on the launching stream; meta = the launch's shape.
event_log = None
event_tags: set = set()


class _Timed:
    def __init__(self, tag, meta=None):
        self.on = event_log is not None and tag in event_tags
        self.tag = tag
        self.meta = meta

    def __enter__(self):
        if self.on:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()

    def __exit__(self, *a):
        if self.on:
            self.e1.record()
            event_log.append((self.tag, self.e0, self.e1, self.meta))


def on_device(fn):
    """Method decorator for the module-level entry points: makes `self.device` the current CUDA device for the call (the C
    ABI launches on the current device and stream)."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        dev = self.device
        if dev.type != "cuda":
            return fn(self, *args, **kwargs)
        with torch.cuda.device(dev):
            return fn(self, *args, **kwargs)

    return wrapper


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype: torch.dtype, name: str) -> None:
    if not t.is_cuda:
        raise _lib.AmbError(f"{name}: expected a CUDA tensor (there is no CPU fallback)")
    if t.dtype != dtype:
        raise _lib.AmbError(f"{name}: expected {dtype}, got {t.dtype}")
    # the C ABI launches on the CURRENT device and stream: a tensor of another device would be an illegal access (or
    # silent peer traffic).  The module-level entry points (B200Denoiser.forward, B200SchedulerFlow.denoise, ...) make
    # their own device current; direct callers of ops must do the same.
    if t.device.index != torch.cuda.current_device():
        raise _lib.AmbError(f"{name}: tensor lives on {t.device} but the current device is cuda:{torch.cuda.current_device()}"
                            " (wrap the call in torch.cuda.device(tensor.device))")


def cfg_euler_step(latents: torch.Tensor, pred: torch.Tensor, scales: list[float], dt_signed: float,
                   frame_update: torch.Tensor, *, n_branches: int, branch_stride: int, frame_stride: int,
                   frame_offset: int, n_per_frame: int) -> None:
    """In-place x[f] += dt * (p0 + sum_i s_i (p_{i+1} - p_i)) on frames with frame_update[f] != 0.

    Replaces guidance.py:95-118 + scheduler.py:238-248 of the reference."""
    global launch_count
    _need(latents, torch.float32, "latents")
    _need(pred, torch.bfloat16, "pred")
    _need(frame_update, torch.uint8, "frame_update")
    n_frames = frame_update.numel()
    arr = (C.c_float * max(1, len(scales)))(*scales)
    rc = _lib.load_library().amb_cfg_euler_step(
        latents.data_ptr(), pred.data_ptr(), n_branches, arr, float(dt_signed), frame_update.data_ptr(), n_frames,
        n_per_frame, branch_stride, frame_stride, frame_offset, _stream())
    _lib.check(rc, "amb_cfg_euler_step")
    launch_count += 1


def layernorm(x: torch.Tensor, gamma: torch.Tensor, beta: torch.Tensor, eps: float,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Affine LayerNorm over the last dim of a 2-D (rows, cols) tensor, fp32 statistics, bf16 (default) or fp32 output."""
    global launch_count
    assert x.dim() == 2 and x.stride(1) == 1
    rows, cols = x.shape
    if out is None:
        out = torch.empty((rows, cols), dtype=torch.bfloat16, device=x.device)
    _need(gamma, torch.float32, "gamma")
    _need(beta, torch.float32, "beta")
    if x.dtype not in (torch.bfloat16, torch.float32) or out.dtype not in (torch.bfloat16, torch.float32):
        raise _lib.AmbError(f"layernorm: unsupported dtype {x.dtype} -> {out.dtype}")
    if not out.is_cuda:
        raise _lib.AmbError("layernorm: out must be a CUDA tensor")
    with _Timed("layernorm", (rows, cols, x.element_size() + out.element_size())):
        rc = _lib.load_library().amb_layernorm(
            x.data_ptr(), int(x.dtype == torch.float32), x.stride(0), gamma.data_ptr(), beta.data_ptr(), out.data_ptr(),
            int(out.dtype == torch.float32), out.stride(0), rows, cols, float(eps), _stream())
    _lib.check(rc, "amb_layernorm")
    launch_count += 1
    return out


def patchify(pixels: torch.Tensor, patch: int, kpad: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """im2col of (T,3,H,W) fp32 pixels -> (T*(H/P)*(W/P), kpad) bf16 rows for the patch-embedding GEMM."""
    global launch_count
    _need(pixels, torch.float32, "pixels")
    assert pixels.is_contiguous() and pixels.dim() == 4 and pixels.shape[1] == 3
    T, _, H, W = pixels.shape
    rows = T * (H // patch) * (W // patch)
    if out is None:
        out = torch.empty(rows, kpad, dtype=torch.bfloat16, device=pixels.device)
    rc = _lib.load_library().amb_patchify(pixels.data_ptr(), out.data_ptr(), T, H, W, patch, kpad, _stream())
    _lib.check(rc, "amb_patchify")
    launch_count += 1
    return out


def alpha_rows(source_alpha: float, target_alpha: float, size: int, out_rows: torch.Tensor) -> None:
    """Write the (source, target) alpha token (2*size fp32 values) into every row of the strided 2-D view `out_rows`."""
    global launch_count
    _need(out_rows, torch.float32, "out_rows")
    assert out_rows.dim() == 2 and out_rows.shape[1] == 2 * size and out_rows.stride(1) == 1
    rc = _lib.load_library().amb_alpha_rows(float(source_alpha), float(target_alpha), size, out_rows.data_ptr(),
                                            out_rows.stride(0), out_rows.shape[0], _stream())
    _lib.check(rc, "amb_alpha_rows")
    launch_count += 1


def point_embedding(points: torch.Tensor, num_freqs: int, include_pi: bool, kpad: int) -> torch.Tensor:
    """(V, 3+E) fp32 query points -> (V, kpad) fp32 [x | sin | cos | extra | 0-pad] rows."""
    global launch_count
    _need(points, torch.float32, "points")
    assert points.dim() == 2 and points.is_contiguous()
    V, in_dim = points.shape
    out = torch.empty(V, kpad, dtype=torch.float32, device=points.device)
    rc = _lib.load_library().amb_point_embedding(points.data_ptr(), V, in_dim, in_dim - 3, num_freqs, int(include_pi),
                                                 out.data_ptr(), kpad, _stream())
    _lib.check(rc, "amb_point_embedding")
    launch_count += 1
    return out


def split3(src: torch.Tensor, out: torch.Tensor, seg: Optional[int] = None, weight: bool = False) -> torch.Tensor:
    """fp32 (rows, cols) -> bf16 (rows, 3*cols) split operand: [hi|lo|hi] per segment (activations) or [hi|hi|lo] (weights)."""
    global launch_count
    _need(src, torch.float32, "src")
    _need(out, torch.bfloat16, "out")
    assert src.dim() == 2 and out.dim() == 2 and src.stride(1) == 1 and out.stride(1) == 1
    rows, cols = src.shape
    assert out.shape[0] >= rows and out.shape[1] == 3 * cols
    rc = _lib.load_library().amb_split3_bf16(src.data_ptr(), src.stride(0), rows, cols, seg or cols, int(weight),
                                             out.data_ptr(), out.stride(0), _stream())
    _lib.check(rc, "amb_split3_bf16")
    launch_count += 1
    return out


def softmax_split3(scores: torch.Tensor, n: int, scale: float, out: torch.Tensor) -> torch.Tensor:
    """Row softmax over the first n columns of fp32 `scores` (rows, n_pad), written as [P_hi|P_lo|P_hi] (rows, 3*n_pad)."""
    global launch_count
    _need(scores, torch.float32, "scores")
    _need(out, torch.bfloat16, "out")
    rows, n_pad = scores.shape
    assert scores.stride(1) == 1 and out.stride(1) == 1 and out.shape == (rows, 3 * n_pad)
    rc = _lib.load_library().amb_softmax_split3(scores.data_ptr(), scores.stride(0), rows, n, n_pad, float(scale),
                                                out.data_ptr(), out.stride(0), _stream())
    _lib.check(rc, "amb_softmax_split3")
    launch_count += 1
    return out


def displacement_out(logits: torch.Tensor, out_dim: int, out: torch.Tensor) -> torch.Tensor:
    global launch_count
    _need(logits, torch.float32, "logits")
    _need(out, torch.float32, "out")
    assert logits.dim() == 2 and logits.stride(1) == 1 and out.is_contiguous()
    rc = _lib.load_library().amb_displacement_out(logits.data_ptr(), logits.stride(0), logits.shape[0], out_dim,
                                                  out.data_ptr(), _stream())
    _lib.check(rc, "amb_displacement_out")
    launch_count += 1
    return out


def resize_h_u8(src: torch.Tensor, y0: int, n_rows: int, bounds: torch.Tensor, coeffs: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
    """Horizontal pass of Pillow's uint8 resample on source rows [y0, y0+n_rows): src (n, H, W, 3|4) u8 -> out (n, n_rows, out_w, 3)."""
    global launch_count
    _need(src, torch.uint8, "src")
    _need(out, torch.uint8, "out")
    _need(bounds, torch.int32, "bounds")
    _need(coeffs, torch.int32, "coeffs")
    assert src.dim() == 4 and src.is_contiguous() and out.is_contiguous() and bounds.is_contiguous() and coeffs.is_contiguous()
    n, H, W, cin = src.shape
    out_w, ksize = coeffs.shape
    assert out.shape == (n, n_rows, out_w, 3) and bounds.shape == (out_w, 2)
    rc = _lib.load_library().amb_resize_h_u8(src.data_ptr(), n, H, W, cin, y0, n_rows, bounds.data_ptr(), coeffs.data_ptr(),
                                             ksize, out_w, out.data_ptr(), _stream())
    _lib.check(rc, "amb_resize_h_u8")
    launch_count += 1
    return out


def resize_v_normalize(src: torch.Tensor, y0: int, bounds: torch.Tensor, coeffs: torch.Tensor, lut: torch.Tensor, mean, std,
                       out: torch.Tensor, out_u8: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Vertical pass + 1/255 rescale (lut) + mean/std + CHW: src (n, n_rows, out_w, 3) u8 -> out (n, 3, out_h, out_w) fp32."""
    global launch_count
    _need(src, torch.uint8, "src")
    _need(out, torch.float32, "out")
    _need(bounds, torch.int32, "bounds")
    _need(coeffs, torch.int32, "coeffs")
    _need(lut, torch.float32, "lut")
    assert src.is_contiguous() and out.is_contiguous() and lut.numel() == 256
    n, n_rows, out_w, _ = src.shape
    out_h, ksize = coeffs.shape
    assert out.shape == (n, 3, out_h, out_w) and bounds.shape == (out_h, 2)
    if out_u8 is not None:
        _need(out_u8, torch.uint8, "out_u8")
        assert out_u8.shape == (n, out_h, out_w, 3) and out_u8.is_contiguous()
    m = (C.c_float * 3)(*[float(v) for v in mean])
    s = (C.c_float * 3)(*[float(v) for v in std])
    rc = _lib.load_library().amb_resize_v_normalize(src.data_ptr(), n, n_rows, y0, out_w, bounds.data_ptr(), coeffs.data_ptr(),
                                                    ksize, out_h, lut.data_ptr(), m, s, out.data_ptr(),
                                                    out_u8.data_ptr() if out_u8 is not None else None, _stream())
    _lib.check(rc, "amb_resize_v_normalize")
    launch_count += 1
    return out


def alpha_stats(rgba: torch.Tensor) -> torch.Tensor:
    """(n, H, W, 4) u8 RGBA frames -> (n, 5) int32: xmin, ymin, xmax, ymax of alpha > 0 and the count of alpha > 127."""
    global launch_count
    _need(rgba, torch.uint8, "rgba")
    assert rgba.dim() == 4 and rgba.shape[3] == 4 and rgba.is_contiguous()
    n, H, W, _ = rgba.shape
    stats = torch.empty(n, 5, dtype=torch.int32, device=rgba.device)
    rc = _lib.load_library().amb_alpha_stats(rgba.data_ptr(), n, H, W, stats.data_ptr(), _stream())
    _lib.check(rc, "amb_alpha_stats")
    launch_count += 2
    return stats


def composite_crop_pad(rgba: torch.Tensor, box: tuple, pad_x: int, pad_y: int) -> torch.Tensor:
    """RGBA frames -> white-composited, cropped to box = (x, y, w, h), padded uint8 RGB frames (n, h + 2 pad_y, w + 2 pad_x, 3)."""
    global launch_count
    _need(rgba, torch.uint8, "rgba")
    assert rgba.dim() == 4 and rgba.shape[3] == 4 and rgba.is_contiguous()
    n, H, W, _ = rgba.shape
    x, y, w, h = (int(v) for v in box)
    out = torch.empty(n, h + 2 * pad_y, w + 2 * pad_x, 3, dtype=torch.uint8, device=rgba.device)
    rc = _lib.load_library().amb_composite_crop_pad(rgba.data_ptr(), n, H, W, x, y, w, h, int(pad_x), int(pad_y),
                                                    out.data_ptr(), _stream())
    _lib.check(rc, "amb_composite_crop_pad")
    launch_count += 1
    return out


def nearest_neighbors(query: torch.Tensor, reference: torch.Tensor, want_index: bool = True):
    """(Q, 3), (R, 3) fp32 CUDA points -> (distance (Q,) fp32, index (Q,) int32) of each query's nearest reference point."""
    global launch_count
    _need(query, torch.float32, "query")
    _need(reference, torch.float32, "reference")
    assert query.dim() == 2 and query.shape[1] == 3 and reference.dim() == 2 and reference.shape[1] == 3
    q, r = query.contiguous(), reference.contiguous()
    dist = torch.empty(q.shape[0], dtype=torch.float32, device=q.device)
    idx = torch.empty(q.shape[0], dtype=torch.int32, device=q.device) if want_index else None
    scratch = torch.empty(q.shape[0], dtype=torch.int64, device=q.device)
    rc = _lib.load_library().amb_nearest_neighbors(q.data_ptr(), q.shape[0], r.data_ptr(), r.shape[0], scratch.data_ptr(),
                                                   dist.data_ptr(), _ptr(idx), _stream())
    _lib.check(rc, "amb_nearest_neighbors")
    launch_count += 3
    return dist, idx


ICP_STARTS = 24


def adam_tables(lr: float, n_iter: int) -> tuple[torch.Tensor, torch.Tensor]:
    """torch Adam's per-step scalars in double, as torch.optim.Adam computes them (betas 0.9 / 0.999), rounded to fp32:
    (lr / (1 - 0.9^t), sqrt(1 - 0.999^t)) for t = 1..n_iter."""
    step = [lr / (1 - 0.9 ** t) for t in range(1, n_iter + 1)]
    bc2 = [(1 - 0.999 ** t) ** 0.5 for t in range(1, n_iter + 1)]
    return torch.tensor(step, dtype=torch.float32), torch.tensor(bc2, dtype=torch.float32)


def _icp_inputs(pred: torch.Tensor, gt: torch.Tensor, r_init: torch.Tensor):
    for t, name in ((pred, "pred"), (gt, "gt"), (r_init, "r_init")):
        _need(t, torch.float32, name)
    assert pred.dim() == 3 and pred.shape[2] == 3 and gt.dim() == 3 and gt.shape[2] == 3 and pred.shape[0] == gt.shape[0]
    assert r_init.shape == (ICP_STARTS, 3, 3)
    F, P, Q = pred.shape[0], pred.shape[1], gt.shape[1]
    if F == 0 or P == 0 or Q == 0:
        raise _lib.AmbError(f"gradient ICP needs non-empty clouds (F={F}, P_pred={P}, P_gt={Q})")
    nbytes = C.c_size_t()
    _lib.check(_lib.load_library().amb_icp_workspace_bytes(F, P, Q, C.byref(nbytes)), "amb_icp_workspace_bytes")
    ws = torch.empty(nbytes.value // 4, dtype=torch.float32, device=pred.device)
    return pred.contiguous(), gt.contiguous(), r_init.contiguous(), ws, F, P, Q


def icp_chamfer_grad(pred: torch.Tensor, gt: torch.Tensor, r_init: torch.Tensor, params: torch.Tensor):
    """(F, P, 3), (F, Q, 3), (24, 3, 3), params (F, 24, 12) = [r6d | T | s] -> (loss (F, 24), gradient (F, 24, 12)):
    the Chamfer loss of x = (s * p) @ (r_init[r] @ rot6d(r6d)) + T against gt, and its gradient, per (problem, start)."""
    global launch_count
    pred, gt, r_init, ws, F, P, Q = _icp_inputs(pred, gt, r_init)
    _need(params, torch.float32, "params")
    assert params.shape == (F, ICP_STARTS, 12)
    params = params.contiguous()
    loss = torch.empty(F, ICP_STARTS, dtype=torch.float32, device=pred.device)
    grad = torch.empty(F, ICP_STARTS, 12, dtype=torch.float32, device=pred.device)
    rc = _lib.load_library().amb_icp_chamfer_grad(pred.data_ptr(), gt.data_ptr(), F, P, Q, r_init.data_ptr(), params.data_ptr(),
                                                  ws.data_ptr(), ws.numel() * 4, loss.data_ptr(), grad.data_ptr(), _stream())
    _lib.check(rc, "amb_icp_chamfer_grad")
    launch_count += 3
    return loss, grad


def gradient_icp(pred: torch.Tensor, gt: torch.Tensor, r_init: torch.Tensor, lr: float = 0.01, n_iter: int = 200,
                 want_trace: bool = False):
    """Batched gradient ICP (actionbench/icp.py:53-112) on the device: (F, P, 3), (F, Q, 3), (24, 3, 3) ->
    (R (F, 3, 3), T (F, 3), s (F, 3), best loss (F,), best start (F,) int32, loss trace (n_iter, F, 24) or None)."""
    global launch_count
    pred, gt, r_init, ws, F, P, Q = _icp_inputs(pred, gt, r_init)
    if n_iter <= 0:
        raise _lib.AmbError(f"gradient_icp: n_iter must be positive (got {n_iter})")
    dev = pred.device
    step, bc2 = (t.to(dev) for t in adam_tables(lr, n_iter))
    R = torch.empty(F, 3, 3, dtype=torch.float32, device=dev)
    T = torch.empty(F, 3, dtype=torch.float32, device=dev)
    s = torch.empty(F, 3, dtype=torch.float32, device=dev)
    loss = torch.empty(F, dtype=torch.float32, device=dev)
    start = torch.empty(F, dtype=torch.int32, device=dev)
    trace = torch.empty(n_iter, F, ICP_STARTS, dtype=torch.float32, device=dev) if want_trace else None
    rc = _lib.load_library().amb_gradient_icp(pred.data_ptr(), gt.data_ptr(), F, P, Q, r_init.data_ptr(), n_iter, step.data_ptr(),
                                              bc2.data_ptr(), ws.data_ptr(), ws.numel() * 4, R.data_ptr(), T.data_ptr(),
                                              s.data_ptr(), loss.data_ptr(), start.data_ptr(), _ptr(trace), _stream())
    _lib.check(rc, "amb_gradient_icp")
    launch_count += 2 + 2 * n_iter
    return R, T, s, loss, start, trace


def transform_points(points: torch.Tensor, R: torch.Tensor, T: torch.Tensor, s: torch.Tensor) -> torch.Tensor:
    """(F, N, 3) points, per-problem R (F, 3, 3), T (F, 3), s (F, 3) -> (x * s) @ R + T, (F, N, 3)."""
    global launch_count
    for t, name in ((points, "points"), (R, "R"), (T, "T"), (s, "s")):
        _need(t, torch.float32, name)
    F = points.shape[0]
    assert points.dim() == 3 and points.shape[2] == 3 and R.shape == (F, 3, 3) and T.shape == (F, 3) and s.shape == (F, 3)
    points, R, T, s = points.contiguous(), R.contiguous(), T.contiguous(), s.contiguous()
    out = torch.empty_like(points)
    rc = _lib.load_library().amb_transform_points(points.data_ptr(), F, points.shape[1], R.data_ptr(), T.data_ptr(), s.data_ptr(),
                                                  out.data_ptr(), _stream())
    _lib.check(rc, "amb_transform_points")
    launch_count += 1
    return out


def cast_bf16(src: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    global launch_count
    _need(src, torch.float32, "src")
    assert src.is_contiguous()
    if out is None:
        out = torch.empty(src.shape, dtype=torch.bfloat16, device=src.device)
    rc = _lib.load_library().amb_cast_f32_bf16(src.data_ptr(), out.data_ptr(), src.numel(), _stream())
    _lib.check(rc, "amb_cast_f32_bf16")
    launch_count += 1
    return out


def timestep_embedding(t: torch.Tensor, channels: int, out: Optional[torch.Tensor] = None, *,
                       mask: Optional[torch.Tensor] = None, rows: Optional[int] = None) -> torch.Tensor:
    """Row r: sinusoidal embedding of t[r % len(t)] * (1 - mask[r]) (temporal_denoiser.py:209-213)."""
    global launch_count
    _need(t, torch.float32, "t")
    if mask is not None:
        _need(mask, torch.float32, "mask")
        rows = mask.numel()
    if rows is None:
        rows = t.numel()
    if out is None:
        out = torch.empty((rows, channels), dtype=torch.bfloat16, device=t.device)
    rc = _lib.load_library().amb_timestep_embedding(t.data_ptr(), t.numel(), _ptr(mask), rows, channels, out.data_ptr(), _stream())
    _lib.check(rc, "amb_timestep_embedding")
    launch_count += 1
    return out


def add_bias_rows(y: torch.Tensor, bias: torch.Tensor) -> None:
    global launch_count
    if y.dtype not in (torch.bfloat16, torch.float32):
        raise _lib.AmbError(f"add_bias_rows: unsupported dtype {y.dtype}")
    _need(y, y.dtype, "y")
    _need(bias, torch.float32, "bias")
    assert y.dim() == 2 and y.stride(1) == 1
    rc = _lib.load_library().amb_add_bias_rows(y.data_ptr(), int(y.dtype == torch.float32), y.stride(0), bias.data_ptr(),
                                               y.shape[0], y.shape[1], _stream())
    _lib.check(rc, "amb_add_bias_rows")
    launch_count += 1


def gemm(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, *, bias: Optional[torch.Tensor] = None,
         a2: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None, act: int = 0,
         col_scale: Optional[torch.Tensor] = None, row_map: Optional[tuple[int, int, int]] = None,
         norm: Optional[dict] = None, out2: Optional[torch.Tensor] = None, tag: str = "gemm") -> torch.Tensor:
    """out = epilogue(cat[a, a2] @ w.T).  a:(m,k1) bf16, a2:(m,k2) bf16 or None, w:(n,k1+k2) bf16, out bf16/fp32.

    norm = dict(cols=, seg=, w0=, w1=, eps=, rope_cols=, cos=, sin=, rows_per_pos=) enables the per-head
    RMSNorm(+RoPE) epilogue of attention_processor.py:106-130."""
    global launch_count
    _need(a, torch.bfloat16, "a")
    _need(w, torch.bfloat16, "w")
    assert a.dim() == 2 and w.dim() == 2 and out.dim() == 2
    assert a.stride(1) == 1 and w.stride(1) == 1 and out.stride(1) == 1
    g = _lib.GemmArgs()
    m, k1 = a.shape
    n, k = w.shape
    g.a, g.lda = a.data_ptr(), a.stride(0)
    if a2 is not None:
        _need(a2, torch.bfloat16, "a2")
        assert a2.shape[0] == m and a2.stride(1) == 1 and k1 + a2.shape[1] == k
        g.a2, g.lda2, g.k_split = a2.data_ptr(), a2.stride(0), k1
    else:
        assert k1 == k, f"a has k={k1}, w has k={k}"
        g.a2, g.lda2, g.k_split = None, 0, 0
    g.w, g.ldw = w.data_ptr(), w.stride(0)
    if out.dtype not in (torch.bfloat16, torch.float32):
        raise _lib.AmbError(f"gemm: unsupported output dtype {out.dtype}")
    g.c, g.ldc, g.c_fp32 = out.data_ptr(), out.stride(0), int(out.dtype == torch.float32)
    g.m, g.n, g.k = m, n, k
    if out2 is not None:  # bf16 copy of the result (GEMM operand of a later linear)
        _need(out2, torch.bfloat16, "out2")
        assert out2.shape == out.shape and out2.stride(1) == 1
        g.c2, g.ldc2 = out2.data_ptr(), out2.stride(0)
    else:
        g.c2, g.ldc2 = None, 0
    if bias is not None:
        _need(bias, torch.float32, "bias")
    g.bias = _ptr(bias)
    if residual is not None:
        assert residual.stride(1) == 1
        g.residual, g.ldr, g.res_fp32 = residual.data_ptr(), residual.stride(0), int(residual.dtype == torch.float32)
    else:
        g.residual, g.ldr, g.res_fp32 = None, 0, 0
    g.act = act
    if col_scale is not None:
        _need(col_scale, torch.float32, "col_scale")
    g.col_scale = _ptr(col_scale)
    if row_map is not None:
        g.grp_rows, g.grp_stride, g.row_off = row_map
    else:
        g.grp_rows = g.grp_stride = g.row_off = 0
    if norm is not None:
        g.norm_cols, g.norm_seg = norm.get("cols", 0), norm.get("seg", norm.get("cols", 0))
        g.norm_w0 = norm["w0"].data_ptr() if norm.get("w0") is not None else None
        g.norm_w1 = norm["w1"].data_ptr() if norm.get("w1") is not None else None
        g.norm_eps = float(norm.get("eps", 0.0))
        g.rope_cols = norm.get("rope_cols", 0)
        g.rope_cos = _ptr(norm.get("cos"))
        g.rope_sin = _ptr(norm.get("sin"))
        g.rope_rows_per_pos = norm.get("rows_per_pos", 1)
    else:
        g.norm_cols = g.norm_seg = g.rope_cols = 0
        g.norm_w0 = g.norm_w1 = g.rope_cos = g.rope_sin = None
        g.norm_eps = 0.0
        g.rope_rows_per_pos = 1
    with _Timed(tag, (m, n, k)):
        rc = _lib.load_library().amb_gemm_bf16(C.byref(g), _stream())
    _lib.check(rc, "amb_gemm_bf16")
    launch_count += 1
    return out


def attn_small_f32(qkv: torch.Tensor, frames: int, seq: int, heads: int, scale: float, out: torch.Tensor,
                   tag: str = "attn_small") -> torch.Tensor:
    """fp32 attention of `frames` independent sequences of `seq` <= 320 tokens, head_dim 64 (DinoV2).
    qkv: fp32 (frames * seq, 3 * heads * 64) = [q | k | v] of a fused projection; out: fp32 (frames * seq, heads * 64)."""
    global launch_count
    _need(qkv, torch.float32, "qkv")
    _need(out, torch.float32, "out")
    D = heads * 64
    assert qkv.dim() == 2 and out.dim() == 2 and qkv.stride(1) == 1 and out.stride(1) == 1
    assert qkv.shape == (frames * seq, 3 * D) and out.shape == (frames * seq, D)
    base = qkv.data_ptr()
    with _Timed(tag, (frames, heads, seq, seq, 64)):
        rc = _lib.load_library().amb_attn_small_f32(base, base + 4 * D, base + 8 * D, qkv.stride(0), frames, seq, heads,
                                                    float(scale), out.data_ptr(), out.stride(0), _stream())
    _lib.check(rc, "amb_attn_small_f32")
    launch_count += 1
    return out


def flash_attn(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, out: torch.Tensor, scale: float, *,
               kv_chunks: int = 1, tag: str = "attn") -> torch.Tensor:
    """softmax(scale q kᵀ) v, non-causal.  q:(B,Sq,H,D) k,v:(B,Sk,H,D) out:(B,Sq,H,D) — arbitrary (16-byte aligned)
    strides with unit stride on D, so views into a fused QKV buffer work in place.

    With kv_chunks > 1, k/v are (B, chunks, Sk_chunk, H, D) (rank-c all-gathered K/V of the frame-sharded window)."""
    global launch_count
    for t, nme in ((q, "q"), (k, "k"), (v, "v"), (out, "out")):
        _need(t, torch.bfloat16, nme)
        assert t.stride(-1) == 1
    a = _lib.AttnArgs()
    B, Sq, H, D = q.shape
    a.q, a.k, a.v, a.o = q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr()
    a.q_stride_b, a.q_stride_s, a.q_stride_h = q.stride(0), q.stride(1), q.stride(2)
    a.o_stride_b, a.o_stride_s, a.o_stride_h = out.stride(0), out.stride(1), out.stride(2)
    if kv_chunks > 1:
        assert k.dim() == 5 and v.dim() == 5 and k.shape[1] == kv_chunks
        a.k_stride_b, a.k_chunk_stride, a.k_stride_s, a.k_stride_h = k.stride(0), k.stride(1), k.stride(2), k.stride(3)
        a.v_stride_b, a.v_chunk_stride, a.v_stride_s, a.v_stride_h = v.stride(0), v.stride(1), v.stride(2), v.stride(3)
        a.sk_chunk = k.shape[2]
        a.sk = k.shape[1] * k.shape[2]
    else:
        assert k.dim() == 4 and v.dim() == 4
        a.k_stride_b, a.k_stride_s, a.k_stride_h = k.stride(0), k.stride(1), k.stride(2)
        a.v_stride_b, a.v_stride_s, a.v_stride_h = v.stride(0), v.stride(1), v.stride(2)
        a.k_chunk_stride = a.v_chunk_stride = 0
        a.sk_chunk = k.shape[1]
        a.sk = k.shape[1]
    a.kv_chunks = kv_chunks
    a.batch, a.heads, a.sq, a.head_dim = B, H, Sq, D
    a.scale = float(scale)
    with _Timed(tag, (B, H, Sq, a.sk, D)):
        rc = _lib.load_library().amb_flash_attn_fwd(C.byref(a), _stream())
    _lib.check(rc, "amb_flash_attn_fwd")
    launch_count += 1
    return out
