"""TEST INFRASTRUCTURE ONLY — fp64 reference and per-element error bound of `amb_gemm_bf16` (C = epilogue(A · Wᵀ)).

`reference()` computes in fp64 from the exact bf16 operand values and follows the documented epilogue order
(include/actionmesh_b200.h, csrc/gemm.cu `epilogue_tile` / `finish_and_store`):

* plain columns: bias -> GELU(erf) -> col_scale -> residual;
* head columns c < H = max(norm_cols, rope_cols), in heads of 128 columns: RMSNorm over the head (weight `w0` for heads
  starting below `norm_seg`, `w1` above) for c < norm_cols, then interleaved-pair RoPE, pair (2i, 2i+1) rotated by
  angle i of the fp32 tables at pos = logical row // rows_per_pos, for c < rope_cols.  Bias is NOT applied on head
  columns; it is applied on the columns past them;
* `row_map = (g, stride, off)` places logical row r at dst = (r // g) * stride + r % g + off; the residual is read at dst.

`bound()` gives a per-element tolerance from a-priori terms; nothing in it was fitted to a run.  u = 2^-24 is the
unit roundoff of fp32.

* Accumulation, ACC_PER_K * K * mag with mag = (|A| @ |W|ᵀ)_ij and ACC_PER_K = 2^-26.  The bf16 x bf16 products are
  exact in fp32 (8 + 8 significant bits).  The tensor core adds them 16 at a time (one UMMA_K step) into the fp32
  accumulator, so there are K/16 steps.  Each step is charged two fp32 ulps of the running magnitude, and the running
  magnitude never exceeds mag.  One ulp is the rounding of the step's result.  The other is the alignment of the 16
  products to the largest term, whose truncated bits are worth at most 16 x 2^-3 ulp when at least 3 guard bits are
  kept.  An ulp is at most 2^-23 |x|, so the bound is (K/16) * 2 * 2^-23 * mag = K * 2^-26 * mag.  For K = 64 that is
  2^-20 * mag.  This is the worst case; errors of random signs grow like sqrt(K), so the measured ratio is expected
  well below 1 and is reported by tests/test_gemm_contract_gpu.py.
* Each fp32 add or multiply in the epilogue adds u * (|a| + |b|) for a sum, u * |a b| for a product.
* GELU: |GELU'(x)| <= 1.13 (its maximum, at x = sqrt(2)), so an input error e becomes at most 1.13 e.  The
  Abramowitz-Stegun 7.1.26 formula the kernel evaluates differs from x * Phi(x) by at most GELU_ABS = 4.2e-7 over all x
  including the rounding of its fp32 result (gemm.cu's comment at `gelu_erf`; for |x| > 13 the tail underflows and the
  result is x exactly).  The approximate rcp / ex2 add about 2^-21 relative to a term below 0.17 |x|, which the extra
  2^-23 |GELU(x)| term covers.
* RMSNorm: the kernel computes rs = rsqrt(sum(v^2) / 128 + eps) and v * (rs * w).  The error of sum(v^2) is at most
  2 * sum(|v| e) from the inputs plus 130 u * sum(v^2) from 128 sequential fp32 adds, one squaring and the scaling.  That
  relative error is halved by the square root.  rsqrtf adds at most 2 ulp (2^-22), and the two products add 2u.  The
  output error is rs |w| e + |y| (rel_rs + 2u).
* RoPE: y0 = a cos - b sin, y1 = b cos + a sin with exact fp32 tables, error |cos| e_a + |sin| e_b + 3u (|a cos| + |b sin|).
* Output rounding: one fp32 ulp, 2^-23 |y|, or for bf16 (8 significant bits, round to nearest) the unit roundoff
  2^-8 |y|.  Both are applied to |y| + e, because the kernel rounds its own value and not the exact one.  A correct bf16
  result can therefore use almost all of its bound.

`guarded()` / `untouched_violations()` put an output into a larger buffer prefilled with a sentinel bit pattern and
check, bit for bit, that nothing outside the written elements changed.
"""
from __future__ import annotations

import math
from typing import Optional

import torch

U32 = 2.0 ** -24          # fp32 unit roundoff
ACC_PER_K = 2.0 ** -26    # accumulation bound per unit of K, times mag (see the module docstring)
GELU_ABS = 4.2e-7         # |kernel GELU - x * Phi(x)| over all x, fp32 result rounding included
GELU_LIP = 1.13           # max |d/dx x * Phi(x)|
RSQRT_REL = 2.0 ** -22    # rsqrtf: at most 2 ulp
BF16_ULP = 2.0 ** -8
F32_ULP = 2.0 ** -23

# Sentinel bit patterns: quiet NaNs with a payload no arithmetic produces.
SENTINEL_BITS = {torch.bfloat16: 0x7FA5, torch.float32: 0x7FA5A5A5}
_INT_VIEW = {torch.bfloat16: torch.int16, torch.float32: torch.int32}


def _f64(t):
    return None if t is None else t.double()


def _dst_rows(m: int, row_map, device) -> torch.Tensor:
    r = torch.arange(m, device=device)
    if row_map is None:
        return r
    g, stride, off = row_map
    return (r // g) * stride + r % g + off


def _evaluate(A, W, *, a2=None, bias=None, act=0, col_scale=None, residual=None, row_map=None, norm=None,
              out_fp32=False):
    """(y, e, dst): fp64 values and error bounds of the m logical rows, and their destination rows."""
    Af = A.double() if a2 is None else torch.cat([A.double(), a2.double()], 1)
    Wf = W.double()
    m, K = Af.shape
    n = Wf.shape[0]
    assert Wf.shape[1] == K
    y = Af @ Wf.t()
    e = ACC_PER_K * K * (Af.abs() @ Wf.abs().t())
    dst = _dst_rows(m, row_map, y.device)
    heads = 0
    if norm is not None:
        heads = max(norm.get("cols", 0), norm.get("rope_cols", 0))
    yh, eh = y[:, :heads].clone(), e[:, :heads].clone()
    yp, ep = y[:, heads:], e[:, heads:]

    # ---- plain columns: bias -> GELU -> col_scale -> residual ----
    if bias is not None:
        b = _f64(bias)[heads:]
        ep = ep + U32 * (yp.abs() + b.abs())
        yp = yp + b
    if act == 1:
        g = 0.5 * yp * torch.erfc(-yp / math.sqrt(2.0))
        ep = GELU_LIP * ep + GELU_ABS + F32_ULP * g.abs()
        yp = g
    if col_scale is not None:
        s = _f64(col_scale)[heads:]
        yp = yp * s
        ep = ep * s.abs() + U32 * yp.abs()
    if residual is not None:
        r = _f64(residual)[dst][:, heads:]
        ep = ep + U32 * (yp.abs() + r.abs())
        yp = yp + r

    # ---- head columns: per-128 RMSNorm, then RoPE; no bias ----
    if heads:
        nc, rc = norm.get("cols", 0), norm.get("rope_cols", 0)
        seg = norm.get("seg", nc)
        eps = float(norm.get("eps", 0.0))
        w0 = norm.get("w0")
        w1 = norm.get("w1") if norm.get("w1") is not None else w0
        rpp = max(int(norm.get("rows_per_pos", 1)), 1)
        for c0 in range(0, heads, 128):
            h, he = yh[:, c0:c0 + 128], eh[:, c0:c0 + 128]
            if c0 < nc:
                w = _f64(w0 if c0 < seg else w1)
                ss = (h * h).sum(-1, keepdim=True)
                den = ss / 128 + eps
                rel_ss = (2 * (h.abs() * he).sum(-1, keepdim=True) + 130 * U32 * ss) / 128 / den
                rs = den.rsqrt()
                hn = h * rs * w
                he = rs * w.abs() * he + hn.abs() * (0.5 * rel_ss + RSQRT_REL + 3 * U32)
                h = hn
            if c0 < rc:
                pos = torch.arange(m, device=y.device) // rpp
                cs, sn = _f64(norm["cos"])[pos], _f64(norm["sin"])[pos]     # (m, 64)
                a, b = h[:, 0::2], h[:, 1::2]
                ea, eb = he[:, 0::2], he[:, 1::2]
                y0, y1 = a * cs - b * sn, b * cs + a * sn
                e0 = cs.abs() * ea + sn.abs() * eb + 3 * U32 * ((a * cs).abs() + (b * sn).abs())
                e1 = cs.abs() * eb + sn.abs() * ea + 3 * U32 * ((b * cs).abs() + (a * sn).abs())
                h = torch.stack([y0, y1], -1).reshape(m, 128)
                he = torch.stack([e0, e1], -1).reshape(m, 128)
            yh[:, c0:c0 + 128], eh[:, c0:c0 + 128] = h, he

    y = torch.cat([yh, yp], 1)
    e = torch.cat([eh, ep], 1)
    e = e + (F32_ULP if out_fp32 else BF16_ULP) * (y.abs() + e)
    return y, e, dst


def reference(A, W, **kw):
    """fp64 result (m, n) of the m logical rows and their destination rows dst (m,) in the output."""
    y, _, dst = _evaluate(A, W, **kw)
    return y, dst


def bound(A, W, **kw):
    """Per-element tolerance (m, n) for the kernel's result of reference(A, W, **kw)."""
    return _evaluate(A, W, **kw)[1]


def bound_violations(out_rows, y, e):
    """Elements of the kernel's rows (m, n) outside |out - y| <= e (NaN counts as a violation), and max(err / bound)."""
    err = (out_rows.double() - y).abs().nan_to_num(nan=math.inf)
    bad = ~(err <= e)
    return int(bad.sum()), float((err / e).max())


def guarded(rows, cols, dtype, device, *, row0=8, col0=64, margin=256):
    """A (rows, cols) view at (row0, col0) of a buffer with `margin` more rows and columns after it, prefilled with the
    dtype's sentinel bit pattern.  Returns (buffer, view)."""
    buf = torch.empty(row0 + rows + margin, col0 + cols + margin, dtype=dtype, device=device)
    buf.view(_INT_VIEW[dtype]).fill_(_signed(SENTINEL_BITS[dtype], dtype))
    return buf, buf[row0:row0 + rows, col0:col0 + cols]


def _signed(bits, dtype):
    width = 16 if dtype == torch.bfloat16 else 32
    return bits - (1 << width) if bits >= 1 << (width - 1) else bits


def untouched_violations(buf, before, written):
    """Elements of `buf` outside the boolean mask `written` whose bits differ from `before` (a copy taken before the call)."""
    it = _INT_VIEW[buf.dtype]
    changed = buf.view(it) != before.view(it)
    return int((changed & ~written).sum())


def bits_equal(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and bool((a.view(_INT_VIEW[a.dtype]) == b.view(_INT_VIEW[b.dtype])).all())
