"""The GEMM error bound has teeth (no GPU): an fp32 stand-in for the kernel (torch's fp32 matmul, epilogue in fp32)
passes oracle.gemm_oracle.bound, and each subtle mistake a kernel could make fails it."""
import math

import pytest
import torch

from oracle import gemm_oracle as go


def _operands(m, n, k, seed=0):
    g = torch.Generator().manual_seed(seed)
    A = (torch.randn(m, k, generator=g) * 0.5).bfloat16()
    W = (torch.randn(n, k, generator=g) / math.sqrt(k)).bfloat16()
    return A, W, g


def _rope_pairs(h, cs, sn, swap=False):
    a, b = h[:, 0::2], h[:, 1::2]
    if swap:
        a, b = b, a
    return torch.stack([a * cs - b * sn, b * cs + a * sn], -1).reshape(h.shape)


def _standin(A, W, *, bias=None, act=0, col_scale=None, residual=None, row_map=None, norm=None, out_fp32=True,
             out_rows=None, mutation=None):
    """What a correct kernel computes, in fp32, with one optional mistake."""
    m, n = A.shape[0], W.shape[0]
    y = A.float() @ W.float().t()
    heads = max(norm.get("cols", 0), norm.get("rope_cols", 0)) if norm else 0
    yp = y[:, heads:]
    if bias is not None:
        b = bias[heads:].clone()
        if mutation == "bias_dropped_on_one_group":
            b[8:16] = 0
        yp = yp + b
    if act == 1:
        yp = torch.nn.functional.gelu(yp, approximate="tanh" if mutation == "tanh_gelu" else "none")
    if col_scale is not None:
        yp = yp * col_scale[heads:]
    dst = go._dst_rows(m, row_map, A.device)
    if mutation == "row_map_off_by_one":
        dst = dst + 1
    if residual is not None:
        r = residual.float()[dst][:, heads:]
        yp = yp + r + (r if mutation == "residual_twice" else 0)
    yh = y[:, :heads].clone()
    for c0 in range(0, heads, 128):
        h = yh[:, c0:c0 + 128]
        if c0 < norm["cols"]:
            w = norm["w0"] if c0 < norm["seg"] and mutation != "w1_for_q_head" else norm["w1"]
            h = h * torch.rsqrt(h.pow(2).mean(-1, keepdim=True) + norm["eps"]) * w
        if c0 < norm["rope_cols"]:
            pos = torch.arange(m) // norm["rows_per_pos"]
            h = _rope_pairs(h, norm["cos"][pos], norm["sin"][pos], swap=mutation == "rope_pairs_swapped")
        yh[:, c0:c0 + 128] = h
    y = torch.cat([yh, yp], 1)
    if mutation == "tail_row_zeroed":
        y[-1] = 0
    y = y if out_fp32 else y.bfloat16()
    out = torch.full((out_rows or m, n), float("nan"), dtype=y.dtype)
    out[dst] = y
    return out


def _norm(g, m, nc, seg, rc, rpp):
    npos = (m + rpp - 1) // rpp
    ang = torch.rand(npos, 64, generator=g) * 6.28
    return dict(cols=nc, seg=seg, w0=torch.rand(128, generator=g) + 0.5, w1=torch.rand(128, generator=g) + 0.5,
                eps=1e-6, rope_cols=rc, cos=ang.cos(), sin=ang.sin(), rows_per_pos=rpp)


def _case(kind, k=448):
    """(A, W, kwargs, out_rows) of a small problem exercising the epilogue feature `kind`."""
    m, n = 37, 256
    A, W, g = _operands(m, n, k)
    kw, out_rows = {}, None
    if kind == "gelu":
        kw = dict(bias=torch.randn(n, generator=g), act=1)
    elif kind == "bias":
        kw = dict(bias=torch.randn(n, generator=g))
    elif kind == "residual":
        kw = dict(bias=torch.randn(n, generator=g), col_scale=torch.randn(n, generator=g),
                  residual=torch.randn(m, n, generator=g))
    elif kind == "row_map":
        row_map = (8, 10, 1)
        out_rows = int(go._dst_rows(m, row_map, "cpu").max()) + 3
        kw = dict(bias=torch.randn(n, generator=g), residual=torch.randn(out_rows, n, generator=g).bfloat16(),
                  row_map=row_map)
    elif kind == "heads":
        kw = dict(bias=torch.randn(n, generator=g), norm=_norm(g, m, 128, 128, 128, 5))
    elif kind == "qk_heads":
        kw = dict(norm=_norm(g, m, 256, 128, 0, 1))
    return A, W, kw, out_rows


def _check(A, W, kw, out, out_rows, out_fp32):
    y, dst = go.reference(A, W, **kw)
    e = go.bound(A, W, out_fp32=out_fp32, **kw)
    bad, ratio = go.bound_violations(out[dst], y, e)
    # rows no logical row maps to must be left alone (NaN here)
    gap = torch.ones(out.shape[0], dtype=torch.bool)
    gap[dst] = False
    return bad + int((~torch.isnan(out[gap].float())).sum()), ratio


@pytest.mark.parametrize("kind", ["gelu", "bias", "residual", "row_map", "heads", "qk_heads"])
@pytest.mark.parametrize("k", [64, 448])
@pytest.mark.parametrize("out_fp32", [True, False])
def test_bound_accepts_fp32_standin(kind, k, out_fp32):
    A, W, kw, out_rows = _case(kind, k)
    out = _standin(A, W, out_fp32=out_fp32, out_rows=out_rows, **kw)
    bad, ratio = _check(A, W, kw, out, out_rows, out_fp32)
    assert bad == 0 and ratio <= 1.0, (bad, ratio)


@pytest.mark.parametrize("mutation,kind", [
    ("tanh_gelu", "gelu"),
    ("bias_dropped_on_one_group", "bias"),
    ("row_map_off_by_one", "row_map"),
    ("residual_twice", "residual"),
    ("rope_pairs_swapped", "heads"),
    ("w1_for_q_head", "qk_heads"),
    ("tail_row_zeroed", "bias"),
])
def test_bound_rejects_mutation(mutation, kind):
    A, W, kw, out_rows = _case(kind)
    out = _standin(A, W, out_fp32=True, out_rows=out_rows, mutation=mutation, **kw)
    bad, ratio = _check(A, W, kw, out, out_rows, True)
    assert bad > 0 and ratio > 1.0, (mutation, bad, ratio)


def test_bias_is_not_applied_on_head_columns():
    """The reference follows the kernel: bias reaches only the columns past the heads."""
    A, W, kw, _ = _case("heads")
    y_b, _ = go.reference(A, W, **kw)
    kw.pop("bias")
    y_nb, _ = go.reference(A, W, **kw)
    assert torch.equal(y_b[:, :128], y_nb[:, :128]) and not torch.equal(y_b[:, 128:], y_nb[:, 128:])


def test_guard_helpers():
    buf, view = go.guarded(5, 16, torch.bfloat16, "cpu")
    assert view.stride(0) == 64 + 16 + 256 and torch.isnan(buf.float()).all()
    before = buf.clone()
    view[1, 2] = 1.0
    written = torch.zeros(buf.shape, dtype=torch.bool)
    assert go.untouched_violations(buf, before, written) == 1
    written[8 + 1, 64 + 2] = True
    assert go.untouched_violations(buf, before, written) == 0
    assert go.bits_equal(buf, buf.clone()) and not go.bits_equal(buf, before)
