"""Kernel parity on the B200 (-m gpu): every C-ABI compute entry point against a torch fp32 reference of the same op
on seeded inputs.  Tolerances: outputs are bf16, so relative Frobenius error <= 4e-3 (bf16 has 8 mantissa bits,
2^-9 = 1.95e-3 per rounding; two roundings on the fused paths) unless the output is fp32 (1e-5)."""
import math
import os
import sys

import pytest
import torch

from conftest import ROOT

sys.path.insert(0, os.path.join(ROOT, "tools"))
pytestmark = pytest.mark.gpu

BF16_REL = 4e-3
F32_REL = 1e-5


@pytest.fixture(scope="module")
def probe(amb_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    import gpu_probe

    return gpu_probe


def test_elementwise_group(probe):
    res = {}
    probe.group_elementwise(res)
    assert res["k9"]["rel_fro"] < 1e-6 and res["k9"]["observed_bit_identical"]
    for k in ("ln_1024_bfloat16", "ln_1024_float32", "ln_2048_bfloat16", "ln_2048_float32"):
        assert res[k]["rel_fro"] < BF16_REL and not res[k]["nan"]
    assert res["cast"]["max_abs"] == 0.0
    assert res["timestep_emb"]["rel_fro"] < BF16_REL
    assert res["add_bias_rows"]["max_abs"] == 0.0


@pytest.mark.parametrize("name,kw", [
    ("basic", dict(m=128, n=256, k=64)),
    ("k128", dict(m=256, n=256, k=128)),
    ("n128_tail", dict(m=300, n=128, k=192)),
    ("persistent_many_tiles", dict(m=128 * 40, n=2048, k=256)),
    ("bias_gelu_res", dict(m=512, n=512, k=256, bias=True, act=1, residual=True)),
    ("two_source_a", dict(m=384, n=256, k=512, a2=True, bias=True)),
    ("row_remap", dict(m=256, n=256, k=64, bias=True, row_map=(64, 65, 1))),
    ("qkv_norm_rope", dict(m=300, n=768, k=256, norm=(512, 256, 512, 100))),
    ("q_norm_only", dict(m=300, n=256, k=256, norm=(256, 256, 0, 1))),
    ("kv_norm_bias", dict(m=300, n=512, k=128, norm=(256, 256, 0, 1), bias=True)),
    ("single_row", dict(m=1, n=128, k=64, bias=True)),
    ("max_rows_default_cfg", dict(m=65568, n=256, k=64)),
])
def test_gemm_bf16_out(probe, name, kw):
    res = {}
    m, n, k = kw.pop("m"), kw.pop("n"), kw.pop("k")
    probe._gemm_case(res, name, m, n, k, **kw)
    assert not res[name]["nan"] and res[name]["rel_fro"] < BF16_REL, res[name]


@pytest.mark.parametrize("name,kw", [
    ("n64_fp32", dict(m=200, n=64, k=128, bias=True, out_fp32=True)),
    ("fp32_res_colscale", dict(m=257, n=256, k=128, bias=True, residual=True, res_fp32=True, out_fp32=True, col_scale=True)),
])
def test_gemm_fp32_out(probe, name, kw):
    res = {}
    m, n, k = kw.pop("m"), kw.pop("n"), kw.pop("k")
    probe._gemm_case(res, name, m, n, k, **kw)
    assert res[name]["rel_fro"] < F32_REL, res[name]


def test_gemm_is_linear_in_a(probe):
    """Size-independent property at full width: gemm(a1 + a2) == gemm(a1) + gemm(a2) up to bf16 rounding, and the
    two-source K split equals the concatenated GEMM bit-for-bit."""
    from actionmesh_b200 import ops

    g = torch.Generator().manual_seed(3)
    a1 = torch.randn(4096, 2048, generator=g).cuda().bfloat16()
    a2 = torch.randn(4096, 2048, generator=g).cuda().bfloat16()
    w = (torch.randn(2048, 4096, generator=g) / 64).cuda().bfloat16()
    cat = torch.cat([a1, a2], 1).contiguous()
    o1 = torch.empty(4096, 2048, device="cuda", dtype=torch.float32)
    o2 = torch.empty_like(o1)
    ops.gemm(cat, w, o1)
    ops.gemm(a1, w, o2, a2=a2)
    assert torch.equal(o1, o2)


@pytest.mark.parametrize("name,args,kw", [
    ("one_tile_vones", (1, 1, 256, 64, 128), dict(mode="vones")),
    ("one_tile_kzero", (1, 1, 256, 64, 128), dict(mode="kzero")),
    ("two_tiles", (1, 1, 256, 128, 128), {}),
    ("stage_wrap", (1, 2, 256, 320, 128), {}),
    ("ragged_q300_k257", (2, 2, 300, 257, 128), {}),
    ("single_query_single_key", (1, 1, 1, 1, 128), {}),
    ("sharp_rescale", (1, 2, 512, 1024, 128), dict(mode="sharp")),
    ("fused_qkv_strided", (2, 4, 520, 520, 128), dict(fused=True)),
    ("kv_chunks2", (2, 2, 256, 400, 128), dict(kv_chunks=2)),
    ("kv_chunks8_rank_of_8", (1, 2, 2 * 2049, 8 * 2 * 2049, 128), dict(kv_chunks=8)),   # 8-GPU frame-sharded window
    ("d64_s257", (3, 4, 257, 257, 64), {}),
    ("d64_fused", (2, 16, 257, 257, 64), dict(fused=True)),
    ("window_t2", (2, 16, 2 * 2049, 2 * 2049, 128), dict(fused=True)),
    # >= 48 key tiles: the CTA-pair kernel.  Logits with std 8 push most rows out of the fixed-reference safe range, so the
    # units are marked dirty by the fast pass and recomputed by the exact pass launched behind it (ragged q and key tails)
    ("pair_dirty_units_fixup", (1, 2, 300, 128 * 50 + 17, 128), dict(mode="sharp8")),
    ("pair_clean_ragged", (2, 2, 300, 128 * 50 + 17, 128), {}),
    # one key far above the row reference, in a key slot whose exp2 is the FMA-pipe polynomial: must be caught (argument clamp
    # at 127 -> 2^127 -> row-sum range check) and the unit redone exactly; the output is then v of that key
    ("pair_single_spike_key", (1, 2, 300, 128 * 50, 128), dict(mode="spike")),
])
def test_flash_attention(probe, name, args, kw):
    res = {}
    probe._attn_case(res, name, *args, **kw)
    assert not res[name]["nan"] and res[name]["rel_fro"] < BF16_REL, res[name]


@pytest.mark.parametrize("name,B,H,Sq,Sk,D", [
    ("d64", 2, 3, 300, 257, 64),
    ("d128_short_keys", 2, 3, 300, 128 * 7 + 5, 128),     # < 48 key tiles: the single-CTA kernel
    ("d128_pair", 2, 2, 300, 128 * 48 + 5, 128),          # >= 48 key tiles: the CTA-pair kernel
])
def test_flash_attention_output_guard_bands(probe, name, B, H, Sq, Sk, D):
    """The output is a strided view (rows, heads and head_dim inside a wider buffer) of a buffer prefilled with a NaN
    sentinel: every element outside the view keeps its bits, with ragged Sq and B, H > 1."""
    from actionmesh_b200 import ops
    from oracle import gemm_oracle as go

    g = torch.Generator().manual_seed(11)
    q = torch.randn(B, Sq, H, D, generator=g).cuda().bfloat16()
    k = torch.randn(B, Sk, H, D, generator=g).cuda().bfloat16()
    v = torch.randn(B, Sk, H, D, generator=g).cuda().bfloat16()
    buf = torch.empty(B, 8 + Sq + 256, H, 32 + D + 64, device="cuda", dtype=torch.bfloat16)
    buf.view(torch.int16).fill_(go.SENTINEL_BITS[torch.bfloat16])
    o = buf[:, 8:8 + Sq, :, 32:32 + D]
    before = buf.clone()
    ops.flash_attn(q, k, v, o, 1 / math.sqrt(D))
    torch.cuda.synchronize()
    written = torch.zeros(buf.shape, dtype=torch.bool, device="cuda")
    written[:, 8:8 + Sq, :, 32:32 + D] = True
    assert go.untouched_violations(buf, before, written) == 0
    ref = probe._attn_ref(q, k, v, 1 / math.sqrt(D))
    err = float((o.float() - ref).norm() / ref.norm())
    assert err < BF16_REL and not torch.isnan(o).any(), err


def test_flash_attention_late_rescale(probe):
    """Running-max rescale AFTER the first key tile: keys are ordered so that every row's maximum keeps growing by more
    than the lazy-rescale threshold (2^8) along the key axis, with a ragged tail tile."""
    from actionmesh_b200 import ops

    g = torch.Generator().manual_seed(5)
    _late_rescale_case(probe, 128 * 9 + 17)


def test_flash_attention_late_rescale_pair_kernel(probe):
    """The same construction over 50 key tiles: the CTA-pair kernel, every unit dirty, exact pass with in-loop rescales."""
    _late_rescale_case(probe, 128 * 50 + 17)


def _late_rescale_case(probe, S):
    from actionmesh_b200 import ops

    g = torch.Generator().manual_seed(5)
    B, H, D = 1, 2, 128
    q = torch.randn(B, S, H, D, generator=g)
    k = torch.randn(B, S, H, D, generator=g) * 0.05
    v = torch.randn(B, S, H, D, generator=g)
    # key t gets a component along the mean query direction growing with t => logits ramp up by ~12 nats per tile
    qdir = q.mean(dim=1, keepdim=True)
    qdir = qdir / qdir.norm(dim=-1, keepdim=True)
    ramp = (torch.arange(S, dtype=torch.float32) / 128.0).floor()[None, :, None, None]
    k = k + ramp * 12.0 * qdir * (math.sqrt(D) / (q * qdir).sum(-1, keepdim=True).abs().mean())
    q, k, v = (t.cuda().bfloat16() for t in (q, k, v))
    o = torch.empty_like(q)
    ops.flash_attn(q, k, v, o, 1 / math.sqrt(D))
    ref = probe._attn_ref(q, k, v, 1 / math.sqrt(D))
    err = float((o.float() - ref).norm() / ref.norm())
    assert err < BF16_REL and not torch.isnan(o).any(), err


def test_flash_attention_full_window_properties(probe):
    """Default-config shape (B=2, H=16, S=32 784): with V == 1 every output must be exactly 1 (softmax rows sum to 1),
    and permuting the keys must not change the result beyond accumulation-order noise."""
    from actionmesh_b200 import ops

    g = torch.Generator().manual_seed(8)
    B, S, H, D = 1, 32784, 2, 128
    q = torch.randn(B, S, H, D, generator=g).cuda().bfloat16()
    k = torch.randn(B, S, H, D, generator=g).cuda().bfloat16()
    v = torch.ones(B, S, H, D, device="cuda", dtype=torch.bfloat16)
    o = torch.empty_like(q)
    ops.flash_attn(q, k, v, o, 1 / math.sqrt(D))
    assert (o.float() - 1).abs().max() < 1e-2
    v = torch.randn(B, S, H, D, generator=g).cuda().bfloat16()
    perm = torch.randperm(S, generator=g).cuda()
    o1, o2 = torch.empty_like(q), torch.empty_like(q)
    ops.flash_attn(q, k, v, o1, 1 / math.sqrt(D))
    ops.flash_attn(q, k[:, perm].contiguous(), v[:, perm].contiguous(), o2, 1 / math.sqrt(D))
    assert (o1.float() - o2.float()).abs().max() < 2e-3
