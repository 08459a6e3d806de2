"""The GEMM contract on the B200 (-m gpu): every kernel path of amb_gemm_bf16 and every epilogue it supports, against the
fp64 reference of oracle/gemm_oracle.py, per element, within its a-priori bound.

amb_gemm_bf16 dispatches to four kernels (csrc/gemm.cu, end of file), mirrored by `dispatch()` below:

    P2    n % 256 == 0 and m >= 256   gemm2_bf16_kernel<6>: CTA pair, 256 x 256 tiles
    P256  n % 256 == 0 and m < 256    gemm_bf16_kernel<256, 4>
    P128  n % 128 == 0 otherwise      gemm_bf16_kernel<128, 6>
    P64   otherwise                   gemm_bf16_kernel<64, 8>

Every output (and `out2`) is a view of a larger buffer prefilled with a sentinel bit pattern: 8 rows and 64 columns
before it, 256 rows and 256 columns after it, so a store outside the view changes a canary instead of unrelated memory.
Every element the call must not write is checked bit for bit afterwards, including the gap rows a `row_map` skips.

Each case prints its max(err / bound); tests/test_gemm_oracle_cpu.py shows the bound rejects subtle mistakes.
"""
import dataclasses
import math
import re

import pytest
import torch

from oracle import gemm_oracle as go

pytestmark = pytest.mark.gpu

PATHS = ("P2", "P256", "P128", "P64")
HEAD_PATHS = ("P2", "P256", "P128")            # the head epilogue needs n % 128 == 0
N_OF = {"P2": 512, "P256": 512, "P128": 384, "P64": 192}
MID_M = {"P2": 400, "P256": 129, "P128": 300, "P64": 300}
TAILS = {"P2": (257, 300, 400), "P256": (1, 127, 129, 255), "P128": (1, 129, 300), "P64": (1, 129, 300)}
ROW0, COL0 = 8, 64
DEV = "cuda"


def dispatch(m, n):
    """Mirror of amb_gemm_bf16's choice of kernel."""
    if n % 256 == 0 and m >= 256:
        return "P2"
    if n % 256 == 0:
        return "P256"
    if n % 128 == 0:
        return "P128"
    return "P64"


def persistent_shape(path, sms):
    """(m, n) with at least 3 x sms tiles, so every CTA (or CTA pair) reuses both TMEM accumulators."""
    if path == "P2":
        return math.ceil(3 * sms / 2) * 256 - 100, 512     # 2 column tiles; the last pair's peer is partly valid
    if path == "P256":
        return 255, 256 * math.ceil(3 * sms / 2)           # 2 row tiles
    return sms * 128 + 77, N_OF[path]                      # 3 column tiles, sms + 1 row tiles


# epilogue features: keyword spec of _run
FEATURES = {
    "none": {},
    "bias": dict(bias=True),
    "bias_gelu": dict(bias=True, act=1),
    "bias_gelu_f32": dict(bias=True, act=1, out_fp32=True),
    "cs_res_bf16": dict(col_scale=True, res="bf16"),
    "cs_res_f32": dict(col_scale=True, res="f32", out_fp32=True),
    "res_alias": dict(bias=True, res="bf16", alias=True),
    "out2_alias_f32": dict(bias=True, res="f32", alias=True, out_fp32=True, out2=True),   # the fp32 residual stream
    "a2_k64": dict(bias=True, a2=64),
    "a2_k192": dict(bias=True, a2=192),
    "row_map_res": dict(bias=True, res="bf16", row_map=(64, 70, 3)),
    "row_map_res_alias": dict(bias=True, res="bf16", alias=True, row_map=(100, 103, 1)),  # the patch-embedding pattern
    "strided": dict(bias=True, res="bf16", strided=True),
}
HEAD_FEATURES = {   # norm = (norm_cols, norm_seg, rope_cols, rows_per_pos)
    "q_norm": dict(norm=(128, 128, 0, 1)),
    "qk_norm_w0w1": dict(norm=(256, 128, 0, 1)),
    "norm_rope_rpp100": dict(norm=(256, 128, 256, 100)),
    "rope_only": dict(norm=(0, 0, 256, 3)),
    "norm_bias_past_heads": dict(norm=(128, 128, 128, 7), bias=True),
}


@dataclasses.dataclass(frozen=True)
class Case:
    name: str
    path: str
    m: int            # 0: persistent shape, sized from the device
    n: int
    k: int
    tags: tuple
    spec: dict = dataclasses.field(default_factory=dict, hash=False)
    det: bool = False

    def shape(self, sms):
        if self.m == 0:
            return persistent_shape(self.path, sms) + (self.k,)
        return self.m, self.n, self.k


def _cases():
    out = []
    for p in PATHS:
        n, mid = N_OF[p], MID_M[p]
        for m in TAILS[p]:
            out.append(Case(f"{p}_tail_m{m}", p, m, n, 448, (f"m{m}",), dict(bias=True, res="bf16")))
        for k in (64, 4096):
            out.append(Case(f"{p}_k{k}", p, mid, n, k, (f"k{k}",), dict(bias=True)))
        feats = dict(FEATURES, **(HEAD_FEATURES if p in HEAD_PATHS else {}))
        for f, spec in feats.items():
            out.append(Case(f"{p}_{f}", p, mid, n, 448, (f, "k448"), spec))
        out.append(Case(f"{p}_persistent", p, 0, 0, 64, ("persist", "det"),
                        dict(bias=True, act=1, col_scale=True, res="bf16"), det=True))
    return out


CASES = _cases()
REQUIRED = {p: set(FEATURES) | ({*HEAD_FEATURES} if p in HEAD_PATHS else set()) | {f"m{m}" for m in TAILS[p]}
            | {"k64", "k448", "k4096", "persist", "det"} for p in PATHS}


@pytest.fixture(scope="module")
def sms(amb_lib):
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.cuda.get_device_properties(0).multi_processor_count


def _operands(case, m, n, k, g, dev):
    A = (torch.randn(m, k, generator=g) * 0.5).bfloat16()
    W = (torch.randn(n, k, generator=g) / math.sqrt(k)).bfloat16()
    if case.spec.get("strided"):    # A a column slice (lda > k); W a row slice and a column slice (ldw > k)
        Abig = torch.zeros(m, k + 128, dtype=torch.bfloat16)
        Abig[:, 64:64 + k] = A
        Wbig = torch.zeros(n + 48, k + 192, dtype=torch.bfloat16)
        Wbig[16:16 + n, 64:64 + k] = W
        return Abig.to(dev)[:, 64:64 + k], Wbig.to(dev)[16:16 + n, 64:64 + k]
    return A.to(dev), W.to(dev)


def _call(case, A, W, kw, mo, n, dtype):
    """One amb_gemm_bf16 call into fresh guarded buffers: (buf, view, before, out2 triple or None, residual values)."""
    from actionmesh_b200 import ops

    s = case.spec
    buf, view = go.guarded(mo, n, dtype, A.device, row0=ROW0, col0=COL0)
    kw = dict(kw)
    res_vals = None
    if s.get("res"):
        R = kw.pop("_R")
        res_vals = R
        if s.get("alias"):
            view.copy_(R)
            kw["residual"] = view
        elif s.get("strided"):
            Rbig = torch.zeros(mo, n + 72, dtype=R.dtype, device=A.device)    # ldr = n + 72 != ldc
            Rbig[:, :n] = R
            kw["residual"] = Rbig[:, :n]
        else:
            kw["residual"] = R
    o2 = None
    if s.get("out2"):
        buf2, view2 = go.guarded(mo, n, torch.bfloat16, A.device, row0=ROW0, col0=COL0)
        kw["out2"] = view2
        o2 = (buf2, view2, buf2.clone())
    before = buf.clone()
    a2 = s.get("a2")
    if a2:
        ops.gemm(A[:, :a2], W, view, a2=A[:, a2:], **kw)
    else:
        ops.gemm(A, W, view, **kw)
    torch.cuda.synchronize()
    return buf, view, before, o2, res_vals


def _written(buf, dst, n):
    w = torch.zeros(buf.shape, dtype=torch.bool, device=buf.device)
    w[ROW0 + dst, COL0:COL0 + n] = True
    return w


def _run(case, sms):
    m, n, k = case.shape(sms)
    assert dispatch(m, n) == case.path, (case.name, m, n)
    s = case.spec
    dev = DEV
    g = torch.Generator().manual_seed(1000 + CASES.index(case))
    A, W = _operands(case, m, n, k, g, dev)
    dtype = torch.float32 if s.get("out_fp32") else torch.bfloat16
    kw = {}
    if s.get("bias"):
        kw["bias"] = torch.randn(n, generator=g).to(dev)
    if s.get("act"):
        kw["act"] = 1
    if s.get("col_scale"):
        kw["col_scale"] = torch.randn(n, generator=g).to(dev)
    row_map = s.get("row_map")
    mo = m
    if row_map:
        kw["row_map"] = row_map
        mo = int(go._dst_rows(m, row_map, "cpu").max()) + 3   # two unused rows at the end of the view as well
    if s.get("norm"):
        nc, seg, rc, rpp = s["norm"]
        ang = torch.rand((m + rpp - 1) // rpp, 64, generator=g) * 6.28
        kw["norm"] = dict(cols=nc, seg=seg, eps=1e-6, rope_cols=rc, rows_per_pos=rpp,
                          w0=(torch.rand(128, generator=g) + 0.5).to(dev) if nc else None,
                          w1=(torch.rand(128, generator=g) + 0.5).to(dev) if nc else None,
                          cos=ang.cos().to(dev) if rc else None, sin=ang.sin().to(dev) if rc else None)
    if s.get("res"):
        kw["_R"] = torch.randn(mo, n, generator=g).to(dev).to(torch.float32 if s["res"] == "f32" else torch.bfloat16)

    buf, view, before, o2, R = _call(case, A, W, kw, mo, n, dtype)

    okw = {key: v for key, v in kw.items() if key != "_R"}
    okw["residual"] = R
    Aref = A if not s.get("a2") else A[:, :s["a2"]]
    a2ref = A[:, s["a2"]:] if s.get("a2") else None
    y, dst = go.reference(Aref, W, a2=a2ref, **okw)
    e = go.bound(Aref, W, a2=a2ref, out_fp32=dtype == torch.float32, **okw)
    bad, ratio = go.bound_violations(view[dst], y, e)
    canaries = go.untouched_violations(buf, before, _written(buf, dst, n))
    extra = {}
    if o2 is not None:
        buf2, view2, before2 = o2
        extra["out2_bits"] = go.bits_equal(view2[dst], view[dst].bfloat16())
        canaries += go.untouched_violations(buf2, before2, _written(buf2, dst, n))
    if s.get("a2"):   # the two-source call equals the concatenated-A call on the same path bit for bit
        cat = dataclasses.replace(case, spec={key: v for key, v in s.items() if key != "a2"})
        _, view_c, _, _, _ = _call(cat, A.contiguous(), W, kw, mo, n, dtype)
        extra["a2_bits"] = go.bits_equal(view_c, view)
    if case.det:      # no atomics: a second identical call is bit-identical
        _, view_d, _, _, _ = _call(case, A, W, kw, mo, n, dtype)
        extra["det_bits"] = go.bits_equal(view_d, view)
    print(f"\ngemm-contract {case.name:<26s} {case.path:<4s} m={m:<6d} n={n:<6d} k={k:<5d} "
          f"max(err/bound)={ratio:.3e} bound_violations={bad} canaries={'intact' if canaries == 0 else canaries} "
          + " ".join(f"{key}={v}" for key, v in extra.items()))
    return bad, ratio, canaries, extra


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_gemm_contract(sms, case):
    bad, ratio, canaries, extra = _run(case, sms)
    assert bad == 0, f"{case.name}: {bad} elements outside the bound, max(err/bound) = {ratio:.3g}"
    assert canaries == 0, f"{case.name}: {canaries} elements outside the output changed"
    assert all(extra.values()), (case.name, extra)


def test_every_path_feature_pair_is_covered(sms):
    """Each required (path, feature) pair has a case whose shape the dispatch mirror sends down that path."""
    covered = {p: set() for p in PATHS}
    for c in CASES:
        m, n, k = c.shape(sms)
        covered[dispatch(m, n)].update(c.tags)
    for p in PATHS:
        print(f"\ngemm-contract coverage {p}: {sorted(covered[p] & REQUIRED[p])}")
        assert REQUIRED[p] <= covered[p], (p, sorted(REQUIRED[p] - covered[p]))


_BN = {"P256": 256, "P128": 128, "P64": 64}


@pytest.mark.parametrize("path", PATHS)
def test_dispatch_mirror_matches_launched_kernel(sms, path):
    """The kernel torch.profiler sees for one shape per path is the one dispatch() names."""
    from actionmesh_b200 import ops

    m, n = MID_M[path], N_OF[path]
    A = torch.randn(m, 64, device="cuda").bfloat16()
    W = torch.randn(n, 64, device="cuda").bfloat16()
    out = torch.empty(m, n, device="cuda", dtype=torch.bfloat16)
    ops.gemm(A, W, out)     # first launch (module load) outside the trace
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        ops.gemm(A, W, out)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if "gemm" in e.name and "bf16_kernel" in e.name]
    if not names:
        pytest.skip("torch.profiler recorded no kernel launched through the C ABI; the dispatch mirror stands alone")
    assert len(names) == 1, f"expected one GEMM kernel in the trace, saw {names}"
    if path == "P2":
        assert "gemm2_bf16_kernel" in names[0], names[0]
    else:   # demangled "gemm_bf16_kernel<256, 4>" or mangled "gemm_bf16_kernelILi256ELi4E"
        got = re.search(r"gemm_bf16_kernel(?:<|ILi)(\d+)", names[0])
        assert got and int(got.group(1)) == _BN[path], names[0]
