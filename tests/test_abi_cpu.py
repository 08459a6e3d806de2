"""C-ABI checks that need no GPU: the library loads, exports every symbol include/actionmesh_b200.h declares, and
argument validation fails loudly with an error code + message (no compute calls)."""
import ctypes as C
import os
import re

import pytest

from conftest import ROOT


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "actionmesh_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(amb_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_expected_entry_points():
    names = _declared_functions()
    for n in ("amb_gemm_bf16", "amb_flash_attn_fwd", "amb_cfg_euler_step", "amb_layernorm", "amb_last_error"):
        assert n in names


def test_library_exports_every_declared_symbol(amb_lib):
    for name in _declared_functions():
        assert hasattr(amb_lib, name), f"{name} declared in the header but not exported"


def test_binding_matches_header(amb_lib):
    from actionmesh_b200 import _lib

    assert sorted(_lib.EXPORTS) == _declared_functions()
    text = open(os.path.join(ROOT, "include", "actionmesh_b200.h")).read()
    ver = int(re.search(r"#define AMB_ABI_VERSION (\d+)", text).group(1))
    assert amb_lib.amb_abi_version() == ver == _lib.ABI_VERSION


def test_struct_layouts_match_header(amb_lib):
    """ctypes struct sizes equal the C structs' (computed from the header field order with natural alignment)."""
    from actionmesh_b200 import _lib

    text = open(os.path.join(ROOT, "include", "actionmesh_b200.h")).read()

    def csize(struct_name):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct_name, struct_name), text, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        off = 0
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            m = re.match(r"(const\s+)?(void|float|int64_t|int32_t)\s*(\*)?\s*(.*)", decl)
            assert m, decl
            base, ptr, names = m.group(2), m.group(3), m.group(4)
            for nm in names.split(","):
                is_ptr = bool(ptr) or nm.strip().startswith("*")
                sz = 8 if (is_ptr or base == "int64_t") else 4
                off = (off + sz - 1) // sz * sz + sz
        return (off + 7) // 8 * 8

    assert C.sizeof(_lib.GemmArgs) == csize("amb_gemm_args")
    assert C.sizeof(_lib.AttnArgs) == csize("amb_attn_args")


def test_argument_validation_fails_loudly(amb_lib):
    from actionmesh_b200 import _lib

    g = _lib.GemmArgs()
    rc = amb_lib.amb_gemm_bf16(C.byref(g), None)
    assert rc < 0 and b"null pointer" in amb_lib.amb_last_error()
    g.a, g.w, g.c = 16, 16, 16  # fake non-null pointers: validation must stop before any launch
    g.m, g.n, g.k = 128, 100, 64
    g.lda = g.ldw = g.ldc = 64
    rc = amb_lib.amb_gemm_bf16(C.byref(g), None)
    assert rc < 0 and b"multiple of 64" in amb_lib.amb_last_error()
    # the epilogue's 16-byte loads and stores need 16-byte aligned bases: a bf16 output view at a column offset of 4, or
    # a misaligned bias / residual / norm / rope pointer, is refused before any tensor map is built
    g.n = 128
    for field, bad in (("c", 16 + 8), ("c2", 16 + 4), ("residual", 16 + 2), ("bias", 16 + 4), ("col_scale", 16 + 8)):
        setattr(g, field, bad)
        rc = amb_lib.amb_gemm_bf16(C.byref(g), None)
        assert rc < 0 and b"16-byte aligned" in amb_lib.amb_last_error(), field
        setattr(g, field, 16 if field == "c" else None)
    g.norm_cols, g.norm_seg, g.norm_w0 = 128, 128, 16
    for field in ("norm_w0", "norm_w1", "rope_cos", "rope_sin"):
        setattr(g, field, 16 + 4)
        rc = amb_lib.amb_gemm_bf16(C.byref(g), None)
        assert rc < 0 and b"16-byte aligned" in amb_lib.amb_last_error(), field
        setattr(g, field, 16 if field == "norm_w0" else None)
    g.norm_cols = g.norm_seg = 0
    g.norm_w0 = None
    a = _lib.AttnArgs()
    a.q = a.k = a.v = a.o = 16
    a.batch = a.heads = 1
    a.sq = a.sk = 64
    a.head_dim = 96
    rc = amb_lib.amb_flash_attn_fwd(C.byref(a), None)
    assert rc < 0 and b"head_dim" in amb_lib.amb_last_error()
    rc = amb_lib.amb_layernorm(None, 0, 0, None, None, None, 0, 0, 1, 2048, 1e-5, None)
    assert rc < 0


def test_product_path_has_no_cpu_fallback():
    """Ops refuse CPU tensors, and nothing under actionmesh_b200/ imports the oracle."""
    import torch

    from actionmesh_b200 import AmbError, ops

    with pytest.raises(AmbError):
        ops.layernorm(torch.zeros(4, 2048, dtype=torch.bfloat16), torch.ones(2048), torch.zeros(2048), 1e-5)
    pkg = os.path.join(ROOT, "actionmesh_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            src = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in src.replace("# oracle", ""), f"{fn} references the oracle"


def test_missing_library_raises(monkeypatch, tmp_path):
    from actionmesh_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(_lib.AmbError):
        _lib.load_library()


def test_argument_validation_of_widened_entry_points(amb_lib):
    """Stage-II helpers and the preprocessing kernels validate their geometry before any launch (fake non-null pointers)."""
    P = 16
    err = lambda: amb_lib.amb_last_error().decode()
    assert amb_lib.amb_split3_bf16(None, 0, 1, 128, 128, 0, None, 0, None) < 0 and "null pointer" in err()
    assert amb_lib.amb_split3_bf16(P, 128, 1, 128, 96, 0, P, 384, None) < 0 and "bad geometry" in err()     # cols % seg != 0
    assert amb_lib.amb_split3_bf16(P, 128, 1, 128, 128, 0, P, 256, None) < 0 and "bad geometry" in err()    # ld_dst < 3*cols
    assert amb_lib.amb_softmax_split3(P, 128, 1, 130, 128, 1.0, P, 384, None) < 0 and "bad geometry" in err()  # n > n_pad
    assert amb_lib.amb_softmax_split3(P, 64, 1, 100, 128, 1.0, P, 384, None) < 0                               # ld_s < n_pad
    assert amb_lib.amb_alpha_rows(0.0, 1.0, 511, P, 1024, 1, None) < 0 and "alpha_rows" in err()               # odd size
    assert amb_lib.amb_point_embedding(P, 4, 6, 3, 8, 0, P, 32, None) < 0 and "bad geometry" in err()          # kpad too small
    assert amb_lib.amb_point_embedding(P, 4, 5, 3, 8, 0, P, 64, None) < 0                                      # in_dim != 3 + extra
    assert amb_lib.amb_displacement_out(P, 2, 4, 3, P, None) < 0                                               # ld < out_dim
    assert amb_lib.amb_resize_h_u8(P, 1, 64, 64, 2, 0, 64, P, P, 9, 32, P, None) < 0 and "bad geometry" in err()  # 2 channels
    assert amb_lib.amb_resize_h_u8(P, 1, 64, 64, 3, 60, 8, P, P, 9, 32, P, None) < 0 and "outside the image" in err()
    m = (C.c_float * 3)(0, 0, 0)
    assert amb_lib.amb_resize_v_normalize(P, 1, 0, 0, 32, P, P, 9, 32, P, m, m, P, None, None) < 0 and "bad geometry" in err()
    assert amb_lib.amb_resize_v_normalize(P, 1, 8, 0, 32, P, P, 9, 32, None, m, m, P, None, None) < 0 and "null pointer" in err()
    # zero-size work is a successful no-op without a launch
    assert amb_lib.amb_split3_bf16(P, 128, 0, 128, 128, 0, P, 384, None) == 0
    assert amb_lib.amb_resize_h_u8(P, 0, 64, 64, 3, 0, 64, P, P, 9, 32, P, None) == 0
