"""The C-ABI library loads and exports every symbol include/ast.h declares (no compute: no GPU needed)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "ast.h")).read()
    return sorted(set(re.findall(r"\b(ast_[a-z0-9_]+)\s*\(", text)))


def test_header_symbols_exported():
    from artist_style_transfer_b200 import _lib
    lib = _lib.load()
    names = _declared()
    assert len(names) >= 18
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/ast.h but not exported by libast_b200.so"
    assert sorted(_lib.EXPORTS) == names, "ctypes binding and header disagree"
    assert lib.ast_abi_version() == 7
    assert lib.ast_instnorm_workspace_bytes(4, 128) > 0
    assert lib.ast_launch_count() >= 0


def test_argument_errors_are_loud():
    from artist_style_transfer_b200 import _lib
    lib = _lib.load()
    rc = lib.ast_pack_weights(None, None, 1, 1, 1, 1, 1, None, 0, None)
    assert rc < 0 and b"null" in lib.ast_last_error()


def test_instnorm_layouts_without_a_kernel_are_errors():
    """InstanceNorm apply / backward run only on the staged kernels: mixed dtypes and a pixel stride other than C are
    argument errors, reported before any CUDA call (the dummy pointers are never dereferenced)."""
    from artist_style_transfer_b200 import _lib
    lib = _lib.load()
    n, h, w, c, pad = 2, 8, 8, 64, 1
    p = ctypes.c_void_p(1 << 20)

    def img(dtype, hh=h, ww=w, sw=c):
        return _lib.Image(1 << 20, dtype, n, hh, ww, c, hh * ww * sw, ww * sw, sw, 1)
    f32, bf16 = _lib.AST_F32, _lib.AST_BF16
    for x, out, what in ((img(f32), img(bf16, h + 2, w + 2), b"dtype"),
                         (img(bf16, sw=2 * c), img(bf16, h + 2, w + 2, sw=2 * c), b"dense")):
        rc = lib.ast_instnorm_apply(ctypes.byref(x), p, p, p, p, None, ctypes.byref(out), pad, 1, None)
        assert rc < 0 and what in lib.ast_last_error(), lib.ast_last_error()
        dx = img(out.dtype, sw=2 * c if what == b"dense" else c)
        rc = lib.ast_instnorm_bwd(ctypes.byref(x), p, p, p, p, ctypes.byref(out), pad, None, 1, p, p, p, ctypes.byref(dx),
                                  None, None)
        assert rc < 0 and what in lib.ast_last_error(), lib.ast_last_error()


def test_no_cpu_fallback():
    import torch
    import artist_style_transfer_b200 as ast
    with pytest.raises(RuntimeError, match="CUDA"):
        ast.gram(torch.zeros(1, 4, 2, 2))
    net = ast.StyleTransfer(device="cpu")
    with pytest.raises(RuntimeError, match="CUDA"):
        net(torch.zeros(1, 3, 8, 8))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "artist_style_transfer_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), f"{f} imports the oracle"
                assert "/root/reference" not in src or f.endswith(".py"), f


def test_ctypes_structs_match_the_header_layout(tmp_path):
    """sizeof / offsetof of ast_image and ast_gather_geom as gcc sees include/ast.h == the ctypes mirror in _lib.py
    (a silent mismatch would shift every field after it, e.g. the `stats` / `pooled` pointers)."""
    import shutil
    import subprocess
    from artist_style_transfer_b200 import _lib
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no C compiler")
    src = tmp_path / "layout.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "ast.h"\n'
        'int main(void) {\n'
        '  printf("%zu %zu %zu %zu\\n", sizeof(ast_image), offsetof(ast_image, sn), offsetof(ast_image, c), offsetof(ast_image, sc));\n'
        '  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(ast_gather_geom), offsetof(ast_gather_geom, dy), offsetof(ast_gather_geom, dx),\n'
        '         offsetof(ast_gather_geom, w_img_stride), offsetof(ast_gather_geom, stats), offsetof(ast_gather_geom, pooled));\n'
        '  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(ast_param_desc), offsetof(ast_param_desc, dim), offsetof(ast_param_desc, g_off),\n'
        '         offsetof(ast_param_desc, g_tap), offsetof(ast_param_desc, pack), sizeof(ast_pack_map));\n'
        '  printf("%zu %zu %zu %zu\\n", sizeof(ast_adam_state), offsetof(ast_adam_state, step), sizeof(ast_reduce_desc), offsetof(ast_reduce_desc, rows));\n'
        '  printf("%zu %zu %zu %zu %zu %zu\\n", sizeof(ast_stacked_geom), offsetof(ast_stacked_geom, oy), offsetof(ast_stacked_geom, nvt),\n'
        '         offsetof(ast_stacked_geom, dy), offsetof(ast_stacked_geom, stats), offsetof(ast_pack_map, rep));\n'
        '  return 0;\n}\n')
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    got = [int(v) for v in out]
    img, geom, pd, ad, rd = _lib.Image, _lib.GatherGeom, _lib.ParamDesc, _lib.AdamState, _lib.ReduceDesc
    sg = _lib.StackedGeom
    want = [ctypes.sizeof(img), img.sn.offset, img.c.offset, img.sc.offset,
            ctypes.sizeof(geom), geom.dy.offset, geom.dx.offset, geom.w_img_stride.offset, geom.stats.offset,
            geom.pooled.offset,
            ctypes.sizeof(pd), pd.dim.offset, pd.g_off.offset, pd.g_tap.offset, pd.pack.offset, ctypes.sizeof(_lib.PackMap),
            ctypes.sizeof(ad), ad.step.offset, ctypes.sizeof(rd), rd.rows.offset,
            ctypes.sizeof(sg), sg.oy.offset, sg.nvt.offset, sg.dy.offset, sg.stats.offset, _lib.PackMap.rep.offset]
    assert got == want, (got, want)
