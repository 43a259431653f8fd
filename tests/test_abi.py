"""CPU-only checks of the drop-in boundary: the C-ABI library loads and exports every symbol include/gms_b200.h
declares; the Python shim mirrors the stock argument checks; nothing in the product imports the oracle."""
import os
import re

import pytest
import torch

from gms_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, "include", "gms_b200.h")).read()
    declared = set(re.findall(r"\b(gms_[a-z_0-9]+)\s*\(", hdr)) - {"gms_alloc_fn"}
    assert declared, "header parse failed"
    assert declared == set(_lib.ABI_SYMBOLS), declared ^ set(_lib.ABI_SYMBOLS)
    for sym in declared:
        assert hasattr(L, sym), f"libgms_b200.so does not export {sym}"
    assert b"sm_100a" in L.gms_version()


def test_header_is_plain_c_and_struct_layouts_match_the_ctypes_mirror(tmp_path):
    """include/gms_b200.h is the contract a C / cgo / JNI binding compiles against: it must be valid C99 on its own, and the
    ctypes structures of gms_b200/_lib.py (what every Python call marshals through) must have the sizes the C compiler gives
    the header's structs, field by field."""
    import ctypes
    import subprocess
    names = {"gms_raster_settings": _lib.RasterSettings, "gms_raster_inputs": _lib.RasterInputs, "gms_raster_outputs": _lib.RasterOutputs,
             "gms_raster_saved": _lib.RasterSaved, "gms_raster_grads": _lib.RasterGrads, "gms_frame_args": _lib.FrameArgs,
             "gms_adam_args": _lib.AdamArgs, "gms_adam_sh_args": _lib.AdamShArgs, "gms_frame_view": _lib.FrameView,
             "gms_debug_views": _lib.DebugViews, "gms_expand_args": _lib.ExpandArgs, "gms_expand_grads": _lib.ExpandGrads,
             "gms_points_args": _lib.PointsArgs, "gms_points_vertices_args": _lib.PointsVerticesArgs, "gms_loss_args": _lib.LossArgs}
    src = tmp_path / "sizes.c"
    body = "".join(f'    printf("{n} %zu\\n", sizeof({n}));\n' for n in names)
    body += "".join(f'    printf("{n}.{f[0]} %zu\\n", offsetof({n}, {f[0]}));\n' for n, cls in names.items() for f in cls._fields_)
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gms_b200.h"\nint main(void) {\n' + body + "    return 0;\n}\n")
    exe = tmp_path / "sizes"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    out = subprocess.check_output([str(exe)], text=True)
    sizes = dict((l.split()[0], int(l.split()[1])) for l in out.strip().split("\n"))
    for n, cls in names.items():
        assert sizes[n] == ctypes.sizeof(cls), (n, sizes[n], ctypes.sizeof(cls))
        for f in cls._fields_:                      # same field names, same offsets (175 fields)
            assert sizes[f"{n}.{f[0]}"] == getattr(cls, f[0]).offset, (n, f[0])


def test_shim_module_name_and_settings_fields():
    import diff_gaussian_rasterization as d
    fields = d.GaussianRasterizationSettings._fields
    assert fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                      "projmatrix", "sh_degree", "campos", "prefiltered", "debug", "antialiasing")
    # 12-field (older API generation) construction still works
    z = torch.zeros(3)
    s = d.GaussianRasterizationSettings(image_height=4, image_width=4, tanfovx=1.0, tanfovy=1.0, bg=z, scale_modifier=1.0,
                                        viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=0, campos=z,
                                        prefiltered=False, debug=False)
    assert s.antialiasing is False


def test_argument_exclusivity_errors_match_stock_messages():
    import diff_gaussian_rasterization as d
    z = torch.zeros(3)
    s = d.GaussianRasterizationSettings(4, 4, 1.0, 1.0, z, 1.0, torch.eye(4), torch.eye(4), 0, z, False, False, False)
    r = d.GaussianRasterizer(raster_settings=s)
    m = torch.zeros(2, 3)
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        r(means3D=m, means2D=m, opacities=torch.ones(2, 1), scales=torch.ones(2, 3), rotations=torch.ones(2, 4))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m, means2D=m, opacities=torch.ones(2, 1), colors_precomp=torch.ones(2, 3))
    with pytest.raises(Exception, match="scale/rotation pair or precomputed 3D covariance"):
        r(means3D=m, means2D=m, opacities=torch.ones(2, 1), colors_precomp=torch.ones(2, 3), scales=torch.ones(2, 3),
          rotations=torch.ones(2, 4), cov3D_precomp=torch.ones(2, 6))


def test_cpu_tensors_fail_loudly_no_fallback():
    import diff_gaussian_rasterization as d
    z = torch.zeros(3)
    s = d.GaussianRasterizationSettings(16, 16, 1.0, 1.0, z, 1.0, torch.eye(4), torch.eye(4), 0, z, False, False, False)
    r = d.GaussianRasterizer(raster_settings=s)
    m = torch.zeros(2, 3)
    with pytest.raises(RuntimeError, match="CUDA tensor"):
        r(means3D=m, means2D=m, opacities=torch.ones(2, 1), colors_precomp=torch.ones(2, 3), scales=torch.ones(2, 3),
          rotations=torch.ones(2, 4))


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "gaussian-mesh-splatting_b200")
    for dp, _, fs in os.walk(pkg):
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), f"{f} imports the oracle"
                assert "gms_oracle" not in txt, f"{f} references the oracle library"


def test_reference_renderer_imports_against_the_shim(golden_dir):
    """Every name the reference's renderer modules import from `diff_gaussian_rasterization` (recorded from the reference by
    tests/golden/make_reference_render_golden.py) resolves in our shim to the product's rasterizer."""
    import numpy as np
    import diff_gaussian_rasterization as d
    import gms_b200.rasterizer as ours
    imports = np.load(os.path.join(golden_dir, "reference_rasterizer_imports.npz"))
    assert set(imports.files) == {"renderer.gaussian_renderer", "renderer.gaussian_animated_renderer"}
    for mod in imports.files:
        names = list(imports[mod])
        assert {"GaussianRasterizationSettings", "GaussianRasterizer"} <= set(names), (mod, names)
        for n in names:
            assert getattr(d, n) is getattr(ours, n), (mod, n)
