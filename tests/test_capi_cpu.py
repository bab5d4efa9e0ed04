"""CPU-side checks of the drop-in boundary: the C-ABI library loads without a GPU and exports every symbol
include/gsplat_b200.h declares; the ctypes mirrors match the C struct layouts; the Python operator surface has
the reference's names, fields and error behaviour.  No compute calls (no GPU here)."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "gsplat_b200.h")


@pytest.fixture(scope="module")
def capi():
    import __graft_entry__ as ge
    ge.build()
    from pf3plat_b200 import _capi
    return _capi


def _declared_functions():
    src = open(HEADER).read()
    return re.findall(r"GS_API\s+[\w\s\*]+?\b(gs_\w+)\s*\(", src)


def test_library_loads_and_exports_every_declared_symbol(capi):
    L = capi.lib()
    declared = _declared_functions()
    assert len(declared) >= 12
    for name in declared:
        assert hasattr(L, name), f"{name} declared in include/gsplat_b200.h but not exported"
        assert name in capi.SYMBOLS, f"{name} has no ctypes prototype"
    assert set(capi.SYMBOLS) == set(declared)
    assert L.gs_abi_version() == capi.ABI_VERSION


def test_ctypes_struct_layouts_match_the_header(capi, tmp_path):
    names = ["GsConfig", "GsInputs", "GsOutputs", "GsOutGrads", "GsInGrads", "GsStats", "GsAdapterConfig",
             "GsAdapterInputs", "GsAdapterOutputs", "GsAdapterOutGrads", "GsAdapterInGrads"]
    prog = tmp_path / "sizes.c"
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "gsplat_b200.h"\nint main(void){'
                    + "".join(f'printf("%zu\\n", sizeof({n}));' for n in names)
                    + 'printf("%zu\\n", offsetof(GsConfig, viewmatrix));printf("%zu\\n", offsetof(GsConfig, tanfovx));'
                    + 'printf("%zu\\n", offsetof(GsAdapterConfig, c2w));printf("%zu\\n", offsetof(GsAdapterConfig, eps));'
                    + "return 0;}")
    exe = tmp_path / "sizes"
    subprocess.run(["/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc", "-I", os.path.join(ROOT, "include"),
                    str(prog), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    for n, sz in zip(names, out):
        assert ctypes.sizeof(getattr(capi, n)) == int(sz), n
    assert capi.GsConfig.viewmatrix.offset == int(out[len(names)])
    assert capi.GsConfig.tanfovx.offset == int(out[len(names) + 1])
    assert capi.GsAdapterConfig.c2w.offset == int(out[len(names) + 2])
    assert capi.GsAdapterConfig.eps.offset == int(out[len(names) + 3])


def test_null_arguments_are_rejected_without_a_device(capi):
    L = capi.lib()
    assert L.gs_forward(None, None, None, None, None, None) == -1
    assert b"null" in L.gs_last_error()
    assert L.gs_backward(None, None, None, None, None, None, None) == -1
    assert L.gs_get_stats(None, None) == -1
    L.gs_saved_free(None, None, None)      # no-op
    L.gs_context_destroy(None)             # no-op
    # the rows next to the rasterizer validate their arguments before touching the device too
    assert L.gs_adapter_forward(None, None, None, None) == -1
    assert L.gs_adapter_backward(None, None, None, None, None) == -1
    assert L.gs_ssim(None, None, 1, 3, 32, 32, None, None, None) == -1
    assert L.gs_psnr(None, None, 1, 10, None, None, None) == -1
    assert L.gs_view_batch(1, 1, None, None, None, None, None, None, None, None, None, None) == -1
    assert L.gs_view_batch(0, 1, None, None, None, None, None, None, None, None, None, None) == 0   # nothing to do
    assert L.gs_ssim_scratch_floats(2, 3, 256, 256) == 2 * 2 * 3 * 64 and L.gs_ssim_scratch_floats(1, 3, 10, 64) == 0
    bad = capi.GsAdapterConfig(V=1, R=1, d_sh=5)
    assert L.gs_adapter_forward(ctypes.byref(bad), ctypes.byref(capi.GsAdapterInputs()), ctypes.byref(capi.GsAdapterOutputs()),
                                None) == -1 and b"d_sh" in L.gs_last_error()


def test_operator_surface_matches_the_reference_call_site():
    import diff_gaussian_rasterization as dgr
    from pf3plat_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    assert dgr.GaussianRasterizer is GaussianRasterizer
    # the 12 fields, keyword-constructible exactly as in cuda_splatting.py:99-112
    s = dgr.GaussianRasterizationSettings(
        image_height=8, image_width=8, tanfovx=0.5, tanfovy=0.5, bg=torch.zeros(3), scale_modifier=1.0,
        viewmatrix=torch.eye(4), projmatrix=torch.eye(4), sh_degree=4, campos=torch.zeros(3), prefiltered=False,
        debug=False)
    assert s._fields == ("image_height", "image_width", "tanfovx", "tanfovy", "bg", "scale_modifier", "viewmatrix",
                         "projmatrix", "sh_degree", "campos", "prefiltered", "debug")
    r = dgr.GaussianRasterizer(s)
    assert isinstance(r, torch.nn.Module) and hasattr(r, "markVisible")
    P = 4
    kw = dict(means3D=torch.zeros(P, 3), means2D=torch.zeros(P, 3), opacities=torch.ones(P, 1))
    with pytest.raises(Exception, match="excatly one of either SHs or precomputed colors"):
        r(**kw, cov3D_precomp=torch.zeros(P, 6))
    with pytest.raises(Exception, match="exactly one of either scale/rotation pair or precomputed 3D covariance"):
        r(**kw, shs=torch.zeros(P, 25, 3))
    # CPU tensors: the product path refuses loudly instead of falling back
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        r(**kw, shs=torch.zeros(P, 25, 3), cov3D_precomp=torch.zeros(P, 6))


def test_product_code_never_touches_the_oracle():
    bad = []
    for pkg in ("pf3plat_b200", "diff_gaussian_rasterization"):
        for dp, _, fs in os.walk(os.path.join(ROOT, pkg)):
            for f in fs:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".sh")):
                    txt = open(os.path.join(dp, f)).read()
                    if re.search(r"(from|import)\s+oracle|oracle/gs_oracle|libgs_oracle", txt) and "oracle/gs_oracle.c" not in txt:
                        bad.append(os.path.join(dp, f))
                    elif re.search(r"^\s*(from|import)\s+oracle", txt, re.M):
                        bad.append(os.path.join(dp, f))
    assert not bad, bad


OPERATOR_CALLS = os.path.join(ROOT, "tests", "golden", "operator_calls.npz")


def _recorded_operator_calls():
    """(settings kwargs, call kwargs) of every operator call in tests/golden/operator_calls.npz, with the Python types
    and requires_grad flags the reference passed."""
    import json
    z = np.load(OPERATOR_CALLS)
    calls = {}
    for key, kind in json.loads(str(z["kinds"])).items():
        i, part, name = key.split(".")
        if kind == "none":
            v = None
        elif kind.startswith("tensor"):
            v = torch.from_numpy(z[key]).requires_grad_(kind == "tensor_grad")
        else:
            v = {"int": int, "float": float, "bool": bool}[kind](z[key])
        calls.setdefault(int(i[1:]), ({}, {}))[part == "call"][name] = v
    return [calls[i] for i in sorted(calls)]


def test_reference_render_glue_imports_and_reaches_our_operator_unmodified():
    """Replays, with CPU tensors, the operator calls the reference's cuda_splatting.py made through the
    `diff_gaussian_rasterization` names (tests/golden/operator_calls.npz, recorded by make_camera_golden.py from
    render_cuda, render_depth_cuda and render_cuda_orthographic): the settings are built with the reference's
    keywords and Python types, the rasterizer is called with its keywords, and every call arrives at our operator,
    which refuses CPU tensors loudly.  (The same call pattern is exercised on the GPU by tests/test_gpu_dropin.py
    through a line-by-line restatement of the reference's glue.)"""
    import diff_gaussian_rasterization as dgr
    calls = _recorded_operator_calls()
    assert len(calls) == 5
    # render_cuda_orthographic hands 0-dim tensors as tanfovx / tanfovy, the other call sites Python floats
    assert isinstance(calls[-1][0]["tanfovx"], torch.Tensor) and isinstance(calls[0][0]["tanfovx"], float)
    for settings, call in calls:
        rasterizer = dgr.GaussianRasterizer(dgr.GaussianRasterizationSettings(**settings))
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            rasterizer(**call)
