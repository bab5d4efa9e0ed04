"""Pins the camera glue (pf3plat_b200/cameras.py: the tensor path here, the gs_view_batch kernel in
tests/test_gpu_dropin.py) to the REFERENCE's own render_cuda: tests/golden/camera_glue.npz holds the
GaussianRasterizationSettings that /root/reference/src/model/decoder/cuda_splatting.py:64-112 handed to a recording
rasterizer stub, view by view (tests/golden/make_camera_golden.py)."""
import os

import numpy as np
import pytest
import torch

from pf3plat_b200.cameras import make_view_batch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "camera_glue.npz")


def check_against_golden(vb, z, tag, tol):
    for name, got in (("viewmatrix", vb.viewmatrix), ("projmatrix", vb.projmatrix), ("campos", vb.campos),
                      ("tanfov", vb.tanfov)):
        want = z[f"{tag}_{name}"].astype(np.float64)
        got = got.detach().cpu().double().numpy()
        assert got.shape == want.shape, name
        assert np.abs(got - want).max() <= tol * max(1.0, np.abs(want).max()), (tag, name, np.abs(got - want).max())
    # the 1/near rescale the reference applies to the Gaussians (cuda_splatting.py:64-71) is what view_scale stands for
    s = vb.scale.detach().cpu().double().numpy()
    np.testing.assert_allclose(z["means"] * s[:, None, None], z[f"{tag}_means"], rtol=1e-6, atol=1e-7)
    c = z["covariances"] * (s ** 2)[:, None, None, None]
    cov6 = np.stack([c[..., 0, 0], c[..., 0, 1], c[..., 0, 2], c[..., 1, 1], c[..., 1, 2], c[..., 2, 2]], -1)
    np.testing.assert_allclose(cov6, z[f"{tag}_cov6"], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("tag,scale_invariant", [("si", True), ("raw", False)])
def test_tensor_path_matches_what_the_reference_hands_its_rasterizer(tag, scale_invariant):
    z = np.load(GOLDEN)
    t = lambda k: torch.from_numpy(z[k])
    vb = make_view_batch(t("extrinsics"), t("intrinsics"), t("near"), t("far"), scale_invariant)
    check_against_golden(vb, z, tag, 2e-6)


def test_fixture_is_what_the_reference_produces_today():
    """The recorded half of the fixture is the reference's fixed render_cuda / render_depth_cuda /
    render_cuda_orthographic / DecoderSplattingCUDA run on the inputs make_camera_golden.py generates; the fixture stays
    what the reference produces as long as the script still generates the stored inputs (to fp32 rounding)."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_camera_golden as mk
    z = np.load(GOLDEN)
    names = ("extrinsics", "intrinsics", "near", "far", "means", "covariances", "sh", "opacities")
    same = lambda got, key: np.testing.assert_allclose(got.numpy(), z[key], rtol=1e-6, atol=1e-7, err_msg=key)
    for name, t in zip(names, mk.glue_inputs()):
        same(t, name)
    for name, t in mk.ortho_inputs().items():
        same(t, "ortho_in_" + name)
    for name, t in mk.decoder_inputs().items():
        same(t, "dec_in_" + name)


def test_callsite_restatement_hands_the_op_what_the_reference_does(monkeypatch):
    """tests/ref_callsite.py (the comparator of the GPU drop-in tests, needed because /root/reference is absent on the GPU
    box) is run against the same recording rasterizer stub as the reference was: every argument it hands the operator --
    settings, rescaled means / covariances, relaid SH, fake depth colours of all four modes, background, flags, the
    zero means2D leaf -- must equal what the reference's render_cuda / render_depth_cuda handed over."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_camera_golden as mk
    from tests import ref_callsite
    monkeypatch.setattr(ref_callsite, "GaussianRasterizer", mk._Recorder)
    monkeypatch.setattr(ref_callsite, "GaussianRasterizationSettings", mk._Settings)
    z = np.load(GOLDEN)
    t = lambda k: torch.from_numpy(z[k])
    ext, intr, near, far, means, cov, sh, opac = (t(k) for k in ("extrinsics", "intrinsics", "near", "far", "means",
                                                                  "covariances", "sh", "opacities"))
    B = ext.shape[0]

    def recorded(keys):
        out = {k: torch.stack([r[k] for r in mk.RECORDED]).numpy() for k in keys}
        mk.RECORDED.clear()
        return out

    same = lambda a, b, name: np.testing.assert_allclose(a, b, rtol=2e-6, atol=2e-6, err_msg=name)
    mk.RECORDED.clear()
    for tag, si in (("si", True), ("raw", False)):
        ref_callsite.render_like_reference(ext, intr, near, far, (16, 24), torch.zeros(B, 3), means, cov, sh, opac,
                                           scale_invariant=si)
        got = recorded(("viewmatrix", "projmatrix", "campos", "tanfov", "means", "cov6"))
        for k, v in got.items():
            same(v, z[f"{tag}_{k}"], f"{tag}_{k}")
    bg = torch.rand(B, 3, generator=torch.Generator().manual_seed(14))
    ref_callsite.render_like_reference(ext, intr, near, far, (16, 24), bg, means, cov, sh, opac)
    for k, v in recorded(("shs", "bg", "opacities", "ints", "scale_modifier", "means2D_is_zero_leaf")).items():
        same(v, z[f"color_{k}"], f"color_{k}")
    for mode in ("depth", "disparity", "relative_disparity", "log"):
        ref_callsite.render_depth_like_reference(ext, intr, near, far, (16, 24), means.abs() + 0.5, cov, opac, mode=mode)
        for k, v in recorded(("colors", "bg", "opacities", "ints", "scale_modifier", "means2D_is_zero_leaf")).items():
            same(v, z[f"depth_{mode}_{k}"], f"depth_{mode}_{k}")


def test_orthographic_restatement_hands_the_op_what_the_reference_does(monkeypatch):
    """ref_callsite.render_orthographic_like_reference against the recorded operator call of the reference's own
    render_cuda_orthographic (cuda_splatting.py:130-220): the moved-back camera, the 0.1-degree field of view, the
    projection built from it."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_camera_golden as mk
    from tests import ref_callsite
    monkeypatch.setattr(ref_callsite, "GaussianRasterizer", mk._Recorder)
    monkeypatch.setattr(ref_callsite, "GaussianRasterizationSettings", mk._Settings)
    z = np.load(GOLDEN)
    t = lambda k: torch.from_numpy(z[k])
    oi = {k: t("ortho_in_" + k) for k in ("extrinsics", "width", "height", "near", "far", "bg")}
    mk.RECORDED.clear()
    ref_callsite.render_orthographic_like_reference(oi["extrinsics"], oi["width"], oi["height"], oi["near"], oi["far"],
                                                    (16, 24), oi["bg"], t("means")[:1], t("covariances")[:1], t("sh")[:1],
                                                    t("opacities")[:1])
    assert len(mk.RECORDED) == 1
    for k in ("viewmatrix", "projmatrix", "campos", "tanfov", "means", "cov6", "shs", "bg", "opacities", "ints",
              "scale_modifier", "means2D_is_zero_leaf"):
        got = torch.stack([r[k] for r in mk.RECORDED]).numpy()
        want = z[f"ortho_{k}"]
        np.testing.assert_allclose(got, want, rtol=2e-6, atol=2e-6 * max(1.0, float(np.abs(want).max())), err_msg=k)
    assert abs(z["ortho_viewmatrix"][0, 3, 2]) > 1000 and z["ortho_tanfov"][0, 0] < 1e-3   # the stressed regime
    mk.RECORDED.clear()
    # the settings helper the GPU test feeds the oracle with is the same computation
    st = ref_callsite.orthographic_settings_like_reference(oi["extrinsics"], oi["width"], oi["height"], oi["near"],
                                                           oi["far"], (16, 24), oi["bg"], 25)[0]
    np.testing.assert_allclose(st["viewmatrix"], z["ortho_viewmatrix"][0], rtol=2e-6, atol=2e-3)
    np.testing.assert_allclose(st["projmatrix"], z["ortho_projmatrix"][0], rtol=2e-6, atol=2e-3)
    np.testing.assert_allclose([st["tanfovx"], st["tanfovy"]], z["ortho_tanfov"][0], rtol=1e-6)


def test_decoder_restatement_hands_the_op_what_the_reference_decoder_does(monkeypatch):
    """ref_callsite.decoder_like_reference against the recorded operator calls of the reference's own
    DecoderSplattingCUDA.forward (2 scenes x 3 views, colour pass then depth pass): same views in the same order, the
    same repeated Gaussians, background and fake depth colours."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden"))
    import make_camera_golden as mk
    from tests import ref_callsite
    monkeypatch.setattr(ref_callsite, "GaussianRasterizer", mk._Recorder)
    monkeypatch.setattr(ref_callsite, "GaussianRasterizationSettings", mk._Settings)
    z = np.load(GOLDEN)
    t = lambda k: torch.from_numpy(z["dec_in_" + k])
    mk.RECORDED.clear()
    color, depth = ref_callsite.decoder_like_reference(t("means"), t("covariances"), t("sh"), t("opacities"), t("extrinsics"),
                                                       t("intrinsics"), t("near"), t("far"), (16, 24),
                                                       torch.tensor([0.1, 0.2, 0.3]), depth_mode="depth")
    assert color.shape == (2, 3, 3, 16, 24) and depth.shape == (2, 3, 16, 24) and len(mk.RECORDED) == 12
    for half, sl in (("color", slice(0, 6)), ("depth", slice(6, 12))):
        for k in mk.DECODER_KEYS:
            got = torch.stack([r[k] for r in mk.RECORDED[sl]]).numpy()
            np.testing.assert_allclose(got, z[f"dec_{half}_{k}"], rtol=2e-6, atol=2e-6, err_msg=f"{half}_{k}")
    mk.RECORDED.clear()
