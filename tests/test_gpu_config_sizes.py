"""GPU parity at the sizes BASELINE.json's configs name (VERDICT r1 item 1), against the CPU oracle on the same seeded
inputs, with the element-wise gradient criterion of tests/util.py and the fragile-pixel exemption stated and bounded:

  C3   500k Gaussians x 256x256, 2 of the 8 views: forward AND every gradient (means, opacities, SH per band, cov6)
  C4   2M Gaussians x 512x512, 1 of the 32 views: colour + composited depth
  C5   the PF3plat-shaped cloud, 2 x 256 x 256 pixel-aligned Gaussians at 256x256: forward + gradients
  ortho  the fake-orthographic settings of render_cuda_orthographic
         (/root/reference/src/model/decoder/cuda_splatting.py:154-165: fov 0.1 deg, camera moved back ~10^3 units)

Every test prints the four image numbers (pixels over 1e-4, fragile fraction, worst non-fragile / fragile error) and,
per gradient tensor, the worst element-wise ratio |a-b| / (|b| + rms(b)) for Gaussians that do / do not contribute to a
fragile pixel."""
import numpy as np
import pytest
import torch

from pf3plat_b200.synthetic import make_pixel_aligned_scene, make_scene
from tests.util import check_image_strict, fwd_bwd_vs_oracle, gpu_device as _dev, oracle_view, render_scene as _render

pytestmark = pytest.mark.gpu


def test_c3_forward_and_all_gradients_at_config_size():
    """BASELINE.json configs[2]: 500k Gaussians, 256x256, forward+backward (MSE to a random target); 2 of the 8 views."""
    sc = make_scene(500_000, 2, 256, 256, seed=0, total_views=8)
    fwd_bwd_vs_oracle(sc, 2, max_fragile_frac=0.03, label="C3")


def test_c5_shape_forward_and_gradients():
    """The cloud PF3plat's encoder emits for 2 context views at 256x256 (131 072 pixel-aligned Gaussians), 2 targets."""
    sc = make_pixel_aligned_scene(256, 256, 2, seed=5)
    assert sc.means.shape[0] == 2 * 256 * 256
    # sub-pixel splats on a smooth surface put more pixels next to an alpha = 1/255 contour: 3.3 % fragile (C3: 1.2 %)
    fwd_bwd_vs_oracle(sc, 2, max_fragile_frac=0.05, label="C5-shape")


def test_c4_forward_and_depth_at_config_size():
    """BASELINE.json configs[3]: 2M Gaussians, 512x512; view 5 of the 32, colour and the fused depth channel."""
    dev = _dev()
    sc = make_scene(2_000_000, 1, 512, 512, seed=0, first_view=5, total_views=32)
    (color, depth), _ = _render(sc, dev, with_depth=True)
    orc = oracle_view(sc, 0, with_depth=True)
    check_image_strict(color[0], orc, 0.03, "C4 view 5")
    derr = np.abs(depth[0].cpu().numpy().astype(np.float64) - orc.depth)
    frag = orc.px_fragile
    rel = derr / np.maximum(np.abs(orc.depth), 1.0)
    print(f"[parity] C4 depth: max rel err non-fragile {rel[~frag].max():.3e}, fragile {rel[frag].max() if frag.any() else 0:.3e}")
    assert rel[~frag].max() <= 1e-4 and (not frag.any() or rel[frag].max() <= 5e-2)


def test_fake_orthographic_settings_match_oracle():
    """render_cuda_orthographic (cuda_splatting.py:130-220): fov 0.1 degrees, camera moved back by 0.5*width/tan(fov/2)
    (~1146 units per unit of width) -- the fp32-stressing regime: view-space depths ~10^3, focal length ~1.5e5 px."""
    from oracle.gs_oracle import OracleRender, OracleSettings
    from tests.ref_callsite import orthographic_settings_like_reference, render_orthographic_like_reference
    dev = _dev()
    g = torch.Generator().manual_seed(11)
    P, h, w = 20000, 96, 128
    means = torch.rand(P, 3, generator=g) * torch.tensor([2.0, 1.5, 2.0]) - torch.tensor([1.0, 0.75, 0.0])
    sc = make_scene(P, 1, h, w, seed=11)
    scales = 0.004 * torch.exp(torch.rand(P, 3, generator=g) * 2.5)
    from pf3plat_b200.synthetic import quat_to_rotmat
    R = quat_to_rotmat(sc.rotations)
    cov = R @ torch.diag_embed(scales * scales) @ R.transpose(-1, -2)
    cov = 0.5 * (cov + cov.transpose(-1, -2))
    ext = torch.eye(4)[None]
    width, height = torch.tensor([2.2]), torch.tensor([1.65])
    near, far = torch.tensor([0.0]), torch.tensor([4.0])
    bg = torch.tensor([[0.1, 0.2, 0.3]])
    args = dict(extrinsics=ext, width=width, height=height, near=near, far=far, image_shape=(h, w), background_color=bg,
                gaussian_means=means[None], gaussian_covariances=cov[None], gaussian_sh_coefficients=sc.harmonics[None],
                gaussian_opacities=sc.opacities[None])
    # camera tensors stay on the CPU (so the oracle below sees bit-identical matrices); the operator moves them itself
    img = render_orthographic_like_reference(**{k: (v.to(dev) if k.startswith("gaussian_") else v) for k, v in args.items()})
    st = orthographic_settings_like_reference(ext, width, height, near, far, (h, w), bg, sc.harmonics.shape[-1])[0]
    assert st["tanfovx"] < 1e-3 and abs(st["viewmatrix"][3, 2]) > 1000.0     # really the stressed regime
    row, col = torch.triu_indices(3, 3)
    # Every depth lies near 1.26e3, where fp32 resolves 1.2e-4: ~40 % of the 20 000 depths are EXACT ties and the order is
    # decided by the index.  The kernels' depth keys are bit-identical to the oracle's (same fma chain) and both order
    # ties by index, so the "depths within 4 ulp" fragility flag is switched off here: ties must not hide differences.
    from oracle import gs_oracle
    gs_oracle.set_depth_tie_ulps(0.0)
    try:
        orc = _ortho_oracle(OracleRender, OracleSettings, st, h, w, bg, means, sc, cov, row, col)
    finally:
        gs_oracle.set_depth_tie_ulps(4.0)
    assert len(np.unique(orc.depths[orc.radii > 0])) < 0.9 * (orc.radii > 0).sum()    # ties really are the rule
    assert orc.num_rendered > 0 and (orc.radii > 0).sum() > 0.5 * P
    check_image_strict(img[0], orc, 0.05, "ortho")


def _ortho_oracle(OracleRender, OracleSettings, st, h, w, bg, means, sc, cov, row, col):
    orc = OracleRender(OracleSettings(image_height=h, image_width=w, tanfovx=st["tanfovx"], tanfovy=st["tanfovy"],
                                      bg=bg[0].numpy(), scale_modifier=1.0, viewmatrix=st["viewmatrix"],
                                      projmatrix=st["projmatrix"], sh_degree=st["sh_degree"], campos=st["campos"]),
                       means3D=means.numpy(), opacities=sc.opacities.numpy(),
                       shs=sc.harmonics.permute(0, 2, 1).contiguous().numpy(), cov3D_precomp=cov[:, row, col].numpy())
    return orc
