"""GPU parity with cameras the way PF3plat renders target views: rotated around the cloud (yaw, pitch, roll; one view
rolled by 90 degrees), tanfovx / tanfovy = 1.3, near in {0.5, 1, 2} (in-kernel view_scale 2, 1, 0.5), a non-zero
background, and Gaussians behind the camera, inside the near cull, just past it, past the guard band and far off-axis
(tests/util.make_posed_scene).  The front-facing scenes of the other GPU tests reach none of these.

Every check prints the four image numbers and the per-gradient worst ratios; the regime assertions make sure the
populations were really reached in the views compared."""
import numpy as np
import pytest
import torch

from pf3plat_b200.synthetic import make_pixel_aligned_scene, make_target
from tests.util import (SH_BANDS, affected_gaussians, camera_space, check_grad, check_image_strict, cov6_of,
                        fwd_bwd_vs_oracle, gpu_device, make_posed_scene, oracle_view, posed_c2w, posed_regimes,
                        view_args, view_scales)

pytestmark = pytest.mark.gpu

N_MIN = 20   # Gaussians per regime and view that must really be in that regime


def _assert_regimes(sc, views, orcs=None):
    vb_scales = view_scales(sc)
    assert len(np.unique(vb_scales)) > 1, vb_scales
    for v in range(views):
        st, _ = view_args(sc, v)
        assert abs(st.tanfovx / st.tanfovy - 1.3) < 0.01 and st.bg.min() > 0
        reg = posed_regimes(sc, v)
        counts = {k: int(reg[k].sum()) for k in ("behind", "near_cull", "x_out", "y_out", "off_axis")}
        print(f"[regimes] view {v}: view_scale {vb_scales[v]}, {counts}")
        assert counts["behind"] >= N_MIN and counts["near_cull"] >= N_MIN and counts["off_axis"] >= 4
        if orcs is not None:
            r = orcs[v]["radii"]
            assert ((reg["x_out"] | reg["y_out"]) & (r > 0)).sum() >= N_MIN
            assert (r[reg["behind"] | reg["near_cull"] | reg["off_axis"]] == 0).all()


def test_posed_forward_depth_radii_and_all_gradients():
    """~40k Gaussians, 4 posed views at 96x128: colour per view, radii (except geom_fragile), the depth channel, and
    dL/d{means, opacities, SH per band, cov6} against the oracle (its gradients taken back through the 1/near rescale)."""
    sc = make_posed_scene(40000, 4, 96, 128, seed=0)
    orcs, grads = fwd_bwd_vs_oracle(sc, 4, max_fragile_frac=0.03, label="posed", with_depth=True, check_radii=True)
    _assert_regimes(sc, 4, orcs)
    gm = grads["means"].cpu().numpy()
    for v in range(4):   # Gaussians clamped by the guard band are seen and get gradients
        reg = posed_regimes(sc, v)
        clamped = (reg["x_out"] | reg["y_out"]) & (orcs[v]["radii"] > 0)
        assert (np.abs(gm[clamped]).sum(axis=1) > 0).sum() >= N_MIN


@pytest.mark.parametrize("mode", ["sh_scalerot", "rgb"])
def test_posed_means2D_and_colour_gradients_per_view(mode):
    """rasterize_batch with a means2D sink: dL/dmeans2D per view, and for per-view colours_precomp (V,P,3) dL/dcolors
    per view; scales / rotations (sh_scalerot) summed over views."""
    from pf3plat_b200.cameras import make_view_batch
    from pf3plat_b200.rasterizer import BatchSettings, rasterize_batch
    from oracle.gs_oracle import OracleRender
    dev = gpu_device()
    V, (h, w) = 3, (64, 96)
    sc = make_posed_scene(8000, V, h, w, seed=3)
    P = sc.means.shape[0]
    d = sc.to(dev)
    vb = make_view_batch(d.extrinsics, d.intrinsics, d.near, d.far)
    bs = BatchSettings(image_height=h, image_width=w, viewmatrix=vb.viewmatrix, projmatrix=vb.projmatrix,
                       campos=vb.campos, bg=d.background, sh_degree=4, tanfov=vb.tanfov, view_scale=vb.scale)
    g = torch.Generator().manual_seed(5)
    colors = torch.rand(V, P, 3, generator=g)
    leaves = {"means3D": d.means[None].clone(), "opacities": d.opacities[None].clone(),
              "means2D": torch.zeros(V, P, 3, device=dev)}
    if mode == "rgb":
        leaves["colors_precomp"] = colors.to(dev)
        leaves["cov3D_precomp"] = torch.as_tensor(cov6_of(sc.covariances), device=dev)[None]
    else:
        leaves["shs"] = d.harmonics.permute(0, 2, 1).contiguous()[None]
        leaves["scales"], leaves["rotations"] = d.scales[None].clone(), d.rotations[None].clone()
    for t in leaves.values():
        t.requires_grad_(True)
    color, radii = rasterize_batch(bs, **leaves)
    target = make_target(V, h, w).to(dev)
    ((color - target) ** 2).mean().backward()
    s = view_scales(sc)
    gsc, grot = np.zeros((P, 3)), np.zeros((P, 4))
    aff_all = np.zeros(P, bool)
    for v in range(V):
        st, kw = view_args(sc, v)
        kw.pop("shs")
        if mode == "rgb":
            kw["colors_precomp"] = colors[v].numpy()
        else:
            kw["shs"] = sc.harmonics.permute(0, 2, 1).contiguous().numpy()
            kw.pop("cov3D_precomp")
            kw["scales"], kw["rotations"] = sc.scales.numpy() * s[v], sc.rotations.numpy()
        orc = OracleRender(st, **kw)
        check_image_strict(color[v], orc, 0.03, f"{mode} view {v}")
        ok = (radii[v].cpu().numpy() == orc.radii) | orc.geom_fragile
        assert ok.all()
        gref = orc.backward((2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32))
        aff = affected_gaussians(orc, orc.px_fragile) | orc.geom_fragile
        aff_all |= aff
        check_grad(f"{mode} view {v} dL/dmeans2D", leaves["means2D"].grad[v], gref["means2D"], aff)
        if mode == "rgb":
            check_grad(f"{mode} view {v} dL/dcolors", leaves["colors_precomp"].grad[v], gref["colors_precomp"], aff)
        else:
            gsc += s[v] * gref["scales"]; grot += gref["rotations"]
    if mode != "rgb":
        check_grad(f"{mode} dL/dscales", leaves["scales"].grad[0], gsc, aff_all)
        check_grad(f"{mode} dL/drotations", leaves["rotations"].grad[0], grot, aff_all)


def test_two_posed_scenes_in_one_call():
    """S = 2 scenes, each with its own posed cameras, in one render_views call: every view against the oracle of its
    own scene, and each scene's dL/dmeans."""
    from pf3plat_b200.render import render_views
    dev = gpu_device()
    V, (h, w) = 3, (64, 80)
    scs = make_posed_scene(10000, V, h, w, seed=7, scenes=2)
    assert not torch.equal(scs[0].extrinsics, scs[1].extrinsics)
    P = min(s.means.shape[0] for s in scs)
    for s in scs:   # same P in both scenes (the operator takes (S, P, ...))
        for name in ("means", "covariances", "harmonics", "opacities", "scales", "rotations"):
            setattr(s, name, getattr(s, name)[:P].contiguous())
    cat = lambda name: torch.cat([getattr(s, name) for s in scs]).to(dev)
    stack = lambda name: torch.stack([getattr(s, name) for s in scs]).to(dev)
    means = stack("means").requires_grad_(True)
    color = render_views(cat("extrinsics"), cat("intrinsics"), cat("near"), cat("far"), (h, w), cat("background"),
                         means, stack("covariances"), stack("harmonics"), stack("opacities"))
    target = make_target(2 * V, h, w).to(dev)
    ((color - target) ** 2).mean().backward()
    for k, sc in enumerate(scs):
        s = view_scales(sc)
        gm, aff = np.zeros((P, 3)), np.zeros(P, bool)
        for v in range(V):
            orc = oracle_view(sc, v)
            check_image_strict(color[k * V + v], orc, 0.03, f"scene {k} view {v}")
            aff |= affected_gaussians(orc, orc.px_fragile) | orc.geom_fragile
            dL = (2 * (orc.color - target[k * V + v].cpu().numpy()) / target.numel()).astype(np.float32)
            gm += s[v] * orc.backward(dL)["means3D"]
        check_grad(f"scene {k} dL/dmeans3D", means.grad[k], gm, aff)


def test_dropin_rasterizer_on_a_posed_view():
    """The drop-in GaussianRasterizer, fed what render_cuda hands it for view 1 (rolled 90 degrees, near 0.5):
    image, radii and every gradient against the oracle."""
    from oracle.gs_oracle import OracleRender
    from pf3plat_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    dev = gpu_device()
    sc = make_posed_scene(6000, 2, 64, 80, seed=9)
    st, kw = view_args(sc, 1)
    orc = OracleRender(st, **kw)
    target = make_target(1, 64, 80)[0].numpy()
    dL = (2 * (orc.color - target) / target.size).astype(np.float32)
    g_ref = orc.backward(dL)
    settings = GaussianRasterizationSettings(
        image_height=64, image_width=80, tanfovx=st.tanfovx, tanfovy=st.tanfovy, bg=torch.tensor(st.bg, device=dev),
        scale_modifier=1.0, viewmatrix=torch.tensor(st.viewmatrix, device=dev),
        projmatrix=torch.tensor(st.projmatrix, device=dev), sh_degree=st.sh_degree,
        campos=torch.tensor(st.campos, device=dev), prefiltered=False, debug=False)
    tk = {k: torch.tensor(np.asarray(a), dtype=torch.float32, device=dev, requires_grad=True) for k, a in kw.items()}
    tk["opacities"] = tk["opacities"].detach().reshape(-1, 1).requires_grad_(True)
    m2d = torch.zeros(sc.means.shape[0], 3, device=dev, requires_grad=True)
    color, radii = GaussianRasterizer(settings)(means2D=m2d, **tk)
    check_image_strict(color, orc, 0.03, "drop-in posed")
    assert ((radii.cpu().numpy() == orc.radii) | orc.geom_fragile).all()
    (color * torch.tensor(dL, device=dev)).sum().backward()
    aff = affected_gaussians(orc, orc.px_fragile) | orc.geom_fragile
    for name, t in tk.items():
        check_grad(f"drop-in posed dL/d{name}", t.grad, g_ref[name], aff, bands=SH_BANDS if name == "shs" else None)
    check_grad("drop-in posed dL/dmeans2D", m2d.grad, g_ref["means2D"], aff)


def test_mark_visible_matches_the_near_cull_on_a_posed_view():
    from pf3plat_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    dev = gpu_device()
    sc = make_posed_scene(6000, 3, 64, 80, seed=11)
    for v in range(3):
        st, kw = view_args(sc, v)
        settings = GaussianRasterizationSettings(
            image_height=64, image_width=80, tanfovx=st.tanfovx, tanfovy=st.tanfovy,
            bg=torch.tensor(st.bg, device=dev), scale_modifier=1.0, viewmatrix=torch.tensor(st.viewmatrix, device=dev),
            projmatrix=torch.tensor(st.projmatrix, device=dev), sh_degree=st.sh_degree,
            campos=torch.tensor(st.campos, device=dev), prefiltered=False, debug=False)
        vis = GaussianRasterizer(settings).markVisible(torch.tensor(kw["means3D"], device=dev)).cpu().numpy()
        z = camera_space(sc, v)[0][:, 2]
        expect = z > 0.2                                  # the oracle's (and upstream's in_frustum) near cull
        orc = oracle_view(sc, v)
        assert not (orc.radii[~expect] > 0).any()
        print(f"[markVisible] view {v}: {int((~vis).sum())} of {len(vis)} culled")
        assert (~expect).sum() >= 2 * N_MIN and np.array_equal(vis, expect)


def _rotate_targets(sc, seed):
    """Target poses yawed and pitched by 5..15 degrees (random signs) about each camera's own centre."""
    rng = np.random.default_rng(seed)
    ext = sc.extrinsics.clone()
    for v in range(ext.shape[0]):
        yaw, pitch = rng.choice([-1, 1], 2) * rng.uniform(5, 15, 2)
        R = torch.tensor(posed_c2w(yaw, pitch, 0.0, dist=0.0)[:3, :3], dtype=ext.dtype)
        ext[v, :3, :3] = ext[v, :3, :3] @ R
    sc.extrinsics = ext
    return sc


def test_pf3plat_shape_from_rotated_target_poses():
    """make_pixel_aligned_scene(128, 128, 3), rendered from target poses rotated 5..15 degrees away from the context
    views: forward, dL/dmeans and dL/dcov (and the rest) against the oracle, fragile fraction <= 5 %."""
    sc = _rotate_targets(make_pixel_aligned_scene(128, 128, 3, seed=2), seed=3)
    fwd_bwd_vs_oracle(sc, 3, max_fragile_frac=0.05, label="pixel-aligned rotated")


def test_binning_paths_agree_bit_for_bit_on_posed_views():
    """Oblique views give tiles whose depth range spans the whole cloud: the exact, trial, stratified, NO_STRATA,
    SEPARATE_EMIT and FORCE_RADIX binning paths must still give bit-identical images."""
    from pf3plat_b200._capi import (GS_TUNE_FORCE_RADIX_BINNING, GS_TUNE_NO_SPECULATION, GS_TUNE_NO_STRATA,
                                    GS_TUNE_SEPARATE_EMIT)
    from tests.test_gpu_parity import _render_with_tuning
    dev = gpu_device()
    sc = make_posed_scene(30000, 3, 64, 96, seed=17)
    exact, st_exact = _render_with_tuning(sc, dev, GS_TUNE_NO_SPECULATION)
    first, st_first = _render_with_tuning(sc, dev, 0)
    spec, st_spec = _render_with_tuning(sc, dev, 0)
    spec2, st_spec2 = _render_with_tuning(sc, dev, GS_TUNE_SEPARATE_EMIT)
    _render_with_tuning(sc, dev, GS_TUNE_NO_STRATA | GS_TUNE_NO_SPECULATION)
    whole, st_whole = _render_with_tuning(sc, dev, GS_TUNE_NO_STRATA)
    slow, st_slow = _render_with_tuning(sc, dev, GS_TUNE_FORCE_RADIX_BINNING)
    print("[binning] speculative states exact/first/spec/separate/whole/radix:",
          [s["speculative"] for s in (st_exact, st_first, st_spec, st_spec2, st_whole, st_slow)])
    assert st_exact["speculative"] == 0 and st_slow["speculative"] == 0 and st_spec["speculative"] >= 1
    assert st_exact["num_rendered"] == st_spec["num_rendered"] == st_slow["num_rendered"]
    for name, img in (("first", first), ("spec", spec), ("separate_emit", spec2), ("whole", whole), ("radix", slow)):
        assert torch.equal(exact, img), name
    check_image_strict(exact[0], oracle_view(sc, 0), 0.03, "binning posed view 0")
