"""GPU parity tests: the sm_100a kernels, called through the C ABI, against the CPU oracle on the same seeded
inputs.  Tolerances are BASELINE.json's: 1e-4 abs RGB, 1e-3 rel gradient -- the gradient criterion is ELEMENT-WISE,
|a-b| <= 1e-3 |b| + 1e-3 rms(b), per tensor and per SH band (tests/util.py).
Pixels the oracle flags as FRAGILE (a discontinuous decision -- alpha<1/255, T<1e-4, ceil/int of the footprint,
near-equal depths -- lies within 1e-4 relative of its threshold, so two correct fp32 implementations may take
either branch) are held to 5e-3 (one flipped 1/255-alpha decision is worth <= 3.9e-3) and must be a small fraction of
the image; Gaussians that contribute to such a pixel carry a 2e-2 gradient bound.  Every check prints its numbers."""
import numpy as np
import pytest
import torch

from pf3plat_b200.synthetic import make_scene, make_target
from tests.util import (FRAGILE_RGB_TOL, RGB_TOL, SH_BANDS, affected_gaussians, check_grad, image_report, oracle_view,
                        view_args)

pytestmark = pytest.mark.gpu


def _dev():
    assert torch.cuda.is_available(), "GPU test needs CUDA"
    return torch.device("cuda:0")


def check_image(gpu_color, orc, max_fragile_frac=0.03):
    rep = image_report(gpu_color, orc)
    print(f"[parity] {rep}")
    assert rep["fragile_frac"] <= max_fragile_frac, rep
    assert rep["max_err_nonfragile"] <= RGB_TOL, rep
    assert rep["max_err_fragile"] <= FRAGILE_RGB_TOL, rep
    return rep


def affected_of(orc):
    return affected_gaussians(orc, orc.px_fragile) | orc.geom_fragile


def check_radii(gpu_radii, orc):
    r = gpu_radii.cpu().numpy()
    ok = (r == orc.radii) | orc.geom_fragile
    assert ok.all(), f"{(~ok).sum()} radii differ on non-fragile Gaussians"


def relerr(a, b):
    a = a.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return np.abs(a - b.reshape(a.shape)).max() / max(np.abs(b).max(), 1e-30)


def _last_stats(dev):
    from pf3plat_b200.rasterizer import last_stats
    return last_stats(dev)


def render_batch(sc, dev, use_sh=True, with_depth=False, requires_grad=False, scale_rot=False):
    from pf3plat_b200.render import render_views
    d = sc.to(dev)
    leaves = {"means": d.means[None].clone(), "cov": d.covariances[None].clone(), "sh": d.harmonics[None].clone(),
              "opac": d.opacities[None].clone()}
    if requires_grad:
        for t in leaves.values():
            t.requires_grad_(True)
    sh = leaves["sh"] if use_sh else leaves["sh"][..., :1]
    out = render_views(d.extrinsics, d.intrinsics, d.near, d.far, d.image_shape, d.background, leaves["means"],
                       leaves["cov"], sh, leaves["opac"], use_sh=use_sh, with_depth=with_depth)
    return out, leaves


@pytest.mark.parametrize("P,hw,views", [(3000, (64, 64), 2), (20000, (70, 50), 3), (500, (16, 16), 1)])
@pytest.mark.parametrize("use_sh", [True, False])
def test_forward_matches_oracle(P, hw, views, use_sh):
    dev = _dev()
    sc = make_scene(P, views, hw[0], hw[1], seed=1)
    color, _ = render_batch(sc, dev, use_sh=use_sh)
    assert color.shape == (views, 3, hw[0], hw[1])
    for v in range(views):
        check_image(color[v], oracle_view(sc, v, use_sh=use_sh))


def test_per_view_dropin_matches_oracle_and_batched_path():
    from tests.ref_callsite import render_like_reference
    dev = _dev()
    views = 3
    sc = make_scene(5000, views, 64, 80, seed=2)
    d = sc.to(dev)
    rep = lambda t: t[None].expand(views, *t.shape)
    img, radii = render_like_reference(d.extrinsics, d.intrinsics, d.near, d.far, d.image_shape, d.background,
                                       rep(d.means), rep(d.covariances), rep(d.harmonics), rep(d.opacities),
                                       return_radii=True)
    batched, _ = render_batch(sc, dev)
    for v in range(views):
        orc = oracle_view(sc, v)
        check_image(img[v], orc)
        check_radii(radii[v], orc)
    # the batched entry applies the 1/near rescale inside the kernel; near == 1 here, so both paths are bit-identical
    assert torch.equal(img, batched)


@pytest.mark.parametrize("mode", ["sh_cov", "rgb_cov", "sh_scalerot"])
def test_backward_matches_oracle(mode):
    from pf3plat_b200.rasterizer import GaussianRasterizationSettings, GaussianRasterizer
    dev = _dev()
    sc = make_scene(4000, 2, 48, 64, seed=3)
    v = 1
    st, kw = view_args(sc, v, use_sh=mode.startswith("sh"))
    if mode.endswith("scalerot"):
        kw.pop("cov3D_precomp")
        kw["scales"] = sc.scales.numpy()
        kw["rotations"] = sc.rotations.numpy()
    from oracle.gs_oracle import OracleRender
    orc = OracleRender(st, **kw)
    assert orc.px_fragile.sum() == 0 or orc.px_fragile.mean() < 0.01
    H, W = sc.image_shape
    target = make_target(1, H, W)[0].numpy()
    dL = (2 * (orc.color - target) / target.size).astype(np.float32)
    g_ref = orc.backward(dL)

    settings = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=st.tanfovx, tanfovy=st.tanfovy, bg=torch.tensor(st.bg, device=dev),
        scale_modifier=1.0, viewmatrix=torch.tensor(st.viewmatrix, device=dev),
        projmatrix=torch.tensor(st.projmatrix, device=dev), sh_degree=st.sh_degree,
        campos=torch.tensor(st.campos, device=dev), prefiltered=False, debug=False)
    tk = {k: torch.tensor(np.asarray(a), dtype=torch.float32, device=dev, requires_grad=True) for k, a in kw.items()}
    tk["opacities"] = tk["opacities"].detach().reshape(-1, 1).requires_grad_(True)
    m2d = torch.zeros(sc.means.shape[0], 3, device=dev, requires_grad=True)
    color, radii = GaussianRasterizer(settings)(means2D=m2d, **tk)
    check_image(color, orc)
    check_radii(radii, orc)
    (color * torch.tensor(dL, device=dev)).sum().backward()
    aff = affected_of(orc)
    for name, t in tk.items():
        check_grad(f"{mode} dL/d{name}", t.grad, g_ref[name], aff, bands=SH_BANDS if name == "shs" else None)
    check_grad(f"{mode} dL/dmeans2D", m2d.grad, g_ref["means2D"], aff)


def test_batched_backward_sums_views_and_matches_oracle():
    dev = _dev()
    views = 3
    sc = make_scene(6000, views, 64, 64, seed=4)
    (color, depth), leaves = render_batch(sc, dev, with_depth=True, requires_grad=True)
    target = make_target(views, 64, 64).to(dev)
    wd = 1e-3
    loss = ((color - target) ** 2).mean() + wd * depth.mean()
    loss.backward()
    gm = np.zeros((6000, 3)); go = np.zeros(6000); gs = np.zeros((6000, 25, 3)); gc = np.zeros((6000, 6))
    aff = np.zeros(6000, bool)
    for v in range(views):
        orc = oracle_view(sc, v, with_depth=True)
        aff |= affected_of(orc)
        check_image(color[v], orc)
        derr = np.abs(depth[v].detach().cpu().numpy() - orc.depth)[~orc.px_fragile].max()
        assert derr <= 1e-3, derr      # depth values reach ~20: 1e-3 abs is ~5e-5 relative
        dL = (2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32)
        dLd = np.full((64, 64), wd / (views * 64 * 64), np.float32)
        g = orc.backward(dL, dLd)
        gm += g["means3D"]; go += g["opacities"][:, 0]; gs += g["shs"]; gc += g["cov3D_precomp"]
    check_grad("batched dL/dmeans", leaves["means"].grad[0], gm, aff)
    check_grad("batched dL/dopacities", leaves["opac"].grad[0].reshape(-1, 1), go.reshape(-1, 1), aff)
    check_grad("batched dL/dshs", leaves["sh"].grad[0].permute(0, 2, 1), gs, aff, bands=SH_BANDS)
    # covariance gradient arrives on the (3,3) matrix; fold it to the 6 unique entries
    G = leaves["cov"].grad[0].cpu().numpy()
    g6 = np.stack([G[:, 0, 0], G[:, 0, 1], G[:, 0, 2], G[:, 1, 1], G[:, 1, 2], G[:, 2, 2]], -1)
    check_grad("batched dL/dcov3D", g6, gc, aff)


@pytest.mark.parametrize("blow_up", [25.0, 400.0])
def test_huge_footprints_backward_matches_oracle(blow_up):
    """A few Gaussians blown up to cover most of the image (every one reaches thousands of pixels in every tile): the
    backward compositor's per-block moment sums are taken about the block centre and shifted to the Gaussian's own offset
    (hundreds of pixels here) -- gradients against the oracle's direct per-pixel sums."""
    dev = _dev()
    views, P, hw = 2, 24, (48, 80)
    sc = make_scene(P, views, *hw, seed=17)
    sc.covariances.mul_(blow_up)
    out, leaves = render_batch(sc, dev, requires_grad=True)
    color = out[0] if isinstance(out, (tuple, list)) else out
    target = make_target(views, *hw).to(dev)
    ((color - target) ** 2).mean().backward()
    gm = np.zeros((P, 3)); go = np.zeros(P); gs = np.zeros((P, 25, 3)); gc = np.zeros((P, 6))
    aff = np.zeros(P, bool)
    for v in range(views):
        orc = oracle_view(sc, v)
        aff |= affected_of(orc)
        check_image(color[v], orc, max_fragile_frac=0.1)
        dL = (2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32)
        g = orc.backward(dL)
        gm += g["means3D"]; go += g["opacities"][:, 0]; gs += g["shs"]; gc += g["cov3D_precomp"]
    aff[:] = False      # with two dozen Gaussians everything touches a fragile pixel: hold them all to the strict bound
    check_grad(f"x{blow_up:g} dL/dmeans", leaves["means"].grad[0], gm, aff)
    check_grad(f"x{blow_up:g} dL/dopacities", leaves["opac"].grad[0].reshape(-1, 1), go.reshape(-1, 1), aff)
    check_grad(f"x{blow_up:g} dL/dshs", leaves["sh"].grad[0].permute(0, 2, 1), gs, aff, bands=SH_BANDS)
    G = leaves["cov"].grad[0].cpu().numpy()
    g6 = np.stack([G[:, 0, 0], G[:, 0, 1], G[:, 0, 2], G[:, 1, 1], G[:, 1, 2], G[:, 2, 2]], -1)
    check_grad(f"x{blow_up:g} dL/dcov3D", g6, gc, aff)


@pytest.mark.parametrize("d_sh,P", [(1, 1000), (4, 1001), (9, 777), (16, 1300), (16, 129), (25, 1301), (25, 63)])
def test_sh_coefficient_counts_and_ragged_blocks(d_sh, P):
    """Every staging path of the SH block, forward and backward, against the oracle: M <= 16 (one bulk TMA copy when the
    CTA's block is 16-byte aligned, the plain loop for ragged tails and unaligned slices), M = 25 (4-byte cp.async gather
    of the 16 evaluated coefficients into odd-stride rows; zero bands appended to the gradient), Gaussian counts that are
    not multiples of the CTA size."""
    from pf3plat_b200.render import render_views
    dev = _dev()
    sc = make_scene(P, 2, 48, 48, seed=40 + d_sh, d_sh=d_sh)
    d = sc.to(dev)
    leaves = [t.clone().requires_grad_(True) for t in (d.means[None], d.covariances[None], d.harmonics[None], d.opacities[None])]
    color = render_views(d.extrinsics, d.intrinsics, d.near, d.far, d.image_shape, d.background, *leaves)
    target = make_target(2, 48, 48).to(dev)
    ((color - target) ** 2).mean().backward()
    gm = np.zeros((P, 3)); gs = np.zeros((P, d_sh, 3))
    aff = np.zeros(P, bool)
    for v in range(2):
        orc = oracle_view(sc, v)
        check_image(color[v], orc)
        aff |= affected_of(orc)
        dL = (2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32)
        g = orc.backward(dL)
        gm += g["means3D"]; gs += g["shs"]
    check_grad(f"d_sh={d_sh} dL/dmeans", leaves[0].grad[0], gm, aff)
    bands = [b for b in SH_BANDS if b[1].start < d_sh]
    check_grad(f"d_sh={d_sh} dL/dshs", leaves[2].grad[0].permute(0, 2, 1), gs, aff, bands=bands)
    if d_sh > 16:
        assert float(leaves[2].grad[0][..., 16:].abs().max()) == 0.0


def test_edge_cases():
    from pf3plat_b200.rasterizer import BatchSettings, rasterize_batch
    dev = _dev()
    eye = torch.eye(4, device=dev)[None]
    proj = torch.tensor([[2.0, 0, 0, 0], [0, 2.0, 0, 0], [0, 0, 100 / 99, 1], [0, 0, -100 / 99, 0]], device=dev)[None]
    bg = torch.tensor([[0.25, 0.5, 0.75]], device=dev)
    bs = BatchSettings(image_height=40, image_width=24, viewmatrix=eye, projmatrix=proj, campos=torch.zeros(1, 3, device=dev),
                       bg=bg, sh_degree=0, tanfovx=0.5, tanfovy=0.5)
    # empty cloud -> background
    color, radii = rasterize_batch(bs, torch.zeros(1, 0, 3, device=dev), torch.zeros(1, 0, device=dev),
                                   colors_precomp=torch.zeros(1, 0, 3, device=dev),
                                   cov3D_precomp=torch.zeros(1, 0, 6, device=dev))
    assert radii.shape == (1, 0) and torch.allclose(color[0, :, 3, 3], bg[0])
    # everything culled (behind the 0.2 near plane) or invisible (opacity below 1/255)
    means = torch.tensor([[[0.0, 0, 0.1], [0, 0, 5.0]]], device=dev)
    cov = torch.tensor([[[0.01, 0, 0, 0.01, 0, 0.01]] * 2], device=dev)
    color, radii = rasterize_batch(bs, means, torch.tensor([[1.0, 0.003]], device=dev),
                                   colors_precomp=torch.ones(1, 2, 3, device=dev), cov3D_precomp=cov)
    assert radii[0, 0] == 0 and radii[0, 1] > 0
    assert torch.allclose(color, bg[0][None, :, None, None].expand_as(color))
    # one huge opaque Gaussian covers the whole (ragged: 40x24 is not a multiple of 16) image
    big = torch.tensor([[[50.0, 0, 0, 50.0, 0, 50.0]]], device=dev)
    color, radii = rasterize_batch(bs, means[:, 1:], torch.ones(1, 1, device=dev),
                                   colors_precomp=torch.full((1, 1, 3), 0.5, device=dev), cov3D_precomp=big)
    expect = 0.99 * 0.5 + 0.01 * bg[0]
    assert torch.allclose(color[0, :, 20, 12], expect, atol=2e-3) and torch.isfinite(color).all()


def test_determinism_and_linearity_at_full_size():
    """BASELINE.json configs[1] size (500k Gaussians, 256x256), 2 of the 8 views: forward is bit-reproducible, one
    view is checked against the oracle, and the backward is linear in dL/dcolor (size-independent properties)."""
    dev = _dev()
    sc = make_scene(500_000, 2, 256, 256, seed=0, total_views=8)
    (c1, leaves) = render_batch(sc, dev, requires_grad=True)
    c2, _ = render_batch(sc, dev)
    assert torch.equal(c1, c2)
    orc = oracle_view(sc, 1)
    check_image(c1[1], orc)
    g = torch.randn_like(c1)
    (ga,) = torch.autograd.grad((c1 * g).sum(), leaves["means"], retain_graph=True)
    (gb,) = torch.autograd.grad((c1 * (2 * g)).sum(), leaves["means"])
    assert relerr(gb, (2 * ga).cpu().numpy()) < 1e-5     # float atomics reorder sums: not bit-exact
    assert torch.isfinite(ga).all()


def _render_with_tuning(sc, dev, tuning):
    from pf3plat_b200.cameras import make_view_batch
    from pf3plat_b200.rasterizer import BatchSettings, last_stats, rasterize_batch
    d = sc.to(dev)
    vb = make_view_batch(d.extrinsics, d.intrinsics, d.near, d.far)
    h, w = sc.image_shape
    bs = BatchSettings(image_height=h, image_width=w, viewmatrix=vb.viewmatrix, projmatrix=vb.projmatrix,
                       campos=vb.campos, bg=d.background, sh_degree=4, tanfov=vb.tanfov, view_scale=vb.scale,
                       tuning=tuning)
    c = d.covariances
    cov6 = torch.stack([c[:, 0, 0], c[:, 0, 1], c[:, 0, 2], c[:, 1, 1], c[:, 1, 2], c[:, 2, 2]], -1)
    color, radii = rasterize_batch(bs, d.means[None], d.opacities[None], shs=d.harmonics.permute(0, 2, 1)[None],
                                   cov3D_precomp=cov6[None])
    return color, last_stats(dev)


def test_compositor_variants_agree():
    """Round-2 kernels against the round-1 kernels they replace (kept behind tuning flags for A/B): the persistent
    warp-specialised forward compositor gives bit-identical images, final T and contributor counts (same arithmetic in
    the same order); the pair-matrix backward gives the same gradients up to the re-association of the sums."""
    from pf3plat_b200._capi import (GS_TUNE_BWD_OCC4, GS_TUNE_BWD_V1, GS_TUNE_FWD_WS, GS_TUNE_PBWD_2PHASE, GS_TUNE_PRE_OCC6,
                                    GS_TUNE_PRE_SH_RAW16)
    from pf3plat_b200.cameras import make_view_batch
    from pf3plat_b200.rasterizer import BatchSettings, rasterize_batch
    dev = _dev()
    from tests.util import make_posed_scene
    for sc, depth in ((make_scene(40000, 3, 80, 112, seed=12), True), (make_scene(300, 1, 16, 16, seed=13), False),
                      (make_scene(150000, 2, 128, 128, seed=14), False),
                      (make_posed_scene(40000, 4, 80, 112, seed=12), True)):   # rotated views, near != 1, clamped
        d = sc.to(dev)
        vb = make_view_batch(d.extrinsics, d.intrinsics, d.near, d.far)
        h, w = sc.image_shape
        c = d.covariances
        cov6 = torch.stack([c[:, 0, 0], c[:, 0, 1], c[:, 0, 2], c[:, 1, 1], c[:, 1, 2], c[:, 2, 2]], -1)[None]
        bg = torch.rand(d.background.shape, device=dev)
        outs, grads = {}, {}
        variants = (GS_TUNE_FWD_WS, GS_TUNE_BWD_V1, GS_TUNE_FWD_WS | GS_TUNE_BWD_V1, GS_TUNE_BWD_OCC4, GS_TUNE_PBWD_2PHASE,
                    GS_TUNE_PRE_OCC6, GS_TUNE_PRE_SH_RAW16)
        for tuning in (0,) + variants:
            bs = BatchSettings(image_height=h, image_width=w, viewmatrix=vb.viewmatrix, projmatrix=vb.projmatrix,
                               campos=vb.campos, bg=bg, sh_degree=4, tanfov=vb.tanfov, view_scale=vb.scale,
                               tuning=tuning, with_depth=depth)
            leaves = [t.clone().requires_grad_(True) for t in (d.means[None], d.opacities[None],
                                                               d.harmonics.permute(0, 2, 1).contiguous()[None], cov6)]
            out = rasterize_batch(bs, leaves[0], leaves[1], shs=leaves[2], cov3D_precomp=leaves[3])
            g = torch.Generator(device="cpu").manual_seed(3)
            wgt = torch.randn(out[0].shape, generator=g).to(dev)
            loss = (out[0] * wgt).sum() + (0.01 * out[2].sum() if depth else 0.0)
            loss.backward()
            outs[tuning] = [o.detach() for o in out]
            grads[tuning] = [t.grad for t in leaves]
        for tuning in variants:
            for a, b in zip(outs[0], outs[tuning]):
                assert torch.equal(a, b), tuning
            for a, b in zip(grads[0], grads[tuning]):
                assert float((a - b).abs().max()) <= 2e-5 * float(b.abs().max()) + 1e-12, tuning


def test_alternating_shapes_keep_their_speculation_state():
    """A context remembers several shapes: a caller that alternates two of them (context / target views of a training step,
    training / validation batches) gets the speculative path for both from their third call on, with the pixels of the exact
    path; cycling through more shapes than there are slots only evicts (every call exact or re-learning, still the same
    pixels)."""
    from pf3plat_b200._capi import GS_TUNE_NO_SPECULATION
    from pf3plat_b200.cameras import make_view_batch
    from pf3plat_b200.rasterizer import BatchSettings, last_stats, rasterize_batch
    dev = _dev()

    def shape(P, V, hw, seed):
        sc = make_scene(P, V, *hw, seed=seed).to(dev)
        vb = make_view_batch(sc.extrinsics, sc.intrinsics, sc.near, sc.far)
        c = sc.covariances
        cov6 = torch.stack([c[:, 0, 0], c[:, 0, 1], c[:, 0, 2], c[:, 1, 1], c[:, 1, 2], c[:, 2, 2]], -1)[None]
        args = (sc.means[None], sc.opacities[None])
        kw = dict(shs=sc.harmonics.permute(0, 2, 1).contiguous()[None], cov3D_precomp=cov6)
        mk = lambda tuning: BatchSettings(image_height=hw[0], image_width=hw[1], viewmatrix=vb.viewmatrix, projmatrix=vb.projmatrix,
                                          campos=vb.campos, bg=sc.background, sh_degree=4, tanfov=vb.tanfov, tuning=tuning)
        with torch.no_grad():
            ref = rasterize_batch(mk(GS_TUNE_NO_SPECULATION), *args, **kw)[0].clone()
        return mk(0), args, kw, ref

    shapes = [shape(20000, 2, (64, 80), 31), shape(30000, 3, (48, 48), 32)]
    states = []
    for it in range(5):
        for bs, args, kw, ref in shapes:
            with torch.no_grad():
                out = rasterize_batch(bs, *args, **kw)[0]
            assert torch.equal(out, ref)
            states.append(last_stats(dev)["speculative"])
    assert all(s >= 1 for s in states[4:]), states     # both shapes speculative from their third call on
    more = shapes + [shape(10000 + 1000 * k, 1 + k % 3, (32, 48), 40 + k) for k in range(4)]
    for it in range(3):
        for bs, args, kw, ref in more:
            with torch.no_grad():
                assert torch.equal(rasterize_batch(bs, *args, **kw)[0], ref)


def test_binning_paths_agree_bit_for_bit():
    """Exact-capacity buckets, speculative-capacity buckets (later calls of a shape; whole-tile sorts or depth strata)
    and the device-wide radix-sort fallback give the same lists, hence the same pixels; overflowing the learned
    capacities is detected and redone; a scene whose densest tile exceeds the shared-memory sort capacity takes the
    radix fallback by itself."""
    from pf3plat_b200._capi import (GS_TUNE_FORCE_RADIX_BINNING, GS_TUNE_NO_SPECULATION, GS_TUNE_NO_STRATA,
                                    GS_TUNE_SEPARATE_EMIT)
    dev = _dev()
    sc = make_scene(30000, 2, 64, 96, seed=7)
    exact, st_exact = _render_with_tuning(sc, dev, GS_TUNE_NO_SPECULATION)   # also learns capacities + depth strata
    first, st_first = _render_with_tuning(sc, dev, 0)          # trial of the strata on doubled capacities
    spec, st_spec = _render_with_tuning(sc, dev, 0)            # strata on their own learned capacities, fused appends
    spec2, st_spec2 = _render_with_tuning(sc, dev, GS_TUNE_SEPARATE_EMIT)   # same, buckets filled by k_emit_buckets
    assert st_first["speculative"] == 2 and st_spec2["speculative"] == 2 and torch.equal(exact, spec2)
    whole, st_whole = _render_with_tuning(sc, dev, GS_TUNE_NO_STRATA | GS_TUNE_NO_SPECULATION)  # re-learn unstratified
    whole, st_whole = _render_with_tuning(sc, dev, GS_TUNE_NO_STRATA)        # speculative, whole-tile sorts
    assert st_whole["speculative"] == 1 and torch.equal(exact, whole)
    slow, st_slow = _render_with_tuning(sc, dev, GS_TUNE_FORCE_RADIX_BINNING)
    assert st_exact["speculative"] == 0 and st_spec["speculative"] == 2 and st_slow["speculative"] == 0
    assert st_exact["num_rendered"] == st_spec["num_rendered"] == st_slow["num_rendered"]
    assert st_exact["max_tile_list"] == st_spec["max_tile_list"] <= 8192
    assert torch.equal(exact, spec) and torch.equal(exact, slow) and torch.equal(exact, first)
    # same shape (2 views, 24 tiles), 2.5x the Gaussians: the learned capacities overflow -> detected, redone exactly
    dense = make_scene(75000, 2, 64, 96, seed=7)
    got, st_got = _render_with_tuning(dense, dev, 0)
    ref, _ = _render_with_tuning(dense, dev, GS_TUNE_NO_SPECULATION)
    assert st_got["speculative"] == 0 and torch.equal(got, ref)
    again, st_again = _render_with_tuning(dense, dev, 0)       # capacities re-learned from the exact pass
    assert st_again["speculative"] >= 1 and torch.equal(again, ref)
    # every Gaussian twice (identical depth, different colour): the radix tile sort (depth bits only) meets ties in
    # every tile and must hand those tiles to the 64-bit merge sort -- index order decides, as in the oracle
    twin = make_scene(30000, 1, 64, 96, seed=9)
    for name in ("means", "covariances", "opacities", "scales", "rotations"):
        setattr(twin, name, torch.cat([getattr(twin, name)] * 2))
    twin.harmonics = torch.cat([twin.harmonics, twin.harmonics.flip(1)])
    tw, st_tw = _render_with_tuning(twin, dev, 0)
    tw_slow, _ = _render_with_tuning(twin, dev, GS_TUNE_FORCE_RADIX_BINNING)
    assert st_tw["max_tile_list"] > 2048 and torch.equal(tw, tw_slow)
    check_image(tw[0], oracle_view(twin, 0), max_fragile_frac=1.0)   # every pixel sees equal depths: all "fragile"
    # 40k Gaussians squeezed into the centre of a 32x32 image: > 8192 entries in one tile
    huge = make_scene(40000, 1, 32, 32, seed=8)
    huge.means[:, :2] *= 0.05
    color, st = _render_with_tuning(huge, dev, 0)
    assert st["max_tile_list"] > 8192 and st["speculative"] == 0
    check_image(color[0], oracle_view(huge, 0), max_fragile_frac=0.2)
    color2, st2 = _render_with_tuning(huge, dev, 0)            # lists too long to speculate on: still exact
    assert st2["speculative"] == 0 and torch.equal(color, color2)


@pytest.mark.parametrize("levels", [8, 64, 4096])
def test_stratum_sort_handles_depth_ties(levels):
    """The hand-written warp-per-stratum sort forms its buckets on the depth bits.  Depths quantised to a few levels put
    EXACT ties en masse into every stratum: 8 levels = one depth per stratum (buckets are then formed on the index), 64
    levels = a handful of crowded buckets per stratum (ranked cooperatively), 4096 = ordinary small ties.  Lists must be
    bit-identical to the exact path's and to the merge-sort kernel's."""
    from pf3plat_b200._capi import GS_TUNE_NO_SPECULATION, GS_TUNE_STRATA_MERGE_SORT
    dev = _dev()
    sc = make_scene(60000, 2, 96, 96, seed=15)
    z = sc.means[:, 2]
    q = torch.exp(torch.round(torch.log(z) * (levels / 3.0)) / (levels / 3.0))     # log-spaced levels between 1.5 and 20
    sc.means = sc.means * (q / z)[:, None]                                          # same pixel, quantised depth
    exact, st0 = _render_with_tuning(sc, dev, GS_TUNE_NO_SPECULATION)
    _render_with_tuning(sc, dev, 0)                                                 # strata trial
    ours, st1 = _render_with_tuning(sc, dev, 0)
    merge, st2 = _render_with_tuning(sc, dev, GS_TUNE_STRATA_MERGE_SORT)
    assert st0["speculative"] == 0
    if st1["speculative"] == 2:      # (a shape whose strata overflow falls back to whole-tile sorts: nothing to compare)
        assert st2["speculative"] == 2
    assert torch.equal(exact, ours) and torch.equal(exact, merge)
    assert st0["num_rendered"] == st1["num_rendered"]


def test_pixel_aligned_pf3plat_shaped_cloud():
    """2 x 128 x 128 pixel-aligned Gaussians (the structure PF3plat's encoder emits): neighbouring indices share
    tiles, lists are short, many splats are sub-pixel.  Forward and backward against the oracle."""
    from pf3plat_b200.synthetic import make_pixel_aligned_scene
    dev = _dev()
    sc = make_pixel_aligned_scene(128, 128, 3, seed=2)
    assert sc.means.shape[0] == 2 * 128 * 128
    color, leaves = render_batch(sc, dev, requires_grad=True)
    target = make_target(3, 128, 128).to(dev)
    ((color - target) ** 2).mean().backward()
    gm = 0
    aff = np.zeros(sc.means.shape[0], bool)
    for v in range(3):
        orc = oracle_view(sc, v)
        check_image(color[v], orc)
        aff |= affected_of(orc)
        dL = (2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32)
        gm = gm + orc.backward(dL)["means3D"]
    check_grad("pixel-aligned dL/dmeans", leaves["means"].grad[0], gm, aff)
    # Depth strata on a cloud whose tiles each see a narrow depth range (a smooth surface): the per-view octiles do
    # not balance such tiles, the trial overflows, and the library switches the shape to per-(view, tile) boundaries
    # (learned from the exact redo's sorted lists, refreshed by every call's sort).  Every call gives the same pixels,
    # and the shape ends up on the stratified path.
    states = []
    for _ in range(7):
        again, _ = render_batch(sc, dev)
        states.append(_last_stats(dev)["speculative"])
        assert torch.equal(again, color.detach())
    print("[strata] pixel-aligned cloud, speculative state per call:", states)
    assert states[-1] == 2, states
