"""Pins the C oracle's hand-written backward: (1) against torch.autograd on an independent vectorised
restatement of the forward (oracle/torch_oracle.py), in fp64; (2) against central finite differences of its own
fp64 forward.  Tolerance 1e-5 relative to each tensor's max-abs (the upstream backward replaces 1/det^2 by
1/(det^2+1e-7), a deliberate ~1e-6-relative deviation from the exact derivative; SURVEY.md Appendix A)."""
import numpy as np
import pytest
import torch

from oracle import torch_oracle
from oracle.gs_oracle import OracleRender
from pf3plat_b200.synthetic import make_scene, make_target
from tests.util import affected_gaussians, make_posed_scene, posed_regimes, view_args, view_scales


def _relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-30)


def _scene(P=300, hw=48, seed=3, views=3):
    return make_scene(P, views, hw, hw, seed=seed, d_sh=25)


def _posed(P=300, hw=48, seed=3, views=3):
    """Rotated cameras (view 1: rolled 90 degrees, near 0.5), tanfovx != tanfovy, a background, and Gaussians behind
    the camera, in the near cull, past the guard band and far off-axis (tests/util.make_posed_scene)."""
    return make_posed_scene(P, views, hw, hw, seed=seed)


@pytest.mark.parametrize("mode", ["sh_cov", "rgb_cov", "sh_scalerot", "rgb_cov_depth",
                                  "posed_sh_cov", "posed_rgb_cov", "posed_sh_scalerot", "posed_rgb_cov_depth"])
def test_c_backward_matches_autograd(mode):
    posed = mode.startswith("posed_")
    mode = mode.removeprefix("posed_")
    sc = _posed() if posed else _scene()
    v = 1
    st, kw = view_args(sc, v, use_sh=mode.startswith("sh"))
    if "scalerot" in mode:
        s = float(view_scales(sc)[v])
        kw.pop("cov3D_precomp")
        kw["scales"] = sc.scales.numpy().astype(np.float64) * s     # the 1/near rescale view_args applies to means
        kw["rotations"] = sc.rotations.numpy().astype(np.float64)
    if posed:      # the regimes this scene exists for are really in view
        reg = posed_regimes(sc, v)
        assert reg["behind"].sum() >= 3 and reg["near_cull"].sum() >= 3 and reg["off_axis"].sum() >= 2
        assert st.tanfovx / st.tanfovy > 1.2 and st.bg.min() > 0
    with_depth = mode.endswith("depth")
    r = OracleRender(st, dtype=np.float64, with_depth=with_depth, **kw)
    H, W = sc.image_shape
    target = make_target(1, H, W)[0].double().numpy()
    dL = 2 * (r.color - target) / target.size
    dLd = (np.cos(np.arange(H * W).reshape(H, W)) * 1e-3) if with_depth else None
    g = r.backward(dL, dLd)

    tk = {k: torch.tensor(np.asarray(a, np.float64), requires_grad=True) for k, a in kw.items()}
    m2d = torch.zeros(sc.means.shape[0], 3, dtype=torch.float64, requires_grad=True)
    out = torch_oracle.render(st, means2D=m2d, with_depth=with_depth, **tk)
    color = out[0]
    assert np.abs(color.detach().numpy() - r.color).max() < 1e-9
    assert (out[1].numpy() == r.radii).all()
    loss = (color * torch.tensor(dL)).sum()
    if with_depth:
        assert np.abs(out[2].detach().numpy() - r.depth).max() < 1e-8
        loss = loss + (out[2] * torch.tensor(dLd)).sum()
    loss.backward()
    assert r.num_rendered > 100
    if posed:
        clamped = (reg["x_out"] | reg["y_out"]) & (r.radii > 0)
        assert clamped.sum() >= 3 and (r.radii[reg["behind"] | reg["near_cull"] | reg["off_axis"]] == 0).all()
    for name, t in tk.items():
        key = name
        ga = t.grad.numpy().reshape(np.asarray(g[key]).shape)
        assert _relerr(g[key], ga) < 1e-5, (name, _relerr(g[key], ga))
    assert _relerr(g["means2D"], m2d.grad.numpy()) < 1e-5


def test_c_backward_matches_finite_differences():
    _finite_differences(_scene(P=60, hw=32, seed=5, views=2), 0, None)
    # posed: view 1 (rolled 90 degrees, near 0.5 -> view_scale 2, tanfovx != tanfovy, background 0.1..0.9).  Indices
    # include Gaussians clamped by the guard band, Gaussians just past the near cull and Gaussians seen over pixels where
    # the background still shows (final T > 0.05).  The means of clamped Gaussians are left out: there the upstream
    # backward (which the oracle follows) is not the derivative of its forward -- it masks d/dt.x and holds the clamped
    # t.x constant in d/dt.z; tests/test_oracle_known_answers.py pins that rule instead.
    sc = _posed(P=200, hw=32, seed=5, views=2)
    st, kw = view_args(sc, 1)
    r = OracleRender(st, dtype=np.float64, **kw)
    reg = posed_regimes(sc, 1)
    vis = r.radii > 0
    clamped = np.nonzero((reg["x_out"] | reg["y_out"]) & vis)[0]
    near = np.nonzero((reg["z"] < 1.0) & vis)[0]
    lit = (r.final_T > 0.05)
    bgpx = np.nonzero(vis & affected_gaussians(r, lit))[0]
    assert len(clamped) >= 2 and len(near) >= 2 and len(bgpx) >= 4 and lit.mean() > 0.05
    _finite_differences(sc, 1, {"clamped": clamped[:4], "near": near[:4], "background": bgpx[:4], "clamped_all": clamped})


def _finite_differences(sc, v, chosen):
    H, W = sc.image_shape
    st, kw = view_args(sc, v, use_sh=True)
    kw = {k: np.asarray(a, np.float64) for k, a in kw.items()}
    rng = np.random.default_rng(0)
    dL = rng.standard_normal((3, H, W))

    def loss(**over):
        k2 = dict(kw)
        k2.update(over)
        return float((OracleRender(st, dtype=np.float64, frag_rel=0, **k2).color * dL).sum())

    g = OracleRender(st, dtype=np.float64, **kw).backward(dL)
    for name in ["means3D", "opacities", "cov3D_precomp", "shs"]:
        base = kw[name]
        flat_g = np.asarray(g[name]).reshape(-1)
        idx = rng.choice(base.size, size=12, replace=False)
        per = base.size // base.shape[0]
        if chosen is not None:      # the first elements of every chosen Gaussian too
            ids = np.unique(np.concatenate(list(chosen.values())))
            idx = np.concatenate([idx, (ids[:, None] * per + np.arange(min(per, 6))[None, :]).reshape(-1)])
            if name == "means3D":   # not the means of the Gaussians the guard band clamps (see above)
                idx = idx[~np.isin(idx // per, chosen["clamped_all"])]
        scale = np.abs(flat_g).max()
        for i in idx:
            eps = 1e-6 * max(1.0, abs(base.reshape(-1)[i]))
            p, m = base.copy().reshape(-1), base.copy().reshape(-1)
            p[i] += eps
            m[i] -= eps
            fd = (loss(**{name: p.reshape(base.shape)}) - loss(**{name: m.reshape(base.shape)})) / (2 * eps)
            assert abs(fd - flat_g[i]) < 2e-4 * scale + 1e-9, (name, i, fd, flat_g[i])


def test_fp32_oracle_agrees_with_fp64_outside_fragile_pixels():
    posed = make_posed_scene(10_000, 4, 96, 128, seed=0)
    for sc, v in [(make_scene(10_000, 1, 256, 256, seed=0), 0)] + [(posed, v) for v in range(4)]:   # C1, posed views
        st, kw = view_args(sc, v)
        r32 = OracleRender(st, dtype=np.float32, **kw)
        r64 = OracleRender(st, dtype=np.float64, **kw)
        frag = r32.px_fragile | r64.px_fragile
        err = np.abs(r32.color.astype(np.float64) - r64.color).max(axis=0)
        assert frag.mean() < 0.02, (v, frag.mean())
        assert err[~frag].max() < 1e-4          # north_star tolerance, abs RGB
        same = r32.radii == r64.radii
        assert (same | r32.geom_fragile | r64.geom_fragile).all()
