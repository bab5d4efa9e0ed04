"""Pins the CPU oracle with closed-form, hand-derived answers (SURVEY.md section 8(c) item 2).

The reference ships no golden vectors for the rasterizer (SURVEY.md section 4), so these cases are what
"pinning" means here; each states the arithmetic it expects in plain Python."""
import math

import numpy as np
import pytest

from oracle.gs_oracle import OracleRender
from tests.util import simple_settings

DT = [np.float32, np.float64]


def _iso_cov6(s):
    return np.array([[s * s, 0, 0, s * s, 0, s * s]], np.float64)


@pytest.mark.parametrize("dt", DT)
def test_single_isotropic_gaussian_on_axis(dt):
    H = W = 64
    st = simple_settings(H, W, tanfov=0.5, bg=(0.1, 0.2, 0.3))
    z, s, o = 5.0, 0.05, 0.6
    c = np.array([[0.9, 0.5, 0.2]])
    r = OracleRender(st, means3D=np.array([[0.0, 0.0, z]]), opacities=np.array([o]), colors_precomp=c,
                     cov3D_precomp=_iso_cov6(s), dtype=dt)
    fx = W / (2 * 0.5)
    var = (fx / z) ** 2 * s * s + 0.3
    # ndc (0,0) -> pixel ((0+1)*64-1)/2 = 31.5
    assert np.allclose(r.xy[0], [31.5, 31.5], atol=1e-5)
    assert np.allclose(r.conic_opacity[0], [1 / var, 0, 1 / var, o], rtol=1e-5)
    # upstream clamps the eigenvalue discriminant at 0.1: lambda = mid + sqrt(max(0.1, mid^2-det))
    assert r.radii[0] == math.ceil(3 * math.sqrt(var + math.sqrt(0.1)))
    for (x, y) in [(31, 31), (32, 31), (30, 33), (35, 35)]:
        dx, dy = 31.5 - x, 31.5 - y
        a = min(0.99, o * math.exp(-0.5 * (dx * dx + dy * dy) / var))
        expect = (a * c[0] + (1 - a) * np.array([0.1, 0.2, 0.3])) if a >= 1 / 255 else np.array([0.1, 0.2, 0.3])
        assert np.allclose(r.color[:, y, x], expect, atol=2e-6)
        assert np.isclose(r.final_T[y, x], 1 - a if a >= 1 / 255 else 1.0, atol=1e-6)
    # far from the Gaussian: background only
    assert np.allclose(r.color[:, 0, 0], [0.1, 0.2, 0.3])
    assert r.num_visible == 1


@pytest.mark.parametrize("dt", DT)
def test_depth_order_independent_of_index_order(dt):
    st = simple_settings(65, 65, bg=(0, 0, 0))
    cols = np.array([[1.0, 0, 0], [0, 1.0, 0]])
    cov = np.repeat(_iso_cov6(0.2), 2, 0)
    out = []
    for zs in ([3.0, 6.0], [6.0, 3.0]):
        r = OracleRender(st, means3D=np.array([[0, 0, zs[0]], [0, 0, zs[1]]]), opacities=np.array([0.5, 0.5]),
                         colors_precomp=cols, cov3D_precomp=cov, dtype=dt)
        out.append(r.color[:, 32, 32].copy())
    # pixel (32,32) is the exact centre for W=65: alpha=0.5 each. front first: 0.5*front + 0.25*back
    assert np.allclose(out[0], [0.5, 0.25, 0], atol=1e-6)
    assert np.allclose(out[1], [0.25, 0.5, 0], atol=1e-6)


@pytest.mark.parametrize("dt", DT)
def test_equal_depth_ties_resolve_by_index(dt):
    st = simple_settings(65, 65)
    cols = np.array([[1.0, 0, 0], [0, 1.0, 0]])
    r = OracleRender(st, means3D=np.array([[0, 0, 4.0], [0, 0, 4.0]]), opacities=np.array([0.5, 0.5]),
                     colors_precomp=cols, cov3D_precomp=np.repeat(_iso_cov6(0.2), 2, 0), dtype=dt)
    assert np.allclose(r.color[:, 32, 32], [0.5, 0.25, 0], atol=1e-6)


@pytest.mark.parametrize("dt", DT)
def test_near_cull_and_alpha_clamp(dt):
    st = simple_settings(65, 65, bg=(0.3, 0.3, 0.3))
    # z = 0.1 <= 0.2: culled, radius 0, picture is background
    r = OracleRender(st, means3D=np.array([[0, 0, 0.1]]), opacities=np.array([1.0]), colors_precomp=np.ones((1, 3)),
                     cov3D_precomp=_iso_cov6(0.01), dtype=dt)
    assert r.radii[0] == 0 and r.num_rendered == 0
    assert np.allclose(r.color, 0.3)
    # opacity 1 at the exact centre: alpha clamps to 0.99
    r = OracleRender(st, means3D=np.array([[0, 0, 2.0]]), opacities=np.array([1.0]), colors_precomp=np.ones((1, 3)),
                     cov3D_precomp=_iso_cov6(0.1), dtype=dt)
    assert np.allclose(r.color[:, 32, 32], 0.99 * 1.0 + 0.01 * 0.3, atol=1e-6)


@pytest.mark.parametrize("dt", DT)
def test_transmittance_termination_excludes_the_stopping_gaussian(dt):
    st = simple_settings(65, 65, bg=(1.0, 1.0, 1.0))
    n = 20
    means = np.array([[0, 0, 2.0 + 0.1 * i] for i in range(n)])
    r = OracleRender(st, means3D=means, opacities=np.full(n, 0.5), colors_precomp=np.full((n, 3), 0.25),
                     cov3D_precomp=np.repeat(_iso_cov6(0.5), n, 0), dtype=dt)
    # T after k contributions = 0.5^k; 0.5^13 = 1.22e-4 >= 1e-4 but 0.5^14 < 1e-4 -> 14th is not added
    assert r.n_contrib[32, 32] == 13
    assert np.isclose(r.final_T[32, 32], 0.5 ** 13, rtol=1e-6)
    expect = 0.25 * (1 - 0.5 ** 13) + 1.0 * 0.5 ** 13
    assert np.allclose(r.color[:, 32, 32], expect, atol=1e-6)


@pytest.mark.parametrize("dt", DT)
def test_tile_rect_and_duplicates(dt):
    st = simple_settings(64, 64)
    # centre 31.5, radius r: rect = [int((31.5-r)/16), int((31.5+r+15)/16))
    s, z = 0.05, 5.0
    r = OracleRender(st, means3D=np.array([[0, 0, z]]), opacities=np.array([0.5]), colors_precomp=np.ones((1, 3)),
                     cov3D_precomp=_iso_cov6(s), dtype=dt)
    rad = r.radii[0]
    lo, hi = int((31.5 - rad) / 16), min(4, int((31.5 + rad + 15) / 16))
    assert r.tiles_touched[0] == (hi - lo) ** 2 == r.num_rendered
    rg = r.ranges
    assert sorted(np.nonzero(rg[:, 1] - rg[:, 0])[0].tolist()) == sorted(y * 4 + x for y in range(lo, hi) for x in range(lo, hi))


@pytest.mark.parametrize("dt", DT)
def test_backward_single_gaussian_closed_form(dt):
    st = simple_settings(65, 65, bg=(0.2, 0.2, 0.2))
    o, c = 0.4, np.array([[0.7, 0.1, 0.5]])
    r = OracleRender(st, means3D=np.array([[0, 0, 3.0]]), opacities=np.array([o]), colors_precomp=c,
                     cov3D_precomp=_iso_cov6(0.1), dtype=dt)
    dL = np.zeros((3, 65, 65))
    dL[:, 32, 32] = [1.0, 2.0, -1.0]       # one-hot at the exact centre: G = 1, alpha = o
    g = r.backward(dL)
    # C = alpha*c + (1-alpha)*bg  ->  dC/dc = alpha ; dC/do = G*(c-bg)
    assert np.allclose(g["colors_precomp"][0], o * dL[:, 32, 32], atol=1e-6)
    assert np.isclose(g["opacities"][0, 0], ((c[0] - 0.2) * dL[:, 32, 32]).sum(), atol=1e-6)
    # at the exact centre dG/dmean = 0
    assert np.allclose(g["means2D"][0], 0, atol=1e-6)


@pytest.mark.parametrize("dt", DT)
def test_sh_degree0_and_clamp(dt):
    st = simple_settings(65, 65, sh_degree=0)
    sh = np.zeros((1, 1, 3))
    sh[0, 0] = [1.0, -5.0, 0.0]
    r = OracleRender(st, means3D=np.array([[0, 0, 3.0]]), opacities=np.array([0.5]), shs=sh,
                     cov3D_precomp=_iso_cov6(0.1), dtype=dt)
    C0 = 0.28209479177387814
    assert np.allclose(r.rgb[0], [C0 + 0.5, 0.0, 0.5], atol=1e-6)
    assert r.clamped[0].tolist() == [False, True, False]
    g = r.backward(np.ones((3, 65, 65)))
    assert g["shs"][0, 0, 1] == 0.0 and g["shs"][0, 0, 0] > 0


def test_argument_validation():
    st = simple_settings(32, 32)
    with pytest.raises(ValueError):
        OracleRender(st, means3D=np.zeros((1, 3)), opacities=np.ones(1), cov3D_precomp=_iso_cov6(1))
    with pytest.raises(ValueError):
        OracleRender(st, means3D=np.zeros((1, 3)), opacities=np.ones(1), colors_precomp=np.ones((1, 3)))


def test_empty_cloud():
    st = simple_settings(32, 48, bg=(0.5, 0.25, 0.0))
    r = OracleRender(st, means3D=np.zeros((0, 3)), opacities=np.zeros(0), colors_precomp=np.zeros((0, 3)),
                     cov3D_precomp=np.zeros((0, 6)))
    assert r.num_rendered == 0 and np.allclose(r.color[1], 0.25)


def test_tile_lists_are_in_depth_then_index_order_for_any_thread_count():
    """The binning's contract (Appendix A "Binning": stable sort of (tile | depth bits) over instances emitted in index
    order): inside every tile range the (fp32 depth bits, Gaussian index) pairs strictly increase, every Gaussian
    appears once per tile of its rect, and the lists do not depend on the number of OpenMP threads."""
    from oracle import gs_oracle
    from pf3plat_b200.synthetic import make_scene
    from tests.util import view_args
    sc = make_scene(20000, 2, 96, 80, seed=5)
    # duplicate some Gaussians so that equal depths occur inside tiles
    import torch
    for name in ("means", "covariances", "opacities", "harmonics", "scales", "rotations"):
        t = getattr(sc, name)
        setattr(sc, name, torch.cat([t, t[:3000]]))
    st, kw = view_args(sc, 1)
    lists = []
    prev = gs_oracle.set_threads(0)
    try:
        for threads in (1, 3, max(prev, 2)):
            gs_oracle.set_threads(threads)
            r = OracleRender(st, **kw)
            pl, rg, tt = r.point_list, r.ranges, r.tiles_touched
            depth_bits = r.depths.astype(np.float32).view(np.uint32).astype(np.uint64)
            assert int(tt.sum()) == r.num_rendered == len(pl)
            assert np.array_equal(np.bincount(pl, minlength=len(tt)), tt)
            key = (depth_bits[pl] << np.uint64(32)) | pl.astype(np.uint64)
            covered = 0
            for a, b in rg:
                if b > a:
                    assert np.all(key[a + 1:b] > key[a:b - 1])
                    covered += b - a
            assert covered == len(pl)
            lists.append((pl.copy(), rg.copy(), r.color.copy()))
            r.close()
    finally:
        gs_oracle.set_threads(prev)
    for pl, rg, col in lists[1:]:
        assert np.array_equal(pl, lists[0][0]) and np.array_equal(rg, lists[0][1]) and np.array_equal(col, lists[0][2])


# ---------------------------------------------------------------------------------------------------------
# rotated cameras: pose convention, rotation equivariance, the roles of x and y, the guard band
# ---------------------------------------------------------------------------------------------------------
def _one_view_scene(c2w, fx, fy, h, w, means, cov, colors, opac, near=1.0, bg=(0.2, 0.3, 0.4)):
    """A one-view fp64 Scene (colours as degree-0 'harmonics', read back by view_args(use_sh=False))."""
    import torch

    from pf3plat_b200.synthetic import Scene
    t = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float64)
    K = np.array([[fx, 0, 0.5], [0, fy, 0.5], [0, 0, 1.0]])
    P = len(means)
    return Scene(t(c2w)[None], t(K)[None], t([near]), t([100.0]), (h, w), t(bg)[None], t(means), t(cov),
                 t(colors)[:, :, None], t(opac), torch.zeros(P, 3, dtype=torch.float64), torch.zeros(P, 4, dtype=torch.float64))


def _render(sc, dt=np.float64, **extra):
    from tests.util import view_args
    st, kw = view_args(sc, 0, use_sh=False)
    return OracleRender(st, dtype=dt, **kw, **extra), st


@pytest.mark.parametrize("dt", DT)
def test_pose_convention_end_to_end(dt):
    """c2w = yaw 90 + pitch 30 at c != 0, through make_view_batch (itself pinned to the reference's glue by
    camera_glue.npz): a Gaussian at c + d * forward lands on the image centre, + delta * right moves it right by
    fx_px * delta / d pixels, + delta * down moves it down by fy_px * delta / d."""
    from tests.util import posed_c2w
    c2w = posed_c2w(90.0, 30.0, 0.0)
    c = np.array([1.5, -0.7, 2.0])
    c2w[:3, 3] = c
    h, w, fx, fy = 64, 80, 0.8, 1.1
    d, delta = 6.0, 0.25
    R = c2w[:3, :3]
    means = np.stack([c + d * R[:, 2], c + d * R[:, 2] + delta * R[:, 0], c + d * R[:, 2] + delta * R[:, 1]])
    cov = np.repeat((0.02 ** 2 * np.eye(3))[None], 3, 0)
    r, _ = _render(_one_view_scene(c2w, fx, fy, h, w, means, cov, np.ones((3, 3)), np.full(3, 0.5)), dt)
    centre = np.array([(w - 1) / 2, (h - 1) / 2])
    assert (r.radii > 0).all()
    assert np.allclose(r.xy[0], centre, atol=1e-4)
    assert np.allclose(r.xy[1], centre + [fx * w * delta / d, 0], atol=1e-4)
    assert np.allclose(r.xy[2], centre + [0, fy * h * delta / d], atol=1e-4)
    assert np.allclose(r.depths, d, rtol=1e-6)


def _random_rotation(rng):
    q, _ = np.linalg.qr(rng.standard_normal((3, 3)))
    return q * np.sign(np.linalg.det(q))


def test_rotation_equivariance():
    """The same world rotation applied to the means, the covariances and the camera leaves the fp64 image (outside
    fragile pixels) and the radii unchanged -- for every view of a posed scene, Gaussians behind the camera, in the
    near cull and past the guard band included.  A view block read transposed anywhere breaks this."""
    import torch

    from pf3plat_b200.synthetic import Scene
    from tests.util import make_posed_scene, view_args
    sc = make_posed_scene(3000, 4, 64, 80, seed=21)
    sc = Scene(**{k: (v.double() if torch.is_tensor(v) else v) for k, v in sc.__dict__.items()})
    Q = torch.tensor(_random_rotation(np.random.default_rng(4)))
    ext = sc.extrinsics.clone()
    ext[:, :3, :3] = Q @ ext[:, :3, :3]
    ext[:, :3, 3] = ext[:, :3, 3] @ Q.T
    rot = Scene(**{**sc.__dict__, "extrinsics": ext, "means": sc.means @ Q.T, "covariances": Q @ sc.covariances @ Q.T})
    for v in range(4):
        a = OracleRender(*_args(view_args(sc, v, use_sh=False)), dtype=np.float64)
        b = OracleRender(*_args(view_args(rot, v, use_sh=False)), dtype=np.float64)
        frag = a.px_fragile | b.px_fragile
        assert frag.mean() < 0.05 and a.num_rendered > 1000
        assert np.abs(a.color - b.color).max(axis=0)[~frag].max() < 1e-9
        assert np.array_equal(a.radii, b.radii)


def _args(st_kw):
    st, kw = st_kw
    return (st,) + tuple(kw[k] for k in ("means3D", "opacities")) + (None, kw["colors_precomp"], None, None, kw["cov3D_precomp"])


@pytest.mark.parametrize("dt", DT)
def test_roll_by_90_degrees_rotates_the_image(dt):
    """Rolling the camera by 90 degrees about its axis, with H <-> W and fx <-> fy swapped, gives np.rot90 of the image:
    fixes which of tanfovx / tanfovy, limx / limy and W / H goes with which image axis.  Footprints are >= 5 px and
    opacities < 0.19, so no Gaussian reaches alpha 1/255 where the tile rectangle (not mirror-symmetric) cuts it off;
    widths are multiples of 16, so the tile grids map onto each other; some Gaussians sit past the guard band."""
    from tests.util import posed_c2w
    rng = np.random.default_rng(8)
    h, w, fx, fy = 64, 96, 0.7, 1.2            # tanfovx = 0.71, tanfovy = 0.42
    tx, ty = 0.5 / fx, 0.5 / fy
    n = 120
    z = rng.uniform(3, 9, n)
    rx = np.where(np.arange(n) % 6 == 0, rng.choice([-1, 1], n) * rng.uniform(1.4, 1.9, n), rng.uniform(-1, 1, n))
    ry = np.where(np.arange(n) % 6 == 1, rng.choice([-1, 1], n) * rng.uniform(1.4, 1.9, n), rng.uniform(-1, 1, n))
    cam = np.stack([rx * tx * z, ry * ty * z, z], -1)
    sig = rng.uniform(5, 12, n) * z / (fx * w) * np.where(np.abs(rx) > 1.3, 4, 1)
    A = rng.standard_normal((n, 3, 3)) * 0.3 + np.eye(3)
    cov = np.einsum("nij,nkj->nik", A, A) * (sig ** 2)[:, None, None]
    cols, opac = rng.uniform(0, 1, (n, 3)), rng.uniform(0.03, 0.19, n)
    c2w = posed_c2w(25.0, -15.0, 10.0)
    means = c2w[:3, 3] + cam @ c2w[:3, :3].T
    a, sa = _render(_one_view_scene(c2w, fx, fy, h, w, means, cov, cols, opac), dt)
    c2w_b = c2w.copy()
    c2w_b[:3, :3] = c2w[:3, :3] @ np.array([[0.0, -1, 0], [1, 0, 0], [0, 0, 1]])
    b, sb = _render(_one_view_scene(c2w_b, fy, fx, w, h, means, cov, cols, opac), dt)
    assert abs(sb.tanfovx - sa.tanfovy) < 1e-12 and abs(sb.tanfovy - sa.tanfovx) < 1e-12 and sa.tanfovx != sa.tanfovy
    rot = np.rot90(a.color, 1, axes=(1, 2))
    frag = np.rot90(a.px_fragile) | b.px_fragile
    assert b.color.shape == rot.shape and frag.mean() < 0.05
    assert np.abs(b.color - rot).max(axis=0)[~frag].max() < (1e-9 if dt == np.float64 else 2e-5)
    assert np.array_equal(a.radii, b.radii) and (a.radii > 0).sum() > 0.9 * n


@pytest.mark.parametrize("dt", DT)
def test_guard_band_clamp(dt):
    """A Gaussian at x/z = 2 limx (limx = 1.3 tanfovx): its 2D covariance is J Sigma J^T + 0.3 I with J taken at the
    CLAMPED position (t.x = limx t.z); in the backward, nothing reaches mean.x through J (the clamped axis), only through
    means2D -- while mean.y, inside the band, gets both."""
    tanfov, z = 0.5, 4.0
    st = simple_settings(48, 64, tanfov=tanfov, bg=(0.1, 0.2, 0.3))
    limx = 1.3 * tanfov
    mean = np.array([2 * limx * z, 0.3 * tanfov * z, z])
    L = np.array([[0.9, 0, 0], [0.4, 0.6, 0], [-0.3, 0.5, 0.7]])
    Sigma = L @ L.T * 1.5
    c6 = Sigma[np.triu_indices(3)][None]
    r = OracleRender(st, means3D=mean[None], opacities=np.array([0.8]), colors_precomp=np.array([[0.9, 0.4, 0.1]]),
                     cov3D_precomp=c6, dtype=dt)
    assert r.radii[0] > 0
    fx, fy = 64 / (2 * tanfov), 48 / (2 * tanfov)
    J = np.array([[fx / z, 0, -fx * limx * z / z ** 2], [0, fy / z, -fy * mean[1] / z ** 2]])
    cov2 = J @ Sigma @ J.T + 0.3 * np.eye(2)
    inv = np.linalg.inv(cov2)
    assert np.allclose(r.conic_opacity[0, :3], [inv[0, 0], inv[0, 1], inv[1, 1]], rtol=1e-5)
    g = r.backward(np.random.default_rng(0).standard_normal((3, 48, 64)))
    # identity view: dL/dmean.x = (through J: masked) + d ndc_x / d mean.x * dL/dmeans2D.x = (1 / tanfov) / z * ...
    gx_proj = (1 / tanfov) / z * g["means2D"][0, 0]
    gy_proj = (1 / tanfov) / z * g["means2D"][0, 1]
    assert abs(g["means2D"][0, 0]) > 1e-3
    assert np.isclose(g["means3D"][0, 0], gx_proj, rtol=1e-5, atol=1e-9)
    assert abs(g["means3D"][0, 1] - gy_proj) > 1e-2 * abs(g["means3D"][0, 1])
