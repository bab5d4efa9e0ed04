"""Shared helpers for the parity tests: turn a synthetic Scene into the exact per-view arguments the
reference call site hands to the rasterizer (/root/reference/src/model/decoder/cuda_splatting.py:64-124)."""
from __future__ import annotations

import math

import numpy as np
import torch

from oracle.gs_oracle import OracleRender, OracleSettings
from pf3plat_b200.cameras import make_view_batch
from pf3plat_b200.synthetic import Scene, make_target, quat_to_rotmat


def view_args(scene, v: int, use_sh: bool = True):
    """Returns (OracleSettings, kwargs) for view v, following render_cuda line by line."""
    vb = make_view_batch(scene.extrinsics, scene.intrinsics, scene.near, scene.far, scale_invariant=True)
    scale = vb.scale[v]
    h, w = scene.image_shape
    means = scene.means * scale
    cov = scene.covariances * scale * scale
    row, col = torch.triu_indices(3, 3)
    cov6 = cov[:, row, col]
    d_sh = scene.harmonics.shape[-1]
    shs = scene.harmonics.permute(0, 2, 1).contiguous()  # (P, d_sh, 3)
    st = OracleSettings(
        image_height=h, image_width=w, tanfovx=float(vb.tanfov[v, 0]), tanfovy=float(vb.tanfov[v, 1]),
        bg=scene.background[v].numpy(), scale_modifier=1.0, viewmatrix=vb.viewmatrix[v].numpy(),
        projmatrix=vb.projmatrix[v].numpy(), sh_degree=math.isqrt(d_sh) - 1, campos=vb.campos[v].numpy())
    kw = dict(means3D=means.numpy(), opacities=scene.opacities.numpy(), cov3D_precomp=cov6.numpy())
    if use_sh:
        kw["shs"] = shs.numpy()
    else:
        kw["colors_precomp"] = shs[:, 0, :].contiguous().numpy()
    return st, kw


def oracle_view(scene, v, use_sh=True, dtype=np.float32, **extra):
    st, kw = view_args(scene, v, use_sh)
    return OracleRender(st, dtype=dtype, **kw, **extra)


def simple_settings(h=64, w=64, tanfov=0.5, bg=(0.0, 0.0, 0.0), near=1.0, far=100.0, sh_degree=0):
    """Identity camera looking down +z, built the way get_projection_matrix does (cuda_splatting.py:17-44)."""
    proj = np.zeros((4, 4), np.float64)
    proj[0, 0] = 1.0 / tanfov
    proj[1, 1] = 1.0 / tanfov
    proj[3, 2] = 1.0
    proj[2, 2] = far / (far - near)
    proj[2, 3] = -(far * near) / (far - near)
    view = np.eye(4)
    full = view.T @ proj.T
    return OracleSettings(image_height=h, image_width=w, tanfovx=tanfov, tanfovy=tanfov, bg=np.array(bg, np.float64),
                          scale_modifier=1.0, viewmatrix=view.T.copy(), projmatrix=full, sh_degree=sh_degree,
                          campos=np.zeros(3))


# ---------------------------------------------------------------------------------------------------------
# parity criteria (BASELINE.json north_star: 1e-4 abs RGB, 1e-3 rel gradient)
# ---------------------------------------------------------------------------------------------------------
RGB_TOL = 1e-4          # non-fragile pixels
FRAGILE_RGB_TOL = 5e-3  # pixels where the oracle saw a discontinuous decision within 1e-4 of its threshold: ONE flipped
                        # alpha >= 1/255 decision moves a channel by at most alpha*T*c <= 1/255 = 3.9e-3
GRAD_RTOL = 1e-3        # element-wise: |a-b| <= GRAD_RTOL*|b| + GRAD_RTOL*rms(b), per tensor and per SH band
# Gaussians that contribute to a fragile pixel: a decision flipped there (alpha >= 1/255 or T < 1e-4 taken the other way
# round) changes T for every Gaussian behind it at that pixel by <= 0.4 % -- and for the flipped Gaussian itself it adds
# or removes that pixel's whole term of its gradient.  They are held to the same element-wise form with 1e-2, except for
# a bounded handful (<= 1e-4 of them + 2: the flipped Gaussians themselves), which must stay below 1e-1.  Measured on C3
# (500k Gaussians, 2 views): 180k affected, worst ratio 3.0e-2.
GRAD_RTOL_AFFECTED = 1e-2
GRAD_RTOL_FLIPPED = 1e-1


def image_report(gpu_color, orc) -> dict:
    """The four numbers SURVEY.md section 7 asks for, of one view against the oracle."""
    g = gpu_color.detach().cpu().numpy() if torch.is_tensor(gpu_color) else np.asarray(gpu_color)
    err = np.abs(g.astype(np.float64) - orc.color.astype(np.float64)).max(axis=0)
    frag = orc.px_fragile
    return {
        "pixels": int(err.size),
        "pixels_over_1e-4": int((err > RGB_TOL).sum()),
        "nonfragile_pixels_over_1e-4": int((err[~frag] > RGB_TOL).sum()),
        "fragile_frac": float(frag.mean()),
        "max_err_nonfragile": float(err[~frag].max()) if (~frag).any() else 0.0,
        "max_err_fragile": float(err[frag].max()) if frag.any() else 0.0,
    }


def check_image_strict(gpu_color, orc, max_fragile_frac: float, label: str = "") -> dict:
    rep = image_report(gpu_color, orc)
    print(f"[parity] {label} {rep}")
    if rep["max_err_nonfragile"] > RGB_TOL:   # say where, so that the pixel can be examined on the CPU
        g = gpu_color.detach().cpu().numpy() if torch.is_tensor(gpu_color) else np.asarray(gpu_color)
        err = np.abs(g.astype(np.float64) - orc.color.astype(np.float64)).max(axis=0) * ~orc.px_fragile
        y, x = np.unravel_index(np.argmax(err), err.shape)
        print(f"[parity] {label} worst non-fragile pixel (y={y}, x={x}): ours {g[:, y, x]}, oracle {orc.color[:, y, x]}, "
              f"final_T {orc.final_T[y, x]}, n_contrib {orc.n_contrib[y, x]}")
    assert rep["fragile_frac"] <= max_fragile_frac, rep
    assert rep["max_err_nonfragile"] <= RGB_TOL, rep
    assert rep["max_err_fragile"] <= FRAGILE_RGB_TOL, rep
    return rep


def affected_gaussians(orc, pixel_mask: np.ndarray) -> np.ndarray:
    """bool[P]: Gaussians that can contribute (alpha >= ~1/255) to a pixel of `pixel_mask` -- a flipped decision at such a
    pixel changes T for every Gaussian behind it there, so their gradients carry the fragile pixel's slack."""
    P = orc.P
    hit = np.zeros(P, bool)
    ys, xs = np.nonzero(pixel_mask)
    if len(ys) == 0:
        return hit
    xy, co, pl, rg = orc.xy.astype(np.float64), orc.conic_opacity.astype(np.float64), orc.point_list, orc.ranges
    gx = (orc.W + 15) // 16
    tiles = (ys // 16) * gx + (xs // 16)
    for t in np.unique(tiles):
        s, e = rg[t]
        ids = pl[s:e]
        if len(ids) == 0:
            continue
        sel = tiles == t
        px, py = xs[sel][None, :].astype(np.float64), ys[sel][None, :].astype(np.float64)
        dx, dy = xy[ids, 0:1] - px, xy[ids, 1:2] - py
        power = -0.5 * (co[ids, 0:1] * dx * dx + co[ids, 2:3] * dy * dy) - co[ids, 1:2] * dx * dy
        alpha = co[ids, 3:4] * np.exp(np.minimum(power, 0.0))
        touch = ((power <= 1e-6) & (alpha >= (1 / 255) * 0.99)).any(axis=1)
        hit[ids[touch]] = True
    return hit


def grad_report(name, a, b, affected=None, bands=None) -> dict:
    """Element-wise gradient criterion.  a: ours, b: oracle, both [P, ...]; affected: bool[P] or None; bands: list of
    (label, slice over axis 1) to apply the criterion per SH band (rms taken per band)."""
    a = a.detach().cpu().numpy().astype(np.float64) if torch.is_tensor(a) else np.asarray(a, np.float64)
    b = np.asarray(b, np.float64).reshape(a.shape)
    P = a.shape[0]
    aff = np.zeros(P, bool) if affected is None else affected
    out = {"name": name, "elements": int(a.size), "affected_gaussians": int(aff.sum())}
    worst_ok, worst_aff, bad, bad_aff, over_strict_aff = 0.0, 0.0, 0, 0, 0
    parts = [("all", slice(None))] if bands is None else bands
    for label, sl in parts:
        aa, bb = (a, b) if bands is None else (a[:, sl], b[:, sl])
        rms = float(np.sqrt(np.mean(bb * bb)))
        ratio = np.abs(aa - bb) / (np.abs(bb) + rms + 1e-300)   # criterion: ratio <= rtol
        r2 = ratio.reshape(P, -1).max(axis=1) if ratio.size else np.zeros(P)
        worst_ok = max(worst_ok, float(r2[~aff].max()) if (~aff).any() else 0.0)
        worst_aff = max(worst_aff, float(r2[aff].max()) if aff.any() else 0.0)
        bad += int((r2[~aff] > GRAD_RTOL).sum())
        bad_aff += int((r2[aff] > GRAD_RTOL_AFFECTED).sum())
        over_strict_aff += int((r2[aff] > GRAD_RTOL).sum())
        out[f"rms_{label}"] = rms
    out.update({"worst_ratio_unaffected": worst_ok, "worst_ratio_affected": worst_aff, "gaussians_over_tol": bad,
                "affected_over_1e-3": over_strict_aff, "affected_over_1e-2": bad_aff})
    return out


SH_BANDS = [("band0", slice(0, 1)), ("band1", slice(1, 4)), ("band2", slice(4, 9)), ("band3", slice(9, 16))]


def check_grad(name, a, b, affected=None, bands=None) -> dict:
    rep = grad_report(name, a, b, affected, bands)
    print(f"[parity] grad {rep}")
    assert rep["gaussians_over_tol"] == 0, rep
    assert rep["affected_over_1e-2"] <= 1e-4 * rep["affected_gaussians"] + 2, rep
    assert rep["worst_ratio_affected"] <= GRAD_RTOL_FLIPPED, rep
    return rep


# ---------------------------------------------------------------------------------------------------------
# posed scenes: rotated cameras around the cloud, fx != fy, near != 1, non-zero background, and labelled populations
# behind the camera, inside the near cull, past the guard band and far off-axis
# ---------------------------------------------------------------------------------------------------------
POSED_TANFOV = (0.585, 0.45)     # tanfovx / tanfovy = 1.3
# (yaw, pitch, roll) in degrees and near of each view; view 1 is rolled by exactly 90 degrees.  Forward axes are >= 20
# degrees apart (checked below), near in {0.5, 1, 2} gives the in-kernel view_scale 2, 1 and 0.5.
_POSES = [(0, 8, 0), (38, -14, 90), (-35, 22, -20), (75, 5, 35), (-70, -25, 60), (150, 15, -45), (-140, -10, 10),
          (110, 40, -75)]
_NEARS = [1.0, 0.5, 2.0, 1.0, 0.5, 2.0, 1.0, 2.0]
_CAM_DIST, _CLOUD_RADIUS = 8.0, 2.8
_MARGIN = 1e-3                   # relative distance every Gaussian keeps from z = near_cull_z and from |x/z| = limx


def _rot(axis, deg):
    if deg % 360 == 90:          # exact, so that the 90-degree roll really swaps the image axes
        c, s = 0.0, 1.0
    else:
        c, s = math.cos(math.radians(deg)), math.sin(math.radians(deg))
    i, j = [(1, 2), (2, 0), (0, 1)][axis]
    R = np.eye(3)
    R[i, i], R[i, j], R[j, i], R[j, j] = c, -s, s, c
    return R


def posed_c2w(yaw, pitch, roll, dist=_CAM_DIST):
    """Camera-to-world (OpenCV axes: x right, y down, z forward) looking at the origin from `dist` away."""
    R = _rot(1, yaw) @ _rot(0, pitch) @ _rot(2, roll)
    T = np.eye(4)
    T[:3, :3] = R
    T[:3, 3] = -dist * R[:, 2]
    return T


def camera_space(scene, v):
    """fp64 camera-space positions of every Gaussian in view v, in the 1/near-rescaled units the kernels work in
    (the same matrices `view_args` hands the oracle), and that view's (tanfovx, tanfovy)."""
    vb = make_view_batch(scene.extrinsics, scene.intrinsics, scene.near, scene.far, scale_invariant=True)
    view = vb.viewmatrix[v].double().numpy()
    m = scene.means.double().numpy() * float(vb.scale[v])
    return m @ view[:3, :3] + view[3, :3], (float(vb.tanfov[v, 0]), float(vb.tanfov[v, 1]))


def posed_regimes(scene, v, near_cull_z=0.2, guard_band=1.3):
    """bool[P] masks of the regimes of view v, from the camera matrices: behind the camera, inside the near cull,
    past the guard band in x / y (among the Gaussians that survive the cull), far off-axis (|x/z| or |y/z| >= 1e3)."""
    t, (tx, ty) = camera_space(scene, v)
    z = t[:, 2]
    live = z > near_cull_z
    with np.errstate(divide="ignore", invalid="ignore"):
        rx, ry = np.abs(t[:, 0] / z), np.abs(t[:, 1] / z)
    return {"behind": z < 0, "near_cull": (z >= 0) & ~live, "live": live,
            "x_out": live & (rx > guard_band * tx), "y_out": live & (ry > guard_band * ty),
            "off_axis": live & ((rx >= 1e3) | (ry >= 1e3)), "z": z, "ratio_x": rx / tx, "ratio_y": ry / ty}


def make_posed_scene(P: int, views: int, h: int, w: int, seed: int = 0, scenes: int = 1, d_sh: int = 25):
    """A cloud seen from cameras placed around it and looking at it, the way PF3plat renders target views at poses
    rotated away from the context views.  Returns a `Scene` (a list of `scenes` of them if scenes > 1, each with its
    own cloud and its own cameras).

    Cameras: distinct yaw / pitch / roll (view 1 rolled by exactly 90 degrees), tanfovx / tanfovy = 1.3, near from
    {0.5, 1, 2}, a non-zero background per view.  Gaussians: the bulk, a ball around the origin, plus per view,
    planted in that view's rescaled camera space: behind the camera (z < 0); inside the near cull (0 < z < 0.2); just
    past it (0.25 <= z <= 1) with large footprints; past the guard band (1.3 < |x/z| / tanfov < 4) with footprints that
    still reach the image; far off-axis (|x/z| >= 1e3).  Bulk Gaussians with zero, rank-1 and rank-2 covariances.
    Every Gaussian keeps 1e-3 relative distance from z = 0.2 and from |x/z| = 1.3 tanfov in EVERY view (resampled
    otherwise), so no test can depend on which side of those discontinuities an fp32 rounding puts it."""
    if scenes > 1:
        return [_posed_scene(P, views, h, w, seed + 1000 * k, d_sh, 13.0 * k) for k in range(scenes)]
    return _posed_scene(P, views, h, w, seed, d_sh, 0.0)


def _posed_scene(P, views, h, w, seed, d_sh, yaw_offset):
    assert 1 <= views <= len(_POSES)
    rng = np.random.default_rng(seed)
    tx, ty = POSED_TANFOV
    c2w = np.stack([posed_c2w(yaw + yaw_offset, pitch, roll) for yaw, pitch, roll in _POSES[:views]])
    fwd = c2w[:, :3, 2]
    cosang = np.clip(fwd @ fwd.T, -1, 1)[~np.eye(views, dtype=bool)]
    assert views == 1 or np.degrees(np.arccos(cosang)).min() >= 20.0
    near = np.array(_NEARS[:views])
    K = np.eye(3)
    K[0, 0], K[1, 1], K[0, 2], K[1, 2] = 0.5 / tx, 0.5 / ty, 0.5, 0.5
    fx_px, fy_px = w / (2 * tx), h / (2 * ty)

    pos, sc, op = [], [], []   # world positions, world-unit scales, opacities

    def plant(n, z, rx, ry, sigma_px, opacity=(0.05, 0.7)):
        """n Gaussians in view v's rescaled camera space at depth z, x/z = rx * tanfovx, y/z = ry * tanfovy,
        isotropic-ish with a footprint of about sigma_px pixels."""
        cam = np.stack([rx * tx * z, ry * ty * z, z], -1) * near[v]
        pos.append(c2w[v, :3, 3] + cam @ c2w[v, :3, :3].T)
        sigma = sigma_px * np.abs(z) / fx_px * near[v]
        sc.append(sigma[:, None] * np.exp(rng.uniform(-0.3, 0.3, (n, 3))))
        op.append(rng.uniform(*opacity, n))

    cnt = lambda frac, lo: max(lo, int(round(frac * P)))
    for v in range(views):
        U = lambda a, b, n: rng.uniform(a, b, n)
        sgn = lambda n: rng.choice([-1.0, 1.0], n)
        n = cnt(4e-3, 4)                                                        # behind the camera
        plant(n, -np.exp(U(np.log(0.3), np.log(6.0), n)), U(-1, 1, n), U(-1, 1, n), U(1, 6, n))
        n = cnt(4e-3, 4)                                                        # inside the near cull
        plant(n, U(0.02, 0.18, n), U(-0.9, 0.9, n), U(-0.9, 0.9, n), U(2, 10, n))
        n = cnt(1.5e-3, 3)                                                      # just past the cull, large footprints
        plant(n, U(0.25, 1.0, n), U(-0.9, 0.9, n), U(-0.9, 0.9, n), U(3, 15, n), (0.05, 0.35))
        n = cnt(1e-3, 6)                                                        # past the guard band
        r_out, r_in = U(1.35, 3.0, n), U(-0.9, 0.9, n)
        axis = np.arange(n) % 3                                                 # x, y or both out
        rx = np.where(axis != 1, sgn(n) * r_out, r_in)
        ry = np.where(axis == 0, U(-0.9, 0.9, n), sgn(n) * np.where(axis == 2, U(1.35, 3.0, n), r_out))
        off = np.maximum((np.abs(rx) - 1) * w / 2, (np.abs(ry) - 1) * h / 2)    # pixels beyond the image edge
        plant(n, U(1.0, 4.0, n), rx, ry, off / 2.2 + 4, (0.05, 0.35))
        n = cnt(1.5e-3, 3)                                                      # far off-axis
        ratio = np.exp(U(np.log(1e3), np.log(1e5), n))
        big_x = np.arange(n) % 2 == 0
        plant(n, U(0.3, 3.0, n), np.where(big_x, sgn(n) * ratio, U(-1, 1, n)), np.where(big_x, U(-1, 1, n), sgn(n) * ratio),
              U(0.5, 3, n))
    planted = np.concatenate(pos)
    planted_sc = np.concatenate(sc)
    planted_op = np.concatenate(op)

    def bulk(n):
        d = rng.standard_normal((n, 3))
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        p = d * _CLOUD_RADIUS * rng.uniform(0, 1, (n, 1)) ** (1 / 3)
        mult = 0.1 * (1.0 / (K[0, 0] * w) + 1.0 / (K[1, 1] * h))
        return p, _CAM_DIST * mult * np.exp(rng.uniform(np.log(0.3), np.log(6.0), (n, 3)))

    def keep(p):
        ok = np.ones(len(p), bool)
        for v in range(views):
            R, c = c2w[v, :3, :3], c2w[v, :3, 3]
            t = (p - c) @ R / near[v]
            z = t[:, 2]
            ok &= np.abs(z - 0.2) > _MARGIN * 0.2
            live = z > 0.2
            for k, tf in ((0, tx), (1, ty)):
                r = np.abs(t[:, k] / np.where(live, z, 1.0))
                ok &= ~live | (np.abs(r - 1.3 * tf) > _MARGIN * 1.3 * tf)
        return ok

    ok = keep(planted)
    planted, planted_sc, planted_op = planted[ok], planted_sc[ok], planted_op[ok]
    nb = max(P - len(planted), 1)
    bp, bs = bulk(nb)
    while (~keep(bp)).any():
        bad = ~keep(bp)
        bp[bad], bs[bad] = bulk(int(bad.sum()))
    # degenerate covariances among the bulk: zero, rank 1, rank 2
    nd = min(cnt(5e-3, 3), nb // 3)
    bs[:nd] = 0.0
    bs[nd:2 * nd, 1:] = 0.0
    bs[2 * nd:3 * nd, 2] = 0.0
    means = np.concatenate([planted, bp])
    scales = np.concatenate([planted_sc, bs])
    Pn = len(means)
    q = rng.standard_normal((Pn, 4))
    q /= np.linalg.norm(q, axis=1, keepdims=True)
    qt = torch.tensor(q, dtype=torch.float64)
    R = quat_to_rotmat(qt)
    s = torch.tensor(scales, dtype=torch.float64)
    cov = R @ torch.diag_embed(s * s) @ R.transpose(-1, -2)
    cov = 0.5 * (cov + cov.transpose(-1, -2))
    opac = np.concatenate([planted_op, rng.uniform(0.05, 0.7, len(bp))])
    mask = np.ones(d_sh)
    for deg in range(1, math.isqrt(d_sh)):
        mask[deg * deg:(deg + 1) * (deg + 1)] = 0.1 * 0.25 ** deg
    mask[16:] = 0.0
    sh = rng.standard_normal((Pn, 3, d_sh)) * mask
    f = lambda a: torch.as_tensor(np.asarray(a), dtype=torch.float32).contiguous()
    return Scene(f(c2w), f(np.repeat(K[None], views, 0)), f(near), f(np.full(views, 100.0)), (h, w),
                 f(rng.uniform(0.1, 0.9, (views, 3))), f(means), cov.float().contiguous(), f(sh), f(opac), f(scales),
                 qt.float().contiguous())


# ---------------------------------------------------------------------------------------------------------
# GPU forward + backward of a whole Scene against the oracle, view by view
# ---------------------------------------------------------------------------------------------------------
def gpu_device():
    assert torch.cuda.is_available(), "GPU test needs CUDA"
    return torch.device("cuda:0")


def render_scene(sc, dev, with_depth=False, requires_grad=False):
    """All views of `sc` through the batched entry (render_views: the 1/near rescale is applied inside the kernels)."""
    from pf3plat_b200.render import render_views
    d = sc.to(dev)
    leaves = {"means": d.means[None].clone(), "cov": d.covariances[None].clone(), "sh": d.harmonics[None].clone(),
              "opac": d.opacities[None].clone()}
    if requires_grad:
        for t in leaves.values():
            t.requires_grad_(True)
    out = render_views(d.extrinsics, d.intrinsics, d.near, d.far, d.image_shape, d.background, leaves["means"],
                       leaves["cov"], leaves["sh"], leaves["opac"], with_depth=with_depth)
    return out, leaves


def cov6_of(G):
    G = G.detach().cpu().numpy() if torch.is_tensor(G) else np.asarray(G)
    return np.stack([G[:, 0, 0], G[:, 0, 1], G[:, 0, 2], G[:, 1, 1], G[:, 1, 2], G[:, 2, 2]], -1)


def view_scales(sc) -> np.ndarray:
    """Per view, the 1/near rescale view_args applies to means (and its square to covariances) before the oracle sees
    them: the oracle's gradients are with respect to the rescaled inputs."""
    return make_view_batch(sc.extrinsics, sc.intrinsics, sc.near, sc.far).scale.double().numpy()


def fwd_bwd_vs_oracle(sc, views, max_fragile_frac, label, d_sh=None, with_depth=False, check_radii=False):
    """Renders `views` views of `sc` on the GPU, MSE to a random target (plus a small depth term if with_depth), and
    holds colour per view, optionally radii and the depth channel, and dL/d{means, opacities, SH per band, cov6} to the
    oracle.  Returns the per-view oracle renders' summary and the GPU gradients."""
    dev = gpu_device()
    h, w = sc.image_shape
    d_sh = sc.harmonics.shape[-1] if d_sh is None else d_sh
    out, leaves = render_scene(sc, dev, with_depth=with_depth, requires_grad=True)
    color, depth = out if with_depth else (out, None)
    target = make_target(views, h, w).to(dev)
    wd = 1e-3
    loss = ((color - target) ** 2).mean()
    if with_depth:
        loss = loss + wd * depth.mean()
    loss.backward()
    radii = None
    if check_radii:
        radii = _radii(sc, dev)
    s = view_scales(sc)
    P = sc.means.shape[0]
    gm = np.zeros((P, 3)); go = np.zeros(P); gs = np.zeros((P, d_sh, 3)); gc = np.zeros((P, 6))
    affected = np.zeros(P, bool)
    orcs = []
    for v in range(views):
        orc = oracle_view(sc, v, with_depth=with_depth)
        check_image_strict(color[v], orc, max_fragile_frac, f"{label} view {v}")
        if check_radii:
            r = radii[v].cpu().numpy()
            ok = (r == orc.radii) | orc.geom_fragile
            assert ok.all(), f"{label} view {v}: {(~ok).sum()} radii differ on non-fragile Gaussians"
        if with_depth:
            derr = np.abs(depth[v].detach().cpu().numpy().astype(np.float64) - orc.depth)
            rel = derr / np.maximum(np.abs(orc.depth), 1.0)
            frag = orc.px_fragile
            print(f"[parity] {label} view {v} depth: max rel err non-fragile {rel[~frag].max():.3e}")
            assert rel[~frag].max() <= 1e-4
        # gradients are compared on the oracle's own image (dL/dC from the oracle's colours), like the small tests
        dL = (2 * (orc.color - target[v].cpu().numpy()) / target.numel()).astype(np.float32)
        dLd = np.full((h, w), wd / (views * h * w), np.float32) if with_depth else None
        g = orc.backward(dL, dLd)
        # the oracle differentiates with respect to the rescaled mean s*m and covariance s^2*Sigma
        gm += s[v] * g["means3D"]; go += g["opacities"][:, 0]; gs += g["shs"]; gc += s[v] ** 2 * g["cov3D_precomp"]
        affected |= affected_gaussians(orc, orc.px_fragile) | orc.geom_fragile
        orcs.append({"radii": orc.radii, "geom_fragile": orc.geom_fragile, "fragile_frac": float(orc.px_fragile.mean())})
        orc.close()
    print(f"[parity] {label}: {int(affected.sum())} of {P} Gaussians contribute to a fragile pixel")
    check_grad(f"{label} dL/dmeans3D", leaves["means"].grad[0], gm, affected)
    check_grad(f"{label} dL/dopacities", leaves["opac"].grad[0].reshape(P, 1), go.reshape(P, 1), affected)
    gsh = leaves["sh"].grad[0].permute(0, 2, 1)          # (P, d_sh, 3)
    check_grad(f"{label} dL/dshs", gsh, gs, affected, bands=[b for b in SH_BANDS if b[1].start < d_sh])
    if d_sh > 16:   # bands the evaluator never reads
        assert float(gsh[:, 16:].abs().max()) == 0.0 and np.abs(gs[:, 16:]).max() == 0.0
    check_grad(f"{label} dL/dcov3D", cov6_of(leaves["cov"].grad[0]), gc, affected)
    return orcs, {k: t.grad[0] for k, t in leaves.items()}


def _radii(sc, dev):
    """Radii per view from the batched operator, configured as render_views configures it."""
    from pf3plat_b200.rasterizer import BatchSettings, rasterize_batch
    d = sc.to(dev)
    vb = make_view_batch(d.extrinsics, d.intrinsics, d.near, d.far)
    h, w = sc.image_shape
    bs = BatchSettings(image_height=h, image_width=w, viewmatrix=vb.viewmatrix, projmatrix=vb.projmatrix,
                       campos=vb.campos, bg=d.background, sh_degree=math.isqrt(d.harmonics.shape[-1]) - 1,
                       tanfov=vb.tanfov, view_scale=vb.scale)
    with torch.no_grad():
        return rasterize_batch(bs, d.means[None], d.opacities[None], shs=d.harmonics.permute(0, 2, 1).contiguous()[None],
                               cov3D_precomp=torch.as_tensor(cov6_of(sc.covariances), device=dev)[None])[1]
