"""Generates tests/golden/camera_glue.npz by running the REFERENCE's own render_cuda
(/root/reference/src/model/decoder/cuda_splatting.py:47-127, imported unmodified from the read-only tree) against a
RECORDING stand-in for `diff_gaussian_rasterization`: the stub rasterizer stores the GaussianRasterizationSettings it is
handed for every view (viewmatrix, projmatrix, campos, tanfovx, tanfovy -- everything lines 64-112 compute) and returns
blank images.  The fixture therefore pins pf3plat_b200.cameras.make_view_batch / gs_view_batch to the reference's own glue.
Also writes tests/golden/operator_calls.npz: the raw arguments of every operator call of the three call sites
(record_operator_calls).
Only runs in the build container (needs /root/reference).   Usage: python tests/golden/make_camera_golden.py"""
import importlib.util
import json
import os
import sys
import types
from typing import NamedTuple

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = "/root/reference"
RECORDED: list = []


class _Settings(NamedTuple):
    image_height: int
    image_width: int
    tanfovx: float
    tanfovy: float
    bg: torch.Tensor
    scale_modifier: float
    viewmatrix: torch.Tensor
    projmatrix: torch.Tensor
    sh_degree: int
    campos: torch.Tensor
    prefiltered: bool
    debug: bool


class _Recorder:
    def __init__(self, raster_settings):
        self.s = raster_settings

    def __call__(self, means3D, means2D, shs=None, colors_precomp=None, opacities=None, cov3D_precomp=None, **kw):
        s = self.s
        RECORDED.append(dict(viewmatrix=s.viewmatrix.detach().clone(), projmatrix=s.projmatrix.detach().clone(),
                             campos=s.campos.detach().clone(), tanfov=torch.tensor([float(s.tanfovx), float(s.tanfovy)]),
                             means=means3D.detach().clone(), cov6=cov3D_precomp.detach().clone(),
                             bg=s.bg.detach().clone().float(), opacities=opacities.detach().clone(),
                             colors=(torch.zeros(0) if colors_precomp is None else colors_precomp.detach().clone()),
                             shs=(torch.zeros(0) if shs is None else shs.detach().clone()),
                             ints=torch.tensor([s.image_height, s.image_width, s.sh_degree, int(s.prefiltered), int(s.debug)]),
                             scale_modifier=torch.tensor(float(s.scale_modifier)),
                             means2D_is_zero_leaf=torch.tensor(int(bool((means2D == 0).all()) and means2D.requires_grad))))
        return torch.zeros(3, s.image_height, s.image_width), torch.zeros(means3D.shape[0], dtype=torch.int32)


def load_reference_render_cuda():
    stub = types.ModuleType("diff_gaussian_rasterization")
    stub.GaussianRasterizationSettings = _Settings
    stub.GaussianRasterizer = _Recorder
    saved = sys.modules.get("diff_gaussian_rasterization")
    sys.modules["diff_gaussian_rasterization"] = stub
    try:
        for name in ("src", "src.model", "src.model.decoder", "src.model.encoder", "src.model.encoder.costvolume", "src.geometry"):
            m = types.ModuleType(name)
            m.__path__ = [os.path.join(REF_ROOT, *name.split("."))]
            sys.modules[name] = m
        path = os.path.join(REF_ROOT, "src/model/decoder/cuda_splatting.py")
        spec = importlib.util.spec_from_file_location("src.model.decoder.cuda_splatting", path)
        mod = importlib.util.module_from_spec(spec)
        sys.modules[spec.name] = mod
        spec.loader.exec_module(mod)
        return mod
    finally:
        if saved is not None:
            sys.modules["diff_gaussian_rasterization"] = saved
        else:
            del sys.modules["diff_gaussian_rasterization"]


def load_reference_decoder():
    """The reference's DecoderSplattingCUDA (/root/reference/src/model/decoder/decoder_splatting_cuda.py), on top of
    load_reference_render_cuda(); `src.dataset` (which pulls in every dataset class) is replaced by an empty stand-in --
    the decoder only reads dataset_cfg.background_color."""
    load_reference_render_cuda()
    ds = types.ModuleType("src.dataset")
    ds.DatasetCfg = type("DatasetCfg", (), {})
    sys.modules["src.dataset"] = ds
    for name, rel in (("src.model.types", "src/model/types.py"), ("src.model.decoder.decoder", "src/model/decoder/decoder.py"),
                      ("src.model.decoder.decoder_splatting_cuda", "src/model/decoder/decoder_splatting_cuda.py")):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF_ROOT, rel))
        mod = importlib.util.module_from_spec(spec)
        sys.modules[name] = mod
        spec.loader.exec_module(mod)
    return sys.modules["src.model.decoder.decoder_splatting_cuda"], sys.modules["src.model.types"]


DECODER_KEYS = ("viewmatrix", "projmatrix", "campos", "tanfov", "means", "cov6", "bg", "opacities", "colors", "shs", "ints")


def decoder_inputs(b=2, v=3, G=2):
    """The inputs run_reference_decoder hands DecoderSplattingCUDA.forward: b scenes of G Gaussians, v views each."""
    ext, intr, near, far = make_cameras(21, b * v)
    g = torch.Generator().manual_seed(22)
    means = torch.randn(b, G, 3, generator=g).abs() + 0.5
    a = torch.randn(b, G, 3, 3, generator=g)
    cov = a @ a.transpose(-1, -2)
    sh = torch.randn(b, G, 3, 25, generator=g)
    opac = torch.rand(b, G, generator=g)
    r4 = lambda t: t.reshape(b, v, *t.shape[1:])
    return dict(extrinsics=r4(ext), intrinsics=r4(intr), near=r4(near), far=r4(far), means=means, covariances=cov, sh=sh,
                opacities=opac)


def run_reference_decoder(b=2, v=3, G=2, depth_mode="depth"):
    """Inputs and the recorded operator calls of one DecoderSplattingCUDA.forward (colour pass, then depth pass)."""
    dec_mod, types_mod = load_reference_decoder()
    inputs = decoder_inputs(b, v, G)
    cfg = types.SimpleNamespace(background_color=[0.1, 0.2, 0.3])
    dec = dec_mod.DecoderSplattingCUDA(dec_mod.DecoderSplattingCUDACfg(name="splatting_cuda"), cfg)
    RECORDED.clear()
    i = inputs
    dec.forward(types_mod.Gaussians(i["means"], i["covariances"], i["sh"], i["opacities"]), i["extrinsics"],
                i["intrinsics"], i["near"], i["far"], (16, 24), depth_mode=depth_mode)
    rec = {k: [r[k] for r in RECORDED] for k in DECODER_KEYS}
    RECORDED.clear()
    return inputs, rec


def ortho_inputs():
    ext = make_cameras(31, 1)[0]
    return dict(extrinsics=ext, width=torch.tensor([2.5]), height=torch.tensor([1.75]), near=torch.tensor([0.0]),
                far=torch.tensor([7.0]), bg=torch.tensor([[0.3, 0.1, 0.2]]))


def make_cameras(seed, B):
    g = torch.Generator().manual_seed(seed)
    ext = torch.eye(4).repeat(B, 1, 1)
    ext[:, :3, :3] = torch.linalg.qr(torch.randn(B, 3, 3, generator=g))[0]
    ext[:, :3, 3] = torch.randn(B, 3, generator=g)
    intr = torch.eye(3).repeat(B, 1, 1)
    intr[:, 0, 0] = 0.6 + 0.6 * torch.rand(B, generator=g)
    intr[:, 1, 1] = 0.6 + 0.6 * torch.rand(B, generator=g)
    intr[:, 0, 2] = 0.5 + 0.03 * torch.randn(B, generator=g)
    intr[:, 1, 2] = 0.5 + 0.03 * torch.randn(B, generator=g)
    near = 0.3 + torch.rand(B, generator=g)
    far = 40 + 100 * torch.rand(B, generator=g)
    return ext, intr, near, far


def glue_inputs(B=9, G=2):
    """The cameras and Gaussians of main(): render_cuda gets them as they are, render_depth_cuda the same cameras with
    means.abs() + 0.5, render_cuda_orthographic only the first scene's Gaussians (with the camera of ortho_inputs())."""
    ext, intr, near, far = make_cameras(12, B)
    g = torch.Generator().manual_seed(13)
    means = torch.randn(B, G, 3, generator=g)
    a = torch.randn(B, G, 3, 3, generator=g)
    cov = a @ a.transpose(-1, -2)
    sh = torch.randn(B, G, 3, 25, generator=g)
    opac = torch.rand(B, G, generator=g)
    return ext, intr, near, far, means, cov, sh, opac


class _RawSettings(dict):
    """Stand-in for GaussianRasterizationSettings that keeps the keyword arguments exactly as they were passed."""

    def __init__(self, **kwargs):
        super().__init__(kwargs)


class _RawRecorder:
    """Stand-in for GaussianRasterizer that keeps its settings and the keyword arguments of every call as handed over."""

    def __init__(self, raster_settings):
        self.s = raster_settings

    def __call__(self, **kwargs):
        OPERATOR_CALLS.append((dict(self.s), kwargs))
        return (torch.zeros(3, self.s["image_height"], self.s["image_width"]),
                torch.zeros(kwargs["means3D"].shape[0], dtype=torch.int32))


OPERATOR_CALLS: list = []


def record_operator_calls():
    """Every operator call of the reference's three call sites (render_cuda, render_cuda_orthographic, and render_cuda
    again through render_depth_cuda) on a small synthetic scene, argument by argument: tensors as arrays (with
    requires_grad), Python scalars with their type.  tests/test_capi_cpu.py replays them against this repository's
    `diff_gaussian_rasterization`."""
    sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
    from pf3plat_b200.synthetic import make_scene
    mod = load_reference_render_cuda()
    mod.GaussianRasterizationSettings, mod.GaussianRasterizer = _RawSettings, _RawRecorder
    sc = make_scene(64, 2, 32, 32)
    rep = lambda t: t[None].expand(2, *t.shape)
    one = lambda t: t[:1]
    OPERATOR_CALLS.clear()
    mod.render_cuda(sc.extrinsics, sc.intrinsics, sc.near, sc.far, sc.image_shape, sc.background, rep(sc.means),
                    rep(sc.covariances), rep(sc.harmonics), rep(sc.opacities))
    mod.render_depth_cuda(sc.extrinsics, sc.intrinsics, sc.near, sc.far, sc.image_shape, rep(sc.means),
                          rep(sc.covariances), rep(sc.opacities), mode="disparity")
    mod.render_cuda_orthographic(one(sc.extrinsics), torch.tensor([2.0]), torch.tensor([2.0]), one(sc.near), one(sc.far),
                                 sc.image_shape, one(sc.background), one(rep(sc.means)), one(rep(sc.covariances)),
                                 one(rep(sc.harmonics)), one(rep(sc.opacities)))
    arrays, kinds = {}, {}
    for i, (settings, call) in enumerate(OPERATOR_CALLS):
        for part, args in (("settings", settings), ("call", call)):
            for name, v in args.items():
                key = f"c{i}.{part}.{name}"
                if isinstance(v, torch.Tensor):
                    arrays[key] = v.detach().numpy()
                    kinds[key] = "tensor_grad" if v.requires_grad else "tensor"
                elif v is None:
                    kinds[key] = "none"
                else:
                    arrays[key] = np.array(v)
                    kinds[key] = type(v).__name__
    arrays["kinds"] = np.array(json.dumps(kinds))
    OPERATOR_CALLS.clear()
    path = os.path.join(HERE, "operator_calls.npz")
    np.savez_compressed(path, **arrays)
    print(len(kinds), "arguments", os.path.getsize(path), "bytes")


def main():
    mod = load_reference_render_cuda()
    B = 9
    ext, intr, near, far, means, cov, sh, opac = glue_inputs(B)
    arrays = dict(extrinsics=ext.numpy(), intrinsics=intr.numpy(), near=near.numpy(), far=far.numpy(),
                  means=means.numpy(), covariances=cov.numpy())
    for tag, si in (("si", True), ("raw", False)):
        RECORDED.clear()
        mod.render_cuda(ext, intr, near, far, (16, 24), torch.zeros(B, 3), means, cov, sh, opac, scale_invariant=si)
        assert len(RECORDED) == B
        for k in ("viewmatrix", "projmatrix", "campos", "tanfov", "means", "cov6"):
            arrays[f"{tag}_{k}"] = torch.stack([r[k] for r in RECORDED]).numpy()
    # the depth renders: what render_depth_cuda (:226-269) hands the op in each of its modes (fake colours, bg, flags)
    for mode in ("depth", "disparity", "relative_disparity", "log"):
        RECORDED.clear()
        mod.render_depth_cuda(ext, intr, near, far, (16, 24), means.abs() + 0.5, cov, opac, mode=mode)
        assert len(RECORDED) == B
        for k in ("colors", "bg", "opacities", "ints", "scale_modifier", "means2D_is_zero_leaf"):
            arrays[f"depth_{mode}_{k}"] = torch.stack([r[k] for r in RECORDED]).numpy()
    # and the colour render's remaining arguments
    RECORDED.clear()
    mod.render_cuda(ext, intr, near, far, (16, 24), torch.rand(B, 3, generator=torch.Generator().manual_seed(14)), means, cov, sh, opac)
    for k in ("shs", "bg", "opacities", "ints", "scale_modifier", "means2D_is_zero_leaf"):
        arrays[f"color_{k}"] = torch.stack([r[k] for r in RECORDED]).numpy()
    arrays["sh"] = sh.numpy()
    arrays["opacities"] = opac.numpy()
    # the fake-orthographic render (render_cuda_orthographic, :130-220; batch of one, as its 0-dim/1-element tensor
    # tanfov arguments require): everything it hands the op
    for k, t in ortho_inputs().items():
        arrays[f"ortho_in_{k}"] = t.numpy()
    RECORDED.clear()
    oi = ortho_inputs()
    mod.render_cuda_orthographic(oi["extrinsics"], oi["width"], oi["height"], oi["near"], oi["far"], (16, 24), oi["bg"],
                                 means[:1], cov[:1], sh[:1], opac[:1])
    assert len(RECORDED) == 1
    for k in ("viewmatrix", "projmatrix", "campos", "tanfov", "means", "cov6", "shs", "bg", "opacities", "ints",
              "scale_modifier", "means2D_is_zero_leaf"):
        arrays[f"ortho_{k}"] = torch.stack([r[k] for r in RECORDED]).numpy()
    # the decoder on top (decoder_splatting_cuda.py:35-91): 2 scenes x 3 views, colour pass then depth pass
    inputs, rec = run_reference_decoder()
    for k, t in inputs.items():
        arrays[f"dec_in_{k}"] = t.numpy()
    for k, lst in rec.items():
        for half, sl in (("color", slice(0, 6)), ("depth", slice(6, 12))):
            arrays[f"dec_{half}_{k}"] = torch.stack(lst[sl]).numpy()
    path = os.path.join(HERE, "camera_glue.npz")
    np.savez_compressed(path, **arrays)
    print({k: v.shape for k, v in arrays.items()}, os.path.getsize(path), "bytes")
    record_operator_calls()


if __name__ == "__main__":
    main()
