"""Generates tests/golden/adapter_*.npz by running the REFERENCE's own GaussianAdapter
(/root/reference/src/model/encoder/common/gaussian_adapter.py, imported unmodified from the read-only tree) on small
seeded inputs, in its native fp32, and recording its outputs and autograd gradients.

Only runs in the build container (needs /root/reference).  Two third-party imports of that module are absent here and
are stubbed for the import:
  * e3nn.o3.matrix_to_angles / wigner_D (used by misc/sh_rotation.py:26-29): the stub hands the rotation matrices
    through and returns the Wigner-D matrices of pf3plat_b200.sh_rotation -- so the reference's own rotate_sh code
    (determinant guard, per-degree einsum, concatenation) runs, with the D matrices as data.  Each fixture stores the
    block-diagonal D it used.
Usage:  python tests/golden/make_adapter_golden.py
"""
import importlib.util
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from pf3plat_b200.sh_rotation import rotations_are_proper, sh_rotation_blocks, wigner_d_from_matrix  # noqa: E402

REF_ROOT = "/root/reference"


def load_reference_adapter():
    """Returns the reference module src.model.encoder.common.gaussian_adapter (package __init__ files, which pull in
    the whole encoder, are bypassed with empty namespace packages)."""
    o3 = types.ModuleType("e3nn.o3")
    o3.matrix_to_angles = lambda rot: (rot, None, None)
    o3.wigner_D = lambda degree, alpha, beta, gamma: wigner_d_from_matrix(degree, alpha)
    e3nn = types.ModuleType("e3nn")
    e3nn.o3 = o3
    sys.modules.setdefault("e3nn", e3nn)
    sys.modules.setdefault("e3nn.o3", o3)
    for name in ("src", "src.model", "src.model.encoder", "src.model.encoder.common", "src.geometry", "src.misc"):
        m = types.ModuleType(name)
        m.__path__ = [os.path.join(REF_ROOT, *name.split("."))]
        sys.modules[name] = m
    path = os.path.join(REF_ROOT, "src/model/encoder/common/gaussian_adapter.py")
    spec = importlib.util.spec_from_file_location("src.model.encoder.common.gaussian_adapter", path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[spec.name] = mod
    spec.loader.exec_module(mod)
    return mod


def random_pose(g, n, proper=True):
    q = torch.randn(n, 4, generator=g)
    q = q / q.norm(dim=-1, keepdim=True)
    r, x, y, z = q.unbind(-1)
    rot = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - r * z), 2 * (x * z + r * y),
                       2 * (x * y + r * z), 1 - 2 * (x * x + z * z), 2 * (y * z - r * x),
                       2 * (x * z - r * y), 2 * (y * z + r * x), 1 - 2 * (x * x + y * y)], -1).reshape(n, 3, 3)
    if not proper:
        rot = rot * 1.05  # determinant 1.16: the reference then rotates the harmonics by the identity
    ext = torch.eye(4).repeat(n, 1, 1)
    ext[:, :3, :3] = rot
    ext[:, :3, 3] = 0.3 * torch.randn(n, 3, generator=g)
    return ext


def make_inputs(seed, b, v, h, w, sh_degree, proper=True, srf=1, spp=1):
    """Shapes of the adapter call at /root/reference/src/model/encoder/encoder_costvolume.py:529-540."""
    g = torch.Generator().manual_seed(seed)
    d_in = 7 + 3 * (sh_degree + 1) ** 2
    r = h * w
    ext = random_pose(g, b * v, proper).reshape(b, v, 1, 1, 1, 4, 4)
    intr = torch.eye(3).repeat(b, v, 1, 1)
    intr[..., 0, 0] = 0.8 + 0.2 * torch.rand(b, v, generator=g)
    intr[..., 1, 1] = 0.8 + 0.2 * torch.rand(b, v, generator=g)
    intr[..., 0, 2] = 0.5 + 0.02 * torch.randn(b, v, generator=g)
    intr[..., 1, 2] = 0.5 + 0.02 * torch.randn(b, v, generator=g)
    intr = intr.reshape(b, v, 1, 1, 1, 3, 3)
    ys, xs = torch.meshgrid((torch.arange(h) + 0.5) / h, (torch.arange(w) + 0.5) / w, indexing="ij")
    xy = torch.stack([xs, ys], -1).reshape(1, 1, r, 1, 1, 2)
    coords = xy + (torch.rand(b, v, r, srf, 1, 2, generator=g) - 0.5) / torch.tensor([w, h])
    depths = 1.0 + 9.0 * torch.rand(b, v, r, 1, 1, generator=g)
    opac = torch.rand(b, v, r, srf, spp, generator=g)
    raw = torch.randn(b, v, r, srf, 1, d_in, generator=g)
    return dict(extrinsics=ext, intrinsics=intr, coordinates=coords, depths=depths, opacities=opac, raw_gaussians=raw)


def make_weights(seed, shapes):
    """Weights w_k of the loss sum_k <w_k, out_k> whose gradients the fixture records, for outputs of the given shapes."""
    g = torch.Generator().manual_seed(100 + seed)
    return {k: torch.randn(s, generator=g) for k, s in shapes.items()}


def sh_rotation_used(extrinsics, b, v, sh_degree):
    """The block-diagonal Wigner-D matrices the e3nn stub hands the reference's rotate_sh (identity for improper
    rotations, which rotate_sh leaves alone)."""
    rot = extrinsics[..., :3, :3].reshape(b, v, 3, 3)
    d_sh = (sh_degree + 1) ** 2
    if rotations_are_proper(rot):
        return sh_rotation_blocks(rot, d_sh)
    return torch.eye(d_sh).expand(b, v, d_sh, d_sh)


CASES = {
    # name: (seed, b, v, h, w, sh_degree, proper rotations)
    "adapter_pf3plat": (0, 1, 2, 6, 8, 4, True),       # PF3plat: sh_degree 4, two context views
    "adapter_deg2_batch": (1, 2, 3, 5, 5, 2, True),
    "adapter_improper": (2, 1, 2, 4, 6, 4, False),     # det != 1 -> identity SH rotation (sh_rotation.py:21-22)
}


def main():
    ref = load_reference_adapter()
    for name, (seed, b, v, h, w, deg, proper) in CASES.items():
        inp = make_inputs(seed, b, v, h, w, deg, proper)
        leaves = {k: t.clone().requires_grad_(k != "opacities") for k, t in inp.items()}
        adapter = ref.GaussianAdapter(ref.GaussianAdapterCfg(gaussian_scale_min=0.5, gaussian_scale_max=15.0, sh_degree=deg))
        out = adapter.forward(leaves["extrinsics"], leaves["intrinsics"], leaves["coordinates"], leaves["depths"],
                              leaves["opacities"], leaves["raw_gaussians"], (h, w))
        outs = dict(means=out.means, covariances=out.covariances, harmonics=out.harmonics, scales=out.scales,
                    rotations=out.rotations)
        weights = make_weights(seed, {k: t.shape for k, t in outs.items()})
        loss = sum((weights[k] * outs[k]).sum() for k in outs)
        loss.backward()
        dmat = sh_rotation_used(inp["extrinsics"], b, v, deg)
        arrays = {f"in_{k}": t.numpy() for k, t in inp.items()}
        arrays.update({f"out_{k}": t.detach().numpy() for k, t in outs.items()})
        arrays.update({f"w_{k}": t.numpy() for k, t in weights.items()})
        arrays.update({f"grad_{k}": leaves[k].grad.numpy() for k in leaves if leaves[k].grad is not None})
        arrays["sh_rotation"] = dmat.numpy().astype(np.float32)
        arrays["meta"] = np.array([b, v, h, w, deg, int(proper)], np.int64)
        path = os.path.join(HERE, f"{name}.npz")
        np.savez_compressed(path, **arrays)
        print(name, {k: tuple(a.shape) for k, a in arrays.items() if k.startswith(("out_", "grad_"))},
              os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
