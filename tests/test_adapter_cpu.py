"""Pins the adapter oracle (oracle/adapter_oracle.py) to the REFERENCE's own outputs: the golden fixtures were
produced by the reference's src/model/encoder/common/gaussian_adapter.py itself (tests/golden/make_adapter_golden.py).
Also: the SH-rotation helper's algebra, and that the generating script still feeds the reference what the fixtures hold."""
import os
import sys

import numpy as np
import pytest
import torch

from tests import adapter_util as au

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from pf3plat_b200 import sh_rotation  # noqa: E402


@pytest.mark.parametrize("name", au.CASES)
def test_oracle_matches_reference_outputs_and_gradients(name):
    z, meta = au.load(name)
    out, grads = au.oracle_run(z, meta)
    # the reference ran in fp32, the oracle in fp64: agreement to fp32 rounding of a ~30-operation chain
    for k in au.OUTPUTS:
        assert out[k].shape == z["out_" + k].shape, k
        assert au.rel_err(out[k], z["out_" + k]) < 2e-6, (k, au.rel_err(out[k], z["out_" + k]))
    for k in au.GRADS:
        assert grads[k].shape == z["grad_" + k].shape, k
        assert au.rel_err(grads[k], z["grad_" + k]) < 2e-5, (k, au.rel_err(grads[k], z["grad_" + k]))


def test_oracle_in_fp32_is_as_close_to_the_reference_as_fp32_allows():
    z, meta = au.load("adapter_pf3plat")
    out, _ = au.oracle_run(z, meta, dtype=torch.float32)
    for k in au.OUTPUTS:
        assert au.rel_err(out[k], z["out_" + k]) < 1e-6, k


def test_improper_rotations_fall_back_to_identity_sh_rotation():
    z, meta = au.load("adapter_improper")
    assert not meta["proper"]
    d = z["sh_rotation"]
    assert np.array_equal(d[0, 0], np.eye(d.shape[-1], dtype=np.float32))
    # harmonics are then just raw * mask, transposed
    raw = z["in_raw_gaussians"][..., 7:].reshape(*z["in_raw_gaussians"].shape[:-1], 3, 25)
    from oracle.adapter_oracle import sh_mask
    np.testing.assert_allclose(z["out_harmonics"], raw * sh_mask(4).numpy(), rtol=1e-6, atol=1e-7)


def test_wigner_matrices_are_orthogonal_homomorphic_and_equal_the_rotation_for_degree_one():
    g = torch.Generator().manual_seed(3)
    q = torch.randn(6, 4, generator=g, dtype=torch.float64)
    q = q / q.norm(dim=-1, keepdim=True)
    from pf3plat_b200.synthetic import quat_to_rotmat
    rot = quat_to_rotmat(q)
    for degree in range(5):
        d = sh_rotation.wigner_d_from_matrix(degree, rot)
        eye = torch.eye(2 * degree + 1, dtype=torch.float64)
        assert (d @ d.transpose(-1, -2) - eye).abs().max() < 1e-12
        assert (sh_rotation.wigner_d_from_matrix(degree, rot[0] @ rot[1]) - d[0] @ d[1]).abs().max() < 1e-12
        # defining property on fresh points
        x = torch.randn(50, 3, generator=g, dtype=torch.float64)
        x = x / x.norm(dim=-1, keepdim=True)
        lhs = sh_rotation.real_sh_basis(degree, x @ rot[2].T)
        rhs = sh_rotation.real_sh_basis(degree, x) @ d[2].T
        assert (lhs - rhs).abs().max() < 1e-12
    assert (sh_rotation.wigner_d_from_matrix(1, rot) - rot).abs().max() < 1e-12
    blocks = sh_rotation.sh_rotation_blocks(rot, 25)
    assert blocks.shape == (6, 25, 25) and blocks[:, 0, 0].sub(1).abs().max() < 1e-12 and blocks[:, 0, 1:].abs().max() == 0
    # rotate_sh keeps the reference's guard: improper input -> coefficients unchanged
    sh = torch.randn(6, 25, generator=g, dtype=torch.float64)
    assert (sh_rotation.rotate_sh(sh, rot * 1.1) - sh).abs().max() < 1e-13


def test_fixtures_are_what_the_reference_module_produces_today():
    """The outputs and gradients of each fixture are the reference module's, a fixed function of what the generating
    script feeds it: the inputs, the loss weights and the Wigner-D matrices its e3nn stub hands over (computed by
    pf3plat_b200.sh_rotation).  The fixture stays what the reference produces as long as the script still generates
    the stored ones to fp32 rounding: guards against a stale fixture after an edit of the script or of sh_rotation."""
    sys.path.insert(0, au.GOLDEN)
    import make_adapter_golden as mk
    for name in au.CASES:
        z, meta = au.load(name)
        seed, b, v, h, w, deg, proper = mk.CASES[name]
        assert (b, v, h, w, deg, proper) == tuple(meta.values()), name
        inp = mk.make_inputs(seed, b, v, h, w, deg, proper)

        def same(got, key):
            np.testing.assert_allclose(got.numpy(), z[key], rtol=1e-6, atol=1e-7, err_msg=f"{name} {key}")
        for k in au.INPUTS:
            same(inp[k], "in_" + k)
        for k, t in mk.make_weights(seed, {k: z["out_" + k].shape for k in au.OUTPUTS}).items():
            same(t, "w_" + k)
        same(mk.sh_rotation_used(inp["extrinsics"], b, v, deg), "sh_rotation")
