"""CPU: the re-implemented coarse-to-fine sweep returns the reference's grid and lattice geometry bit-for-bit when
both use the same query function (tests/golden/c2f_grid.npz and c2f_lattice.npz hold what the reference class
computes, tests/golden/make_golden_c2f.py)."""
import os

import numpy as np
import torch

from conftest import GOLDEN, load_golden
from recmv_b200.MCAcc import Seg3dLossless, create_grid3D


def sphere_query(points):
    # min distance to three spheres, returned as [1,1,M] like OptimNetwork.discretizeSDF's query_func
    p = points.reshape(-1, 3)
    c = torch.tensor([[0.1, -0.2, 0.05], [-0.35, 0.3, -0.1], [0.3, 0.35, 0.3]], dtype=p.dtype, device=p.device)
    r = torch.tensor([0.45, 0.3, 0.22], dtype=p.dtype, device=p.device)
    d = ((p[:, None, :] - c[None]).norm(dim=2) - r[None]).min(dim=1).values
    return d.reshape(1, 1, -1)


PYR = [(9, 13, 7), (17, 25, 13), (33, 49, 25), (65, 97, 49)]
KW = dict(b_min=[-1.0, -1.2, -0.9], b_max=[1.0, 1.2, 0.9], resolutions=PYR, align_corners=False,
          balance_value=0.0, visualize=False, debug=False, use_cuda_impl=False, faster=False)


def test_create_grid3d_order():
    g = create_grid3D(0, 8, steps=(3, 5, 2), device="cpu")
    assert g.shape == (30, 3) and g[1].tolist() == [4, 0, 0] and g[3].tolist() == [0, 2, 0]


def test_matches_golden_grid():
    eng = Seg3dLossless(sphere_query, **KW)
    out = eng.forward()
    gold = np.load(os.path.join(GOLDEN, "c2f_grid.npz"))["grid"]
    assert out.shape == (1, 1, 49, 97, 65)
    assert np.array_equal(out[0, 0].numpy(), gold)
    # the sweep is "lossless" where it matters: same sign as the dense evaluation everywhere
    dense = sphere_query(((create_grid3D(0, (64, 96, 48), steps=(65, 97, 49), device="cpu").float()
                           / torch.tensor([65., 97., 49.]) + 0.5 / torch.tensor([65., 97., 49.]))
                          * (eng.b_max - eng.b_min)[0] + eng.b_min[0])).view(49, 97, 65)
    assert bool(((dense > 0) == (out[0, 0] > 0)).all())
    assert sum(s[3] for s in eng.stats) < 0.4 * 49 * 97 * 65  # and it evaluates a fraction of the lattice


def test_bit_identical_to_reference_class():
    grid, lattice = load_golden("c2f_grid.npz")["grid"], load_golden("c2f_lattice.npz")
    ours = Seg3dLossless(sphere_query, **KW)
    b = ours.forward()
    assert torch.equal(b, torch.from_numpy(grid)[None, None])
    for name in ("spacing_x", "spacing_y", "spacing_z", "bx", "by", "bz"):
        assert float(lattice[name]) == getattr(ours, name)


def test_interp2x_boundary_oracle_pins():
    """The restated upsampler against an independent implementation: values == F.interpolate(trilinear,
    align_corners=True) up to fp32 rounding, flags == 'interpolated 0/1 occupancy strictly between 0 and 1' (the
    reference's default path, seg3d_lossless.py:270-281), backward == autograd of the interpolation."""
    import torch.nn.functional as F
    from oracle import oracle_torch as ot
    g = torch.Generator().manual_seed(4)
    x = torch.randn((1, 2, 5, 6, 7), generator=g)
    out, flag = ot.interp2x_boundary3d(x, 0.1)
    size = (9, 11, 13)
    ref = F.interpolate(x, size=size, mode="trilinear", align_corners=True)
    valid = F.interpolate((x > 0.1).float(), size=size, mode="trilinear", align_corners=True)
    assert out.shape == ref.shape and (out - ref).abs().max() < 1e-6
    assert torch.equal(flag, (valid > 0) & (valid < 1))
    go = torch.randn(ref.shape, generator=g)
    xr = x.clone().requires_grad_(True)
    F.interpolate(xr, size=size, mode="trilinear", align_corners=True).backward(go)
    assert (ot.interp2x_boundary3d_backward(go) - xr.grad).abs().max() < 1e-5
