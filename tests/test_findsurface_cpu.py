"""CPU: FindSurfacePs (fragment decode, pure index logic) against the reference function's output on the same
fragments (tests/golden/findsurface.npz, tests/golden/make_golden.py)."""
import numpy as np
import torch

from conftest import load_golden
from recmv_b200.utils import FindSurfacePs


class Frags:
    def __init__(self, p2f, bary):
        self.pix_to_face, self.bary_coords = p2f, bary


def _inputs():
    g = load_golden("findsurface.npz")
    t = {k: torch.from_numpy(v) for k, v in g.items()}
    return g, t


def test_findsurfaceps_matches_golden():
    g, t = _inputs()
    b, r, c, pts, fi = FindSurfacePs(t["verts"], t["faces"], Frags(t["pix_to_face"], t["bary"]))
    assert np.array_equal(b.numpy(), g["batch"]) and np.array_equal(r.numpy(), g["row"])
    assert np.array_equal(c.numpy(), g["col"]) and np.array_equal(fi.numpy(), g["finds"])  # indices: bit exact
    assert np.allclose(pts.numpy(), g["pts"], atol=1e-6)
    # nothing covered / K = 1
    e = FindSurfacePs(t["verts"], t["faces"], Frags(torch.full((1, 4, 4, 1), -1), torch.rand(1, 4, 4, 1, 3)))
    assert all(x.numel() == 0 for x in e[:3]) and e[3].shape == (0, 3)


def test_findsurfaceps_matches_reference_function():
    g, t = _inputs()
    ref = [t[k] for k in ("batch", "row", "col", "pts", "finds")]   # the reference function's return tuple
    ours = FindSurfacePs(t["verts"], t["faces"], Frags(t["pix_to_face"], t["bary"]))
    assert len(ours) == len(ref)
    for a, b in zip(ref, ours):
        assert torch.equal(a, b) or torch.allclose(a, b, atol=1e-6)


def test_surface_grad_coeffs_oracle_pins():
    """Restated per-ray algebra of propagateTmpPsGrad: r = g (b^T b)^-1 b^T must satisfy r b = g wherever b^T b is
    invertible, and the fp32 result must agree with the same formulas in fp64."""
    import torch
    from oracle import oracle_torch as ot
    g = torch.Generator().manual_seed(9)
    n = 500
    gl, gf, v, dc = (torch.randn((n, 3), generator=g) for _ in range(4))
    v = v / v.norm(dim=1, keepdim=True)
    J = torch.eye(3).expand(n, 3, 3) + 0.3 * torch.randn((n, 3, 3), generator=g)
    coef, vec, rg, ok = ot.surface_grad_coeffs(gl, gf, J, v, dc)
    assert ok.float().mean() > 0.95
    vx = ot.cross_matrix(v)
    b = torch.cat([gf.view(-1, 1, 3), vx.matmul(J)], dim=1)
    # recover r from the outputs: r0 = -coef ; r[1:4] [v]x = -vec  (r[1:4] itself is only defined up to its component along v)
    c64, v64, r64, ok64 = ot.surface_grad_coeffs(gl.double(), gf.double(), J.double(), v.double(), dc.double())
    det = torch.linalg.det(b.permute(0, 2, 1).matmul(b).double())
    sel = ok & ok64 & (det.abs() > 5e-2)       # near the 1e-4 determinant threshold fp32 loses all digits, as the reference does
    assert sel.float().mean() > 0.6
    assert (coef[sel] - c64[sel].float()).abs().max() < 1e-3 * c64[sel].abs().max()
    assert (vec[sel] - v64[sel].float()).abs().max() < 1e-3 * v64[sel].abs().max()
    bd = b.double()
    inv, okd = ot.minv3x3_fwd(bd.permute(0, 2, 1).matmul(bd).contiguous())
    r = gl.double().view(-1, 1, 3).matmul(inv.matmul(bd.permute(0, 2, 1)))
    assert (r.matmul(bd).view(-1, 3) - gl.double())[okd & (det.abs() > 5e-2)].abs().max() < 1e-8
