"""GPU: the mesh rasteriser (recmv_rasterize / ops.rasterize) against the float64 brute force of oracle/raster_oracle.py on
triangle soups, a deformed marching-cubes mesh and a close-up with faces larger than the warp threshold and faces behind
the camera; determinism; the chain rasteriser -> FindSurfacePsRays; render.render_colors against the same steps written
out with the public functions; render.MaskRasterizer on a meshes object."""
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN
sys.path.insert(0, GOLDEN)
import make_golden as mg  # noqa: E402  (scene builder shared with the surface tests)
from oracle import raster_oracle as ro  # noqa: E402
from recmv_b200 import ops, render, synth, testing  # noqa: E402
from recmv_b200 import model as M  # noqa: E402
from recmv_b200 import utils as U  # noqa: E402
from recmv_b200.MCAcc import Seg3dLossless  # noqa: E402
from recmv_b200.discretize import discretize_sdf  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H, W = 64, 96                       # H != W
WARP_FACE_PIXELS = 128              # faces with a larger clipped bounding box are swept by a warp (csrc/raster.cu)
RATIO = {"sdfRatio": 0.8, "deformerRatio": 0.6, "renderRatio": 0.9}


class _Mods:  # the scene builder expects module namespaces
    getTmpSdf = staticmethod(M.getTmpSdf)
    MLPTranslator, LBSkinner, CompositeDeformer = M.MLPTranslator, M.LBSkinner, M.CompositeDeformer


def _rot(ax, ay, az):
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    Rx = np.array([[1, 0, 0], [0, cx, -sx], [0, sx, cx]])
    Ry = np.array([[cy, 0, sy], [0, 1, 0], [-sy, 0, cy]])
    Rz = np.array([[cz, -sz, 0], [sz, cz, 0], [0, 0, 1]])
    return Rx @ Ry @ Rz


def _camera(R, T, fx=1.2 * W, fy=1.2 * W, px=(W - 1) / 2, py=(H - 1) / 2):
    R = torch.tensor(np.asarray(R), dtype=torch.float32).reshape(-1, 3, 3)
    T = torch.tensor(np.asarray(T), dtype=torch.float32).reshape(-1, 3)
    return fx, fy, px, py, R.to(DEV), T.to(DEV)


def _check_against_oracle(verts, faces, cam, size=(H, W)):
    fr = ops.rasterize(verts, faces, cam, size)
    fx, fy, px, py, R, T = cam
    ref_f, ref_z, ref_b, amb = ro.rasterize(verts.cpu().numpy(), faces.cpu().numpy(),
                                            (fx, fy, px, py, R.cpu().numpy(), T.cpu().numpy()), size)
    p2f, zbuf, bary = fr.pix_to_face.cpu().numpy(), fr.zbuf.cpu().numpy(), fr.bary_coords.cpu().numpy()
    bg = p2f[..., 0] < 0
    assert (zbuf[bg] == -1).all() and (bary[bg] == -1).all()            # background: exactly -1 everywhere
    assert ((p2f < 0) == (p2f == -1)).all()
    covered = ref_f[..., 0] >= 0
    same = p2f[..., 0] == ref_f[..., 0]
    n_amb = int((amb & covered).sum())
    print(f"covered {int(covered.sum())}, ambiguous {n_amb}, mismatches on ambiguous pixels {int((~same & amb).sum())}")
    assert covered.sum() > 500 and n_amb < 0.005 * covered.sum()
    assert same[~amb].all(), np.argwhere(~same & ~amb)[:10]
    hit = same & covered
    assert np.abs(bary[hit] - ref_b[hit]).max() < 2e-4
    assert (np.abs(zbuf[hit] - ref_z[hit]) / ref_z[hit]).max() < 1e-5
    again = ops.rasterize(verts, faces, cam, size)                      # determinism: bit-identical second call
    assert all(torch.equal(a, b) for a, b in zip(fr[:3], again[:3])) and fr.dists is None
    return fr


def _bbox_pixels(verts, faces, cam, size):
    """Clipped pixel-box sizes of the faces with all three vertices in front of camera 0."""
    fx, fy, px, py, R, T = cam
    h, w = size
    x, y, z = ro.project(verts.reshape(-1, 3), R[0].cpu().numpy(), T[0].cpu().numpy(), fx, fy, px, py)
    fa = faces.cpu().numpy()
    x, y, z = x[fa], y[fa], z[fa]
    front = (z > 0).all(1)
    w_ = np.clip(np.floor(x.max(1)), -1, w - 1) - np.clip(np.ceil(x.min(1)), 0, w) + 1
    h_ = np.clip(np.floor(y.max(1)), -1, h - 1) - np.clip(np.ceil(y.min(1)), 0, h) + 1
    return np.where(front, np.maximum(w_, 0) * np.maximum(h_, 0), 0)


def test_triangle_soup_two_frames_per_frame_cameras():
    g = np.random.default_rng(11)
    F = 500
    N = 2
    Rs = np.stack([_rot(0.1, -0.2, 0.05), _rot(-0.15, 0.3, -0.1)])
    Ts = np.array([[0.1, -0.05, 3.0], [-0.2, 0.1, 2.6]])
    verts = []
    for n in range(N):
        # camera-space triangles in the view frustum, sizes from ~1 px to ~60 px, mapped to world: Xw = (Xc - T) R^T
        c = g.uniform([-1.1, -0.7, 2.0], [1.1, 0.7, 4.5], (F, 1, 3))
        size = np.exp(g.uniform(np.log(0.02), np.log(0.8), (F, 1, 1)))
        xc = c + size * g.normal(0, 1, (F, 3, 3))
        verts.append(((xc.reshape(-1, 3) - Ts[n]) @ Rs[n].T))
    verts = torch.tensor(np.stack(verts), dtype=torch.float32, device=DEV)
    faces = torch.arange(3 * F, device=DEV).view(F, 3)
    cam = _camera(Rs, Ts, fx=80.0, fy=84.0, px=47.3, py=31.6)
    _check_against_oracle(verts, faces, cam)


def _mc_scene():
    sdf = synth.sphere_sdf_grid(res=49, num=8, seed=3, device=DEV)
    step = 2.0 / 48
    v, f = ops.mc_gpu(sdf, step, step, step, -1.0, -1.0, -1.0)
    assert f.min() >= 0
    _, deformer = mg.surface_scene(_Mods, _Mods, device="cpu")
    deformer = deformer.to(DEV)
    poses, trans = synth.poses_trans(2, seed=11)
    conds = torch.randn((2, 128), generator=synth.generator(5)) * 0.1
    defconds = [conds.to(DEV), [poses.to(DEV), trans.to(DEV)]]
    with torch.no_grad():
        dv = deformer(v[None].expand(2, -1, 3), defconds, ratio=RATIO, offset_type="body")
    cam = _camera(np.eye(3), [0.0, 0.0, 2.4])
    return v, f, dv.contiguous(), cam


def test_deformed_marching_cubes_mesh_and_the_chain_to_find_surface_rays():
    v, f, dv, cam = _mc_scene()
    fr = _check_against_oracle(dv, f, cam)
    # every row FindSurfacePsRays returns: the interpolated DEFORMED point lies on the returned ray, at depth zbuf
    fx, fy, px, py, R, T = cam
    b, r, c, pts, fi, rays = U.FindSurfacePsRays(v, f, fr, (fx, fy, px, py, R[0].cpu()))
    assert b.numel() > 1000
    Rd, Td = R[0].double(), T[0].double()
    bc = fr.bary_coords[b, r, c, 0].double()
    P = (bc[:, :, None] * dv[b[:, None], f[fi]].double()).sum(1)
    off = P + Rd.matmul(Td)                                             # P - cam_pos, cam_pos = -R T
    cosang = (off * rays.double()).sum(1) / off.norm(dim=1) / rays.double().norm(dim=1)
    ang = torch.rad2deg(torch.arccos(cosang.clamp(max=1.0)))
    zc = (P.matmul(Rd) + Td)[:, 2]
    zb = fr.zbuf[b, r, c, 0].double()
    print(f"chain: max angle {ang.max().item():.2e} deg, max depth error {((zc - zb).abs() / zb).max().item():.2e}")
    assert ang.max() < 1e-4 and ((zc - zb).abs() / zb).max() < 1e-5


def test_large_faces_and_faces_behind_the_camera():
    g = np.random.default_rng(3)
    tris = []
    for _ in range(6):                                   # close-up faces spanning a large part of the image
        c = g.uniform([-0.3, -0.2, 0.6], [0.3, 0.2, 1.6], (1, 3))
        tris.append(c + g.normal(0, 0.6, (3, 3)) * [1, 1, 0.2])
    for _ in range(40):                                  # small faces, some in front of, some behind the large ones
        z = g.uniform(0.5, 2.5)
        c = np.array([[g.uniform(-0.4, 0.4) * z, g.uniform(-0.26, 0.26) * z, z]])
        tris.append(c + g.normal(0, 0.02 * z, (3, 3)))
    for _ in range(6):                                   # one vertex behind the camera (Zc < 0): skipped
        c = g.uniform([-0.3, -0.2, 0.4], [0.3, 0.2, 0.8], (1, 3))
        t = c + g.normal(0, 0.3, (3, 3)) * [1, 1, 0]
        t[0, 2] = -0.5
        tris.append(t)
    verts = torch.tensor(np.concatenate(tris), dtype=torch.float32, device=DEV)[None]
    faces = torch.arange(verts.shape[1], device=DEV).view(-1, 3)
    cam = _camera(np.eye(3), [0.0, 0.0, 0.0])
    px_count = _bbox_pixels(verts[0].cpu().numpy(), faces, cam, (H, W))
    assert (px_count > WARP_FACE_PIXELS).sum() >= 4 and ((px_count > 0) & (px_count <= WARP_FACE_PIXELS)).sum() >= 20
    fr = _check_against_oracle(verts, faces, cam)
    behind = set(range(46, 52))
    assert not behind & set(fr.pix_to_face.unique().tolist())


def test_render_colors_matches_the_steps_written_out():
    sdf, deformer = mg.surface_scene(_Mods, _Mods, device="cpu")
    sdf, deformer = sdf.to(DEV), deformer.to(DEV)
    torch.manual_seed(2)
    rn = M.RenderingNetwork_view_norm(256, d_in=9, d_out=3, dims=[512] * 4, mode="idr", weight_norm=True,
                                      multires_v=4, multires_n=0)
    testing.perturb_module(rn, 303)
    rn = rn.to(DEV)
    eng = Seg3dLossless(None, b_min=[-1, -1, -1], b_max=[1, 1, 1], resolutions=[17, 33, 65], align_corners=False,
                        balance_value=0.0).to(DEV)
    v, f = discretize_sdf(sdf, eng, RATIO)
    poses, trans = synth.poses_trans(2, seed=11)
    conds = torch.randn((2, 128), generator=synth.generator(5)) * 0.1
    defconds = [conds.to(DEV), [poses.to(DEV), trans.to(DEV)]]
    size = (48, 64)
    cam = _camera(np.eye(3), [0.0, 0.0, 2.4], fx=80.0, fy=80.0, px=31.5, py=23.5)
    kw = dict(offset_type="body", dthreshold=1e-4, times=10)
    colors, mask, fr = render.render_colors(v, f, sdf, deformer, defconds, rn, cam, size, RATIO, 0.05, **kw)
    # the nine steps with the existing public functions, on the same fragments, in one chunk
    fx, fy, px, py, R, T = cam
    with torch.no_grad():
        dv = deformer(v[None].expand(2, -1, 3), defconds, ratio=RATIO, offset_type="body")
    fr2 = ops.rasterize(dv.contiguous(), f, cam, size)
    assert all(torch.equal(a, b) for a, b in zip(fr[:3], fr2[:3]))
    b, r, c, seeds, _, rays = U.FindSurfacePsRays(v, f, fr, (fx, fy, px, py, R[0].cpu()))
    assert b.numel() > 300
    cam_pos = -R[0].matmul(T[0].view(3, 1)).view(3)
    ps, _ = U.OptimizeGarmentSurfaceSinlge(cam_pos, rays, seeds.clone(), b, sdf, RATIO, deformer, defconds, dthreshold=1e-4,
                                           athreshold=0.05, w1=3.05, w2=1., times=10, offset_type="body")
    with torch.no_grad():
        _, gr = sdf.value_and_grad(ps, RATIO, want_feat=True)
        feat = sdf.rendcond
        nx = gr / gr.norm(dim=1, keepdim=True)
    crays, _ = U.compute_cardinal_rays(deformer, ps, rays, defconds, b, RATIO, 'test', offset_type="body")
    with torch.no_grad():
        col = torch.clamp((rn(ps, nx, crays, feat, RATIO) / 2. + 0.5) * 255., min=0., max=255.)
    ref = torch.full((2,) + size + (3,), 255., device=DEV)
    ref[b, r, c] = col
    assert torch.equal(mask, fr.pix_to_face[..., 0] >= 0) and colors.shape == (2,) + size + (3,)
    assert (colors - ref).abs().max() < 1e-4 and (colors[mask] < 254.).any() and (colors[~mask] == 255.).all()
    colors2, _, _ = render.render_colors(v, f, sdf, deformer, defconds, rn, cam, size, RATIO, 0.05, chunk=97, **kw)
    assert (colors2 - colors).abs().max() < 1e-4
    ops.check_async_errors()


def test_mask_rasterizer_on_a_meshes_object_and_input_checks():
    v, f, dv, cam = _mc_scene()

    class Meshes:                                        # duck-typed: the two methods maskRender's callers use
        def __init__(self, verts, faces):
            self.v, self.f = verts, faces

        def verts_padded(self):
            return self.v

        def faces_padded(self):
            return self.f

    mr = render.MaskRasterizer(cam, (H, W))
    imgs, fr = mr(Meshes(dv, f[None].expand(2, -1, 3)))
    ref = ops.rasterize(dv, f, cam, (H, W))
    assert imgs is None and all(torch.equal(a, b) for a, b in zip(fr[:3], ref[:3]))
    _, fr2 = mr(dv, f)
    assert torch.equal(fr2.pix_to_face, ref.pix_to_face)
    f2 = torch.stack([f, f.flip(0)])
    with pytest.raises(RuntimeError):
        mr(Meshes(dv, f2))
    with pytest.raises(RuntimeError):                    # CPU input: no fallback
        ops.rasterize(dv.cpu(), f.cpu(), cam, (H, W))
    with pytest.raises(RuntimeError):                    # non-contiguous input
        ops.rasterize(dv.transpose(0, 1), f, cam, (H, W))
    one = ops.rasterize(dv[0], f, cam, (H, W))           # [V,3]: one mesh
    assert torch.equal(one.pix_to_face, ref.pix_to_face[:1])
