"""GPU: the points rasteriser + alpha compositor (recmv_points_* / ops.rasterize_points / render.PointsRenderer) against
the float64 brute force of oracle/points_oracle.py -- random clouds at H != W with per-frame cameras, discs clipped at the
image border, points behind the camera, a dense case where K = 8 and K = 50 truncate, a large radius with pixels over 1024
candidates, the deformed marching-cubes vertices at 512^2 -- with the gradient against the float64 composite of the
kernel's own selection; determinism; the `_Split` form; and the mask-loss chain through the deformer's training path."""
import sys

import numpy as np
import pytest
import torch

from conftest import GOLDEN
sys.path.insert(0, GOLDEN)
import make_golden as mg  # noqa: E402  (scene builder shared with the surface tests)
from oracle import points_oracle as po  # noqa: E402
from recmv_b200 import ops, render, synth  # noqa: E402
from recmv_b200 import model as M  # noqa: E402

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
H, W = 64, 96                       # H != W
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


def _np_camera(cam):
    fx, fy, px, py, R, T = cam
    return fx, fy, px, py, R.cpu().numpy(), T.cpu().numpy()


def _camera(R, T, fx=1.2 * W, fy=1.2 * W, px=(W - 1) / 2, py=(H - 1) / 2):
    R = torch.tensor(np.asarray(R), dtype=torch.float32).reshape(-1, 3, 3)
    T = torch.tensor(np.asarray(T), dtype=torch.float32).reshape(-1, 3)
    return fx, fy, px, py, R.to(DEV), T.to(DEV)


def _world(xc, R, T):
    """Camera-space points [P,3] of camera (R, T) -> world: Xw = (Xc - T) R^T."""
    return (xc - T) @ R.T


def _check_against_oracle(points, feats, cam, size, radius, K, min_covered=500):
    """Every assertion of the comparison; returns (images, fragments, oracle outputs)."""
    pts = points.detach().requires_grad_(True)
    images, fr = ops.rasterize_points(pts, feats, cam, size, radius, K)
    ref_i, ref_z, ref_d, ref_img, amb = po.rasterize_points(points.detach().cpu().numpy(), feats.cpu().numpy(),
                                                            _np_camera(cam), size, radius, K)
    idx, zbuf, dists = fr.idx.cpu().numpy(), fr.zbuf.cpu().numpy(), fr.dists.cpu().numpy()
    img = images.detach().cpu().numpy()
    empty = idx < 0
    assert (idx[empty] == -1).all() and (zbuf[empty] == -1).all() and (dists[empty] == -1).all()
    covered = ref_i[..., 0] >= 0
    n_amb = int((amb & covered).sum())
    same = (idx == ref_i).all(-1)
    print(f"covered {int(covered.sum())}, ambiguous {n_amb}, mismatches on ambiguous pixels {int((~same & amb).sum())}, "
          f"truncated pixels {int((ref_i[..., -1] >= 0).sum())}")
    assert covered.sum() > min_covered and n_amb < 0.005 * covered.sum()
    assert same[~amb].all(), np.argwhere(~same & ~amb)[:10]
    ok = (~amb)[..., None] & (idx >= 0)
    assert (np.abs(dists[ok] - ref_d[ok]) <= 1e-5 * ref_d[ok] + 1e-12).all()
    assert (np.abs(zbuf[ok] - ref_z[ok]) <= 1e-6 * ref_z[ok]).all()
    assert np.abs(img[~amb] - ref_img[~amb]).max() < 1e-5
    # determinism: a second call is bit-identical, images and fragments
    images2, fr2 = ops.rasterize_points(points.detach(), feats, cam, size, radius, K)
    assert torch.equal(images2, images.detach())
    assert all(torch.equal(a, b) for a, b in zip((fr.idx, fr.zbuf, fr.dists), (fr2.idx, fr2.zbuf, fr2.dists)))
    # gradient: against the float64 composite of the kernel's own selection
    g = torch.randn(images.shape, generator=torch.Generator().manual_seed(7)).to(DEV)
    (images * g).sum().backward()
    p64 = points.detach().double().requires_grad_(True)
    (po.composite_given(p64, feats, fr.idx, _np_camera(cam), size, radius) * g.double()).sum().backward()
    g64 = p64.grad
    err = (pts.grad.double() - g64).abs().max().item()
    print(f"grad_points: max |g - g64| {err:.3e}, max |g64| {g64.abs().max().item():.3e}")
    assert g64.abs().max() > 0 and err <= 1e-4 * g64.abs().max().item()
    ops.check_async_errors()
    return images, fr, (ref_i, ref_z, ref_d, ref_img, amb)


def test_random_clouds_two_frames_per_frame_cameras():
    g = np.random.default_rng(11)
    N, P = 2, 3000
    Rs = np.stack([_rot(0.1, -0.2, 0.05), _rot(-0.15, 0.3, -0.1)])
    Ts = np.array([[0.1, -0.05, 3.0], [-0.2, 0.1, 2.6]])
    xc = np.stack([np.stack([g.uniform(-1.3, 1.3, P), g.uniform(-0.9, 0.9, P), g.uniform(2.0, 5.0, P)], 1)
                   for _ in range(N)])
    pts = torch.tensor(np.stack([_world(xc[n], Rs[n], Ts[n]) for n in range(N)]), dtype=torch.float32, device=DEV)
    feats = torch.tensor(g.uniform(0, 1, (P, 3)), dtype=torch.float32, device=DEV)
    cam = _camera(Rs, Ts, fx=80.0, fy=84.0, px=47.3, py=31.6)
    _, fr, (ref_i, _, _, _, _) = _check_against_oracle(pts, feats, cam, (H, W), 0.05, 8)
    assert (ref_i[1] >= P).sum() == (ref_i[1] >= 0).sum() > 0        # packed index n * P + p


def test_discs_clipped_at_the_border_and_points_behind_the_camera():
    g = np.random.default_rng(3)
    P = 1500
    # screen positions around and beyond the image edges, depth 1.5 - 3; a fifth of the points behind the camera
    sx, sy, z = g.uniform(-6, W + 6, P), g.uniform(-6, H + 6, P), g.uniform(1.5, 3.0, P)
    fx = fy = 70.0
    px, py = (W - 1) / 2, (H - 1) / 2
    xc = np.stack([(px - sx) * z / fx, (py - sy) * z / fy, z], 1)
    behind = g.uniform(0, 1, P) < 0.2
    xc[behind, 2] *= -1
    pts = torch.tensor(xc, dtype=torch.float32, device=DEV)[None]
    feats = torch.ones((P, 1), device=DEV)
    cam = _camera(np.eye(3), np.zeros(3), fx=fx, fy=fy, px=px, py=py)
    radius = 0.15                                                     # 4.8 px: discs cut by the border
    _, fr, _ = _check_against_oracle(pts, feats, cam, (H, W), radius, 8)
    assert not set(np.nonzero(behind)[0].tolist()) & set(fr.idx.unique().tolist())
    r = radius * H / 2
    border = ((sx < 0) | (sx > W - 1) | (sy < 0) | (sy > H - 1)) & ~behind
    assert border.sum() > 100 and ((sx > -r) & (sx < 0)).sum() > 10
    assert (fr.idx[0, :, 0] >= 0).any() and (fr.idx[0, :, -1] >= 0).any()


@pytest.mark.parametrize("K", [8, 50])
def test_dense_cloud_truncates(K):
    g = np.random.default_rng(5)
    P_bg, P_cl = 1500, 1200
    # a sparse cloud over the whole image and a dense cluster (sigma 4 px, over 300 candidates at its centre); depth
    # spread 1 - 20, so few near-equal depths
    z = g.uniform(1.0, 20.0, P_bg + P_cl)
    sx = np.concatenate([g.uniform(0, W, P_bg), g.normal(40, 4, P_cl)])
    sy = np.concatenate([g.uniform(0, H, P_bg), g.normal(30, 4, P_cl)])
    fx = fy = 90.0
    px, py = 47.5, 31.5
    xc = np.stack([(px - sx) * z / fx, (py - sy) * z / fy, z], 1)
    pts = torch.tensor(xc, dtype=torch.float32, device=DEV)[None]
    feats = torch.tensor(g.uniform(0, 1, (P_bg + P_cl, 2)), dtype=torch.float32, device=DEV)
    cam = _camera(np.eye(3), np.zeros(3), fx=fx, fy=fy, px=px, py=py)
    _, _, (ref_i, _, _, _, _) = _check_against_oracle(pts, feats, cam, (H, W), 0.1, K)
    assert (ref_i[..., -1] >= 0).sum() > 100                          # pixels with more than K candidates


def test_large_radius_long_segments():
    g = np.random.default_rng(8)
    P = 3000
    sx, sy, z = g.normal(W / 2, 4, P), g.normal(H / 2, 4, P), g.uniform(1.0, 30.0, P)
    fx = fy = 90.0
    px, py = 47.5, 31.5
    xc = np.stack([(px - sx) * z / fx, (py - sy) * z / fy, z], 1)
    pts = torch.tensor(xc, dtype=torch.float32, device=DEV)[None]
    feats = torch.ones((P, 1), device=DEV)
    cam = _camera(np.eye(3), np.zeros(3), fx=fx, fy=fy, px=px, py=py)
    radius = 0.4                                                      # 12.8 px
    r = radius * H / 2
    cand = ((sx - W / 2) ** 2 + (sy - H / 2) ** 2 < r * r).sum()
    assert cand > 1024                                                # the centre pixel's segment
    _check_against_oracle(pts, feats, cam, (H, W), radius, 8)


def _mc_scene(N=2):
    sdf = synth.sphere_sdf_grid(res=49, num=8, seed=3, device=DEV)
    step = 2.0 / 48
    v, _ = ops.mc_gpu(sdf, step, step, step, -1.0, -1.0, -1.0)
    _, deformer = mg.surface_scene(_Mods, _Mods, device="cpu")
    deformer = deformer.to(DEV)
    poses, trans = synth.poses_trans(N, seed=11)
    conds = torch.randn((N, 128), generator=synth.generator(5)) * 0.1
    defconds = [conds.to(DEV), [poses.to(DEV), trans.to(DEV)]]
    return v, deformer, defconds


def test_deformed_marching_cubes_vertices_at_512():
    v, deformer, defconds = _mc_scene()
    with torch.no_grad():
        dv = deformer(v[None].expand(2, -1, 3), defconds, ratio=RATIO, offset_type="body").contiguous()
    S = 512
    cam = _camera(np.eye(3), [0.0, 0.0, 2.4], fx=1.2 * S, fy=1.2 * S, px=(S - 1) / 2, py=(S - 1) / 2)
    feats = torch.ones((v.shape[0], 1), device=DEV)
    _check_against_oracle(dv, feats, cam, (S, S), 0.006, 50, min_covered=5000)


def test_points_renderer_split_matches_single_channel_composites():
    v, deformer, defconds = _mc_scene()
    with torch.no_grad():
        dv = deformer(v[None].expand(2, -1, 3), defconds, ratio=RATIO, offset_type="body").contiguous()
    V = v.shape[0]
    split = V // 3
    cam = _camera(np.eye(3), [0.0, 0.0, 2.4])
    pr = render.PointsRenderer(cam, (H, W), 0.03)
    (up, lo), fr = pr(list(dv), split_size=split, all_size=V)
    upper = (torch.arange(V, device=DEV) < split).float()[:, None]
    up1, fr1 = ops.rasterize_points(dv, upper, cam, (H, W), 0.03, 50)
    lo1, _ = ops.rasterize_points(dv, (1 - upper).contiguous(), cam, (H, W), 0.03, 50)
    assert up.shape == (2, H, W, 1) and torch.equal(up, up1) and torch.equal(lo, lo1)
    assert (up > 0).any() and (lo > 0).any() and torch.equal(fr.idx, fr1.idx)

    class Clouds:                                                     # duck-typed Pointclouds
        def points_list(self):
            return list(dv)

    ones, _ = pr(Clouds())
    assert ones.shape == (2, H, W, 1) and (ones - (up + lo)).abs().max() < 1e-6
    pr.camera = _camera(np.eye(3), [0.05, 0.0, 2.4])                  # settable, as the training step reassigns it
    moved, _ = pr(dv)
    assert not torch.equal(moved, ones) and pr.radius == 0.03
    with pytest.raises(RuntimeError):                                 # non-contiguous input
        ops.rasterize_points(dv.transpose(0, 1), upper, cam, (H, W), 0.03)
    with pytest.raises(RuntimeError):                                 # CPU input: no fallback
        ops.rasterize_points(dv.cpu(), upper.cpu(), cam, (H, W), 0.03)


def _iou_loss(imgs, gt):
    """The reference's mask loss (OptimGarmentNetwork.py:621-629)."""
    N = gt.shape[0]
    m = imgs[..., -1]
    return (1. - (m * gt).view(N, -1).sum(1) / (m + gt - m * gt).abs().view(N, -1).sum(1)).mean()


def test_mask_loss_chain_through_the_deformer_training_path():
    v, deformer, defconds = _mc_scene()
    V = v.shape[0]
    split = V // 2
    cam = _camera(np.eye(3), [0.0, 0.0, 2.4])
    rows, cols = torch.meshgrid(torch.arange(H, device=DEV), torch.arange(W, device=DEV), indexing="ij")
    gts = [(((rows - 30.0) ** 2 + (cols - 44.0) ** 2) < 18.0 ** 2).float()[None].expand(2, H, W),
           (((rows - 36.0) ** 2 + (cols - 52.0) ** 2) < 14.0 ** 2).float()[None].expand(2, H, W)]
    upper = (torch.arange(V, device=DEV) < split).double()[:, None]

    def chain(composite):
        cv = v.detach().clone().requires_grad_(True)
        dv = deformer(cv[None].expand(2, -1, 3), defconds, ratio=RATIO, offset_type="body")
        masks = composite(dv)
        loss = sum(_iou_loss(m, gt) for m, gt in zip(masks, gts))
        loss.backward()
        return loss.item(), cv.grad

    pr = render.PointsRenderer(cam, (H, W), 0.03)
    frags = []

    def kernel(dv):
        masks, fr = pr(list(dv), split_size=split, all_size=V)
        frags.append(fr)
        return masks

    def reference(dv):
        f = torch.cat([upper, 1 - upper], 1)
        img = po.composite_given(dv, f, frags[0].idx, _np_camera(cam), (H, W), 0.03)
        return [img[..., :1], img[..., 1:]]

    loss, grad = chain(kernel)
    loss64, grad64 = chain(reference)
    err = (grad - grad64.float()).abs().max().item()
    print(f"chain: loss {loss:.6f} vs {loss64:.6f}, max |g - g64| {err:.3e}, max |g64| {grad64.abs().max().item():.3e}")
    assert abs(loss - loss64) < 1e-5 and grad64.abs().max() > 0 and err <= 1e-4 * grad64.abs().max().item()
    ops.check_async_errors()
