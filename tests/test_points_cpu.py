"""CPU: the float64 points-rasteriser oracle (oracle/points_oracle.py) on hand-built cases, the pixel convention written
out in pytorch3d's NDC terms, the given-selection composite and its gradient, and the host-side argument checks of
recmv_points_* / ops.rasterize_points / render.PointsRenderer."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import points_oracle as po
from recmv_b200 import _lib, ops, render

# camera at the origin looking down +z: screen x = 4 - 8 X/Z, y = 4 - 8 Y/Z; 8 x 8 image
H = W = 8
CAM = (8.0, 8.0, 4.0, 4.0, np.eye(3), np.zeros(3))
RADIUS = 0.375            # r = 0.375 * 8 / 2 = 1.5 pixels, exact in float32
R2 = 1.5 ** 2


def _world(x, y, z):
    """World point whose projection through CAM is the screen point (x, y) at depth z."""
    return [(4.0 - x) * z / 8.0, (4.0 - y) * z / 8.0, z]


def _run(pts, K=4, feats=None, radius=RADIUS, cam=CAM, size=(H, W)):
    pts = np.asarray(pts, np.float64)[None]                        # one cloud
    feats = np.ones((pts.shape[1], 1)) if feats is None else feats
    return po.rasterize_points(pts, feats, cam, size, radius, K)


def test_one_centred_point():
    idx, zbuf, dists, img, amb = _run([_world(3, 2, 2.0)])
    # pixel (row 2, col 3) is the point's own centre: weight 1; the pixels at distance 1 and sqrt 2 are covered
    assert idx[0, 2, 3, 0] == 0 and img[0, 2, 3, 0] == 1.0 and dists[0, 2, 3, 0] == 0.0 and zbuf[0, 2, 3, 0] == 2.0
    assert np.isclose(img[0, 2, 4, 0], 1 - 1 / R2) and np.isclose(img[0, 3, 4, 0], 1 - 2 / R2)
    assert np.isclose(dists[0, 3, 4, 0], 2 * (2 / 8) ** 2)
    covered = idx[0, :, :, 0] >= 0
    assert covered.sum() == 9 and (idx[0, :, :, 1:] == -1).all()
    assert (img[0, ~covered] == 0).all() and (zbuf[0][~covered] == -1).all() and (dists[0][~covered] == -1).all()
    assert not amb.any()


def test_two_overlapping_points_composite_front_to_back():
    near, far = _world(3, 3, 2.0), _world(3.5, 3, 3.0)
    for pts, i_near in (([near, far], 0), ([far, near], 1)):
        idx, zbuf, dists, img, amb = _run(pts)
        a1 = 1 - 0.0 / R2
        a2 = 1 - 0.25 / R2
        assert list(idx[0, 3, 3, :3]) == [i_near, 1 - i_near, -1]
        assert np.allclose(zbuf[0, 3, 3, :2], [2.0, 3.0])
        assert np.isclose(img[0, 3, 3, 0], a1 + (1 - a1) * a2)
        # pixel (3, 4): d^2 = 1 to the near point, 0.25 to the far one
        b1, b2 = 1 - 1 / R2, 1 - 0.25 / R2
        assert np.isclose(img[0, 3, 4, 0], b1 + (1 - b1) * b2)
        assert not amb[0, 3, 3] and not amb[0, 3, 4] and amb[0, 3, 5]     # (3, 5) is exactly r from the far point


def test_k_truncation_keeps_the_nearest():
    pts = [_world(3, 3, z) for z in (4.0, 2.0, 3.0, 5.0)]
    idx, zbuf, _, img, _ = _run(pts, K=2)
    assert list(idx[0, 3, 3]) == [1, 2] and list(zbuf[0, 3, 3]) == [2.0, 3.0]
    assert img[0, 3, 3, 0] == 1.0                                 # weight 1 in front: nothing behind shows
    idx4, _, _, _, _ = _run(pts, K=4)
    assert list(idx4[0, 3, 3]) == [1, 2, 0, 3]
    # an exact depth tie goes to the smaller index and is flagged
    idx, _, _, _, amb = _run([_world(3, 3, 2.0), _world(3.2, 3, 2.0)], K=1)
    assert idx[0, 3, 3, 0] == 0 and amb[0, 3, 3]


def test_points_behind_the_camera_are_skipped():
    behind = [0.0, 0.0, -2.0]                                     # projects to the image centre from behind
    on_plane = [0.1, 0.1, 0.0]
    idx, _, _, img, _ = _run([behind, on_plane])
    assert (idx == -1).all() and (img == 0).all()
    idx, _, _, _, _ = _run([behind, _world(4, 4, 3.0)])
    assert idx[0, 4, 4, 0] == 1 and (idx[..., 0][idx[..., 0] >= 0] == 1).all()


def test_strict_radius_boundary():
    # r = 2 exactly (radius 0.5 at 8 x 8); the point sits on pixel centre (3, 3): (3, 5) is exactly r away
    idx, _, _, img, amb = _run([[0.125, 0.125, 1.0]], radius=0.5)
    assert idx[0, 3, 3, 0] == 0 and idx[0, 3, 4, 0] == 0 and idx[0, 4, 4, 0] == 0
    assert idx[0, 3, 5, 0] == -1 and img[0, 3, 5, 0] == 0 and idx[0, 5, 3, 0] == -1
    assert amb[0, 3, 5] and amb[0, 5, 3] and not amb[0, 3, 3] and not amb[0, 3, 4]


def test_split_channels_are_the_composites_of_masked_features():
    g = np.random.default_rng(2)
    pts = [_world(*g.uniform(1, 7, 2), g.uniform(2, 4)) for _ in range(30)]
    split = 12
    upper = (np.arange(30) < split)[:, None].astype(np.float64)
    _, _, _, both, _ = _run(pts, K=8, feats=np.concatenate([upper, 1 - upper], 1))
    _, _, _, up, _ = _run(pts, K=8, feats=upper)
    _, _, _, lo, _ = _run(pts, K=8, feats=1 - upper)
    _, _, _, ones, _ = _run(pts, K=8)
    assert np.allclose(both[..., :1], up, rtol=0, atol=1e-15) and np.allclose(both[..., 1:], lo, rtol=0, atol=1e-15)
    assert np.allclose(up + lo, ones) and (up > 0).any() and (lo > 0).any()


def test_pixel_convention_matches_pytorch3d_ndc_for_square_images():
    # _get_sfm_calibration_matrix (CameraMine.py:273-287) puts a point with screen x at NDC 1 - (2 x + 1) / W; pytorch3d's
    # pixel (i, j) has its centre at NDC (1 - (2 j + 1) / W, 1 - (2 i + 1) / H).  The NDC distance is then 2 / W times the
    # pixel distance, and pytorch3d's weight 1 - dist_ndc^2 / radius^2 equals the pixel-space 1 - d^2 / r_pix^2.
    g = np.random.default_rng(9)
    n = 40
    S = 16
    fx, fy, px, py = 20.0, 22.0, 7.25, 8.125
    xc = np.stack([g.uniform(-1, 1, n), g.uniform(-1, 1, n), g.uniform(2, 5, n)], 1)
    cam = (fx, fy, px, py, np.eye(3), np.zeros(3))
    radius = 0.3
    K = 6
    idx, _, dists, img, _ = po.rasterize_points(xc, np.ones((n, 1)), cam, (S, S), radius, K)
    sx, sy = px - fx * xc[:, 0] / xc[:, 2], py - fy * xc[:, 1] / xc[:, 2]
    ndc_x, ndc_y = 1 - (2 * sx + 1) / S, 1 - (2 * sy + 1) / S
    r32 = float(np.float32(radius))
    want = np.zeros((S, S))
    for i in range(S):
        for j in range(S):
            cx, cy = 1 - (2 * j + 1) / S, 1 - (2 * i + 1) / S
            d = (ndc_x - cx) ** 2 + (ndc_y - cy) ** 2
            sel = [p for p in np.argsort(xc[:, 2], kind="stable") if d[p] < r32 ** 2][:K]
            assert list(idx[0, i, j][:len(sel)]) == sel and (idx[0, i, j][len(sel):] == -1).all()
            assert np.allclose(dists[0, i, j][:len(sel)], d[sel], rtol=1e-12, atol=1e-15)
            t = 1.0
            for p in sel:
                a = 1 - d[p] / r32 ** 2
                want[i, j] += t * a
                t *= 1 - a
    assert np.allclose(img[0, :, :, 0], want, atol=1e-12) and (want > 0).sum() > 50


def test_composite_given_matches_the_oracle_and_has_the_finite_difference_gradient():
    g = np.random.default_rng(4)
    N, P = 2, 25
    Rs = np.stack([np.eye(3), np.array([[0.8, 0, 0.6], [0, 1, 0], [-0.6, 0, 0.8]])])
    Ts = np.array([[0.0, 0.0, 0.0], [0.1, -0.1, 0.3]])
    pts = np.stack([np.stack([_world(*g.uniform(1, 7, 2), g.uniform(2, 4)) for _ in range(P)]) for _ in range(N)])
    pts[1] = (pts[1] - Ts[1]) @ Rs[1].T                           # the same camera-space cloud seen by camera 1
    feats = np.stack([np.ones(P), g.uniform(0, 1, P)], 1)
    cam = (8.0, 8.0, 4.0, 4.0, Rs, Ts)
    idx, _, _, img, _ = po.rasterize_points(pts, feats, cam, (H, W), RADIUS, 5)
    assert (idx[1] >= P).sum() == (idx[1] >= 0).sum() > 20        # packed n * P + p
    t = torch.tensor(pts, requires_grad=True)
    out = po.composite_given(t, feats, idx, cam, (H, W), RADIUS)
    assert np.allclose(out.detach().numpy(), img, atol=1e-12)
    assert torch.autograd.gradcheck(lambda x: po.composite_given(x, feats, idx, cam, (H, W), RADIUS), (t,))


def test_points_argument_checks_without_gpu():
    lib = _lib.load()
    nbytes = ctypes.c_size_t(0)
    assert lib.recmv_points_scratch_bytes(2, 1000, 96, 64, ctypes.byref(nbytes)) == 0
    assert nbytes.value >= 2 * 1000 * 28 + 2 * 96 * 64 * 12
    assert lib.recmv_points_scratch_bytes(0, 1000, 96, 64, ctypes.byref(nbytes)) == -3
    assert lib.recmv_points_scratch_bytes(1, 1000, 96, 64, None) == -1
    assert lib.recmv_points_scratch_bytes(2, 1 << 31, 96, 64, ctypes.byref(nbytes)) == -4   # packed index > 32 bits
    assert lib.recmv_points_scratch_bytes(1, 10, 1 << 16, 1 << 16, ctypes.byref(nbytes)) == -4
    cam = (ctypes.c_float * 4)(1, 1, 0, 0)
    p = ctypes.c_void_p(16)   # never dereferenced: every call below fails validation first
    total = ctypes.c_int64(0)
    cnt = lambda N, P, cm, NR, r, tot: lib.recmv_points_count(p, N, P, cm, p, p, NR, 8, 8, r, p, tot, None)  # noqa: E731
    assert cnt(1, 10, cam, 1, 0.1, None) == -1
    assert cnt(1, 10, None, 1, 0.1, ctypes.byref(total)) == -1
    assert cnt(2, 10, cam, 3, 0.1, ctypes.byref(total)) == -3     # NR not in {1, N}
    assert cnt(1, 0, cam, 1, 0.1, ctypes.byref(total)) == -3
    assert cnt(1, 10, cam, 1, 0.0, ctypes.byref(total)) == -3     # radius must be > 0
    assert cnt(1, 10, cam, 1, float("nan"), ctypes.byref(total)) == -3
    assert cnt(1, 10, cam, 1, float("inf"), ctypes.byref(total)) == -3
    ren = lambda C, K, cand, tot: lib.recmv_points_render(p, C, 1, 10, 8, 8, 0.1, K, p, cand, tot, p, None)  # noqa: E731
    assert ren(0, 8, p, 5) == -3 and ren(5, 8, p, 5) == -3        # 1 <= C <= 4
    assert ren(1, 0, p, 5) == -3 and ren(1, 65, p, 5) == -3       # 1 <= K <= 64
    assert ren(1, 8, p, -1) == -3 and ren(1, 8, p, 1 << 31) == -4
    assert ren(1, 8, None, 5) == -1
    bwd = lambda C, K, NR: lib.recmv_points_render_backward(p, 1, 10, cam, p, p, NR, 8, 8, 0.1, p, C, K, p, p, p, p, None)  # noqa: E731,E501
    assert bwd(5, 8, 1) == -3 and bwd(1, 65, 1) == -3 and bwd(1, 8, 2) == -3
    assert lib.recmv_points_render_backward(p, 1, 10, cam, p, p, 1, 8, 8, 0.1, p, 1, 8, p, p, None, p, None) == -1
    assert lib.recmv_points_fragments(1, 10, 8, 8, 0.1, 0, p, p, p, p, p, None) == -3
    assert lib.recmv_points_fragments(1, 10, 8, 8, 0.1, 8, p, p, None, p, p, None) == -1


def test_rasterize_points_rejects_cpu_tensors_and_feature_gradients():
    pts = torch.randn(1, 6, 3)
    cam = (1.0, 1.0, 0.0, 0.0, torch.eye(3), torch.zeros(3))
    with pytest.raises(RuntimeError):
        ops.rasterize_points(pts, torch.ones(6, 1), cam, (8, 8), 0.1)
    with pytest.raises(RuntimeError, match="features"):
        ops.rasterize_points(pts, torch.ones(6, 1, requires_grad=True), cam, (8, 8), 0.1)
    pr = render.PointsRenderer(cam, (8, 8), 0.1)
    assert pr.radius == 0.1 and pr.points_per_pixel == 50
    with pytest.raises(RuntimeError):                             # no CPU fallback
        pr([torch.randn(6, 3), torch.randn(6, 3)])
    with pytest.raises(RuntimeError, match="all_size"):
        pr(pts, split_size=2, all_size=4)
