"""CPU: the float64 rasteriser oracle (oracle/raster_oracle.py) on hand-built cases, the consistency of its hits with the
camera functions it restates, and the host-side argument checks of recmv_rasterize / ops.rasterize."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import raster_oracle as ro
from recmv_b200 import _lib, ops

# camera at the origin looking down +z: screen x = 5 - 10 X/Z, y = 5 - 10 Y/Z
CAM = (10.0, 10.0, 5.0, 5.0, np.eye(3), np.zeros(3))
H, W = 10, 10


def _world(x, y, z):
    """World point whose projection through CAM is the screen point (x, y) at depth z."""
    return [(5.0 - x) * z / 10.0, (5.0 - y) * z / 10.0, z]


def _tri(z, screen=((0.5, 0.5), (7.7, 0.5), (0.5, 7.7))):
    return [_world(x, y, z) for x, y in screen]


def _hand_mask():
    # screen triangle (0.5,0.5) (7.7,0.5) (0.5,7.7): the pixel centres inside have col >= 1, row >= 1, col + row <= 8
    # (nearest centre to an edge: 0.2 / sqrt2 px off the hypotenuse)
    m = np.zeros((H, W), bool)
    for r in range(H):
        for c in range(W):
            m[r, c] = c >= 1 and r >= 1 and c + r <= 8
    return m


def test_single_triangle_against_hand_computed_pixels():
    p2f, zbuf, bary, amb = ro.rasterize(np.array(_tri(2.0)), np.array([[0, 1, 2]]), CAM, (H, W))
    m = _hand_mask()
    assert m.sum() == 28
    assert np.array_equal(p2f[0, :, :, 0] == 0, m) and (p2f[0, :, :, 0][~m] == -1).all()
    assert np.allclose(zbuf[0, :, :, 0][m], 2.0, atol=1e-12) and (zbuf[0, :, :, 0][~m] == -1).all()
    assert (bary[0, :, :, 0][~m] == -1).all()
    for r, c in zip(*np.nonzero(m)):
        # constant depth: perspective-correct = screen-space barycentrics, b1 = (col - 0.5) / 7.2, b2 = (row - 0.5) / 7.2
        want = [1 - (c - 0.5) / 7.2 - (r - 0.5) / 7.2, (c - 0.5) / 7.2, (r - 0.5) / 7.2]
        assert np.allclose(bary[0, r, c, 0], want, atol=1e-12)
    assert not amb.any()
    # tilted face: perspective-correct barycentrics interpolate camera-space points along the ray
    tri = np.array([_world(0.5, 0.5, 2.0), _world(7.7, 0.5, 4.0), _world(0.5, 7.7, 3.0)])
    p2f, zbuf, bary, _ = ro.rasterize(tri, np.array([[0, 1, 2]]), CAM, (H, W))
    assert np.array_equal(p2f[0, :, :, 0] == 0, m)
    b = bary[0, 3, 2, 0]
    assert np.isclose(b @ tri[:, 2], zbuf[0, 3, 2, 0]) and not np.allclose(b, [1 - 4 / 7.2, 1.5 / 7.2, 2.5 / 7.2])


def test_overlapping_triangles_nearest_wins_and_ties_go_to_the_smaller_index():
    m = _hand_mask()
    # same screen triangle at depth 3 (face 0) and 2 (face 1), then the order swapped
    verts = np.array(_tri(3.0) + _tri(2.0))
    for faces, near in ((np.array([[0, 1, 2], [3, 4, 5]]), 1), (np.array([[3, 4, 5], [0, 1, 2]]), 0)):
        p2f, zbuf, _, amb = ro.rasterize(verts, faces, CAM, (H, W))
        assert (p2f[0, :, :, 0][m] == near).all() and np.allclose(zbuf[0, :, :, 0][m], 2.0)
        assert not amb.any()
    # an exactly equal depth: the smaller face index, flagged ambiguous
    p2f, _, _, amb = ro.rasterize(np.array(_tri(2.0)), np.array([[0, 1, 2], [0, 1, 2]]), CAM, (H, W))
    assert (p2f[0, :, :, 0][m] == 0).all() and amb[0][m].all()
    # two frames: the packed index is n * F + f
    p2f, _, _, _ = ro.rasterize(np.stack([verts, verts]), np.array([[0, 1, 2], [3, 4, 5]]), CAM, (H, W))
    assert (p2f[1, :, :, 0][m] == 2 + 1).all()


def test_back_facing_face_counts():
    p2f, _, bary, _ = ro.rasterize(np.array(_tri(2.0)), np.array([[0, 2, 1]]), CAM, (H, W))
    m = _hand_mask()
    assert np.array_equal(p2f[0, :, :, 0] == 0, m)
    r, c = 3, 2                                      # bary in the face's own vertex order (0, 2, 1)
    assert np.allclose(bary[0, r, c, 0], [1 - (c - 0.5) / 7.2 - (r - 0.5) / 7.2, (r - 0.5) / 7.2, (c - 0.5) / 7.2])


def test_face_with_a_vertex_behind_the_camera_is_skipped():
    tri = _tri(2.0)
    tri[2] = [tri[2][0], tri[2][1], -1.0]
    p2f, zbuf, bary, _ = ro.rasterize(np.array(tri), np.array([[0, 1, 2]]), CAM, (H, W))
    assert (p2f == -1).all() and (zbuf == -1).all() and (bary == -1).all()
    # ... and does not hide a visible face behind it
    verts = np.array(tri + _tri(4.0))
    p2f, _, _, _ = ro.rasterize(verts, np.array([[0, 1, 2], [3, 4, 5]]), CAM, (H, W))
    assert (p2f[0, :, :, 0][_hand_mask()] == 1).all()


def test_zero_area_faces_are_skipped():
    # a repeated vertex, and three distinct collinear screen points (a face seen edge-on)
    degenerate = np.array(_tri(2.0) + [_world(1, 1, 2.0), _world(4, 4, 3.0), _world(7, 7, 2.5)])
    p2f, _, _, _ = ro.rasterize(degenerate, np.array([[0, 1, 1], [3, 4, 5]]), CAM, (H, W))
    assert (p2f == -1).all()


def test_pixel_centres_on_or_near_an_edge_are_flagged():
    # screen triangle (1,1) (7,1) (1,7): its edges pass through pixel centres, where the sign of a zero barycentric is
    # rounding; such a pixel is either not covered or covered and flagged ambiguous, the centres inside are neither
    p2f, _, _, amb = ro.rasterize(np.array(_tri(2.0, ((1, 1), (7, 1), (1, 7)))), np.array([[0, 1, 2]]), CAM, (H, W))
    rr, cc = np.mgrid[0:H, 0:W]
    inside = (cc > 1) & (rr > 1) & (cc + rr < 8)
    edge = ((cc == 1) & (rr >= 1) & (rr <= 7)) | ((rr == 1) & (cc >= 1) & (cc <= 7)) | ((cc + rr == 8) & (cc >= 1) & (rr >= 1))
    cov = p2f[0, :, :, 0] == 0
    assert (cov[inside] & ~amb[0][inside]).all() and not cov[~inside & ~edge].any()
    assert (~cov[edge] | amb[0][edge]).all()
    # a pixel 1e-6 px inside an edge is covered but ambiguous
    shifted = [_world(1 - 1e-6, 0.5, 2.0), _world(7.7, 0.5, 2.0), _world(1 - 1e-6, 7.7, 2.0)]
    p2f, _, _, amb = ro.rasterize(np.array(shifted), np.array([[0, 1, 2]]), CAM, (H, W))
    assert p2f[0, 3, 1, 0] == 0 and amb[0, 3, 1] and not amb[0, 3, 3]


def test_hits_lie_on_the_view_rays_and_project_back():
    g = np.random.default_rng(5)
    F = 60
    centres = g.uniform([-0.8, -0.6, 2.0], [0.8, 0.6, 4.0], (F, 1, 3))
    verts = (centres + g.normal(0, 0.25, (F, 3, 3))).reshape(-1, 3)
    faces = np.arange(3 * F).reshape(F, 3)
    ang = 0.2
    R = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]])
    T = np.array([0.3, -0.1, 0.4])
    fx, fy, px, py = 40.0, 44.0, 23.5, 15.2
    h, w = 32, 48
    p2f, zbuf, bary, amb = ro.rasterize(verts, faces, (fx, fy, px, py, R, T), (h, w))
    hit = p2f[0, :, :, 0] >= 0
    assert hit.sum() > 200 and amb.sum() < hit.sum()
    rows, cols = np.nonzero(hit)
    f = p2f[0, rows, cols, 0]
    P = (bary[0, rows, cols, 0][:, :, None] * verts[faces[f]]).sum(1)
    o = ro.cam_pos(R, T)
    d = ro.view_rays(cols, rows, fx, fy, px, py, R)
    off = P - o
    assert np.abs(np.cross(off, d)).max() < 1e-9 and ((off * d).sum(1) > 0).all()
    x, y, z = ro.project(P, R, T, fx, fy, px, py)
    assert np.abs(z - zbuf[0, rows, cols, 0]).max() < 1e-9
    assert np.abs(x - cols).max() < 1e-9 and np.abs(y - rows).max() < 1e-9


def test_rasterize_argument_checks_without_gpu():
    lib = _lib.load()
    nbytes = ctypes.c_size_t(0)
    assert lib.recmv_raster_scratch_bytes(2, 96, 64, ctypes.byref(nbytes)) == 0 and nbytes.value == 2 * 96 * 64 * 8
    assert lib.recmv_raster_scratch_bytes(0, 96, 64, ctypes.byref(nbytes)) == -3
    cam = (ctypes.c_float * 4)(1, 1, 0, 0)
    p = ctypes.c_void_p(16)   # never dereferenced: every call below fails validation first
    args = lambda N, V, F, cm, NR, Hh, Ww: (p, p, N, V, F, cm, p, p, NR, Hh, Ww, p, p, p, p, None)  # noqa: E731
    assert lib.recmv_rasterize(None, p, 1, 3, 1, cam, p, p, 1, 4, 4, p, p, p, p, None) == -1
    assert lib.recmv_rasterize(*args(1, 3, 1, None, 1, 4, 4)) == -1
    assert lib.recmv_rasterize(*args(2, 3, 1, cam, 3, 4, 4)) == -3      # NR not in {1, N}
    assert lib.recmv_rasterize(*args(1, 0, 1, cam, 1, 4, 4)) == -3
    assert lib.recmv_rasterize(*args(1, 3, 0, cam, 1, 4, 4)) == -3
    assert lib.recmv_rasterize(*args(1, 3, 1, cam, 1, 0, 4)) == -3
    assert lib.recmv_rasterize(*args(1, 3, 1 << 33, cam, 1, 4, 4)) == -4


def test_rasterize_rejects_cpu_tensors():
    verts = torch.randn(1, 6, 3)
    faces = torch.tensor([[0, 1, 2], [3, 4, 5]])
    with pytest.raises(RuntimeError):
        ops.rasterize(verts, faces, (1.0, 1.0, 0.0, 0.0, torch.eye(3), torch.zeros(3)), (8, 8))
