"""Float64 brute-force points rasteriser + alpha compositor: the definition `recmv_points_*` (csrc/points.cu) is tested
against.

Our restatement of what `pcRender` gets from pytorch3d's PointsRasterizer + AlphaCompositor (model/CameraMine.py:306-415),
in the reference camera's convention (CameraMine.py:169-173, `raster_oracle.project`): Xc = Xw R + T, screen
x = px - fx Xc/Zc, y = py - fy Yc/Zc, pixel (row i, col j) is the screen point (j, i).  Point p covers pixel (i, j) when
Zc > 0 and d^2 = (x - j)^2 + (y - i)^2 < r^2 with r = radius min(H, W) / 2 (radius in NDC units; it and the camera
intrinsics are taken as the float32 values the kernel receives).  Per pixel the K covering points with the smallest Zc
are kept, ascending, ties to the smaller packed index n P + p; weight a = 1 - d^2 / r^2; image
I_c = sum_k T_k a_k f[idx_k, c], T_0 = 1, T_{k+1} = T_k (1 - a_k).

`rasterize_points` tests every point against every pixel of its bounding square (a pixel outside it lies at least r away,
so this is the all-pairs test) in NumPy float64.  `composite_given` composites a GIVEN selection (e.g. the kernel's own
fragments) in torch float64, so its autograd gradient is a reference that the ambiguous pixels do not contaminate.
"""
import numpy as np
import torch

from .raster_oracle import project

BOUNDARY_RTOL = 1e-4    # |d^2 - r^2| < BOUNDARY_RTOL r^2: fp32 / fp64 rounding may decide the coverage either way
DEPTH_RTOL = 1e-6       # two covering depths this close may be ordered differently once rounded to fp32


def pixel_radius(radius, image_size):
    H, W = image_size
    return float(np.float32(radius)) * min(H, W) / 2.0


def _cameras(camera, N):
    """Per-frame (fx, fy, px, py, R, T), the intrinsics as the float32 values the kernel receives."""
    fx, fy, px, py, R, T = camera
    fx, fy, px, py = (float(np.float32(v)) for v in (fx, fy, px, py))
    R = np.asarray(R, np.float64).reshape(-1, 3, 3)
    T = np.asarray(T, np.float64).reshape(-1, 3)
    return [(fx, fy, px, py, R[0 if R.shape[0] == 1 else n], T[0 if T.shape[0] == 1 else n]) for n in range(N)]


def rasterize_points(points, features, camera, image_size, radius, K):
    """points [N,P,3] or [P,3], features [P,C], camera = (fx, fy, px, py, R [NR,3,3] or [3,3], T [NR,3] or [3]) with
    NR = 1 or N, image_size = (H, W).  Returns (idx [N,H,W,K] int64 packed n*P + p, zbuf [N,H,W,K] Zc, dists [N,H,W,K]
    = d^2 (2 / min(H, W))^2, images [N,H,W,C], ambiguous [N,H,W] bool), -1 in empty slots.  A pixel is ambiguous when
    fp32 arithmetic may legitimately select differently: a candidate with |d^2 - r^2| < 1e-4 r^2 that is not behind the
    K-th covering point, or two covering depths within 1e-6 relative among the first K + 1."""
    pts = np.asarray(points, np.float64)
    if pts.ndim == 2:
        pts = pts[None]
    feats = np.asarray(features, np.float64)
    N, P = pts.shape[:2]
    H, W = image_size
    r = pixel_radius(radius, image_size)
    r2 = r * r
    reach = int(np.ceil(r * (1 + BOUNDARY_RTOL))) + 1
    oy, ox = (a.ravel() for a in np.mgrid[-reach:reach + 1, -reach:reach + 1])
    idx = np.full((N, H * W, K), -1, np.int64)
    zbuf = np.full((N, H * W, K), -1.0)
    dists = np.full((N, H * W, K), -1.0)
    images = np.zeros((N, H * W, feats.shape[1]))
    amb = np.zeros((N, H * W), bool)
    for n, (fx, fy, px, py, R, T) in enumerate(_cameras(camera, N)):
        with np.errstate(divide="ignore", invalid="ignore"):
            x, y, z = project(pts[n], R, T, fx, fy, px, py)
        front = np.nonzero((z > 0) & np.isfinite(x) & np.isfinite(y))[0]
        cx, cy = np.round(x[front]), np.round(y[front])
        cols = (cx[:, None] + ox[None]).ravel()
        rows = (cy[:, None] + oy[None]).ravel()
        p = np.repeat(front, ox.size)
        inside = (cols >= 0) & (cols < W) & (rows >= 0) & (rows < H)
        cols, rows, p = cols[inside].astype(np.int64), rows[inside].astype(np.int64), p[inside]
        d2 = (x[p] - cols) ** 2 + (y[p] - rows) ** 2
        near = d2 < r2 * (1 + BOUNDARY_RTOL)
        cols, rows, p, d2 = cols[near], rows[near], p[near], d2[near]
        pix = rows * W + cols
        cov = d2 < r2
        # covering candidates sorted by (pixel, Zc, index), ranked within their pixel
        cp, cpix, cd2 = p[cov], pix[cov], d2[cov]
        order = np.lexsort((cp, z[cp], cpix))
        cp, cpix, cd2 = cp[order], cpix[order], cd2[order]
        first = np.searchsorted(cpix, cpix, side="left")
        rank = np.arange(cpix.size) - first
        keep = rank < K
        kp, kpix, krank, kd2 = cp[keep], cpix[keep], rank[keep], cd2[keep]
        idx[n, kpix, krank] = n * P + kp
        zbuf[n, kpix, krank] = z[kp]
        dists[n, kpix, krank] = kd2 * (2.0 / min(H, W)) ** 2
        a = np.zeros((H * W, K))
        a[kpix, krank] = 1.0 - kd2 / r2
        tr = np.cumprod(np.concatenate([np.ones((H * W, 1)), 1.0 - a[:, :-1]], 1), 1)
        f = np.zeros((H * W, K, feats.shape[1]))
        f[kpix, krank] = feats[kp]
        images[n] = ((tr * a)[..., None] * f).sum(1)
        # ambiguity: a near-boundary candidate not behind the K-th covering point ...
        zk = np.full(H * W, np.inf)
        last = rank == K - 1
        zk[cpix[last]] = z[cp[last]]
        band = np.abs(d2 - r2) < BOUNDARY_RTOL * r2
        amb[n, pix[band][z[p[band]] <= zk[pix[band]]]] = True
        # ... or two covering depths within DEPTH_RTOL among the first K + 1
        first_k1 = rank <= K
        zs, ps = z[cp[first_k1]], cpix[first_k1]
        tie = (ps[1:] == ps[:-1]) & (np.abs(zs[1:] - zs[:-1]) < DEPTH_RTOL * zs[:-1])
        amb[n, ps[1:][tie]] = True
    shape = (N, H, W)
    return (idx.reshape(shape + (K,)), zbuf.reshape(shape + (K,)), dists.reshape(shape + (K,)),
            images.reshape(shape + (feats.shape[1],)), amb.reshape(shape))


def composite_given(points, features, idx, camera, image_size, radius):
    """The alpha composite of a given selection in torch float64, differentiable in `points`.  points [N,P,3] (any float
    tensor; promoted to float64), features [P,C], idx [N,H,W,K] packed n*P + p with -1 in empty slots (nearest first),
    camera as rasterize_points.  Returns images [N,H,W,C] float64 on the device of `points`."""
    pts = points.double()
    dev = pts.device
    N, P = pts.shape[:2]
    H, W = image_size
    r2 = pixel_radius(radius, image_size) ** 2
    xs, ys = [], []
    for n, (fx, fy, px, py, R, T) in enumerate(_cameras(camera, N)):
        xc = pts[n] @ torch.as_tensor(R, device=dev) + torch.as_tensor(T, device=dev)
        xs.append(px - fx * xc[:, 0] / xc[:, 2])
        ys.append(py - fy * xc[:, 1] / xc[:, 2])
    sx, sy = torch.cat(xs), torch.cat(ys)
    idx = torch.as_tensor(idx, device=dev)
    valid = idx >= 0
    i = idx.clamp(min=0)
    rows = torch.arange(H, device=dev, dtype=torch.float64)[None, :, None, None]
    cols = torch.arange(W, device=dev, dtype=torch.float64)[None, None, :, None]
    d2 = (sx[i] - cols) ** 2 + (sy[i] - rows) ** 2
    a = torch.where(valid, 1.0 - d2 / r2, torch.zeros_like(d2))
    tr = torch.cumprod(torch.cat([torch.ones_like(a[..., :1]), 1.0 - a[..., :-1]], -1), -1)
    f = torch.as_tensor(features, device=dev, dtype=torch.float64)[i % P] * valid[..., None]
    return ((tr * a)[..., None] * f).sum(-2)
