"""Float64 brute-force rasteriser: the definition `recmv_rasterize` (csrc/raster.cu) is tested against.

Our restatement of the reference camera (model/CameraMine.py): `project` (:169-173) Xc = Xw R + T, x = px - fx Xc/Zc,
y = py - fy Yc/Zc; `view_rays` (:146-167) for pixel (row, col) the world direction of ((px - col)/fx, (py - row)/fy, 1)
rotated by R^T; `cam_pos` (:207-208) = -R T.  Every pixel's ray is intersected with every face (Moller-Trumbore in world
space).  A face covers the pixel when the hit's barycentrics are all > 0 and its three vertices have Zc > 0 -- for Zc > 0 the
signs of the perspective-correct barycentrics are those of the screen-space ones, so this is the screen-space rule; a face of
zero screen area lies in a plane through the camera and is never hit at a positive depth.  The covering face with the
smallest Zc wins, an exact tie goes to the smallest face index.  NumPy only.
"""
import numpy as np


def cam_pos(R, T):
    """-R T (CameraMine.cam_pos) for one camera: R [3,3], T [3]."""
    return -np.asarray(R, np.float64) @ np.asarray(T, np.float64)


def view_rays(cols, rows, fx, fy, px, py, R):
    """CameraMine.view_rays of the pixel centres (col, row, 1): unit world directions [P,3]."""
    d = np.stack([(px - np.asarray(cols, np.float64)) / fx, (py - np.asarray(rows, np.float64)) / fy,
                  np.ones(np.shape(cols))], axis=1)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    return d @ np.asarray(R, np.float64).T


def project(X, R, T, fx, fy, px, py):
    """CameraMine.project with the depth kept: [P,3] world -> (x, y, Zc) each [P]."""
    Xc = np.asarray(X, np.float64) @ np.asarray(R, np.float64) + np.asarray(T, np.float64)
    return px - fx * Xc[:, 0] / Xc[:, 2], py - fy * Xc[:, 1] / Xc[:, 2], Xc[:, 2]


def _frame(V, faces, fx, fy, px, py, R, T, H, W, chunk):
    R = np.asarray(R, np.float64)
    T = np.asarray(T, np.float64)
    tri = np.asarray(V, np.float64)[faces]                         # [F,3,3]
    F = tri.shape[0]
    zc = (tri @ R + T)[..., 2]                                     # [F,3] vertex depths
    front = (zc > 0).all(1)
    o = cam_pos(R, T)
    v0, e1, e2 = tri[:, 0], tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]
    s = o[None] - v0                                               # [F,3]
    # hit o + t d = v0 + u e1 + v e2; the pixel-independent factors of Moller-Trumbore's triple products:
    q = np.cross(s, e1)                                            # v det = d . (s x e1)
    a = np.cross(e2, e1)                                          # det  = d . (e2 x e1)   (= e1 . (d x e2))
    b = np.cross(e2, s)                                            # u det = d . (e2 x s)   (= s . (d x e2))
    tnum = (e2 * q).sum(1)                                         # t det = e2 . (s x e1)
    rows, cols = np.divmod(np.arange(H * W), W)
    out_f = np.full(H * W, -1, np.int64)
    out_b = np.full((H * W, 3), -1.0)
    out_z = np.full(H * W, -1.0)
    amb = np.zeros(H * W, bool)
    for c0 in range(0, H * W, chunk):
        sl = slice(c0, min(c0 + chunk, H * W))
        d = view_rays(cols[sl], rows[sl], fx, fy, px, py, R)        # [P,3]
        det = d @ a.T                                              # [P,F]
        with np.errstate(divide="ignore", invalid="ignore"):
            inv = 1.0 / det
            u = (d @ b.T) * inv
            v = (d @ q.T) * inv
            w0 = 1.0 - u - v
            t = tnum[None] * inv
        # (w0, u, v) are the perspective-correct barycentrics; Zc of the hit is linear in them (camera space), the
        # screen-space barycentrics are b_i = bp_i Zc_i / Zc
        valid = (det != 0) & front[None] & (t > 0)
        zhit = w0 * zc[None, :, 0] + u * zc[None, :, 1] + v * zc[None, :, 2]
        with np.errstate(divide="ignore", invalid="ignore"):
            sbmin = np.minimum(np.minimum(w0 * zc[None, :, 0], u * zc[None, :, 1]), v * zc[None, :, 2]) / zhit
        cover = valid & (w0 > 0) & (u > 0) & (v > 0)
        z = np.where(cover, zhit, np.inf)
        win = np.argmin(z, axis=1)                                 # first minimum = smallest face index
        idx = np.arange(z.shape[0])
        zw = z[idx, win]
        hit = np.isfinite(zw)
        bw = np.stack([w0[idx, win], u[idx, win], v[idx, win]], 1)
        z2 = z.copy()
        z2[idx, win] = np.inf
        second = z2.min(1)
        # a face whose smallest screen-space barycentric is within 1e-4 of 0 and that lies in front of the winner (or in
        # front of nothing) decides the pixel by rounding; so does a second covering face at the winner's depth
        border = valid & (np.abs(sbmin) < 1e-4) & (zhit <= np.where(hit, zw * (1 + 1e-5), np.inf)[:, None])
        with np.errstate(invalid="ignore"):            # inf - inf where fewer than two faces cover
            ambig = border.any(1) | (hit & (np.abs(second - zw) < 1e-5 * zw))
        pix = np.arange(sl.start, sl.stop)[hit]
        out_f[pix] = win[hit]
        out_b[pix] = bw[hit]
        out_z[pix] = zw[hit]
        amb[sl] = ambig
    return out_f.reshape(H, W), out_z.reshape(H, W), out_b.reshape(H, W, 3), amb.reshape(H, W), F


def rasterize(verts, faces, camera, image_size, chunk=None):
    """verts [N,V,3] or [V,3], faces [F,3], camera = (fx, fy, px, py, R [NR,3,3] or [3,3], T [NR,3] or [3]) with NR = 1
    or N, image_size = (H, W).  Returns (pix_to_face [N,H,W,1] int64 (packed n*F + f), zbuf [N,H,W,1], bary_coords
    [N,H,W,1,3] (perspective-correct, vertex order of the face), ambiguous [N,H,W] bool), -1 on background.  A pixel is
    ambiguous when fp32 arithmetic may decide it differently: the winner's smallest screen-space barycentric is < 1e-4,
    the two nearest covering depths differ by < 1e-5 relative, or a face in front of the winner (or in front of nothing,
    on background) misses the pixel centre by less than 1e-4 in screen-space barycentrics."""
    verts = np.asarray(verts, np.float64)
    if verts.ndim == 2:
        verts = verts[None]
    faces = np.asarray(faces, np.int64)
    fx, fy, px, py, R, T = camera
    R = np.asarray(R, np.float64).reshape(-1, 3, 3)
    T = np.asarray(T, np.float64).reshape(-1, 3)
    H, W = image_size
    N = verts.shape[0]
    chunk = chunk or max(16, 2_000_000 // max(len(faces), 1))    # [pixels, faces] float64 temporaries of ~16 MB
    outs = []
    for n in range(N):
        c = 0 if R.shape[0] == 1 else n
        f, z, b, a, F = _frame(verts[n], faces, float(fx), float(fy), float(px), float(py), R[c], T[c], H, W, chunk)
        outs.append((np.where(f >= 0, f + n * F, -1), z, b, a))
    p2f, zbuf, bary, amb = (np.stack(x) for x in zip(*outs))
    return p2f[..., None], zbuf[..., None], bary[:, :, :, None, :], amb
