"""The fused render path as a user-facing object, plus its data-parallel sharding.

`SdfRenderer` owns the device-resident state of one scene (packed SDF weights, channels-last skinning
voxel, skeleton) and exposes

    render(ray_dirs, poses, trans)           device tensors in, device tensors out
    render_host(ray_dirs_pinned, poses, ...) HOST buffers in, HOST result out (H2D + kernels + D2H) --
                                             the call bench.py times as `e2e`

Sharding (`shard_rows`): rays are independent given replicated weights / voxel / bone matrices
(SURVEY 8e), so ranks take contiguous blocks of image rows (or whole frames) and there is NO
data-path collective; gradients -- when training -- are exchanged by `allreduce_grads`.

`MaskRasterizer` / `render_colors`: from a (marching-cubes) mesh to rasteriser fragments and to the colour frame of
`infer_garment`, on the device (`ops.rasterize`, csrc/raster.cu).

`PointsRenderer`: the point-cloud silhouette renderer `pcRender` of the training step's mask loss, on the device and
differentiable in the point positions (`ops.rasterize_points`, csrc/points.cu).
"""
import torch

from . import ops, synth
from .model import LBSkinner, getTmpSdf


def shard_rows(height, rank, world):
    """Contiguous block of image rows for `rank` (first `height % world` ranks get one extra row)."""
    base, extra = divmod(height, world)
    row0 = rank * base + min(rank, extra)
    return row0, base + (1 if rank < extra else 0)


def shard_frames(num_frames, rank, world):
    """Frames a rank owns when there are at least as many frames as ranks."""
    return list(range(rank, num_frames, world))


def allreduce_grads(params, group=None, comm_stream=None):
    """ONE flat fp32 all-reduce (sum) over the gradients of `params` (SDF nets + translator + rendnet;
    deformer + pose only in large-pose mode), issued on `comm_stream` so it overlaps the caller's
    remaining backward work.  Returns a handle whose .wait() scatters the reduced bucket back."""
    import torch.distributed as dist
    grads = [p.grad for p in params if p.grad is not None]
    if not grads or not dist.is_initialized() or dist.get_world_size(group) == 1:
        class _Done:
            def wait(self):
                return None
        return _Done()
    dev = grads[0].device
    flat = torch.cat([g.reshape(-1).float() for g in grads])
    if comm_stream is not None and dev.type == "cuda":
        comm_stream.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(comm_stream):
            work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True)
    else:
        work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group, async_op=True)

    class _Handle:
        def wait(self_inner):
            work.wait()
            if comm_stream is not None and dev.type == "cuda":
                torch.cuda.current_stream(dev).wait_stream(comm_stream)
            off = 0
            for g in grads:
                n = g.numel()
                g.copy_(flat[off:off + n].view_as(g))
                off += n
    return _Handle()


class SdfRenderer:
    """`sdf_net` / `skinner`: an existing `ImplicitNetwork` / `LBSkinner` pair (what `getOptNet` builds,
    model/network.py:204-272) -- the renderer then marches THAT scene; without them a seeded synthetic scene of the
    BASELINE shapes is fabricated (bench / tests).  The packed weight blob is fetched per call from the network's
    version-keyed cache, so an optimizer step or `load_state_dict` between renders is picked up."""

    def __init__(self, device, sdf_net=None, voxel_shape=(65, 225, 129), seed=0, mode=None,
                 samples=64, t_near=synth.T_NEAR, t_far=synth.T_FAR, cam_pos=synth.CAM_POS, skinner=None):
        self.device = torch.device(device)
        self.mode = ops.DEFAULT_MLP_MODE if mode is None else mode
        self.samples, self.t_near, self.t_far, self.cam_pos = samples, t_near, t_far, cam_pos
        if sdf_net is None:
            torch.manual_seed(seed)
            sdf_net = getTmpSdf(self.device, 6, 0.6, 256)
        self.sdf_net = sdf_net
        if skinner is None:
            Js, parents, init = synth.skeleton()
            ws = synth.skinning_voxel(voxel_shape, seed=7, device=self.device)
            skinner = LBSkinner(ws, [-1.1] * 3, [1.1] * 3, Js, parents, init_pose=init,
                                bbox_extend=torch.tensor(synth.BBOX_EXTEND),
                                bbox_center=torch.tensor(synth.BBOX_CENTER)).to(self.device)
        self.skinner = skinner
        self.pe_w = [1.0] * 12
        self._sdf_buf = None

    @property
    def ws_cl(self):
        return self.skinner.ws_channels_last()

    @property
    def packed(self):
        return self.sdf_net.packed_weights()

    def _bbox(self):
        return self.skinner.bbox_host()

    def bone_matrices(self, poses, trans):
        with torch.no_grad():
            A = self.skinner.bone_matrices(poses)
            t = trans + self.skinner.extra_trans
        return A.contiguous(), t.contiguous()

    def render(self, ray_dirs, A, trans, rays_per_frame=0, want_xc=False):
        R = ray_dirs.shape[0]
        if self._sdf_buf is None or self._sdf_buf.shape[0] != R:
            self._sdf_buf = torch.empty((R, self.samples), dtype=torch.float32, device=self.device)
        center, extend = self._bbox()
        return ops.render_sdf(ray_dirs, self.cam_pos, self.t_near, self.t_far, self.samples, A, trans,
                              self.ws_cl, center, extend, self.packed, self.pe_w,
                              self.mode, None, rays_per_frame or R, want_xc, True, self._sdf_buf)

    def render_host(self, ray_dirs_pinned, A_pinned, trans_pinned, out_hit_t_pinned, out_hit_idx_pinned,
                    rays_per_frame=0):
        """End-to-end call on HOST buffers (pinned): H2D inputs, fused render, D2H per-ray result."""
        d = ray_dirs_pinned.to(self.device, non_blocking=True)
        A = A_pinned.to(self.device, non_blocking=True)
        t = trans_pinned.to(self.device, non_blocking=True)
        _, _, hit_idx, hit_t = self.render(d, A, t, rays_per_frame=rays_per_frame)
        out_hit_t_pinned.copy_(hit_t, non_blocking=True)
        out_hit_idx_pinned.copy_(hit_idx, non_blocking=True)
        return out_hit_t_pinned, out_hit_idx_pinned


    # ---- full per-ray render: sdf march -> surface point -> normal -> colour --------------------------------
    def surface_points(self, ray_dirs, A, trans, frame_of_ray=None, refine=3):
        """Observation-space surface point per ray: first sign change of the 64-sample march, then `refine`
        secant steps on the bracketing interval (each step = one inverse-LBS launch + one fused SDF launch on
        the hit rays only).  Returns (hit mask [R], t [R], x_obs [R,3], x_can [R,3], sdf at the point [R])."""
        R = ray_dirs.shape[0]
        rpf = 0 if frame_of_ray is not None else R // max(int(A.shape[0]), 1)
        center, extend = self._bbox()
        sdf, _, hit_idx, hit_t = ops.render_sdf(ray_dirs, self.cam_pos, self.t_near, self.t_far, self.samples, A,
                                                trans, self.ws_cl, center, extend,
                                                self.packed, self.pe_w, self.mode, frame_of_ray, rpf, False, True)
        hit = hit_idx > 0
        idx = hit.nonzero(as_tuple=False).view(-1)
        cam = torch.tensor(self.cam_pos, device=self.device, dtype=torch.float32)
        dt = (self.t_far - self.t_near) / self.samples
        k = hit_idx[idx].long()
        t0 = self.t_near + (k.float() - 0.5) * dt          # sample k-1 (outside) .. sample k (inside)
        t1 = t0 + dt
        s0 = sdf[idx, k - 1]
        s1 = sdf[idx, k]
        d = ray_dirs[idx]
        frames = (frame_of_ray[idx].long() if frame_of_ray is not None
                  else torch.div(idx, max(rpf, 1), rounding_mode="floor").clamp_max(A.shape[0] - 1))

        def eval_at(t):
            xo = cam[None] + t[:, None] * d
            xc, ok = ops.lbs_inverse(xo, A, trans, self.ws_cl, center, extend, frames, 0)
            v = ops.sdf_mlp_forward(xc, self.packed, self.pe_w, self.mode, want_feat=False)[0][:, 0]   # same weights and
            # precision mode as the march (not sdf_net.mlp_mode)
            return xo, xc, torch.where(ok, v, torch.full_like(v, 1e10))
        t = t0 + (t1 - t0) * s0 / (s0 - s1)
        xo, xc, v = eval_at(t)
        for _ in range(refine):
            inside = v <= 0                                  # keep the root bracketed (regula falsi)
            t1 = torch.where(inside, t, t1); s1 = torch.where(inside, v, s1)
            t0 = torch.where(inside, t0, t); s0 = torch.where(inside, s0, v)
            t = t0 + (t1 - t0) * s0 / (s0 - s1)
            xo, xc, v = eval_at(t)
        full = lambda z, fill: torch.full((R,) + z.shape[1:], fill, device=self.device, dtype=z.dtype).index_copy_(0, idx, z)  # noqa: E731
        return hit, full(t, 0.0), full(xo, 0.0), full(xc, 0.0), full(v, 0.0)

    def render_image(self, ray_dirs, A, trans, render_net, ratio=None, frame_of_ray=None, refine=3):
        """RGB per ray (background 0): surface point -> canonical normal from the fused value+gradient launch
        (which also returns the 256 features) -> IDR colour MLP on (x_can, normal, view dir, features).
        The view direction is the observation-space ray (the reference pulls it back through the deformer's
        Jacobian, utils/utils.py:232-250; that belongs to the training path, see DESIGN.md)."""
        hit, t, xo, xc, v = self.surface_points(ray_dirs, A, trans, frame_of_ray, refine)
        idx = hit.nonzero(as_tuple=False).view(-1)
        rgb = torch.zeros((ray_dirs.shape[0], 3), device=self.device)
        if idx.numel() == 0:
            return rgb, hit, t
        sdf_ratio = ratio.get("sdfRatio") if isinstance(ratio, dict) else ratio
        _, grad = self.sdf_net.value_and_grad(xc[idx], sdf_ratio, want_feat=True)
        n = torch.nn.functional.normalize(grad, dim=1)
        with torch.no_grad():
            col = render_net(xc[idx], n, ray_dirs[idx], self.sdf_net.rendcond,
                             {"renderRatio": ratio.get("renderRatio") if isinstance(ratio, dict) else ratio})
        rgb.index_copy_(0, idx, col)
        return rgb, hit, t


# ---- mesh rasterisation and the colour frame of infer_garment ---------------------------------------------------------
class MaskRasterizer:
    """The `maskRender` of the reference (model/network.py:307-322) for the call sites that read only the fragments,
    `__, frags = self.maskRender(meshes)` (OptimGarmentNetwork.py:767,1397,1448,1492; OptimNetwork.py:437): callable on
    (verts [N,V,3] | [V,3], faces [F,3]) or on a meshes object with verts_padded() / faces_padded() whose faces are the
    same for every mesh.  Returns (None, ops.Fragments) -- no shaded image.
    camera = (fx, fy, px, py, R, T) as for ops.rasterize; image_size = (H, W)."""

    def __init__(self, camera, image_size):
        self.camera = camera
        self.image_size = image_size

    def __call__(self, meshes, faces=None):
        if faces is None:
            verts, fp = meshes.verts_padded(), meshes.faces_padded()
            faces = fp[0]
            if not all(torch.equal(f, faces) for f in fp[1:]):
                raise RuntimeError("MaskRasterizer: every mesh must have the same face list")
        else:
            verts = meshes
        return None, ops.rasterize(verts.detach().contiguous(), faces.contiguous(), self.camera, self.image_size)


def render_colors(canon_verts, faces, sdf_net, deformer, defconds, render_net, camera, image_size, ratio, ang_threshold,
                  offset_type=None, dthreshold=1e-4, times=30, chunk=10000):
    """The colour branch of infer_garment (OptimGarmentNetwork.py:3128-3204) on the device: deform the canonical mesh
    for the N frames of `defconds`, rasterise, seed points + view rays (FindSurfacePsRays), surface solve per chunk of
    `chunk` rays, canonical normal from the fused value+gradient launch, cardinal rays, colour network, and
    clamp((c/2 + 0.5) * 255) scattered into a white [N,H,W,3] image.  The rays and the camera position use camera 0
    (cam_pos = -R[0] T[0]), as the reference does.  Returns (colors [N,H,W,3] float, mask [N,H,W] bool, fragments)."""
    from . import utils
    fx, fy, px, py, R, T = camera
    R = torch.as_tensor(R, dtype=torch.float32, device=canon_verts.device).reshape(-1, 3, 3)
    T = torch.as_tensor(T, dtype=torch.float32, device=canon_verts.device).reshape(-1, 3)
    N = defconds[1][0].shape[0]
    H, W = (image_size, image_size) if isinstance(image_size, int) else image_size
    with torch.no_grad():
        verts = canon_verts.detach().contiguous()
        def_verts = deformer(verts[None].expand(N, -1, 3), defconds, ratio=ratio, offset_type=offset_type)
        frags = ops.rasterize(def_verts.contiguous(), faces, (fx, fy, px, py, R, T), (H, W))
        b, r, c, seeds, _, rays = utils.FindSurfacePsRays(verts, faces, frags, (fx, fy, px, py, R[0].cpu()))
        cam_pos = -R[0].matmul(T[0].view(3, 1)).view(3)
    cols = []
    for rays_, seeds_, b_ in zip(torch.split(rays, chunk), torch.split(seeds, chunk), torch.split(b, chunk)):
        if rays_.shape[0] == 0:
            continue
        ps, _ = utils.OptimizeGarmentSurfaceSinlge(cam_pos, rays_, seeds_.clone(), b_, sdf_net, ratio, deformer, defconds,
                                                   dthreshold=dthreshold, athreshold=ang_threshold, w1=3.05, w2=1.,
                                                   times=times, offset_type=offset_type)
        with torch.no_grad():
            _, g = sdf_net.value_and_grad(ps, ratio, want_feat=True)
            feat = sdf_net.rendcond
            nx = g / g.norm(dim=1, keepdim=True)
        crays, _ = utils.compute_cardinal_rays(deformer, ps, rays_, defconds, b_, ratio, 'test', offset_type=offset_type)
        with torch.no_grad():
            cols.append(render_net(ps, nx, crays, feat, ratio))
    with torch.no_grad():
        tcolors = torch.cat(cols, 0) if cols else torch.zeros((0, 3), device=canon_verts.device)
        tcolors = torch.clamp((tcolors / 2. + 0.5) * 255., min=0., max=255.)
        colors = torch.full((N, H, W, 3), 255., device=canon_verts.device)
        colors[b, r, c, :] = tcolors
    return colors, frags.pix_to_face[..., 0] >= 0, frags


# ---- point-cloud silhouettes of the training step's mask loss ----------------------------------------------------------
class PointsRenderer:
    """The reference's `pcRender` (OptimNetwork.py:87-100): PointsRendererWithFrags / PointsRendererWithFrags_Split
    (model/CameraMine.py:306-415) over PointsRasterizer + AlphaCompositor(background_color=None).
    camera = (fx, fy, px, py, R, T) as for ops.rasterize_points, settable between calls; image_size = (H, W) or an int;
    radius in NDC units (`point_render.radius`).  Call on points [N,P,3], a list of N [P,3] tensors or an object with
    points_list() (equal-size clouds), with features [P,C] (None: ones [P,1]).  Returns (images [N,H,W,C], fragments);
    with split_size= and all_size= the `_Split` form: ([upper [N,H,W,C], lower [N,H,W,C]], fragments), upper holding the
    points with p % all_size < split_size, both composited in one launch.  Differentiable in the points."""

    def __init__(self, camera, image_size, radius, points_per_pixel=50):
        self.camera = camera
        self.image_size = image_size
        self.radius = radius
        self.points_per_pixel = points_per_pixel

    def __call__(self, point_clouds, features=None, split_size=None, all_size=None):
        if hasattr(point_clouds, "points_list"):
            point_clouds = point_clouds.points_list()
        points = torch.stack(list(point_clouds)) if isinstance(point_clouds, (list, tuple)) else point_clouds
        points = points.float().contiguous()
        P = points.shape[-2]
        if features is None:
            features = torch.ones((P, 1), dtype=torch.float32, device=points.device)
        if split_size is not None:
            if all_size is None or all_size <= 0 or P % all_size:
                raise RuntimeError("PointsRenderer: all_size must divide the number of points of a cloud")
            upper = (torch.arange(P, device=points.device) % all_size < split_size)[:, None]
            features = torch.cat([features * upper, features * ~upper], 1)
        images, frags = ops.rasterize_points(points, features.float().contiguous(), self.camera, self.image_size,
                                             self.radius, self.points_per_pixel)
        if split_size is not None:
            C = images.shape[-1] // 2
            return [images[..., :C], images[..., C:]], frags
        return images, frags
