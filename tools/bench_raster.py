"""Timing of the mesh rasteriser (ops.rasterize, csrc/raster.cu) and of render.render_colors stage by stage.

Cases (CUDA events after warm-up, mean over --iters calls):
  * the 257^3 marching-cubes mesh of the synthetic sphere set (SURVEY 8d) at 1 x 512 x 512 and at 4 x 1080 x 1080 (four
    cameras rotated about the vertical axis);
  * the same mesh through a zoomed camera (fx = 40000 at 512 x 512), where the visible faces span hundreds of pixels and
    take the warp-per-face path;
  * render_colors on the marching-cubes mesh of the SDF network's own level set (the colour branch of infer_garment), at
    1 x 512 x 512, each of its stages bracketed by events.
Share of the HBM bound, from shapes: per face 3 vertices (36 B) + indices (24 B), per pixel an 8 B key + 24 B of outputs,
over 7.7 TB/s (HBM3e, HGX B200 data sheet).  The 1 x 512^2 working set (~10 MB) stays in L2 between calls; the 4 x 1080^2
one (~150 MB) does not.  The card's name and power limit are read in the same run and written next to the numbers.

    python tools/bench_raster.py [--out profiles/r03_raster.json] [--iters 20]
"""
import argparse
import json
import math
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from recmv_b200 import model as M  # noqa: E402
from recmv_b200 import ops, render, synth, testing, utils as U  # noqa: E402
from recmv_b200.MCAcc import Seg3dLossless  # noqa: E402
from recmv_b200.discretize import discretize_sdf  # noqa: E402

DEV = "cuda:0"
HBM_BYTES_PER_S = 7.7e12
RATIO = {"sdfRatio": 0.8, "deformerRatio": 0.6, "renderRatio": 0.9}


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n0 = ops.launch_count()
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3, (ops.launch_count() - n0) / iters


def rot_y(a):
    c, s = math.cos(a), math.sin(a)
    return [[c, 0.0, s], [0.0, 1.0, 0.0], [-s, 0.0, c]]


def raster_case(name, verts, faces, cam, size, iters):
    N, F = verts.shape[0], faces.shape[0]
    H, W = size
    t, launches = timed(lambda: ops.rasterize(verts, faces, cam, size), iters)
    fr = ops.rasterize(verts, faces, cam, size)
    nbytes = N * F * (36 + 24) + N * H * W * (8 + 24)
    res = {"case": name, "N": N, "H": H, "W": W, "faces": F, "vertices": int(verts.shape[1]), "ms": t * 1e3,
           "faces_per_s": N * F / t, "pixels_per_s": N * H * W / t, "kernel_launches_per_call": launches,
           "memsets_per_call": 1, "hbm_bytes_model": nbytes, "hbm_bound_share": nbytes / HBM_BYTES_PER_S / t,
           "covered_pixels": int((fr.pix_to_face >= 0).sum())}
    print(json.dumps(res))
    return res


def render_colors_stages(v, f, sdf, deformer, defconds, rn, cam, size, iters):
    """The steps of render.render_colors in one chunk, each bracketed by CUDA events."""
    fx, fy, px, py, R, T = cam
    names = ["deform", "rasterize", "find_surface_rays", "surface_solve", "normal", "cardinal_rays", "colour_net",
             "clamp_scatter"]
    acc = dict.fromkeys(names, 0.0)
    for it in range(iters + 1):
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
        ev[0].record()
        with torch.no_grad():
            dv = deformer(v[None].expand(1, -1, 3), defconds, ratio=RATIO, offset_type="body")
        ev[1].record()
        fr = ops.rasterize(dv.contiguous(), f, cam, size)
        ev[2].record()
        b, r, c, seeds, _, rays = U.FindSurfacePsRays(v, f, fr, (fx, fy, px, py, R[0].cpu()))
        ev[3].record()
        cam_pos = -R[0].matmul(T[0].view(3, 1)).view(3)
        ps, _ = U.OptimizeGarmentSurfaceSinlge(cam_pos, rays, seeds.clone(), b, sdf, RATIO, deformer, defconds,
                                               dthreshold=1e-4, athreshold=0.05, w1=3.05, w2=1., times=30,
                                               offset_type="body")
        ev[4].record()
        with torch.no_grad():
            _, g = sdf.value_and_grad(ps, RATIO, want_feat=True)
            nx = g / g.norm(dim=1, keepdim=True)
        ev[5].record()
        crays, _ = U.compute_cardinal_rays(deformer, ps, rays, defconds, b, RATIO, 'test', offset_type="body")
        ev[6].record()
        with torch.no_grad():
            col = rn(ps, nx, crays, sdf.rendcond, RATIO)
        ev[7].record()
        with torch.no_grad():
            img = torch.full((1,) + tuple(size) + (3,), 255., device=DEV)
            img[b, r, c] = torch.clamp((col / 2. + 0.5) * 255., min=0., max=255.)
        ev[8].record()
        torch.cuda.synchronize()
        if it:                                                         # the first pass is the warm-up
            for i, n in enumerate(names):
                acc[n] += ev[i].elapsed_time(ev[i + 1]) / iters
    t, launches = timed(lambda: render.render_colors(v, f, sdf, deformer, defconds, rn, cam, size, RATIO, 0.05,
                                                     offset_type="body"), iters, warmup=1)
    res = {"case": "render_colors", "H": size[0], "W": size[1], "faces": int(f.shape[0]), "rays": int(b.numel()),
           "stage_ms": acc, "total_ms": t * 1e3, "kernel_launches_per_call": launches}
    print(json.dumps(res))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_raster.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_raster: no CUDA device (timings need the GPU)")
    out = {"card": card(), "hbm_bytes_per_s_assumed": HBM_BYTES_PER_S, "results": []}
    print(json.dumps(out["card"]))
    step = 2.0 / 256
    v, f = ops.mc_gpu(synth.sphere_sdf_grid(res=257, device=DEV), step, step, step, -1.0, -1.0, -1.0)
    eye = torch.eye(3, device=DEV)[None]
    T0 = torch.tensor([[0.0, 0.0, 2.4]], device=DEV)
    cam512 = (1.2 * 512, 1.2 * 512, 255.5, 255.5, eye, T0)
    out["results"].append(raster_case("mc257_1x512x512", v[None].contiguous(), f, cam512, (512, 512), args.iters))
    R4 = torch.tensor([rot_y(a) for a in (0.0, 0.4, 0.8, 1.2)], device=DEV)
    cam1080 = (1.2 * 1080, 1.2 * 1080, 539.5, 539.5, R4, T0.expand(4, 3).contiguous())
    out["results"].append(raster_case("mc257_4x1080x1080", v[None].expand(4, -1, 3).contiguous(), f, cam1080, (1080, 1080),
                                      args.iters))
    # zoom onto the vertex nearest to the camera: faces of ~0.008 units at ~2 units span ~150 px
    k = int((v[:, 2]).argmin())
    fz = 40000.0
    zc = float(v[k, 2]) + 2.4
    camz = (fz, fz, 255.5 + fz * float(v[k, 0]) / zc, 255.5 + fz * float(v[k, 1]) / zc, eye, T0)
    out["results"].append(raster_case("mc257_closeup_1x512x512", v[None].contiguous(), f, camz, (512, 512), args.iters))

    sdf = testing.build_sdf(M.getTmpSdf, seed=0, perturb_seed=101, device=DEV)
    torch.manual_seed(1)
    tr = M.MLPTranslator(128, 6)
    testing.perturb_module(tr, 202, scale=0.5)
    Js, parents, init = synth.skeleton()
    sk = M.LBSkinner(synth.skinning_voxel((65, 225, 129), seed=7), [-1.1] * 3, [1.1] * 3, Js, parents, init_pose=init,
                     bbox_extend=torch.tensor(synth.BBOX_EXTEND), bbox_center=torch.tensor(synth.BBOX_CENTER))
    deformer = M.CompositeDeformer([tr, sk]).to(DEV)
    torch.manual_seed(2)
    rn = M.RenderingNetwork_view_norm(256, d_in=9, d_out=3, dims=[512] * 4, mode="idr", weight_norm=True,
                                      multires_v=4, multires_n=0)
    testing.perturb_module(rn, 303)
    rn = rn.to(DEV)
    eng = Seg3dLossless(None, b_min=[-1, -1, -1], b_max=[1, 1, 1], resolutions=[17, 33, 65, 129, 257],
                        align_corners=False, balance_value=0.0).to(DEV)
    vs, fs = discretize_sdf(sdf, eng, RATIO)
    poses, trans = synth.poses_trans(1, seed=11)
    conds = torch.randn((1, 128), generator=synth.generator(5)) * 0.1
    defconds = [conds.to(DEV), [poses.to(DEV), trans.to(DEV)]]
    out["results"].append(render_colors_stages(vs, fs, sdf, deformer, defconds, rn, cam512, (512, 512),
                                               max(args.iters // 5, 2)))
    ops.check_async_errors()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
