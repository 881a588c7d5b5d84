"""Timing of the points rasteriser + alpha compositor (ops.rasterize_points, csrc/points.cu): forward, backward and the
dense fragment expansion, each on its own.

Cases (CUDA events after warm-up, mean over --iters calls): the vertices of the 257^3 marching-cubes mesh of the synthetic
sphere set (SURVEY 8d, ~100 k points) as one point cloud per frame, at 1 and 4 frames (four cameras rotated about the
vertical axis), 512^2 and 1080^2, radius 0.006 and 0.0041 (the `point_render.radius` values of the configs), K = 50, one
feature channel.  The forward includes its one host synchronisation (the candidate count).  Next to each time: the
candidate total, the kept entries (sum over pixels of min(candidates, K)) and a byte model of the traffic each pass needs,
from these counts (per point 12 B read + 28 B of projection state; per pixel counter, offsets and image; per candidate
the counting atomics, the key write and read; per kept entry the projection read).  The card's name and power limit are
read in the same run and written next to the numbers.

    python tools/bench_points.py [--out profiles/r04_points.json] [--iters 20]
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
from recmv_b200 import ops, synth  # noqa: E402

DEV = "cuda:0"
HBM_BYTES_PER_S = 7.7e12
K = 50


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


def case(name, pts, cam, S, radius, iters):
    N, P = pts.shape[0], pts.shape[1]
    feats = torch.ones((P, 1), device=DEV)
    npix = N * S * S
    t_fwd, l_fwd = timed(lambda: ops.rasterize_points(pts, feats, cam, S, radius, K), iters)
    p = pts.detach().requires_grad_(True)
    images, fr = ops.rasterize_points(p, feats, cam, S, radius, K)
    g = torch.randn_like(images)
    t_bwd, l_bwd = timed(lambda: torch.autograd.grad(images, p, g, retain_graph=True), iters)

    def expand():
        ops.PointFragments(fr._meta, fr._scratch, fr._cand, fr.candidates).idx

    t_frag, l_frag = timed(expand, max(iters // 4, 2), warmup=1)
    total = fr.candidates
    kept = int((fr.idx >= 0).sum())
    fwd_bytes = N * P * (12 + 28 + 20) + npix * (4 + 8 + 4 + 8 + 8 + 4) + total * (4 + 4 + 8 + 8 + 8) + kept * (8 + 16 + 4)
    bwd_bytes = npix * (8 + 8 + 4) + kept * (8 + 16 + 4 + 8) + N * P * (12 + 8 + 4 + 12 + 8)
    frag_bytes = npix * 16 + kept * (8 + 16) + npix * K * 16
    res = {"case": name, "N": N, "H": S, "W": S, "points_per_frame": P, "radius": radius, "K": K,
           "candidates": total, "kept_entries": kept, "covered_pixels": int((fr.idx[..., 0] >= 0).sum()),
           "forward_ms": t_fwd * 1e3, "forward_launches": l_fwd, "forward_bytes_model": fwd_bytes,
           "forward_hbm_bound_share": fwd_bytes / HBM_BYTES_PER_S / t_fwd,
           "backward_ms": t_bwd * 1e3, "backward_launches": l_bwd, "backward_bytes_model": bwd_bytes,
           "backward_hbm_bound_share": bwd_bytes / HBM_BYTES_PER_S / t_bwd,
           "fragments_ms": t_frag * 1e3, "fragments_launches": l_frag, "fragments_bytes_model": frag_bytes,
           "fragments_hbm_bound_share": frag_bytes / HBM_BYTES_PER_S / t_frag}
    print(json.dumps(res))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_points.json"))
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_points: no CUDA device (timings need the GPU)")
    out = {"card": card(), "hbm_bytes_per_s_assumed": HBM_BYTES_PER_S, "results": []}
    print(json.dumps(out["card"]))
    step = 2.0 / 256
    v, _ = ops.mc_gpu(synth.sphere_sdf_grid(res=257, device=DEV), step, step, step, -1.0, -1.0, -1.0)
    T0 = torch.tensor([[0.0, 0.0, 2.4]], device=DEV)
    R4 = torch.tensor([rot_y(a) for a in (0.0, 0.4, 0.8, 1.2)], device=DEV)
    for S in (512, 1080):
        for N in (1, 4):
            cam = (1.2 * S, 1.2 * S, (S - 1) / 2, (S - 1) / 2, R4[:N].contiguous(), T0.expand(N, 3).contiguous())
            pts = v[None].expand(N, -1, 3).contiguous()
            for radius in (0.006, 0.0041):
                out["results"].append(case(f"mc257_{N}x{S}x{S}_r{radius}", pts, cam, S, radius, args.iters))
    ops.check_async_errors()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
