#!/usr/bin/env python
"""bench.py -- rays/sec of the fused SDF render path (BASELINE.json metric) on N B200s of one node.

A "step" = one pass of the hot path over one 512x512-ray x 64-sample frame per GPU:
rays -> sample points -> skinning-voxel sample -> inverse LBS -> PE -> 9-layer SDF MLP -> per-ray first
hit.  Inputs are seeded synthetic data of the BASELINE shapes (no dataset / checkpoint exists offline).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mode tc3|tc1|simt] [--impl reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement" for every field.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H = W = 512
S = 64
FLOP_PER_SAMPLE = 2 * 1966592  # SURVEY 8d: 3 933 184 FLOP per SDF forward
METRIC = "rays/sec at 512x512x64-samp SDF render"
MODES = {"simt": 0, "tc3": 1, "tc1": 2}
# dram__bytes_read.sum + dram__bytes_write.sum of ONE full-frame launch of the dominant kernel, from the
# ncu capture of the final round-1 kernel, profiles/r01_ncu_tc3_current.txt (142.3 MB read + 54.8 MB written; the
# algorithmic minimum is the 67 MB sdf output + the touched part of the 181 MB voxel + 8.6 MB of weights)
TRAFFIC_BYTES = {"tc3": 197053696}
DUMP_SDF_RAYS = 65536   # rays of the per-sample SDF written by --dump-outputs (all 512x512 of them would be 64 MiB)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d, "measured"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock / power / throttle reasons sampled DURING the timed region (B200_PROFILING.md): NVML in-process
    every 20 ms (>= 20 samples even for a 0.5 s region); `nvidia-smi` as the fallback when NVML is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")

    def __init__(self, cuda_index):
        super().__init__(daemon=True)
        self.gpu, self.rows, self.stop_flag, self.h, self.nv = cuda_index, [], False, None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            self.h = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
            self.nv = pynvml
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.h = None

    def _nvml_row(self):
        nv = self.nv
        sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
        pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
        r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        bits = (nv.nvmlClocksEventReasonHwSlowdown, nv.nvmlClocksEventReasonHwThermalSlowdown,
                nv.nvmlClocksEventReasonSwThermalSlowdown, nv.nvmlClocksEventReasonSwPowerCap)
        return [str(self.gpu), str(sm), str(self.sm_max), str(pw)] + ["Active" if r & b else "Not Active" for b in bits]

    def run(self):
        while not self.stop_flag:
            try:
                if self.h is not None:
                    self.rows.append(self._nvml_row())
                    time.sleep(0.02)
                    continue
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.gpu)], capture_output=True, text=True, timeout=5).stdout
                for line in out.strip().splitlines():
                    self.rows.append([c.strip() for c in line.split(",")])
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        num = lambda v: v.replace(".", "", 1).isdigit()  # noqa: E731
        sm = sorted(float(r[1]) for r in self.rows if len(r) > 2 and num(r[1]))
        mx = [float(r[2]) for r in self.rows if len(r) > 2 and num(r[2])]
        pw = [float(r[3]) for r in self.rows if len(r) > 3 and num(r[3])]
        reasons = set()
        for r in self.rows:
            for name, v in zip(self.NAMES, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows), "power_w_max": max(pw) if pw else None,
                "source": "nvml" if self.h is not None else "nvidia-smi"}


_CPU_SCENE = {}


def _cpu_scene():
    """Weights, skinning voxel and skeleton of the CPU legs (built once per process)."""
    if not _CPU_SCENE:
        from oracle import oracle_torch as ot
        from recmv_b200 import synth
        from recmv_b200.model import LBSkinner, getTmpSdf
        torch.manual_seed(0)
        net = getTmpSdf("cpu", 6, 0.6, 256)
        Ws, bs = net.effective_weights()
        Js, parents, init = synth.skeleton()
        ws = synth.skinning_voxel((65, 225, 129), seed=7)
        sk = LBSkinner(ws, [-1.1] * 3, [1.1] * 3, Js, parents, init_pose=init,
                       bbox_extend=torch.tensor(synth.BBOX_EXTEND), bbox_center=torch.tensor(synth.BBOX_CENTER))
        poses, trans = synth.poses_trans(1, seed=11)
        _CPU_SCENE.update(Ws=[w.detach() for w in Ws], bs=[b.detach() for b in bs], ws=ws, trans=trans,
                          A=ot.bone_matrices(poses, Js, parents, sk.init_pose))
    return _CPU_SCENE


def cpu_port_rate(samples_rays, threads):
    """The oracle's CPU restatement of the same path (inverse LBS + SDF MLP), timed on the host cores.
    Bounded sample of the workload: `samples_rays` rays x 64 samples of frame 0."""
    from oracle import oracle_torch as ot
    from recmv_b200 import synth
    torch.set_num_threads(threads)
    sc = _cpu_scene()
    Ws, bs, ws, trans, A = sc["Ws"], sc["bs"], sc["ws"], sc["trans"], sc["A"]
    dirs = synth.pinhole_rays(H, W)[H * W // 2: H * W // 2 + samples_rays]
    cam = torch.tensor(synth.CAM_POS)
    dt = (synth.T_FAR - synth.T_NEAR) / S
    tk = synth.T_NEAR + (torch.arange(S, dtype=torch.float32) + 0.5) * dt
    pe_w = ot.annealing_weights(6, None)
    bi = torch.zeros(samples_rays * S, dtype=torch.long)

    def step():
        with torch.no_grad():
            x = (cam[None, None] + tk[None, :, None] * dirs[:, None, :]).reshape(-1, 3)
            xc, ok = ot.lbs_inverse(x, A, trans, ws, torch.tensor(synth.BBOX_CENTER), synth.BBOX_EXTEND, bi)
            out = []
            for c in range(0, xc.shape[0], 65536):  # 65 536-sample slabs (BASELINE.md section 3)
                out.append(ot.sdf_mlp(xc[c:c + 65536], Ws, bs, pe_w)[0])
            return torch.cat(out)
    return step


def best_cpu_threads():
    """torch-CPU throughput of the port peaks well below the core count of the GPU host (measured on the
    128-thread B200 host: 8 thr 1201, 16 thr 1443, 32 thr 1405, 64 thr 1022, 128 thr 37 rays/s --
    profiles/r01_notes.md): calibrate on a small sample and use the fastest setting.  Bounded: candidates are
    8/16/32/64 (never more threads than cores), each probe is 2 x 128 rays and the loop stops after 20 s."""
    if os.environ.get("RECMV_BENCH_CPU_THREADS"):     # skip the calibration (tests)
        return max(1, int(os.environ["RECMV_BENCH_CPU_THREADS"]))
    n = os.cpu_count() or 1
    best, best_rate = min(n, 8), 0.0
    t_start = time.perf_counter()
    for th in (16, 8, 32, 64):
        if th > n or time.perf_counter() - t_start > 20.0:
            continue
        step = cpu_port_rate(128, th)
        step()
        t0 = time.perf_counter()
        step()
        rate = 128 / (time.perf_counter() - t0)
        if rate > best_rate:
            best, best_rate = th, rate
    return best


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  /root/reference does not exist
    on the GPU box and its natives are CUDA-only, so this is the oracle PORT (torch CPU restatement,
    pinned against the imported reference modules -- tests/golden) on all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = best_cpu_threads()
    rays = int(os.environ.get("RECMV_BENCH_REF_RAYS", "4096"))
    step = cpu_port_rate(rays, threads)
    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    val = rays / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "rays/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "gpu_launches": 0,
            "config": {"workload": "512x512 rays x 64 samples: inverse-LBS + SDF MLP (configs[1])",
                       "sample": f"{rays} rays x 64 samples per step (bounded sample of the frame)"},
            "cpu_baseline": {"value": val, "unit": "rays/s", "cores": threads, "kind": "port",
                             "sample": f"{rays} rays x 64 samples, torch CPU fp32, {threads} threads (fastest of 8/16/32/64)"},
            "e2e": {"value": val, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


def secondary_rates(dev, ren, mode):
    """Throughput of the other fused launches of the path at 1 M points (tcgen05 modes): translator + LBS
    (CompositeDeformer.forward), its forward-mode Jacobian variant, the SDF value+gradient launch and the colour
    network.  ALGORITHMIC FLOP per point: SURVEY 8d (translator 1 746 944, colour net 1 871 872, SDF 3 933 184;
    the forward-mode launches carry 4 rows per point)."""
    import recmv_b200.model as M
    from recmv_b200 import ops
    from recmv_b200 import synth as sy
    P = 1 << 20
    g = sy.generator(21)
    pts = ((torch.rand((P, 3), generator=g) - 0.5) * 1.2).to(dev)
    unit = torch.nn.functional.normalize(torch.randn((P, 3), generator=g), dim=1).to(dev)
    feats = (torch.randn((P, 256), generator=g) * 0.1).to(dev)
    conds = (torch.randn((1, 128), generator=g) * 0.1).to(dev)
    poses, trans = sy.poses_trans(1, seed=11)
    poses, trans = poses.to(dev), trans.to(dev)
    torch.manual_seed(3)
    tr = M.MLPTranslator(128, 6).to(dev)
    rn = M.RenderingNetwork_view_norm(256, d_in=9, d_out=3, dims=[512] * 4, mode="idr", weight_norm=True,
                                      multires_v=4, multires_n=0).to(dev)
    tr.mlp_mode = rn.mlp_mode = mode
    deformer = M.CompositeDeformer([tr, ren.skinner])
    ratio = {"sdfRatio": None, "deformerRatio": None, "renderRatio": None}
    bi = torch.zeros((P,), dtype=torch.long, device=dev)
    sdf_net = ren.sdf_net
    sdf_net.mlp_mode = mode

    def rate(fn, flop_per_point):
        with torch.no_grad():
            for _ in range(2):
                fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                fn()
            e1.record()
            torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 5
        return {"points_per_s": P / (ms * 1e-3), "ms_per_1M_points": ms,
                "algorithmic_tflops": flop_per_point * P / (ms * 1e-3) / 1e12}

    # training step of the SDF network on the same engine: fused forward that saves the layer inputs + tcgen05 backward
    # GEMMs (backward-data and weight gradient per layer, all on the operand planes) behind loss.backward(); ALGORITHMIC FLOP per point =
    # 3 x 3 933 184 (forward, backward-data, weight gradient), each issued as 3 fp16 MMAs per product
    Pt = 1 << 17
    xt = pts[:Pt].clone()
    c_sdf = (torch.randn((Pt, 1), generator=g) / Pt).to(dev)
    c_feat = (torch.randn((Pt, 256), generator=g) / Pt * 0.1).to(dev)

    def train_step():
        for p_ in sdf_net.parameters():
            p_.grad = None
        xg = xt.detach().requires_grad_(True)
        y = sdf_net(xg, None)
        ((y * c_sdf).sum() + (sdf_net.rendcond * c_feat).sum()).backward()

    def rate_train():
        for _ in range(2):
            train_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            train_step()
        e1.record()
        torch.cuda.synchronize(dev)
        ms = e0.elapsed_time(e1) / 5
        tf = 3 * FLOP_PER_SAMPLE * Pt / (ms * 1e-3) / 1e12
        peaks, _ = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
        return {"points_per_s": Pt / (ms * 1e-3), "ms_per_step": ms, "points": Pt, "path": sdf_net.last_path,
                "backward": ops.SdfMlpTrainFunction.last_backward, "algorithmic_tflops": tf,
                "roofline": {"bound": "tensor", "achieved": tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": tf / peak_tf,
                             "mma_passes": 3, "issued_frac": 3 * tf / peak_tf},
                "includes": "weight-norm graph, cotangent packing, 9 backward-data launches, 9 weight-gradient launches + bias column sums, "
                            "PE Jacobian, autograd bookkeeping (everything loss.backward() runs)"}
    train = rate_train()
    # the same step through torch autograd over cuBLAS fp32 (what the reference runs): informative, same GPU, same run
    sdf_net.train_fused = False
    allow = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref = rate_train()
    finally:
        sdf_net.train_fused = True
        torch.backends.cuda.matmul.allow_tf32 = allow
    train["torch_autograd_cublas_fp32_ms_per_step"] = ref["ms_per_step"]
    train["speedup_vs_torch_autograd"] = ref["ms_per_step"] / train["ms_per_step"]

    # second order (SURVEY 8f row 4): the eikonal term of the training step -- net.gradient(x) with create_graph=True, then
    # ((|grad| - 1)^2).mean().backward() -- on the tcgen05 GEMMs (recmv_b200/second_order.py) and, for comparison, through
    # torch autograd over cuBLAS fp32.  The reference draws ~8-16 k points per step for this term (OptimGarmentNetwork.py:1107).
    from recmv_b200 import utils as U
    Pe = 1 << 14
    xe = pts[:Pe].clone()

    def eik_step():
        for p_ in sdf_net.parameters():
            p_.grad = None
        U.eikonal_loss(sdf_net, xe.detach().clone(), None).backward()

    def rate_eik():
        for _ in range(2):
            eik_step()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            eik_step()
        e1.record()
        torch.cuda.synchronize(dev)
        return e0.elapsed_time(e1) / 5
    eik_ms = rate_eik()
    eik = {"ms_per_step": eik_ms, "points": Pe, "points_per_s": Pe / (eik_ms * 1e-3), "path": sdf_net.last_path,
           "backward": ops.SdfMlpTrainFunction.last_backward,
           "gemm_launches": "9 forward + 9 reverse + 9 tangent + 8 backward-data layer GEMMs, 2 weight-gradient launches"}
    sdf_net.train_fused = False
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        eik_ref = rate_eik()
    finally:
        sdf_net.train_fused = True
        torch.backends.cuda.matmul.allow_tf32 = allow
    eik["torch_autograd_cublas_fp32_ms_per_step"] = eik_ref
    eik["speedup_vs_torch_autograd"] = eik_ref / eik_ms

    return {
        "sdf_train_step (fused forward + tcgen05 backward, loss.backward())": train,
        "sdf_eikonal_step (second order: gradient(create_graph) + loss.backward())": eik,
        "deformer_fwd (MLPTranslator + LBS, one launch)": rate(
            lambda: deformer(pts, [conds, [poses, trans]], bi, ratio=ratio, offset_type="body"), 1746944),
        "deformer_fwd_jac (value + 3x3 Jacobian, forward mode)": rate(
            lambda: deformer.value_and_jacobian(pts, [conds, [poses, trans]], bi, ratio=ratio, offset_type="body"), 4 * 1746944),
        "sdf_value_and_grad (forward mode)": rate(lambda: sdf_net.value_and_grad(pts, None), 4 * FLOP_PER_SAMPLE),
        "rendernet_fwd (colour MLP)": rate(lambda: rn(pts, unit, unit, feats, ratio), 1871872),
    }


def dump_outputs(out_dir, sdf, hit_idx, hit_t):
    """What render() returned in the last timed step, as <out_dir>/<name>.npy: the per-ray first-hit sample index
    (float64, exact) and distance of every ray, and the per-sample SDF of a fixed seeded sample of DUMP_SDF_RAYS rays
    (ascending ray order).  The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    R = sdf.shape[0]
    rows = torch.randperm(R, generator=torch.Generator().manual_seed(0))[:DUMP_SDF_RAYS].sort().values
    arrays = {"sdf": sdf[rows.to(sdf.device)].float(), "hit_idx": hit_idx.double(), "hit_t": hit_t.float()}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


_JSON_OUT = None


def _claim_stdout():
    """stdout carries exactly ONE line (the JSON).  Libraries print there too (NCCL's "NCCL version ..." banner goes to
    stdout at NCCL_DEBUG >= VERSION), so the process' fd 1 is pointed at stderr and the JSON line is written to a private
    duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--mode", default=os.environ.get("RECMV_BENCH_MODE", "tc3"), choices=sorted(MODES))
    ap.add_argument("--scaling", default=os.environ.get("RECMV_BENCH_SCALING", "strong"), choices=("strong", "weak"),
                    help="N > 1: strong = the SAME job (--frames 512x512x64 frames) row-sharded over the ranks with a "
                         "flat gradient all-reduce per step (default); weak = one full frame per rank, no collective")
    ap.add_argument("--frames", type=int, default=1, help="frames per step of the strong-scaling job (4 = configs[3])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write the last step's render outputs to DIR/<name>.npy (rank 0's rays)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; the reference arm has none")
    if args.impl == "reference":
        return run_reference(args)

    from recmv_b200 import ops, synth
    from recmv_b200.render import SdfRenderer, shard_rows
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback of the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # NCCL logging only when asked for (RECMV_NCCL_DEBUG=INFO shows the NVLS / ring choice); it lands on stderr
        os.environ["NCCL_DEBUG"] = os.environ.get("RECMV_NCCL_DEBUG", "WARN")
        dist.init_process_group("nccl", device_id=dev)
    warmup = max(args.warmup, 3)
    strong = args.scaling == "strong"
    frames = max(args.frames, 1) if strong else 1

    # ---- scene -------------------------------------------------------------------------------------------
    # strong: ONE job of `frames` 512x512 frames; every rank renders a contiguous block of image rows of every
    #         frame (render.shard_rows), weights / voxel / bone matrices replicated (SURVEY 8e); per step one flat
    #         fp32 all-reduce of the SDF-MLP gradient bucket (1 975 220 floats) on a side stream.
    # weak:   every rank renders its own full frame (its own pose), no collective.
    mode = MODES[args.mode]
    ren = SdfRenderer(dev, mode=mode, samples=S)
    if strong:
        poses, trans = synth.poses_trans(frames, seed=11, device="cpu")
        A, t = ren.bone_matrices(poses.to(dev), trans.to(dev))
        row0, rows = shard_rows(H, rank, world)
        d1 = synth.pinhole_rays(H, W, device=dev, row0=row0, rows=rows)
        dirs = d1.repeat(frames, 1).contiguous()          # frame-major: rays of frame f = [f*rows*W, (f+1)*rows*W)
        rays_per_frame = rows * W
        total_rays = frames * H * W
    else:
        poses, trans = synth.poses_trans(world, seed=11, device="cpu")
        A, t = ren.bone_matrices(poses[rank:rank + 1].to(dev), trans[rank:rank + 1].to(dev))
        dirs = synth.pinhole_rays(H, W, device=dev)
        rays_per_frame = dirs.shape[0]
        total_rays = world * H * W
    R = dirs.shape[0]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    # gradient bucket of the SDF network (synthetic values; the all-reduce is the real collective of a training step)
    n_grad = sum(p.numel() for p in ren.sdf_net.parameters())
    grad_bucket = torch.randn(n_grad, device=dev, generator=torch.Generator(device=dev).manual_seed(5 + rank))
    comm = torch.cuda.Stream(dev) if world > 1 else None
    use_coll = world > 1 and strong

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def step_device():
        """One step with inputs resident in HBM: [all-reduce of the gradient bucket on the side stream ||] render."""
        work = None
        if use_coll:
            comm.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(comm):
                work = dist.all_reduce(grad_bucket, op=dist.ReduceOp.SUM, async_op=True)
        out = ren.render(dirs, A, t, rays_per_frame=rays_per_frame)
        if work is not None:
            work.wait()
            torch.cuda.current_stream(dev).wait_stream(comm)
        return out

    def max_over_ranks(x):
        tt = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item())

    # ---- value: inputs resident in HBM ---------------------------------------------------------------
    for _ in range(warmup):
        step_device()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = ops.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_beg, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_beg.record()
    for i in range(args.steps):
        flush.zero_()  # L2 flush between timed iterations (inside the bracket, ~0.05 ms)
        ev[i][0].record()
        sdf, _, hit_idx, hit_t = step_device()
        ev[i][1].record()
    t_end.record()
    barrier()
    launches = ops.launch_count() - launches0
    ops.check_async_errors()
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:   # before the e2e leg: render() reuses its sdf buffer
        dump_outputs(args.dump_outputs, sdf, hit_idx, hit_t)
    step_ms = [a.elapsed_time(b) for a, b in ev]
    dev_s = max_over_ranks(t_beg.elapsed_time(t_end) * 1e-3)   # device time of the K steps, max over ranks
    ms_per_step = dev_s * 1e3 / args.steps
    value = total_rays / (dev_s / args.steps)
    kernel_ms = sum(step_ms) / len(step_ms)  # device time of one step's launch sequence on this rank
    nhit = int((hit_idx >= 0).sum().item())
    comm_ok = None
    if use_coll:   # the reduced bucket must be the same on every rank (sum of the per-rank seeds' buckets)
        chk = torch.stack([grad_bucket[:1024].double().sum()])
        lo, hi = chk.clone(), chk.clone()
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        comm_ok = bool((lo == hi).all().item()) and bool(torch.isfinite(chk).all().item())

    # ---- e2e: HOST buffers in / HOST result out through the public call ---------------------------------
    dirs_h = dirs.cpu().pin_memory()
    A_h, t_h = A.cpu().pin_memory(), t.cpu().pin_memory()
    o_t = torch.empty(R, dtype=torch.float32).pin_memory()
    o_i = torch.empty(R, dtype=torch.int32).pin_memory()
    grad_h = grad_bucket.cpu().pin_memory() if use_coll else None

    def step_host():
        work = None
        if use_coll:   # gradients arrive from the host side too in this leg (H2D counted below)
            with torch.cuda.stream(comm):
                grad_bucket.copy_(grad_h, non_blocking=True)
                work = dist.all_reduce(grad_bucket, op=dist.ReduceOp.SUM, async_op=True)
        ren.render_host(dirs_h, A_h, t_h, o_t, o_i, rays_per_frame=rays_per_frame)
        if work is not None:
            work.wait()
            torch.cuda.current_stream(dev).wait_stream(comm)
        torch.cuda.current_stream(dev).synchronize()  # the host result must be readable every step

    for _ in range(2):
        step_host()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_host()
    e2e_s = max_over_ranks(time.perf_counter() - t0)   # host clock: the region ends when the HOST holds the result
    barrier()
    e2e = total_rays / (e2e_s / args.steps)
    h2d = dirs_h.numel() * 4 + A_h.numel() * 4 + t_h.numel() * 4 + (grad_h.numel() * 4 if use_coll else 0)
    d2h = o_t.numel() * 4 + o_i.numel() * 4

    # ---- second half of the BASELINE metric: marching-cubes cells/s on a 257^3 grid (256^3 cells) -----------
    mc = None
    if rank == 0 and world == 1:   # the MC half of the metric and the secondary launches: N=1 line only
        grid = synth.sphere_sdf_grid(257, num=8, seed=3, device=dev)
        for _ in range(3):
            v, f = ops.mc_gpu(grid, 2 / 256, 2 / 256, 2 / 256, -1.0, -1.0, -1.0, 0.0)
        torch.cuda.synchronize(dev)
        reps = 20
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            v, f = ops.mc_gpu(grid, 2 / 256, 2 / 256, 2 / 256, -1.0, -1.0, -1.0, 0.0)
        e1.record()
        torch.cuda.synchronize(dev)
        mc_ms = e0.elapsed_time(e1) / reps
        mc_bytes = 4 * 257 ** 3 + 12 * v.shape[0] + 24 * f.shape[0]   # SURVEY 8d algorithmic bytes
        mc = {"cells_per_s": 256 ** 3 / (mc_ms * 1e-3), "ms_per_call": mc_ms, "grid": "257^3", "verts": int(v.shape[0]),
              "faces": int(f.shape[0]), "algorithmic_bytes": mc_bytes,
              "note": "sign mask + count + scan + vertex + face passes queued by one call, one host sync at the end, fresh output tensors"}

    # ---- the other networks of the path on the same engine (reported next to the headline, not part of it) -----------
    secondary = None
    if rank == 0 and world == 1 and mode != 0 and not args.no_secondary:
        secondary = secondary_rates(dev, ren, mode)

    if rank == 0:
        peaks, src = measured_peaks()
        peak_tf = float(peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))
        flop = FLOP_PER_SAMPLE * R * S
        ach = flop / (kernel_ms * 1e-3) / 1e12
        issued = {0: None, 1: 3, 2: 1}[mode]
        roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                "traffic": TRAFFIC_BYTES.get(args.mode) if world == 1 else None,
                "peak_source": f"{src} bf16_tflops_sustained (kernel timed inside a long step)",
                "kernel_ms": kernel_ms, "algorithmic_flop_per_launch": flop,
                "mma_passes": issued,
                "issued_frac": (ach * issued / peak_tf) if issued else None,
                "note": "frac = ALGORITHMIC fp32-equivalent FLOP/s over dense-bf16 peak; tc3 issues 3 fp16 MMAs "
                        "per product to meet the fp32 parity bar, so frac <= 1/3 by construction; "
                        "issued_frac = tensor-pipe work actually issued over the same peak"}
        cpu = None
        if not args.no_cpu_baseline and world == 1:   # reported at N=1 only
            threads = best_cpu_threads()
            rays = 2048
            step = cpu_port_rate(rays, threads)
            step()
            c0 = time.perf_counter()
            n = 0
            while time.perf_counter() - c0 < 10.0 or n < 2:
                step()
                n += 1
            cdt = (time.perf_counter() - c0) / n
            cpu = {"value": rays / cdt, "unit": "rays/s", "cores": threads, "kind": "port",
                   "sample": f"{rays} rays x 64 samples x {n} reps (oracle torch-CPU restatement of inverse-LBS + "
                             f"SDF MLP, fp32; {threads} threads = fastest of 8/16/32/64 on this host)"}
        if strong:
            workload = (f"configs[1]: {frames} frame(s) of 512x512 rays x 64 samples/ray, 9-layer x512 SDF MLP "
                        "(PeopleSnapshot-shaped synthetic scene), inverse-LBS on a 24x65x225x129 skinning voxel"
                        + (f"; image rows sharded over {world} ranks, one flat fp32 all-reduce of the SDF-MLP gradient "
                           f"bucket ({n_grad} floats) per step on a side stream" if world > 1 else ""))
        else:
            workload = ("configs[1]: 512x512 rays x 64 samples/ray, 9-layer x512 SDF MLP (PeopleSnapshot-shaped "
                        "synthetic scene), inverse-LBS on a 24x65x225x129 skinning voxel, one frame per GPU")
        line = {"metric": METRIC, "value": value, "unit": "rays/s", "n_gpus": world, "steps": args.steps,
                "warmup": warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
                "scaling": "strong" if strong else "weak",
                "vs_baseline": None, "dtype": {0: "f32", 1: "f16x3->f32", 2: "f16->f32"}[mode],
                "data": "synthetic",
                "config": {"workload": workload,
                           "mlp_mode": args.mode, "rays_per_gpu": R, "samples_per_ray": S, "frames": frames,
                           "l2": "256 MiB buffer written between timed steps (inside the bracket)",
                           "timing": "CUDA events around the K steps on the launching stream, max over ranks",
                           "collective": ({"op": "all_reduce(sum, fp32)", "bytes": 4 * n_grad, "backend": "nccl",
                                           "inside_timed_region": True, "result_identical_on_all_ranks": comm_ok}
                                          if use_coll else None),
                           "hits": nhit},
                "clocks": sampler.summary(), "gpu_launches": launches,
                "e2e": {"value": e2e, "unit": "rays/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
                "roofline": roof, "cpu_baseline": cpu, "mc": mc, "secondary": secondary}
        if mc is not None:
            hbm = float(peaks.get("hbm_gbs", 6650.0))
            mc["roofline"] = {"bound": "hbm", "achieved": mc["algorithmic_bytes"] / (mc["ms_per_call"] * 1e-3) / 1e9,
                              "peak": hbm, "unit": "GB/s",
                              "frac": mc["algorithmic_bytes"] / (mc["ms_per_call"] * 1e-3) / 1e9 / hbm}
        _emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
