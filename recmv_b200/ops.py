"""Torch-facing wrappers over the C ABI: allocate outputs, pass raw pointers + the current stream,
raise on non-zero status, wire autograd.  PyTorch is plumbing here (device memory, streams,
autograd graph); all arithmetic happens in librecmv_b200.so.
"""
import collections
import ctypes
from ctypes import byref, c_float, c_int64, c_size_t

import torch

from . import _lib
from ._lib import (F32, F64, LAYOUT_NCDHW, LAYOUT_NDHWC, MLP_FP32_SIMT, MLP_TC_F16X1, MLP_TC_F16X3,
                   RayMarch, Voxel, check)

DEFAULT_MLP_MODE = MLP_TC_F16X3


def _stream(t):
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _check_input(t, name):
    # reference: CHECK_INPUT (FastMinv/M3x3Inv.cpp:4-6, MCGpu/MCGpu.cpp:3-5)
    if not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor")
    if not t.is_contiguous():
        raise RuntimeError(f"{name} must be contiguous")


def _dtype_code(t, name):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float64:
        return F64
    raise RuntimeError(f"{name} must be a float/double tensor")


# --------------------------------------------------------------------------------------------------
# FastMinv
# --------------------------------------------------------------------------------------------------
def minv3x3(ms):
    """FastMinv.Fast3x3Minv(ms) -> [invs, checks]  (FastMinv/M3x3Inv.cpp:12-37)."""
    _check_input(ms, "ms")
    code = _dtype_code(ms, "ms")
    n = ms.size(0)
    invs = torch.empty((n, 3, 3), dtype=ms.dtype, device=ms.device)
    ok = torch.empty((n,), dtype=torch.uint8, device=ms.device)
    with torch.cuda.device(ms.device):
        check(_lib.load().recmv_minv3x3_fwd(_ptr(ms), _ptr(invs), _ptr(ok), n, code, _stream(ms)),
              "recmv_minv3x3_fwd")
    return [invs, ok.view(torch.bool)]


def minv3x3_backward(grads, invs):
    """FastMinv.Fast3x3Minv_backward(grads, invs) -> outs  (FastMinv/M3x3Inv.cpp:39-59)."""
    _check_input(grads, "grads")
    _check_input(invs, "invs")
    if grads.dtype != invs.dtype:
        raise RuntimeError("invs must have same type with grads")
    code = _dtype_code(invs, "invs")
    n = invs.size(0)
    outs = torch.empty((n, 3, 3), dtype=invs.dtype, device=invs.device)
    with torch.cuda.device(invs.device):
        check(_lib.load().recmv_minv3x3_bwd(_ptr(grads), _ptr(invs), _ptr(outs), n, code,
                                            _stream(invs)), "recmv_minv3x3_bwd")
    return outs


class FastDiff3x3MinvFunction(torch.autograd.Function):
    """utils/utils.py:8-18."""

    @staticmethod
    def forward(ctx, input):
        invs, chk = minv3x3(input.contiguous())
        ctx.save_for_backward(invs, chk)
        ctx.mark_non_differentiable(chk)
        return invs, chk

    @staticmethod
    def backward(ctx, grad_input, grad_check):
        invs, _ = ctx.saved_tensors
        return minv3x3_backward(grad_input.contiguous(), invs), None


# --------------------------------------------------------------------------------------------------
# GridSamplerMine
# --------------------------------------------------------------------------------------------------
def _gs_dims(inp, grid, layout):
    if inp.dim() != 5 or grid.dim() != 5:
        raise RuntimeError("grid_sampler(): expected 5D input and grid")
    if inp.size(0) != grid.size(0) or grid.size(-1) != 3:
        raise RuntimeError("grid_sampler(): inconsistent input / grid sizes")
    if inp.dtype != grid.dtype:
        raise RuntimeError("grid_sampler(): expected input and grid to have same dtype")
    if layout == LAYOUT_NCDHW:
        N, C, D, H, W = inp.shape
    else:
        N, D, H, W, C = inp.shape
    P = grid.size(1) * grid.size(2) * grid.size(3)
    return N, C, D, H, W, P


def grid_sample3d_forward(inp, grid, layout=LAYOUT_NCDHW):
    """GridSamplerMine.forward(input, grid, 0, 1)  (MCAcc/cuda/GridSamplerMine.cpp:75-81)."""
    _check_input(inp, "input")
    _check_input(grid, "grid")
    code = _dtype_code(inp, "input")
    N, C, D, H, W, P = _gs_dims(inp, grid, layout)
    out = torch.empty((N, C, grid.size(1), grid.size(2), grid.size(3)), dtype=inp.dtype,
                      device=inp.device)
    with torch.cuda.device(inp.device):
        check(_lib.load().recmv_gridsample3d_fwd(_ptr(inp), _ptr(grid), _ptr(out), N, C, D, H, W, P,
                                                 code, layout, _stream(inp)),
              "recmv_gridsample3d_fwd")
    return out


def grid_sample3d_backward(inp, grid, grad_out, layout=LAYOUT_NCDHW, need_grad_input=True):
    """GridSamplerMine.backward(input, grid, grad_output, 0, 1) -> (grad_input, grad_grid)."""
    _check_input(inp, "input")
    _check_input(grid, "grid")
    grad_out = grad_out.contiguous()
    code = _dtype_code(inp, "input")
    N, C, D, H, W, P = _gs_dims(inp, grid, layout)
    gi = torch.zeros_like(inp) if need_grad_input else None
    gg = torch.empty_like(grid)
    with torch.cuda.device(inp.device):
        check(_lib.load().recmv_gridsample3d_bwd(_ptr(inp), _ptr(grid), _ptr(grad_out), _ptr(gi),
                                                 _ptr(gg), N, C, D, H, W, P, code, layout,
                                                 _stream(inp)), "recmv_gridsample3d_bwd")
    return gi, gg


def grid_sample3d_dbackward(gg_input, gg_grid, inp, grid, grad_out, layout=LAYOUT_NCDHW,
                            need_grad_input=True):
    """GridSamplerMine.dbackward(ggI, ggG, input, grid, grad_output, 0, 1) -> (gI, gG, ggO)."""
    _check_input(inp, "input")
    _check_input(grid, "grid")
    grad_out = grad_out.contiguous()
    gg_grid = gg_grid.contiguous()
    if gg_input is not None:
        gg_input = gg_input.contiguous()
    code = _dtype_code(inp, "input")
    N, C, D, H, W, P = _gs_dims(inp, grid, layout)
    gi = torch.zeros_like(inp) if need_grad_input else None
    gg = torch.empty_like(grid)
    ggo = torch.empty_like(grad_out)
    with torch.cuda.device(inp.device):
        check(_lib.load().recmv_gridsample3d_bwd2(_ptr(gg_input), _ptr(gg_grid), _ptr(inp), _ptr(grid),
                                                  _ptr(grad_out), _ptr(gi), _ptr(gg), _ptr(ggo), N, C,
                                                  D, H, W, P, code, layout, _stream(inp)),
              "recmv_gridsample3d_bwd2")
    return gi, gg, ggo


class GridSamplerMine3dFunction(torch.autograd.Function):
    """MCAcc/grid_sampler_mine.py:8-46 -- twice differentiable trilinear/border sampler."""

    @staticmethod
    def forward(ctx, input, grid, mode="bilinear", padding_mode="border", align_corners=False):
        if align_corners:
            raise NotImplementedError
        input = input.contiguous()
        grid = grid.contiguous()
        ctx.save_for_backward(input, grid)
        return grid_sample3d_forward(input, grid)

    @staticmethod
    def backward(ctx, grad_output):
        input, grid = ctx.saved_tensors
        o0, o1 = GridSamplerMine3dBackwardFunction.apply(input, grid, grad_output)
        return o0, o1, None, None, None


class GridSamplerMine3dBackwardFunction(torch.autograd.Function):
    """MCAcc/grid_sampler_mine.py:48-65.  grad_input is only materialised when the voxel itself
    requires grad (the reference always fills a full zero volume, GridSamplerMineKernel.cu:955)."""

    @staticmethod
    def forward(ctx, input, grid, grad_output):
        ctx.save_for_backward(input, grid, grad_output)
        ctx.need_gi = bool(input.requires_grad)
        gi, gg = grid_sample3d_backward(input, grid, grad_output, need_grad_input=ctx.need_gi)
        if gi is None:
            gi = input.new_zeros(())  # placeholder, never consumed (input does not require grad)
            ctx.mark_non_differentiable(gi)
        return gi, gg

    @staticmethod
    def backward(ctx, grad_output_input, grad_output_grid):
        input, grid, grad_output = ctx.saved_tensors
        ggi = grad_output_input if ctx.need_gi else None
        if grad_output_grid is None:
            grad_output_grid = torch.zeros_like(grid)
        o0, o1, o2 = grid_sample3d_dbackward(ggi, grad_output_grid, input, grid, grad_output,
                                             need_grad_input=ctx.need_gi)
        return o0, o1, o2


class FrozenVoxelSampleFunction(torch.autograd.Function):
    """Twice-differentiable trilinear / border sample of a FROZEN channels-last voxel [1,D,H,W,C] (the cached layout of
    LBSkinner.ws: one corner = C contiguous floats) -- the autograd path of LBSkinner.forward.  Same kernels as
    GridSamplerMine3dFunction (recmv_gridsample3d_{fwd,bwd,bwd2}) with layout NDHWC; the voxel gets no gradient."""

    @staticmethod
    def forward(ctx, voxel_cl, grid):
        grid = grid.contiguous()
        ctx.save_for_backward(voxel_cl, grid)
        return grid_sample3d_forward(voxel_cl, grid, LAYOUT_NDHWC)

    @staticmethod
    def backward(ctx, grad_output):
        voxel_cl, grid = ctx.saved_tensors
        return None, _FrozenVoxelSampleBackward.apply(voxel_cl, grid, grad_output)


class _FrozenVoxelSampleBackward(torch.autograd.Function):
    @staticmethod
    def forward(ctx, voxel_cl, grid, grad_output):
        ctx.save_for_backward(voxel_cl, grid, grad_output)
        return grid_sample3d_backward(voxel_cl, grid, grad_output, LAYOUT_NDHWC, need_grad_input=False)[1]

    @staticmethod
    def backward(ctx, gg_grid):
        voxel_cl, grid, grad_output = ctx.saved_tensors
        _, g_grid, gg_out = grid_sample3d_dbackward(None, gg_grid.contiguous(), voxel_cl, grid, grad_output, LAYOUT_NDHWC,
                                                    need_grad_input=False)
        return None, g_grid, gg_out


def voxel_to_channels_last(ws):
    """[1,C,D,H,W] fp32 -> [D,H,W,C] (private, coalesced copy of LBSkinner.ws)."""
    _check_input(ws, "ws")
    _, C, D, H, W = ws.shape
    out = torch.empty((D, H, W, C), dtype=torch.float32, device=ws.device)
    with torch.cuda.device(ws.device):
        check(_lib.load().recmv_voxel_to_channels_last(_ptr(ws), _ptr(out), C, D, H, W, _stream(ws)),
              "recmv_voxel_to_channels_last")
    return out


# --------------------------------------------------------------------------------------------------
# MCGpu
# --------------------------------------------------------------------------------------------------
_mc_state = {}   # per device: grow-only scratch + output buffers (like the MCGpu singleton, MCGpu/CudaKernels.cu:524-604)


def _mc_buffers(dev, nbytes, cap_v, cap_f):
    st = _mc_state.setdefault(dev.index, {})
    if st.get("scratch") is None or st["scratch"].numel() < nbytes:
        st["scratch"] = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    if st.get("verts") is None or st["verts"].shape[0] < cap_v:
        st["verts"] = torch.empty((cap_v, 3), dtype=torch.float32, device=dev)
    if st.get("faces") is None or st["faces"].shape[0] < cap_f:
        st["faces"] = torch.empty((cap_f, 3), dtype=torch.int64, device=dev)
    if st.get("counts") is None:
        st["counts"] = torch.zeros((4,), dtype=torch.int32, device=dev)
        st["counts_host"] = torch.zeros((4,), dtype=torch.int32).pin_memory()
    return st


def mc_gpu(sdfs, xstep=1.0, ystep=1.0, zstep=1.0, xmin=0.0, ymin=0.0, zmin=0.0, fTargetValue=0.0):
    """MCGpu.mc_gpu(sdfs, steps, mins, iso) -> [verts [V,3] f32, faces [F,3] i64]
    (MCGpu/MCGpu.cpp:20-56).  Wrong dtype returns [] exactly like the reference (:41-42).

    One C call queues every pass (sign mask, count, scan, vertices, faces) into grow-only capacity buffers; the single
    host synchronisation is the read of (V, F) AFTER everything is queued (the reference blocks between its kernels,
    CudaKernels.cu:628).  The results are fresh tensors, as the reference returns (MCGpu.cpp:49-54)."""
    _check_input(sdfs, "sdfs")
    if sdfs.dtype != torch.float32:
        return []
    if sdfs.dim() != 3 or min(sdfs.shape) <= 0:
        return []
    NX, NY, NZ = sdfs.shape
    lib = _lib.load()
    nbytes = c_size_t(0)
    check(lib.recmv_mc_scratch_bytes(NX, NY, NZ, byref(nbytes)), "recmv_mc_scratch_bytes")
    dev = sdfs.device
    prev = _mc_state.get(dev.index, {})
    cap_v = max(4096, prev["verts"].shape[0] if prev.get("verts") is not None else 0)
    cap_f = max(8192, prev["faces"].shape[0] if prev.get("faces") is not None else 0)
    step = (c_float * 3)(xstep, ystep, zstep)
    org = (c_float * 3)(xmin, ymin, zmin)
    with torch.cuda.device(dev):
        stream = _stream(sdfs)
        for _ in range(2):
            st = _mc_buffers(dev, nbytes.value, cap_v, cap_f)
            check(lib.recmv_mc_run(_ptr(sdfs), NX, NY, NZ, float(fTargetValue), _ptr(st["scratch"]), step, org,
                                   _ptr(st["verts"]), st["verts"].shape[0], _ptr(st["faces"]), st["faces"].shape[0],
                                   _ptr(st["counts"]), stream), "recmv_mc_run")
            st["counts_host"].copy_(st["counts"], non_blocking=True)
            torch.cuda.current_stream(dev).synchronize()
            V, F, overflow = (int(v) for v in st["counts_host"][:3])
            if V >= (1 << 25):
                check(_lib.RECMV_E_RANGE, "recmv_mc_run (more than 2^25 vertices)")
            if not overflow:
                break
            cap_v, cap_f = int(V * 1.25) + 1024, int(F * 1.25) + 2048   # grow once, re-run (buffers are kept)
        else:
            raise _lib.RecmvError("recmv_mc_run: output buffers still too small after growing")
        return [st["verts"][:V].clone(), st["faces"][:F].clone()]


def mc_gpu_two_call(sdfs, step=(1.0, 1.0, 1.0), origin=(0.0, 0.0, 0.0), iso=0.0):
    """The count / emit pair of the C ABI (exact-size outputs; synchronises between the two calls like the reference)."""
    _check_input(sdfs, "sdfs")
    NX, NY, NZ = sdfs.shape
    lib = _lib.load()
    nbytes = c_size_t(0)
    check(lib.recmv_mc_scratch_bytes(NX, NY, NZ, byref(nbytes)), "recmv_mc_scratch_bytes")
    scratch = torch.empty((nbytes.value,), dtype=torch.uint8, device=sdfs.device)
    V, F = c_int64(0), c_int64(0)
    with torch.cuda.device(sdfs.device):
        st = _stream(sdfs)
        check(lib.recmv_mc_count(_ptr(sdfs), NX, NY, NZ, float(iso), _ptr(scratch), byref(V), byref(F), st), "recmv_mc_count")
        verts = torch.empty((V.value, 3), dtype=torch.float32, device=sdfs.device)
        faces = torch.empty((F.value, 3), dtype=torch.int64, device=sdfs.device)
        if V.value > 0:
            check(lib.recmv_mc_emit(_ptr(sdfs), NX, NY, NZ, float(iso), _ptr(scratch), (c_float * 3)(*step),
                                    (c_float * 3)(*origin), _ptr(verts), _ptr(faces) if F.value > 0 else None, st),
                  "recmv_mc_emit")
    return [verts, faces]


# --------------------------------------------------------------------------------------------------
# LBS
# --------------------------------------------------------------------------------------------------
def make_voxel(ws_cl, center, extend):
    v = Voxel()
    v.ws_cl = ws_cl.data_ptr()
    v.D, v.H, v.W = int(ws_cl.shape[0]), int(ws_cl.shape[1]), int(ws_cl.shape[2])
    c = [float(x) for x in center]
    v.center = (c_float * 3)(*c)
    v.extend = float(extend)
    return v


def lbs_forward(ps, A, trans, ws_cl, center, extend, batch_inds=None, points_per_frame=0, tps=None,
                want_weights=False):
    ps = ps.contiguous().float()
    A = A.contiguous().float()
    trans = trans.contiguous().float()
    P = ps.numel() // 3
    out = torch.empty_like(ps)
    wout = torch.empty((P, 24), dtype=torch.float32, device=ps.device) if want_weights else None
    if tps is not None:
        tps = tps.contiguous().float()
    if batch_inds is not None:
        batch_inds = batch_inds.contiguous().long()
    vox = make_voxel(ws_cl, center, extend)
    with torch.cuda.device(ps.device):
        check(_lib.load().recmv_lbs_fwd(_ptr(ps), _ptr(tps), _ptr(A), _ptr(trans), _ptr(batch_inds),
                                        int(points_per_frame), int(A.shape[0]), byref(vox), _ptr(out),
                                        _ptr(wout), P, _stream(ps)), "recmv_lbs_fwd")
    return (out, wout) if want_weights else out


def lbs_inverse(x_obs, A, trans, ws_cl, center, extend, batch_inds=None, points_per_frame=0):
    x_obs = x_obs.contiguous().float()
    A = A.contiguous().float()
    trans = trans.contiguous().float()
    P = x_obs.numel() // 3
    xc = torch.empty_like(x_obs)
    valid = torch.empty((P,), dtype=torch.uint8, device=x_obs.device)
    if batch_inds is not None:
        batch_inds = batch_inds.contiguous().long()
    vox = make_voxel(ws_cl, center, extend)
    with torch.cuda.device(x_obs.device):
        check(_lib.load().recmv_lbs_inverse(_ptr(x_obs), _ptr(A), _ptr(trans), _ptr(batch_inds),
                                            int(points_per_frame), int(A.shape[0]), byref(vox),
                                            _ptr(xc), _ptr(valid), P, _stream(x_obs)),
              "recmv_lbs_inverse")
    return xc, valid.view(torch.bool)


def bone_matrices(poses, Js, parents_i32, init_pose=None, want_A=True):
    """(G [F,24,4,4], A [F,24,4,4] or None): the kinematic chain of LBSkinner in one launch (no autograd)."""
    poses = poses.detach().contiguous().float()
    _check_input(poses, "poses")
    F_ = poses.shape[0]
    dev = poses.device
    G = torch.empty((F_, 24, 4, 4), dtype=torch.float32, device=dev)
    A = torch.empty((F_, 24, 4, 4), dtype=torch.float32, device=dev) if want_A else None
    ip = init_pose.contiguous().float() if init_pose is not None else None
    with torch.cuda.device(dev):
        check(_lib.load().recmv_bone_matrices(_ptr(poses), _ptr(Js.contiguous().float()), _ptr(parents_i32), _ptr(ip),
                                              _ptr(G), _ptr(A), F_, _stream(poses)), "recmv_bone_matrices")
    return G, A


# --------------------------------------------------------------------------------------------------
# SDF MLP
# --------------------------------------------------------------------------------------------------
SDF_LAYER_SHAPES = [(512, 39), (512, 512), (512, 512), (473, 512), (512, 512), (512, 512), (512, 512),
                    (512, 512), (257, 512)]


def sdf_pack_weights(Ws, bs):
    """Ws[l] [out,in] effective fp32 weights (weight-norm applied), bs[l] [out] -> packed device blob."""
    dev = Ws[0].device
    for (o, i), W, b in zip(SDF_LAYER_SHAPES, Ws, bs):
        if tuple(W.shape) != (o, i) or tuple(b.shape) != (o,):
            raise RuntimeError(f"unexpected SDF layer shape {tuple(W.shape)} (want {(o, i)})")
    W_all = torch.cat([W.detach().reshape(-1).float() for W in Ws]).contiguous()
    b_all = torch.cat([b.detach().reshape(-1).float() for b in bs]).contiguous()
    lib = _lib.load()
    nbytes = lib.recmv_sdf_packed_bytes()
    # 1 KiB alignment for the TMA-visible planes
    raw = torch.empty((nbytes + 1024,), dtype=torch.uint8, device=dev)
    off = (-raw.data_ptr()) % 1024
    packed = raw[off:off + nbytes]
    with torch.cuda.device(dev):
        check(lib.recmv_sdf_pack_weights(_ptr(W_all), _ptr(b_all), _ptr(packed), _stream(W_all)),
              "recmv_sdf_pack_weights")
    packed._keepalive = raw
    return packed


def _pe_array(pe_w):
    pe_w = [1.0] * 12 if pe_w is None else [float(w) for w in pe_w]
    if len(pe_w) != 12:
        raise RuntimeError("pe_w must hold 12 annealing weights")
    return (c_float * 12)(*pe_w)


def sdf_mlp_forward(x, packed, pe_w=None, mode=None, want_feat=True):
    """ImplicitNetwork.forward on canonical points x [P,3] -> (sdf [P,1], feat [P,256] or None)."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    x = x.contiguous().float()
    _check_input(x, "x")
    P = x.shape[0]
    sdf = torch.empty((P, 1), dtype=torch.float32, device=x.device)
    feat = torch.empty((P, 256), dtype=torch.float32, device=x.device) if want_feat else None
    with torch.cuda.device(x.device):
        check(_lib.load().recmv_sdf_mlp_fwd(_ptr(x), _ptr(packed), _pe_array(pe_w), _ptr(sdf),
                                            _ptr(feat), P, mode, _stream(x)), "recmv_sdf_mlp_fwd")
    return sdf, feat


def sdf_value_and_grad(x, packed, pe_w=None, mode=None, want_feat=False):
    """(sdf [P,1], d sdf/d x [P,3], feat or None) in ONE forward-mode launch (no graph is recorded)."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    if mode == MLP_FP32_SIMT:
        raise _lib.RecmvError("the fused value+gradient launch exists for the tcgen05 modes only")
    x = x.contiguous().float()
    _check_input(x, "x")
    P = x.shape[0]
    sdf = torch.empty((P, 1), dtype=torch.float32, device=x.device)
    grad = torch.empty((P, 3), dtype=torch.float32, device=x.device)
    feat = torch.empty((P, 256), dtype=torch.float32, device=x.device) if want_feat else None
    with torch.cuda.device(x.device):
        check(_lib.load().recmv_sdf_mlp_fwd_grad(_ptr(x), _ptr(packed), _pe_array(pe_w), _ptr(sdf), _ptr(feat),
                                                 _ptr(grad), P, mode, _stream(x)), "recmv_sdf_mlp_fwd_grad")
    return sdf, grad, feat


# --------------------------------------------------------------------------------------------------
# Training path: fused forward that saves the layer inputs + tcgen05 backward GEMMs (csrc/gemm3.cu)
# --------------------------------------------------------------------------------------------------
ACT_NONE, ACT_SOFTPLUS100, ACT_RELU = 0, 1, 2
# "planes": forward / backward-data layer GEMMs fed by TMA from fp16 hi / lo operand planes (csrc/gemm3_tma.cu);
# "producers": the first-generation kernel that converts fp32 operands in its main loop (csrc/gemm3.cu).  The weight
# gradient uses the latter in both settings.
import os as _os
TRAIN_GEMM = _os.environ.get("RECMV_TRAIN_GEMM", "planes")
# create_graph=True input gradients: "1" = differentiable reverse chain on the tcgen05 GEMMs (second_order.py), "0" = torch graph
SECOND_ORDER_FUSED = _os.environ.get("RECMV_SECOND_ORDER", "1") != "0"
_INPUT_GRAD_ONLY = [0]


class input_grad_only:
    """`with ops.input_grad_only(): torch.autograd.grad(y, x, ..., create_graph=True)` -- tells the training Functions that
    this differentiation asks for INPUT gradients only (ctx.needs_input_grad cannot: it reflects requires_grad at forward
    time, and the parameters always require grad while training).  The mirrors of the reference's call sites use it
    (ImplicitNetwork.gradient, utils.compute_Jacobian, utils.compute_deformed_normals).  The backward runs on autograd's
    device thread, so the flag is process-wide, not thread-local (one process drives one GPU)."""

    def __enter__(self):
        _INPUT_GRAD_ONLY[0] += 1
        return self

    def __exit__(self, *exc):
        _INPUT_GRAD_ONLY[0] -= 1
        return False


def _inputs_only(need_params):
    return SECOND_ORDER_FUSED and (not need_params or _INPUT_GRAD_ONLY[0] > 0)
_INV_SQRT2 = 0.70710678118654752440


def _ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() if t is not None else None for t in tensors])


def grad_dyn_scale(*cotangents):
    """Device scalar 2^-floor(log2(max|g|)) (1 for an all-zero cotangent): brings the largest cotangent entry into
    [1, 2) before the fp16 hi/lo split of the backward GEMMs; no host synchronisation."""
    m = torch.stack([c.detach().abs().amax() for c in cotangents if c is not None]).amax().float()
    e = torch.floor(torch.log2(m.clamp_min(1e-30)))
    s = torch.exp2(-e.clamp(-100.0, 100.0))
    return torch.where(m > 0, s, torch.ones_like(s)).reshape(1).contiguous()


def mlp_bwd_data_layer(G, W, out_dim, in_dim, saved_input, act, G_prev, split=0, D2=None, out_scale=1.0, dyn_scale=None):
    """G_prev[:, :split] = ((G[:, :out_dim] @ W) * out_scale)[:, :split] * act'(saved_input); columns >= split -> D2."""
    P = G.shape[0]
    with torch.cuda.device(G.device):
        check(_lib.load().recmv_mlp_bwd_data_layer(
            _ptr(G), G.stride(0), _ptr(W), int(out_dim), int(in_dim), _ptr(saved_input),
            saved_input.stride(0) if saved_input is not None else 0, int(act), int(split), _ptr(G_prev), G_prev.stride(0),
            _ptr(D2), D2.stride(0) if D2 is not None else 0, float(out_scale), _ptr(dyn_scale), P, _stream(G)),
            "recmv_mlp_bwd_data_layer")
    return G_prev


def mlp_bwd_weight(Gs, Xs, out_dims, in_dims, out_scales=None, dyn_scale=None, want_bias=True):
    """dW[l] = out_scale[l] * Gs[l][:, :out]^T @ Xs[l][:, :in] and db[l] = Gs[l][:, :out].sum(0), all layers in one launch."""
    n = len(Gs)
    dev = Gs[0].device
    P = Gs[0].shape[0]
    dW = [torch.empty((o, i), dtype=torch.float32, device=dev) for o, i in zip(out_dims, in_dims)]
    db = [torch.zeros((o,), dtype=torch.float32, device=dev) for o in out_dims] if want_bias else None
    scales = (c_float * n)(*[float(v) for v in (out_scales or [1.0] * n)])
    with torch.cuda.device(dev):
        check(_lib.load().recmv_mlp_bwd_weight(
            n, _ptr_array(Gs), (c_int64 * n)(*[g.stride(0) for g in Gs]), _ptr_array(Xs),
            (c_int64 * n)(*[x.stride(0) for x in Xs]), (ctypes.c_int * n)(*out_dims), (ctypes.c_int * n)(*in_dims),
            _ptr_array(dW), _ptr_array(db) if db is not None else None, scales, _ptr(dyn_scale), P, _stream(Gs[0])),
            "recmv_mlp_bwd_weight")
    return dW, db


def mlp_fwd_layer(X, W, bias, out_dim, in_dim, act, Y, pre_scale=1.0, split=0, Y2=None):
    """Y[:, :split or out] (and Y2) = act(pre_scale * X[:, :in] @ W.T + bias) on tcgen05 (training forward, one layer)."""
    P = X.shape[0]
    with torch.cuda.device(X.device):
        check(_lib.load().recmv_mlp_fwd_layer(_ptr(X), X.stride(0), _ptr(W), _ptr(bias), int(out_dim), int(in_dim), int(act),
                                              float(pre_scale), int(split), _ptr(Y), Y.stride(0), _ptr(Y2),
                                              Y2.stride(0) if Y2 is not None else 0, P, _stream(X)), "recmv_mlp_fwd_layer")
    return Y


def pe_forward(x, pe_w, bands, out, out2=None):
    """out[:, :3 + 6 bands] (and out2) = positional encoding of x [P,3] with annealing weights pe_w."""
    w = (c_float * (2 * bands))(*[float(v) for v in pe_w[:2 * bands]])
    with torch.cuda.device(x.device):
        check(_lib.load().recmv_pe_forward(_ptr(x), w, int(bands), _ptr(out), out.stride(0), _ptr(out2),
                                           out2.stride(0) if out2 is not None else 0, x.shape[0], _stream(x)),
              "recmv_pe_forward")
    return out


def _pad8(n):
    return (int(n) + 7) // 8 * 8


def split_planes(t, rows, cols, scale, scale_dev=None, transpose=False, ldp=None):
    """fp32 [rows, >= cols] -> (hi, lo) fp16 planes of scale (* scale_dev) * t, [rows][ldp] or transposed [cols][ldp]."""
    dev = t.device
    ldp = ldp or _pad8(rows if transpose else cols)
    shape = (cols, ldp) if transpose else (rows, ldp)
    hi = torch.zeros(shape, dtype=torch.float16, device=dev)
    lo = torch.zeros(shape, dtype=torch.float16, device=dev)
    with torch.cuda.device(dev):
        check(_lib.load().recmv_split_planes(_ptr(t), t.stride(0), int(rows), int(cols), float(scale), _ptr(scale_dev),
                                             1 if transpose else 0, _ptr(hi), _ptr(lo), ldp, _stream(t)), "recmv_split_planes")
    return hi, lo


def weight_planes(W, transpose=False):
    """Operand planes of a layer's weight matrix ([out][in], scale 1024; transpose=True: [in][out], the backward-data
    operand), computed once per tensor OBJECT and version: the forward, the reverse chain and the two second-order passes of
    one training step all see the same weight tensor, so three of four splits are cache hits.  The cache lives on the tensor
    (an attribute), so it dies with it -- no address-keyed table that could go stale."""
    if W.is_leaf:
        # a Parameter can be rewritten through `.data` without a version bump: never cache on leaves (weight-normed layers
        # hand over a fresh non-leaf W = g v / |v| every forward, which is the case the cache is for)
        Wd = W.detach().contiguous().float()
        return split_planes(Wd, Wd.shape[0], Wd.shape[1], 1024.0, transpose=transpose)
    ver = W._version
    cache = getattr(W, "_recmv_planes", None)
    if cache is None or cache[0] != ver:
        cache = (ver, {})
        try:
            W._recmv_planes = cache
        except AttributeError:
            pass
    if transpose not in cache[1]:
        Wd = W.detach().contiguous().float()
        cache[1][transpose] = split_planes(Wd, Wd.shape[0], Wd.shape[1], 1024.0, transpose=transpose)
    return cache[1][transpose]


def pe_forward_planes(x, pe_w, bands, out, out_hi, out_lo):
    w = (c_float * (2 * bands))(*[float(v) for v in pe_w[:2 * bands]])
    with torch.cuda.device(x.device):
        check(_lib.load().recmv_pe_forward_planes(_ptr(x), w, int(bands), _ptr(out), out.stride(0) if out is not None else 0,
                                                  _ptr(out_hi), _ptr(out_lo), out_hi.stride(0), x.shape[0], _stream(x)),
              "recmv_pe_forward_planes")


def mlp_layer_planes(a_planes, b_planes, M, N, K, mode, Y, bias=None, saved_input=None, scale=1.0, dyn=None, a_has_dyn=False,
                     split=0, Y2=None, y_planes=None, planes_with_dyn=False):
    """One TMA-fed layer GEMM on operand planes (recmv_mlp_layer_planes); modes: 4/5/6 forward none/softplus/relu,
    0/1/2 backward-data none/softplus'/relu'."""
    ah, al = a_planes
    bh, bl = b_planes
    yh, yl = y_planes if y_planes is not None else (None, None)
    with torch.cuda.device(Y.device):
        check(_lib.load().recmv_mlp_layer_planes(
            _ptr(ah), _ptr(al), ah.stride(0), _ptr(bh), _ptr(bl), bh.stride(0), int(M), int(N), int(K), int(mode), _ptr(bias),
            _ptr(saved_input), saved_input.stride(0) if saved_input is not None else 0, float(scale), _ptr(dyn),
            1 if a_has_dyn else 0, int(split), _ptr(Y), Y.stride(0), _ptr(Y2), Y2.stride(0) if Y2 is not None else 0, _ptr(yh),
            _ptr(yl), yh.stride(0) if yh is not None else 0, 1 if planes_with_dyn else 0, _stream(Y)), "recmv_mlp_layer_planes")
    return Y


_WGRAD_WS = {}


def _wgrad_workspace(dev):
    key = (dev.type, dev.index)
    if key not in _WGRAD_WS:
        with torch.cuda.device(dev):
            n = int(_lib.load().recmv_mlp_wgrad_workspace_floats())
        _WGRAD_WS[key] = (torch.empty((n,), dtype=torch.float32, device=dev), torch.empty((128 * 512,), dtype=torch.float32, device=dev))
    return _WGRAD_WS[key]


def mlp_wgrad_planes(g_planes, x_planes, P, out_dim, in_dim, scale=1.0, dyn=None, want_bias=False):
    """dW [out_dim, in_dim] = scale * G^T X from the operand planes the layer GEMMs wrote (recmv_mlp_wgrad_planes); with
    want_bias also db [out_dim] = sum over samples of g (same launch) -> (dW, db)."""
    gh, gl = g_planes
    xh, xl = x_planes
    dev = gh.device
    ws, _ = _wgrad_workspace(dev)
    dW = torch.empty((out_dim, in_dim), dtype=torch.float32, device=dev)
    db = torch.empty((out_dim,), dtype=torch.float32, device=dev) if want_bias else None
    with torch.cuda.device(dev):
        check(_lib.load().recmv_mlp_wgrad_planes(_ptr(gh), _ptr(gl), gh.stride(0), _ptr(xh), _ptr(xl), xh.stride(0), int(P),
                                                 int(out_dim), int(in_dim), float(scale), _ptr(dyn), _ptr(ws), _ptr(dW), _ptr(db),
                                                 _stream(gh)), "recmv_mlp_wgrad_planes")
    return (dW, db) if want_bias else dW


def colsum(G, cols):
    """sum over rows of G[:, :cols] (fp32, deterministic two-stage reduction): the bias gradient."""
    _, part = _wgrad_workspace(G.device)
    out = torch.empty((cols,), dtype=torch.float32, device=G.device)
    with torch.cuda.device(G.device):
        check(_lib.load().recmv_colsum(_ptr(G), G.stride(0), G.shape[0], int(cols), _ptr(part), _ptr(out), _stream(G)),
              "recmv_colsum")
    return out


def softplus_tangent_planes(tz, a, h, cols, u, u_planes, inj, plane_scale=64.0):
    """u[:, :cols] = softplus_100'(z) * tz (+ planes), inj[:, :cols] = softplus_100''(z) * (h / softplus') * tz, from the saved
    softplus output a (second_order.py's tangent pass; one launch)."""
    with torch.cuda.device(tz.device):
        check(_lib.load().recmv_softplus_tangent_planes(
            _ptr(tz), tz.stride(0), _ptr(a), a.stride(0), _ptr(h), h.stride(0), tz.shape[0], int(cols), float(plane_scale), _ptr(u),
            u.stride(0), _ptr(u_planes[0]), _ptr(u_planes[1]), u_planes[0].stride(0), _ptr(inj), inj.stride(0), _stream(tz)),
            "recmv_softplus_tangent_planes")


def add_split_planes(y, addend, cols, y_planes, scale=64.0, scale_dev=None):
    """y[:, :cols] += addend[:, :cols] in place, and the planes of the sum scaled scale (* scale_dev)."""
    with torch.cuda.device(y.device):
        check(_lib.load().recmv_add_split_planes(_ptr(y), y.stride(0), _ptr(addend), addend.stride(0), y.shape[0], int(cols),
                                                 float(scale), _ptr(scale_dev), _ptr(y_planes[0]), _ptr(y_planes[1]),
                                                 y_planes[0].stride(0), _stream(y)), "recmv_add_split_planes")


def pe_backward(x, g, g2, pe_w, bands, dx=None):
    """dx (+)= (d PE/d x)^T (g + g2); g / g2 [P, >= 3 + 6 bands] (row stride free), x [P,3]."""
    P = x.shape[0]
    acc = dx is not None
    if dx is None:
        dx = torch.empty((P, 3), dtype=torch.float32, device=x.device)
    w = (c_float * (2 * bands))(*[float(v) for v in pe_w[:2 * bands]])
    with torch.cuda.device(x.device):
        check(_lib.load().recmv_pe_backward(_ptr(x), _ptr(g), g.stride(0), _ptr(g2), g2.stride(0) if g2 is not None else 0,
                                            w, int(bands), _ptr(dx), 1 if acc else 0, P, _stream(x)), "recmv_pe_backward")
    return dx


def _pe_torch(x, pe_w, bands):
    outs, f = [x], 1.0
    for k in range(bands):
        outs += [pe_w[2 * k] * torch.sin(x * f), pe_w[2 * k + 1] * torch.cos(x * f)]
        f *= 2.0
    return torch.cat(outs, -1)


def _sdf_composite(x, Ws, bs, pe_w):
    """The same network as a torch graph (model/network.py:89-119) -- the twice-differentiable fallback of the
    training Function's backward when the caller asked for create_graph=True."""
    pe = _pe_torch(x, pe_w, 6)
    h = pe
    for l in range(9):
        if l == 4:
            h = torch.cat([h, pe], 1) * _INV_SQRT2
        h = torch.nn.functional.linear(h, Ws[l], bs[l])
        if l < 8:
            h = torch.nn.functional.softplus(h, beta=100)
    return h[:, :1], h[:, 1:]


class SdfMlpTrainFunction(torch.autograd.Function):
    """ImplicitNetwork.forward with gradients (model/network.py:89-119 inside train.py:317-330), all GEMMs on tcgen05
    in the engine's fp32-grade arithmetic (csrc/gemm3.cu: fp16 hi/lo split, 3 MMAs per product, fp32 accumulation).

    forward : PE kernel + 9 layer launches  Y = softplus(X W^T + b)  whose outputs stay in HBM as the next layer's input
              AND as what the backward needs (16 KB per point -- what autograd keeps for the reference's graph); the skip
              concatenation is a column range of layer 4's input buffer, its 1/sqrt2 a scale of that layer's GEMM.
              (The inference engine keeps activations on-chip; a variant of it that also streamed them to HBM was
              built and dropped: it fails above ~50 k points per call, profiles/r02_notes.md.)
    backward: first order (`loss.backward()`, parameter VJPs of propagateTmpPsGrad) -> 9 backward-data launches + nine
              weight-gradient launches on the same operand planes (recmv_mlp_wgrad_planes) + the PE Jacobian; weight-norm's
              (g, v) and anything upstream of x stay ordinary autograd.  Called with create_graph=True for the INPUT gradient
              (eikonal / normals, network.py:121-133, inside ops.input_grad_only()) the backward returns the reverse chain as
              a differentiable op on the same GEMMs (recmv_b200/second_order.py); a create_graph call that also wants
              parameter gradients with a graph re-runs the network as a torch graph (cuBLAS); `last_backward` says which ran."""
    last_backward = None

    @staticmethod
    def forward(ctx, x, pe_w, mode, packed, *Wb):
        Ws, bs = Wb[:9], Wb[9:]
        W_in = Ws
        if not (x.is_contiguous() and x.dtype == torch.float32 and x.dim() == 2):
            raise RuntimeError("SdfMlpTrainFunction expects a contiguous float32 [P,3] tensor (convert outside, in the graph)")
        P = x.shape[0]
        dev = x.device
        Ws = [w.detach().contiguous().float() for w in Ws]
        bs = [b.detach().contiguous().float() for b in bs]
        act = [torch.empty((P, 64), dtype=torch.float32, device=dev)] + \
              [torch.empty((P, 512), dtype=torch.float32, device=dev) for _ in range(8)]
        sdf = torch.empty((P, 1), dtype=torch.float32, device=dev)
        feat = torch.empty((P, 256), dtype=torch.float32, device=dev)
        if TRAIN_GEMM == "planes":
            # operands as fp16 hi / lo planes, TMA-fed GEMMs (csrc/gemm3_tma.cu): each layer writes its output in fp32
            # (kept for the backward) AND as the next layer's A planes
            xp = [(torch.empty((P, 64), dtype=torch.float16, device=dev), torch.empty((P, 64), dtype=torch.float16, device=dev))]
            xp += [(torch.empty((P, 512), dtype=torch.float16, device=dev), torch.empty((P, 512), dtype=torch.float16, device=dev))
                   for _ in range(8)]
            pe_forward_planes(x, pe_w, 6, act[0], xp[0][0], xp[0][1])
            pe_forward_planes(x, pe_w, 6, act[4][:, 473:], xp[4][0][:, 473:], xp[4][1][:, 473:])
            for l in range(9):
                o, i = Ws[l].shape
                wp = weight_planes(W_in[l])
                if l < 8:
                    mlp_layer_planes(xp[l], wp, P, o, i, 5, act[l + 1], bias=bs[l], scale=_INV_SQRT2 if l == 4 else 1.0,
                                     y_planes=xp[l + 1])
                else:
                    mlp_layer_planes(xp[8], wp, P, 257, 512, 4, sdf, bias=bs[8], split=1, Y2=feat)
        else:
            pe_forward(x, pe_w, 6, act[0], act[4][:, 473:])
            for l in range(8):
                mlp_fwd_layer(act[l], Ws[l], bs[l], Ws[l].shape[0], Ws[l].shape[1], ACT_SOFTPLUS100, act[l + 1],
                              pre_scale=_INV_SQRT2 if l == 4 else 1.0)
            mlp_fwd_layer(act[8], Ws[8], bs[8], 257, 512, ACT_NONE, sdf, split=1, Y2=feat)
        ctx.pe_w, ctx.mode = [float(w) for w in pe_w], mode
        ctx.has_planes = TRAIN_GEMM == "planes"
        if ctx.has_planes:      # the layer inputs' operand planes feed the weight gradient too (recmv_mlp_wgrad_planes)
            ctx.save_for_backward(x, *Wb, *act, *[t for pair in xp for t in pair])
        else:
            ctx.save_for_backward(x, *Wb, *act)
        return sdf, feat

    @staticmethod
    def backward(ctx, g_sdf, g_feat):
        saved = ctx.saved_tensors
        x, Ws, bs, act = saved[0], saved[1:10], saved[10:19], saved[19:28]
        P = x.shape[0]
        dev = x.device
        need_x = ctx.needs_input_grad[0]
        need_w = any(ctx.needs_input_grad[4:])
        if torch.is_grad_enabled() and _inputs_only(need_w):
            # create_graph=True for the INPUT gradient only (ImplicitNetwork.gradient / deformed normals): the reverse
            # chain as a differentiable op whose own backward is tangent + backward GEMMs on tcgen05 (second_order.py)
            from . import second_order
            SdfMlpTrainFunction.last_backward = "fused-tcgen05 (create_graph, input gradient)"
            dx = second_order.sdf_input_grad(x, g_sdf, g_feat, ctx.pe_w, act, Ws, bs,
                                             saved[28:46] if ctx.has_planes else ()) if need_x else None
            return (dx, None, None, None, *([None] * 18))
        if torch.is_grad_enabled():
            # create_graph=True with parameter gradients in the graph: differentiate a torch graph of the same network
            SdfMlpTrainFunction.last_backward = "autograd-composite (create_graph)"
            xi = x if x.requires_grad else x.detach().requires_grad_(need_x)
            with torch.enable_grad():
                sdf, feat = _sdf_composite(xi, Ws, bs, ctx.pe_w)
                ins = [t for t in [xi] + list(Ws) + list(bs) if t.requires_grad]
                outs, gos = [sdf], [g_sdf if g_sdf is not None else torch.zeros_like(sdf)]
                if g_feat is not None:
                    outs.append(feat); gos.append(g_feat)
                gr = torch.autograd.grad(outs, ins, gos, create_graph=True, allow_unused=True)
            it = iter(gr)
            res = [next(it) if t.requires_grad else None for t in [xi] + list(Ws) + list(bs)]
            return (res[0] if need_x else None, None, None, None, *res[1:])
        SdfMlpTrainFunction.last_backward = "fused-tcgen05"
        G8 = torch.zeros((P, 264), dtype=torch.float32, device=dev)
        if g_sdf is not None:
            G8[:, 0:1] = g_sdf
        if g_feat is not None:
            G8[:, 1:257] = g_feat
        dyn = grad_dyn_scale(G8)
        G = [None] * 9
        G[8] = G8
        dpe4 = torch.empty((P, 40), dtype=torch.float32, device=dev)
        outs = [w.shape[0] for w in Ws]
        ins = [w.shape[1] for w in Ws]
        dx = None
        planes = TRAIN_GEMM == "planes" and ctx.has_planes
        GP = [None] * 9
        if planes:
            gp = split_planes(G8, P, 257, 64.0, scale_dev=dyn, ldp=264)       # cotangent planes carry 64 * dyn
            GP[8] = gp
            for l in range(8, 0, -1):
                G[l - 1] = torch.empty((P, 512), dtype=torch.float32, device=dev)
                gprev = (torch.empty((P, 512), dtype=torch.float16, device=dev), torch.empty((P, 512), dtype=torch.float16, device=dev))
                wtp = weight_planes(Ws[l], transpose=True)                                     # [in][out]: B of backward-data
                mlp_layer_planes(gp, wtp, P, ins[l], outs[l], 1, G[l - 1], saved_input=act[l], scale=_INV_SQRT2 if l == 4 else 1.0,
                                 dyn=dyn, a_has_dyn=True, split=473 if l == 4 else 0, Y2=dpe4 if l == 4 else None,
                                 y_planes=gprev, planes_with_dyn=True)
                gp = gprev
                GP[l - 1] = gp
            if need_x:
                dpe0 = torch.empty((P, 40), dtype=torch.float32, device=dev)
                mlp_layer_planes(gp, weight_planes(Ws[0], transpose=True), P, ins[0], outs[0], 0, dpe0, dyn=dyn, a_has_dyn=True)
                dx = pe_backward(x, dpe0, dpe4, ctx.pe_w, 6)
        else:
            for l in range(8, 0, -1):
                G[l - 1] = torch.empty((P, 512), dtype=torch.float32, device=dev)
                mlp_bwd_data_layer(G[l], Ws[l].detach(), outs[l], ins[l], act[l], ACT_SOFTPLUS100, G[l - 1],
                                   split=473 if l == 4 else 0, D2=dpe4 if l == 4 else None,
                                   out_scale=_INV_SQRT2 if l == 4 else 1.0, dyn_scale=dyn)
            if need_x:
                dpe0 = torch.empty((P, 40), dtype=torch.float32, device=dev)
                mlp_bwd_data_layer(G[0], Ws[0], outs[0], ins[0], None, ACT_NONE, dpe0, dyn_scale=dyn)
                dx = pe_backward(x, dpe0, dpe4, ctx.pe_w, 6)
        dW, db = [None] * 9, [None] * 9
        if need_w and planes:
            # weight gradient straight from the planes both passes wrote (MN-major operands, no transposed copies)
            xpl = saved[28:46]
            for l in range(9):
                dW[l], db[l] = mlp_wgrad_planes(GP[l], (xpl[2 * l], xpl[2 * l + 1]), P, outs[l], ins[l],
                                                _INV_SQRT2 if l == 4 else 1.0, dyn, want_bias=True)
        elif need_w:
            dW, db = mlp_bwd_weight(G, list(act), outs, ins, [_INV_SQRT2 if l == 4 else 1.0 for l in range(9)], dyn)
        return (dx, None, None, None, *dW, *db)


def _plain_mlp_forward(X0, Ws, bs):
    """ReLU MLP on tcgen05 layer GEMMs: returns (output [P, out_last], saved layer inputs [X0, X1, ...])."""
    P, dev = X0.shape[0], X0.device
    Ws = [w.detach().contiguous().float() for w in Ws]
    bs = [b.detach().contiguous().float() for b in bs]
    acts = [X0]
    n = len(Ws)
    planes = TRAIN_GEMM == "planes"
    xp = split_planes(X0, P, Ws[0].shape[1], 64.0, ldp=_pad8(X0.shape[1])) if planes else None
    xplanes = []
    for l in range(n):
        o, i = Ws[l].shape
        last = l == n - 1
        Y = torch.empty((P, o if not last else ((o + 3) // 4) * 4), dtype=torch.float32, device=dev)
        if planes:
            yp = None if last else (torch.empty((P, _pad8(o)), dtype=torch.float16, device=dev),
                                    torch.empty((P, _pad8(o)), dtype=torch.float16, device=dev))
            mlp_layer_planes(xp, split_planes(Ws[l], o, i, 1024.0), P, o, i, 4 if last else 6, Y, bias=bs[l], y_planes=yp)
            xplanes += [xp[0], xp[1]]
            xp = yp
        else:
            mlp_fwd_layer(acts[l], Ws[l], bs[l], o, i, ACT_NONE if last else ACT_RELU, Y)
        acts.append(Y)
    return acts[-1][:, :Ws[-1].shape[0]], acts[:-1], xplanes


def _plain_mlp_backward(g_out, Ws, acts, need_w, need_x0, xplanes=()):
    """g_out [P, out_last] -> (dX0 [P, in_0 padded] or None, dW list, db list) for the ReLU MLP.  xplanes: the layer inputs'
    operand planes from the forward (flat hi, lo list) -- with them the weight gradient runs on the planes as well."""
    P, dev = g_out.shape[0], g_out.device
    n = len(Ws)
    o_last = Ws[-1].shape[0]
    G = [None] * n
    G[n - 1] = torch.zeros((P, _pad8(o_last)), dtype=torch.float32, device=dev)
    G[n - 1][:, :o_last] = g_out
    dyn = grad_dyn_scale(G[n - 1])
    planes = TRAIN_GEMM == "planes"
    gp = split_planes(G[n - 1], P, o_last, 64.0, scale_dev=dyn, ldp=_pad8(o_last)) if planes else None
    GP = [None] * n
    GP[n - 1] = gp
    for l in range(n - 1, 0, -1):
        o, i = Ws[l].shape
        G[l - 1] = torch.empty((P, i), dtype=torch.float32, device=dev)
        if planes:
            gprev = (torch.empty((P, _pad8(i)), dtype=torch.float16, device=dev), torch.empty((P, _pad8(i)), dtype=torch.float16, device=dev))
            mlp_layer_planes(gp, split_planes(Ws[l].detach(), o, i, 1024.0, transpose=True), P, i, o, 2, G[l - 1],
                             saved_input=acts[l], dyn=dyn, a_has_dyn=True, y_planes=gprev, planes_with_dyn=True)
            gp = gprev
            GP[l - 1] = gp
        else:
            mlp_bwd_data_layer(G[l], Ws[l], o, i, acts[l], ACT_RELU, G[l - 1], dyn_scale=dyn)
    dX0 = None
    if need_x0:
        o, i = Ws[0].shape
        dX0 = torch.empty((P, ((i + 3) // 4) * 4), dtype=torch.float32, device=dev)
        if planes:
            mlp_layer_planes(gp, split_planes(Ws[0].detach(), o, i, 1024.0, transpose=True), P, i, o, 0, dX0, dyn=dyn,
                             a_has_dyn=True)
        else:
            mlp_bwd_data_layer(G[0], Ws[0], o, i, None, ACT_NONE, dX0, dyn_scale=dyn)
    dW, db = [None] * n, [None] * n
    if need_w and planes and len(xplanes) == 2 * n:
        for l in range(n):
            o, i = Ws[l].shape
            dW[l], db[l] = mlp_wgrad_planes(GP[l], (xplanes[2 * l], xplanes[2 * l + 1]), P, o, i, 1.0, dyn, want_bias=True)
    elif need_w:
        dW, db = mlp_bwd_weight(G, list(acts), [w.shape[0] for w in Ws], [w.shape[1] for w in Ws], None, dyn)
    return dX0, dW, db


def _plain_composite(X0, Ws, bs):
    h = X0
    for l in range(len(Ws)):
        h = torch.nn.functional.linear(h, Ws[l], bs[l])
        if l < len(Ws) - 1:
            h = torch.relu(h)
    return h


class TranslatorTrainFunction(torch.autograd.Function):
    """MLPTranslator offset MLP with gradients (model/Deformer.py:171-206): input row [PE6(p) 39 | cond[frame] 128] ->
    512 x4 ReLU -> 3, forward / backward-data / weight gradient on tcgen05 (csrc/gemm3.cu); returns the OFFSET (the caller
    adds p).  create_graph=True falls back to a torch graph inside backward, like SdfMlpTrainFunction."""
    last_backward = None

    @staticmethod
    def forward(ctx, ps, conds, batch_inds, pe_w, *Wb):
        n = len(Wb) // 2
        Ws, bs = Wb[:n], Wb[n:]
        P, dev = ps.shape[0], ps.device
        X0 = torch.zeros((P, 168), dtype=torch.float32, device=dev)
        pe_forward(ps, pe_w, 6, X0)
        X0[:, 39:167] = conds.detach()[batch_inds]
        out, acts, xplanes = _plain_mlp_forward(X0, Ws, bs)
        ctx.pe_w, ctx.n = [float(w) for w in pe_w], n
        ctx.save_for_backward(ps, conds, batch_inds, *Wb, *acts, *xplanes)
        return out.contiguous()

    @staticmethod
    def backward(ctx, g_off):
        n = ctx.n
        saved = ctx.saved_tensors
        ps, conds, batch_inds = saved[:3]
        Ws, bs, acts, xplanes = saved[3:3 + n], saved[3 + n:3 + 2 * n], saved[3 + 2 * n:3 + 3 * n], saved[3 + 3 * n:]
        need = ctx.needs_input_grad
        if torch.is_grad_enabled() and _inputs_only(any(need[4:])):
            # utils.compute_Jacobian(..., create_graph=True) of the deformation regulariser: see second_order.py
            from . import second_order
            TranslatorTrainFunction.last_backward = "fused-tcgen05 (create_graph, input gradient)"
            dX0 = second_order.PlainMlpInputGradFunction.apply(g_off.contiguous().float(), n, *acts, *Ws)
            dps = second_order.pe_vjp_torch(ps, dX0, ctx.pe_w, 6) if need[0] else None
            dconds = torch.zeros_like(conds).index_add(0, batch_inds, dX0[:, 39:167]) if need[1] else None
            return (dps, dconds, None, None, *([None] * (2 * n)))
        if torch.is_grad_enabled():
            TranslatorTrainFunction.last_backward = "autograd-composite (create_graph)"
            with torch.enable_grad():
                x0 = torch.cat([_pe_torch(ps, ctx.pe_w, 6), conds[batch_inds]], 1)
                out = _plain_composite(x0, Ws, bs)
                ins = [t for t in [ps, conds] + list(Ws) + list(bs) if t.requires_grad]
                gr = iter(torch.autograd.grad([out], ins, [g_off], create_graph=True, allow_unused=True))
            res = [next(gr) if t.requires_grad else None for t in [ps, conds] + list(Ws) + list(bs)]
            return (res[0], res[1], None, None, *res[2:])
        TranslatorTrainFunction.last_backward = "fused-tcgen05"
        dX0, dW, db = _plain_mlp_backward(g_off.contiguous().float(), Ws, acts, any(need[4:]), need[0] or need[1], xplanes)
        dps = dconds = None
        if need[0]:
            dps = pe_backward(ps, dX0, None, ctx.pe_w, 6)
        if need[1]:
            dconds = torch.zeros_like(conds).index_add_(0, batch_inds, dX0[:, 39:167])
        return (dps, dconds, None, None, *dW, *db)


class RenderNetTrainFunction(torch.autograd.Function):
    """RenderingNetwork_view_norm ('idr', model/RenderNet.py:59-96) with gradients: input row [p 3 | PE4(v) 27 | n 3 |
    feat 256] -> 512 x4 ReLU -> 3 (pre-tanh; the caller applies tanh), all GEMMs on tcgen05."""
    last_backward = None

    @staticmethod
    def forward(ctx, points, normals, view_dirs, feats, pe_w, *Wb):
        n = len(Wb) // 2
        Ws, bs = Wb[:n], Wb[n:]
        P, dev = points.shape[0], points.device
        X0 = torch.zeros((P, 292), dtype=torch.float32, device=dev)
        X0[:, 0:3] = points.detach()
        pe_forward(view_dirs.detach().contiguous(), pe_w, 4, X0[:, 3:])
        X0[:, 30:33] = normals.detach()
        X0[:, 33:289] = feats.detach()
        out, acts, xplanes = _plain_mlp_forward(X0, Ws, bs)
        ctx.pe_w, ctx.n = [float(w) for w in pe_w], n
        ctx.save_for_backward(points, normals, view_dirs, feats, *Wb, *acts, *xplanes)
        return out.contiguous()

    @staticmethod
    def backward(ctx, g_out):
        n = ctx.n
        saved = ctx.saved_tensors
        points, normals, view_dirs, feats = saved[:4]
        Ws, bs, acts, xplanes = saved[4:4 + n], saved[4 + n:4 + 2 * n], saved[4 + 2 * n:4 + 3 * n], saved[4 + 3 * n:]
        need = ctx.needs_input_grad
        if torch.is_grad_enabled() and _inputs_only(any(need[5:])):
            from . import second_order
            RenderNetTrainFunction.last_backward = "fused-tcgen05 (create_graph, input gradient)"
            dX0 = second_order.PlainMlpInputGradFunction.apply(g_out.contiguous().float(), n, *acts, *Ws)
            dp = dX0[:, 0:3] if need[0] else None
            dn = dX0[:, 30:33] if need[1] else None
            dv = second_order.pe_vjp_torch(view_dirs, dX0[:, 3:30], ctx.pe_w, 4) if need[2] else None
            df = dX0[:, 33:289] if need[3] else None
            return (dp, dn, dv, df, None, *([None] * (2 * n)))
        if torch.is_grad_enabled():
            RenderNetTrainFunction.last_backward = "autograd-composite (create_graph)"
            with torch.enable_grad():
                x0 = torch.cat([points, _pe_torch(view_dirs, ctx.pe_w, 4), normals, feats], 1)
                out = _plain_composite(x0, Ws, bs)
                allin = [points, normals, view_dirs, feats] + list(Ws) + list(bs)
                ins = [t for t in allin if t.requires_grad]
                gr = iter(torch.autograd.grad([out], ins, [g_out], create_graph=True, allow_unused=True))
            res = [next(gr) if t.requires_grad else None for t in allin]
            return (*res[:4], None, *res[4:])
        RenderNetTrainFunction.last_backward = "fused-tcgen05"
        dX0, dW, db = _plain_mlp_backward(g_out.contiguous().float(), Ws, acts, any(need[5:]), any(need[:4]), xplanes)
        dp = dn = dv = df = None
        if need[0]:
            dp = dX0[:, 0:3].contiguous()
        if need[1]:
            dn = dX0[:, 30:33].contiguous()
        if need[2]:
            dv = pe_backward(view_dirs.detach().contiguous(), dX0[:, 3:], None, ctx.pe_w, 4)
        if need[3]:
            df = dX0[:, 33:289].contiguous()
        return (dp, dn, dv, df, None, *dW, *db)


TRANSLATOR_LAYER_SHAPES = [(512, 167), (512, 512), (512, 512), (512, 512), (3, 512)]


def _aligned_blob(nbytes, dev):
    raw = torch.empty((nbytes + 1024,), dtype=torch.uint8, device=dev)
    off = (-raw.data_ptr()) % 1024
    blob = raw[off:off + nbytes]
    blob._keepalive = raw
    return blob


def translator_pack_weights(Ws, bs):
    """MLPTranslator weights (lin0..lin4, no weight-norm) -> packed fp16 hi/lo panels for the tcgen05 engine."""
    dev = Ws[0].device
    for (o, i), W, b in zip(TRANSLATOR_LAYER_SHAPES, Ws, bs):
        if tuple(W.shape) != (o, i) or tuple(b.shape) != (o,):
            raise RuntimeError(f"unexpected translator layer shape {tuple(W.shape)} (want {(o, i)})")
    W_all = torch.cat([W.detach().reshape(-1).float() for W in Ws]).contiguous()
    b_all = torch.cat([b.detach().reshape(-1).float() for b in bs]).contiguous()
    lib = _lib.load()
    packed = _aligned_blob(lib.recmv_translator_packed_bytes(), dev)
    with torch.cuda.device(dev):
        check(lib.recmv_translator_pack_weights(_ptr(W_all), _ptr(b_all), _ptr(packed), _stream(W_all)),
              "recmv_translator_pack_weights")
    return packed


def deformer_forward(ps, conds, packed, pe_w, batch_inds=None, points_per_frame=0, skin=None, mode=None,
                     want_offset=True, want_translated=True, want_jacobian=False):
    """MLPTranslator (+ LBS forward when skin = (A, trans, ws_cl, center, extend)) in one fused launch.
    Returns (translated [P,3] or None, offset [P,3] or None, posed [P,3] or None) -- plus the Jacobian [P,3,3]
    of the last stage w.r.t. ps (forward-mode launch) when want_jacobian."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    ps = ps.contiguous().float()
    _check_input(ps, "ps")
    conds = conds.contiguous().float()
    P = ps.shape[0]
    dev = ps.device
    tr = torch.empty((P, 3), dtype=torch.float32, device=dev) if want_translated else None
    off = torch.empty((P, 3), dtype=torch.float32, device=dev) if want_offset else None
    posed, A, trans, vox = None, None, None, None
    if skin is not None:
        A, trans, ws_cl, center, extend = skin
        A, trans = A.contiguous().float(), trans.contiguous().float()
        vox = byref(make_voxel(ws_cl, center, extend))
        posed = torch.empty((P, 3), dtype=torch.float32, device=dev)
    if batch_inds is not None:
        batch_inds = batch_inds.contiguous().long()
    with torch.cuda.device(dev):
        if want_jacobian:
            jac = torch.empty((P, 3, 3), dtype=torch.float32, device=dev)
            check(_lib.load().recmv_deformer_fwd_jac(_ptr(ps), _ptr(conds), _ptr(batch_inds), int(points_per_frame),
                                                     int(conds.shape[0]), _ptr(packed), _pe_array(pe_w), _ptr(A),
                                                     _ptr(trans), vox, _ptr(tr), _ptr(off), _ptr(posed), _ptr(jac), P,
                                                     mode, _stream(ps)), "recmv_deformer_fwd_jac")
            return tr, off, posed, jac
        check(_lib.load().recmv_deformer_fwd(_ptr(ps), _ptr(conds), _ptr(batch_inds), int(points_per_frame),
                                             int(conds.shape[0]), _ptr(packed), _pe_array(pe_w), _ptr(A), _ptr(trans),
                                             vox, _ptr(tr), _ptr(off), _ptr(posed), P, mode, _stream(ps)),
              "recmv_deformer_fwd")
    return tr, off, posed


RENDERNET_LAYER_SHAPES = [(512, 289), (512, 512), (512, 512), (512, 512), (3, 512)]


def rendernet_pack_weights(Ws, bs):
    """Effective colour-network weights (weight norm already applied) -> packed fp16 hi/lo panels."""
    dev = Ws[0].device
    for (o, i), W, b in zip(RENDERNET_LAYER_SHAPES, Ws, bs):
        if tuple(W.shape) != (o, i) or tuple(b.shape) != (o,):
            raise RuntimeError(f"unexpected colour-network layer shape {tuple(W.shape)} (want {(o, i)})")
    W_all = torch.cat([W.detach().reshape(-1).float() for W in Ws]).contiguous()
    b_all = torch.cat([b.detach().reshape(-1).float() for b in bs]).contiguous()
    lib = _lib.load()
    packed = _aligned_blob(lib.recmv_rendernet_packed_bytes(), dev)
    with torch.cuda.device(dev):
        check(lib.recmv_rendernet_pack_weights(_ptr(W_all), _ptr(b_all), _ptr(packed), _stream(W_all)),
              "recmv_rendernet_pack_weights")
    return packed


def rendernet_forward(points, normals, view_dirs, feats, packed, pe_w8, mode=None):
    """Fused colour MLP: [P,3] x3 + [P,256] -> rgb [P,3] (tanh)."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    args = [t.contiguous().float() for t in (points, normals, view_dirs, feats)]
    for t, n in zip(args, ("points", "normals", "view_dirs", "feature_vectors")):
        _check_input(t, n)
    P = args[0].shape[0]
    if args[3].shape != (P, 256) or any(a.shape != (P, 3) for a in args[:3]):
        raise RuntimeError("rendernet_forward: expected [P,3] x3 and [P,256]")
    out = torch.empty((P, 3), dtype=torch.float32, device=args[0].device)
    pe = (c_float * 8)(*[float(w) for w in pe_w8])
    with torch.cuda.device(out.device):
        check(_lib.load().recmv_rendernet_fwd(*[_ptr(a) for a in args], _ptr(packed), pe, _ptr(out), P, mode,
                                              _stream(out)), "recmv_rendernet_fwd")
    return out


def make_raymarch(cam_pos, t_near, t_far, samples):
    rm = RayMarch()
    rm.cam_pos = (c_float * 3)(*[float(c) for c in cam_pos])
    rm.t_near, rm.t_far, rm.samples_per_ray = float(t_near), float(t_far), int(samples)
    return rm


def render_sdf(ray_dirs, cam_pos, t_near, t_far, samples, A, trans, ws_cl, center, extend, packed,
               pe_w=None, mode=None, frame_of_ray=None, rays_per_frame=0, want_xc=False, want_hit=True,
               out_sdf=None):
    """The fused render path: rays -> samples -> inverse LBS -> PE -> SDF MLP -> sdf [R,S] (+ first hit)."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    ray_dirs = ray_dirs.contiguous().float()
    _check_input(ray_dirs, "ray_dirs")
    A = A.contiguous().float()
    trans = trans.contiguous().float()
    R = ray_dirs.shape[0]
    dev = ray_dirs.device
    sdf = out_sdf if out_sdf is not None else torch.empty((R, samples), dtype=torch.float32, device=dev)
    xc = torch.empty((R, samples, 3), dtype=torch.float32, device=dev) if want_xc else None
    hit_idx = torch.empty((R,), dtype=torch.int32, device=dev) if want_hit else None
    hit_t = torch.empty((R,), dtype=torch.float32, device=dev) if want_hit else None
    if frame_of_ray is not None:
        frame_of_ray = frame_of_ray.contiguous().to(torch.int32)
    rm = make_raymarch(cam_pos, t_near, t_far, samples)
    vox = make_voxel(ws_cl, center, extend)
    with torch.cuda.device(dev):
        check(_lib.load().recmv_render_sdf(_ptr(ray_dirs), byref(rm), _ptr(A), _ptr(trans),
                                           _ptr(frame_of_ray), int(rays_per_frame), int(A.shape[0]),
                                           byref(vox), _ptr(packed), _pe_array(pe_w), _ptr(sdf), _ptr(xc),
                                           _ptr(hit_idx), _ptr(hit_t), R, mode, _stream(ray_dirs)),
              "recmv_render_sdf")
    return sdf, xc, hit_idx, hit_t


def interp2x_boundary3d_forward(inp, balance_value, order=0):
    """[N,C,D,H,W] f32 -> (output [N,C,2D-1,2H-1,2W-1] f32, is_boundary bool): the reference's optional
    `interp2x_boundary3d.forward` (order 0: its rounding; order 1: the rounding of F.interpolate(trilinear,
    align_corners=True), the default path of Seg3dLossless)."""
    _check_input(inp, "input")
    if inp.dtype != torch.float32 or inp.dim() != 5:
        raise RuntimeError("interp2x_boundary3d: expected a float32 [N,C,D,H,W] tensor")
    N, C, D, H, W = inp.shape
    out = torch.empty((N, C, 2 * D - 1, 2 * H - 1, 2 * W - 1), dtype=torch.float32, device=inp.device)
    flag = torch.empty(out.shape, dtype=torch.uint8, device=inp.device)
    with torch.cuda.device(inp.device):
        check(_lib.load().recmv_interp2x_boundary3d_fwd(_ptr(inp), _ptr(out), _ptr(flag), N * C, D, H, W,
                                                        float(balance_value), int(order), _stream(inp)),
              "recmv_interp2x_boundary3d_fwd")
    return [out, flag.view(torch.bool)]


def interp2x_boundary3d_backward(grad_output):
    """grad_output [N,C,2D-1,2H-1,2W-1] f32 -> grad_input [N,C,D,H,W] (`interp2x_boundary3d.backward`)."""
    _check_input(grad_output, "grad_output")
    if grad_output.dtype != torch.float32 or grad_output.dim() != 5:
        raise RuntimeError("interp2x_boundary3d: expected a float32 [N,C,d,h,w] tensor")
    N, C, d, h, w = grad_output.shape
    D, H, W = (d + 1) // 2, (h + 1) // 2, (w + 1) // 2
    gi = torch.empty((N, C, D, H, W), dtype=torch.float32, device=grad_output.device)
    with torch.cuda.device(gi.device):
        check(_lib.load().recmv_interp2x_boundary3d_bwd(_ptr(grad_output), _ptr(gi), N * C, D, H, W, _stream(gi)),
              "recmv_interp2x_boundary3d_bwd")
    return gi


def c2f_todo_mask(is_boundary, done):
    """(3x3x3 dilation of is_boundary [D,H,W] bool) & ~done [D,H,W] bool -> bool [D,H,W]."""
    _check_input(is_boundary, "is_boundary")
    _check_input(done, "done")
    D, H, W = is_boundary.shape
    todo = torch.empty((D, H, W), dtype=torch.uint8, device=done.device)
    with torch.cuda.device(done.device):
        check(_lib.load().recmv_c2f_todo_mask(_ptr(is_boundary.view(torch.uint8)), _ptr(done.view(torch.uint8)),
                                              _ptr(todo), D, H, W, _stream(todo)), "recmv_c2f_todo_mask")
    return todo.view(torch.bool)


def fragment_decode(pix_to_face, bary, verts, faces, mask=None, camera=None):
    """Fragments -> (batch, row, col, seed points, face ids[, rays]) of the covered pixels in (n, row, col) order
    (recmv_fragment_decode).  camera = (fx, fy, px, py, R [3,3]) as host numbers / CPU tensor, or None.
    One host synchronisation: the read of the row count (the reference's `nonzero` has the same one)."""
    pix_to_face = pix_to_face.contiguous().long()
    bary = bary.contiguous().float()
    _check_input(pix_to_face, "pix_to_face")
    N, H, W, K = pix_to_face.shape
    dev = pix_to_face.device
    verts = verts.detach().contiguous().float()
    faces = faces.contiguous().long()
    npix = N * H * W
    lib = _lib.load()
    scratch = torch.empty((lib.recmv_fragment_decode_scratch_bytes(npix),), dtype=torch.uint8, device=dev)
    ob, orow, ocol, ofi = (torch.empty((npix,), dtype=torch.int64, device=dev) for _ in range(4))
    opts = torch.empty((npix, 3), dtype=torch.float32, device=dev)
    orays = torch.empty((npix, 3), dtype=torch.float32, device=dev) if camera is not None else None
    cam = None
    if camera is not None:
        fx, fy, px, py, R = camera
        cam = (c_float * 13)(float(fx), float(fy), float(px), float(py), *[float(v) for v in torch.as_tensor(R).reshape(-1).tolist()])
    counters = torch.zeros((1,), dtype=torch.int32, device=dev)
    if mask is not None:
        mask = mask.contiguous().float()
    with torch.cuda.device(dev):
        check(lib.recmv_fragment_decode(_ptr(pix_to_face), _ptr(bary), N, H, W, K, _ptr(verts), _ptr(faces), int(faces.shape[0]),
                                        _ptr(mask), cam, _ptr(scratch), _ptr(ob), _ptr(orow), _ptr(ocol), _ptr(opts), _ptr(ofi),
                                        _ptr(orays), _ptr(counters), _stream(bary)), "recmv_fragment_decode")
    n = int(counters.item())
    out = (ob[:n], orow[:n], ocol[:n], opts[:n], ofi[:n])
    return out + (orays[:n],) if camera is not None else out


Fragments = collections.namedtuple("Fragments", ["pix_to_face", "zbuf", "bary_coords", "dists"])


def rasterize(verts, faces, camera, image_size):
    """Mesh rasteriser (recmv_rasterize): one face per pixel, the convention of pytorch3d's MeshRasterizer with
    faces_per_pixel=1, blur_radius=0, perspective_correct=True and no culling, in the reference camera's pixel grid
    (CameraMine.project / view_rays: pixel (row, col) is the screen point (col, row)).
    verts [N,V,3] (or [V,3]: one mesh) float32, faces [F,3] int64 shared by the N meshes, both CUDA and contiguous;
    camera = (fx, fy, px, py, R [NR,3,3] or [3,3], T [NR,3] or [3]) with NR = 1 or N; image_size = (H, W) or an int.
    Returns Fragments(pix_to_face [N,H,W,1] int64 packed n*F + f, zbuf [N,H,W,1] camera-space Zc, bary_coords
    [N,H,W,1,3] perspective-correct, dists=None), -1 everywhere on background."""
    _check_input(verts, "verts")
    _check_input(faces, "faces")
    if verts.dtype != torch.float32 or faces.dtype != torch.int64:
        raise RuntimeError("rasterize: verts must be float32 and faces int64")
    if verts.dim() == 2:
        verts = verts.unsqueeze(0)
    if verts.dim() != 3 or verts.shape[2] != 3 or faces.dim() != 2 or faces.shape[1] != 3:
        raise RuntimeError("rasterize: expected verts [N,V,3] or [V,3] and faces [F,3]")
    H, W = (image_size, image_size) if isinstance(image_size, int) else (int(image_size[0]), int(image_size[1]))
    N, V = verts.shape[0], verts.shape[1]
    fx, fy, px, py, R, T = camera
    dev = verts.device
    R = torch.as_tensor(R, dtype=torch.float32, device=dev).reshape(-1, 3, 3).contiguous()
    T = torch.as_tensor(T, dtype=torch.float32, device=dev).reshape(-1, 3).contiguous()
    if R.shape[0] != T.shape[0]:
        raise RuntimeError("rasterize: R and T must hold the same number of cameras")
    lib = _lib.load()
    nbytes = c_size_t(0)
    check(lib.recmv_raster_scratch_bytes(N, H, W, byref(nbytes)), "recmv_raster_scratch_bytes")
    scratch = torch.empty((nbytes.value,), dtype=torch.uint8, device=dev)
    p2f = torch.empty((N, H, W, 1), dtype=torch.int64, device=dev)
    zbuf = torch.empty((N, H, W, 1), dtype=torch.float32, device=dev)
    bary = torch.empty((N, H, W, 1, 3), dtype=torch.float32, device=dev)
    cam = (c_float * 4)(float(fx), float(fy), float(px), float(py))
    with torch.cuda.device(dev):
        check(lib.recmv_rasterize(_ptr(verts), _ptr(faces), N, V, int(faces.shape[0]), cam, _ptr(R), _ptr(T),
                                  int(R.shape[0]), H, W, _ptr(scratch), _ptr(p2f), _ptr(zbuf), _ptr(bary), _stream(verts)),
              "recmv_rasterize")
    return Fragments(p2f, zbuf, bary, None)


def _camera_tensors(camera, dev):
    fx, fy, px, py, R, T = camera
    R = torch.as_tensor(R, dtype=torch.float32, device=dev).detach().reshape(-1, 3, 3).contiguous()
    T = torch.as_tensor(T, dtype=torch.float32, device=dev).detach().reshape(-1, 3).contiguous()
    if R.shape[0] != T.shape[0]:
        raise RuntimeError("R and T must hold the same number of cameras")
    return (c_float * 4)(float(fx), float(fy), float(px), float(py)), R, T


class PointFragments:
    """The selection of one `rasterize_points` call.  The dense pytorch3d layout -- idx [N,H,W,K] int64 (packed n*P + p),
    zbuf [N,H,W,K] (camera-space Zc) and dists [N,H,W,K] (squared NDC distance), -1 in empty slots, nearest first -- is
    expanded on the device on first access (recmv_points_fragments): at 4 x 1080^2 with K = 50 it takes 3.7 GB.
    `candidates` is the number of (point, pixel) coverings before the per-pixel selection."""

    def __init__(self, meta, scratch, cand, candidates):
        self._meta, self._scratch, self._cand = meta, scratch, cand
        self.candidates = candidates
        self._dense = None

    def _expand(self):
        if self._dense is None:
            N, P, H, W, radius, K = self._meta
            dev = self._scratch.device
            idx = torch.empty((N, H, W, K), dtype=torch.int64, device=dev)
            zbuf = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
            dists = torch.empty((N, H, W, K), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                check(_lib.load().recmv_points_fragments(N, P, H, W, radius, K, _ptr(self._scratch), _ptr(self._cand),
                                                         _ptr(idx), _ptr(zbuf), _ptr(dists), _stream(idx)),
                      "recmv_points_fragments")
            self._dense = (idx, zbuf, dists)
        return self._dense

    @property
    def idx(self):
        return self._expand()[0]

    @property
    def zbuf(self):
        return self._expand()[1]

    @property
    def dists(self):
        return self._expand()[2]


class _RasterizePointsFunction(torch.autograd.Function):
    """images = composite(points); differentiable in `points` only (features and camera are constants)."""

    @staticmethod
    def forward(ctx, points, features, cam, R, T, size, radius, K, out):
        N, P = points.shape[0], points.shape[1]
        H, W = size
        C = features.shape[1]
        dev = points.device
        lib = _lib.load()
        nbytes = c_size_t(0)
        check(lib.recmv_points_scratch_bytes(N, P, H, W, byref(nbytes)), "recmv_points_scratch_bytes")
        scratch = torch.empty((nbytes.value,), dtype=torch.uint8, device=dev)
        total = c_int64(0)
        images = torch.empty((N, H, W, C), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            st = _stream(points)
            check(lib.recmv_points_count(_ptr(points), N, P, cam, _ptr(R), _ptr(T), int(R.shape[0]), H, W, radius,
                                         _ptr(scratch), byref(total), st), "recmv_points_count")
            cand = torch.empty((max(total.value, 1),), dtype=torch.int64, device=dev)
            check(lib.recmv_points_render(_ptr(features), C, N, P, H, W, radius, K, _ptr(scratch), _ptr(cand),
                                          total.value, _ptr(images), st), "recmv_points_render")
        ctx.save_for_backward(points, features, R, T, scratch, cand)
        ctx.meta = (cam, size, radius, K)
        out.append(PointFragments((N, P, H, W, radius, K), scratch, cand, total.value))
        return images

    @staticmethod
    def backward(ctx, grad_images):
        if not ctx.needs_input_grad[0]:
            return (None,) * 9
        points, features, R, T, scratch, cand = ctx.saved_tensors
        cam, (H, W), radius, K = ctx.meta
        N, P = points.shape[0], points.shape[1]
        grad_images = grad_images.contiguous().float()
        grad_points = torch.empty_like(points)
        with torch.cuda.device(points.device):
            check(_lib.load().recmv_points_render_backward(
                _ptr(points), N, P, cam, _ptr(R), _ptr(T), int(R.shape[0]), H, W, radius, _ptr(features),
                int(features.shape[1]), K, _ptr(scratch), _ptr(cand), _ptr(grad_images), _ptr(grad_points),
                _stream(points)), "recmv_points_render_backward")
        return (grad_points,) + (None,) * 8


def rasterize_points(points, features, camera, image_size, radius, points_per_pixel=50):
    """Points rasteriser + alpha compositor (recmv_points_*): pytorch3d's PointsRasterizer + AlphaCompositor
    (background_color=None) as `pcRender` uses them, in the reference camera's pixel grid (pixel (row, col) is the screen
    point (col, row), as ops.rasterize).  points [N,P,3] (or [P,3]: one cloud) float32 and features [P,C] float32
    (1 <= C <= 4, the same for every cloud), both CUDA and contiguous; camera = (fx, fy, px, py, R [NR,3,3] or [3,3],
    T [NR,3] or [3]) with NR = 1 or N, a constant; radius in NDC units (a disc of radius * min(H, W) / 2 pixels);
    1 <= points_per_pixel <= 64.  Differentiable in `points` only: features that require grad are refused.
    Returns (images [N,H,W,C], PointFragments).  One host synchronisation (the candidate count)."""
    if features.requires_grad:
        raise RuntimeError("rasterize_points: no gradient with respect to features; pass features.detach()")
    _check_input(points, "points")
    _check_input(features, "features")
    if points.dtype != torch.float32 or features.dtype != torch.float32:
        raise RuntimeError("rasterize_points: points and features must be float32")
    if points.dim() == 2:
        points = points.unsqueeze(0)
    if points.dim() != 3 or points.shape[2] != 3 or features.dim() != 2 or features.shape[0] != points.shape[1]:
        raise RuntimeError("rasterize_points: expected points [N,P,3] or [P,3] and features [P,C]")
    size = (image_size, image_size) if isinstance(image_size, int) else (int(image_size[0]), int(image_size[1]))
    cam, R, T = _camera_tensors(camera, points.device)
    out = []
    images = _RasterizePointsFunction.apply(points, features, cam, R, T, size, float(radius), int(points_per_pixel), out)
    return images, out[0]


class C2fLevel:
    """Device worklist of one pyramid level (recmv_c2f_refine / recmv_sdf_mlp_fwd_counted / recmv_c2f_scatter_list /
    recmv_c2f_mark_conflicts): one fused full-grid pass builds the level and its worklist, conflict rounds are driven by
    lists; no host round trip inside the level."""

    def __init__(self, coarse_dhw, final_whd, b_min, b_max, device, capacity):
        D, H, W = coarse_dhw
        self.coarse = (int(D), int(H), int(W))
        self.D, self.H, self.W = 2 * D - 1, 2 * H - 1, 2 * W - 1
        self.level = (ctypes.c_int * 3)(self.W, self.H, self.D)
        self.final = (ctypes.c_int * 3)(*[int(v) for v in final_whd])
        self.bmin = (c_float * 3)(*[float(v) for v in b_min])
        self.bmax = (c_float * 3)(*[float(v) for v in b_max])
        self.cap = int(capacity)
        self.dev = device
        self.idx = torch.empty((self.cap,), dtype=torch.int32, device=device)
        self.pts = torch.empty((self.cap, 3), dtype=torch.float32, device=device)
        self.vals = torch.empty((self.cap, 1), dtype=torch.float32, device=device)
        self.clist = [torch.empty((self.cap,), dtype=torch.int32, device=device) for _ in range(2)]
        # [0:2] worklist {count, overflow}; [2], [3] conflict counts of the two lists; [4] queried total
        self.ctr = torch.zeros((8,), dtype=torch.int32, device=device)
        self.claim = torch.zeros((self.D, self.H, self.W), dtype=torch.uint8, device=device)
        self.mixed = torch.empty((max(D - 1, 1) * max(H - 1, 1) * max(W - 1, 1),), dtype=torch.uint8, device=device)
        self.cur = 0     # which conflict list the last scatter filled

    def refine(self, occ_coarse, done_coarse, balance, order):
        occ_f = torch.empty((1, 1, self.D, self.H, self.W), dtype=torch.float32, device=self.dev)
        done_f = torch.empty((self.D, self.H, self.W), dtype=torch.uint8, device=self.dev)
        D, H, W = self.coarse
        with torch.cuda.device(self.dev):
            check(_lib.load().recmv_c2f_refine(_ptr(occ_coarse), _ptr(done_coarse), D, H, W, self.final, self.bmin, self.bmax,
                                               float(balance), int(order), _ptr(self.mixed), _ptr(occ_f), _ptr(done_f),
                                               _ptr(self.idx), _ptr(self.pts), _ptr(self.ctr), self.cap, _stream(occ_f)),
                  "recmv_c2f_refine")
        return occ_f, done_f

    def evaluate(self, packed, pe_w, mode, occ, done_u8, calculated_u8, balance):
        """SDF on the current worklist, scatter, conflicts -> the other conflict list."""
        lib = _lib.load()
        self.cur ^= 1
        cc = self.ctr[2 + self.cur:3 + self.cur]
        with torch.cuda.device(self.dev):
            st = _stream(occ)
            check(lib.recmv_sdf_mlp_fwd_counted(_ptr(self.pts), _ptr(packed), _pe_array(pe_w), _ptr(self.vals), None,
                                                self.cap, _ptr(self.ctr), mode, st), "recmv_sdf_mlp_fwd_counted")
            cc.zero_()
            check(lib.recmv_c2f_scatter_list(_ptr(self.idx), _ptr(self.vals), _ptr(self.ctr), self.cap, self.level,
                                             self.final, _ptr(occ), _ptr(done_u8), _ptr(calculated_u8), _ptr(self.claim),
                                             float(balance), _ptr(self.clist[self.cur]), _ptr(cc), _ptr(self.ctr[4:5]), st),
                  "recmv_c2f_scatter_list")

    def next_from_conflicts(self, calculated_u8):
        """Worklist of the next round from the conflict list the last evaluate() filled."""
        cc = self.ctr[2 + self.cur:3 + self.cur]
        with torch.cuda.device(self.dev):
            self.ctr[0:1].zero_()
            check(_lib.load().recmv_c2f_mark_conflicts(_ptr(self.clist[self.cur]), _ptr(cc), self.cap, _ptr(calculated_u8),
                                                       self.level, self.final, self.bmin, self.bmax, _ptr(self.claim),
                                                       _ptr(self.idx), _ptr(self.pts), _ptr(self.ctr), self.cap,
                                                       _stream(calculated_u8)), "recmv_c2f_mark_conflicts")

    def read(self):
        """(queried so far, conflicts of the last round, overflow) -- the level's host synchronisation."""
        h = self.ctr.tolist()
        return h[4], h[2 + self.cur], h[1]


def c2f_done_up(done_u8):
    D, H, W = done_u8.shape
    up = torch.empty((2 * D - 1, 2 * H - 1, 2 * W - 1), dtype=torch.uint8, device=done_u8.device)
    with torch.cuda.device(up.device):
        check(_lib.load().recmv_c2f_done_up(_ptr(done_u8), D, H, W, _ptr(up), _stream(up)), "recmv_c2f_done_up")
    return up


def surface_solve(cam_pos, rays, seeds, batch_inds, sdf_packed, sdf_pe_w, tr_packed, tr_pe_w, conds, skin, dthreshold,
                  athreshold, w1, w2, times, mode=None):
    """Device-resident surface solve (recmv_surface_solve).  skin = (A, trans, ws_cl, center, extend).
    Returns (points [P,3], ok [P] bool); `seeds` is not modified."""
    mode = DEFAULT_MLP_MODE if mode is None else mode
    ps = seeds.detach().contiguous().float().clone()
    rays = rays.contiguous().float()
    _check_input(ps, "seeds")
    _check_input(rays, "rays")
    P = ps.shape[0]
    dev = ps.device
    A, trans, ws_cl, center, extend = skin
    A, trans, conds = A.contiguous().float(), trans.contiguous().float(), conds.contiguous().float()
    bi = batch_inds.contiguous().long() if batch_inds is not None else None
    lib = _lib.load()
    wsz = lib.recmv_surface_solve_workspace(P)
    work = torch.empty((max(wsz, 1),), dtype=torch.uint8, device=dev)
    ok = torch.empty((P,), dtype=torch.uint8, device=dev)
    cam = (c_float * 3)(*[float(v) for v in cam_pos.view(-1).tolist()])
    with torch.cuda.device(dev):
        check(lib.recmv_surface_solve(cam, _ptr(rays), _ptr(ps), _ptr(bi), _ptr(sdf_packed), _pe_array(sdf_pe_w),
                                      _ptr(tr_packed), _pe_array(tr_pe_w), _ptr(conds), int(conds.shape[0]), _ptr(A),
                                      _ptr(trans), byref(make_voxel(ws_cl, center, extend)), float(dthreshold),
                                      float(athreshold), float(w1), float(w2), int(times), mode, _ptr(work), wsz,
                                      _ptr(ok), P, _stream(ps)), "recmv_surface_solve")
    return ps, ok.view(torch.bool)


def surface_grad_coeffs(grad_l_p, grad_f_p, jac, rays, d_minus_c=None):
    """Per-ray algebra of propagateTmpPsGrad (OptimNetwork.py:788-851) in one launch.
    Returns (sdf_coef [n], def_vec [n,3], ray_grad [n,3] or None, ok [n] bool)."""
    args = [t.contiguous().float() for t in (grad_l_p, grad_f_p, jac, rays)]
    for t, name in zip(args, ("grad_l_p", "grad_f_p", "jac", "rays")):
        _check_input(t, name)
    n = args[0].shape[0]
    if args[2].shape != (n, 3, 3) or any(a.shape != (n, 3) for a in (args[0], args[1], args[3])):
        raise RuntimeError("surface_grad_coeffs: expected [n,3], [n,3], [n,3,3], [n,3]")
    dev = args[0].device
    dc = d_minus_c.contiguous().float() if d_minus_c is not None else None
    coef = torch.empty((n,), dtype=torch.float32, device=dev)
    vec = torch.empty((n, 3), dtype=torch.float32, device=dev)
    rg = torch.empty((n, 3), dtype=torch.float32, device=dev) if dc is not None else None
    ok = torch.empty((n,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(_lib.load().recmv_surface_grad_coeffs(*[_ptr(a) for a in args], _ptr(dc), _ptr(coef), _ptr(vec), _ptr(rg),
                                                    _ptr(ok), n, _stream(coef)), "recmv_surface_grad_coeffs")
    return coef, vec, rg, ok.view(torch.bool)


class Svd3x3Function(torch.autograd.Function):
    """(U, S, V) = svd(J), J [N,3,3] float32 CUDA, J = U diag(S) V^T with S descending -- torch.svd's contract, computed
    per matrix in registers (csrc/svd3.cu) instead of the reference's round trip through the host
    (`torch.svd(Jacobs.cpu())`, engineer/networks/OptimGarmentNetwork.py:1148).  Differentiable through S (dJ = U diag(dS)
    V^T, one launch); a cotangent on U or V raises (the reference's loss reads the singular values only)."""

    @staticmethod
    def forward(ctx, J):
        _check_input(J, "J")
        if J.dtype != torch.float32 or J.dim() != 3 or tuple(J.shape[1:]) != (3, 3):
            raise TypeError("svd3x3 expects a float32 [N,3,3] tensor")
        N = J.shape[0]
        U = torch.empty((N, 3, 3), dtype=torch.float32, device=J.device)
        V = torch.empty((N, 3, 3), dtype=torch.float32, device=J.device)
        S = torch.empty((N, 3), dtype=torch.float32, device=J.device)
        with torch.cuda.device(J.device):
            check(_lib.load().recmv_svd3x3(_ptr(J), N, _ptr(U), _ptr(S), _ptr(V), _stream(J)), "recmv_svd3x3")
        ctx.save_for_backward(U, V)
        ctx.set_materialize_grads(False)
        ctx.mark_non_differentiable(U, V)
        return U, S, V

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, gU, gS, gV):
        if gU is not None or gV is not None:
            raise NotImplementedError("svd3x3 is differentiable through the singular values only")
        if gS is None:
            return None
        U, V = ctx.saved_tensors
        gS = gS.contiguous().float()
        dJ = torch.empty_like(U)
        with torch.cuda.device(U.device):
            check(_lib.load().recmv_svd3x3_backward_s(_ptr(U), _ptr(V), _ptr(gS), U.shape[0], _ptr(dJ), _stream(U)),
                  "recmv_svd3x3_backward_s")
        return dJ


def svd3x3(J):
    """torch.svd for a batch of 3x3 matrices on the device: returns (U, S, V)."""
    return Svd3x3Function.apply(J.contiguous())


def check_async_errors(clear=False):
    """Raise if a tcgen05 launch on the current device aborted on a bounded wait (non-blocking check)."""
    info = (ctypes.c_int * 3)()
    st = _lib.load().recmv_check_async_errors(info, 1 if clear else 0)
    if st != 0:
        if info[0] == 2:
            raise _lib.RecmvError(f"tcgen05 operand range exceeded (|activation| >= 1023.5 or |weight| >= 63.97 does not "
                                  f"fit the scaled fp16 operands; results were saturated): site tag={info[1]} block={info[2]}")
        raise _lib.RecmvError(f"tcgen05 kernel aborted: code={info[0]} barrier tag={info[1]} block={info[2]}")


def launch_count():
    return int(_lib.load().recmv_launch_count())
