/* recmv_b200.h -- C ABI of the B200-native REC-MV hot path (librecmv_b200.so).
 *
 * Every entry point takes raw DEVICE pointers (unless a parameter says "host"), plain sizes and a
 * cudaStream_t passed as void*.  No torch types.  Return value: 0 = ok, negative = argument error
 * (RECMV_E_*), positive = cudaError_t raised by the launch.  Nothing here allocates result storage
 * of data-dependent size: marching cubes is a count call followed by an emit call.  All kernels run
 * on the caller's stream and never synchronise the device, except recmv_mc_count (it has to return
 * two integers to the host, like the reference's blocking cudaMemcpy at MCGpu/CudaKernels.cu:628) and
 * recmv_points_count (it returns the candidate total that sizes the caller's list).
 *
 * Each block cites the reference interface (path:line under /root/reference) it replaces.
 */
#ifndef RECMV_B200_H_
#define RECMV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* recmv_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define RECMV_API __attribute__((visibility("default")))
#else
#define RECMV_API
#endif

enum {
  RECMV_OK = 0,
  RECMV_E_NULL = -1,      /* required pointer is NULL            */
  RECMV_E_DTYPE = -2,     /* dtype / layout / mode flag unknown  */
  RECMV_E_SHAPE = -3,     /* non-positive or inconsistent extent */
  RECMV_E_RANGE = -4,     /* size exceeds an implementation limit (e.g. > 2^26 MC vertices) */
  RECMV_E_UNSUPPORTED = -5,
  RECMV_E_DEVICE = -6     /* a tcgen05 launch aborted on a bounded mbarrier wait (see recmv_check_async_errors) */
};

enum { RECMV_F32 = 0, RECMV_F64 = 1 };
enum { RECMV_LAYOUT_NCDHW = 0, RECMV_LAYOUT_NDHWC = 1 };

/* SDF-MLP arithmetic.  All modes accumulate in fp32.
 *   FP32_SIMT : fp32 FMA on CUDA cores (exact-fp32 verification mode, slow)
 *   TC_F16X3  : tcgen05 kind::f16, operands split a = hi + lo (fp16 each), 3 MMAs per product
 *               (hi*hi + lo*hi + hi*lo) -> ~2^-21 relative per product; meets the 1e-4 parity bar
 *   TC_F16X1  : tcgen05 kind::f16 single pass (11-bit operands, like the TF32 the reference ran
 *               with on Ampere); ~1e-3, NOT parity grade                                          */
enum { RECMV_MLP_FP32_SIMT = 0, RECMV_MLP_TC_F16X3 = 1, RECMV_MLP_TC_F16X1 = 2 };

RECMV_API int recmv_version(void);
RECMV_API const char* recmv_error_string(int status);
/* number of kernels this library has launched since load (bench.py's gpu_launches) */
RECMV_API int64_t recmv_launch_count(void);

/* ---- A6: FastMinv.Fast3x3Minv / Fast3x3Minv_backward --------------------------------------
 * replaces FastMinv/M3x3Inv.cpp:12-59 (pybind) + Matrix3x3InvKernels.cu:21-142.
 * ms/invs/grads/outs: [n,3,3] contiguous; ok: [n] bytes (1 = invertible, |det| >= 1e-4).        */
RECMV_API int recmv_minv3x3_fwd(const void* ms, void* invs, uint8_t* ok, int64_t n, int dtype,
                      recmv_stream_t stream);
RECMV_API int recmv_minv3x3_bwd(const void* grads, const void* invs, void* outs, int64_t n, int dtype,
                      recmv_stream_t stream);

/* ---- K4-K6: GridSamplerMine.forward / backward / dbackward --------------------------------
 * replaces MCAcc/cuda/GridSamplerMine.cpp:75-103 + GridSamplerMineKernel.cu:160-1022.
 * trilinear, border padding, align_corners=False.  input [N,C,D,H,W] (layout NCDHW) or
 * [N,D,H,W,C] (NDHWC, the coalesced internal layout); grid [N,P,3] (x->W, y->H, z->D);
 * output / grad_out / gg_out [N,C,P].
 * bwd : grad_input may be NULL (skipped -- the skinning voxel is a frozen buffer); otherwise it
 *       must be zero-filled by the caller and has the layout of `input`.
 * bwd2: cotangents gg_input (layout of input, may be NULL = zeros) and gg_grid [N,P,3];
 *       outputs g_input (may be NULL; else zero-filled), g_grid [N,P,3], gg_out [N,C,P].         */
RECMV_API int recmv_gridsample3d_fwd(const void* input, const void* grid, void* output, int N, int C, int D,
                           int H, int W, int64_t P, int dtype, int layout, recmv_stream_t stream);
RECMV_API int recmv_gridsample3d_bwd(const void* input, const void* grid, const void* grad_out,
                           void* grad_input, void* grad_grid, int N, int C, int D, int H, int W,
                           int64_t P, int dtype, int layout, recmv_stream_t stream);
RECMV_API int recmv_gridsample3d_bwd2(const void* gg_input, const void* gg_grid, const void* input,
                            const void* grid, const void* grad_out, void* g_input, void* g_grid,
                            void* gg_out, int N, int C, int D, int H, int W, int64_t P, int dtype,
                            int layout, recmv_stream_t stream);
/* [C,D,H,W] -> [D,H,W,C] copy (private cache of LBSkinner.ws) */
RECMV_API int recmv_voxel_to_channels_last(const float* src, float* dst, int C, int D, int H, int W,
                                 recmv_stream_t stream);

/* ---- A12: MCGpu.mc_gpu --------------------------------------------------------------------
 * replaces MCGpu/MCGpu.cpp:20-56 + CudaKernels.cu:316-521.  sdf [NX,NY,NZ] f32, z fastest.
 * Deterministic: vertices and faces come out in the order a sequential sweep of the reference
 * kernel (cell index ascending) would create them; faces int64 with the reference's reversed
 * winding; vertices referenced on the far boundary planes get index -1 exactly as the reference.
 * count: fills host V,F (blocks on the stream).  emit: must follow count on the same stream with
 * the same sdf/iso/scratch; writes verts [V,3] = v*step+origin and faces [F,3].                 */
RECMV_API int recmv_mc_scratch_bytes(int NX, int NY, int NZ, size_t* bytes /*host*/);
RECMV_API int recmv_mc_count(const float* sdf, int NX, int NY, int NZ, float iso, void* scratch,
                   int64_t* num_verts /*host*/, int64_t* num_faces /*host*/, recmv_stream_t stream);
RECMV_API int recmv_mc_emit(const float* sdf, int NX, int NY, int NZ, float iso, void* scratch,
                  const float step[3] /*host*/, const float origin[3] /*host*/, float* verts,
                  int64_t* faces, recmv_stream_t stream);
/* One call, NO host synchronisation (the reference blocks on a cudaMemcpy between its two kernels,
 * MCGpu/CudaKernels.cu:628): classify + count + scan + emit into caller-provided buffers of capacity cap_verts /
 * cap_faces rows.  counts (DEVICE, int32[4]) receives {V, F, overflow, 0}; overflow != 0 = a buffer was too small
 * (re-run with V / F rows).  Rows beyond V / F are left untouched.                                              */
RECMV_API int recmv_mc_run(const float* sdf, int NX, int NY, int NZ, float iso, void* scratch,
                 const float step[3] /*host*/, const float origin[3] /*host*/, float* verts, int64_t cap_verts,
                 int64_t* faces, int64_t cap_faces, int32_t* counts /*device*/, recmv_stream_t stream);

/* ---- A5 / A5': LBSkinner.forward and the inverse warp ----------------------------------------
 * replaces model/Deformer.py:359-445 (+342-355, GridSamplerMine3dFunction at :421).
 * ws_cl: skinning voxel channels-last [D,H,W,24] f32; A [F,24,4,4] row-major bone matrices
 * (G*init_pose, computed on the host side); trans [F,3] (already + extra_trans);
 * batch_inds [P] int64 or NULL (then frame = point / points_per_frame).
 * fwd: out = (sum_j w_j(tp) A_j) [p;1] + trans;  tps may be NULL (= ps).
 *      weights_out [P,24] optional (NULL to skip).
 * inverse: x_c = M^-1 (x_obs - trans - t), [M|t] = sum_j w_j(x_obs) A_j ; valid=0 and x_c=0 when
 *      |det M| < 1e-4 (FastMinv rule, Matrix3x3InvKernels.cu:40).                                */
typedef struct {
  const float* ws_cl;
  int D, H, W;
  float center[3];
  float extend; /* nps = 2 (p - center) / extend   (Deformer.py:342-355) */
} recmv_voxel_t;

RECMV_API int recmv_lbs_fwd(const float* ps, const float* tps, const float* A, const float* trans,
                  const int64_t* batch_inds, int64_t points_per_frame, int num_frames,
                  const recmv_voxel_t* vox /*host*/, float* out, float* weights_out, int64_t P,
                  recmv_stream_t stream);
RECMV_API int recmv_lbs_inverse(const float* x_obs, const float* A, const float* trans,
                      const int64_t* batch_inds, int64_t points_per_frame, int num_frames,
                      const recmv_voxel_t* vox /*host*/, float* x_can, uint8_t* valid, int64_t P,
                      recmv_stream_t stream);

/* Bone matrices of the SMPL kinematic chain: replaces the 24-joint python loop of model/Deformer.py:372-405 (and
 * posedSkeleton, :305-326) when no autograd graph is needed.  poses [F,24,3] axis-angle, Js [24,3], parents [24] int32
 * (device), init_pose [24,4,4] or NULL (Deformer.py:397-404).  G [F,24,4,4] = chained joint transforms (always
 * written; G[:,:,:3,3] is the posed skeleton), A [F,24,4,4] = G . init_pose (may be NULL).                       */
RECMV_API int recmv_bone_matrices(const float* poses, const float* Js, const int* parents, const float* init_pose,
                        float* G, float* A, int num_frames, recmv_stream_t stream);

/* ---- A1+A2: Embedder + ImplicitNetwork.forward -------------------------------------------------
 * replaces model/Embedder.py:43-50 + model/network.py:89-119 (+ utils/utils.py:40-46 weights).
 * Network shape is the reference's getTmpSdf: PE(6) 39 -> 512 x3 -> 473 (+39 skip)/sqrt2 -> 512 x4
 * -> 257, softplus(beta=100, threshold 20) on layers 0..7.
 * pack: W_l [out_l, in_l] row-major fp32 EFFECTIVE weights (weight-norm already applied by the host
 * shim), concatenated l = 0..8; b likewise.  `packed` (recmv_sdf_packed_bytes() bytes) holds the
 * fp32 copy used by FP32_SIMT and the padded fp16 hi/lo K-major planes the TMA descriptors read.  */
RECMV_API size_t recmv_sdf_packed_bytes(void);
RECMV_API int recmv_sdf_pack_weights(const float* W_all, const float* b_all, void* packed,
                           recmv_stream_t stream);
/* x [P,3] canonical points; pe_w [12] host (annealing weights); out_sdf [P]; out_feat [P,256] or
 * NULL.                                                                                           */
RECMV_API int recmv_sdf_mlp_fwd(const float* x, const void* packed, const float* pe_w /*host*/,
                      float* out_sdf, float* out_feat, int64_t P, int mode, recmv_stream_t stream);
/* the same with the point count read from DEVICE memory: *count_dev points (clamped to `capacity`, for which the launch
 * is sized) -- consumer of device-built worklists (recmv_c2f_compact).  TC modes only.                             */
RECMV_API int recmv_sdf_mlp_fwd_counted(const float* x, const void* packed, const float* pe_w /*host*/, float* out_sdf,
                              float* out_feat, int64_t capacity, const int* count_dev, int mode,
                              recmv_stream_t stream);

/* ---- A2/A3 training path: what `loss.backward()` (train.py:325) runs through model/network.py:89-119 ---------
 * (and through Deformer.py:171-206 / RenderNet.py:59-96 -- the entry points below are generic over the layer list).
 *
 * recmv_mlp_fwd_layer: Y = act(pre_scale * (X . W^T) + bias) for ONE layer on tcgen05 (3 fp16 MMAs per product, fp32
 *   accumulation) -- the TRAINING forward, whose layer outputs stay in HBM as the inputs the backward needs (what
 *   autograd would save): X [P][ldx] (in_dim columns used), W [out_dim][in_dim] row-major fp32 (nn.Linear layout),
 *   bias [out_dim] or NULL, act: 0 none, 1 softplus(beta 100, threshold 20), 2 ReLU.  Columns n < split -> Y[p*ldy+n],
 *   columns n >= split -> Y2[p*ldy2 + n - split] (split <= 0: all to Y; the SDF output layer splits sdf | features).
 * recmv_pe_forward: positional encoding rows (model/Embedder.py:43-50 with the annealing weights pe_w [2*bands] host)
 *   written as a saved layer input: out[p*ld + e], e < 3 + 6*bands; out2 (optional) gets the same row.
 *
 * recmv_mlp_bwd_data_layer: G_prev = (G . W) * act'(saved_input)  for ONE layer, on tcgen05 (3 fp16 MMAs per product):
 *   G [P][ldg] cotangent of the layer output (out_dim columns used), W [out_dim][in_dim] row-major fp32 (the
 *   nn.Linear layout -- no transposed copy), saved_input [P][lds] = the layer's input as saved by the forward
 *   (= the previous layer's activation output), act: 0 none, 1 softplus(beta 100) -> 1 - exp(-100 a), 2 ReLU -> a > 0.
 *   Columns n < split go to G_prev[p * ldgp + n] with the activation derivative; columns n >= split (the PE part
 *   of the SDF skip layer; split <= 0 = none) go to D2[p * ldd2 + n - split] untouched.  out_scale multiplies
 *   everything (1/sqrt2 for the SDF skip layer).  dyn_scale: optional DEVICE scalar, a power of two that brings
 *   max|G| near 1 before the fp16 split (gradients of mean-reduced losses are ~1/P); results are unscaled again.
 *
 * recmv_mlp_bwd_weight: for every layer l < num_layers in ONE launch:  dW[l] [out][in] = out_scale[l] * G[l]^T X[l]
 *   (reduction over the P samples, accumulated in chunks of 2048 samples; tile owner adds chunks in fp32 -- no atomics,
 *   deterministic) and db[l] [out] += column sums of G[l] (db must be zero-filled by the caller; may be NULL).
 *   G, ldg, X, ldx, out_dim, in_dim, dW, db, out_scale are HOST arrays of length num_layers (<= 10).
 *
 * recmv_pe_backward: dx [P,3] (+)= (d PE / d x)^T (g + g2): g [P][ldg] cotangent of the 3 + 6*bands encoding
 *   (model/Embedder.py:43-50 order), g2 optional second cotangent of the same encoding, pe_w [2*bands] host.       */
RECMV_API int recmv_mlp_fwd_layer(const float* X, int64_t ldx, const float* W, const float* bias, int out_dim, int in_dim,
                        int act, float pre_scale, int split, float* Y, int64_t ldy, float* Y2, int64_t ldy2, int64_t P,
                        recmv_stream_t stream);
RECMV_API int recmv_pe_forward(const float* x, const float* pe_w /*host*/, int bands, float* out, int64_t ld, float* out2,
                     int64_t ld2, int64_t P, recmv_stream_t stream);
RECMV_API int recmv_mlp_bwd_data_layer(const float* G, int64_t ldg, const float* W, int out_dim, int in_dim,
                             const float* saved_input, int64_t lds, int act, int split, float* G_prev, int64_t ldgp,
                             float* D2, int64_t ldd2, float out_scale, const float* dyn_scale /*device*/, int64_t P,
                             recmv_stream_t stream);
RECMV_API int recmv_mlp_bwd_weight(int num_layers, const float* const* G, const int64_t* ldg, const float* const* X,
                         const int64_t* ldx, const int* out_dim, const int* in_dim, float* const* dW, float* const* db,
                         const float* out_scale, const float* dyn_scale /*device*/, int64_t P, recmv_stream_t stream);
RECMV_API int recmv_pe_backward(const float* x, const float* g, int64_t ldg, const float* g2, int64_t ldg2,
                      const float* pe_w /*host*/, int bands, float* dx, int accumulate, int64_t P,
                      recmv_stream_t stream);

/* Second-generation layer GEMMs: operands as fp16 hi / lo PLANES in HBM, fed by TMA (csrc/gemm3_tma.cu) -- every tensor a
 * later GEMM consumes is written in consumable form by its producer, the main loop converts nothing.
 *  recmv_split_planes      : fp32 [R][C] (row stride ld) -> planes hi = fp16(s v), lo = fp16(s v - hi), s = scale * (*scale_dev
 *                            if given); transpose != 0 writes [C][R].  ldp = plane row stride in elements (multiple of 8, plane
 *                            base 16-byte aligned).  Weights: scale 1024 ([out][in] for the forward, transposed for
 *                            backward-data); the loss cotangent: scale 64 with scale_dev = the call's dyn scale.
 *  recmv_pe_forward_planes : recmv_pe_forward + the planes (scale 64) of the same rows.
 *  recmv_mlp_layer_planes  : one layer.  mode 4 / 5 / 6 = forward with none / softplus(100) / ReLU:
 *                              Y = act(scale * (A . B^T) + bias);
 *                            mode 0 / 1 / 2 = backward-data with none / softplus' / ReLU':
 *                              Y = scale * (A . B^T) * act'(saved_input); columns >= split -> Y2 without the derivative.
 *                            A planes [M][lda_p] hold 64 (x dyn if a_has_dyn) * value, B planes [N][ldb_p] 1024 * weight; K
 *                            columns of each are used.  Y fp32 [M][ldy] (+ Y2); y_hi / y_lo (optional) receive the planes
 *                            of Y's columns < split, scaled 64 (x dyn if planes_with_dyn) -- the next GEMM's A operand.      */
RECMV_API int recmv_split_planes(const float* in, int64_t ld, int64_t R, int C, float scale, const float* scale_dev /*device*/,
                       int transpose, void* hi, void* lo, int64_t ldp, recmv_stream_t stream);
RECMV_API int recmv_pe_forward_planes(const float* x, const float* pe_w /*host*/, int bands, float* out, int64_t ld,
                            void* out_hi, void* out_lo, int64_t ldp, int64_t P, recmv_stream_t stream);
RECMV_API int recmv_mlp_layer_planes(const void* a_hi, const void* a_lo, int64_t lda_p, const void* b_hi, const void* b_lo,
                           int64_t ldb_p, int64_t M, int N, int K, int mode, const float* bias, const float* saved_input,
                           int64_t lds, float scale, const float* dyn_scale /*device*/, int a_has_dyn, int split, float* Y,
                           int64_t ldy, float* Y2, int64_t ldy2, void* y_hi, void* y_lo, int64_t ldyp, int planes_with_dyn,
                           recmv_stream_t stream);

/* Weight gradient from the same planes, no transposed copies (tcgen05 reads the row-major planes as MN-major operands):
 *   dW [out_dim][in_dim] = scale * G^T X,  g planes [P][ldg_p] = 64 * dyn * g (columns < out_dim), x planes [P][ldx_p] = 64 * x.
 * The sample range is split over the SMs, partial tiles are summed in a fixed order (deterministic).  db [out_dim] (optional)
 * = sum_p g[p][:] = the bias gradient, from one more product of the G tiles with a tile of ones in the same launch.  workspace:
 * device fp32, recmv_mlp_wgrad_workspace_floats() elements, reusable across calls on one stream.
 *   recmv_colsum: out[c] = sum_r g[r][c] (the bias gradient from the fp32 cotangent); partial = scratch of 128 * cols floats. */
RECMV_API size_t recmv_mlp_wgrad_workspace_floats(void);
RECMV_API int recmv_mlp_wgrad_planes(const void* g_hi, const void* g_lo, int64_t ldg_p, const void* x_hi, const void* x_lo,
                                     int64_t ldx_p, int64_t P, int out_dim, int in_dim, float scale,
                                     const float* dyn_scale /*device*/, float* workspace, float* dW, float* db /*or NULL*/,
                                     recmv_stream_t stream);
RECMV_API int recmv_colsum(const float* g, int64_t ld, int64_t rows, int cols, float* partial, float* out,
                           recmv_stream_t stream);
/* (f4) element-wise steps of the second-order pass between two plane GEMMs (recmv_b200/second_order.py), each one launch that
 * also writes the next GEMM's A planes (scaled plane_scale [x *scale_dev]):
 *   softplus_tangent: u = s tz (fp32 + planes), inj = 100 (1 - s) h tz,  s = 1 - exp(-100 a)  (softplus_100' from the saved
 *                     output a; h = first-order cotangent at the same pre-activation)
 *   add_split:        y += addend (in place), planes of y                                                                   */
RECMV_API int recmv_softplus_tangent_planes(const float* tz, int64_t ldt, const float* a, int64_t lda, const float* h,
                                            int64_t ldh, int64_t rows, int cols, float plane_scale, float* u, int64_t ldu,
                                            void* u_hi, void* u_lo, int64_t ldp, float* inj, int64_t ldi,
                                            recmv_stream_t stream);
RECMV_API int recmv_add_split_planes(float* y, int64_t ldy, const float* addend, int64_t lda, int64_t rows, int cols,
                                     float scale, const float* scale_dev, void* y_hi, void* y_lo, int64_t ldp,
                                     recmv_stream_t stream);

/* ---- A3: sdf and its input gradient (ImplicitNetwork.gradient, model/network.py:121-133; the
 * autograd.grad(sdf, p) of utils/FindSurfacePs.py:176 and OptimGarmentNetwork.py:1171,3192) --------------
 * One forward-mode launch of the tcgen05 kernel: every point occupies four tile rows (value and the three
 * directional derivatives), no activations are stored and no transposed weights are needed.
 * out_grad [P,3] = d sdf / d x.  TC modes only (RECMV_E_UNSUPPORTED otherwise).                            */
RECMV_API int recmv_sdf_mlp_fwd_grad(const float* x, const void* packed, const float* pe_w /*host*/,
                           float* out_sdf, float* out_feat, float* out_grad, int64_t P, int mode,
                           recmv_stream_t stream);

/* ---- A4 + A5: MLPTranslator.forward followed by LBSkinner.forward (CompositeDeformer) in ONE launch ------
 * replaces model/Deformer.py:171-206 (PE ++ cond[batch] -> 512 x4 ReLU -> 3, p + offset) and :406-445.
 * Same tcgen05 engine as the SDF network (3 input K blocks, 4 hidden layers, 32-wide tail tile).
 * pack: W_l [out,in] row-major fp32, l = 0..4 concatenated (167->512, 512->512 x3, 512->3); b likewise.
 * conds [F,128]; batch_inds [P] i64 or NULL (frame = p / points_per_frame); pe_w [12] host.
 * Outputs (each may be NULL): out_translated = p + offset, out_offset, out_posed = LBS(p + offset) (needs
 * A [F,24,4,4], trans [F,3] (+extra_trans) and the channels-last voxel).  TC modes only.                   */
RECMV_API size_t recmv_translator_packed_bytes(void);
RECMV_API int recmv_translator_pack_weights(const float* W_all, const float* b_all, void* packed,
                                  recmv_stream_t stream);
RECMV_API int recmv_deformer_fwd(const float* ps, const float* conds, const int64_t* batch_inds,
                       int64_t points_per_frame, int num_frames, const void* packed,
                       const float* pe_w /*host*/, const float* A, const float* trans,
                       const recmv_voxel_t* vox /*host, may be NULL*/, float* out_translated,
                       float* out_offset, float* out_posed, int64_t P, int mode, recmv_stream_t stream);

/* Forward-mode variant of recmv_deformer_fwd (A7, utils/utils.py:133-156 compute_Jacobian without autograd): every
 * point travels as 4 tile rows (value + 3 tangents); out_jac [P,9] row-major, J[i][j] = d out_i / d p_j where
 * `out` is out_posed when the skeleton/voxel are given, else out_translated.  The skinning weights' own
 * dependence on the point (d w / d q, sampler backward semantics incl. zero gradient on clamped axes) is included. */
RECMV_API int recmv_deformer_fwd_jac(const float* ps, const float* conds, const int64_t* batch_inds,
                           int64_t points_per_frame, int num_frames, const void* packed,
                           const float* pe_w /*host*/, const float* A, const float* trans,
                           const recmv_voxel_t* vox /*host, may be NULL*/, float* out_translated,
                           float* out_offset, float* out_posed, float* out_jac, int64_t P, int mode,
                           recmv_stream_t stream);

/* ---- A8: RenderingNetwork_view_norm.forward, mode 'idr' (model/RenderNet.py:59-96) in one launch -----------------
 * cat[points 3 | PE4(view_dirs) 27 | normals 3 | feature_vectors 256] = 289 -> 512 x4 ReLU -> 3 -> tanh.
 * pack: effective (weight-norm materialised) W_l [out,in] row-major fp32 concatenated, l = 0..4; b likewise.
 * pe_w [8] host = annealing weights of the 4-band view-direction encoding.  All tensors [P,*] row-major fp32.
 * TC modes only.                                                                                              */
RECMV_API size_t recmv_rendernet_packed_bytes(void);
RECMV_API int recmv_rendernet_pack_weights(const float* W_all, const float* b_all, void* packed,
                                 recmv_stream_t stream);
RECMV_API int recmv_rendernet_fwd(const float* points, const float* normals, const float* view_dirs,
                        const float* feats, const void* packed, const float* pe_w /*host*/, float* out_rgb,
                        int64_t P, int mode, recmv_stream_t stream);

/* ---- coarse-to-fine sweep helpers (A11, MCAcc/seg3d_lossless.py:233-428) -------------------------------------------
 * interp2x_boundary3d: replaces MCAcc/cuda/interp2x_boundary3d.cpp:18-35 (forward(input, balance) -> [output,
 * is_boundary]; backward(grad_output) -> grad_input).  input [NC,D,H,W] f32 -> output [NC,2D-1,2H-1,2W-1] f32 and
 * is_boundary (1 byte per voxel: the contributing coarse voxels are not all on one side of balance_value).
 * order 0 = the rounding of the reference extension (sequential sum / count), order 1 = the rounding of
 * F.interpolate(mode='trilinear', align_corners=True), the reference's default path (seg3d_lossless.py:270-281).
 * recmv_c2f_todo_mask: todo = (3x3x3 dilation of is_boundary) & ~done  (seg3d_lossless.py:297-303).                */
RECMV_API int recmv_interp2x_boundary3d_fwd(const float* input, float* output, uint8_t* is_boundary, int NC,
                                  int D, int H, int W, float balance_value, int order,
                                  recmv_stream_t stream);
RECMV_API int recmv_interp2x_boundary3d_bwd(const float* grad_output, float* grad_input, int NC, int D, int H,
                                  int W, recmv_stream_t stream);
RECMV_API int recmv_c2f_todo_mask(const uint8_t* is_boundary, const uint8_t* done, uint8_t* todo, int D, int H,
                        int W, recmv_stream_t stream);

/* ---- A9 + (f3): FindSurfacePs + view_rays + the mask filter of sample_train_ray ------------------------------------
 * replaces utils/FindSurfacePs.py:7-60 (nonzero / torch_scatter scatter(min) / gathers), model/CameraMine.py:146-167
 * (view_rays) and the `gt_mask > 0` selection of OptimGarmentNetwork.py:1006-1011, in three launches and one ordered
 * compaction.  pix_to_face [N,H,W,K] int64, bary [N,H,W,K,3] f32 (pytorch3d Fragments), verts [V,3], faces [F,3] int64,
 * mask [N,H,W] f32 or NULL, camera = host float[13] {fx, fy, px, py, R row-major} or NULL.
 * Outputs have capacity N*H*W rows and are filled in (n, row, col) order -- the order of the reference's `nonzero`:
 * out_batch/out_row/out_col/out_finds int64, out_pts [.,3] (barycentric seed point on the canonical mesh), out_rays [.,3]
 * (only with a camera).  counters (device int32[1]) <- number of rows.  scratch: recmv_fragment_decode_scratch_bytes.   */
RECMV_API size_t recmv_fragment_decode_scratch_bytes(int64_t npix);
RECMV_API int recmv_fragment_decode(const int64_t* pix_to_face, const float* bary, int N, int H, int W, int K,
                          const float* verts, const int64_t* faces, int64_t num_faces, const float* mask,
                          const float* camera /*host[13]*/, void* scratch, int64_t* out_batch, int64_t* out_row,
                          int64_t* out_col, float* out_pts, int64_t* out_finds, float* out_rays, int32_t* counters,
                          recmv_stream_t stream);

/* ---- mesh rasteriser: what `maskRender` gets from pytorch3d's MeshRasterizer (model/network.py:307-322; faces_per_pixel=1,
 * blur_radius=0, perspective_correct=True, no culling), in the camera convention of model/CameraMine.py:146-173 --------------
 * verts [N,V,3] f32 (N posed meshes sharing faces [F,3] int64), cam = host float[4] {fx, fy, px, py} shared by all frames,
 * R [NR,3,3] row-major and T [NR,3] device f32 with NR = 1 or N: Xc = Xw R + T, screen x = px - fx Xc/Zc, y = py - fy Yc/Zc,
 * pixel (row, col) = screen point (x = col, y = row).  A face covers a pixel when its three screen-space barycentrics at the
 * pixel centre are > 0 (either winding) and its three vertices have Zc > 0; zero-area faces cover nothing.  Winner: smallest
 * perspective-correct Zc, then smallest face index (deterministic).  Outputs (pytorch3d layout, -1 on background):
 * pix_to_face [N,H,W] int64 = n*F + f, zbuf [N,H,W] f32 = Zc, bary [N,H,W,3] f32 perspective-correct, vertex order of
 * the face.  Faces with a clipped bounding box over 128 pixels are swept by a warp.  Face indices must be in range.
 * scratch: recmv_raster_scratch_bytes(N, H, W) bytes.  Two kernels + one memset, no host synchronisation.           */
RECMV_API int recmv_raster_scratch_bytes(int N, int H, int W, size_t* bytes /*host*/);
RECMV_API int recmv_rasterize(const float* verts, const int64_t* faces, int N, int64_t V, int64_t F,
                    const float* cam /*host float[4]: fx fy px py*/, const float* R, const float* T, int NR, int H, int W,
                    void* scratch, int64_t* pix_to_face, float* zbuf, float* bary, recmv_stream_t stream);

/* ---- points rasteriser + alpha compositor: what `pcRender` gets from pytorch3d's PointsRasterizer + AlphaCompositor
 * (model/CameraMine.py:306-415, OptimNetwork.py:87-100), in the camera convention of recmv_rasterize --------------------
 * points [N,P,3] f32 (N clouds of P points), cam = host float[4] {fx, fy, px, py}, R [NR,3,3] row-major and T [NR,3]
 * device f32 with NR = 1 or N.  Point p covers pixel (row i, col j) when Zc > 0 and d^2 = (sx - j)^2 + (sy - i)^2 < r^2,
 * r = radius min(H, W) / 2 (radius > 0 in NDC units).  Per pixel the K (1..64) covering points with the smallest Zc,
 * ties to the smaller packed index n*P + p; weight a = 1 - d^2 / r^2; images [N,H,W,C] = alpha composite of
 * features [P,C] (C = 1..4, shared by the clouds), no background.  N*P < 2^32, N*H*W < 2^31.
 * scratch: recmv_points_scratch_bytes(N, P, H, W) bytes, kept from the count call to the last backward / fragments call.
 * recmv_points_count: projection, per-pixel candidate counts and their scan; ONE blocking read: *total (host) = the
 *   candidate total, RECMV_E_RANGE above 2^31 - 1.
 * recmv_points_render: once per count call (it consumes the counts); cand = total x 8 bytes (device; may be NULL when
 *   total = 0).  Images and the kept lists are bit-identical from call to call.
 * recmv_points_render_backward: grad_points [N,P,3] = dL/dpoints from grad_images [N,H,W,C], with the scratch and cand
 *   of the render call; fp32 atomics (sums not deterministic), no host synchronisation.
 * recmv_points_fragments: dense idx [N,H,W,K] int64 (packed n*P + p), zbuf (Zc), dists (d^2 (2 / min(H, W))^2),
 *   -1 in empty slots.                                                                                                  */
RECMV_API int recmv_points_scratch_bytes(int N, int64_t P, int H, int W, size_t* bytes /*host*/);
RECMV_API int recmv_points_count(const float* points, int N, int64_t P, const float* cam /*host float[4]: fx fy px py*/,
                       const float* R, const float* T, int NR, int H, int W, float radius, void* scratch,
                       int64_t* total /*host*/, recmv_stream_t stream);
RECMV_API int recmv_points_render(const float* features, int C, int N, int64_t P, int H, int W, float radius, int K,
                        void* scratch, void* cand, int64_t total, float* images, recmv_stream_t stream);
RECMV_API int recmv_points_render_backward(const float* points, int N, int64_t P, const float* cam /*host float[4]*/,
                                 const float* R, const float* T, int NR, int H, int W, float radius,
                                 const float* features, int C, int K, void* scratch, const void* cand,
                                 const float* grad_images, float* grad_points, recmv_stream_t stream);
RECMV_API int recmv_points_fragments(int N, int64_t P, int H, int W, float radius, int K, const void* scratch,
                           const void* cand, int64_t* idx, float* zbuf, float* dists, recmv_stream_t stream);

/* ---- A11 / (f2): the sweep of one pyramid level as a DEVICE WORKLIST (SURVEY 8b `recmv_c2f_sweep`) -----------------
 * replaces the coordinate-list bookkeeping of MCAcc/seg3d_lossless.py:306-428 (nonzero / unique / index scatter, a
 * host sync per step).  level / final_res are (W, H, D) = (x, y, z) lattice sizes (host).
 *  recmv_c2f_done_up      : done_up[2z,2y,2x] = done[z,y,x], 0 elsewhere.
 *  recmv_c2f_compact      : voxels with todo != 0 -> idx_out[i] (flat level index), points_out[i] = the query point of
 *                           batch_eval (:89-100), bit-identical arithmetic; counters (device int32[2] = {count, overflow},
 *                           zeroed by the caller) is advanced with one atomic per warp; order is unspecified.
 *  recmv_sdf_mlp_fwd_counted (above): evaluates points_out[0 .. *counters) without the host knowing the count.
 *  recmv_c2f_scatter      : occ[idx] = vals, done[idx] = 1, calculated[final-lattice position] = 1; a sign flip against
 *                           the interpolated value sets conflict_flag[idx] (caller zeroes it); stats (device int32[2])
 *                           += {queried, conflicts}.
 *  recmv_c2f_conflict_todo: todo = dilate3x3x3(conflict_flag) & ~calculated[z*sz, y*sy, x*sx]  (:392-420).          */
RECMV_API int recmv_c2f_done_up(const uint8_t* done, int D, int H, int W, uint8_t* done_up, recmv_stream_t stream);
RECMV_API int recmv_c2f_compact(const uint8_t* todo, const int level[3] /*host*/, const int final_res[3] /*host*/,
                      const float b_min[3] /*host*/, const float b_max[3] /*host*/, int32_t* idx_out, float* points_out,
                      int32_t* counters, int capacity, recmv_stream_t stream);
RECMV_API int recmv_c2f_scatter(const int32_t* idx, const float* vals, const int32_t* counters, int capacity,
                      const int level[3] /*host*/, const int final_res[3] /*host*/, float* occ, uint8_t* done,
                      uint8_t* calculated, uint8_t* conflict_flag, float balance_value, int32_t* stats,
                      recmv_stream_t stream);
RECMV_API int recmv_c2f_conflict_todo(const uint8_t* conflict_flag, const uint8_t* calculated, const int level[3] /*host*/,
                            const int final_res[3] /*host*/, uint8_t* todo, recmv_stream_t stream);
/* The fused form Seg3dLossless._forward_device uses -- ONE full-grid pass per level instead of four:
 *  recmv_c2f_refine       : coarse level (D,H,W) -> fine level (2D-1,2H-1,2W-1): upsampled values (order as
 *                           recmv_interp2x_boundary3d_fwd), the level's done lattice, and the voxels to query appended to
 *                           (idx_out, points_out).  The 3x3x3 dilation of the mixed-stencil flags is evaluated exactly
 *                           from a coarse "mixed cell" mask (mixed_scratch, (D-1)(H-1)(W-1) bytes).
 *  recmv_c2f_scatter_list : as recmv_c2f_scatter, conflicts appended to conflict_list / conflict_count (zeroed by the
 *                           caller); clears the claim bytes of the consumed voxels.
 *  recmv_c2f_mark_conflicts: next worklist = not-yet-evaluated 3x3x3 neighbours of the conflicting voxels, each claimed
 *                           once through `claim` (level-lattice bytes, 4-byte aligned, all zero between rounds).      */
RECMV_API int recmv_c2f_refine(const float* occ_coarse, const uint8_t* done_coarse, int D, int H, int W,
                     const int final_res[3] /*host*/, const float b_min[3] /*host*/, const float b_max[3] /*host*/,
                     float balance_value, int order, uint8_t* mixed_scratch, float* occ_fine, uint8_t* done_fine,
                     int32_t* idx_out, float* points_out, int32_t* counters, int capacity, recmv_stream_t stream);
RECMV_API int recmv_c2f_scatter_list(const int32_t* idx, const float* vals, const int32_t* counters, int capacity,
                           const int level[3] /*host*/, const int final_res[3] /*host*/, float* occ, uint8_t* done,
                           uint8_t* calculated, uint8_t* claim, float balance_value, int32_t* conflict_list,
                           int32_t* conflict_count, int32_t* stats, recmv_stream_t stream);
RECMV_API int recmv_c2f_mark_conflicts(const int32_t* conflict_list, const int32_t* conflict_count, int list_capacity,
                             const uint8_t* calculated, const int level[3] /*host*/, const int final_res[3] /*host*/,
                             const float b_min[3] /*host*/, const float b_max[3] /*host*/, uint8_t* claim,
                             int32_t* idx_out, float* points_out, int32_t* counters, int capacity,
                             recmv_stream_t stream);

/* ---- A10: surface-point solve of a batch of rays on the device (utils/FindSurfacePs.py:145-353) -------------------
 * ps [P,3]: in = seeds (FindSurfacePs), out = solution; ok [P] = converged (|f| < dthreshold and the angle between
 * D(p) - cam and the ray < athreshold_deg).  Networks: packed SDF weights, packed translator weights + conds
 * [F,128] + skeleton (A [F,24,4,4], trans [F,3]) + channels-last voxel, i.e. the CompositeDeformer
 * [MLPTranslator, LBSkinner]; batch_inds [P] i64 (or NULL: one frame).  `times` steps = times + 1 rounds of two
 * forward-mode launches + one update kernel; no host synchronisation.  workspace: recmv_surface_solve_workspace(P)
 * bytes of device memory.  TC modes only.                                                                            */
RECMV_API size_t recmv_surface_solve_workspace(int64_t P);
RECMV_API int recmv_surface_solve(const float* cam_pos /*host[3]*/, const float* rays, float* ps,
                        const int64_t* batch_inds, const void* sdf_packed, const float* sdf_pe_w /*host[12]*/,
                        const void* tr_packed, const float* tr_pe_w /*host[12]*/, const float* conds,
                        int num_frames, const float* A, const float* trans, const recmv_voxel_t* vox /*host*/,
                        float dthreshold, float athreshold_deg, float w1, float w2, int times, int mode,
                        void* workspace, size_t workspace_bytes, uint8_t* ok, int64_t P, recmv_stream_t stream);

/* ---- implicit-surface gradient, per-ray algebra (SURVEY 8f rank 1; engineer/networks/OptimNetwork.py:788-851) -------
 * b = [grad_f_p ; [v]x J] (4x3), r = grad_l_p (b^T b)^-1 b^T with FastMinv's |det| < 1e-4 rule (ok = 0, zeros).
 * Outputs: sdf_coef [n] = -r[0] (the cotangent the reference feeds to autograd.grad(sdf(p), params, .)),
 * def_vec [n,3] = r[1:4] (-[v]x) (the cotangent for autograd.grad(D(p), params, .)), optional ray_grad [n,3] =
 * r[1:4] [d - c]x (needs d_minus_c [n,3]).  All inputs [n,3] except jac [n,3,3] (row i = gradient of D_i), fp32.   */
RECMV_API int recmv_surface_grad_coeffs(const float* grad_l_p, const float* grad_f_p, const float* jac,
                              const float* rays, const float* d_minus_c /*may be NULL*/, float* sdf_coef,
                              float* def_vec, float* ray_grad /*may be NULL*/, uint8_t* ok, int64_t n,
                              recmv_stream_t stream);

/* Calibration knob of the tcgen05 modes.  The tensor core accumulates in fp32 with truncation: each of the K/16
 * MMAs that adds into the full-size accumulator loses on average ~2^-24 of it, a systematic bias towards zero.  The
 * epilogue therefore scales a layer's raw accumulators by (1 + gain_per_kblock * K/64); the default gain is
 * 4 * 2^-24 (measured optimum against the reference's fp32 results, tools/calibrate_acc_gain.py; 0 disables).      */
RECMV_API int recmv_tc_set_acc_gain(int mode, float gain_per_kblock);

/* Non-blocking health check of the tcgen05 path on the current device: every mbarrier wait in the kernel is
 * bounded; a wait that times out records {code, barrier tag, block} in mapped host memory and later launches
 * are refused with RECMV_E_DEVICE.  info may be NULL; clear != 0 resets the record.                        */
RECMV_API int recmv_check_async_errors(int* info /*host [3]*/, int clear);

/* ---- (f4) deformation regulariser: 3x3 SVD of the translator Jacobians ---------------------------------------------
 * replaces `_, s, _ = torch.svd(Jacobs.cpu())` and its autograd backward (engineer/networks/OptimGarmentNetwork.py:1148:
 * device -> host copy, LAPACK, host -> device copy on every training step).  J [N,3,3] f32 row-major = U diag(S) V^T,
 * S [N,3] descending (torch.svd's convention); U, V [N,3,3] may be NULL.  One-sided Jacobi in registers, one matrix per
 * thread.  recmv_svd3x3_backward_s: dJ = U diag(dS) V^T -- the VJP of S alone (what a loss on the singular values needs). */
RECMV_API int recmv_svd3x3(const float* J, int64_t N, float* U, float* S, float* V, recmv_stream_t stream);
RECMV_API int recmv_svd3x3_backward_s(const float* U, const float* V, const float* dS, int64_t N, float* dJ,
                                      recmv_stream_t stream);

/* Diagnostics (tcgen05 bring-up trace entry, issue-rate microbenchmark) are NOT part of this ABI: include/recmv_b200_diag.h,
 * librecmv_b200_diag.so (tools/ only).                                                                                  */

/* ---- the fused render path (BASELINE north star) -------------------------------------------------
 * One launch: ray r, sample k -> x_obs = cam_pos + t_k dir_r, t_k = t_near + (k+1/2)(t_far-t_near)/S
 * -> inverse LBS (frame = frame_of_ray[r] or r / rays_per_frame) -> PE -> SDF MLP -> sdf [R,S].
 * Per ray also: hit_idx[r] = first k with sdf_k <= 0 (-1 if none or if sample 0 is already inside),
 * hit_t[r] = depth of the linear zero crossing between samples k-1 and k.
 * out_xc [R,S,3] optional (NULL).  Samples whose inverse warp is singular get sdf = +1e10 (never hit).*/
typedef struct {
  float cam_pos[3];
  float t_near, t_far;
  int samples_per_ray;
} recmv_raymarch_t;

RECMV_API int recmv_render_sdf(const float* ray_dirs /*[R,3]*/, const recmv_raymarch_t* rm /*host*/,
                     const float* A, const float* trans, const int32_t* frame_of_ray,
                     int64_t rays_per_frame, int num_frames, const recmv_voxel_t* vox /*host*/,
                     const void* packed, const float* pe_w /*host*/, float* out_sdf, float* out_xc,
                     int32_t* hit_idx, float* hit_t, int64_t R, int mode, recmv_stream_t stream);
/* second pass of the same launch sequence: per-ray first-hit scan over out_sdf (exposed for tests) */
RECMV_API int recmv_ray_first_hit(const float* sdf /*[R,S]*/, const recmv_raymarch_t* rm /*host*/,
                        int32_t* hit_idx, float* hit_t, int64_t R, recmv_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RECMV_B200_H_ */
