// Mesh rasteriser: N posed meshes that share one face list -> one face per pixel.  What the reference gets from
// pytorch3d's MeshRasterizer with faces_per_pixel=1, blur_radius=0, perspective_correct=True and no culling
// (model/network.py:307-322), stated in the reference camera's own convention (model/CameraMine.py:169-173 `project`,
// :146-167 `view_rays`):
//   Xc = Xw R + T,   screen x = px - fx Xc/Zc,  y = py - fy Yc/Zc,   pixel (row, col) <-> screen point (x = col, y = row).
// A face covers a pixel when the three screen-space barycentrics at the pixel centre are > 0 (either winding) and the three
// vertices have Zc > 0; a face of zero screen area covers nothing.  Among the covering faces the smallest perspective-correct
// Zc wins, an exact tie goes to the smallest face index: one 64-bit atomicMin of (float bits of Zc) << 32 | f per pixel
// (Zc > 0, so the bits order like the values), which makes the result independent of launch order.
//
// Passes: clear the per-pixel keys (memset), face pass, resolve pass.
//  * face pass, one thread per (frame, face): setup in fp64 (projection, signed area, bounding box clipped to the image,
//    edge functions divided by the area and anchored at the first pixel of the box), so the per-pixel test is three fp32
//    FMAs on numbers of the order of the barycentrics.  A face whose clipped box holds <= kWarpFacePixels pixels is swept
//    by its own thread; a larger one (camera close-ups, coarse meshes) by the whole warp, pixel k of the box on lane k % 32.
//  * resolve, one thread per pixel: decode the winner, recompute its screen barycentrics and depth at the pixel centre in
//    fp64, write the perspective-correct barycentrics, Zc and the packed face index n*F + f (-1 everywhere on background).
// HBM: per face 3 x 12 B of vertices + 24 B of indices, per pixel an 8 B key (cleared, atomics, read) + 24 B of output.
#include "common.cuh"

namespace recmv {
namespace {

constexpr int kRasterThreads = 256;
constexpr int kWarpFacePixels = 128;
constexpr unsigned long long kEmptyKey = ~0ull;   // high word 0xffffffff is a NaN pattern: never a depth

struct RasterCam {
  double fx, fy, px, py;
};

struct FaceSetup {
  float ba[3], bb[3], bc[3];   // screen bary_i at anchor + (dx, dy) = ba_i dx + bb_i dy + bc_i
  float iz[3];                 // 1 / Zc_i
  int x0, y0, bw, bh;          // anchor (first pixel of the clipped box) and box size
};

__device__ __forceinline__ void project_vertex(const float* __restrict__ v, const float* __restrict__ R,
                                               const float* __restrict__ T, const RasterCam& cam, double& sx, double& sy,
                                               double& z) {
  const double X = v[0], Y = v[1], Z = v[2];
  const double cx = X * R[0] + Y * R[3] + Z * R[6] + T[0];
  const double cy = X * R[1] + Y * R[4] + Z * R[7] + T[1];
  z = X * R[2] + Y * R[5] + Z * R[8] + T[2];
  const double rz = 1.0 / z;
  sx = cam.px - cam.fx * cx * rz;
  sy = cam.py - cam.fy * cy * rz;
}

// the three projected vertices of face f; false when one of them has Zc <= 0
__device__ __forceinline__ bool project_face(const float* __restrict__ verts_n, const long long* __restrict__ faces,
                                             long long f, const float* __restrict__ R, const float* __restrict__ T,
                                             const RasterCam& cam, double sx[3], double sy[3], double z[3]) {
  bool ok = true;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    project_vertex(verts_n + 3 * faces[3 * f + i], R, T, cam, sx[i], sy[i], z[i]);
    ok = ok && z[i] > 0.0;
  }
  return ok;
}

// edge function of vertex i (zero on the opposite edge), evaluated at (x, y): sum over i = the signed double area
__device__ __forceinline__ double edge_fn(const double sx[3], const double sy[3], int i, double x, double y) {
  const int a = (i + 1) % 3, b = (i + 2) % 3;
  return (sx[b] - sx[a]) * (y - sy[a]) - (sy[b] - sy[a]) * (x - sx[a]);
}

__device__ __forceinline__ bool face_setup(const float* __restrict__ verts_n, const long long* __restrict__ faces,
                                           long long f, const float* __restrict__ R, const float* __restrict__ T,
                                           const RasterCam& cam, int H, int W, FaceSetup& s) {
  double sx[3], sy[3], z[3];
  if (!project_face(verts_n, faces, f, R, T, cam, sx, sy, z)) return false;
  const double area = edge_fn(sx, sy, 0, sx[0], sy[0]);
  if (!(area != 0.0) || !isfinite(area)) return false;
  // pixel centres strictly inside lie in [ceil(min), floor(max)]; clip before converting to int
  const double xlo = fmax(ceil(fmin(fmin(sx[0], sx[1]), sx[2])), 0.0);
  const double xhi = fmin(floor(fmax(fmax(sx[0], sx[1]), sx[2])), (double)(W - 1));
  const double ylo = fmax(ceil(fmin(fmin(sy[0], sy[1]), sy[2])), 0.0);
  const double yhi = fmin(floor(fmax(fmax(sy[0], sy[1]), sy[2])), (double)(H - 1));
  if (!(xlo <= xhi && ylo <= yhi)) return false;
  s.x0 = (int)xlo; s.y0 = (int)ylo;
  s.bw = (int)(xhi - xlo) + 1; s.bh = (int)(yhi - ylo) + 1;
  const double inv_area = 1.0 / area;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int a = (i + 1) % 3, b = (i + 2) % 3;
    s.ba[i] = (float)(-(sy[b] - sy[a]) * inv_area);
    s.bb[i] = (float)((sx[b] - sx[a]) * inv_area);
    s.bc[i] = (float)(edge_fn(sx, sy, i, xlo, ylo) * inv_area);
    s.iz[i] = (float)(1.0 / z[i]);
  }
  return true;
}

__device__ __forceinline__ void raster_pixel(const FaceSetup& s, int dx, int dy, unsigned f,
                                             unsigned long long* __restrict__ keys_n, int W) {
  const float fx = (float)dx, fy = (float)dy;
  const float b0 = fmaf(s.ba[0], fx, fmaf(s.bb[0], fy, s.bc[0]));
  const float b1 = fmaf(s.ba[1], fx, fmaf(s.bb[1], fy, s.bc[1]));
  const float b2 = fmaf(s.ba[2], fx, fmaf(s.bb[2], fy, s.bc[2]));
  if (!(b0 > 0.f && b1 > 0.f && b2 > 0.f)) return;
  const float z = __frcp_rn(fmaf(b0, s.iz[0], fmaf(b1, s.iz[1], b2 * s.iz[2])));   // perspective-correct Zc
  const unsigned long long key = ((unsigned long long)__float_as_uint(z) << 32) | f;
  unsigned long long* k = keys_n + (size_t)(s.y0 + dy) * W + (s.x0 + dx);
  if (key < *k) atomicMin(k, key);   // keys only decrease: a stale read can only cause a redundant atomic
}

__device__ __forceinline__ FaceSetup shfl_setup(const FaceSetup& s, int src) {
  FaceSetup q;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    q.ba[i] = __shfl_sync(0xffffffffu, s.ba[i], src);
    q.bb[i] = __shfl_sync(0xffffffffu, s.bb[i], src);
    q.bc[i] = __shfl_sync(0xffffffffu, s.bc[i], src);
    q.iz[i] = __shfl_sync(0xffffffffu, s.iz[i], src);
  }
  q.x0 = __shfl_sync(0xffffffffu, s.x0, src);
  q.y0 = __shfl_sync(0xffffffffu, s.y0, src);
  q.bw = __shfl_sync(0xffffffffu, s.bw, src);
  q.bh = __shfl_sync(0xffffffffu, s.bh, src);
  return q;
}

__global__ void __launch_bounds__(kRasterThreads) raster_faces_kernel(
    const float* __restrict__ verts, const long long* __restrict__ faces, int N, long long V, long long F,
    const float* __restrict__ R, const float* __restrict__ T, int NR, RasterCam cam, int H, int W,
    unsigned long long* __restrict__ keys) {
  const long long t = blockIdx.x * (long long)kRasterThreads + threadIdx.x;
  const int lane = threadIdx.x & 31;
  FaceSetup s = {};
  bool ok = false;
  int n = 0;
  long long f = 0;
  if (t < (long long)N * F) {   // no early return: the whole warp takes part in the large-face sweep below
    n = (int)(t / F);
    f = t - (long long)n * F;
    const int c = NR == 1 ? 0 : n;
    ok = face_setup(verts + (size_t)n * V * 3, faces, f, R + 9 * c, T + 3 * c, cam, H, W, s);
  }
  const long long hw = (long long)H * W;
  const bool big = ok && s.bw * s.bh > kWarpFacePixels;
  if (ok && !big) {
    unsigned long long* keys_n = keys + (size_t)n * hw;
    for (int dy = 0; dy < s.bh; ++dy)
      for (int dx = 0; dx < s.bw; ++dx) raster_pixel(s, dx, dy, (unsigned)f, keys_n, W);
  }
  unsigned m = __ballot_sync(0xffffffffu, big);
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const FaceSetup q = shfl_setup(s, src);
    const int qn = __shfl_sync(0xffffffffu, n, src);
    const unsigned qf = __shfl_sync(0xffffffffu, (unsigned)f, src);
    unsigned long long* keys_n = keys + (size_t)qn * hw;
    const int npx = q.bw * q.bh;
    for (int k = lane; k < npx; k += 32) {
      const int dy = k / q.bw;
      raster_pixel(q, k - dy * q.bw, dy, qf, keys_n, W);
    }
  }
}

__global__ void __launch_bounds__(kRasterThreads) raster_resolve_kernel(
    const unsigned long long* __restrict__ keys, const float* __restrict__ verts, const long long* __restrict__ faces,
    long long V, long long F, const float* __restrict__ R, const float* __restrict__ T, int NR, RasterCam cam, int H,
    int W, long long npix, long long* __restrict__ p2f, float* __restrict__ zbuf, float* __restrict__ bary) {
  const long long p = blockIdx.x * (long long)kRasterThreads + threadIdx.x;
  if (p >= npix) return;
  const unsigned long long key = keys[p];
  if (key == kEmptyKey) {
    p2f[p] = -1;
    zbuf[p] = -1.f;
    bary[3 * p] = -1.f; bary[3 * p + 1] = -1.f; bary[3 * p + 2] = -1.f;
    return;
  }
  const long long hw = (long long)H * W;
  const int n = (int)(p / hw);
  const int rem = (int)(p - (long long)n * hw);
  const int row = rem / W, col = rem - row * W;
  const long long f = (long long)(key & 0xffffffffull);
  const int c = NR == 1 ? 0 : n;
  double sx[3], sy[3], z[3];
  project_face(verts + (size_t)n * V * 3, faces, f, R + 9 * c, T + 3 * c, cam, sx, sy, z);
  // bary_i = e_i / area;  perspective-correct bary_i ~ e_i / z_i ~ u_i = e_i z_{i+1} z_{i+2};  Zc = area z0 z1 z2 / sum u
  const double area = edge_fn(sx, sy, 0, sx[0], sy[0]);
  double u[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) u[i] = edge_fn(sx, sy, i, (double)col, (double)row) * z[(i + 1) % 3] * z[(i + 2) % 3];
  const double inv_s = 1.0 / (u[0] + u[1] + u[2]);
  p2f[p] = (long long)n * F + f;
  zbuf[p] = (float)(area * z[0] * z[1] * z[2] * inv_s);
#pragma unroll
  for (int i = 0; i < 3; ++i) bary[3 * p + i] = (float)(u[i] * inv_s);
}

int check_sizes(int N, int H, int W) {
  if (N <= 0 || H <= 0 || W <= 0) return RECMV_E_SHAPE;
  if ((int64_t)H * W > 0x7fffffffLL) return RECMV_E_RANGE;
  return RECMV_OK;
}

}  // namespace
}  // namespace recmv

using namespace recmv;

extern "C" int recmv_raster_scratch_bytes(int N, int H, int W, size_t* bytes) {
  const int s = check_sizes(N, H, W);
  if (s) return s;
  if (!bytes) return RECMV_E_NULL;
  *bytes = (size_t)N * H * W * sizeof(unsigned long long);
  return RECMV_OK;
}

extern "C" int recmv_rasterize(const float* verts, const int64_t* faces, int N, int64_t V, int64_t F, const float* cam,
                               const float* R, const float* T, int NR, int H, int W, void* scratch, int64_t* pix_to_face,
                               float* zbuf, float* bary, recmv_stream_t stream) {
  int s = check_sizes(N, H, W);
  if (s) return s;
  if (V <= 0 || F <= 0 || (NR != 1 && NR != N)) return RECMV_E_SHAPE;
  if (F > 0xffffffffLL) return RECMV_E_RANGE;   // the face index is the low word of the key
  const long long max_threads = 0x7fffffffLL * kRasterThreads;   // one-dimensional grids
  if ((long long)N * F > max_threads || (long long)N * H * W > max_threads) return RECMV_E_RANGE;
  if (!verts || !faces || !cam || !R || !T || !scratch || !pix_to_face || !zbuf || !bary) return RECMV_E_NULL;
  cudaStream_t st = (cudaStream_t)stream;
  const RasterCam c = {cam[0], cam[1], cam[2], cam[3]};
  const long long npix = (long long)N * H * W;
  unsigned long long* keys = (unsigned long long*)scratch;
  cudaError_t e = cudaMemsetAsync(keys, 0xff, (size_t)npix * sizeof(unsigned long long), st);
  if (e != cudaSuccess) return (int)e;
  const long long nf = (long long)N * F;
  raster_faces_kernel<<<(unsigned)((nf + kRasterThreads - 1) / kRasterThreads), kRasterThreads, 0, st>>>(
      verts, (const long long*)faces, N, V, F, R, T, NR, c, H, W, keys);
  s = launch_status();
  if (s) return s;
  raster_resolve_kernel<<<(unsigned)((npix + kRasterThreads - 1) / kRasterThreads), kRasterThreads, 0, st>>>(
      keys, verts, (const long long*)faces, V, F, R, T, NR, c, H, W, npix, (long long*)pix_to_face, zbuf, bary);
  return launch_status();
}
