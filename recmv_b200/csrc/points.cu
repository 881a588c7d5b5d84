// Points rasteriser + alpha compositor with its backward: what the reference's point-cloud silhouette renderer `pcRender`
// gets from pytorch3d's PointsRasterizer + AlphaCompositor (model/CameraMine.py:306-415, OptimNetwork.py:87-100), in the
// reference camera's own convention (CameraMine.py:169-173), as `recmv_rasterize` uses it:
//   Xc = Xw R + T,   screen x = px - fx Xc/Zc,  y = py - fy Yc/Zc,   pixel (row i, col j) <-> screen point (x = j, y = i).
// Point p covers pixel (i, j) when Zc > 0 and d^2 = (sx - j)^2 + (sy - i)^2 < r^2 (strict), r = radius min(H, W) / 2
// (radius in pytorch3d's NDC units).  Per pixel the K covering points with the smallest Zc are kept, in ascending order;
// an exact tie in float Zc goes to the smaller packed index n P + p.  Weight a_k = 1 - d_k^2 / r^2, image
// I_c = sum_k T_k a_k f[idx_k, c] with T_0 = 1, T_{k+1} = T_k (1 - a_k), no background.
//
// Forward, two C calls:
//  * recmv_points_count: memset of the per-pixel counters; point pass (one thread per (frame, point): fp64 projection
//    stored, atomicAdd over the covered pixels of the disc's clipped bounding box); three-kernel exclusive scan of the
//    counts into per-pixel segment offsets (int64); ONE blocking read: the candidate total, which sizes the list.
//  * recmv_points_render: emit (every candidate writes (float bits of Zc) << 32 | packed index into its pixel's segment,
//    at a slot taken by counting the pixel's counter back down to 0); resolve (one warp per pixel): the K smallest keys of
//    the segment -- chunks of 32 keys ranked in shared memory and merged into a sorted list of at most K, chunks that
//    cannot enter a full list skipped -- are written back, sorted, to the front of the segment; d^2 is recomputed in fp64
//    from the stored screen position and the C <= 4 channels are composited in fp32.  The selection depends only on the
//    set of keys, so images and fragments are bit-identical from call to call whatever the emit order.
// Backward (recmv_points_render_backward), no host synchronisation: one warp per pixel runs the division-free reverse
// sweep dI_c/da_k = T_k (f_kc - R_kc), R_k = a_{k+1} f_{k+1} + (1 - a_{k+1}) R_{k+1}, over the saved sorted keys and
// accumulates dL/d(sx, sy) = dL/da (-2 (s - pixel) / r^2) per point with fp32 atomicAdd (not deterministic, as
// pytorch3d's); a per-point pass applies the projection Jacobian and writes dL/dXw.  The selection carries no gradient.
// Fragments on request (recmv_points_fragments): the sorted keys expanded to pytorch3d's dense idx / zbuf / dists
// [N,H,W,K] with -1 in empty slots, dists in NDC units d^2 (2 / min(H, W))^2.
#include <cmath>

#include "common.cuh"

namespace recmv {
namespace {

constexpr int kPtsThreads = 256;
constexpr int kPtsWarps = kPtsThreads / 32;
constexpr int kScanItems = 8;                           // pixels per thread in the scan passes
constexpr int kScanTile = kPtsThreads * kScanItems;
constexpr int kMaxK = 64;
constexpr int kMaxC = 4;
constexpr unsigned long long kNoKey = ~0ull;            // pads a chunk; never a candidate (high word is a NaN pattern)

struct PtsCam {
  double fx, fy, px, py;
};

struct PtsScratch {
  double2* scr;        // [N P] screen position (fp64)
  float* zc;           // [N P] Zc, or -1 for a point that covers nothing (Zc <= 0 or a non-finite projection)
  float2* gscr;        // [N P] dL/d(sx, sy), backward only
  int* counts;         // [npix] candidates per pixel; counted back down to 0 by the emit pass
  long long* offs;     // [npix + 1] exclusive scan of the counts, offs[npix] = candidate total
  long long* bsums;    // [tiles] per-tile sums of the scan
};

size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

long long scan_tiles(long long npix) { return (npix + kScanTile - 1) / kScanTile; }

PtsScratch carve(void* base, long long np, long long npix, size_t* bytes) {
  PtsScratch s;
  size_t o = 0;
  char* b = (char*)base;
  s.scr = (double2*)(b + o);  o += align256((size_t)np * sizeof(double2));
  s.zc = (float*)(b + o);     o += align256((size_t)np * sizeof(float));
  s.gscr = (float2*)(b + o);  o += align256((size_t)np * sizeof(float2));
  s.counts = (int*)(b + o);   o += align256((size_t)npix * sizeof(int));
  s.offs = (long long*)(b + o); o += align256((size_t)(npix + 1) * sizeof(long long));
  s.bsums = (long long*)(b + o); o += align256((size_t)scan_tiles(npix) * sizeof(long long));
  if (bytes) *bytes = o;
  return s;
}

__device__ __forceinline__ void project_point(const float* __restrict__ v, const float* __restrict__ R,
                                              const float* __restrict__ T, const PtsCam& cam, double& cx, double& cy,
                                              double& z) {
  const double X = v[0], Y = v[1], Z = v[2];
  cx = X * R[0] + Y * R[3] + Z * R[6] + T[0];
  cy = X * R[1] + Y * R[4] + Z * R[7] + T[1];
  z = X * R[2] + Y * R[5] + Z * R[8] + T[2];
}

// d^2 of a screen position to the centre of pixel (row y, col x); one rounding order at every use, so the coverage test
// of the count and emit passes agrees bit for bit and the weights of forward, backward and fragments are the same
__device__ __forceinline__ double dist2(double2 s, int x, int y) {
  const double dx = s.x - (double)x, dy = s.y - (double)y;
  return __fma_rn(dx, dx, __dmul_rn(dy, dy));
}

struct Box {
  int x0, x1, y0, y1;
};

// pixel centres strictly inside the disc lie in [ceil(s - r), floor(s + r)]; clip before converting to int
__device__ __forceinline__ bool disc_box(double2 s, double r, int H, int W, Box& b) {
  const double xlo = fmax(ceil(s.x - r), 0.0), xhi = fmin(floor(s.x + r), (double)(W - 1));
  const double ylo = fmax(ceil(s.y - r), 0.0), yhi = fmin(floor(s.y + r), (double)(H - 1));
  if (!(xlo <= xhi && ylo <= yhi)) return false;
  b.x0 = (int)xlo; b.x1 = (int)xhi; b.y0 = (int)ylo; b.y1 = (int)yhi;
  return true;
}

__global__ void __launch_bounds__(kPtsThreads) pts_count_kernel(
    const float* __restrict__ points, int N, long long P, const float* __restrict__ R, const float* __restrict__ T,
    int NR, PtsCam cam, int H, int W, double r, double r2, double2* __restrict__ scr, float* __restrict__ zc,
    int* __restrict__ counts) {
  const long long t = blockIdx.x * (long long)kPtsThreads + threadIdx.x;
  if (t >= (long long)N * P) return;
  const int n = (int)(t / P);
  const int c = NR == 1 ? 0 : n;
  double cx, cy, z;
  project_point(points + 3 * t, R + 9 * c, T + 3 * c, cam, cx, cy, z);
  const double rz = 1.0 / z;
  const double2 s = make_double2(cam.px - cam.fx * cx * rz, cam.py - cam.fy * cy * rz);
  Box b;
  const bool ok = z > 0.0 && (float)z > 0.f && disc_box(s, r, H, W, b);
  scr[t] = s;
  zc[t] = ok ? (float)z : -1.f;
  if (!ok) return;
  int* cnt = counts + (size_t)n * H * W;
  for (int y = b.y0; y <= b.y1; ++y)
    for (int x = b.x0; x <= b.x1; ++x)
      if (dist2(s, x, y) < r2) atomicAdd(cnt + (size_t)y * W + x, 1);
}

__global__ void __launch_bounds__(kPtsThreads) pts_emit_kernel(
    const double2* __restrict__ scr, const float* __restrict__ zc, long long np, long long P, int H, int W, double r,
    double r2, int* __restrict__ counts, const long long* __restrict__ offs, unsigned long long* __restrict__ cand) {
  const long long t = blockIdx.x * (long long)kPtsThreads + threadIdx.x;
  if (t >= np) return;
  const float z = zc[t];
  if (!(z > 0.f)) return;
  const double2 s = scr[t];
  Box b;
  disc_box(s, r, H, W, b);   // true: the count pass kept this point
  const int n = (int)(t / P);
  const unsigned long long key = ((unsigned long long)__float_as_uint(z) << 32) | (unsigned long long)(unsigned)t;
  const size_t base = (size_t)n * H * W;
  for (int y = b.y0; y <= b.y1; ++y)
    for (int x = b.x0; x <= b.x1; ++x)
      if (dist2(s, x, y) < r2) {
        const size_t pix = base + (size_t)y * W + x;
        const int slot = atomicSub(counts + pix, 1) - 1;
        cand[offs[pix] + slot] = key;
      }
}

// CTA-wide exclusive scan (kPtsThreads threads); total in *tot for every thread
__device__ __forceinline__ long long block_excl_scan(long long v, long long* tot) {
  __shared__ long long warp_sums[kPtsWarps];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  long long inc = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const long long a = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= o) inc += a;
  }
  if (lane == 31) warp_sums[wid] = inc;
  __syncthreads();
  long long before = 0, all = 0;
#pragma unroll
  for (int w = 0; w < kPtsWarps; ++w) {
    const long long ws = warp_sums[w];
    before += w < wid ? ws : 0;
    all += ws;
  }
  __syncthreads();   // warp_sums is reused by the next call
  *tot = all;
  return before + inc - v;
}

__global__ void __launch_bounds__(kPtsThreads) pts_scan_reduce_kernel(const int* __restrict__ counts, long long npix,
                                                                      long long* __restrict__ bsums) {
  const long long i0 = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  long long sum = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (i0 + j < npix) sum += counts[i0 + j];
  long long tot;
  block_excl_scan(sum, &tot);
  if (threadIdx.x == 0) bsums[blockIdx.x] = tot;
}

// exclusive scan of the tile sums in one CTA; the total -> offs[npix]
__global__ void __launch_bounds__(kPtsThreads) pts_scan_tiles_kernel(long long* __restrict__ bsums, long long nb,
                                                                     long long* __restrict__ total) {
  long long carry = 0;
  for (long long base = 0; base < nb; base += kPtsThreads) {
    const long long b = base + threadIdx.x;
    const long long v = b < nb ? bsums[b] : 0;
    long long tot;
    const long long ex = block_excl_scan(v, &tot);
    if (b < nb) bsums[b] = carry + ex;
    carry += tot;
  }
  if (threadIdx.x == 0) *total = carry;
}

__global__ void __launch_bounds__(kPtsThreads) pts_scan_down_kernel(const int* __restrict__ counts, long long npix,
                                                                    const long long* __restrict__ bsums,
                                                                    long long* __restrict__ offs) {
  const long long i0 = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * kScanItems;
  int c[kScanItems];
  long long sum = 0;
#pragma unroll
  for (int j = 0; j < kScanItems; ++j) {
    c[j] = i0 + j < npix ? counts[i0 + j] : 0;
    sum += c[j];
  }
  long long tot;
  long long run = bsums[blockIdx.x] + block_excl_scan(sum, &tot);
#pragma unroll
  for (int j = 0; j < kScanItems; ++j)
    if (i0 + j < npix) {
      offs[i0 + j] = run;
      run += c[j];
    }
}

// number of entries of the sorted a[0, n) below key
__device__ __forceinline__ int count_below(const unsigned long long* a, int n, unsigned long long key) {
  int lo = 0, hi = n;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (a[mid] < key) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// The K smallest keys of seg[0, L) (distinct), sorted, into list[which][0, n); returns n = min(L, K).  Warp-collective.
__device__ int warp_select(const unsigned long long* __restrict__ seg, long long L, int K,
                           unsigned long long (*list)[kMaxK], unsigned long long* chunk, int lane, int& which) {
  int n = 0;
  which = 0;
  for (long long base = 0; base < L; base += 32) {
    const int m = (int)min(32LL, L - base);
    const unsigned long long key = lane < m ? seg[base + lane] : kNoKey;
    if (n == K) {   // a full list: skip a chunk whose smallest key does not beat the K-th
      unsigned long long mn = key;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long q = __shfl_xor_sync(0xffffffffu, mn, o);
        mn = q < mn ? q : mn;
      }
      if (mn > list[which][K - 1]) continue;
    }
    chunk[lane] = key;
    __syncwarp();
    int rank = 0;
    for (int j = 0; j < m; ++j) rank += chunk[j] < key;
    __syncwarp();
    if (lane < m) chunk[rank] = key;
    __syncwarp();
    const unsigned long long* cur = list[which];
    unsigned long long* nxt = list[which ^ 1];
    if (lane < m) {
      const int pos = rank + count_below(cur, n, key);
      if (pos < K) nxt[pos] = key;
    }
    for (int i = lane; i < n; i += 32) {
      const unsigned long long v = cur[i];
      const int pos = i + count_below(chunk, m, v);
      if (pos < K) nxt[pos] = v;
    }
    __syncwarp();
    n = min(K, n + m);
    which ^= 1;
  }
  return n;
}

__global__ void __launch_bounds__(kPtsThreads) pts_resolve_kernel(
    const long long* __restrict__ offs, unsigned long long* __restrict__ cand, const double2* __restrict__ scr,
    const float* __restrict__ features, long long P, int C, int K, int H, int W, long long npix, double r2,
    float* __restrict__ images) {
  __shared__ unsigned long long s_list[kPtsWarps][2][kMaxK];
  __shared__ unsigned long long s_chunk[kPtsWarps][32];
  __shared__ float s_a[kPtsWarps][kMaxK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long hw = (long long)H * W;
  for (long long pix = (long long)blockIdx.x * kPtsWarps + w; pix < npix; pix += (long long)gridDim.x * kPtsWarps) {
    const long long beg = offs[pix];
    unsigned long long* seg = cand + beg;
    int which;
    const int n = warp_select(seg, offs[pix + 1] - beg, K, s_list[w], s_chunk[w], lane, which);
    const unsigned long long* lst = s_list[w][which];
    const int rem = (int)(pix % hw);
    const int row = rem / W, col = rem - row * W;
    for (int k = lane; k < n; k += 32) {
      const unsigned long long key = lst[k];
      seg[k] = key;   // sorted kept keys at the front of the segment: what backward and fragments read
      s_a[w][k] = (float)(1.0 - dist2(scr[(unsigned)key], col, row) / r2);
    }
    __syncwarp();
    if (lane < C) {
      float tr = 1.f, acc = 0.f;
      for (int k = 0; k < n; ++k) {
        const float a = s_a[w][k];
        const float f = features[((long long)(unsigned)lst[k] % P) * C + lane];
        acc = fmaf(tr * a, f, acc);
        tr *= 1.f - a;
      }
      images[pix * C + lane] = acc;
    }
    __syncwarp();
  }
}

__global__ void __launch_bounds__(kPtsThreads) pts_backward_kernel(
    const long long* __restrict__ offs, const unsigned long long* __restrict__ cand, const double2* __restrict__ scr,
    const float* __restrict__ features, const float* __restrict__ grad_images, long long P, int C, int K, int H, int W,
    long long npix, double r2, float2* __restrict__ gscr) {
  __shared__ unsigned s_idx[kPtsWarps][kMaxK];
  __shared__ float s_a[kPtsWarps][kMaxK];
  __shared__ float s_g[kPtsWarps][kMaxC][kMaxK];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const long long hw = (long long)H * W;
  for (long long pix = (long long)blockIdx.x * kPtsWarps + w; pix < npix; pix += (long long)gridDim.x * kPtsWarps) {
    const long long beg = offs[pix];
    const int n = (int)min((long long)K, offs[pix + 1] - beg);
    if (n == 0) continue;
    const float g = lane < C ? grad_images[pix * C + lane] : 0.f;
    if (!__any_sync(0xffffffffu, g != 0.f)) continue;
    const int rem = (int)(pix % hw);
    const int row = rem / W, col = rem - row * W;
    for (int k = lane; k < n; k += 32) {
      const unsigned i = (unsigned)cand[beg + k];
      s_idx[w][k] = i;
      s_a[w][k] = (float)(1.0 - dist2(scr[i], col, row) / r2);
    }
    __syncwarp();
    if (lane < C) {
      // lane c: its row of s_g first holds T_k, then g_c dI_c/da_k = g_c T_k (f_kc - R_kc), swept back to front
      float* sg = s_g[w][lane];
      float tr = 1.f;
      for (int k = 0; k < n; ++k) {
        sg[k] = tr;
        tr *= 1.f - s_a[w][k];
      }
      float rc = 0.f;
      for (int k = n - 1; k >= 0; --k) {
        const float a = s_a[w][k];
        const float f = features[((long long)s_idx[w][k] % P) * C + lane];
        sg[k] = g * (sg[k] * (f - rc));
        rc = fmaf(a, f, (1.f - a) * rc);
      }
    }
    __syncwarp();
    for (int k = lane; k < n; k += 32) {
      const unsigned i = s_idx[w][k];
      const double2 s = scr[i];
      float ga = s_g[w][0][k];
      for (int c = 1; c < C; ++c) ga += s_g[w][c][k];
      const double q = -2.0 * (double)ga / r2;   // dL/da * da/ds = dL/da * (-2 (s - pixel) / r^2)
      atomicAdd(&gscr[i].x, (float)(q * (s.x - (double)col)));
      atomicAdd(&gscr[i].y, (float)(q * (s.y - (double)row)));
    }
    __syncwarp();
  }
}

// dL/dXw = J^T dL/d(sx, sy):  sx = px - fx Xc/Zc, sy = py - fy Yc/Zc, Xc = Xw R + T
__global__ void __launch_bounds__(kPtsThreads) pts_grad_points_kernel(
    const float* __restrict__ points, int N, long long P, const float* __restrict__ R, const float* __restrict__ T,
    int NR, PtsCam cam, const float* __restrict__ zc, const float2* __restrict__ gscr, float* __restrict__ grad_points) {
  const long long t = blockIdx.x * (long long)kPtsThreads + threadIdx.x;
  if (t >= (long long)N * P) return;
  float* out = grad_points + 3 * t;
  if (!(zc[t] > 0.f)) {
    out[0] = 0.f; out[1] = 0.f; out[2] = 0.f;
    return;
  }
  const int n = (int)(t / P);
  const int c = NR == 1 ? 0 : n;
  const float* Rc = R + 9 * c;
  double cx, cy, z;
  project_point(points + 3 * t, Rc, T + 3 * c, cam, cx, cy, z);
  const float2 g = gscr[t];
  const double rz = 1.0 / z;
  const double gx = -(double)g.x * cam.fx * rz, gy = -(double)g.y * cam.fy * rz;
  const double gz = -(gx * cx + gy * cy) * rz;
#pragma unroll
  for (int i = 0; i < 3; ++i) out[i] = (float)(Rc[3 * i] * gx + Rc[3 * i + 1] * gy + Rc[3 * i + 2] * gz);
}

__global__ void __launch_bounds__(kPtsThreads) pts_fragments_kernel(
    const long long* __restrict__ offs, const unsigned long long* __restrict__ cand, const double2* __restrict__ scr,
    int K, int H, int W, long long total, double ndc2, long long* __restrict__ idx, float* __restrict__ zbuf,
    float* __restrict__ dists) {
  const long long t = blockIdx.x * (long long)kPtsThreads + threadIdx.x;
  if (t >= total) return;
  const long long pix = t / K;
  const int k = (int)(t - pix * K);
  const long long beg = offs[pix];
  if (k >= offs[pix + 1] - beg) {
    idx[t] = -1; zbuf[t] = -1.f; dists[t] = -1.f;
    return;
  }
  const unsigned long long key = cand[beg + k];
  const unsigned i = (unsigned)key;
  const int rem = (int)(pix % ((long long)H * W));
  const int row = rem / W;
  idx[t] = (long long)i;
  zbuf[t] = __uint_as_float((unsigned)(key >> 32));
  dists[t] = (float)(dist2(scr[i], rem - row * W, row) * ndc2);
}

constexpr long long kMaxThreads = 0x7fffffffLL * kPtsThreads;   // one-dimensional grids

int check_sizes(int N, int64_t P, int H, int W, float radius) {
  if (N <= 0 || P <= 0 || H <= 0 || W <= 0 || !(radius > 0.f) || !std::isfinite(radius)) return RECMV_E_SHAPE;
  if ((int64_t)N * H * W > 0x7fffffffLL) return RECMV_E_RANGE;
  if ((int64_t)N * P > 0xffffffffLL) return RECMV_E_RANGE;   // the packed index is the low word of the key
  return RECMV_OK;
}

double pix_radius(float radius, int H, int W) { return (double)radius * (double)(H < W ? H : W) * 0.5; }

unsigned blocks_for(long long work) { return (unsigned)((work + kPtsThreads - 1) / kPtsThreads); }

}  // namespace
}  // namespace recmv

using namespace recmv;

extern "C" int recmv_points_scratch_bytes(int N, int64_t P, int H, int W, size_t* bytes) {
  const int s = check_sizes(N, P, H, W, 1.f);
  if (s) return s;
  if (!bytes) return RECMV_E_NULL;
  carve(nullptr, (long long)N * P, (long long)N * H * W, bytes);
  return RECMV_OK;
}

extern "C" int recmv_points_count(const float* points, int N, int64_t P, const float* cam, const float* R,
                                  const float* T, int NR, int H, int W, float radius, void* scratch, int64_t* total,
                                  recmv_stream_t stream) {
  int s = check_sizes(N, P, H, W, radius);
  if (s) return s;
  if (NR != 1 && NR != N) return RECMV_E_SHAPE;
  if (!points || !cam || !R || !T || !scratch || !total) return RECMV_E_NULL;
  cudaStream_t st = (cudaStream_t)stream;
  const long long np = (long long)N * P, npix = (long long)N * H * W;
  const PtsScratch sc = carve(scratch, np, npix, nullptr);
  const PtsCam c = {cam[0], cam[1], cam[2], cam[3]};
  const double r = pix_radius(radius, H, W);
  cudaError_t e = cudaMemsetAsync(sc.counts, 0, (size_t)npix * sizeof(int), st);
  if (e != cudaSuccess) return (int)e;
  pts_count_kernel<<<blocks_for(np), kPtsThreads, 0, st>>>(points, N, P, R, T, NR, c, H, W, r, r * r, sc.scr, sc.zc,
                                                           sc.counts);
  if ((s = launch_status())) return s;
  const long long nb = scan_tiles(npix);
  pts_scan_reduce_kernel<<<(unsigned)nb, kPtsThreads, 0, st>>>(sc.counts, npix, sc.bsums);
  if ((s = launch_status())) return s;
  pts_scan_tiles_kernel<<<1, kPtsThreads, 0, st>>>(sc.bsums, nb, sc.offs + npix);
  if ((s = launch_status())) return s;
  pts_scan_down_kernel<<<(unsigned)nb, kPtsThreads, 0, st>>>(sc.counts, npix, sc.bsums, sc.offs);
  if ((s = launch_status())) return s;
  long long h = 0;
  e = cudaMemcpyAsync(&h, sc.offs + npix, sizeof(h), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return (int)e;
  *total = h;
  return h > 0x7fffffffLL ? RECMV_E_RANGE : RECMV_OK;
}

extern "C" int recmv_points_render(const float* features, int C, int N, int64_t P, int H, int W, float radius, int K,
                                   void* scratch, void* cand, int64_t total, float* images, recmv_stream_t stream) {
  int s = check_sizes(N, P, H, W, radius);
  if (s) return s;
  if (C < 1 || C > kMaxC || K < 1 || K > kMaxK || total < 0) return RECMV_E_SHAPE;
  if (total > 0x7fffffffLL) return RECMV_E_RANGE;
  if (!features || !scratch || !images || (total > 0 && !cand)) return RECMV_E_NULL;
  cudaStream_t st = (cudaStream_t)stream;
  const long long np = (long long)N * P, npix = (long long)N * H * W;
  const PtsScratch sc = carve(scratch, np, npix, nullptr);
  const double r = pix_radius(radius, H, W);
  unsigned long long* keys = (unsigned long long*)cand;
  if (total > 0) {
    pts_emit_kernel<<<blocks_for(np), kPtsThreads, 0, st>>>(sc.scr, sc.zc, np, P, H, W, r, r * r, sc.counts, sc.offs,
                                                            keys);
    if ((s = launch_status())) return s;
  }
  pts_resolve_kernel<<<stride_grid(npix * 32, kPtsThreads, 8), kPtsThreads, 0, st>>>(
      sc.offs, keys, sc.scr, features, P, C, K, H, W, npix, r * r, images);
  return launch_status();
}

extern "C" int recmv_points_render_backward(const float* points, int N, int64_t P, const float* cam, const float* R,
                                            const float* T, int NR, int H, int W, float radius, const float* features,
                                            int C, int K, void* scratch, const void* cand, const float* grad_images,
                                            float* grad_points, recmv_stream_t stream) {
  int s = check_sizes(N, P, H, W, radius);
  if (s) return s;
  if (NR != 1 && NR != N) return RECMV_E_SHAPE;
  if (C < 1 || C > kMaxC || K < 1 || K > kMaxK) return RECMV_E_SHAPE;
  if (!points || !cam || !R || !T || !features || !scratch || !grad_images || !grad_points) return RECMV_E_NULL;
  cudaStream_t st = (cudaStream_t)stream;
  const long long np = (long long)N * P, npix = (long long)N * H * W;
  const PtsScratch sc = carve(scratch, np, npix, nullptr);
  const PtsCam c = {cam[0], cam[1], cam[2], cam[3]};
  const double r = pix_radius(radius, H, W);
  cudaError_t e = cudaMemsetAsync(sc.gscr, 0, (size_t)np * sizeof(float2), st);
  if (e != cudaSuccess) return (int)e;
  pts_backward_kernel<<<stride_grid(npix * 32, kPtsThreads, 8), kPtsThreads, 0, st>>>(
      sc.offs, (const unsigned long long*)cand, sc.scr, features, grad_images, P, C, K, H, W, npix, r * r, sc.gscr);
  if ((s = launch_status())) return s;
  pts_grad_points_kernel<<<blocks_for(np), kPtsThreads, 0, st>>>(points, N, P, R, T, NR, c, sc.zc, sc.gscr,
                                                                 grad_points);
  return launch_status();
}

extern "C" int recmv_points_fragments(int N, int64_t P, int H, int W, float radius, int K, const void* scratch,
                                      const void* cand, int64_t* idx, float* zbuf, float* dists,
                                      recmv_stream_t stream) {
  int s = check_sizes(N, P, H, W, radius);
  if (s) return s;
  if (K < 1 || K > kMaxK) return RECMV_E_SHAPE;
  const long long n = (long long)N * H * W * K;
  if (n > kMaxThreads) return RECMV_E_RANGE;
  if (!scratch || !idx || !zbuf || !dists) return RECMV_E_NULL;
  const PtsScratch sc = carve((void*)scratch, (long long)N * P, (long long)N * H * W, nullptr);
  const double ndc = 2.0 / (double)(H < W ? H : W);
  pts_fragments_kernel<<<blocks_for(n), kPtsThreads, 0, (cudaStream_t)stream>>>(
      sc.offs, (const unsigned long long*)cand, sc.scr, K, H, W, n, ndc * ndc, (long long*)idx, zbuf, dists);
  return launch_status();
}
