// Image quality measures of an estimate against a reference (RMSE, SRE, SAM, UIQ; dsen2_b200/metrics.py derives them).
//
// Both images are contiguous HWC (H, W, C), 1 <= C <= 16, each float32, float64 or uint16; every value is read exactly as
// float64 and all arithmetic is float64.  With nodata v a pixel is invalid iff every band of the REFERENCE equals v in the
// reference's element type (exact as doubles: float32 and uint16 widen exactly).
//   quality_pixel_kernel: one grid-stride pass over the pixels -> per band E_b = sum (est - ref)^2, S_b = sum ref, the
//                         valid-pixel count and the spectral angle of every valid pixel whose two vectors are non-zero.
//   quality_uiq_kernel:   Wang-Bovik Q of every 8 x 8 window whose 64 pixels are valid.  A CTA owns 32 x 32 window origins
//                         and stages the 39 x 39 footprint of one band of both images (float64) in shared memory; a thread
//                         owns 4 origins of one column and streams the 11 footprint rows they cover through registers, once
//                         for the means (row sums, then rows in order) and once for the centred sums (two passes).
//   quality_final_kernel: one block per output sum adds the per-CTA partials in a fixed order.
// No floating-point atomics anywhere: every partial has its own slot and every sum a fixed order, so the same inputs give
// bit-identical sums on the same device.  The grids depend on H, W and C only.
#include "common.cuh"

namespace dsen2 {

static constexpr int kMaxBands = 16;
static constexpr int kPixThreads = 256;
static constexpr int kPixMaxBlocks = 2048;
static constexpr int kWin = 8;                        // UIQ window
static constexpr int kTile = 32;                      // window origins per CTA side
static constexpr int kRowsPerThread = 4;              // origins of one column per thread
static constexpr int kUiqThreads = kTile * (kTile / kRowsPerThread);   // 256
static constexpr int kFoot = kTile + kWin - 1;        // 39: footprint side
static constexpr int kFinalThreads = 256;

__device__ __forceinline__ double ld_d(const float* p) { return (double)__ldg(p); }
__device__ __forceinline__ double ld_d(const double* p) { return __ldg(p); }
__device__ __forceinline__ double ld_d(const uint16_t* p) { return (double)__ldg(p); }

// Sum of v over the block in a fixed tree (warp butterfly-free shuffle-down, then the warps in order); result in thread 0.
template <int kThreads>
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();                                    // red[] may still be read from the previous call
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
  return s;
}

static inline int pix_blocks(long long npix) {
  const long long b = (npix + kPixThreads * 8 - 1) / (kPixThreads * 8);
  return (int)(b < 1 ? 1 : (b > kPixMaxBlocks ? kPixMaxBlocks : b));
}
static inline long long uiq_tiles(int H, int W) {
  if (H < kWin || W < kWin) return 0;
  return (long long)ceil_div(H - kWin + 1, kTile) * ceil_div(W - kWin + 1, kTile);
}

// partials[block][q]: q = 2c: E_c, 2c + 1: S_c (c < C), then 2C: n, 2C + 1: sum of angles (radians), 2C + 2: SAM pixels
template <typename TE, typename TR>
__global__ void __launch_bounds__(kPixThreads) quality_pixel_kernel(const TE* __restrict__ est, const TR* __restrict__ ref,
                                                                    long long npix, int C, int use_nodata, double v,
                                                                    double* __restrict__ partials) {
  __shared__ double red[kPixThreads / 32];
  double E[kMaxBands], S[kMaxBands];
#pragma unroll
  for (int c = 0; c < kMaxBands; ++c) E[c] = S[c] = 0.0;
  double n = 0.0, ang = 0.0, nsam = 0.0;
  for (long long p = blockIdx.x * (long long)kPixThreads + threadIdx.x; p < npix; p += (long long)gridDim.x * kPixThreads) {
    const TE* e = est + p * C;
    const TR* r = ref + p * C;
    double xr[kMaxBands];
    bool nd = use_nodata != 0;
#pragma unroll
    for (int c = 0; c < kMaxBands; ++c)
      if (c < C) {
        xr[c] = ld_d(r + c);
        nd &= xr[c] == v;
      }
    if (nd) continue;
    n += 1.0;
    double dot = 0.0, ne = 0.0, nr = 0.0;
#pragma unroll
    for (int c = 0; c < kMaxBands; ++c)
      if (c < C) {
        const double xe = ld_d(e + c), d = xe - xr[c];
        E[c] = fma(d, d, E[c]);
        S[c] += xr[c];
        dot = fma(xe, xr[c], dot);
        ne = fma(xe, xe, ne);
        nr = fma(xr[c], xr[c], nr);
      }
    if (ne > 0.0 && nr > 0.0) {
      ang += acos(fmin(fmax(dot / (sqrt(ne) * sqrt(nr)), -1.0), 1.0));
      nsam += 1.0;
    }
  }
  double* out = partials + (long long)blockIdx.x * (2 * C + 3);
#pragma unroll
  for (int c = 0; c < kMaxBands; ++c)
    if (c < C) {
      const double se = block_sum<kPixThreads>(E[c], red);
      if (threadIdx.x == 0) out[2 * c] = se;
      const double ss = block_sum<kPixThreads>(S[c], red);
      if (threadIdx.x == 0) out[2 * c + 1] = ss;
    }
  const double sn = block_sum<kPixThreads>(n, red);
  if (threadIdx.x == 0) out[2 * C] = sn;
  const double sa = block_sum<kPixThreads>(ang, red);
  if (threadIdx.x == 0) out[2 * C + 1] = sa;
  const double sc = block_sum<kPixThreads>(nsam, red);
  if (threadIdx.x == 0) out[2 * C + 2] = sc;
}

// partials[tile][2c]: sum of Q over the used windows of band c, [2c + 1]: their number
template <typename TE, typename TR>
__global__ void __launch_bounds__(kUiqThreads) quality_uiq_kernel(const TE* __restrict__ est, const TR* __restrict__ ref,
                                                                  int H, int W, int C, int use_nodata, double v, int tiles_x,
                                                                  double* __restrict__ partials) {
  __shared__ double xs[kFoot][kFoot + 1];
  __shared__ double ys[kFoot][kFoot + 1];
  __shared__ unsigned char valid[kFoot][kFoot + 1];
  __shared__ double red[kUiqThreads / 32];
  const int tile = blockIdx.x;
  const int oy0 = (tile / tiles_x) * kTile, ox0 = (tile % tiles_x) * kTile;
  const int tx = threadIdx.x % kTile, ty = threadIdx.x / kTile;
  const int ry = ty * kRowsPerThread;                 // first of this thread's origins, tile-relative
  const int fh = min(kFoot, H - oy0), fw = min(kFoot, W - ox0);

  // per-pixel validity of the footprint (every band of ref equal to v -> invalid); outside the image: invalid
  for (int i = threadIdx.x; i < kFoot * kFoot; i += kUiqThreads) {
    const int fy = i / kFoot, fx = i - fy * kFoot;
    bool ok = fy < fh && fx < fw;
    if (ok && use_nodata) {
      const TR* r = ref + ((long long)(oy0 + fy) * W + (ox0 + fx)) * C;
      bool nd = true;
      for (int c = 0; c < C; ++c) nd &= ld_d(r + c) == v;
      ok = !nd;
    }
    valid[fy][fx] = ok;
  }
  __syncthreads();
  // window k of this thread (origin (ry + k, tx)) is used only if its origin lies in the image and its 64 pixels are valid
  unsigned wmask = 0;
  {
    int bad[kRowsPerThread + kWin - 1];
#pragma unroll
    for (int i = 0; i < kRowsPerThread + kWin - 1; ++i) {
      int b = 0;
      const int fy = min(ry + i, kFoot - 1);
#pragma unroll
      for (int j = 0; j < kWin; ++j) b |= !valid[fy][min(tx + j, kFoot - 1)];
      bad[i] = b;
    }
#pragma unroll
    for (int k = 0; k < kRowsPerThread; ++k) {
      int b = 0;
#pragma unroll
      for (int i = 0; i < kWin; ++i) b |= bad[k + i];
      if (!b && oy0 + ry + k <= H - kWin && ox0 + tx <= W - kWin) wmask |= 1u << k;
    }
  }

  double* out = partials + (long long)tile * (2 * C);
  for (int c = 0; c < C; ++c) {
    __syncthreads();                                  // previous band's tiles are no longer read
    for (int i = threadIdx.x; i < kFoot * kFoot; i += kUiqThreads) {
      const int fy = i / kFoot, fx = i - fy * kFoot;
      double a = 0.0, b = 0.0;
      if (fy < fh && fx < fw) {
        const long long off = ((long long)(oy0 + fy) * W + (ox0 + fx)) * C + c;
        a = ld_d(est + off);
        b = ld_d(ref + off);
      }
      xs[fy][fx] = a;
      ys[fy][fx] = b;
    }
    __syncthreads();
    double qsum = 0.0, used = 0.0;
    if (wmask) {
      // pass 1: window sums = row sums (left to right), then rows top to bottom
      double mx[kRowsPerThread], my[kRowsPerThread];
#pragma unroll
      for (int k = 0; k < kRowsPerThread; ++k) mx[k] = my[k] = 0.0;
#pragma unroll 1
      for (int i = 0; i < kRowsPerThread + kWin - 1; ++i) {
        double rx = 0.0, rr = 0.0;
#pragma unroll
        for (int j = 0; j < kWin; ++j) {
          rx += xs[ry + i][tx + j];
          rr += ys[ry + i][tx + j];
        }
#pragma unroll
        for (int k = 0; k < kRowsPerThread; ++k)
          if (i >= k && i < k + kWin) {
            mx[k] += rx;
            my[k] += rr;
          }
      }
#pragma unroll
      for (int k = 0; k < kRowsPerThread; ++k) {
        mx[k] *= 1.0 / 64.0;
        my[k] *= 1.0 / 64.0;
      }
      // pass 2: centred sums
      double sxx[kRowsPerThread], syy[kRowsPerThread], sxy[kRowsPerThread];
#pragma unroll
      for (int k = 0; k < kRowsPerThread; ++k) sxx[k] = syy[k] = sxy[k] = 0.0;
#pragma unroll 1
      for (int i = 0; i < kRowsPerThread + kWin - 1; ++i) {
        double rx[kWin], rr[kWin];
#pragma unroll
        for (int j = 0; j < kWin; ++j) {
          rx[j] = xs[ry + i][tx + j];
          rr[j] = ys[ry + i][tx + j];
        }
#pragma unroll
        for (int k = 0; k < kRowsPerThread; ++k)
          if (i >= k && i < k + kWin) {
#pragma unroll
            for (int j = 0; j < kWin; ++j) {
              const double dx = rx[j] - mx[k], dy = rr[j] - my[k];
              sxx[k] = fma(dx, dx, sxx[k]);
              syy[k] = fma(dy, dy, syy[k]);
              sxy[k] = fma(dx, dy, sxy[k]);
            }
          }
      }
#pragma unroll
      for (int k = 0; k < kRowsPerThread; ++k) {
        const double vx = sxx[k] * (1.0 / 64.0), vy = syy[k] * (1.0 / 64.0), cxy = sxy[k] * (1.0 / 64.0);
        const double den = (vx + vy) * (mx[k] * mx[k] + my[k] * my[k]);
        if ((wmask >> k & 1u) && den != 0.0) {
          qsum += 4.0 * cxy * mx[k] * my[k] / den;
          used += 1.0;
        }
      }
    }
    const double sq = block_sum<kUiqThreads>(qsum, red);
    if (threadIdx.x == 0) out[2 * c] = sq;
    const double su = block_sum<kUiqThreads>(used, red);
    if (threadIdx.x == 0) out[2 * c + 1] = su;
  }
}

// Output slot s of d_sums (band b = s / 5 for s < 5C: E_b, S_b, n, sum Q_b, used_b; then sum of angles, SAM pixels) is the
// sum over `count` partials of src[i * stride + off], i ascending within a thread, threads in a fixed tree.
__global__ void __launch_bounds__(kFinalThreads) quality_final_kernel(const double* __restrict__ pix, int pix_blocks,
                                                                      const double* __restrict__ uiq, long long tiles, int C,
                                                                      double* __restrict__ sums) {
  __shared__ double red[kFinalThreads / 32];
  const int s = blockIdx.x;
  const double* src;
  long long count;
  int stride, off;
  if (s < 5 * C) {
    const int b = s / 5, f = s % 5;
    if (f < 3) {
      src = pix, count = pix_blocks, stride = 2 * C + 3, off = f == 0 ? 2 * b : (f == 1 ? 2 * b + 1 : 2 * C);
    } else {
      src = uiq, count = tiles, stride = 2 * C, off = 2 * b + (f - 3);
    }
  } else {
    src = pix, count = pix_blocks, stride = 2 * C + 3, off = 2 * C + 1 + (s - 5 * C);
  }
  double acc = 0.0;
  for (long long i = threadIdx.x; i < count; i += kFinalThreads) acc += src[i * stride + off];
  const double t = block_sum<kFinalThreads>(acc, red);
  if (threadIdx.x == 0) sums[s] = t;
}

template <typename TE, typename TR>
static int launch_quality(const void* d_est, const void* d_ref, int H, int W, int C, int use_nodata, double v, double* pix,
                          int nb, double* uiq, long long tiles, cudaStream_t st) {
  const TE* e = static_cast<const TE*>(d_est);
  const TR* r = static_cast<const TR*>(d_ref);
  quality_pixel_kernel<TE, TR><<<nb, kPixThreads, 0, st>>>(e, r, (long long)H * W, C, use_nodata, v, pix);
  int rc = check_launch("quality_pixel_kernel");
  if (rc || tiles == 0) return rc;
  quality_uiq_kernel<TE, TR><<<(unsigned)tiles, kUiqThreads, 0, st>>>(e, r, H, W, C, use_nodata, v,
                                                                      ceil_div(W - kWin + 1, kTile), uiq);
  return check_launch("quality_uiq_kernel");
}

template <typename TE>
static int dispatch_ref(int ref_dtype, const void* d_est, const void* d_ref, int H, int W, int C, int use_nodata, double v,
                        double* pix, int nb, double* uiq, long long tiles, cudaStream_t st) {
  switch (ref_dtype) {
    case DSEN2_IMG_F32: return launch_quality<TE, float>(d_est, d_ref, H, W, C, use_nodata, v, pix, nb, uiq, tiles, st);
    case DSEN2_IMG_U16: return launch_quality<TE, uint16_t>(d_est, d_ref, H, W, C, use_nodata, v, pix, nb, uiq, tiles, st);
    default: return launch_quality<TE, double>(d_est, d_ref, H, W, C, use_nodata, v, pix, nb, uiq, tiles, st);
  }
}

}  // namespace dsen2

using namespace dsen2;

static size_t quality_workspace(int H, int W, int C) {
  const long long npix = (long long)H * W;
  return ((size_t)pix_blocks(npix) * (2 * C + 3) + (size_t)uiq_tiles(H, W) * (2 * C)) * sizeof(double);
}

extern "C" size_t dsen2_image_quality_workspace_bytes(int H, int W, int C) {
  if (H < 1 || W < 1 || C < 1 || C > kMaxBands) return 0;
  return quality_workspace(H, W, C);
}

extern "C" int dsen2_image_quality(const void* d_est, int est_dtype, const void* d_ref, int ref_dtype, int H, int W, int C,
                                   int use_nodata, float nodata, void* d_workspace, size_t workspace_bytes, double* d_sums,
                                   void* stream) {
  static const char* name = "dsen2_image_quality";
  DSEN2_REQUIRE(d_est && d_ref && d_workspace && d_sums, DSEN2_E_BADARG, "%s: null pointer", name);
  DSEN2_REQUIRE(H >= 1 && W >= 1, DSEN2_E_BADARG, "%s: size %dx%d", name, H, W);
  DSEN2_REQUIRE(C >= 1 && C <= kMaxBands, DSEN2_E_BADARG, "%s: C = %d outside 1..%d", name, C, kMaxBands);
  const auto known = [](int t) { return t == DSEN2_IMG_F32 || t == DSEN2_IMG_U16 || t == DSEN2_IMG_F64; };
  DSEN2_REQUIRE(known(est_dtype) && known(ref_dtype), DSEN2_E_BADARG,
                "%s: dtypes must be DSEN2_IMG_F32, DSEN2_IMG_U16 or DSEN2_IMG_F64 (got %d, %d)", name, est_dtype, ref_dtype);
  DSEN2_REQUIRE(!use_nodata || nodata == nodata, DSEN2_E_BADARG, "%s: nodata is NaN", name);
  DSEN2_REQUIRE(!use_nodata || ref_dtype != DSEN2_IMG_U16 ||
                    (nodata >= 0.f && nodata <= 65535.f && nodata == (float)(int)nodata),
                DSEN2_E_BADARG, "%s: nodata %g is not a uint16 value", name, (double)nodata);
  const size_t need = quality_workspace(H, W, C);
  DSEN2_REQUIRE(workspace_bytes >= need, DSEN2_E_BADARG, "%s: workspace of %zu bytes, %zu needed", name, workspace_bytes,
                need);
  const int nb = pix_blocks((long long)H * W);
  const long long tiles = uiq_tiles(H, W);
  double* pix = static_cast<double*>(d_workspace);
  double* uiq = pix + (size_t)nb * (2 * C + 3);
  const cudaStream_t st = (cudaStream_t)stream;
  const int un = use_nodata ? 1 : 0;
  const double v = (double)nodata;
  int rc;
  switch (est_dtype) {
    case DSEN2_IMG_F32: rc = dispatch_ref<float>(ref_dtype, d_est, d_ref, H, W, C, un, v, pix, nb, uiq, tiles, st); break;
    case DSEN2_IMG_U16: rc = dispatch_ref<uint16_t>(ref_dtype, d_est, d_ref, H, W, C, un, v, pix, nb, uiq, tiles, st); break;
    default: rc = dispatch_ref<double>(ref_dtype, d_est, d_ref, H, W, C, un, v, pix, nb, uiq, tiles, st); break;
  }
  if (rc) return rc;
  quality_final_kernel<<<5 * C + 2, kFinalThreads, 0, st>>>(pix, nb, uiq, tiles, C, d_sums);
  return check_launch("quality_final_kernel");
}
