// HBM-bound kernels of the DSen2 path: patch extraction, bilinear / bicubic upsampling, stitching,
// operand packing.  All are pure gathers with coalesced stores; grids are sized in multiples of the
// SM count and grid-stride over the work.
#include <stdarg.h>

#include "common.cuh"
#include "tiling.cuh"

namespace dsen2 {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ------------------------------------------------------------------------------------------ //
// extract: one thread per output pixel, all C bands (HWC gather -> C coalesced plane stores)
// ------------------------------------------------------------------------------------------ //
template <int C>
__global__ void extract_patches_kernel(const float* __restrict__ img, int H, int W, int ratio, int p, int b,
                                       Tiling tl, int first_patch, long long total, float divisor,
                                       float* __restrict__ out) {
  const long long pp = (long long)p * p;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int local = (int)(idx / pp);
    const int rem = (int)(idx - (long long)local * pp);
    const int y = rem / p, x = rem - y * p;
    const int patch = first_patch + local;
    float v[C];
    if (patch < tl.n_i * tl.n_j) {
      const int ti = patch / tl.n_j, tj = patch - ti * tl.n_j;
      const int si = (ti < tl.k_i ? ti * tl.stride : tl.last_i) * ratio;
      const int sj = (tj < tl.k_j ? tj * tl.stride : tl.last_j) * ratio;
      const int sy = sym_index(si + y - b, H);
      const int sx = sym_index(sj + x - b, W);
      const float* src = img + ((long long)sy * W + sx) * C;
      if (C == 4) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(src));
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3 % C] = q.w;
      } else if (C % 2 == 0) {
#pragma unroll
        for (int c = 0; c < C; c += 2) {
          const float2 q = __ldg(reinterpret_cast<const float2*>(src + c));
          v[c] = q.x; v[(c + 1) % C] = q.y;
        }
      } else {
#pragma unroll
        for (int c = 0; c < C; ++c) v[c] = __ldg(src + c);
      }
    } else {
#pragma unroll
      for (int c = 0; c < C; ++c) v[c] = 0.f;
    }
    float* dst = out + (long long)local * C * pp + rem;
#pragma unroll
    for (int c = 0; c < C; ++c) dst[c * pp] = (divisor == 1.0f) ? v[c] : __fdiv_rn(v[c], divisor);
  }
}

__global__ void extract_patches_generic_kernel(const float* __restrict__ img, int H, int W, int C, int ratio, int p,
                                               int b, Tiling tl, int first_patch, long long total, float divisor,
                                               float* __restrict__ out) {
  const long long pp = (long long)p * p;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int local = (int)(idx / pp);
    const int rem = (int)(idx - (long long)local * pp);
    const int y = rem / p, x = rem - y * p;
    const int patch = first_patch + local;
    float* dst = out + (long long)local * C * pp + rem;
    if (patch < tl.n_i * tl.n_j) {
      const int ti = patch / tl.n_j, tj = patch - ti * tl.n_j;
      const int si = (ti < tl.k_i ? ti * tl.stride : tl.last_i) * ratio;
      const int sj = (tj < tl.k_j ? tj * tl.stride : tl.last_j) * ratio;
      const float* src = img + ((long long)sym_index(si + y - b, H) * W + sym_index(sj + x - b, W)) * C;
      for (int c = 0; c < C; ++c) {
        const float v = __ldg(src + c);
        dst[c * pp] = (divisor == 1.0f) ? v : __fdiv_rn(v, divisor);
      }
    } else {
      for (int c = 0; c < C; ++c) dst[c * pp] = 0.f;
    }
  }
}

// ------------------------------------------------------------------------------------------ //
// bilinear, mirror boundary, integer scale s (patches.py:11-16): u = (o + .5)/s - .5
// ------------------------------------------------------------------------------------------ //
// a * (1 - f) + b * f as every bilinear kernel here (and prep_gather) evaluates it: the first product fused into the sum,
// the second rounded.  Spelled out so that the compiler cannot contract the expression differently in each kernel: the
// kernels below must give the same bits for the same plane.
__device__ __forceinline__ float lerp_rn(float a, float b, float f) { return __fmaf_rn(a, 1.0f - f, __fmul_rn(b, f)); }

__global__ void bilinear_mirror_kernel(const float* __restrict__ in, int p, int s, long long total, float post_div,
                                       float* __restrict__ out) {
  const int P = p * s;
  const long long PP = (long long)P * P;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long plane = idx / PP;
    const int rem = (int)(idx - plane * PP);
    const int oy = rem / P, ox = rem - oy * P;
    int y0, y1, x0, x1;
    float fy, fx;
    bilin_tap(oy, s, p, y0, y1, fy);
    bilin_tap(ox, s, p, x0, x1, fx);
    if (p == 1) y0 = x0 = 0;                 // bilin_tap mirrors the tap -1 to 1, which a one-pixel plane does not have
    const float* src = in + plane * (long long)p * p;
    const float k = 30000.0f;                // the reference scales by 1/30000 around the resize
    const float v00 = __fdiv_rn(__ldg(src + y0 * p + x0), k), v01 = __fdiv_rn(__ldg(src + y0 * p + x1), k);
    const float v10 = __fdiv_rn(__ldg(src + y1 * p + x0), k), v11 = __fdiv_rn(__ldg(src + y1 * p + x1), k);
    const float c0 = lerp_rn(v00, v10, fy);  // rows first, then columns (as the oracle)
    const float c1 = lerp_rn(v01, v11, fy);
    const float r = __fmul_rn(lerp_rn(c0, c1, fx), k);
    out[idx] = (post_div == 1.0f) ? r : __fdiv_rn(r, post_div);
  }
}

// Row-band form of the same arithmetic: a block owns kBilRows input rows of one plane (+ one mirrored halo row / column
// on each side), divides every input value by 30000 ONCE into shared memory (the direct kernel does it four times per
// output) and produces the s * kBilRows output rows from there.  A thread owns FOUR consecutive output columns (their x
// taps are computed once, the row is written with 16-byte stores; blockDim.x = P / 4) and walks the band's output rows.
// Same operations per output as bilinear_mirror_kernel (lerp_rn) => same bits.
constexpr int kBilRows = 16, kBilThreads = 256, kBilMaxP = 1024;

__device__ __forceinline__ int mirror_index(int g, int n) {
  if (g < 0) g = -g;
  if (g > n - 1) g = 2 * (n - 1) - g;
  return g < 0 ? 0 : g;
}

// u = (o + .5)/s - .5 = t / (2 s) with t = 2 o + 1 - s: integer part (floor) and fraction.  SC > 0: compile-time scale
// (the divisions become multiplications); SC == 0: run-time scale.
template <int SC>
__device__ __forceinline__ void bilin_split(int o, int s, int& i0, float& f) {
  const int d = 2 * (SC > 0 ? SC : s);
  const int t = 2 * o + 1 - (SC > 0 ? SC : s);
  i0 = (t >= 0) ? t / d : -((-t + d - 1) / d);
  f = (float)(t - i0 * d) / (float)d;
}

template <int SC>
__global__ void __launch_bounds__(kBilThreads) bilinear_mirror_band_kernel(const float* __restrict__ in, int p, int s, int bands,
                                                                          float post_div, float* __restrict__ out) {
  extern __shared__ float s_src[];                         // [kBilRows + 2][p + 2], value / 30000
  const int plane = blockIdx.x / bands, band = blockIdx.x - plane * bands;
  const int r0 = band * kBilRows, rows = min(kBilRows, p - r0);
  const int pitch = p + 2, P = p * s;
  const float k = 30000.0f;                                // the reference scales by 1/30000 around the resize
  const float* src = in + (long long)plane * p * p;
  for (int lr = threadIdx.y; lr < rows + 2; lr += blockDim.y) {
    const float* srow = src + mirror_index(r0 - 1 + lr, p) * p;
    for (int lc = threadIdx.x; lc < pitch; lc += blockDim.x)
      s_src[lr * pitch + lc] = __fdiv_rn(__ldg(srow + mirror_index(lc - 1, p)), k);
  }
  // x taps of this thread's four output columns: local column of the left tap and the fraction
  int xl[4];
  float fx[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    int i0;
    bilin_split<SC>(threadIdx.x * 4 + j, s, i0, fx[j]);
    xl[j] = i0 + 1;
  }
  __syncthreads();
  float* dst = out + (long long)plane * P * P + threadIdx.x * 4;
  for (int oyl = threadIdx.y; oyl < rows * s; oyl += blockDim.y) {
    const int oy = r0 * s + oyl;
    int i0;
    float fy;
    bilin_split<SC>(oy, s, i0, fy);
    const float* row0 = s_src + (i0 - (r0 - 1)) * pitch;
    const float* row1 = row0 + pitch;
    float r[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float v00 = row0[xl[j]], v01 = row0[xl[j] + 1], v10 = row1[xl[j]], v11 = row1[xl[j] + 1];
      const float c0 = lerp_rn(v00, v10, fy);          // rows first, then columns (as the oracle)
      const float c1 = lerp_rn(v01, v11, fy);
      const float v = __fmul_rn(lerp_rn(c0, c1, fx[j]), k);
      r[j] = (post_div == 1.0f) ? v : __fdiv_rn(v, post_div);
    }
    *reinterpret_cast<float4*>(dst + (long long)oy * P) = make_float4(r[0], r[1], r[2], r[3]);
  }
}

// The DSen2_20 shape (20 m patches of 64 x 64 -> 128 x 128, supres.py:27): fractions are 1/4 and 3/4, a warp is one source
// row (lane t = columns 2t, 2t+1; the neighbours 2t-1 and 2t+2 come from the adjacent lanes), and it walks down a band of
// 16 source rows with the previous row in registers: one 8-byte load and two shuffles per lane and source row, no shared
// memory, ~6 instructions per output instead of ~17.  Same float32 expressions as the band kernel above.
__global__ void __launch_bounds__(256) bilinear_mirror_x2_p64_kernel(const float* __restrict__ in, long long planes,
                                                                     float post_div, float* __restrict__ out) {
  const long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  const long long plane = w >> 2;
  if (plane >= planes) return;
  const int r0 = (int)(w & 3) * 16;
  const float* src = in + plane * 4096;
  float* dst = out + plane * 16384 + lane * 4;
  const float k = 30000.0f;
  float top[4], bot[4];
  auto load_row = [&](int r, float (&v)[4]) {   // columns 2t-1 .. 2t+2 of source row r (mirrored), / 30000
    const float2 a = __ldg(reinterpret_cast<const float2*>(src + mirror_index(r, 64) * 64) + lane);
    const float a0 = __fdiv_rn(a.x, k), a1 = __fdiv_rn(a.y, k);
    const float l = __shfl_up_sync(0xffffffffu, a1, 1), r2 = __shfl_down_sync(0xffffffffu, a0, 1);
    v[0] = lane == 0 ? a1 : l;                  // column -1 mirrors to column 1
    v[1] = a0;
    v[2] = a1;
    v[3] = lane == 31 ? a0 : r2;                // column 64 mirrors to column 62
  };
  load_row(r0 - 1, top);
#pragma unroll 2
  for (int r = r0 - 1; r < r0 + 16; ++r) {      // source rows (r, r+1) -> output rows 2r+1 (fy = 1/4) and 2r+2 (fy = 3/4)
    load_row(r + 1, bot);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int oy = 2 * r + 1 + h;
      if (oy < 2 * r0 || oy >= 2 * r0 + 32) continue;      // the neighbouring band's row
      const float fy = h ? 0.75f : 0.25f;
      float c[4], o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) c[j] = lerp_rn(top[j], bot[j], fy);      // rows first, then columns
      o[0] = __fmul_rn(lerp_rn(c[0], c[1], 0.75f), k);
      o[1] = __fmul_rn(lerp_rn(c[1], c[2], 0.25f), k);
      o[2] = __fmul_rn(lerp_rn(c[1], c[2], 0.75f), k);
      o[3] = __fmul_rn(lerp_rn(c[2], c[3], 0.25f), k);
      if (post_div != 1.0f) {
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = __fdiv_rn(o[j], post_div);
      }
      *reinterpret_cast<float4*>(dst + oy * 128) = make_float4(o[0], o[1], o[2], o[3]);
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) top[j] = bot[j];
  }
}

// ------------------------------------------------------------------------------------------ //
// stitch (patches.py:374-405): patch t writes the output pixels whose LAST writer it is
// ------------------------------------------------------------------------------------------ //
// generic form: thread per (patch, interior pixel), writes the C contiguous HWC floats it owns
__global__ void recompose_kernel(const float* __restrict__ pred, int first_patch, int C, int P, int border, int H,
                                 int W, int ny, int nx, float mul, long long total, float* __restrict__ out) {
  const int S = P - 2 * border;
  const long long SS = (long long)S * S, PP = (long long)P * P;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int local = (int)(idx / SS);
    const int rem = (int)(idx - (long long)local * SS);
    const int yy = rem / S, xx = rem - yy * S;
    const int patch = first_patch + local;
    if (patch >= ny * nx) continue;
    const int ty = patch / nx, tx = patch - ty * nx;
    const int oy = min(ty * S, H - S), ox = min(tx * S, W - S);
    const int y = oy + yy, x = ox + xx;
    if (tile_of(y, H, S, ny) != ty || tile_of(x, W, S, nx) != tx) continue;   // a later patch overwrites it
    const float* src = pred + (long long)local * C * PP + (long long)(border + yy) * P + (border + xx);
    float* dst = out + ((long long)y * W + x) * C;
    for (int c = 0; c < C; ++c) dst[c] = __ldg(src + c * PP) * mul;
  }
}

// vector form (C = 2 or 6, S and border multiples of 4, even W): a thread owns FOUR consecutive interior pixels of one
// patch row -- C 16-byte plane loads in flight, then its 4 * C HWC floats (16 * C contiguous bytes) as 16-byte stores
template <int C>
__global__ void __launch_bounds__(256) recompose_vec4_kernel(const float* __restrict__ pred, int first_patch, int P, int border,
                                                             int H, int W, int ny, int nx, float mul, long long total,
                                                             float* __restrict__ out) {
  const int S = P - 2 * border, S4 = S / 4;
  const long long PP = (long long)P * P;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long row = idx / S4;
    const int xx = (int)(idx - row * S4) * 4;
    const int local = (int)(row / S), yy = (int)(row - (long long)local * S);
    const int patch = first_patch + local;
    if (patch >= ny * nx) continue;
    const int ty = patch / nx, tx = patch - ty * nx;
    const int oy = min(ty * S, H - S), ox = min(tx * S, W - S);
    const int y = oy + yy, x = ox + xx;
    if (tile_of(y, H, S, ny) != ty) continue;
    const bool o0 = tile_of(x, W, S, nx) == tx, o3 = tile_of(x + 3, W, S, nx) == tx;   // ownership is a contiguous run
    if (!o0 && !o3) continue;
    const float* src = pred + (long long)local * C * PP + (long long)(border + yy) * P + (border + xx);
    float4 v[C];
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = __ldg(reinterpret_cast<const float4*>(src + c * PP));
    float o[4 * C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
      o[0 * C + c] = v[c].x * mul; o[1 * C + c] = v[c].y * mul; o[2 * C + c] = v[c].z * mul; o[3 * C + c] = v[c].w * mul;
    }
    float* dst = out + ((long long)y * W + x) * C;
    if (o0 && o3) {
#pragma unroll
      for (int q = 0; q < C; ++q) reinterpret_cast<float4*>(dst)[q] = make_float4(o[4 * q], o[4 * q + 1], o[4 * q + 2], o[4 * q + 3]);
    } else {                                               // the seam of the clamped last tile column
      for (int i = 0; i < 4; ++i)
        if (tile_of(x + i, W, S, nx) == tx)
          for (int c = 0; c < C; ++c) dst[i * C + c] = o[i * C + c];
    }
  }
}

// ------------------------------------------------------------------------------------------ //
// MATLAB bicubic (imresize.py:50-74): float64 products, left-to-right sums, no FMA contraction
// ------------------------------------------------------------------------------------------ //
template <typename TIn>
__global__ void bicubic_kernel(const TIn* __restrict__ in, int h, int w, int C, const double* __restrict__ wy,
                               const int32_t* __restrict__ iy, int ty, int out_h, const double* __restrict__ wx,
                               const int32_t* __restrict__ ix, int tx, int out_w, int first_dim, long long total,
                               double* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    const long long pix = idx / C;
    const int ox = (int)(pix % out_w), oy = (int)(pix / out_w);
    double acc = 0.0;
    if (first_dim == 0) {  // rows first: inter[oy, col] then along x
      for (int b = 0; b < tx; ++b) {
        const int col = ix[ox * tx + b];
        double inter = 0.0;
        for (int a = 0; a < ty; ++a) {
          const double v = (double)in[((long long)iy[oy * ty + a] * w + col) * C + c];
          const double pr = __dmul_rn(v, wy[oy * ty + a]);
          inter = (a == 0) ? pr : __dadd_rn(inter, pr);
        }
        const double pr = __dmul_rn(inter, wx[ox * tx + b]);
        acc = (b == 0) ? pr : __dadd_rn(acc, pr);
      }
    } else {               // columns first
      for (int a = 0; a < ty; ++a) {
        const int row = iy[oy * ty + a];
        double inter = 0.0;
        for (int b = 0; b < tx; ++b) {
          const double v = (double)in[((long long)row * w + ix[ox * tx + b]) * C + c];
          const double pr = __dmul_rn(v, wx[ox * tx + b]);
          inter = (b == 0) ? pr : __dadd_rn(inter, pr);
        }
        const double pr = __dmul_rn(inter, wy[oy * ty + a]);
        acc = (a == 0) ? pr : __dadd_rn(acc, pr);
      }
    }
    out[idx] = acc;
  }
}

// Tiled two-pass form of the same arithmetic (what resizeAlongDim does: dim `first` completely, then the other):
// a block owns a TR x TC tile of output pixels, computes the first-pass intermediate it needs ONCE into shared
// memory (float64, the values the reference stores in its intermediate array) and combines it along the second
// dimension.  Per output 4 + ~2.4 products instead of 20, four + ~2.4 global loads instead of 16, 32-bit index
// arithmetic, stores contiguous over (x, c).  Products and left-to-right sums are the same operations in the same
// order as bicubic_kernel, so the result is bit-identical.  Falls back to the direct form for a tile whose
// first-pass footprint exceeds the buffer (strong down-scaling).
constexpr int kBicTR = 16;                                // output rows per tile (columns and the intermediate extent follow C)
constexpr int kBicMaxTaps = 8;                            // taps per dimension the tiled path keeps in registers / smem

// TAPS > 0: both dimensions have exactly TAPS taps (4 for every up-scaling factor: imresize.py:35-47 trims the six
// candidates to the non-zero columns) -- the tap loops are fully unrolled without predicates; TAPS == 0: run-time counts.
template <typename TIn, bool FIRST0, int TAPS>
__global__ void __launch_bounds__(256) bicubic_tiled_kernel(const TIn* __restrict__ in, int h, int w, int C,
                                                            const double* __restrict__ wy, const int32_t* __restrict__ iy,
                                                            int ty, int out_h, const double* __restrict__ wx,
                                                            const int32_t* __restrict__ ix, int tx, int out_w,
                                                            int kBicTC, int kBicSpan, double* __restrict__ out) {
  extern __shared__ double s_inter[];                      // FIRST0: [TR][span][C]   else: [span][TC][C]
  __shared__ int s_lo, s_hi, s_ylo, s_yhi;
  __shared__ double s_wy[kBicTR * kBicMaxTaps];            // y taps of the tile's rows (uniform across a row's threads)
  __shared__ int s_iy[kBicTR * kBicMaxTaps];
  const int ox0 = blockIdx.x * kBicTC, oy0 = blockIdx.y * kBicTR;
  const int tc = min(kBicTC, out_w - ox0), tr = min(kBicTR, out_h - oy0);
  if (threadIdx.x == 0) { s_lo = 0x7fffffff; s_hi = -1; s_ylo = 0x7fffffff; s_yhi = -1; }
  __syncthreads();
  // footprint of the SECOND-pass taps along the dimension the intermediate keeps at input resolution
  {
    const int32_t* idx2 = FIRST0 ? ix + (long long)ox0 * tx : iy + (long long)oy0 * ty;
    const int cnt = FIRST0 ? tc * tx : tr * ty;
    int lo = 0x7fffffff, hi = -1;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
      const int v = idx2[i];
      lo = min(lo, v); hi = max(hi, v);
    }
    if (hi >= 0) { atomicMin(&s_lo, lo); atomicMax(&s_hi, hi); }
  }
  constexpr int NT = TAPS > 0 ? TAPS : kBicMaxTaps;          // unrolled tap-loop length
  if (TAPS > 0) { ty = TAPS; tx = TAPS; }                        // compile-time counts from here on
  const bool taps_fit = ty <= kBicMaxTaps && tx <= kBicMaxTaps;
  if (taps_fit) {
    int ylo = 0x7fffffff, yhi = -1;
    for (int i = threadIdx.x; i < tr * ty; i += blockDim.x) {
      s_wy[i] = wy[(long long)oy0 * ty + i];
      const int v = iy[(long long)oy0 * ty + i];
      s_iy[i] = v;
      ylo = min(ylo, v); yhi = max(yhi, v);
    }
    if (FIRST0 && yhi >= 0) { atomicMin(&s_ylo, ylo); atomicMax(&s_yhi, yhi); }
  }
  __syncthreads();
  const int lo = s_lo, span = s_hi - s_lo + 1;
  if (span <= kBicSpan && taps_fit) {
    const int rowc = tc * C;                               // (x, c) pairs of an output row of the tile
    if (FIRST0) {
      // pass 1 along y: inter[r][col][c] = sum_a in[iy[oy][a]][lo + col][c] * wy[oy][a]; a thread keeps its (col, c)
      const int colc = span * C;
      const long long wc = (long long)w * C;
      // row offsets of the y taps relative to the tile's first input row, in ELEMENTS and 32 bits (a 64-bit product per tap was
      // half of the first pass's instructions); tables whose tile footprint would overflow that keep the 64-bit form
      const int ylo = s_ylo;
      if ((long long)(s_yhi - ylo) * wc < (1LL << 30)) {
        for (int i = threadIdx.x; i < tr * ty; i += blockDim.x) s_iy[i] = (s_iy[i] - ylo) * (int)wc;
        __syncthreads();
        int r = threadIdx.x / colc, cc = threadIdx.x - r * colc;
        const int dr = blockDim.x / colc, dc = blockDim.x - dr * colc;
        const TIn* base0 = in + ((long long)ylo * w + lo) * C;
        for (int i = threadIdx.x; i < tr * colc; i += blockDim.x) {
          const TIn* base = base0 + cc;
          double inter = 0.0;
#pragma unroll
          for (int a = 0; a < NT; ++a)
            if (TAPS > 0 || a < ty) {
              const double pr = __dmul_rn((double)base[s_iy[r * ty + a]], s_wy[r * ty + a]);
              inter = (a == 0) ? pr : __dadd_rn(inter, pr);
            }
          s_inter[i] = inter;
          r += dr;
          cc += dc;
          if (cc >= colc) { cc -= colc; ++r; }
        }
      } else {
        // flattened over (row, column-channel) so that all threads stay busy; (r, cc) advance incrementally -- a division
        // by the run-time extent per item was a fifth of this issue-bound kernel's instructions
        int r = threadIdx.x / colc, cc = threadIdx.x - r * colc;
        const int dr = blockDim.x / colc, dc = blockDim.x - dr * colc;
        const TIn* base0 = in + (long long)lo * C;
        for (int i = threadIdx.x; i < tr * colc; i += blockDim.x) {
          const TIn* base = base0 + cc;
          double inter = 0.0;
#pragma unroll
          for (int a = 0; a < NT; ++a)
            if (TAPS > 0 || a < ty) {
              const double pr = __dmul_rn((double)base[s_iy[r * ty + a] * wc], s_wy[r * ty + a]);
              inter = (a == 0) ? pr : __dadd_rn(inter, pr);
            }
          s_inter[i] = inter;
          r += dr;
          cc += dc;
          if (cc >= colc) { cc -= colc; ++r; }
        }
      }
      __syncthreads();
      // pass 2 along x: a thread keeps its (x, c) and the x taps, walks the tile's rows
      for (int xc = threadIdx.x; xc < rowc; xc += blockDim.x) {
        const int x = xc / C, c = xc - x * C;
        int off[NT];
        double wgt[NT];
#pragma unroll
        for (int b = 0; b < NT; ++b)
          if (TAPS > 0 || b < tx) {
            off[b] = (ix[(ox0 + x) * tx + b] - lo) * C + c;
            wgt[b] = wx[(ox0 + x) * tx + b];
          }
        double* dst = out + ((long long)oy0 * out_w + ox0) * C + xc;
        for (int r = 0; r < tr; ++r) {
          double acc = 0.0;
#pragma unroll
          for (int b = 0; b < NT; ++b)
            if (TAPS > 0 || b < tx) {
              const double pr = __dmul_rn(s_inter[r * colc + off[b]], wgt[b]);
              acc = (b == 0) ? pr : __dadd_rn(acc, pr);
            }
          dst[(long long)r * out_w * C] = acc;
        }
      }
    } else {
      // pass 1 along x: inter[row][x][c] = sum_b in[lo + row][ix[ox][b]][c] * wx[ox][b]; a thread keeps (x, c) and the x taps
      for (int xc = threadIdx.x; xc < rowc; xc += blockDim.x) {
        const int x = xc / C, c = xc - x * C;
        int off[NT];
        double wgt[NT];
#pragma unroll
        for (int b = 0; b < NT; ++b)
          if (TAPS > 0 || b < tx) {
            off[b] = ix[(ox0 + x) * tx + b] * C + c;
            wgt[b] = wx[(ox0 + x) * tx + b];
          }
        for (int row = 0; row < span; ++row) {
          const TIn* base = in + (long long)(lo + row) * w * C;
          double inter = 0.0;
#pragma unroll
          for (int b = 0; b < NT; ++b)
            if (TAPS > 0 || b < tx) {
              const double pr = __dmul_rn((double)base[off[b]], wgt[b]);
              inter = (b == 0) ? pr : __dadd_rn(inter, pr);
            }
          s_inter[row * rowc + xc] = inter;
        }
      }
      __syncthreads();
      // pass 2 along y
      for (int xc = threadIdx.x; xc < rowc; xc += blockDim.x) {
        double* dst = out + ((long long)oy0 * out_w + ox0) * C + xc;
        for (int r = 0; r < tr; ++r) {
          double acc = 0.0;
#pragma unroll
          for (int a = 0; a < NT; ++a)
            if (TAPS > 0 || a < ty) {
              const double pr = __dmul_rn(s_inter[(s_iy[r * ty + a] - lo) * rowc + xc], s_wy[r * ty + a]);
              acc = (a == 0) ? pr : __dadd_rn(acc, pr);
            }
          dst[(long long)r * out_w * C] = acc;
        }
      }
    }
    return;
  }
  // direct form (same operations as bicubic_kernel)
  const int outs = tr * tc * C;
  for (int i = threadIdx.x; i < outs; i += blockDim.x) {
    const int r = i / (tc * C), xc = i - r * (tc * C);
    const int x = xc / C, c = xc - x * C;
    const int oy = oy0 + r, ox = ox0 + x;
    double acc = 0.0;
    if (FIRST0) {
      for (int b = 0; b < tx; ++b) {
        const int col = ix[ox * tx + b];
        double inter = 0.0;
        for (int a = 0; a < ty; ++a) {
          const double pr = __dmul_rn((double)in[((long long)iy[oy * ty + a] * w + col) * C + c], wy[oy * ty + a]);
          inter = (a == 0) ? pr : __dadd_rn(inter, pr);
        }
        const double pr = __dmul_rn(inter, wx[ox * tx + b]);
        acc = (b == 0) ? pr : __dadd_rn(acc, pr);
      }
    } else {
      for (int a = 0; a < ty; ++a) {
        const int row = iy[oy * ty + a];
        double inter = 0.0;
        for (int b = 0; b < tx; ++b) {
          const double pr = __dmul_rn((double)in[((long long)row * w + ix[ox * tx + b]) * C + c], wx[ox * tx + b]);
          inter = (b == 0) ? pr : __dadd_rn(inter, pr);
        }
        const double pr = __dmul_rn(inter, wy[oy * ty + a]);
        acc = (a == 0) ? pr : __dadd_rn(acc, pr);
      }
    }
    out[((long long)oy * out_w + ox0) * C + xc] = acc;
  }
}

// ------------------------------------------------------------------------------------------ //
// downPixelAggr (patches.py:353-371): scipy gaussian_filter(sigma = 1/s) per band, then s x s block mean.
// scipy filters axis 0 then axis 1 in double precision, storing each pass in the array dtype (float32 here), with
// 'reflect' (= numpy 'symmetric') boundaries and the symmetric-kernel summation order of correlate1d.
// ------------------------------------------------------------------------------------------ //
__device__ __forceinline__ double gauss_line(const float* __restrict__ base, long long stride, int pos, int n, const double* w,
                                             int radius) {
  double acc = __dmul_rn((double)base[(long long)pos * stride], w[radius]);
  for (int i = 1; i <= radius; ++i) {
    const double pair = __dadd_rn((double)base[(long long)sym_index(pos - i, n) * stride],
                                  (double)base[(long long)sym_index(pos + i, n) * stride]);
    acc = __dadd_rn(acc, __dmul_rn(pair, w[radius - i]));
  }
  return acc;
}

// integer_input: the image holds integers (the uint16 digital numbers GDAL hands create_patches.py) -- scipy then stores each
// pass in THAT dtype, i.e. truncates the float64 result towards zero (C cast); the truncated values are exact in float32.
__global__ void gauss_rows_kernel(const float* __restrict__ img, int H, int W, int C, const double* __restrict__ w, int radius,
                                  int integer_input, long long total, float* __restrict__ tmp) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long col = idx % ((long long)W * C);               // (x, c) flattened: contiguous across threads
    const int y = (int)(idx / ((long long)W * C));
    const double v = gauss_line(img + col, (long long)W * C, y, H, w, radius);
    tmp[idx] = integer_input ? (float)trunc(v) : (float)v;
  }
}

__global__ void gauss_cols_mean_kernel(const float* __restrict__ tmp, int H, int W, int C, const double* __restrict__ w,
                                       int radius, int s, int integer_input, long long total, double* __restrict__ out) {
  const int ow = W / s;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % C);
    const int ox = (int)((idx / C) % ow);
    const int oy = (int)(idx / ((long long)C * ow));
    double sum = 0.0;
    for (int dy = 0; dy < s; ++dy) {
      const float* row = tmp + ((long long)(oy * s + dy) * W) * C + c;
      for (int dx = 0; dx < s; ++dx) {
        const double v = gauss_line(row, C, ox * s + dx, W, w, radius);
        const float blurred = integer_input ? (float)trunc(v) : (float)v;              // second pass, stored in the image dtype
        sum = (dy == 0 && dx == 0) ? (double)blurred : __dadd_rn(sum, (double)blurred);
      }
    }
    out[idx] = __ddiv_rn(sum, (double)(s * s));
  }
}

// ------------------------------------------------------------------------------------------ //
// operand packing for the tensor-core path
// ------------------------------------------------------------------------------------------ //
__global__ void pack_weights_kernel(const float* __restrict__ hwio, int cin, int cout, int cin_pad, int cout_pad,
                                    long long total, __half* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(idx % cin_pad);
    const int o = (int)((idx / cin_pad) % cout_pad);
    const int t = (int)(idx / ((long long)cin_pad * cout_pad));
    float v = 0.f;
    if (o < cout && i < cin) v = hwio[((long long)t * cin + i) * cout + o];
    out[idx] = __float2half_rn(v);
  }
}

}  // namespace dsen2

// ============================================================================================ //
// C ABI
// ============================================================================================ //
using namespace dsen2;

extern "C" int dsen2_abi_version(void) { return DSEN2_ABI_VERSION; }
extern "C" const char* dsen2_last_error(void) { return g_err; }

extern "C" int dsen2_patch_counts(int grid_h, int grid_w, int patch_lr, int border_lr, int* allocated, int* filled) {
  DSEN2_REQUIRE(grid_h > 0 && grid_w > 0 && patch_lr > 0 && border_lr >= 0 && patch_lr > 2 * border_lr, DSEN2_E_BADARG,
                "dsen2_patch_counts: bad geometry (grid %dx%d patch %d border %d)", grid_h, grid_w, patch_lr, border_lr);
  const Tiling t = make_tiling(grid_h, grid_w, patch_lr, border_lr);
  if (allocated) *allocated = (t.k_i + 1) * (t.k_j + 1);
  if (filled) *filled = t.n_i * t.n_j;
  return 0;
}

extern "C" int dsen2_extract_patches(const float* d_img, int grid_h, int grid_w, int C, int ratio, int patch_lr,
                                     int border_lr, int first_patch, int num_patches, float divisor, float* d_out,
                                     void* stream) {
  DSEN2_REQUIRE(d_img && d_out, DSEN2_E_BADARG, "dsen2_extract_patches: null pointer");
  DSEN2_REQUIRE(grid_h > 0 && grid_w > 0 && C > 0 && ratio > 0 && patch_lr > 2 * border_lr && border_lr >= 0,
                DSEN2_E_BADARG, "dsen2_extract_patches: bad geometry");
  DSEN2_REQUIRE(grid_h + 2 * border_lr >= patch_lr && grid_w + 2 * border_lr >= patch_lr, DSEN2_E_BADARG,
                "dsen2_extract_patches: image (%dx%d on the tiling grid) smaller than one patch (%d)", grid_h, grid_w,
                patch_lr);
  DSEN2_REQUIRE(first_patch >= 0 && num_patches >= 0 && divisor != 0.f, DSEN2_E_BADARG,
                "dsen2_extract_patches: bad patch range / divisor");
  if (num_patches == 0) return 0;
  const Tiling tl = make_tiling(grid_h, grid_w, patch_lr, border_lr);
  DSEN2_REQUIRE(first_patch + num_patches <= (tl.k_i + 1) * (tl.k_j + 1), DSEN2_E_BADARG,
                "dsen2_extract_patches: patch range [%d,%d) exceeds the %d allocated patches", first_patch,
                first_patch + num_patches, (tl.k_i + 1) * (tl.k_j + 1));
  const int H = grid_h * ratio, W = grid_w * ratio, p = patch_lr * ratio, b = border_lr * ratio;
  const long long total = (long long)num_patches * p * p;
  const int block = 256;
  const dim3 grid = grid_for(total, block);
  cudaStream_t s = (cudaStream_t)stream;
  const bool aligned = ((uintptr_t)d_img % 16) == 0;
  if (C == 4 && aligned)
    extract_patches_kernel<4><<<grid, block, 0, s>>>(d_img, H, W, ratio, p, b, tl, first_patch, total, divisor, d_out);
  else if (C == 6 && aligned)
    extract_patches_kernel<6><<<grid, block, 0, s>>>(d_img, H, W, ratio, p, b, tl, first_patch, total, divisor, d_out);
  else if (C == 2 && aligned)
    extract_patches_kernel<2><<<grid, block, 0, s>>>(d_img, H, W, ratio, p, b, tl, first_patch, total, divisor, d_out);
  else
    extract_patches_generic_kernel<<<grid, block, 0, s>>>(d_img, H, W, C, ratio, p, b, tl, first_patch, total, divisor,
                                                          d_out);
  return check_launch("extract_patches");
}

extern "C" int dsen2_bilinear_mirror_up(const float* d_in, int planes, int p, int s, float post_divisor, float* d_out,
                                        void* stream) {
  DSEN2_REQUIRE(d_in && d_out, DSEN2_E_BADARG, "dsen2_bilinear_mirror_up: null pointer");
  DSEN2_REQUIRE(planes >= 0 && p > 0 && s > 0 && post_divisor != 0.f, DSEN2_E_BADARG,
                "dsen2_bilinear_mirror_up: bad sizes");
  if (planes == 0) return 0;
  const long long total = (long long)planes * p * s * p * s;
  const int bands = (p + kBilRows - 1) / kBilRows;
  const size_t band_smem = (size_t)(kBilRows + 2) * (p + 2) * sizeof(float);
  const int P = p * s;
  if (s == 2 && p == 64 && ((uintptr_t)d_in % 8) == 0 && ((uintptr_t)d_out % 16) == 0) {
    const long long warps = (long long)planes * 4;
    bilinear_mirror_x2_p64_kernel<<<(unsigned)((warps + 7) / 8), 256, 0, (cudaStream_t)stream>>>(d_in, planes, post_divisor, d_out);
    return check_launch("bilinear_mirror_up");
  }
  if (p >= 2 && P % 4 == 0 && P <= kBilMaxP && band_smem <= 48 * 1024 && (long long)planes * bands < (1LL << 31) &&
      ((uintptr_t)d_out % 16) == 0) {
    const int tx = P / 4, ty = kBilThreads / tx > 0 ? kBilThreads / tx : 1;
    const dim3 grid((unsigned)(planes * bands)), block(tx, ty);
    if (s == 2)
      bilinear_mirror_band_kernel<2><<<grid, block, band_smem, (cudaStream_t)stream>>>(d_in, p, s, bands, post_divisor, d_out);
    else if (s == 6)
      bilinear_mirror_band_kernel<6><<<grid, block, band_smem, (cudaStream_t)stream>>>(d_in, p, s, bands, post_divisor, d_out);
    else
      bilinear_mirror_band_kernel<0><<<grid, block, band_smem, (cudaStream_t)stream>>>(d_in, p, s, bands, post_divisor, d_out);
    return check_launch("bilinear_mirror_up");
  }
  const int block = 256;
  bilinear_mirror_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_in, p, s, total, post_divisor,
                                                                                     d_out);
  return check_launch("bilinear_mirror_up");
}

extern "C" int dsen2_recompose(const float* d_pred, int first_patch, int num_patches, int C, int P, int border, int H,
                               int W, float mul, float* d_out, void* stream) {
  DSEN2_REQUIRE(d_pred && d_out, DSEN2_E_BADARG, "dsen2_recompose: null pointer");
  const int S = P - 2 * border;
  DSEN2_REQUIRE(C > 0 && P > 0 && border >= 0 && S > 0, DSEN2_E_BADARG, "dsen2_recompose: bad patch geometry");
  DSEN2_REQUIRE(H >= S && W >= S, DSEN2_E_BADARG,
                "dsen2_recompose: image %dx%d smaller than the patch interior %d (patches.py:394-401 needs size >= patch)",
                H, W, S);
  DSEN2_REQUIRE(first_patch >= 0 && num_patches >= 0, DSEN2_E_BADARG, "dsen2_recompose: bad patch range");
  if (num_patches == 0) return 0;
  const int ny = ceil_div(H, S), nx = ceil_div(W, S);
  const int block = 256;
  // vector form: 16-byte plane loads need P, border (and so S) multiples of 4; 16-byte HWC stores need (y * W + x) * C * 4
  // bytes 16-byte aligned for x a multiple of 4: W * C a multiple of 4
  if ((C == 2 || C == 6) && P % 4 == 0 && border % 4 == 0 && (W * C) % 4 == 0 && (W - S) % 4 == 0 &&
      ((uintptr_t)d_pred % 16) == 0 && ((uintptr_t)d_out % 16) == 0) {
    const long long total4 = (long long)num_patches * S * (S / 4);
    if (C == 6)
      recompose_vec4_kernel<6><<<grid_for(total4, block, 32), block, 0, (cudaStream_t)stream>>>(d_pred, first_patch, P, border, H,
                                                                                              W, ny, nx, mul, total4, d_out);
    else
      recompose_vec4_kernel<2><<<grid_for(total4, block, 32), block, 0, (cudaStream_t)stream>>>(d_pred, first_patch, P, border, H,
                                                                                              W, ny, nx, mul, total4, d_out);
    return check_launch("recompose");
  }
  const long long total = (long long)num_patches * S * S;
  recompose_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_pred, first_patch, C, P, border, H, W,
                                                                               ny, nx, mul, total, d_out);
  return check_launch("recompose");
}

extern "C" int dsen2_bicubic_imresize(const void* d_in, int in_is_f64, int h, int w, int C, const double* d_wy,
                                      const int32_t* d_iy, int taps_y, int out_h, const double* d_wx,
                                      const int32_t* d_ix, int taps_x, int out_w, int first_dim, double* d_out,
                                      void* stream) {
  DSEN2_REQUIRE(d_in && d_wy && d_iy && d_wx && d_ix && d_out, DSEN2_E_BADARG, "dsen2_bicubic_imresize: null pointer");
  DSEN2_REQUIRE(h > 0 && w > 0 && C > 0 && taps_y > 0 && taps_x > 0 && out_h > 0 && out_w > 0 &&
                    (first_dim == 0 || first_dim == 1),
                DSEN2_E_BADARG, "dsen2_bicubic_imresize: bad sizes");
  const long long total = (long long)out_h * out_w * C;
  cudaStream_t s = (cudaStream_t)stream;
  // tile: 16 rows x TC columns with TC * C ~ 256-384 (x, c) pairs per row; the intermediate gets 40 KB of shared memory
  const int tcol = C >= 6 ? 64 : (C >= 3 ? 96 : 128);
  const int span_cap = (int)((40 * 1024 / sizeof(double)) / ((size_t)(first_dim == 0 ? kBicTR : tcol) * C));
  const size_t inter_bytes = (size_t)(first_dim == 0 ? kBicTR : tcol) * span_cap * C * sizeof(double);
  const long long gy = ((long long)out_h + kBicTR - 1) / kBicTR;
  if (span_cap >= 8 && gy <= 65535 && (long long)out_w * taps_x < (1LL << 29) && (long long)out_h * taps_y < (1LL << 29)) {
    const dim3 tgrid((unsigned)((out_w + tcol - 1) / tcol), (unsigned)gy);
    // a thread owns one (x, c) pair of the tile row in the second pass: 64 x 6 = 384 pairs are two rounds of 192 threads
    // (a third of the threads would idle in the second round of 256)
    const int bthreads = (tcol * C) % 256 != 0 && (tcol * C) % 192 == 0 ? 192 : 256;
#define DSEN2_BIC(T, F0, NTAPS)                                                                                            \
  bicubic_tiled_kernel<T, F0, NTAPS><<<tgrid, bthreads, inter_bytes, s>>>((const T*)d_in, h, w, C, d_wy, d_iy, taps_y, out_h, \
                                                                     d_wx, d_ix, taps_x, out_w, tcol, span_cap, d_out)
#define DSEN2_BIC2(T, F0) do { if (taps_y == 4 && taps_x == 4) DSEN2_BIC(T, F0, 4); else DSEN2_BIC(T, F0, 0); } while (0)
    if (in_is_f64) { if (first_dim == 0) DSEN2_BIC2(double, true); else DSEN2_BIC2(double, false); }
    else           { if (first_dim == 0) DSEN2_BIC2(float, true);  else DSEN2_BIC2(float, false); }
#undef DSEN2_BIC2
#undef DSEN2_BIC
    return check_launch("bicubic_imresize");
  }
  const int block = 256;
  const dim3 grid = grid_for(total, block);
  if (in_is_f64)
    bicubic_kernel<double><<<grid, block, 0, s>>>((const double*)d_in, h, w, C, d_wy, d_iy, taps_y, out_h, d_wx, d_ix,
                                                  taps_x, out_w, first_dim, total, d_out);
  else
    bicubic_kernel<float><<<grid, block, 0, s>>>((const float*)d_in, h, w, C, d_wy, d_iy, taps_y, out_h, d_wx, d_ix,
                                                 taps_x, out_w, first_dim, total, d_out);
  return check_launch("bicubic_imresize");
}

extern "C" int dsen2_down_pixel_aggr(const float* d_img, int integer_input, int H, int W, int C, int scale,
                                     const double* d_weights, int radius, float* d_tmp, double* d_out, void* stream) {
  DSEN2_REQUIRE(d_img && d_weights && d_tmp && d_out, DSEN2_E_BADARG, "dsen2_down_pixel_aggr: null pointer");
  DSEN2_REQUIRE(H > 0 && W > 0 && C > 0 && scale > 0 && radius >= 0 && H >= scale && W >= scale, DSEN2_E_BADARG,
                "dsen2_down_pixel_aggr: bad sizes");
  const long long total = (long long)H * W * C;
  const int block = 256;
  gauss_rows_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_img, H, W, C, d_weights, radius, integer_input,
                                                                                total, d_tmp);
  int rc = check_launch("gauss_rows");
  if (rc) return rc;
  const long long ototal = (long long)(H / scale) * (W / scale) * C;
  gauss_cols_mean_kernel<<<grid_for(ototal, block), block, 0, (cudaStream_t)stream>>>(d_tmp, H, W, C, d_weights, radius, scale,
                                                                                    integer_input, ototal, d_out);
  return check_launch("gauss_cols_mean");
}

extern "C" int dsen2_pack_conv_weights(const float* d_hwio, int cin, int cout, int cin_pad, int cout_pad, void* d_packed_f16,
                                       void* stream) {
  DSEN2_REQUIRE(d_hwio && d_packed_f16, DSEN2_E_BADARG, "dsen2_pack_conv_weights: null pointer");
  DSEN2_REQUIRE(cin > 0 && cout > 0 && cin_pad % 64 == 0 && cin_pad >= cin && cout_pad >= cout && cout_pad % 16 == 0,
                DSEN2_E_BADARG, "dsen2_pack_conv_weights: bad channel padding (cin %d->%d, cout %d->%d)", cin, cin_pad, cout,
                cout_pad);
  const long long total = 9LL * cout_pad * cin_pad;
  const int block = 256;
  pack_weights_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_hwio, cin, cout, cin_pad, cout_pad, total,
                                                                                  (__half*)d_packed_f16);
  return check_launch("pack_conv_weights");
}
