// Network-input preparation and weight packing for the CTA-pair convolution kernels (conv_pair.cu).
//
// Inference: "x_in16", NHWC fp16 with 16 channels per pixel as a hi tensor and a lo tensor (v = hi + lo to ~22 bits);
// channel c = band c of the channel concatenation X of the network inputs (DSen2Net.py:24,26), zero above.
//   dsen2_prep16_from_patches : X given as NCHW fp32 patch stacks (model.predict drop-in, supres.py:65)
//   dsen2_prep16_from_images  : X gathered straight from the HWC images (float32 or uint16 DN) -- fuses get_test_patches /
//                               get_test_patches60 (patches.py:19-156: symmetric pad, crop), interp_patches
//                               (patches.py:11-16: per-patch bilinear with mirror boundary) and the /2000 scaling
//                               (supres.py:23-24,42-44) with the arithmetic of the standalone kernels.
//   dsen2_prep16_from_images_offset : the same with a radiometric offset added to every loaded band value first
//   dsen2_prep16_from_chips   : the same from stacks of same-size chips, patches indexed chip * ppc + patch
// Training step (and networks without resblocks): "x_in", 64 channels per pixel = the three HORIZONTAL taps of the first
// 3x3 convolution pre-gathered, x_in[n][y][x][t*16 + c] = X[n][c][y][x + t - 1] (zero outside the patch), because the
// first layer's weight-gradient GEMM wants 128-byte pixel rows (dsen2_prep_from_patches).
#include "common.cuh"
#include "tiling.cuh"

namespace dsen2 {

struct __align__(16) Half16 {
  __half v[16];
};

__device__ __forceinline__ void split16(const float (&x)[16], Half16& hi, Half16& lo) {
#pragma unroll
  for (int c = 0; c < 16; ++c) {
    hi.v[c] = __float2half_rn(x[c]);
    lo.v[c] = __float2half_rn(x[c] - __half2float(hi.v[c]));
  }
}

__device__ __forceinline__ void store32(__half* dst, const Half16& h) {
  const uint4* s = reinterpret_cast<const uint4*>(&h);
  uint4* d = reinterpret_cast<uint4*>(dst);
  d[0] = s[0];
  d[1] = s[1];
}

struct PrepSource {
  const void* img;    // (H, W, C) HWC, float32 or uint16 DN; C = 4 / 6 / 2 for the 10 / 20 / 60 m inputs
  int H, W;
  int ratio;          // source pixels per tiling-grid pixel
  int s;              // upsampling factor to the 10 m patch (1 = none)
};

// A band value as the arithmetic below takes it: the stored element, or with ADD fl32(x + add_offset) (the radiometric
// offset of Sentinel-2 products since processing baseline 04.00).  ADD is a template switch, not an add of 0: -0 + 0 is +0.
template <bool ADD, typename T>
__device__ __forceinline__ float ld_band(const T* p, float add_offset) {
  return ADD ? __fadd_rn(ld_px(p), add_offset) : ld_px(p);
}

// value of band c of `src` at 10 m patch pixel (y, x): crop + symmetric pad (+ mirror bilinear) + /divisor
template <typename T, int C, int OFF, bool ADD>
__device__ __forceinline__ void prep_gather(const PrepSource& src, int si, int sj, int plr, int blr, int y, int x,
                                            float divisor, float add_offset, float (&v)[16]) {
  const T* img = reinterpret_cast<const T*>(src.img);
  const int p = plr * src.ratio, b = blr * src.ratio;
  const int oi = si * src.ratio - b, oj = sj * src.ratio - b;
  if (src.s == 1) {
    const T* q = img + ((long long)sym_index(oi + y, src.H) * src.W + sym_index(oj + x, src.W)) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) v[OFF + c] = __fdiv_rn(ld_band<ADD>(q + c, add_offset), divisor);
    return;
  }
  int y0, y1, x0, x1;
  float fy, fx;
  bilin_tap(y, src.s, p, y0, y1, fy);
  bilin_tap(x, src.s, p, x0, x1, fx);
  const long long r0 = (long long)sym_index(oi + y0, src.H) * src.W, r1 = (long long)sym_index(oi + y1, src.H) * src.W;
  const int q0 = sym_index(oj + x0, src.W), q1 = sym_index(oj + x1, src.W);
  const T* p00 = img + (r0 + q0) * C;
  const T* p01 = img + (r0 + q1) * C;
  const T* p10 = img + (r1 + q0) * C;
  const T* p11 = img + (r1 + q1) * C;
  const float k = 30000.0f;                  // the reference scales by 1/30000 around the resize (patches.py:15)
#pragma unroll
  for (int c = 0; c < C; ++c) {
    const float v00 = __fdiv_rn(ld_band<ADD>(p00 + c, add_offset), k), v01 = __fdiv_rn(ld_band<ADD>(p01 + c, add_offset), k);
    const float v10 = __fdiv_rn(ld_band<ADD>(p10 + c, add_offset), k), v11 = __fdiv_rn(ld_band<ADD>(p11 + c, add_offset), k);
    const float c0 = v00 * (1.0f - fy) + v10 * fy;   // rows first, then columns (as bilinear_mirror_kernel)
    const float c1 = v01 * (1.0f - fy) + v11 * fy;
    const float r = (c0 * (1.0f - fx) + c1 * fx) * k;
    v[OFF + c] = __fdiv_rn(r, divisor);
  }
}

// ---- un-gathered 16-channel prepared input (inference path) ---------------------------------------------------------
// x_in16[n][y][x][c] = X[n][c][y][x] (c >= ctot zero), hi and lo tensors: 32 bytes per pixel each instead of 128.
// The head convolution then runs all nine taps as shifted descriptors into a 32-byte-row halo box (conv_pair.cu,
// CfgHead16); a thread writes its own pixel only, consecutive threads consecutive 32-byte chunks.
__global__ void prep16_from_patches_kernel(const float* __restrict__ x0, int c0, const float* __restrict__ x1, int c1,
                                           const float* __restrict__ x2, int c2, int P, long long total,
                                           __half* __restrict__ out_hi, __half* __restrict__ out_lo) {
  const long long PP = (long long)P * P;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const long long n = idx / PP;
    const int rem = (int)(idx - n * PP);
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      float t = 0.f;
      if (c < c0) t = __ldg(x0 + (n * c0 + c) * PP + rem);
      else if (c < c0 + c1) t = __ldg(x1 + (n * c1 + (c - c0)) * PP + rem);
      else if (c < c0 + c1 + c2) t = __ldg(x2 + (n * c2 + (c - c0 - c1)) * PP + rem);
      v[c] = t;
    }
    Half16 hi, lo;
    split16(v, hi, lo);
    store32(out_hi + idx * 16, hi);
    store32(out_lo + idx * 16, lo);
  }
}

// The source of chip `chip` of a stack of same-size images (N, H, W, C): the image pointer advanced by chip * H * W * C
// elements, in 64 bits (100k chips of 120 x 120 x 4 are 5.8e9 elements).
template <typename T, int C>
__device__ __forceinline__ PrepSource chip_source(PrepSource s, int chip) {
  s.img = reinterpret_cast<const T*>(s.img) + (long long)chip * s.H * s.W * C;
  return s;
}

// IDS: batch entry b is patch ids[b] (a list of active patches) instead of first_patch + b.  ADD: add_offset is added to
// every loaded band value (ld_band); it is the last parameter, so the other instances keep their parameter layout.
// CHIPS: the images are stacks of same-size chips and first_patch + b indexes the flat list chip * ppc + patch, with ppc =
// n_i * n_j the filled patches of one chip; the chip and its patch are resolved per patch index with one 32-bit division.
template <typename T, bool IDS, bool ADD, bool CHIPS>
__global__ void prep16_from_images_kernel(PrepSource s0, PrepSource s1, PrepSource s2, int nsrc, int plr, int blr, int P,
                                          Tiling tl, int first_patch, const int* __restrict__ ids, long long total,
                                          float divisor, __half* __restrict__ out_hi, __half* __restrict__ out_lo,
                                          float add_offset) {
  const int PP = P * P;
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int local = (int)(idx / PP);
    const int rem = (int)(idx - (long long)local * PP);
    const int y = rem / P, x = rem - y * P;
    int patch = IDS ? __ldg(ids + local) : first_patch + local;
    int chip = 0;
    if constexpr (CHIPS) {
      chip = patch / (tl.n_i * tl.n_j);
      patch -= chip * (tl.n_i * tl.n_j);
    }
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) v[c] = 0.f;
    // surplus patches of the allocated stack stay zero (patches.py:32-39), and so do ids outside the tiling
    if ((!IDS || patch >= 0) && patch < tl.n_i * tl.n_j) {
      const int ti = patch / tl.n_j, tj = patch - ti * tl.n_j;
      const int si = ti < tl.k_i ? ti * tl.stride : tl.last_i;
      const int sj = tj < tl.k_j ? tj * tl.stride : tl.last_j;
      if constexpr (CHIPS) {
        prep_gather<T, 4, 0, ADD>(chip_source<T, 4>(s0, chip), si, sj, plr, blr, y, x, divisor, add_offset, v);
        prep_gather<T, 6, 4, ADD>(chip_source<T, 6>(s1, chip), si, sj, plr, blr, y, x, divisor, add_offset, v);
        if (nsrc == 3) prep_gather<T, 2, 10, ADD>(chip_source<T, 2>(s2, chip), si, sj, plr, blr, y, x, divisor, add_offset, v);
      } else {
        prep_gather<T, 4, 0, ADD>(s0, si, sj, plr, blr, y, x, divisor, add_offset, v);     // 10 m bands   (DSen2Net.py:24,26 order)
        prep_gather<T, 6, 4, ADD>(s1, si, sj, plr, blr, y, x, divisor, add_offset, v);     // 20 m bands
        if (nsrc == 3) prep_gather<T, 2, 10, ADD>(s2, si, sj, plr, blr, y, x, divisor, add_offset, v);   // 60 m bands
      }
    }
    Half16 hi, lo;
    split16(v, hi, lo);
    store32(out_hi + idx * 16, hi);
    store32(out_lo + idx * 16, lo);
  }
}

// head weights for the 16-channel input: [tap = dy*3+dx][2F rows = W_hi ; W_lo][16: c]
__global__ void pack_head16_weights_kernel(const float* __restrict__ hwio, int cin, int F, long long total,
                                           __half* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(idx % 16);
    const int r = (int)((idx / 16) % (2 * F));
    const int tap = (int)(idx / (16LL * 2 * F));
    float v = 0.f;
    if (c < cin) v = hwio[((long long)tap * cin + c) * F + (r % F)];
    const __half hi = __float2half_rn(v);
    out[idx] = r < F ? hi : __float2half_rn(v - __half2float(hi));
  }
}

// ---- 64-channel form (P <= 256): coalesced x_in stores ---------------------------------------------------------
// A block owns R = 256 / P whole patch rows: each thread
// computes its pixel's 16-channel vector once, parks hi / lo in shared memory, and the block then writes the rows
// out as contiguous 16-byte chunks (lane = chunk: a warp store covers four full 128-byte lines).
__device__ __forceinline__ void rowblock_store(const Half16& hi, const Half16& lo, bool active, int r, int x, int P, int R,
                                               long long first_row, long long total_rows, __half* __restrict__ out_hi,
                                               __half* __restrict__ out_lo) {
  extern __shared__ uint4 s_rows[];                       // [2 (hi, lo)][R][P + 2][2 x 16 B]; columns 0 and P + 1 are zero
  const int pitch = (P + 2) * 2;
  uint4* s_hi = s_rows;
  uint4* s_lo = s_rows + R * pitch;
  const uint4 z = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < R * 2; i += blockDim.x) {  // guard columns
    const int rr = i >> 1, side = i & 1;
    const int col = side ? P + 1 : 0;
    s_hi[rr * pitch + col * 2] = z; s_hi[rr * pitch + col * 2 + 1] = z;
    s_lo[rr * pitch + col * 2] = z; s_lo[rr * pitch + col * 2 + 1] = z;
  }
  if (active) {
    const uint4* h = reinterpret_cast<const uint4*>(&hi);
    const uint4* l = reinterpret_cast<const uint4*>(&lo);
    const int o = r * pitch + (x + 1) * 2;
    s_hi[o] = h[0]; s_hi[o + 1] = h[1];
    s_lo[o] = l[0]; s_lo[o + 1] = l[1];
  }
  __syncthreads();
  // chunk c of pixel x: taps t = c / 2 (pixel x + t - 1 -> column x + t of the guarded row), half c % 2; chunks 6, 7 zero
  const int chunks = R * P * 8;
  for (int i = threadIdx.x; i < chunks; i += blockDim.x) {
    const int pix = i >> 3, c = i & 7;
    const int rr = pix / P, xx = pix - rr * P;
    const long long row = first_row + rr;
    if (row >= total_rows) break;
    uint4 vh = z, vl = z;
    if (c < 6) {
      const int o = rr * pitch + (xx + (c >> 1)) * 2 + (c & 1);
      vh = s_hi[o];
      vl = s_lo[o];
    }
    const long long dst = (row * P + xx) * 8 + c;          // in 16-byte units
    reinterpret_cast<uint4*>(out_hi)[dst] = vh;
    reinterpret_cast<uint4*>(out_lo)[dst] = vl;
  }
}

__global__ void prep_from_patches_rows_kernel(const float* __restrict__ x0, int c0, const float* __restrict__ x1, int c1,
                                              const float* __restrict__ x2, int c2, int P, int R, long long total_rows,
                                              __half* __restrict__ out_hi, __half* __restrict__ out_lo) {
  const long long PP = (long long)P * P;
  const long long first_row = (long long)blockIdx.x * R;
  const int r = threadIdx.x / P, x = threadIdx.x - r * P;
  const long long row = first_row + r;
  const bool active = r < R && row < total_rows;
  Half16 hi, lo;
  if (active) {
    const long long n = row / P;
    const int rem = (int)(row - n * P) * P + x;
    float v[16];
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      float t = 0.f;
      if (c < c0) t = __ldg(x0 + (n * c0 + c) * PP + rem);
      else if (c < c0 + c1) t = __ldg(x1 + (n * c1 + (c - c0)) * PP + rem);
      else if (c < c0 + c1 + c2) t = __ldg(x2 + (n * c2 + (c - c0 - c1)) * PP + rem);
      v[c] = t;
    }
    split16(v, hi, lo);
  }
  rowblock_store(hi, lo, active, r, x, P, R, first_row, total_rows, out_hi, out_lo);
}

// launch geometry of the row-block kernels: R rows per block, R * P threads rounded up to whole warps
struct RowBlock { int R, threads; size_t smem; };
static RowBlock row_block(int P) {
  RowBlock g;
  g.R = 256 / P > 0 ? 256 / P : 1;
  g.threads = (g.R * P + 31) / 32 * 32;
  g.smem = (size_t)2 * g.R * (P + 2) * 2 * sizeof(uint4);
  return g;
}

// head weights: [dy][2F rows = W_hi ; W_lo][64: k = dxi*16 + c]
__global__ void pack_head_weights_kernel(const float* __restrict__ hwio, int cin, int F, long long total,
                                         __half* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % 64);
    const int r = (int)((idx / 64) % (2 * F));
    const int dy = (int)(idx / (64LL * 2 * F));
    const int dxi = k >> 4, c = k & 15;
    float v = 0.f;
    if (dxi < 3 && c < cin) v = hwio[((long long)(dy * 3 + dxi) * cin + c) * F + (r % F)];
    const __half hi = __float2half_rn(v);
    out[idx] = r < F ? hi : __float2half_rn(v - __half2float(hi));
  }
}

// tail weights: [tap][32 rows = W_hi (16) ; W_lo (16)][F]
__global__ void pack_tail_weights_kernel(const float* __restrict__ hwio, int F, int cout, long long total,
                                         __half* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % F);
    const int r = (int)((idx / F) % 32);
    const int tap = (int)(idx / (32LL * F));
    const int co = r & 15;
    float v = 0.f;
    if (co < cout) v = hwio[((long long)tap * F + k) * cout + co];
    const __half hi = __float2half_rn(v);
    out[idx] = r < 16 ? hi : __float2half_rn(v - __half2float(hi));
  }
}

}  // namespace dsen2

using namespace dsen2;

extern "C" int dsen2_prep_from_patches(const float* d_x0, int c0, const float* d_x1, int c1, const float* d_x2, int c2,
                                       int n, int P, void* d_xin_hi, void* d_xin_lo, void* stream) {
  DSEN2_REQUIRE(d_x0 && d_x1 && d_xin_hi && d_xin_lo && (c2 == 0 || d_x2), DSEN2_E_BADARG,
                "dsen2_prep_from_patches: null pointer");
  DSEN2_REQUIRE(c0 > 0 && c1 > 0 && c2 >= 0 && c0 + c1 + c2 <= 16 && n >= 0 && P > 0, DSEN2_E_BADARG,
                "dsen2_prep_from_patches: bad sizes (%d+%d+%d channels, at most 16)", c0, c1, c2);
  DSEN2_REQUIRE(((uintptr_t)d_xin_hi % 16) == 0 && ((uintptr_t)d_xin_lo % 16) == 0, DSEN2_E_ALIGN,
                "dsen2_prep_from_patches: outputs must be 16-byte aligned");
  DSEN2_REQUIRE(P <= 256, DSEN2_E_BADARG, "dsen2_prep_from_patches: patches of at most 256 x 256 (got %d)", P);
  if (n == 0) return 0;
  const RowBlock g = row_block(P);
  const long long rows = (long long)n * P;
  prep_from_patches_rows_kernel<<<(unsigned)((rows + g.R - 1) / g.R), g.threads, g.smem, (cudaStream_t)stream>>>(
      d_x0, c0, d_x1, c1, d_x2, c2, P, g.R, rows, (__half*)d_xin_hi, (__half*)d_xin_lo);
  return check_launch("prep_from_patches");
}

extern "C" int dsen2_pack_head_weights(const float* d_hwio, int cin, int feature_size, void* d_packed, void* stream) {
  DSEN2_REQUIRE(d_hwio && d_packed, DSEN2_E_BADARG, "dsen2_pack_head_weights: null pointer");
  DSEN2_REQUIRE(cin > 0 && cin <= 16 && feature_size > 0, DSEN2_E_BADARG,
                "dsen2_pack_head_weights: at most 16 input channels (got %d)", cin);
  const long long total = 3LL * 2 * feature_size * 64;
  const int block = 256;
  pack_head_weights_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_hwio, cin, feature_size, total,
                                                                                       (__half*)d_packed);
  return check_launch("pack_head_weights");
}

extern "C" int dsen2_pack_tail_weights(const float* d_hwio, int feature_size, int cout, void* d_packed, void* stream) {
  DSEN2_REQUIRE(d_hwio && d_packed, DSEN2_E_BADARG, "dsen2_pack_tail_weights: null pointer");
  DSEN2_REQUIRE(cout > 0 && cout <= 16 && feature_size > 0, DSEN2_E_BADARG,
                "dsen2_pack_tail_weights: at most 16 output bands (got %d)", cout);
  const long long total = 9LL * 32 * feature_size;
  const int block = 256;
  pack_tail_weights_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_hwio, feature_size, cout, total,
                                                                                       (__half*)d_packed);
  return check_launch("pack_tail_weights");
}

extern "C" int dsen2_prep16_from_patches(const float* d_x0, int c0, const float* d_x1, int c1, const float* d_x2, int c2,
                                         int n, int P, void* d_xin_hi, void* d_xin_lo, void* stream) {
  DSEN2_REQUIRE(d_x0 && d_x1 && d_xin_hi && d_xin_lo && (c2 == 0 || d_x2), DSEN2_E_BADARG,
                "dsen2_prep16_from_patches: null pointer");
  DSEN2_REQUIRE(c0 > 0 && c1 > 0 && c2 >= 0 && c0 + c1 + c2 <= 16 && n >= 0 && P > 0, DSEN2_E_BADARG,
                "dsen2_prep16_from_patches: bad sizes (%d+%d+%d channels, at most 16)", c0, c1, c2);
  DSEN2_REQUIRE(((uintptr_t)d_xin_hi % 16) == 0 && ((uintptr_t)d_xin_lo % 16) == 0, DSEN2_E_ALIGN,
                "dsen2_prep16_from_patches: outputs must be 16-byte aligned");
  if (n == 0) return 0;
  const long long total = (long long)n * P * P;
  const int block = 256;
  prep16_from_patches_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(
      d_x0, c0, d_x1, c1, d_x2, c2, P, total, (__half*)d_xin_hi, (__half*)d_xin_lo);
  return check_launch("prep16_from_patches");
}

template <typename T, bool IDS, bool ADD, bool CHIPS>
static void launch_prep16(PrepSource s0, PrepSource s1, PrepSource s2, int nsrc, int plr, int blr, int P, Tiling tl,
                          int first_patch, const int* d_patch_ids, long long total, float divisor, float add_offset,
                          void* d_xin_hi, void* d_xin_lo, cudaStream_t stream) {
  const int block = 256;
  prep16_from_images_kernel<T, IDS, ADD, CHIPS><<<grid_for(total, block), block, 0, stream>>>(
      s0, s1, s2, nsrc, plr, blr, P, tl, first_patch, d_patch_ids, total, divisor, (__half*)d_xin_hi, (__half*)d_xin_lo,
      add_offset);
}

// the instance for (add, chips); the chip form exists for the range form only
template <typename T, bool IDS>
static void launch_prep16_of(bool add, bool chips, PrepSource s0, PrepSource s1, PrepSource s2, int nsrc, int plr, int blr,
                             int P, Tiling tl, int first_patch, const int* d_patch_ids, long long total, float divisor,
                             float add_offset, void* d_xin_hi, void* d_xin_lo, cudaStream_t st) {
  if (!IDS && chips) {
    if (add) launch_prep16<T, false, true, true>(s0, s1, s2, nsrc, plr, blr, P, tl, first_patch, nullptr, total, divisor,
                                                 add_offset, d_xin_hi, d_xin_lo, st);
    else launch_prep16<T, false, false, true>(s0, s1, s2, nsrc, plr, blr, P, tl, first_patch, nullptr, total, divisor,
                                              add_offset, d_xin_hi, d_xin_lo, st);
  } else if (add) {
    launch_prep16<T, IDS, true, false>(s0, s1, s2, nsrc, plr, blr, P, tl, first_patch, d_patch_ids, total, divisor,
                                       add_offset, d_xin_hi, d_xin_lo, st);
  } else {
    launch_prep16<T, IDS, false, false>(s0, s1, s2, nsrc, plr, blr, P, tl, first_patch, d_patch_ids, total, divisor,
                                        add_offset, d_xin_hi, d_xin_lo, st);
  }
}

// add: run the ADD instances with add_offset (finite; checked by the caller).  num_chips >= 0: the images are stacks of
// num_chips same-size chips and [first_patch, first_patch + num_patches) a range of their flat filled-patch list (CHIPS
// instances; IDS is false); -1: one image.
template <bool IDS>
static int prep16_from_images(const char* name, const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype,
                              int H, int W, int patch, int border, int first_patch, const int* d_patch_ids, int num_patches,
                              float divisor, bool add, float add_offset, void* d_xin_hi, void* d_xin_lo, void* stream,
                              int num_chips = -1) {
  DSEN2_REQUIRE(d_img10 && d_img20 && d_xin_hi && d_xin_lo && (!IDS || d_patch_ids), DSEN2_E_BADARG, "%s: null pointer", name);
  DSEN2_REQUIRE(img_dtype == DSEN2_IMG_F32 || img_dtype == DSEN2_IMG_U16, DSEN2_E_BADARG,
                "%s: img_dtype must be DSEN2_IMG_F32 or DSEN2_IMG_U16 (got %d)", name, img_dtype);
  const int r = d_img60 ? 6 : 2;                 // the tiling grid is the coarsest input (patches.py:45-53,114-122)
  DSEN2_REQUIRE(H > 0 && W > 0 && H % r == 0 && W % r == 0, DSEN2_E_BADARG,
                "%s: 10 m size %dx%d must be a multiple of %d", name, H, W, r);
  DSEN2_REQUIRE(patch > 0 && border >= 0 && patch % r == 0 && border % r == 0 && patch > 2 * border, DSEN2_E_BADARG,
                "%s: patch %d / border %d must be multiples of %d", name, patch, border, r);
  DSEN2_REQUIRE(first_patch >= 0 && num_patches >= 0 && divisor != 0.f, DSEN2_E_BADARG,
                "%s: bad patch range / divisor", name);
  DSEN2_REQUIRE(((uintptr_t)d_xin_hi % 16) == 0 && ((uintptr_t)d_xin_lo % 16) == 0, DSEN2_E_ALIGN,
                "%s: outputs must be 16-byte aligned", name);
  const int plr = patch / r, blr = border / r, gh = H / r, gw = W / r;
  DSEN2_REQUIRE(gh + 2 * blr >= plr && gw + 2 * blr >= plr, DSEN2_E_BADARG,
                "%s: image %dx%d smaller than one patch (%d)", name, H, W, patch);
  const Tiling tl = make_tiling(gh, gw, plr, blr);
  const bool chips = num_chips >= 0;
  if (chips) {
    const long long flat = (long long)num_chips * tl.n_i * tl.n_j;
    DSEN2_REQUIRE(flat < (1LL << 31) && (long long)first_patch + num_patches <= flat, DSEN2_E_BADARG,
                  "%s: patch range [%d,%lld) outside the %lld filled patches of %d chips", name, first_patch,
                  (long long)first_patch + num_patches, flat, num_chips);
  }
  if (num_patches == 0) return 0;
  DSEN2_REQUIRE(IDS || chips || first_patch + num_patches <= (tl.k_i + 1) * (tl.k_j + 1), DSEN2_E_BADARG,
                "%s: patch range [%d,%d) exceeds the %d allocated patches", name, first_patch,
                first_patch + num_patches, (tl.k_i + 1) * (tl.k_j + 1));
  PrepSource s0{d_img10, H, W, r, 1};
  PrepSource s1{d_img20, H / 2, W / 2, r / 2, 2};
  PrepSource s2{d_img60, H / 6, W / 6, 1, 6};
  const long long total = (long long)num_patches * patch * patch;
  const int nsrc = d_img60 ? 3 : 2;
  const cudaStream_t st = (cudaStream_t)stream;
  if (img_dtype == DSEN2_IMG_U16)
    launch_prep16_of<uint16_t, IDS>(add, chips, s0, s1, s2, nsrc, plr, blr, patch, tl, first_patch, d_patch_ids, total,
                                    divisor, add ? add_offset : 0.f, d_xin_hi, d_xin_lo, st);
  else
    launch_prep16_of<float, IDS>(add, chips, s0, s1, s2, nsrc, plr, blr, patch, tl, first_patch, d_patch_ids, total,
                                 divisor, add ? add_offset : 0.f, d_xin_hi, d_xin_lo, st);
  return check_launch(name);
}

extern "C" int dsen2_prep16_from_images(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H,
                                        int W, int patch, int border, int first_patch, int num_patches, float divisor,
                                        void* d_xin_hi, void* d_xin_lo, void* stream) {
  return prep16_from_images<false>("dsen2_prep16_from_images", d_img10, d_img20, d_img60, img_dtype, H, W, patch, border,
                                   first_patch, nullptr, num_patches, divisor, false, 0.f, d_xin_hi, d_xin_lo, stream);
}

extern "C" int dsen2_prep16_from_images_ids(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype,
                                            int H, int W, int patch, int border, const int* d_patch_ids, int num_patches,
                                            float divisor, void* d_xin_hi, void* d_xin_lo, void* stream) {
  return prep16_from_images<true>("dsen2_prep16_from_images_ids", d_img10, d_img20, d_img60, img_dtype, H, W, patch, border,
                                  0, d_patch_ids, num_patches, divisor, false, 0.f, d_xin_hi, d_xin_lo, stream);
}

extern "C" int dsen2_prep16_from_images_offset(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype,
                                               int H, int W, int patch, int border, int first_patch, const int* d_patch_ids,
                                               int num_patches, float divisor, float add_offset, void* d_xin_hi,
                                               void* d_xin_lo, void* stream) {
  const char* name = "dsen2_prep16_from_images_offset";
  DSEN2_REQUIRE(isfinite(add_offset), DSEN2_E_BADARG, "%s: add_offset must be finite", name);
  if (d_patch_ids)
    return prep16_from_images<true>(name, d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, 0, d_patch_ids,
                                    num_patches, divisor, true, add_offset, d_xin_hi, d_xin_lo, stream);
  return prep16_from_images<false>(name, d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, first_patch, nullptr,
                                   num_patches, divisor, true, add_offset, d_xin_hi, d_xin_lo, stream);
}

extern "C" int dsen2_prep16_from_chips(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype,
                                       int num_chips, int H, int W, int patch, int border, int first_patch, int num_patches,
                                       float divisor, int add, float add_offset, void* d_xin_hi, void* d_xin_lo,
                                       void* stream) {
  const char* name = "dsen2_prep16_from_chips";
  DSEN2_REQUIRE(num_chips >= 0, DSEN2_E_BADARG, "%s: num_chips %d < 0", name, num_chips);
  DSEN2_REQUIRE(add == 0 || add == 1, DSEN2_E_BADARG, "%s: add must be 0 or 1 (got %d)", name, add);
  DSEN2_REQUIRE(!add || isfinite(add_offset), DSEN2_E_BADARG, "%s: add_offset must be finite", name);
  return prep16_from_images<false>(name, d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, first_patch, nullptr,
                                   num_patches, divisor, add != 0, add_offset, d_xin_hi, d_xin_lo, stream, num_chips);
}

extern "C" int dsen2_pack_head16_weights(const float* d_hwio, int cin, int feature_size, void* d_packed, void* stream) {
  DSEN2_REQUIRE(d_hwio && d_packed, DSEN2_E_BADARG, "dsen2_pack_head16_weights: null pointer");
  DSEN2_REQUIRE(cin > 0 && cin <= 16 && feature_size > 0, DSEN2_E_BADARG,
                "dsen2_pack_head16_weights: at most 16 input channels (got %d)", cin);
  const long long total = 9LL * 2 * feature_size * 16;
  const int block = 256;
  pack_head16_weights_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_hwio, cin, feature_size, total,
                                                                                         (__half*)d_packed);
  return check_launch("pack_head16_weights");
}
