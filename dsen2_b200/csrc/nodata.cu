// Nodata handling of the tile pipeline (opt-in `nodata` value v of supres.DSen2_20 / DSen2_60).
//
// Output pixel (y, x) is NODATA iff every band of img10[y, x], of img20[y / 2, x / 2] and (60 m path) of img60[y / 6, x / 6]
// equals v, compared in the element type of the images (uint16 DN exactly, float32 as stored).  A pixel with data in any
// band of any input is valid: the rule never discards a measurement.
//   dsen2_nodata_patches: the ACTIVE patches of a range -- those that own (last writer wins, patches.py:394-403) at least one
//                         valid pixel -- as an ascending id list.  One block per patch reads the patch's owned rectangle
//                         and stops at the first valid pixel; a single-block scan then compacts the flags in place.
//   dsen2_nodata_fill:    v into every nodata pixel the range owns, after the last layer has stitched the active patches
//                         (dsen2_nodata_fill_u16: the same into a uint16 canvas).
// Together they read the inputs about once (1.3 GB of uint16 for a full 10980^2 tile, all of it only where it is empty).
#include "common.cuh"
#include "tiling.cuh"

namespace dsen2 {

struct NodataImages {
  const void* img10;
  const void* img20;
  const void* img60;    // null: the 20 m path
  int H, W;             // 10 m size
  float v;
};

template <typename T, int C>
__device__ __forceinline__ bool bands_equal(const T* px, float v) {
  bool eq = true;
#pragma unroll
  for (int c = 0; c < C; ++c) eq &= ld_px(px + c) == v;      // no short circuit: all loads in flight at once
  return eq;
}

template <typename T>
__device__ __forceinline__ bool is_nodata(const NodataImages& m, int y, int x) {
  const T* p10 = reinterpret_cast<const T*>(m.img10) + ((long long)y * m.W + x) * 4;
  const T* p20 = reinterpret_cast<const T*>(m.img20) + ((long long)(y >> 1) * (m.W >> 1) + (x >> 1)) * 6;
  bool nd = bands_equal<T, 4>(p10, m.v) & bands_equal<T, 6>(p20, m.v);
  if (m.img60) nd &= bands_equal<T, 2>(reinterpret_cast<const T*>(m.img60) + ((long long)(y / 6) * (m.W / 6) + x / 6) * 2, m.v);
  return nd;
}

static constexpr int kScanThreads = 256;
static constexpr int kScanPx = 4;       // pixels per thread per step: a block tests 1024 pixels between two barriers

// flags[b] = 1 iff patch first_patch + b owns a valid pixel
template <typename T>
__global__ void __launch_bounds__(kScanThreads) nodata_patch_flags_kernel(NodataImages m, int S, int ny, int nx,
                                                                           int first_patch, int* __restrict__ flags) {
  const int t = first_patch + blockIdx.x;
  const int ty = t / nx, tx = t - ty * nx;
  int y0, y1, x0, x1;
  owned_span(ty, m.H, S, ny, y0, y1);
  owned_span(tx, m.W, S, nx, x0, x1);
  const int w = x1 - x0, area = (y1 - y0) * w;
  int valid = 0;
  for (int base = 0; base < area; base += kScanThreads * kScanPx) {
    bool any = false;
#pragma unroll
    for (int k = 0; k < kScanPx; ++k) {
      const int i = base + k * kScanThreads + threadIdx.x;
      if (i < area) {
        const int dy = i / w;
        any |= !is_nodata<T>(m, y0 + dy, x0 + i - dy * w);
      }
    }
    if (__syncthreads_or(any)) { valid = 1; break; }        // uniform across the block
  }
  if (threadIdx.x == 0) flags[blockIdx.x] = valid;
}

// In place: ids[0, n) holds 0/1 flags -> ids[0, count) the ascending patch ids first_patch + b of the set flags.  One block,
// 1024 flags per step; an id is written at or before its own flag's index, after the step has read all of its flags.
__global__ void __launch_bounds__(1024) nodata_compact_kernel(int* __restrict__ ids, int n, int first_patch,
                                                              int* __restrict__ count) {
  __shared__ int warp_sums[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int base = 0;                                              // ids written by the previous steps (same in every thread)
  for (int step = 0; step < n; step += 1024) {
    const int i = step + threadIdx.x;
    const bool f = i < n && ids[i] != 0;
    const unsigned ball = __ballot_sync(0xffffffffu, f);
    if (lane == 0) warp_sums[warp] = __popc(ball);
    __syncthreads();                                         // every flag of this step has been read
    int off = base + __popc(ball & ((1u << lane) - 1u)), tot = 0;
    for (int k = 0; k < 32; ++k) {
      if (k == warp) off += tot;
      tot += warp_sums[k];
    }
    if (f) ids[off] = first_patch + i;
    base += tot;
    __syncthreads();                                         // warp_sums are rewritten by the next step
  }
  if (threadIdx.x == 0) *count = base;
}

// v into the nodata pixels of rows [y0, y0 + total / W) whose owner lies in [first_patch, end_patch); OutT: the canvas
// element type, float or uint16_t (v is then an integer in [0, 65535])
template <typename T, typename OutT>
__global__ void nodata_fill_kernel(NodataImages m, int S, int ny, int nx, int first_patch, int end_patch, int y0,
                                   long long total, int cout, OutT* __restrict__ canvas) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    const int dy = (int)(idx / m.W);
    const int y = y0 + dy, x = (int)(idx - (long long)dy * m.W);
    const int owner = tile_of(y, m.H, S, ny) * nx + tile_of(x, m.W, S, nx);
    if (owner >= first_patch && owner < end_patch && is_nodata<T>(m, y, x)) {
      OutT* o = canvas + ((long long)y * m.W + x) * cout;
      for (int c = 0; c < cout; ++c) o[c] = (OutT)m.v;
    }
  }
}

// Checks shared by both entry points; on success `tl` is the tiling and `S` the 10 m stride.
static int nodata_args(const char* name, const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H,
                       int W, int patch, int border, int first_patch, int num_patches, float nodata, Tiling& tl, int& S) {
  DSEN2_REQUIRE(d_img10 && d_img20, DSEN2_E_BADARG, "%s: null pointer", name);
  DSEN2_REQUIRE(img_dtype == DSEN2_IMG_F32 || img_dtype == DSEN2_IMG_U16, DSEN2_E_BADARG,
                "%s: img_dtype must be DSEN2_IMG_F32 or DSEN2_IMG_U16 (got %d)", name, img_dtype);
  DSEN2_REQUIRE(nodata == nodata, DSEN2_E_BADARG, "%s: nodata is NaN", name);
  const int r = d_img60 ? 6 : 2;
  DSEN2_REQUIRE(H > 0 && W > 0 && H % r == 0 && W % r == 0, DSEN2_E_BADARG,
                "%s: 10 m size %dx%d must be a multiple of %d", name, H, W, r);
  DSEN2_REQUIRE(patch > 0 && border >= 0 && patch % r == 0 && border % r == 0 && patch > 2 * border, DSEN2_E_BADARG,
                "%s: patch %d / border %d must be multiples of %d", name, patch, border, r);
  const int plr = patch / r, blr = border / r, gh = H / r, gw = W / r;
  DSEN2_REQUIRE(gh + 2 * blr >= plr && gw + 2 * blr >= plr, DSEN2_E_BADARG,
                "%s: image %dx%d smaller than one patch (%d)", name, H, W, patch);
  tl = make_tiling(gh, gw, plr, blr);
  S = tl.stride * r;
  DSEN2_REQUIRE(first_patch >= 0 && num_patches >= 0 && first_patch + num_patches <= tl.n_i * tl.n_j, DSEN2_E_BADARG,
                "%s: patch range [%d,%d) outside the %d filled patches", name, first_patch, first_patch + num_patches,
                tl.n_i * tl.n_j);
  return 0;
}

}  // namespace dsen2

using namespace dsen2;

extern "C" int dsen2_nodata_patches(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H,
                                    int W, int patch, int border, int first_patch, int num_patches, float nodata, int* d_ids,
                                    int* d_count, void* stream) {
  Tiling tl;
  int S = 0;
  int rc = nodata_args("dsen2_nodata_patches", d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, first_patch,
                       num_patches, nodata, tl, S);
  if (rc) return rc;
  DSEN2_REQUIRE(d_ids && d_count, DSEN2_E_BADARG, "dsen2_nodata_patches: null pointer");
  const cudaStream_t st = (cudaStream_t)stream;
  if (num_patches == 0) {
    DSEN2_CUDA(cudaMemsetAsync(d_count, 0, sizeof(int), st));
    return 0;
  }
  const NodataImages m{d_img10, d_img20, d_img60, H, W, nodata};
  if (img_dtype == DSEN2_IMG_U16)
    nodata_patch_flags_kernel<uint16_t><<<num_patches, kScanThreads, 0, st>>>(m, S, tl.n_i, tl.n_j, first_patch, d_ids);
  else
    nodata_patch_flags_kernel<float><<<num_patches, kScanThreads, 0, st>>>(m, S, tl.n_i, tl.n_j, first_patch, d_ids);
  if ((rc = check_launch("nodata_patch_flags")) != 0) return rc;
  nodata_compact_kernel<<<1, 1024, 0, st>>>(d_ids, num_patches, first_patch, d_count);
  return check_launch("nodata_compact");
}

template <typename OutT>
static int nodata_fill(const char* name, const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H,
                       int W, int patch, int border, int first_patch, int num_patches, float nodata, int cout,
                       OutT* d_canvas, void* stream) {
  Tiling tl;
  int S = 0;
  int rc = nodata_args(name, d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, first_patch, num_patches, nodata,
                       tl, S);
  if (rc) return rc;
  DSEN2_REQUIRE(d_canvas && cout > 0, DSEN2_E_BADARG, "%s: null canvas or cout %d", name, cout);
  if (num_patches == 0) return 0;
  // rows owned by the range: from the first patch's patch row to the last one's
  int y0, y1, unused;
  owned_span(first_patch / tl.n_j, H, S, tl.n_i, y0, unused);
  owned_span((first_patch + num_patches - 1) / tl.n_j, H, S, tl.n_i, unused, y1);
  const long long total = (long long)(y1 - y0) * W;
  const NodataImages m{d_img10, d_img20, d_img60, H, W, nodata};
  const int block = 256;
  const cudaStream_t st = (cudaStream_t)stream;
  if (img_dtype == DSEN2_IMG_U16)
    nodata_fill_kernel<uint16_t, OutT><<<grid_for(total, block), block, 0, st>>>(m, S, tl.n_i, tl.n_j, first_patch,
                                                                                first_patch + num_patches, y0, total, cout,
                                                                                d_canvas);
  else
    nodata_fill_kernel<float, OutT><<<grid_for(total, block), block, 0, st>>>(m, S, tl.n_i, tl.n_j, first_patch,
                                                                             first_patch + num_patches, y0, total, cout,
                                                                             d_canvas);
  return check_launch("nodata_fill");
}

extern "C" int dsen2_nodata_fill(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H, int W,
                                 int patch, int border, int first_patch, int num_patches, float nodata, int cout,
                                 float* d_canvas, void* stream) {
  return nodata_fill<float>("dsen2_nodata_fill", d_img10, d_img20, d_img60, img_dtype, H, W, patch, border, first_patch,
                            num_patches, nodata, cout, d_canvas, stream);
}

extern "C" int dsen2_nodata_fill_u16(const void* d_img10, const void* d_img20, const void* d_img60, int img_dtype, int H,
                                     int W, int patch, int border, int first_patch, int num_patches, float nodata, int cout,
                                     uint16_t* d_canvas, void* stream) {
  DSEN2_REQUIRE(nodata >= 0.f && nodata <= 65535.f && nodata == (float)(int)nodata, DSEN2_E_BADARG,
                "dsen2_nodata_fill_u16: nodata %g is not a uint16 value", (double)nodata);
  return nodata_fill<uint16_t>("dsen2_nodata_fill_u16", d_img10, d_img20, d_img60, img_dtype, H, W, patch, border,
                               first_patch, num_patches, nodata, cout, d_canvas, stream);
}
