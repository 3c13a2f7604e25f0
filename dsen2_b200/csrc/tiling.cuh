// Tiling / resampling index arithmetic shared by the patch, prep and stitch kernels.
#pragma once
#include "common.cuh"

namespace dsen2 {

inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

inline dim3 grid_for(long long work_items, int block, int max_waves = 16) {
  long long blocks = (work_items + block - 1) / block;
  long long cap = (long long)sm_count() * max_waves;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return dim3((unsigned)blocks);
}

// ------------------------------------------------------------------------------------------ //
// tiling arithmetic shared by host and device (patches.py:32-53, SURVEY appendix A)
// ------------------------------------------------------------------------------------------ //
struct Tiling {
  int k_i, k_j;    // full strides per axis
  int n_i, n_j;    // filled crop starts per axis
  int stride;      // patch_lr - 2*border_lr
  int last_i, last_j;  // clamped start (padded lr coords) of the extra crop, if any
};

__host__ __device__ inline Tiling make_tiling(int grid_h, int grid_w, int patch_lr, int border_lr) {
  Tiling t;
  t.stride = patch_lr - 2 * border_lr;
  t.k_i = grid_h / t.stride;
  t.k_j = grid_w / t.stride;
  t.n_i = t.k_i + (grid_h % t.stride != 0);
  t.n_j = t.k_j + (grid_w % t.stride != 0);
  t.last_i = grid_h + 2 * border_lr - patch_lr;
  t.last_j = grid_w + 2 * border_lr - patch_lr;
  return t;
}

struct PrepSource {
  const void* img;    // (H, W, C) HWC, float32 or uint16 DN; C = 4 / 6 / 2 for the 10 / 20 / 60 m inputs
  int H, W;
  int ratio;          // source pixels per tiling-grid pixel
  int s;              // upsampling factor to the 10 m patch (1 = none)
};

// One scene of a scene list (dsen2_scene_table): everything the preparation and the last layer take from the single
// geometry of a 3-D call, precomputed on the host, so that a kernel resolves a flat patch's scene with loads only (the
// patch -> scene map, then this entry).  The 10 m size is src[0].H x src[0].W; the stitch grid is tl.n_i x tl.n_j.
struct SceneGeom {
  PrepSource src[3];  // 10, 20, 60 m images as the 3-D preparation takes them (src[2].img null on the 20 m path)
  Tiling tl;          // the scene's own tiling: n_i * n_j filled patches
  int first;          // flat index of the scene's first patch (prefix sum of the filled-patch counts before it)
  void* canvas;       // (H, W, cout) output of the scene: float or uint16, the canvas type of the call
};
static_assert(sizeof(SceneGeom) == 112, "the scene table layout is private, but its size is what dsen2_scene_table_bytes reports");

__device__ __forceinline__ int sym_index(int j, int n) {  // numpy pad(mode='symmetric')
  if (j < 0) j = -j - 1;
  if (j >= n) j = 2 * n - 1 - j;
  return j;
}

__device__ __forceinline__ void bilin_tap(int o, int s, int n, int& a0, int& a1, float& f) {
  const int t = 2 * o + 1 - s;               // u = t / (2 s)
  int i0 = (t >= 0) ? t / (2 * s) : -((-t + 2 * s - 1) / (2 * s));
  f = (float)(t - i0 * 2 * s) / (float)(2 * s);
  int i1 = i0 + 1;
  if (i0 < 0) i0 = -i0;                      // mirror: -1 -> 1
  if (i1 > n - 1) i1 = 2 * (n - 1) - i1;     // mirror:  n -> n-2
  if (i1 < 0) i1 = 0;                        // n == 1
  a0 = i0; a1 = i1;
}

__device__ __forceinline__ int tile_of(int y, int size, int S, int n) {
  return (size % S != 0 && y >= size - S) ? n - 1 : y / S;
}

// [lo, hi) of the output coordinates along one axis whose last writer is tile t (the set where tile_of(y) == t): tile t
// starts at min(t * S, size - S), and the next tile's start ends it
__host__ __device__ inline void owned_span(int t, int size, int S, int n, int& lo, int& hi) {
  lo = t * S < size - S ? t * S : size - S;
  hi = t + 1 < n ? ((t + 1) * S < size - S ? (t + 1) * S : size - S) : size;
}

// image element -> float: exact for uint16 digital numbers (what GDAL hands s2_tiles_supres.py:311-315), so a
// uint16 image and its float32 copy prepare bit-identical inputs
__device__ __forceinline__ float ld_px(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_px(const uint16_t* p) { return (float)__ldg(p); }


}  // namespace dsen2
