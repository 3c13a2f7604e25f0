// Last layer of the network, Conv2D(cout, 3x3) + Add(last input) (DSen2Net.py:35,38,41), for the few output bands DSen2 has
// (6 at 20 m, 2 at 60 m): a tcgen05 GEMM with the roles of the operands SWAPPED.
//
// With pixels on the M side (conv_pair.cu) every one of the nine taps re-reads the whole activation tile from shared memory
// for an N = 32 MMA: 590 KB of A-operand reads per 128-pixel tile at 128 B/clk = 4608 clocks -- as long as a 128 -> 128 trunk
// layer for a quarter of a percent of its FLOPs (ncu: tensor pipe 37 %, shared-memory data path 82 %).  Here the WEIGHTS
// are the M side, all taps at once:
//     A (M = 128 rows)  row (tap * 2 + hl) * cout + c  = W_hl[tap][:, c]   (hl: fp16 hi / lo part of the fp32 kernel)
//     B (N = 192 rows)  the 18 x 10 pixel halo box of the tile, as it lies in shared memory after ONE TMA load
//     D[(tap, hl, c)][box pixel] = sum_k W_hl[tap][k, c] * x[box pixel][k]            (x = x_hi k-blocks, then x_lo k-blocks)
// so an activation element crosses the shared-memory read port once per k-step instead of nine times, 16 MMAs of M = 128,
// N = 192 per tile (1536 tensor clocks), and the 3x3 structure moves to the epilogue:
//     out[c][y, x] = sum_tap sum_hl D[(tap, hl, c)][(y + dy) * 10 + (x + dx)]
// a shifted gather over TMEM LANES, done through a shared-memory copy of the accumulator (thread = lane writes its row,
// thread = pixel gathers its 18 terms per band).  All four products (hi + lo) x (W_hi + W_lo) are kept: fp32-equivalent.
// The epilogue then adds bias and the global skip, scales, and writes NCHW predictions or the stitched HWC canvas with the
// last-writer-wins ownership of patches.py:394-403 (supres.py:29).
// Shared-memory port budget per tile (128 B/clk): MMA operands 160 KB + TMA fill 92 KB + accumulator copy 83 KB in, 55 KB
// out = 390 KB ~ 3100 clocks (was 590 + 92 KB); measured 28 ms per 10980^2 tile instead of 37, DRAM at 44-53 % of the copy
// peak (profiles/r02_tail_swapped_ncu.txt).  The global skip is loaded one tile ahead: as a dependent load inside the
// per-tile chain (wait, copy, barrier, gather, barrier) it cost a DRAM latency per tile (33 ms).
//
// One CTA per SM (cta_group::1), persistent over the tile list.  Warps 0-7 epilogue (two per TMEM lane quarter: half of the
// accumulator columns each on the way to shared memory, half of the output bands each in the gather), warp 8 TMA producer,
// warp 9 TMEM alloc + MMA issue; two TMEM accumulators of 192 columns.
#include "common.cuh"
#include "tiling.cuh"

namespace dsen2 {

static constexpr int kTBoxH = 18, kTBoxW = 10;
static constexpr int kTBoxBytes = kTBoxH * kTBoxW * 128;          // 23040: one 64-channel k-block of the halo box
static constexpr int kTStage = 23552;                              // rounded up to the 1 KB swizzle atom
static constexpr int kTN = 192;                                    // UMMA N: the 180 box pixels, padded (the 12 rows past the box
                                                                   // are whatever follows in shared memory; their columns are never read)
static constexpr int kTZPitch = 196;                               // floats per accumulator row in shared memory (16-byte stores, conflict-free)
static constexpr int kTZBytes = 128 * kTZPitch * 4;
static constexpr int kTEpiWarps = 8;                               // two per TMEM lane quarter
static constexpr int kTThreads = (kTEpiWarps + 2) * 32;
static constexpr int kTMaxCout = 7;                                // 9 taps * 2 * cout <= 128 rows

struct TailParams {
  int n, H, W;
  int tiles_x, tiles_y, tx0;          // tile columns [tx0, tx0 + tiles_x) of a patch (the stitching form skips the border columns)
  uint32_t num_tiles;
  const float* bias;
  const __half* skip_hi;              // prepared input x_in16 (n, H, W, 16): the global skip
  const __half* skip_lo;
  int skip_ch0, cout;
  float out_mul;
  // Instances with SCENES take the scene list in the fields of the single-canvas geometry they do not read (each scene's
  // canvas, size and grid are in its table entry): the struct stays at 128 bytes.  A larger parameter struct is read
  // through its address instead of with direct parameter loads, which changes the code of every other instance.
  union {
    void* out;                        // float, or (stitched canvas only) uint16_t: the OutT of the kernel instance
    const SceneGeom* scenes;          // SCENES: the scene table (num_scenes entries)
  };
  int tail_mode;                      // 0: NCHW (n, cout, H, W) predictions; 1: stitched HWC canvas
  int first_patch;
  union { int img_h; int num_scenes; };
  union { int img_w; int num_flat; };  // SCENES: entries of patch_scene, the flat patches of the list
  int border, grid_ny, grid_nx;
  union {
    const int* patch_ids;             // stitching form with IDS: batch entry b is patch patch_ids[b], not first_patch + b
    const int* patch_scene;           // SCENES: the scene of every flat patch
  };
  int avoid;                          // uint16 canvas: a value the network must not write (the nodata value), -1 none
  float add_offset;                   // instances with ADD: subtracted from every stitched value (the product's radiometric offset)
};
static_assert(sizeof(TailParams) == 128, "TailParams grew: see the comment on its unions");

// The uint16 (digital number) canvas value of the float f the float canvas receives: NaN -> 0, else rint(clip(f, 0, 65535))
// (round half to even; fmaxf returns 0 for a NaN f).  A value equal to `avoid` (>= 0) moves one step away from it, so a
// dark or negative network output never reads as nodata.
__device__ __forceinline__ uint16_t dn_of(float f, int avoid) {
  int q = (int)__float2uint_rn(fminf(fmaxf(f, 0.f), 65535.f));
  if (q == avoid) q = avoid == 65535 ? 65534 : q + 1;
  return (uint16_t)q;
}

__device__ __forceinline__ void store_out(float* o, float f, int) { *o = f; }
__device__ __forceinline__ void store_out(uint16_t* o, float f, int avoid) { *o = dn_of(f, avoid); }

template <int KPM>                     // 64-channel k-blocks per activation tensor: 2 (128 features) or 4 (256)
struct TailCfg {
  static constexpr int STAGES = KPM == 2 ? 4 : 2;
  static constexpr int W_BYTES = KPM * 16384;
  static constexpr int BAR_BYTES = 1024;
  static constexpr int SMEM_BYTES = W_BYTES + STAGES * kTStage + BAR_BYTES + kTZBytes + 1024 /*align slack*/;
  static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of shared memory a CTA can opt into");
};

__device__ __forceinline__ int tail_stitch_tile_of(int y, int size, int S, int n) {
  return (size % S != 0 && y >= size - S) ? n - 1 : y / S;
}

// CHIPS (stitching form): the canvas is a stack of same-size chip canvases (num_chips, img_h, img_w, cout) and
// first_patch + b indexes the flat list chip * ppc + patch (ppc = grid_ny * grid_nx); ownership stays inside the chip.
// SCENES (stitching form): first_patch + b indexes the flat patch list of a scene list; locate() resolves the tile's scene
// once (the map p.patch_scene, then its table entry) and writes into that scene's own canvas with its own geometry.
template <int KPM, bool IDS, typename OutT, bool ADD, bool CHIPS, bool SCENES>
__global__ void __launch_bounds__(kTThreads, 1)
conv_tail_swapped_kernel(const __grid_constant__ CUtensorMap tm_hi, const __grid_constant__ CUtensorMap tm_lo,
                         const __grid_constant__ CUtensorMap tm_w, const TailParams p) {
  using Cfg = TailCfg<KPM>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* s_w = smem;
  uint8_t* s_a = smem + Cfg::W_BYTES;
  uint8_t* bar_base = s_a + Cfg::STAGES * kTStage;
  uint64_t* full = reinterpret_cast<uint64_t*>(bar_base);
  uint64_t* empty = full + Cfg::STAGES;
  uint64_t* wfull = empty + Cfg::STAGES;
  uint64_t* tmem_full = wfull + 1;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
  float* s_bias = reinterpret_cast<float*>(bar_base + 512);
  float* s_z = reinterpret_cast<float*>(bar_base + Cfg::BAR_BYTES);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == kTEpiWarps && lane == 0) {
    tma_prefetch_desc(&tm_hi);
    tma_prefetch_desc(&tm_lo);
    tma_prefetch_desc(&tm_w);
    for (int i = 0; i < Cfg::STAGES; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(wfull, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], kTEpiWarps);        // one arrival per epilogue warp
    }
    mbar_fence_init();
  }
  if (warp == kTEpiWarps + 1) tmem_alloc<512>(tmem_ptr);
  if (threadIdx.x < 16) s_bias[threadIdx.x] = threadIdx.x < p.cout ? p.bias[threadIdx.x] : 0.f;
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr;

  if (warp == kTEpiWarps) {
    // ================================ TMA producer ================================
    if (elect_one()) {
      mbar_expect_tx(wfull, Cfg::W_BYTES);
      for (int kb = 0; kb < KPM; ++kb) tma_load_2d(s_w + kb * 16384, &tm_w, wfull, kb * 64, 0);
      int stage = 0;
      uint32_t phase = 0;
      for (uint32_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        const uint32_t row = tile / (uint32_t)p.tiles_x;
        const int tx = (int)(tile - row * (uint32_t)p.tiles_x) + p.tx0;
        const int b = (int)(row / (uint32_t)p.tiles_y), ty = (int)(row - (uint32_t)b * (uint32_t)p.tiles_y);
#pragma unroll 1
        for (int kb = 0; kb < 2 * KPM; ++kb) {
          mbar_wait(&empty[stage], phase ^ 1);
          mbar_expect_tx(&full[stage], kTBoxBytes);
          tma_load_4d(s_a + stage * kTStage, kb < KPM ? &tm_hi : &tm_lo, &full[stage], (kb % KPM) * 64, tx * 8 - 1, ty * 16 - 1, b);
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == kTEpiWarps + 1) {
    // ================================ MMA issuer ==================================
    if (elect_one()) {
      constexpr uint32_t idesc = umma_idesc_f16(128, kTN);
      mbar_wait(wfull, 0);
      tc_fence_after();
      int stage = 0, acc = 0;
      uint32_t phase = 0, acc_phase = 0;
      for (uint32_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
        mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * kTN);
#pragma unroll 1
        for (int kb = 0; kb < 2 * KPM; ++kb) {
          mbar_wait(&full[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(s_w) + (uint32_t)((kb % KPM) * 16384);
          const uint32_t sb = smem_u32(s_a) + (uint32_t)(stage * kTStage);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            umma_f16_ss(d_tmem, umma_desc_sw128(sa + k * 32), umma_desc_sw128(sb + k * 32), idesc, (uint32_t)((kb | k) != 0));
          umma_commit(&empty[stage]);
          if (kb == 2 * KPM - 1) umma_commit(&tmem_full[acc]);
          if (++stage == Cfg::STAGES) { stage = 0; phase ^= 1; }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ================================ epilogue (256 threads) ======================
    // phase 1: thread = (TMEM lane = accumulator row (tap, hl, c), half of the columns); phase 2: thread = (tile pixel, half
    // of the output bands)
    const int lane_row = (warp & 3) * 32 + lane, half = warp >> 2;
    const int rows_used = 18 * p.cout;
    const int pix_t = threadIdx.x & 127, yy = pix_t >> 3, xx = pix_t & 7;
    const int cper = (p.cout + 1) >> 1, c_lo = half * cper, c_hi = min(p.cout, c_lo + cper);   // this thread's bands
    const int hl_stride = p.cout * kTZPitch, tap_stride = 2 * hl_stride;
    int acc = 0;
    uint32_t acc_phase = 0;
    // Where a tile's pixel of this thread goes (and whether this patch owns it), and its global skip.  The skip is loaded
    // ONE TILE AHEAD: a dependent global load inside the per-tile chain (wait, copy, barrier, gather, barrier) would put
    // a DRAM latency on every tile -- measured: the tile took 4.4 us for 1.2 us of MMAs.
    // SCENES: `out` receives the canvas of the tile's scene (the other instances write into p.out)
    struct Dest { bool write; long long obase, ostride; };
    auto locate = [&](uint32_t tile, Dest& d, __half (&sk_hi)[(kTMaxCout + 1) / 2], __half (&sk_lo)[(kTMaxCout + 1) / 2],
                      OutT*& out) {
      const uint32_t rowi = tile / (uint32_t)p.tiles_x;
      const int tx = (int)(tile - rowi * (uint32_t)p.tiles_x) + p.tx0;
      const int b = (int)(rowi / (uint32_t)p.tiles_y), ty = (int)(rowi - (uint32_t)b * (uint32_t)p.tiles_y);
      const int y = ty * 16 + yy, x = tx * 8 + xx;
      d.write = tile < p.num_tiles && (b < p.n) && (y < p.H) && (x < p.W) && c_lo < c_hi;
      d.obase = 0; d.ostride = 0;
      if (d.write) {
        if (p.tail_mode == 0) {
          d.ostride = (long long)p.H * p.W;
          d.obase = (long long)b * p.cout * d.ostride + (long long)y * p.W + x;
        } else if constexpr (SCENES) {
          // a scene or patch index outside the table writes nothing
          const int S = p.H - 2 * p.border;
          const int patch = p.first_patch + b;
          const int sc = patch < p.num_flat ? __ldg(p.patch_scene + patch) : -1;
          d.write = sc >= 0 && sc < p.num_scenes;
          if (d.write) {
            const SceneGeom* g = p.scenes + sc;
            const int img_h = g->src[0].H, img_w = g->src[0].W, gny = g->tl.n_i, gnx = g->tl.n_j;
            const int q = patch - g->first;
            const int pty = q / gnx, ptx = q - pty * gnx;
            const int gy = min(pty * S, img_h - S) + y - p.border;
            const int gx = min(ptx * S, img_w - S) + x - p.border;
            d.write = q >= 0 && q < gny * gnx &&
                      y >= p.border && y < p.H - p.border && x >= p.border && x < p.W - p.border &&
                      tail_stitch_tile_of(gy, img_h, S, gny) == pty && tail_stitch_tile_of(gx, img_w, S, gnx) == ptx;
            d.ostride = 1;
            d.obase = ((long long)gy * img_w + gx) * p.cout;
            out = static_cast<OutT*>(g->canvas);
          }
        } else {
          const int S = p.H - 2 * p.border;
          int patch = IDS ? __ldg(p.patch_ids + b) : p.first_patch + b;
          long long chip_base = 0;                     // CHIPS: first element of the chip's canvas (64-bit)
          if constexpr (CHIPS) {
            const int chip = patch / (p.grid_ny * p.grid_nx);
            patch -= chip * (p.grid_ny * p.grid_nx);
            chip_base = (long long)chip * p.img_h * p.img_w * p.cout;
          }
          const int pty = patch / p.grid_nx, ptx = patch - pty * p.grid_nx;
          const int gy = min(pty * S, p.img_h - S) + y - p.border;
          const int gx = min(ptx * S, p.img_w - S) + x - p.border;
          d.write = (!IDS || (patch >= 0 && patch < p.grid_ny * p.grid_nx)) &&
                    y >= p.border && y < p.H - p.border && x >= p.border && x < p.W - p.border &&
                    tail_stitch_tile_of(gy, p.img_h, S, p.grid_ny) == pty && tail_stitch_tile_of(gx, p.img_w, S, p.grid_nx) == ptx;
          d.ostride = 1;
          d.obase = chip_base + ((long long)gy * p.img_w + gx) * p.cout;
        }
      }
      if (d.write) {
        const long long pix = ((long long)b * p.H + y) * p.W + x;
        const __half* sh = p.skip_hi + pix * 16 + p.skip_ch0 + c_lo;
        const __half* sl = p.skip_lo + pix * 16 + p.skip_ch0 + c_lo;
#pragma unroll
        for (int i = 0; i < (kTMaxCout + 1) / 2; ++i)
          if (c_lo + i < c_hi) { sk_hi[i] = __ldg(sh + i); sk_lo[i] = __ldg(sl + i); }
      }
    };
    Dest cur, nxt;
    OutT *cur_out = nullptr, *nxt_out = nullptr;
    __half ch[(kTMaxCout + 1) / 2], cl[(kTMaxCout + 1) / 2], nh[(kTMaxCout + 1) / 2], nl[(kTMaxCout + 1) / 2];
#pragma unroll
    for (int i = 0; i < (kTMaxCout + 1) / 2; ++i) ch[i] = cl[i] = nh[i] = nl[i] = __float2half_rn(0.f);
    locate(blockIdx.x, cur, ch, cl, cur_out);
    for (uint32_t tile = blockIdx.x; tile < p.num_tiles; tile += gridDim.x) {
      locate(tile + gridDim.x, nxt, nh, nl, nxt_out);                 // next tile's destination and skip loads, in flight during this tile
      const bool write = cur.write;
      const long long obase = cur.obase, ostride = cur.ostride;
      // ---- phase 1: accumulator rows -> shared memory
      mbar_wait(&tmem_full[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)(acc * kTN + half * (kTN / 2));
      const uint32_t zrow = smem_u32(s_z) + (uint32_t)((lane_row * kTZPitch + half * (kTN / 2)) * 4);
#pragma unroll 1
      for (int chunk = 0; chunk < kTN / 64; ++chunk) {
        uint32_t r[32];
        tmem_ld_32x32(taddr + chunk * 32, r);
        tmem_ld_wait();
        if (lane_row < rows_used) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            sts128(zrow + (uint32_t)((chunk * 32 + q * 4) * 4), make_uint4(r[4 * q], r[4 * q + 1], r[4 * q + 2], r[4 * q + 3]));
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tmem_empty[acc]);          // the TMEM buffer is free for the tile after next
      asm volatile("bar.sync 1, 256;" ::: "memory");          // all rows of this tile are in shared memory
      // ---- phase 2: gather the 18 terms of each band of this pixel, shifted by the tap offsets
      if (write) {
        const float* z0 = s_z + c_lo * kTZPitch + yy * kTBoxW + xx;     // band c_lo, tap (0, 0), W_hi row
#pragma unroll
        for (int i = 0; i < (kTMaxCout + 1) / 2; ++i) {
          if (c_lo + i < c_hi) {
            const float* z = z0 + i * kTZPitch;
            float vh = 0.f, vl = 0.f;
#pragma unroll
            for (int tap = 0; tap < 9; ++tap) {
              const int off = (tap / 3) * kTBoxW + (tap % 3);
              vh += z[tap * tap_stride + off];                 // W_hi row of this tap
              vl += z[tap * tap_stride + hl_stride + off];     // W_lo row
            }
            const float v = (vh + vl) + s_bias[c_lo + i];
            const float skip = __half2float(ch[i]) + __half2float(cl[i]);
            // Add (DSen2Net.py:38), x SCALE; ADD: - add_offset, back to the product's convention (__fsub_rn is never
            // contracted into an FMA with the multiply)
            store_out((SCENES ? cur_out : static_cast<OutT*>(p.out)) + obase + (c_lo + i) * ostride,
                      ADD ? __fsub_rn((v + skip) * p.out_mul, p.add_offset) : (v + skip) * p.out_mul, p.avoid);
          }
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");          // the shared-memory copy may be overwritten
      cur = nxt;
      cur_out = nxt_out;
#pragma unroll
      for (int i = 0; i < (kTMaxCout + 1) / 2; ++i) { ch[i] = nh[i]; cl[i] = nl[i]; }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }

  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (warp == kTEpiWarps + 1) tmem_dealloc<512>(tmem_base);
}

// tail weights for the swapped form: [128 rows: (tap * 2 + hl) * cout + c][F channels] fp16, K-major; unused rows zero
__global__ void pack_tail16_weights_kernel(const float* __restrict__ hwio, int F, int cout, long long total, __half* __restrict__ out) {
  for (long long idx = blockIdx.x * (long long)blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(idx % F);
    const int r = (int)(idx / F);
    __half v = __float2half_rn(0.f);
    if (r < 18 * cout) {
      const int g = r / cout, c = r - g * cout;
      const int tap = g >> 1, hl = g & 1;
      const float w = hwio[((long long)tap * F + k) * cout + c];
      const __half hi = __float2half_rn(w);
      v = hl == 0 ? hi : __float2half_rn(w - __half2float(hi));
    }
    out[idx] = v;
  }
}

template <int KPM, bool IDS, typename OutT, bool ADD, bool CHIPS, bool SCENES>
static int launch_tail(const TailParams& p, const void* d_x_hi, const void* d_x_lo, const void* d_w, int sms, cudaStream_t stream) {
  using Cfg = TailCfg<KPM>;
  static bool configured[64] = {};
  if (needs_config(configured)) {
    DSEN2_CUDA(cudaFuncSetAttribute(conv_tail_swapped_kernel<KPM, IDS, OutT, ADD, CHIPS, SCENES>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
  }
  const int F = KPM * 64;
  CUtensorMap hi, lo, w;
  const uint64_t dims[4] = {(uint64_t)F, (uint64_t)p.W, (uint64_t)p.H, (uint64_t)p.n};
  const uint32_t box[4] = {64, (uint32_t)kTBoxW, (uint32_t)kTBoxH, 1};
  int rc = make_tmap_f16_sw(&hi, d_x_hi, 4, dims, box, 128);
  if (rc) return rc;
  if ((rc = make_tmap_f16_sw(&lo, d_x_lo, 4, dims, box, 128)) != 0) return rc;
  const uint64_t wd[2] = {(uint64_t)F, 128};
  const uint32_t wb[2] = {64, 128};
  if ((rc = make_tmap_f16_sw(&w, d_w, 2, wd, wb, 128)) != 0) return rc;
  const int grid = (int)(p.num_tiles < (uint32_t)sms ? p.num_tiles : (uint32_t)sms);
  conv_tail_swapped_kernel<KPM, IDS, OutT, ADD, CHIPS, SCENES><<<grid, kTThreads, Cfg::SMEM_BYTES, stream>>>(hi, lo, w, p);
  return check_launch("conv_tail_swapped");
}

template <bool IDS, typename OutT, bool ADD, bool CHIPS = false, bool SCENES = false>
static int launch_tail_f(const TailParams& p, int features, const void* d_x_hi, const void* d_x_lo, const void* d_w, int sms,
                         cudaStream_t stream) {
  return features == 256 ? launch_tail<4, IDS, OutT, ADD, CHIPS, SCENES>(p, d_x_hi, d_x_lo, d_w, sms, stream)
                         : launch_tail<2, IDS, OutT, ADD, CHIPS, SCENES>(p, d_x_hi, d_x_lo, d_w, sms, stream);
}

// add: run the ADD instances, which subtract p.add_offset from every stitched value; chips: the CHIPS instances (range form);
// scenes: the SCENES instances (range form), with p.scenes and p.patch_scene set and no d_out (the canvases are in the table)
template <typename OutT>
static int tail16_common(TailParams& p, int features, const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                         const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int n, int H, int W, OutT* d_out,
                         bool add, void* stream, bool chips = false, bool scenes = false) {
  DSEN2_REQUIRE(d_x_hi && d_x_lo && d_w && d_bias && d_xin_hi && d_xin_lo && (scenes || d_out), DSEN2_E_BADARG,
                "dsen2_conv_tail16: null pointer");
  DSEN2_REQUIRE(features == 128 || features == 256, DSEN2_E_BADARG, "dsen2_conv_tail16: feature_size must be 128 or 256 (got %d)",
                features);
  DSEN2_REQUIRE(n >= 0 && H > 0 && W > 0 && cout > 0 && cout <= kTMaxCout && skip_ch0 >= 0 && skip_ch0 + cout <= 16, DSEN2_E_BADARG,
                "dsen2_conv_tail16: bad shape (cout %d of at most %d, skip_ch0 %d)", cout, kTMaxCout, skip_ch0);
  DSEN2_REQUIRE(((uintptr_t)d_x_hi % 16) == 0 && ((uintptr_t)d_x_lo % 16) == 0 && ((uintptr_t)d_w % 16) == 0, DSEN2_E_ALIGN,
                "dsen2_conv_tail16: pointers must be 16-byte aligned");
  if (n == 0) return 0;
  int sms = 0;
  int rc = device_sm_count_and_check(&sms);
  if (rc) return rc;
  p.n = n; p.H = H; p.W = W;
  p.tiles_x = ceil_div(W, 8);
  p.tiles_y = ceil_div(H, 16);
  p.tx0 = 0;
  if (p.tail_mode == 1) {
    // recompose_images copies only [border, P - border) of every patch (patches.py:402): tile columns that lie inside the
    // border produce nothing -- leave them out of the tile list (P 128 / border 8: 14 of 16 columns)
    p.tx0 = p.border / 8;
    p.tiles_x = (W - p.border - 1) / 8 - p.tx0 + 1;
  }
  const long long tiles = (long long)n * p.tiles_x * p.tiles_y;
  DSEN2_REQUIRE(tiles < (1LL << 31), DSEN2_E_BADARG, "dsen2_conv_tail16: batch too large (%lld tiles)", tiles);
  p.num_tiles = (uint32_t)tiles;
  p.bias = d_bias;
  p.skip_hi = (const __half*)d_xin_hi; p.skip_lo = (const __half*)d_xin_lo; p.skip_ch0 = skip_ch0;
  p.cout = cout;
  if (!scenes) p.out = d_out;
  const cudaStream_t st = (cudaStream_t)stream;
  if (scenes)
    return add ? launch_tail_f<false, OutT, true, false, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st)
               : launch_tail_f<false, OutT, false, false, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st);
  if (chips)
    return add ? launch_tail_f<false, OutT, true, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st)
               : launch_tail_f<false, OutT, false, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st);
  if (p.patch_ids)
    return add ? launch_tail_f<true, OutT, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st)
               : launch_tail_f<true, OutT, false>(p, features, d_x_hi, d_x_lo, d_w, sms, st);
  return add ? launch_tail_f<false, OutT, true>(p, features, d_x_hi, d_x_lo, d_w, sms, st)
             : launch_tail_f<false, OutT, false>(p, features, d_x_hi, d_x_lo, d_w, sms, st);
}

}  // namespace dsen2

using namespace dsen2;

extern "C" int dsen2_pack_tail16_weights(const float* d_hwio, int feature_size, int cout, void* d_packed, void* stream) {
  DSEN2_REQUIRE(d_hwio && d_packed, DSEN2_E_BADARG, "dsen2_pack_tail16_weights: null pointer");
  DSEN2_REQUIRE(cout > 0 && cout <= kTMaxCout && feature_size > 0 && feature_size % 64 == 0, DSEN2_E_BADARG,
                "dsen2_pack_tail16_weights: at most %d output bands (got %d), feature_size a multiple of 64", kTMaxCout, cout);
  const long long total = 128LL * feature_size;
  const int block = 256;
  pack_tail16_weights_kernel<<<grid_for(total, block), block, 0, (cudaStream_t)stream>>>(d_hwio, feature_size, cout, total,
                                                                                         (__half*)d_packed);
  return check_launch("pack_tail16_weights");
}

extern "C" int dsen2_conv_tail16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                 const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size, int n,
                                 int H, int W, float* d_pred_nchw, void* stream) {
  TailParams p{};
  p.tail_mode = 0;
  p.out_mul = 1.0f;
  p.avoid = -1;
  return tail16_common<float>(p, feature_size, d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, n, H, W, d_pred_nchw,
                       false, stream);
}

// the stitching form: patches first_patch + b, or d_patch_ids[b] when d_patch_ids is not null; float or uint16 canvas;
// with add, add_offset is subtracted from every value after the scale.  num_chips >= 0: the canvas is a stack of num_chips
// chip canvases and first_patch + b indexes their flat patch list (no id list); -1: one canvas.
template <typename OutT>
static int tail16_stitch(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias, const void* d_xin_hi,
                         const void* d_xin_lo, int skip_ch0, int cout, int feature_size, int n, int P, int first_patch,
                         const int* d_patch_ids, int border, int img_h, int img_w, float mul, int avoid, OutT* d_canvas,
                         void* stream, bool add = false, float add_offset = 0.f, int num_chips = -1) {
  const int S = P - 2 * border;
  DSEN2_REQUIRE(P > 0 && border >= 0 && S > 0 && img_h >= S && img_w >= S && first_patch >= 0, DSEN2_E_BADARG,
                "dsen2_conv_tail16_stitch: bad stitch geometry (P %d border %d image %dx%d)", P, border, img_h, img_w);
  DSEN2_REQUIRE(avoid >= -1 && avoid <= 65535, DSEN2_E_BADARG, "dsen2_conv_tail16_stitch: avoid %d outside [-1, 65535]", avoid);
  TailParams p{};
  p.tail_mode = 1;
  p.out_mul = mul;
  p.avoid = avoid;
  p.add_offset = add_offset;
  p.first_patch = first_patch; p.img_h = img_h; p.img_w = img_w; p.border = border;
  p.grid_ny = ceil_div(img_h, S); p.grid_nx = ceil_div(img_w, S);
  p.patch_ids = d_patch_ids;
  if (num_chips >= 0) {
    const long long flat = (long long)num_chips * p.grid_ny * p.grid_nx;
    DSEN2_REQUIRE(!d_patch_ids && n >= 0 && flat < (1LL << 31) && (long long)first_patch + n <= flat, DSEN2_E_BADARG,
                  "dsen2_conv_tail16_stitch_chips: patch range [%d,%lld) outside the %lld patches of %d chips", first_patch,
                  (long long)first_patch + n, flat, num_chips);
  } else {
    DSEN2_REQUIRE(d_patch_ids || first_patch + n <= p.grid_ny * p.grid_nx, DSEN2_E_BADARG,
                  "dsen2_conv_tail16_stitch: patch range [%d,%d) exceeds the %d tiles of the canvas", first_patch,
                  first_patch + n, p.grid_ny * p.grid_nx);
  }
  return tail16_common<OutT>(p, feature_size, d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, n, P, P,
                             d_canvas, add, stream, num_chips >= 0);
}

extern "C" int dsen2_conv_tail16_stitch(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                        const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout, int feature_size,
                                        int n, int P, int first_patch, int border, int img_h, int img_w, float mul,
                                        float* d_canvas, void* stream) {
  return tail16_stitch<float>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P,
                              first_patch, nullptr, border, img_h, img_w, mul, -1, d_canvas, stream);
}

extern "C" int dsen2_conv_tail16_stitch_ids(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                            const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                            int feature_size, int n, int P, const int* d_patch_ids, int border, int img_h,
                                            int img_w, float mul, float* d_canvas, void* stream) {
  DSEN2_REQUIRE(d_patch_ids, DSEN2_E_BADARG, "dsen2_conv_tail16_stitch_ids: null pointer");
  return tail16_stitch<float>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P, 0,
                              d_patch_ids, border, img_h, img_w, mul, -1, d_canvas, stream);
}

extern "C" int dsen2_conv_tail16_stitch_u16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                            const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                            int feature_size, int n, int P, int first_patch, int border, int img_h,
                                            int img_w, float mul, int avoid, uint16_t* d_canvas, void* stream) {
  return tail16_stitch<uint16_t>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P,
                                 first_patch, nullptr, border, img_h, img_w, mul, avoid, d_canvas, stream);
}

extern "C" int dsen2_conv_tail16_stitch_ids_u16(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                                const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                                int feature_size, int n, int P, const int* d_patch_ids, int border,
                                                int img_h, int img_w, float mul, int avoid, uint16_t* d_canvas,
                                                void* stream) {
  DSEN2_REQUIRE(d_patch_ids, DSEN2_E_BADARG, "dsen2_conv_tail16_stitch_ids_u16: null pointer");
  return tail16_stitch<uint16_t>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P, 0,
                                 d_patch_ids, border, img_h, img_w, mul, avoid, d_canvas, stream);
}

extern "C" int dsen2_conv_tail16_stitch_offset(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                               const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                               int feature_size, int n, int P, int first_patch, const int* d_patch_ids,
                                               int border, int img_h, int img_w, float mul, float add_offset,
                                               int canvas_dtype, int avoid, void* d_canvas, void* stream) {
  DSEN2_REQUIRE(isfinite(add_offset), DSEN2_E_BADARG, "dsen2_conv_tail16_stitch_offset: add_offset must be finite");
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_F32 || canvas_dtype == DSEN2_IMG_U16, DSEN2_E_BADARG,
                "dsen2_conv_tail16_stitch_offset: canvas_dtype must be DSEN2_IMG_F32 or DSEN2_IMG_U16 (got %d)", canvas_dtype);
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_U16 || avoid == -1, DSEN2_E_BADARG,
                "dsen2_conv_tail16_stitch_offset: avoid must be -1 for a float canvas (got %d)", avoid);
  const int first = d_patch_ids ? 0 : first_patch;
  if (canvas_dtype == DSEN2_IMG_U16)
    return tail16_stitch<uint16_t>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P,
                                   first, d_patch_ids, border, img_h, img_w, mul, avoid, (uint16_t*)d_canvas, stream, true,
                                   add_offset);
  return tail16_stitch<float>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P, first,
                              d_patch_ids, border, img_h, img_w, mul, -1, (float*)d_canvas, stream, true, add_offset);
}

extern "C" int dsen2_conv_tail16_stitch_chips(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                              const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                              int feature_size, int n, int P, int first_patch, int border, int num_chips,
                                              int img_h, int img_w, float mul, int add, float add_offset, int canvas_dtype,
                                              int avoid, void* d_canvas, void* stream) {
  const char* name = "dsen2_conv_tail16_stitch_chips";
  DSEN2_REQUIRE(num_chips >= 0, DSEN2_E_BADARG, "%s: num_chips %d < 0", name, num_chips);
  DSEN2_REQUIRE(add == 0 || add == 1, DSEN2_E_BADARG, "%s: add must be 0 or 1 (got %d)", name, add);
  DSEN2_REQUIRE(!add || isfinite(add_offset), DSEN2_E_BADARG, "%s: add_offset must be finite", name);
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_F32 || canvas_dtype == DSEN2_IMG_U16, DSEN2_E_BADARG,
                "%s: canvas_dtype must be DSEN2_IMG_F32 or DSEN2_IMG_U16 (got %d)", name, canvas_dtype);
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_U16 || avoid == -1, DSEN2_E_BADARG,
                "%s: avoid must be -1 for a float canvas (got %d)", name, avoid);
  const float a = add ? add_offset : 0.f;
  if (canvas_dtype == DSEN2_IMG_U16)
    return tail16_stitch<uint16_t>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P,
                                   first_patch, nullptr, border, img_h, img_w, mul, avoid, (uint16_t*)d_canvas, stream,
                                   add != 0, a, num_chips);
  return tail16_stitch<float>(d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, feature_size, n, P,
                              first_patch, nullptr, border, img_h, img_w, mul, -1, (float*)d_canvas, stream, add != 0, a,
                              num_chips);
}

extern "C" int dsen2_conv_tail16_stitch_scenes(const void* d_x_hi, const void* d_x_lo, const void* d_w, const float* d_bias,
                                               const void* d_xin_hi, const void* d_xin_lo, int skip_ch0, int cout,
                                               int feature_size, int n, int P, int first_patch, int border,
                                               const void* d_table, const int* d_patch_scene, int num_scenes,
                                               long long total_patches, float mul, int add, float add_offset,
                                               int canvas_dtype, int avoid, void* stream) {
  const char* name = "dsen2_conv_tail16_stitch_scenes";
  DSEN2_REQUIRE(d_table && d_patch_scene, DSEN2_E_BADARG, "%s: null pointer", name);
  DSEN2_REQUIRE(num_scenes >= 0, DSEN2_E_BADARG, "%s: num_scenes %d < 0", name, num_scenes);
  DSEN2_REQUIRE(add == 0 || add == 1, DSEN2_E_BADARG, "%s: add must be 0 or 1 (got %d)", name, add);
  DSEN2_REQUIRE(!add || isfinite(add_offset), DSEN2_E_BADARG, "%s: add_offset must be finite", name);
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_F32 || canvas_dtype == DSEN2_IMG_U16, DSEN2_E_BADARG,
                "%s: canvas_dtype must be DSEN2_IMG_F32 or DSEN2_IMG_U16 (got %d)", name, canvas_dtype);
  DSEN2_REQUIRE(canvas_dtype == DSEN2_IMG_U16 || avoid == -1, DSEN2_E_BADARG,
                "%s: avoid must be -1 for a float canvas (got %d)", name, avoid);
  DSEN2_REQUIRE(avoid >= -1 && avoid <= 65535, DSEN2_E_BADARG, "%s: avoid %d outside [-1, 65535]", name, avoid);
  const int S = P - 2 * border;
  DSEN2_REQUIRE(P > 0 && border >= 0 && S > 0, DSEN2_E_BADARG, "%s: bad stitch geometry (P %d border %d)", name, P, border);
  DSEN2_REQUIRE(total_patches >= 0 && total_patches < (1LL << 31) && first_patch >= 0 && n >= 0 &&
                (long long)first_patch + n <= total_patches, DSEN2_E_BADARG,
                "%s: patch range [%d,%lld) outside the %lld patches of %d scenes", name, first_patch,
                (long long)first_patch + n, total_patches, num_scenes);
  TailParams p{};
  p.tail_mode = 1;
  p.out_mul = mul;
  p.avoid = avoid;
  p.add_offset = add ? add_offset : 0.f;
  p.first_patch = first_patch; p.border = border;
  p.scenes = static_cast<const SceneGeom*>(d_table);
  p.patch_scene = d_patch_scene;
  p.num_scenes = num_scenes; p.num_flat = (int)total_patches;
  if (canvas_dtype == DSEN2_IMG_U16)
    return tail16_common<uint16_t>(p, feature_size, d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, n, P, P,
                                   nullptr, add != 0, stream, false, true);
  return tail16_common<float>(p, feature_size, d_x_hi, d_x_lo, d_w, d_bias, d_xin_hi, d_xin_lo, skip_ch0, cout, n, P, P,
                              nullptr, add != 0, stream, false, true);
}
