// ms_fused.cu -- the throughput path: MS feature volume [N][8][D][h][w] straight from
// the uint8 pair, no intermediate cost volumes except the sadsob scratch.
//
// Replaces, in one pass, get_costs (census + nccNister + zsad + sobel/sadsob +
// 3x swap_axes + border crop, cbmv_generator.py:27-79) and extract_features_left
// (clip/normalise, 4x extract_likelihood, float64 scratch, transpose + cast,
// cbmv_generator.py:258-308) for the default windows 11/3/5/5.
//
// Launch sequence (all on one stream):
//   1. ms_prep_kernel    per padded pixel of every image: census code (4x u32), ZSAD
//                        window mean, NCC window sum A and fp64 C = 1/sqrt(9B - A^2),
//                        float copy of the pixel, Sobel response.
//   2. sadsob vband+scan (sadsob.cu) -> raw SAD-of-Sobel volume [N][D][H][W]; its fp32
//                        summed-area table needs whole-row sequential scans, so it
//                        cannot live inside an x-tile.
//   3. ms_fused_kernel   one CTA = one output row y x 32 pixels x ALL D:
//        stage    right-image row data (census codes, stats, 5 float rows) and the tile's
//                 SAD-of-Sobel costs stream into shared memory through TMA (cp.async.bulk /
//                 cp.async.bulk.tensor; LDGSTS fallback for D > 256).
//        phase 1  8 warps split D; lane = pixel.  Per (pixel, d): census popcount, NCC (9 fp32
//                 products of exact integers, fp64 scaling), ZSAD over a register-resident
//                 right window that slides with d -- two disparities at a time with packed
//                 FADD2, every add still an IEEE fp32 add in the reference's order; raw costs
//                 are parked in shared memory (13 B/voxel: three floats + census byte);
//                 per-pixel minima.
//        phase 2  warp-specialised, both halves only READ the parked costs:
//                 warps 0-3: one thread per (pixel, matcher) adds the AML denominator in
//                 d order (the reference's sequential fp32 sum, featextract.cpp:444-447);
//                 warps 4-7: thread = (pixel quad, d): channels 0-3 normalised and stored
//                 as 128-bit row segments.
//        phase 3  channels 4-7 = exp(-(c-m)^2/sigma) / den, 128-bit row segments.
//
// Bounding resource: HBM writes (32 B per voxel), co-limited by the FP32 pipe -- ZSAD alone is
// 75 ordered adds per voxel -- and by shared-memory/LSU traffic (DESIGN.md has the arithmetic).
#include "ms_fused.cuh"

#include <cuda.h>
#include <cuda_bf16.h>
#include <stdlib.h>

#include <mutex>
#include <vector>

#include "feature_math.cuh"

namespace msn {

namespace {

constexpr int kTileMax = 32;  // widest tile (pixels per CTA) the geometry allows for
constexpr int kGroups = 8;    // d-groups per tile: a phase-1 thread owns (pixel, d-group)
constexpr int kSlack = 24;    // right-image columns left of X-(D-1) that dummy steps (d >= D) may read: groups*DC - D < 2*groups
constexpr int kPadT = 2;      // padded rows above/below (ZSAD halo)
constexpr int kPadR = 40;     // padded columns to the right (tile overhang + halo)
constexpr int kCensW = 11, kNccW = 3, kSadW = 5;
constexpr int kMaxFusedD = 448;

struct __align__(16) RStat {
  float mean;  // ZSAD window mean (matchers.cpp:482)
  float A;     // NCC window sum, exact integer <= 2295 (matchers.cpp:140)
  double C;    // 1/sqrt(9*B - A*A) in fp64 (matchers.cpp:146)
};

struct FusedGeom {
  int N, H, W, h, w, bh, bwl;   // h: output rows of THIS launch (a row band when y0 / row_count are set)
  int y0;   // first cropped-image row of the band (0 unless the caller shards a frame by rows)
  int D;    // disparities handled by this launch: [d0, d0 + D)
  int d0;   // first disparity (> 0 only for a disparity slab, SURVEY.md 8e)
  int d_inner;  // SAD-of-Sobel scratch layout: 0 [N][Dl][H][Ws], 1 [N][H][Dl][Ws] (sub-slab launches, see sadsob.cu)
  int Dl;   // disparities of the whole launch (= D unless the launch is cut into sub-slabs, kModeXchg)
  int Hp, Wp, padL;
  int sxo, Ws;   // SAD-of-Sobel scratch: column offset and row pitch (tile starts land on 16 B)
  int lr;        // both views (p->lr): the right-view tiles slide the LEFT window rightwards, so the planes carry
                 // D + slack padded columns on the right as well, and the left image's statistics get planes too
  __host__ __device__ size_t img_px() const { return (size_t)Hp * Wp; }
};

FusedGeom make_geom(int N, int H, int W, const msn_ms_params* p) {
  FusedGeom g;
  g.N = N; g.H = H; g.W = W;
  g.d0 = p->d_count > 0 ? p->d_begin : 0;
  g.D = p->d_count > 0 ? p->d_count : p->ndisp;
  g.Dl = g.D; g.d_inner = 0;
  g.bh = p->board_h; g.bwl = p->board_w_left;
  g.h = p->row_count > 0 ? p->row_count : H - 2 * p->board_h;
  g.y0 = p->row_count > 0 ? p->row_begin : 0;
  g.w = W - p->board_w_left - p->board_w_right;
  g.padL = (g.d0 + g.D + 1 + kSlack + 8 + 7) & ~7;  // d0+D-1 columns of disparity + dummy-step slack + halo/alignment
  g.Hp = H + 2 * kPadT;
  g.lr = p->lr ? 1 : 0;
  g.Wp = (W + g.padL + (g.lr ? g.D + kSlack + kPadR + 16 : kPadR) + 3) & ~3;
  g.sxo = (4 - (g.bwl & 3)) & 3;            // x0 + bwl + sxo is a multiple of 4 for every tile
  g.Ws = sadsob_fast_pitch(W + g.sxo + kTileMax);  // compile-time pitch of the scan kernels (0: too wide)
  return g;
}

struct FusedWs {
  uint4* desc[2];
  RStat* stat[2];   // [1] (right image) is only read through the planes below
  float* fimg[2];
  float* sob[2];
  float* meanR;    // right image: ZSAD window means as a plain float plane
  float* AR;       // right image: NCC window sums A as a plain float plane
  double* CR;      // right image: NCC 1/sqrt(9B - A^2) as a plain double plane
  float* meanL;    // left image: the same three planes (both views only: the right-view tiles read them per column)
  float* AL;
  double* CL;
  float* first4;   // [N][4] raw costs of cropped voxel (0,0,0): what get_right_cost fills with (featextract.cpp:151)
  float* luts;     // [128] census AML exponentials + [256] census byte -> channel 0
  float* sadsob;   // [N][D][H][Ws], or [N][H][D][Ws] (FusedGeom::d_inner)
  void* sad_ws;
  size_t total;
  void carve(char* base, const FusedGeom& g) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char* q = base ? base + off : nullptr; off += (bytes + 255) & ~(size_t)255; return q; };
    const size_t np = (size_t)g.N * g.img_px();
    for (int i = 0; i < 2; ++i) desc[i] = (uint4*)take(np * sizeof(uint4));
    for (int i = 0; i < 2; ++i) stat[i] = (RStat*)take(np * sizeof(RStat));
    for (int i = 0; i < 2; ++i) fimg[i] = (float*)take(np * sizeof(float));
    for (int i = 0; i < 2; ++i) sob[i] = (float*)take((size_t)g.N * (g.H + kSadRowPad) * g.Ws * sizeof(float));  // zero padded
    meanR = (float*)take((np + 16) * sizeof(float));
    AR = (float*)take((np + 16) * sizeof(float));
    CR = (double*)take((np + 16) * sizeof(double));
    meanL = AL = first4 = nullptr; CL = nullptr;
    if (g.lr) {
      meanL = (float*)take((np + 16) * sizeof(float));
      AL = (float*)take((np + 16) * sizeof(float));
      CL = (double*)take((np + 16) * sizeof(double));
      first4 = (float*)take((size_t)g.N * 4 * sizeof(float));
    }
    luts = (float*)take(384 * sizeof(float));
    sadsob = (float*)take((size_t)g.N * g.Dl * g.H * g.Ws * sizeof(float) + 256);
    sad_ws = take(sadsob_workspace_bytes_n(g.N, g.H, g.W, g.Dl, kSadW));
    total = off;
  }
};

// ------------------------------------------------------------------ prep --
// grid (ceil(Wp/128), Hp, 2N); blockIdx.z = 2*n + side.
__global__ void __launch_bounds__(128)
ms_prep_kernel(const uint8_t* __restrict__ left, const uint8_t* __restrict__ right, FusedGeom g,
               uint4* __restrict__ descL, uint4* __restrict__ descR, RStat* __restrict__ statL,
               RStat* __restrict__ statR, float* __restrict__ fL, float* __restrict__ fR,
               float* __restrict__ sobL, float* __restrict__ sobR, float* __restrict__ meanR,
               float* __restrict__ AR, double* __restrict__ CR, float* __restrict__ meanL,
               float* __restrict__ AL, double* __restrict__ CL, float* __restrict__ luts, float k_cen) {
  if (blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0) {
    // tables for the fused kernel: census AML exponentials exp(-(k^2)/sigma), k = 0..120, and the
    // channel-0 value k/120 of a parked census byte (a true IEEE division; 255 = no cost ->
    // clip(fill, 0, 120)/120 = 1)
    for (int kk = threadIdx.x; kk < 256; kk += blockDim.x) {
      if (kk < 128) luts[kk] = (kk <= 120) ? aml_e((float)kk, 0.f, k_cen) : 0.f;   // (either AML mode)
      luts[128 + kk] = (kk <= 120) ? __fdiv_rn((float)kk, 120.0f) : 1.0f;
    }
  }
  const int xp = blockIdx.x * blockDim.x + threadIdx.x;
  const int yp = blockIdx.y;
  const int n = blockIdx.z >> 1, side = blockIdx.z & 1;
  if (xp >= g.Wp) return;
  const int H = g.H, W = g.W;
  // A row band (the caller shards a frame by rows): the tiles only read padded rows [y0 + bh, y0 + bh + h + 3]
  // (the band's rows and the ZSAD halo); every other row only feeds the SAD-of-Sobel table, whose scan walks down
  // from row 0 -- and nothing below the band's last scan band is read at all.
  const bool feat_row = yp >= g.y0 + g.bh && yp <= g.y0 + g.bh + g.h + 2 * kPadT - 1;
  if (!feat_row) {
    const int Xs = xp - g.padL, Ys = yp - kPadT;
    if (Ys < 0 || Ys >= H || Xs < 0 || Xs >= W || Ys > g.y0 + g.bh + g.h + 64) return;   // (the last scan band reads up to 59 rows past the band)
    const uint8_t* im = (side ? right : left) + (size_t)n * H * W;
    float sv = 0.f;
    if (Ys >= 1 && Ys < H - 2 && Xs >= 1 && Xs < W - 2) {
      const uint8_t* p = im + (size_t)(Ys - 1) * W + (Xs - 1);
      sv = (float)(((int)p[2] - (int)p[0]) + 2 * ((int)p[W + 2] - (int)p[W]) + ((int)p[2 * W + 2] - (int)p[2 * W]));
    }
    (side ? sobR : sobL)[(size_t)n * (H + kSadRowPad) * g.Ws + (size_t)Ys * g.Ws + Xs] = sv;
    return;
  }
  const uint8_t* img = (side ? right : left) + (size_t)n * H * W;
  const int X = xp - g.padL, Y = yp - kPadT;
  const bool inside = (X >= 0 && X < W && Y >= 0 && Y < H);
  const size_t po = (size_t)n * g.img_px() + (size_t)yp * g.Wp + xp;

  uint32_t w0 = 0, w1 = 0, w2 = 0, w3 = 0;
  RStat st;
  st.mean = 0.f; st.A = 0.f; st.C = 0.0;
  float pix = 0.f;
  if (inside) {
    const int c = img[(size_t)Y * W + X];
    pix = (float)c;
    // census 11x11: bit k = a*11+b set iff centre < tap (matchers.cpp:290-297)
    if (Y >= 5 && Y < H - 6 && X >= 5 && X < W - 6) {
      const uint8_t* org = img + (size_t)(Y - 5) * W + (X - 5);
      uint32_t words[4] = {0u, 0u, 0u, 0u};
#pragma unroll
      for (int a = 0; a < kCensW; ++a) {
#pragma unroll
        for (int b = 0; b < kCensW; ++b) {
          const int bit = a * kCensW + b;
          const uint32_t v = (c < (int)__ldg(org + (size_t)a * W + b)) ? 1u : 0u;
          words[bit >> 5] |= v << (bit & 31);
        }
      }
      w0 = words[0]; w1 = words[1]; w2 = words[2]; w3 = words[3];
    }
    // ZSAD 5x5 mean: exact integer sum, one IEEE division (matchers.cpp:472-485)
    if (Y >= 2 && Y < H - 3 && X >= 2 && X < W - 3) {
      const uint8_t* org = img + (size_t)(Y - 2) * W + (X - 2);
      int sum = 0;
#pragma unroll
      for (int a = 0; a < kSadW; ++a)
#pragma unroll
        for (int b = 0; b < kSadW; ++b) sum += __ldg(org + (size_t)a * W + b);
      st.mean = __fdiv_rn((float)sum, 25.0f);
    }
    // NCC 3x3: A, and C in fp64 exactly as matchers.cpp:146
    if (Y >= 1 && Y < H - 2 && X >= 1 && X < W - 2) {
      const uint8_t* org = img + (size_t)(Y - 1) * W + (X - 1);
      unsigned a_sum = 0, b_sum = 0;
#pragma unroll
      for (int a = 0; a < kNccW; ++a)
#pragma unroll
        for (int b = 0; b < kNccW; ++b) {
          const unsigned v = __ldg(org + (size_t)a * W + b);
          a_sum += v;
          b_sum += v * v;
        }
      st.A = (float)a_sum;
      const double var = __dsub_rn((double)(9u * b_sum), __dmul_rn((double)a_sum, (double)a_sum));
      st.C = __ddiv_rn(1.0, __dsqrt_rn(var));
    }
    // Sobel Gx (matchers.cpp:538-547); unpadded array feeds the sadsob scan
    float sv = 0.f;
    if (Y >= 1 && Y < H - 2 && X >= 1 && X < W - 2) {
      const uint8_t* p = img + (size_t)(Y - 1) * W + (X - 1);
      sv = (float)(((int)p[2] - (int)p[0]) + 2 * ((int)p[W + 2] - (int)p[W]) +
                   ((int)p[2 * W + 2] - (int)p[2 * W]));
    }
    (side ? sobR : sobL)[(size_t)n * (H + kSadRowPad) * g.Ws + (size_t)Y * g.Ws + X] = sv;
  }
  (side ? descR : descL)[po] = make_uint4(w0, w1, w2, w3);
  (side ? statR : statL)[po] = st;
  (side ? fR : fL)[po] = pix;
  if (side) {
    // the fused kernel reads the right image's statistics lane-per-column: separate planes keep
    // those shared loads free of bank conflicts (a 16-byte struct per column is a 4-way conflict)
    meanR[po] = st.mean;
    AR[po] = st.A;
    CR[po] = st.C;
  } else if (meanL) {   // both views: the right-view tiles read the left image the same way
    meanL[po] = st.mean;
    AL[po] = st.A;
    CL[po] = st.C;
  }
}

// ----------------------------------------------------------------- fused --
constexpr int kMaxRanks = 8;
constexpr int kXLineWords = 32, kXLines = 5;   // 128 values travel as 5 lines of 31 values + 1 flag word
struct FusedXchg {
  unsigned* peer[kMaxRanks];   // table of every (physical) rank; peer[rank] is this rank's own
  int G, rank;        // physical ranks (GPUs)
  int V, v;           // virtual ranks = sources per tile (G x sub-slabs per launch) and this CTA's index among them
  unsigned epoch;     // > 0, the same on every rank, +1 per frame: flag value and (its low bit) table half
};
struct FusedArgs {
  FusedGeom g;
  const uint4 *descL, *descR;
  const RStat *statL, *statR;
  const float *fL, *fR;
  const float *meanR, *AR;       // right-image ZSAD means / NCC window sums, float planes
  const double* CR;              // right-image NCC scale, double plane
  const float *meanL, *AL;       // the left image's planes (kModeRight)
  const double* CL;
  const float* first4;           // kModeRight: [N][4] raw costs that stand in where x + d >= w (get_right_cost's fill)
  float* first4_out;             // full mode, both views requested: where the left-view launch leaves those four
  int out_ch0;                   // first channel this launch writes (8 for the right view)
  const float* luts;    // [128] + [256], see ms_prep_kernel
  const float* sadsob;  // see FusedWs
  float* out;           // [N][8][D][h][w]
  float* mins;          // slab phase A only: [N][mins_planes][h][w], planes 0-3 = per-pixel minima of this launch's disparities
  int out_channels;     // channel count of the output tensor (pair stride): 8, or 16 when the caller adds the right view
  int mins_planes;      // 4, or 8 when the caller adds the right view
  int out_D, out_d0;    // slab phase A: disparity count of the output tensor and where this launch's slab sits in it
  int mins_accumulate;  // slab phase A: fold into the minima already in `mins` (a later slab of the same volume)
  float k_cen, k_ncc, k_sad;
  int DC;               // disparity steps per d-group (even: phase 1 walks disparity pairs)
  int tiles_x;
  // Disparity-slab exchange (mode kModeXchg): the tables of all ranks (xchg.peer[rank] is this rank's own),
  // peer-mapped device pointers.  See tile_back_half.
  FusedXchg xchg;
  long long n_tiles;
  // optional by-products (nullptr: off): winner-take-all over each of channels 0-3 -- np.argmin's rule, what
  // main_msnet.py:443-448 does on the host with the whole volume -- and the two smallest values, as planes
  // [subs][N][4][h][w]; the disparity index is absolute (first disparity of the launch / sub-slab added)
  int32_t* wta_idx;
  float *wta_min1, *wta_min2;
  int subs;             // kModeXchg: sub-slabs of g.D disparities the launch's slab is cut into (virtual ranks)
};

constexpr int kTile = 32;   // pixels per tile: one output row segment of 128 bytes
constexpr int kModeRight = 5;   // the RIGHT view (channels 8-15 of extract_features_lr): see phase1_tile_right
constexpr int kModeFull = 0, kModeSlabA = 1, kModeXchg = 2, kModeBf16 = 3, kModeExact = 4;   // kModeBf16: kModeFull writing a bf16 volume; kModeExact: kModeFull with the reference's own AML arithmetic

// Staging buffer of one tile: right-image row data for the D + 31 (+ slack) columns the tile
// can touch.  Row strides are compile-time so every shared access in the hot loop is
// "pointer + immediate".
template <int DMAX, int SLACK>
struct StageLay {
  static constexpr int kSl = SLACK;
  static constexpr int RW = (DMAX + kTile - 1 + SLACK + 3) & ~3;   // desc / stat entries
  static constexpr int RWF = RW + 8;                               // float row: halo 2+2, align shift <= 3
  static constexpr size_t st_desc = 0;                                   // [RW] uint4 census codes
  static constexpr size_t st_c = st_desc + (size_t)RW * 16;              // [RW + 2] double NCC scale C (aligned start: shift <= 1)
  static constexpr size_t st_rf = st_c + (size_t)(RW + 2) * 8;           // [7][RWF] float rows: 5 pixel rows, NCC sums A, ZSAD means
  static constexpr size_t st_bytes = (st_rf + (size_t)7 * RWF * 4 + 127) & ~(size_t)127;
};

// Parking buffer of one tile: raw costs (later: AML exponentials) for every (d, pixel).
//   [3][DS][32] floats (ncc, sadsob, zsad) + [DS][32] census bytes; plane DMAX is scratch for
//   dummy steps.  Plane 1 is a TMA destination: DS * 128 bytes keeps it 128-byte aligned.
template <int DMAX>
struct ParkLay {
  static constexpr int DS = DMAX + 1;
  static constexpr int PS = DS * kTile;                                  // floats per parked matcher
  static constexpr size_t pk_cen = (size_t)3 * PS * 4;
  static constexpr size_t pk_bytes = (pk_cen + (size_t)DS * kTile + 127) & ~(size_t)127;
};

// Shared memory of one CTA = one tile (2 CTAs per SM).
template <int DMAX, int SLACK>
struct Lay : StageLay<DMAX, SLACK>, ParkLay<DMAX> {
  using S = StageLay<DMAX, SLACK>;
  using P = ParkLay<DMAX>;
  static constexpr size_t off_red = S::st_bytes;                                  // [kGroups][4][32] per-group minima
  static constexpr size_t off_min = off_red + (size_t)kGroups * 4 * kTile * 4;    // [4][32]
  static constexpr size_t off_inv = off_min + 4 * kTile * 4;                      // [4][32]
  static constexpr size_t off_lut = off_inv + 4 * kTile * 4;                      // [128] census AML exponentials
  static constexpr size_t off_lutn = off_lut + 128 * 4;                           // [256] census byte -> channel 0 (loaded, not read)
  static constexpr size_t off_par = (off_lutn + 256 * 4 + 127) & ~(size_t)127;    // 128 B aligned: TMA destination
  static constexpr size_t off_bar = off_par + P::pk_bytes;                        // 2 mbarriers
  static constexpr size_t bytes = off_bar + 32;
};

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// ---- TMA / bulk-copy helpers (cp.async.bulk*, completion through an mbarrier) ----------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, unsigned count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_init_fence() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Waits for the phase with the given parity.  try_wait suspends the warp in hardware (up to the
// hint, in ns) instead of polling, so waiting warps leave the issue slots to the working ones.
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, unsigned parity) {
  const uint32_t addr = smem_u32(bar);
  unsigned done;
  do {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(1000000u)
        : "memory");
  } while (!done);
}
// 1-D bulk copy global -> shared (bytes multiple of 16, both sides 16 B aligned)
__device__ __forceinline__ void bulk_load(void* dst, const void* src, unsigned bytes, unsigned long long* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// 3-D tiled tensor copy global -> shared through a CUtensorMap (out-of-range elements read as 0)
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            unsigned long long* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
          smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}

// ---- packed fp32x2 arithmetic (Blackwell FADD2: two IEEE round-to-nearest adds per issue slot;
//      operand B may be a scalar register broadcast to both halves, |x| is an operand modifier)
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void upk2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
// AML exponentials of two costs at once: 2^(-(c-m)^2 k) for (c.lo, m.lo) and (c.hi, m.hi); the packed
// subtract / square / scale round exactly like aml_e's scalar ones (each half is an IEEE fp32 operation)
__device__ __forceinline__ void aml_e2(f32x2 c, f32x2 m, f32x2 negk, float& e_lo, float& e_hi) {
  const f32x2 t = sub2(c, m);
  float a_lo, a_hi;
  upk2(mul2(mul2(t, t), negk), a_lo, a_hi);
  e_lo = ex2_approx(a_lo);
  e_hi = ex2_approx(a_hi);
}
__device__ __forceinline__ f32x2 abs2(f32x2 v) {
  float lo, hi;
  upk2(v, lo, hi);
  return pk2(fabsf(lo), fabsf(hi));
}

struct TileId {
  int n, y, x0;   // y: row of the cropped image
  int yl;     // row inside this launch's band (output indexing)
  int d0;     // first disparity of this CTA (the launch's, plus its sub-slab offset)
  int sub0;   // offset of this CTA's sub-slab inside the launch's slab (0 unless the launch is cut, kModeXchg)
  int v;      // kModeXchg: this CTA's virtual rank (row in the exchange tables)
};
__device__ __forceinline__ TileId decode_tile(int tile, const FusedArgs& a, int sub = 0) {
  TileId t;
  t.sub0 = sub * a.g.D;
  t.d0 = a.g.d0 + t.sub0;
  t.v = a.xchg.v + sub;
  const int xt = tile % a.tiles_x;
  tile /= a.tiles_x;
  t.yl = tile % a.g.h;
  t.y = t.yl + a.g.y0;
  t.n = tile / a.g.h;
  t.x0 = xt * kTile;
  return t;
}

// Asynchronously copies the right-image row data of `t` into a staging buffer with LDGSTS:
// census codes and stats of the D+31(+slack) columns the tile can touch and the five float
// rows of the ZSAD/NCC windows (the float rows start at a 4-float aligned column).
template <class L, int NT>
__device__ __forceinline__ void stage_right(const FusedArgs& a, const TileId& t, unsigned char* buf) {
  const FusedGeom& g = a.g;
  const int D = g.D;
  const int RWn = D + kTile - 1 + L::kSl;
  const int XbaseP = t.x0 + g.bwl - (t.d0 + D - 1) - L::kSl + g.padL;
  const int Yp = t.y + g.bh + kPadT;
  const size_t img_off = (size_t)t.n * g.img_px();
  const uint4* gd = a.descR + img_off + (size_t)Yp * g.Wp + XbaseP;
  uint4* s_desc = reinterpret_cast<uint4*>(buf + L::st_desc);
  float* s_rf = reinterpret_cast<float*>(buf + L::st_rf);
  for (int i = threadIdx.x; i < RWn; i += NT) cp_async16(s_desc + i, gd + i);
  {   // NCC scale C: doubles from the even column at or before XbaseP
    const int cstart = XbaseP & ~1;
    const int nc = (RWn + 1 + 1) >> 1;   // 16-byte groups
    const double* gc = a.CR + img_off + (size_t)Yp * g.Wp + cstart;
    double* s_c = reinterpret_cast<double*>(buf + L::st_c);
    for (int i = threadIdx.x; i < nc; i += NT) cp_async16(s_c + 2 * i, gc + 2 * i);
  }
  const int fstart = (XbaseP - 2) & ~3;                 // aligned first float column
  const int nvec = (RWn + 4 + 3 + 3) >> 2;              // 16-byte groups per row (covers any shift)
  for (int i = threadIdx.x; i < 5 * nvec; i += NT) {
    const int r = i / nvec, v = i - r * nvec;
    cp_async16(s_rf + r * L::RWF + 4 * v, a.fR + img_off + (size_t)(Yp - 2 + r) * g.Wp + fstart + 4 * v);
  }
  for (int i = threadIdx.x; i < 2 * nvec; i += NT) {   // rows 5 (A) and 6 (mean), same alignment as the pixel rows
    const int c = i / nvec, v = i - c * nvec;
    cp_async16(s_rf + (5 + c) * L::RWF + 4 * v, (c ? a.meanR : a.AR) + img_off + (size_t)Yp * g.Wp + fstart + 4 * v);
  }
}

// Same data through the TMA engine: nine 1-D bulk copies issued by a single thread,
// completion counted in bytes on `bar`.
// kRightView: the LEFT image's rows for columns X0 + d0 .. (the window of a right-view tile slides rightwards).
template <class L, bool kRightView = false>
__device__ __forceinline__ void stage_rows_tma(const FusedArgs& a, const TileId& t, unsigned char* buf,
                                               unsigned long long* bar) {
  const FusedGeom& g = a.g;
  const int D = g.D;
  const int RWn = D + kTile - 1 + L::kSl;
  const int XbaseP = kRightView ? t.x0 + g.bwl + t.d0 + g.padL : t.x0 + g.bwl - (t.d0 + D - 1) - L::kSl + g.padL;
  const int Yp = t.y + g.bh + kPadT;
  const size_t img_off = (size_t)t.n * g.img_px();
  const int fstart = (XbaseP - 2) & ~3;
  const int nvec = (RWn + 4 + 3 + 3) >> 2;
  const unsigned row_bytes = (unsigned)RWn * 16u, frow_bytes = (unsigned)nvec * 16u;
  const int cstart = XbaseP & ~1;
  const unsigned crow_bytes = (unsigned)((RWn + 1 + 1) >> 1) * 16u;
  const uint4* desc = kRightView ? a.descL : a.descR;
  const double* C = kRightView ? a.CL : a.CR;
  const float* f = kRightView ? a.fL : a.fR;
  const float* A = kRightView ? a.AL : a.AR;
  const float* mean = kRightView ? a.meanL : a.meanR;
  mbar_expect_tx(bar, row_bytes + crow_bytes + 7u * frow_bytes);
  bulk_load(buf + L::st_desc, desc + img_off + (size_t)Yp * g.Wp + XbaseP, row_bytes, bar);
  bulk_load(buf + L::st_c, C + img_off + (size_t)Yp * g.Wp + cstart, crow_bytes, bar);
  float* s_rf = reinterpret_cast<float*>(buf + L::st_rf);
#pragma unroll
  for (int r = 0; r < 5; ++r)
    bulk_load(s_rf + r * L::RWF, f + img_off + (size_t)(Yp - 2 + r) * g.Wp + fstart, frow_bytes, bar);
  bulk_load(s_rf + 5 * L::RWF, A + img_off + (size_t)Yp * g.Wp + fstart, frow_bytes, bar);
  bulk_load(s_rf + 6 * L::RWF, mean + img_off + (size_t)Yp * g.Wp + fstart, frow_bytes, bar);
}

// The tile's D x 32 SAD-of-Sobel costs: ONE 3-D tensor copy straight into parking plane 1.
// They come from DRAM and are only needed after phase 1, hence their own barrier.
__device__ __forceinline__ void stage_sad_tma(const FusedArgs& a, const CUtensorMap* sad_map, const TileId& t,
                                              float* park_plane1, unsigned long long* bar_sad) {
  const FusedGeom& g = a.g;
  mbar_expect_tx(bar_sad, (unsigned)g.D * kTile * 4u);
  if (g.d_inner) tma_load_3d(park_plane1, sad_map, t.x0 + g.bwl + g.sxo, t.sub0, t.n * g.H + t.y + g.bh, bar_sad);
  else tma_load_3d(park_plane1, sad_map, t.x0 + g.bwl + g.sxo, t.y + g.bh, t.n * g.Dl + t.sub0, bar_sad);  // inner coordinate % 4 == 0
}

// A pixel's own left-image data: census code, stats, 5x5 float window.  Loaded straight from
// global memory before the staging barrier, so the latency overlaps the TMA round trip
// (staging it through TMA as well was measured 1.5 % slower).
struct LeftRegs {
  uint4 desc;
  uint4 stat;
  float px[5][5];
};
template <bool kRightView = false>   // kRightView: the pixel's RIGHT-image data (the fixed side of a right-view tile)
__device__ __forceinline__ void load_left(const FusedArgs& a, const TileId& t, int px, LeftRegs& lr) {
  const FusedGeom& g = a.g;
  const int Yp = t.y + g.bh + kPadT;
  const int Xp = t.x0 + px + g.bwl + g.padL;
  const size_t img_off = (size_t)t.n * g.img_px();
  lr.desc = __ldg((kRightView ? a.descR : a.descL) + img_off + (size_t)Yp * g.Wp + Xp);
  lr.stat = __ldg(reinterpret_cast<const uint4*>((kRightView ? a.statR : a.statL) + img_off + (size_t)Yp * g.Wp + Xp));
#pragma unroll
  for (int r = 0; r < 5; ++r) {
    const float* gf = (kRightView ? a.fR : a.fL) + img_off + (size_t)(Yp - 2 + r) * g.Wp + (Xp - 2);
#pragma unroll
    for (int c = 0; c < 5; ++c) lr.px[r][c] = __ldg(gf + c);
  }
}

// ---- phase 1 of a tile for one thread = (pixel px, d-group [d_lo, d_lo + DC)) ---------------
// Per (pixel, d): census popcount, NCC (9 fp32 products of exact integers, fp64 scaling), ZSAD
// over a register-resident right window that slides with d; raw costs are parked in shared
// memory (ncc -> plane 0, zsad -> plane 2, census byte); running minima are returned.
//
// ZSAD evaluates disparities in pairs (dA = d, dB = d + 1) with packed FADD2, dB in the low
// half.  The right windows of the pair overlap: dB's is dA's shifted one column left, so with
// wv[r][j] = right pixel at column (X - dB - 2) + j, j = 0..5, tap c of dA reads wv[c+1] and
// tap c of dB reads wv[c].  Pairing tap j of dB with tap j-1 of dA gives both halves the SAME
// right pixel (a broadcast operand) and a constant left operand ap[r][j-1] =
// (L[r][j] - mL, L[r][j-1] - mL), hoisted over all d (matchers.cpp:503).  Per window row: one
// scalar step (dB tap 0), four packed steps, one scalar step (dA tap 4) -- each half still adds
// its 25 taps in row-major order, every operation an IEEE fp32 add: bit-exact.
struct Phase1Out {
  int min_cen;
  float min_ncc, min_sad;
  int dmax_sad;
};

// Per-thread state of the phase-1 loop: staging pointers (they fall by two columns per disparity
// pair), the register-resident right window and the running minima.
template <class L>
struct P1State {
  const float* rfp;    // column (X - dB - 2) of the pair's second disparity
  const uint4* dscp;
  const double* ccp;   // NCC scale C of column X - dA (C of X - dB is ccp[-1])
  float wv[5][6];      // sliding 5x6 right window; logical column j lives in wv[.][(j - 2*s) mod 6]
  int min_cen;
  float min_ncc, min_sad;
};

// One BLOCK of phase 1 = three disparity pairs (the rotation period of the window registers).
// kClean: every disparity of the block has all three costs for this thread's pixel and the block is
// whole (no dummy steps): no validity selects, one basic block.  Otherwise validity is checked per
// voxel and `steps` (<= 3) pairs are walked.
template <class L, bool kClean>
__device__ __forceinline__ void p1_block(P1State<L>& st, int dblk, int steps, int D, const f32x2 (&ap)[5][4],
                                         const float (&l3)[3][3], const uint4& ld, const RStat& ls, int dmax_cen,
                                         int dmax_ncc, int dmax_sad, float* s_par, uint8_t* s_cen, int px) {
  constexpr int PS = L::PS;
#pragma unroll
  for (int sI = 0; sI < 3; ++sI) {
#define WV(r, j) st.wv[r][((j) + 12 - 2 * sI) % 6]
    if (!kClean && sI > 0 && sI >= steps) break;
    const int dA = dblk + 2 * sI, dB = dA + 1;
    const uint4 rdA = st.dscp[0], rdB = st.dscp[-1];
    // rfp[2] / rfp[3] are columns X - dB / X - dA: rows 5 and 6 hold the NCC sums and the ZSAD means
    RStat rsA, rsB;
    rsA.A = st.rfp[5 * L::RWF + 3]; rsB.A = st.rfp[5 * L::RWF + 2];
    rsA.C = st.ccp[0]; rsB.C = st.ccp[-1];
    const float2 mBA = make_float2(st.rfp[6 * L::RWF + 2], st.rfp[6 * L::RWF + 3]);   // (mean at X - dB, mean at X - dA)

    // census: Hamming distance of the packed codes (matchers.cpp:323-337)
    const int cenA = __popc(ld.x ^ rdA.x) + __popc(ld.y ^ rdA.y) + __popc(ld.z ^ rdA.z) + __popc(ld.w ^ rdA.w);
    const int cenB = __popc(ld.x ^ rdB.x) + __popc(ld.y ^ rdB.y) + __popc(ld.z ^ rdB.z) + __popc(ld.w ^ rdB.w);
    const int cen_bA = (kClean || dA <= dmax_cen) ? cenA : 255;
    const int cen_bB = (kClean || dB <= dmax_cen) ? cenB : 255;

    // NCC: P exact in fp32 (< 2^24); scaling in fp64 left to right (matchers.cpp:200-201)
    float PA = 0.f, PB = 0.f;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        PA = __fmaf_rn(l3[r][c], WV(r + 1, c + 2), PA);
        PB = __fmaf_rn(l3[r][c], WV(r + 1, c + 1), PB);
      }
    const float numA = __fmaf_rn(9.0f, PA, -__fmul_rn(ls.A, rsA.A));
    const float numB = __fmaf_rn(9.0f, PB, -__fmul_rn(ls.A, rsB.A));
    float nccA = (float)__dmul_rn(__dmul_rn(-(double)numA, ls.C), rsA.C);
    float nccB = (float)__dmul_rn(__dmul_rn(-(double)numB, ls.C), rsB.C);
    nccA = (fabsf(nccA) <= 3.0e38f) ? nccA : 1.0f;  // either C was inf (flat window), :196,204
    nccB = (fabsf(nccB) <= 3.0e38f) ? nccB : 1.0f;
    nccA = (kClean || dA <= dmax_ncc) ? nccA : kFill;
    nccB = (kClean || dB <= dmax_ncc) ? nccB : kFill;

    // ZSAD: 25 taps row-major, ((L - mL) - R) + mR, sequential fp32 (matchers.cpp:499-506)
    const f32x2 m2 = pk2(mBA.x, mBA.y);
    f32x2 acc = pk2(0.f, 0.f);   // (dB, dA)
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      float a_first, a_last, dum, accA, accB;
      upk2(ap[r][0], dum, a_first);   // L[r][0] - mL
      upk2(ap[r][3], a_last, dum);    // L[r][4] - mL
      upk2(acc, accB, accA);
      accB = __fadd_rn(accB, fabsf(__fadd_rn(__fsub_rn(a_first, WV(r, 0)), mBA.x)));   // dB tap 0
      acc = pk2(accB, accA);
#pragma unroll
      for (int j = 1; j <= 4; ++j) {
        const float wj = WV(r, j);
        const f32x2 u = add2(sub2(ap[r][j - 1], pk2(wj, wj)), m2);                    // dB tap j, dA tap j-1
        acc = add2(acc, abs2(u));
      }
      upk2(acc, accB, accA);
      accA = __fadd_rn(accA, fabsf(__fadd_rn(__fsub_rn(a_last, WV(r, 5)), mBA.y)));    // dA tap 4
      acc = pk2(accB, accA);
    }
    float zA, zB;
    upk2(acc, zB, zA);
    zA = (kClean || dA <= dmax_sad) ? zA : kFill;
    zB = (kClean || dB <= dmax_sad) ? zB : kFill;

    const int dsA = kClean ? dA : min(dA, D);   // dummy steps (d >= D) park into the scratch plane
    const int dsB = kClean ? dB : min(dB, D);
    s_cen[dsA * kTile + px] = (uint8_t)cen_bA;
    s_cen[dsB * kTile + px] = (uint8_t)cen_bB;
    s_par[dsA * kTile + px] = nccA;
    s_par[dsB * kTile + px] = nccB;
    s_par[2 * PS + dsA * kTile + px] = zA;
    s_par[2 * PS + dsB * kTile + px] = zB;
    st.min_cen = min(st.min_cen, min(cen_bA, cen_bB));
    st.min_ncc = fminf(st.min_ncc, fminf(nccA, nccB));
    st.min_sad = fminf(st.min_sad, fminf(zA, zB));
    // slide the window two columns left: the next pair's new columns 0 and 1
    st.rfp -= 2; st.dscp -= 2; st.ccp -= 2;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      st.wv[r][(0 + 12 - 2 * (sI + 1)) % 6] = st.rfp[r * L::RWF];
      st.wv[r][(1 + 12 - 2 * (sI + 1)) % 6] = st.rfp[r * L::RWF + 1];
    }
#undef WV
  }
}

// ---- phase 1 of a tile for one thread = (pixel px, d-group [d_lo, d_lo + DC)) ---------------
// Per (pixel, d): census popcount, NCC (9 fp32 products of exact integers, fp64 scaling), ZSAD
// over a register-resident right window that slides with d; raw costs are parked in shared
// memory (ncc -> plane 0, zsad -> plane 2, census byte); running minima are returned.
//
// ZSAD evaluates disparities in pairs (dA = d, dB = d + 1) with packed FADD2, dB in the low
// half.  The right windows of the pair overlap: dB's is dA's shifted one column left, so with
// wv[r][j] = right pixel at column (X - dB - 2) + j, j = 0..5, tap c of dA reads wv[c+1] and
// tap c of dB reads wv[c].  Pairing tap j of dB with tap j-1 of dA gives both halves the SAME
// right pixel (a broadcast operand) and a constant left operand ap[r][j-1] =
// (L[r][j] - mL, L[r][j-1] - mL), hoisted over all d (matchers.cpp:503).  Per window row: one
// scalar step (dB tap 0), four packed steps, one scalar step (dA tap 4) -- each half still adds
// its 25 taps in row-major order, every operation an IEEE fp32 add: bit-exact.
//
// The d-group is walked in BLOCKS of six disparities.  A cost exists for d <= dmax (the window must
// fit left of x - d), so per warp (ballot, no divergence) a block is: clean -- every lane has every
// cost: the body without validity selects; past the valid range of every lane (monotone in d:
// nothing after it has a cost either) -- fill is parked and NOTHING is computed; else the generic
// body.  Tiles near the left image border spend about half their blocks in the second kind.
template <class L>
__device__ __forceinline__ Phase1Out phase1_tile(const FusedArgs& a, const TileId& t, const unsigned char* stage,
                                                 float* s_par, uint8_t* s_cen, const LeftRegs& lr, int px,
                                                 int d_lo) {
  constexpr int PS = L::PS;
  const FusedGeom& g = a.g;
  const int D = g.D, H = g.H, W = g.W;
  const int X = t.x0 + px + g.bwl;        // bordered image column of this thread's pixel
  const int Y = t.y + g.bh;               // bordered image row
  const uint4 ld = lr.desc;
  const RStat ls = *reinterpret_cast<const RStat*>(&lr.stat);
  f32x2 ap[5][4];   // ap[r][j-1] for j = 1..4
  float l3[3][3];   // centre 3x3 of L as float for NCC
#pragma unroll
  for (int r = 0; r < 5; ++r) {
    float av[5];
#pragma unroll
    for (int c = 0; c < 5; ++c) {
      av[c] = __fsub_rn(lr.px[r][c], ls.mean);
      if (r >= 1 && r <= 3 && c >= 1 && c <= 3) l3[r - 1][c - 1] = lr.px[r][c];
    }
#pragma unroll
    for (int j = 1; j <= 4; ++j) {
      // + (+0, +0) is value-preserving (a difference is never -0) and makes the pair a value of its
      // own to ptxas, which otherwise shares the overlapping halves and rebuilds the pairs with MOVs
      ap[r][j - 1] = add2(pk2(av[j], av[j - 1]), pk2(0.f, 0.f));
    }
  }
  // validity: cost(y,x,d) exists iff the window origin is inside and x - wc >= d (and d < D)
  // (dmax_* are local to the launch: disparity d0 + d of the image is step d here)
  const int dmax_cen = min(D - 1, ((Y >= 5 && Y < H - 6 && X >= 5 && X < W - 6) ? X - 5 : -1) - t.d0);
  const int dmax_ncc = min(D - 1, ((Y >= 1 && Y < H - 2 && X >= 1 && X < W - 2) ? X - 1 : -1) - t.d0);
  const int dmax_sad = min(D - 1, ((Y >= 2 && Y < H - 3 && X >= 2 && X < W - 3) ? X - 2 : -1) - t.d0);

  const uint4* s_desc = reinterpret_cast<const uint4*>(stage + L::st_desc);
  const double* s_c = reinterpret_cast<const double*>(stage + L::st_c);
  const float* s_rf = reinterpret_cast<const float*>(stage + L::st_rf);
  // shared index of right column X - d is ir = px + L::kSl + (D-1) - d; falls by one per step
  const int XbaseP = t.x0 + g.bwl - (t.d0 + D - 1) - L::kSl + g.padL;
  const int shift = (XbaseP - 2) & 3;
  const int ir0 = px + L::kSl + (D - 1) - d_lo;
  P1State<L> st;
  st.rfp = s_rf + shift + ir0 - 1;
  st.dscp = s_desc + ir0;
  st.ccp = s_c + (XbaseP & 1) + ir0;
#pragma unroll
  for (int r = 0; r < 5; ++r)
#pragma unroll
    for (int j = 0; j < 6; ++j) st.wv[r][j] = st.rfp[r * L::RWF + j];
  st.min_cen = 255;
  st.min_ncc = kFill;
  st.min_sad = kFill;

  for (int base = 0; base < a.DC; base += 6) {
    const int dblk = d_lo + base;
    const int left = a.DC - base;                        // disparities left in the d-group (even)
    const bool clean = (left >= 6) && (dblk + 5 <= dmax_cen);   // census has the tightest bound
    const bool none = dblk > dmax_ncc;                          // NCC the loosest
    if (__all_sync(0xffffffffu, clean)) {
      p1_block<L, true>(st, dblk, 3, D, ap, l3, ld, ls, dmax_cen, dmax_ncc, dmax_sad, s_par, s_cen, px);
    } else if (__all_sync(0xffffffffu, none)) {
      const int nd = min(left, 6);
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        if (k >= nd) break;
        const int ds = min(dblk + k, D);
        s_cen[ds * kTile + px] = 255;
        s_par[ds * kTile + px] = kFill;
        s_par[2 * PS + ds * kTile + px] = kFill;
      }
      st.rfp -= 6; st.dscp -= 6; st.ccp -= 6;   // (the window registers are never used again)
    } else {
      p1_block<L, false>(st, dblk, min(left, 6) >> 1, D, ap, l3, ld, ls, dmax_cen, dmax_ncc, dmax_sad, s_par, s_cen, px);
    }
  }
  Phase1Out o;
  o.min_cen = st.min_cen;
  o.min_ncc = st.min_ncc;
  o.min_sad = st.min_sad;
  o.dmax_sad = dmax_sad;
  return o;
}

// ---- phase 1 of a RIGHT-VIEW tile (channels 8-15 of extract_features_lr, cbmv_generator.py:84-254) ----------
// get_right_cost (featextract.cpp:136-172): right(y, x, d) = cost(y, x + d, d) for x + d < w, else c.flat[0].
// A right-view tile therefore needs the costs of a PARALLELOGRAM of the left-view volume; instead of parking
// raw costs in HBM and gathering them back (the three-phase route of slab.cu: 2.7x the traffic), the tile
// recomputes them with the roles swapped: thread = (RIGHT pixel xr, d-group), the right window is fixed in
// registers and the LEFT window (pixel xr + d) slides rightwards with d.  Every cost is the same sequence of IEEE
// operations as in the left-view tile:
//  census  popc(codeL[xr+d] ^ codeR[xr]);
//  NCC     9P - A_L A_R exact in fp32, then (-num * C_L) * C_R in fp64 -- the LEFT scale first (matchers.cpp:200);
//  ZSAD    ((L - mL) - R) + mR per tap, row-major.  Disparities dA = d, dB = d + 1 are packed: tap j of dA and
//          tap j-1 of dB read the SAME left pixel (a broadcast operand).  Both mL and L change with d, so a tap
//          is evaluated NEGATED, three packed operations: (mL - L) + R - mR = -(((L - mL) - R) + mR) -- each step
//          is the exact negative of the reference's (round-to-nearest is symmetric) and |.| drops the sign.
//          100 adds per voxel instead of the left view's 75 (the left view hoists L - mL over d).
// Validity: the cost exists iff the LEFT window at xr + d is inside -- d <= dmax with dmax falling as xr grows --
// and xr itself is right of the window radius; beyond x + d = w - 1 the caller's first4 stands in (finish_right).
template <class L, bool kClean>
__device__ __forceinline__ void p1_block_right(P1State<L>& st, int dblk, int steps, int D, const f32x2 (&rp)[5][4],
                                               const float (&r3)[3][3],
                                               const uint4& rd, const RStat& rs, int dmax_cen, int dmax_ncc,
                                               int dmax_sad, float* s_par, uint8_t* s_cen, int px) {
  constexpr int PS = L::PS;
  const f32x2 mR2 = pk2(rs.mean, rs.mean);
#pragma unroll
  for (int sI = 0; sI < 3; ++sI) {
#define LV(r, j) st.wv[r][((j) + 2 * sI) % 6]
    if (!kClean && sI > 0 && sI >= steps) break;
    const int dA = dblk + 2 * sI, dB = dA + 1;
    const uint4 ldA = st.dscp[0], ldB = st.dscp[1];
    // rfp[2] / rfp[3] are left columns xr + dA / xr + dB: rows 5 and 6 hold the NCC sums and the ZSAD means
    const float aLA = st.rfp[5 * L::RWF + 2], aLB = st.rfp[5 * L::RWF + 3];
    const double cLA = st.ccp[0], cLB = st.ccp[1];
    const float mLA = st.rfp[6 * L::RWF + 2], mLB = st.rfp[6 * L::RWF + 3];

    const int cenA = __popc(ldA.x ^ rd.x) + __popc(ldA.y ^ rd.y) + __popc(ldA.z ^ rd.z) + __popc(ldA.w ^ rd.w);
    const int cenB = __popc(ldB.x ^ rd.x) + __popc(ldB.y ^ rd.y) + __popc(ldB.z ^ rd.z) + __popc(ldB.w ^ rd.w);
    const int cen_bA = (kClean || dA <= dmax_cen) ? cenA : 255;
    const int cen_bB = (kClean || dB <= dmax_cen) ? cenB : 255;

    float PA = 0.f, PB = 0.f;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        PA = __fmaf_rn(LV(r + 1, c + 1), r3[r][c], PA);
        PB = __fmaf_rn(LV(r + 1, c + 2), r3[r][c], PB);
      }
    const float numA = __fmaf_rn(9.0f, PA, -__fmul_rn(aLA, rs.A));
    const float numB = __fmaf_rn(9.0f, PB, -__fmul_rn(aLB, rs.A));
    float nccA = (float)__dmul_rn(__dmul_rn(-(double)numA, cLA), rs.C);
    float nccB = (float)__dmul_rn(__dmul_rn(-(double)numB, cLB), rs.C);
    nccA = (fabsf(nccA) <= 3.0e38f) ? nccA : 1.0f;
    nccB = (fabsf(nccB) <= 3.0e38f) ? nccB : 1.0f;
    nccA = (kClean || dA <= dmax_ncc) ? nccA : kFill;
    nccB = (kClean || dB <= dmax_ncc) ? nccB : kFill;

    const f32x2 mL2 = pk2(mLA, mLB);
    f32x2 acc = pk2(0.f, 0.f);   // (dA, dB)
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      float accA, accB, r0, r4, dum;
      upk2(rp[r][0], dum, r0);   // R[r][0] and R[r][4] are halves of the hoisted pairs
      upk2(rp[r][3], r4, dum);
      upk2(acc, accA, accB);
      accA = __fadd_rn(accA, fabsf(__fadd_rn(__fsub_rn(__fsub_rn(LV(r, 0), mLA), r0), rs.mean)));   // dA tap 0
      acc = pk2(accA, accB);
#pragma unroll
      for (int j = 1; j <= 4; ++j) {
        const float lj = LV(r, j);
        const f32x2 n = sub2(add2(sub2(mL2, pk2(lj, lj)), rp[r][j - 1]), mR2);   // dA tap j, dB tap j-1 (negated)
        acc = add2(acc, abs2(n));
      }
      upk2(acc, accA, accB);
      accB = __fadd_rn(accB, fabsf(__fadd_rn(__fsub_rn(__fsub_rn(LV(r, 5), mLB), r4), rs.mean)));   // dB tap 4
      acc = pk2(accA, accB);
    }
    float zA, zB;
    upk2(acc, zA, zB);
    zA = (kClean || dA <= dmax_sad) ? zA : kFill;
    zB = (kClean || dB <= dmax_sad) ? zB : kFill;

    const int dsA = kClean ? dA : min(dA, D);
    const int dsB = kClean ? dB : min(dB, D);
    s_cen[dsA * kTile + px] = (uint8_t)cen_bA;
    s_cen[dsB * kTile + px] = (uint8_t)cen_bB;
    s_par[dsA * kTile + px] = nccA;
    s_par[dsB * kTile + px] = nccB;
    s_par[2 * PS + dsA * kTile + px] = zA;
    s_par[2 * PS + dsB * kTile + px] = zB;
    st.min_cen = min(st.min_cen, min(cen_bA, cen_bB));
    st.min_ncc = fminf(st.min_ncc, fminf(nccA, nccB));
    st.min_sad = fminf(st.min_sad, fminf(zA, zB));
    // slide the window two columns right: the next pair's new columns 4 and 5
    st.rfp += 2; st.dscp += 2; st.ccp += 2;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
      st.wv[r][(4 + 2 * (sI + 1)) % 6] = st.rfp[r * L::RWF + 4];
      st.wv[r][(5 + 2 * (sI + 1)) % 6] = st.rfp[r * L::RWF + 5];
    }
#undef LV
  }
}

struct Phase1RightOut {
  Phase1Out o;
  int dcrop;   // last disparity (local to the launch) with x + d < w: beyond it first4 stands in
};

template <class L>
__device__ __forceinline__ Phase1RightOut phase1_tile_right(const FusedArgs& a, const TileId& t, const unsigned char* stage,
                                                            float* s_par, uint8_t* s_cen, const LeftRegs& rr, int px,
                                                            int d_lo) {
  constexpr int PS = L::PS;
  const FusedGeom& g = a.g;
  const int D = g.D, H = g.H, W = g.W;
  const int Xr = t.x0 + px + g.bwl;       // bordered image column of this thread's RIGHT pixel
  const int Y = t.y + g.bh;
  const uint4 rd = rr.desc;
  const RStat rs = *reinterpret_cast<const RStat*>(&rr.stat);
  f32x2 rp[5][4];   // rp[r][j-1] = (R[r][j], R[r][j-1]) for j = 1..4
  float r3[3][3];
#pragma unroll
  for (int r = 0; r < 5; ++r) {
#pragma unroll
    for (int c = 0; c < 5; ++c)
      if (r >= 1 && r <= 3 && c >= 1 && c <= 3) r3[r - 1][c - 1] = rr.px[r][c];
#pragma unroll
    for (int j = 1; j <= 4; ++j) rp[r][j - 1] = add2(pk2(rr.px[r][j], rr.px[r][j - 1]), pk2(0.f, 0.f));   // (own value per pair, see phase1_tile)
  }
  // the cost of (xr, d) is the left-view cost of pixel X = xr + d: window origin inside <=> X below the right
  // margin; X - wc >= d <=> xr >= wc
  const int dcrop = (g.w - 1 - (t.x0 + px)) - t.d0;
  const int dmax_cen = min(min(D - 1, dcrop), ((Y >= 5 && Y < H - 6 && Xr >= 5) ? W - 7 - Xr : -1) - t.d0);
  const int dmax_ncc = min(min(D - 1, dcrop), ((Y >= 1 && Y < H - 2 && Xr >= 1) ? W - 3 - Xr : -1) - t.d0);
  const int dmax_sad = min(min(D - 1, dcrop), ((Y >= 2 && Y < H - 3 && Xr >= 2) ? W - 4 - Xr : -1) - t.d0);

  const uint4* s_desc = reinterpret_cast<const uint4*>(stage + L::st_desc);
  const double* s_c = reinterpret_cast<const double*>(stage + L::st_c);
  const float* s_rf = reinterpret_cast<const float*>(stage + L::st_rf);
  // shared index of left column xr + d is px + d; rises by one per step
  const int XbaseP = t.x0 + g.bwl + t.d0 + g.padL;
  const int shift = (XbaseP - 2) & 3;
  P1State<L> st;
  st.rfp = s_rf + shift + px + d_lo;        // column (xr + dA) - 2 of the pair's first disparity
  st.dscp = s_desc + px + d_lo;
  st.ccp = s_c + (XbaseP & 1) + px + d_lo;
#pragma unroll
  for (int r = 0; r < 5; ++r)
#pragma unroll
    for (int j = 0; j < 6; ++j) st.wv[r][j] = st.rfp[r * L::RWF + j];
  st.min_cen = 255;
  st.min_ncc = kFill;
  st.min_sad = kFill;

  for (int base = 0; base < a.DC; base += 6) {
    const int dblk = d_lo + base;
    const int left = a.DC - base;
    const bool clean = (left >= 6) && (dblk + 5 <= dmax_cen);
    const bool none = dblk > dmax_ncc;
    if (__all_sync(0xffffffffu, clean)) {
      p1_block_right<L, true>(st, dblk, 3, D, rp, r3, rd, rs, dmax_cen, dmax_ncc, dmax_sad, s_par, s_cen, px);
    } else if (__all_sync(0xffffffffu, none)) {
      const int nd = min(left, 6);
#pragma unroll
      for (int k = 0; k < 6; ++k) {
        if (k >= nd) break;
        const int ds = min(dblk + k, D);
        s_cen[ds * kTile + px] = 255;
        s_par[ds * kTile + px] = kFill;
        s_par[2 * PS + ds * kTile + px] = kFill;
      }
      st.rfp += 6; st.dscp += 6; st.ccp += 6;
    } else {
      p1_block_right<L, false>(st, dblk, min(left, 6) >> 1, D, rp, r3, rd, rs, dmax_cen, dmax_ncc, dmax_sad, s_par, s_cen, px);
    }
  }
  Phase1RightOut o;
  o.o.min_cen = st.min_cen;
  o.o.min_ncc = st.min_ncc;
  o.o.min_sad = st.min_sad;
  o.o.dmax_sad = dmax_sad;
  o.dcrop = dcrop;
  return o;
}

// Right view, after phase 1: SAD-of-Sobel validity and minima as in finish_phase1, then get_right_cost's fill --
// where x + d >= w all four matchers hold the volume's first element (featextract.cpp:151), which takes part in
// the minima like any cost.
template <class L>
__device__ __forceinline__ void finish_right(float* s_par, uint8_t* s_cen, float* s_red, const Phase1RightOut& ro,
                                             const float* first4, int px, int grp, int d_lo, int d_end) {
  constexpr int PS = L::PS;
  const Phase1Out& o = ro.o;
  float mn[4] = {(o.min_cen == 255) ? kFill : (float)o.min_cen, o.min_ncc, kFill, o.min_sad};
  float* sp = s_par + PS + d_lo * kTile + px;
  for (int d = d_lo; d < d_end; ++d, sp += kTile) {
    float v = *sp;
    if (d > o.dmax_sad) {
      v = kFill;
      *sp = v;
    }
    mn[2] = fminf(mn[2], v);
  }
  const int df = max(d_lo, ro.dcrop + 1);
  if (df < d_end) {
    const float f0 = first4[0], f1 = first4[1], f2 = first4[2], f3 = first4[3];
    const uint8_t b0 = (f0 == kFill) ? (uint8_t)255 : (uint8_t)f0;
    for (int d = df; d < d_end; ++d) {
      s_cen[d * kTile + px] = b0;
      s_par[d * kTile + px] = f1;
      s_par[PS + d * kTile + px] = f2;
      s_par[2 * PS + d * kTile + px] = f3;
    }
    mn[0] = fminf(mn[0], f0); mn[1] = fminf(mn[1], f1); mn[2] = fminf(mn[2], f2); mn[3] = fminf(mn[3], f3);
  }
#pragma unroll
  for (int m = 0; m < 4; ++m) s_red[(grp * 4 + m) * kTile + px] = mn[m];
}

// After phase 1 and once the tile's SAD-of-Sobel costs have landed in plane 1: this thread's
// disparities outside the valid region become fill; per-group minima go to s_red[grp][4][32].
template <class L>
__device__ __forceinline__ void finish_phase1(float* s_par, float* s_red, const Phase1Out& o, int px, int grp,
                                              int d_lo, int d_end) {
  float min_sob = kFill;
  float* sp = s_par + L::PS + d_lo * kTile + px;
  if (__all_sync(0xffffffffu, d_end - 1 <= o.dmax_sad)) {
    // every disparity of the warp's group has its cost (most tiles): loads and three-input minima only --
    // the guarded form below spends 7.5 mostly ALU-pipe instructions per voxel-row on predicates
    int d = d_lo;
    for (; d + 4 <= d_end; d += 4, sp += 4 * kTile) {
      const float v0 = sp[0], v1 = sp[kTile], v2 = sp[2 * kTile], v3 = sp[3 * kTile];
      min_sob = fminf(fminf(min_sob, v0), v1);
      min_sob = fminf(fminf(min_sob, v2), v3);
    }
    for (; d < d_end; ++d, sp += kTile) min_sob = fminf(min_sob, *sp);
  } else {
#pragma unroll 4
    for (int d = d_lo; d < d_end; ++d, sp += kTile) {
      float v = *sp;
      if (d > o.dmax_sad) {
        v = kFill;
        *sp = v;
      }
      min_sob = fminf(min_sob, v);
    }
  }
  s_red[(grp * 4 + 0) * kTile + px] = (o.min_cen == 255) ? kFill : (float)o.min_cen;
  s_red[(grp * 4 + 1) * kTile + px] = o.min_ncc;
  s_red[(grp * 4 + 2) * kTile + px] = min_sob;
  s_red[(grp * 4 + 3) * kTile + px] = o.min_sad;
}

// Census channels from a parked census byte (255 = no cost), by arithmetic:
//  channel 0 = min(k,120)/120 as q = k*r, q' = fma(fma(-120, q, k), r, q) with r = fl(1/120): correctly
//  rounded (= the true IEEE division NumPy does) for every k in 0..255, checked exhaustively in
//  tests/test_host_math.py;  AML term = 2^(-(k-m)^2 k_cen), 0 for "no cost".
// Only the denominator chain takes the AML term from a shared-memory table instead (random indices: ~2.2
// wavefronts per load).  Measured at config B (ms/pair): no table 0.796, table in the chain 0.777 (the census
// chain is phase 2's critical path: a table load is its cheapest step), also for channel 0 0.787, also in
// phase 3 0.786.
__device__ __forceinline__ float cen_ch0(int cb) {
  const float k = (float)min(cb, 120);
  const float r = 1.0f / 120.0f;
  const float q = __fmul_rn(k, r);
  return __fmaf_rn(__fmaf_rn(-120.0f, q, k), r, q);
}
// The four parked census bytes of a pixel quad as floats WITHOUT integer conversions: PRMT drops a byte into
// the mantissa of 2^23, so as_float(word) - 2^23 is the byte (one packed FADD2 per two pixels, and the
// subtraction can carry any other integer with it).  kSignFill: bit 7 of the byte (set only by the 255 that
// stands for "no cost") is replicated into mantissa bits 8-15, so "no cost" becomes 65535 -- an AML argument
// that underflows to exactly 0 for every sigma below 1e7 (checked by the launcher), which is what the
// reference's fill does.
template <unsigned kSel>   // prmt.b32 in its default mode: a selector nibble with bit 3 set replicates the byte's sign
__device__ __forceinline__ float prmt_f(uint32_t a, uint32_t b) {   // (__byte_perm masks that bit away)
  float r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=f"(r) : "r"(a), "r"(b), "n"(kSel));
  return r;
}
template <bool kSignFill>
__device__ __forceinline__ float4 cen_bytes_as_biased_floats(uint32_t cw) {
  constexpr unsigned base = 0x4B000000u;   // 2^23
  float4 f;
  f.x = prmt_f<kSignFill ? 0x7480u : 0x7440u>(cw, base);
  f.y = prmt_f<kSignFill ? 0x7491u : 0x7441u>(cw, base);
  f.z = prmt_f<kSignFill ? 0x74A2u : 0x7442u>(cw, base);
  f.w = prmt_f<kSignFill ? 0x74B3u : 0x7443u>(cw, base);
  return f;
}
// Channel 0 of four pixels, min(k,120)/120 with cen_ch0's three operations per value, packed.  The clamp moves to
// the end as a free saturation: k <= 120 gives a quotient <= 1 that the saturation leaves alone, and the only other
// byte, 255 ("no cost"), gives 2.125, which saturates to the 1.0 that clip(fill, 0, 120) / 120 is.
__device__ __forceinline__ float4 cen_ch0_quad(uint32_t cw) {
  const float4 f = cen_bytes_as_biased_floats<false>(cw);
  const f32x2 b2 = pk2(8388608.0f, 8388608.0f), r2 = pk2(1.0f / 120.0f, 1.0f / 120.0f), n2 = pk2(-120.0f, -120.0f);
  const f32x2 k01 = sub2(pk2(f.x, f.y), b2), k23 = sub2(pk2(f.z, f.w), b2);
  const f32x2 q01 = mul2(k01, r2), q23 = mul2(k23, r2);
  float4 q, e;
  upk2(q01, q.x, q.y); upk2(q23, q.z, q.w);
  upk2(fma2(n2, q01, k01), e.x, e.y); upk2(fma2(n2, q23, k23), e.z, e.w);
  const float r = 1.0f / 120.0f;
  return make_float4(__saturatef(__fmaf_rn(e.x, r, q.x)), __saturatef(__fmaf_rn(e.y, r, q.y)),
                     __saturatef(__fmaf_rn(e.z, r, q.z)), __saturatef(__fmaf_rn(e.w, r, q.w)));
}
template <bool kLut, bool kExact = false>
__device__ __forceinline__ float cen_e(int cb, int mc, const float* s_lut, float k_cen) {
  if (kLut) return s_lut[min(cb - mc, 127)];     // (the table is built in the launch's AML mode)
  const float t = (float)(cb - mc);
  const float e = kExact ? aml_e_exact(t, 0.f, -k_cen) : aml_e_fast(t, 0.f, k_cen);
  return (cb - mc > 120) ? 0.f : e;
}
// AML term in the kernel's mode: kExact instantiations carry k = -sigma (feature_math.cuh)
template <bool kExact>
__device__ __forceinline__ float aml_t(float c, float m, float k) {
  return kExact ? aml_e_exact(c, m, -k) : aml_e_fast(c, m, k);
}

// Stores four channel planes' 4-pixel row segments: 128-bit streaming stores when the rows are
// 16 B aligned and the quad is fully inside the image (kVec), guarded scalars otherwise.
template <bool kVec, class T>
__device__ __forceinline__ void store_quads(T* o, size_t chan, int nlive, const float4& c0, const float4& c1,
                                            const float4& c2, const float4& c3) {
  if (kVec) {
    st_stream4(o, c0);
    st_stream4(o + chan, c1);
    st_stream4(o + 2 * chan, c2);
    st_stream4(o + 3 * chan, c3);
  } else {
    const float cc[4][4] = {{c0.x, c0.y, c0.z, c0.w}, {c1.x, c1.y, c1.z, c1.w}, {c2.x, c2.y, c2.z, c2.w},
                            {c3.x, c3.y, c3.z, c3.w}};
#pragma unroll
    for (int ch = 0; ch < 4; ++ch)
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (i < nlive) st_stream(o + ch * chan + i, cc[ch][i]);
  }
}

// ---- back half of a tile: channels 0-3, AML denominators, channels 4-7 --------------------
// Channels 0-3 (cbmv_generator.py:283-287) for thread = (pixel quad q4, disparities d0, d0+16, ... < d1):
// normalised costs stored as 128-bit row segments.
template <bool kVec, class T>
__device__ __forceinline__ void store_ch03(const float* s_par, const uint8_t* s_cen, int PS, int q4, int d0, int d1,
                                           T* orow, size_t plane, size_t chan, int nlive) {
  // (the output row is a pointer that advances by 16 planes per sweep: written as orow + d * plane, ptxas
  // redoes the 64-bit product every iteration -- ten more ALU-pipe instructions per four stores)
  T* o = orow + (size_t)d0 * plane;
  const size_t ostep = 16 * plane;
#pragma unroll 1   // (measured: unrolling the back half's sweeps is slower)
  for (int d = d0; d < d1; d += 16, o += ostep) {
    const float* e0 = s_par + d * kTile + q4;
    const uint32_t cw = *reinterpret_cast<const uint32_t*>(s_cen + d * kTile + q4);
    const float4 v1 = *reinterpret_cast<const float4*>(e0);
    const float4 v2 = *reinterpret_cast<const float4*>(e0 + PS);
    const float4 v3 = *reinterpret_cast<const float4*>(e0 + 2 * PS);
    const float4 c0 = cen_ch0_quad(cw);
    const float4 c1 = make_float4(normalise_cost(v1.x, 1), normalise_cost(v1.y, 1), normalise_cost(v1.z, 1),
                                  normalise_cost(v1.w, 1));
    const float4 c2 = make_float4(normalise_cost(v2.x, 2), normalise_cost(v2.y, 2), normalise_cost(v2.z, 2),
                                  normalise_cost(v2.w, 2));
    const float4 c3 = make_float4(normalise_cost(v3.x, 3), normalise_cost(v3.y, 3), normalise_cost(v3.z, 3),
                                  normalise_cost(v3.w, 3));
    store_quads<kVec>(o, chan, nlive, c0, c1, c2, c3);
  }
}

// Four pixels of one matcher: exp(-(c-m)^2/sigma) * (1/den), two pixels per packed operation.
__device__ __forceinline__ void p3_quad(const float4& v, const f32x2 (&m)[2], const f32x2 (&inv)[2], f32x2 negk,
                                        float4& out) {
  float e0, e1, e2, e3;
  aml_e2(pk2(v.x, v.y), m[0], negk, e0, e1);
  aml_e2(pk2(v.z, v.w), m[1], negk, e2, e3);
  upk2(mul2(pk2(e0, e1), inv[0]), out.x, out.y);
  upk2(mul2(pk2(e2, e3), inv[1]), out.z, out.w);
}

__device__ __forceinline__ void p3_quad_exact(const float4& v, const float4& m, const float4& den, float sigma, float4& out) {
  out.x = __fdiv_rn(aml_e_exact(v.x, m.x, sigma), den.x);
  out.y = __fdiv_rn(aml_e_exact(v.y, m.y, sigma), den.y);
  out.z = __fdiv_rn(aml_e_exact(v.z, m.z, sigma), den.z);
  out.w = __fdiv_rn(aml_e_exact(v.w, m.w, sigma), den.w);
}

// Channels 4-7 = exp(-(c-m)^2/sigma) / den for thread = (pixel quad q4, disparities dl, dl+32, ...),
// exponentials recomputed from the parked costs, 128-bit row segments.
template <bool kVec, class T, bool kExact = false>
__device__ __forceinline__ void phase3_quads(const float* s_par, const uint8_t* s_cen, const float* s_lut,
                                             const float* s_min, const float* s_inv, int PS, int q4, int dl, int D,
                                             T* arow, size_t plane, size_t chan, int nlive, float k0, float k1, float k2) {
  const float4 m_cen4 = *reinterpret_cast<const float4*>(s_min + q4);
  const float4 m1 = *reinterpret_cast<const float4*>(s_min + kTile + q4);
  const float4 m2 = *reinterpret_cast<const float4*>(s_min + 2 * kTile + q4);
  const float4 m3 = *reinterpret_cast<const float4*>(s_min + 3 * kTile + q4);
  const float4 i0 = *reinterpret_cast<const float4*>(s_inv + q4);
  const float4 i1 = *reinterpret_cast<const float4*>(s_inv + kTile + q4);
  const float4 i2 = *reinterpret_cast<const float4*>(s_inv + 2 * kTile + q4);
  const float4 i3 = *reinterpret_cast<const float4*>(s_inv + 3 * kTile + q4);
  const f32x2 mp1[2] = {pk2(m1.x, m1.y), pk2(m1.z, m1.w)}, ip1[2] = {pk2(i1.x, i1.y), pk2(i1.z, i1.w)};
  const f32x2 mp2[2] = {pk2(m2.x, m2.y), pk2(m2.z, m2.w)}, ip2[2] = {pk2(i2.x, i2.y), pk2(i2.z, i2.w)};
  const f32x2 mp3[2] = {pk2(m3.x, m3.y), pk2(m3.z, m3.w)}, ip3[2] = {pk2(i3.x, i3.y), pk2(i3.z, i3.w)};
  const f32x2 nk1 = pk2(-k1, -k1), nk2 = pk2(-k2, -k2), nk0 = pk2(-k0, -k0);
  const int mcx = (m_cen4.x == kFill) ? 0 : (int)m_cen4.x, mcy = (m_cen4.y == kFill) ? 0 : (int)m_cen4.y;
  const int mcz = (m_cen4.z == kFill) ? 0 : (int)m_cen4.z, mcw = (m_cen4.w == kFill) ? 0 : (int)m_cen4.w;
  // census minima biased by 2^23 (exact: the minima are integers <= 120), see cen_bytes_as_biased_floats
  const f32x2 mp0[2] = {pk2(8388608.0f + (float)mcx, 8388608.0f + (float)mcy), pk2(8388608.0f + (float)mcz, 8388608.0f + (float)mcw)};
  const f32x2 ip0[2] = {pk2(i0.x, i0.y), pk2(i0.z, i0.w)};
#pragma unroll 1   // (measured: unrolling by 2 is slower)
  for (int d = dl; d < D; d += 32) {
    const float* e0 = s_par + d * kTile + q4;
    const uchar4 cb = *reinterpret_cast<const uchar4*>(s_cen + d * kTile + q4);
    const float4 v1 = *reinterpret_cast<const float4*>(e0);
    const float4 v2 = *reinterpret_cast<const float4*>(e0 + PS);
    const float4 v3 = *reinterpret_cast<const float4*>(e0 + 2 * PS);
    float4 a0, a1, a2, a3;
    if (kExact) {   // s_inv holds the denominators themselves (INFINITY where the pixel has no cost)
      a0 = make_float4(__fdiv_rn(cen_e<false, true>(cb.x, mcx, s_lut, k0), i0.x), __fdiv_rn(cen_e<false, true>(cb.y, mcy, s_lut, k0), i0.y),
                       __fdiv_rn(cen_e<false, true>(cb.z, mcz, s_lut, k0), i0.z), __fdiv_rn(cen_e<false, true>(cb.w, mcw, s_lut, k0), i0.w));
      p3_quad_exact(v1, m1, i1, -k1, a1);
      p3_quad_exact(v2, m2, i2, -k2, a2);
      p3_quad_exact(v3, m3, i3, -k2, a3);
    } else {
      // (byte + 2^23) - (min + 2^23) = the integer difference cen_e squares; "no cost" is 65535 - min: exactly 0
      p3_quad(cen_bytes_as_biased_floats<true>(*reinterpret_cast<const uint32_t*>(&cb)), mp0, ip0, nk0, a0);
      p3_quad(v1, mp1, ip1, nk1, a1);
      p3_quad(v2, mp2, ip2, nk2, a2);
      p3_quad(v3, mp3, ip3, nk2, a3);
    }
    store_quads<kVec>(arow + (size_t)d * plane, chan, nlive, a0, a1, a2, a3);
  }
}

// AML denominator of one (pixel, matcher) over the launch's disparities: exponentials evaluated on the fly
// and added in the reference's order -- sequential fp32 over d (featextract.cpp:444-447; a tree sum is
// measurably outside the 2e-6 bound).  warp = matcher, lane = pixel, mm = the minimum the exponent refers to.
template <class L, bool kExact = false>
__device__ __forceinline__ float den_chain(const FusedArgs& a, int warp, int lane, float mm, const float* s_par,
                                           const uint8_t* s_cen, const float* s_lut) {
  constexpr int PS = L::PS;
  const int D = a.g.D;
  float den = 0.f;
  constexpr int B = 8;           // exponentials evaluated ahead of the denominator's dependent adds
  const int Dfull = D - D % B;   // groups of B without guards, then a guarded tail
  if (warp == 0) {
    const int mc = (mm == kFill) ? 0 : (int)mm;
    const uint8_t* c = s_cen + lane;
    for (int d0 = 0; d0 < Dfull; d0 += B, c += B * kTile) {
      float ev[B];
#pragma unroll
      for (int j = 0; j < B; ++j) ev[j] = cen_e<true, kExact>(c[j * kTile], mc, s_lut, a.k_cen);
#pragma unroll
      for (int j = 0; j < B; ++j) den = __fadd_rn(den, ev[j]);
    }
    for (int d = Dfull; d < D; ++d, c += kTile) den = __fadd_rn(den, cen_e<true, kExact>(c[0], mc, s_lut, a.k_cen));
  } else {
    const float kq = (warp == 1) ? a.k_ncc : a.k_sad;
    const f32x2 mm2 = pk2(mm, mm), nkq = pk2(-kq, -kq);
    const float* e = s_par + (warp - 1) * PS + lane;
    for (int d0 = 0; d0 < Dfull; d0 += B, e += B * kTile) {
      float ev[B];
#pragma unroll
      for (int j = 0; j < B; j += 2) {
        if (kExact) { ev[j] = aml_e_exact(e[j * kTile], mm, -kq); ev[j + 1] = aml_e_exact(e[(j + 1) * kTile], mm, -kq); }
        else aml_e2(pk2(e[j * kTile], e[(j + 1) * kTile]), mm2, nkq, ev[j], ev[j + 1]);
      }
#pragma unroll
      for (int j = 0; j < B; ++j) den = __fadd_rn(den, ev[j]);
    }
    for (int d = Dfull; d < D; ++d, e += kTile) den = __fadd_rn(den, aml_t<kExact>(e[0], mm, kq));
  }
  return den;
}

// ---- disparity-slab exchange between ranks, inside the tile (SURVEY.md 8e) -------------------------
// Every rank computes its own slab of disparities for the SAME tiles; the AML minimum and denominator of
// a pixel need all slabs.  Instead of parking raw costs in HBM and making two more passes over the volume
// around two NCCL all-reduces, the tile keeps its costs in shared memory and trades 2 x 128 floats with the
// other ranks through peer-mapped memory (NVLink / NVSwitch): it WRITES its per-pixel minima into every
// rank's table and reads the other ranks' values from its own.  The payload travels LL128-style: a line is
// 31 values + a flag word (the frame's epoch), written by one warp as one aligned 128-byte store, so a
// reader that sees the flag in a line it loaded in one piece has the line's values -- no fence, no separate
// flag round trip.  Tables are double-buffered by the epoch's low bit: a rank can only be two frames ahead
// of a peer's unread data after that peer has finished the frame in between.
__device__ __forceinline__ size_t xchg_line0(const FusedArgs& a, int round, long long tile, int src) {
  return (((((size_t)(a.xchg.epoch & 1u) * 2 + round) * a.n_tiles + tile) * a.xchg.V + src) * kXLines) *
         kXLineWords;
}
// Warps 0-3: the 128 values in vals[] (shared memory) go to every rank's table as lines k = warp (+ 4 for warp 0).
__device__ __forceinline__ void xchg_publish(const FusedArgs& a, int round, long long tile, int v, int warp, int lane,
                                             const float* vals) {
  for (int k = warp; k < kXLines; k += 4) {
    const int i = 31 * k + lane;
    const unsigned w = (lane == 31) ? a.xchg.epoch : ((i < 128) ? __float_as_uint(vals[i]) : 0u);
    const size_t off = xchg_line0(a, round, tile, v) + (size_t)k * kXLineWords + lane;
    for (int p = 0; p < a.xchg.G; ++p)
      asm volatile("st.volatile.global.u32 [%0], %1;" ::"l"(a.xchg.peer[p] + off), "r"(w) : "memory");
  }
}
// Warps 0-3: waits for every source's lines of this tile and folds them in source order (kSum: a + b, else
// min) into out[0..128).  All the loads of a polling round are issued before the first flag is examined (8
// sources at a time), so a round costs one trip to L2, not one per source.  A peer that never shows up
// (crashed rank, mismatched launch) trips a trap after ~2 s instead of hanging the GPU.
template <bool kSum>
__device__ __forceinline__ void xchg_collect(const FusedArgs& a, int round, long long tile, int warp, int lane,
                                             float* out) {
  const unsigned* mine = a.xchg.peer[a.xchg.rank];
  const unsigned epoch = a.xchg.epoch;
  for (int k = warp; k < kXLines; k += 4) {
    float acc = kSum ? 0.f : kFill;
    for (int s0 = 0; s0 < a.xchg.V; s0 += 8) {
      const int ns = min(8, a.xchg.V - s0);
      const unsigned* line = mine + xchg_line0(a, round, tile, s0) + (size_t)k * kXLineWords + lane;
      unsigned w[8];
      unsigned pending = (1u << ns) - 1u;
      long long t0 = 0;
      for (unsigned spins = 0; pending; ++spins) {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if ((pending >> j) & 1u)
            asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(w[j]) : "l"(line + (size_t)j * kXLines * kXLineWords) : "memory");
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (((pending >> j) & 1u) && __shfl_sync(0xffffffffu, w[j], 31) == epoch) pending &= ~(1u << j);
        if (pending) {
          if (spins == 16) t0 = clock64();
          if (spins > 16) {
            __nanosleep(100);
            if (clock64() - t0 > 4000000000LL) __trap();
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j)
        if (j < ns) {
          const float v = __uint_as_float(w[j]);
          acc = kSum ? __fadd_rn(acc, v) : fminf(acc, v);
        }
    }
    const int i = 31 * k + lane;
    if (lane < 31 && i < 128) out[i] = acc;
  }
}
__device__ __forceinline__ void bar_sync_128() { asm volatile("bar.sync 1, 128;" ::: "memory"); }

// Winner-take-all by-product for one (pixel, matcher): a sequential sweep over the parked costs with the values
// channels 0-3 carry (the reference takes np.argmin of those, main_msnet.py:444-448): first minimal index wins;
// min2 is the second smallest entry counting duplicates (oracle/ms_oracle.py wta).  m = matcher, lane = pixel.
template <class L>
__device__ __forceinline__ void wta_scan(const FusedArgs& a, const TileId& t, int m, int lane, const float* s_par,
                                         const uint8_t* s_cen) {
  constexpr int PS = L::PS;
  const int D = a.g.D;
  float m1 = INFINITY, m2 = INFINITY;
  int idx = 0;
  if (m == 0) {
    const uint8_t* c = s_cen + lane;
#pragma unroll 4
    for (int d = 0; d < D; ++d) {
      const float v = cen_ch0(c[d * kTile]);
      if (v < m1) { m2 = m1; m1 = v; idx = d; }
      else if (v < m2) m2 = v;
    }
  } else {
    const float* e = s_par + (m - 1) * PS + lane;
#pragma unroll 4
    for (int d = 0; d < D; ++d) {
      const float v = normalise_cost(e[d * kTile], m);
      if (v < m1) { m2 = m1; m1 = v; idx = d; }
      else if (v < m2) m2 = v;
    }
  }
  const int x = t.x0 + lane;
  if (x < a.g.w) {
    const size_t plane = (size_t)a.g.h * a.g.w;
    const size_t o = (((size_t)(t.sub0 / a.g.D) * a.g.N + t.n) * 4 + m) * plane + (size_t)t.yl * a.g.w + x;
    a.wta_idx[o] = t.d0 + idx;
    a.wta_min1[o] = m1;
    a.wta_min2[o] = m2;
  }
}

// Phases 2 and 3 for the 256 threads of a CTA.  s_red holds the per-group minima of phase 1.
//   phase 2 (warp-specialised; both halves only READ the parked costs, so they overlap without
//            hazards):
//     warps 0-3  one thread per (pixel, matcher): AML denominator (den_chain);
//     warps 4-7  thread = (pixel quad, d): channels 0-3 normalised and stored.
//   phase 3      all warps: channels 4-7.
// kXchg (disparity-slab sharding): warps 0-3 first trade the slab's minima with the other ranks, add the
// denominator of their OWN disparities against the global minimum, trade the partial denominators and add
// them in rank order -- while warps 4-7 store channels 0-3, which need nothing from anybody.
// Measured alternatives (DESIGN.md section 4): writing each exponential back in place and adding
// the denominators in a phase of their own (fewer instructions, 6 % slower: the chain is
// exposed), the same behind a progress counter (slower still: the chain warps spin), handing
// part of the channel 0-3 stores to the chain warps statically or through a work counter (no
// gain: the halves are already balanced), a warp-specialised persistent producer/consumer
// kernel (15 % slower).
template <class L, bool kXchg, class T = float, bool kExact = false>
__device__ __forceinline__ void tile_back_half(const FusedArgs& a, const TileId& t, long long tile, int tid,
                                               const float* s_par, const uint8_t* s_cen, float* s_red, float* s_min,
                                               float* s_inv, const float* s_lut) {
  constexpr int PS = L::PS;
  const FusedGeom& g = a.g;
  const int D = g.D;
  const size_t plane = (size_t)g.h * g.w;
  const size_t chan = plane * a.out_D;
  // Minima across the d-groups.  Only the chain warps need them before phase 3 and thread tid < 128 is exactly the
  // (matcher, pixel) whose chain it runs, so outside the exchange form each of them folds its own eight values and
  // no barrier separates this from phase 2 (the store warps start on channels 0-3 at once).
  float mm_own = kFill;
  if (tid < 4 * kTile) {
#pragma unroll
    for (int gq = 0; gq < kGroups; ++gq) mm_own = fminf(mm_own, s_red[gq * 4 * kTile + tid]);
    (kXchg ? s_inv : s_min)[tid] = mm_own;   // (kXchg: this rank's slab minima, staged in s_inv for the exchange)
  }
  if (kXchg) __syncthreads();
  const int warp = tid >> 5, lane = tid & 31;
  const int q4 = (tid & 7) * 4;
  // 128-bit stores need 16-byte aligned rows
  const bool vec_ok = ((g.w & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.out) & 15) == 0);
  T* orow = reinterpret_cast<T*>(a.out) + ((size_t)t.n * a.out_channels + a.out_ch0) * chan + (size_t)(a.out_d0 + t.sub0) * plane + (size_t)t.yl * g.w + (t.x0 + q4);
  const int nlive = min(4, g.w - (t.x0 + q4));  // live pixels of this quad (<= 0: none)
  const bool vec = vec_ok && nlive == 4;
  if (warp < 4) {
    if (kXchg) {
      xchg_publish(a, 0, tile, t.v, warp, lane, s_inv);
      xchg_collect<false>(a, 0, tile, warp, lane, s_min);
      bar_sync_128();
    }
    const float mm = kXchg ? s_min[warp * kTile + lane] : mm_own;
    float den = den_chain<L, kExact>(a, warp, lane, mm, s_par, s_cen, s_lut);
    if (kXchg) {
      s_red[warp * kTile + lane] = den;        // (the per-group minima are dead since the barrier above)
      bar_sync_128();
      xchg_publish(a, 1, tile, t.v, warp, lane, s_red);
      xchg_collect<true>(a, 1, tile, warp, lane, s_red + 4 * kTile);
      bar_sync_128();
      den = s_red[4 * kTile + warp * kTile + lane];
    }
    s_inv[warp * kTile + lane] = kExact ? ((mm == kFill) ? INFINITY : den) : ((mm == kFill) ? 0.f : 1.0f / den);
  }
  else {
    // channels 0-3: thread = (pixel quad, d), 16 disparities per sweep of the four warps
    if (vec) store_ch03<true>(s_par, s_cen, PS, q4, (tid >> 3) - 16, D, orow, plane, chan, nlive);
    else store_ch03<false>(s_par, s_cen, PS, q4, (tid >> 3) - 16, D, orow, plane, chan, nlive);
    if (a.wta_idx) wta_scan<L>(a, t, warp - 4, lane, s_par, s_cen);
  }
  __syncthreads();
  const int dl = tid >> 3;
  if (vec) phase3_quads<true, T, kExact>(s_par, s_cen, s_lut, s_min, s_inv, PS, q4, dl, D, orow + 4 * chan, plane, chan, nlive, a.k_cen, a.k_ncc, a.k_sad);
  else phase3_quads<false, T, kExact>(s_par, s_cen, s_lut, s_min, s_inv, PS, q4, dl, D, orow + 4 * chan, plane, chan, nlive, a.k_cen, a.k_ncc, a.k_sad);
}

// Back half of a tile for DISPARITY-SLAB SHARDING (phase A of slab.cu, SURVEY.md 8e): the AML
// minimum and denominator need the other ranks' disparities, so the tile only stores channels
// 0-3, parks the RAW costs in channels 4-7 (census as float; fill where there is no cost) and
// writes the slab's per-pixel minima; slab_phase_b/c finish the job after the all-reduces.
template <class L>
__device__ __forceinline__ void tile_slab_a(const FusedArgs& a, const TileId& t, int tid, const float* s_par,
                                            const uint8_t* s_cen, const float* s_red) {
  constexpr int PS = L::PS;
  const FusedGeom& g = a.g;
  const int D = g.D;
  const size_t plane = (size_t)g.h * g.w;
  const size_t chan = plane * a.out_D;
  if (tid < 4 * kTile) {  // minima across the d-groups -> global
    float v = kFill;
#pragma unroll
    for (int gq = 0; gq < kGroups; ++gq) v = fminf(v, s_red[gq * 4 * kTile + tid]);
    const int m = tid / kTile, x = t.x0 + tid % kTile;
    if (x < g.w) {
      float* mp = a.mins + (((size_t)t.n * a.mins_planes + m) * g.h + t.yl) * g.w + x;
      *mp = a.mins_accumulate ? fminf(*mp, v) : v;
    }
  }
  const int q4 = (tid & 7) * 4;
  const int dl = tid >> 3;
  const bool vec_ok = ((g.w & 3) == 0) && ((reinterpret_cast<uintptr_t>(a.out) & 15) == 0);
  float* orow = a.out + (size_t)t.n * a.out_channels * chan + (size_t)t.yl * g.w + (t.x0 + q4);
  const int nlive = min(4, g.w - (t.x0 + q4));
  const bool vec = vec_ok && nlive == 4;
#pragma unroll 2
  for (int d = dl; d < D; d += 32) {
    const float* e0 = s_par + d * kTile + q4;
    const uchar4 cb = *reinterpret_cast<const uchar4*>(s_cen + d * kTile + q4);
    const float4 v1 = *reinterpret_cast<const float4*>(e0);
    const float4 v2 = *reinterpret_cast<const float4*>(e0 + PS);
    const float4 v3 = *reinterpret_cast<const float4*>(e0 + 2 * PS);
    const float4 v0 = make_float4(cb.x == 255 ? kFill : (float)cb.x, cb.y == 255 ? kFill : (float)cb.y,
                                  cb.z == 255 ? kFill : (float)cb.z, cb.w == 255 ? kFill : (float)cb.w);
    const float4 c0 = make_float4(cen_ch0(cb.x), cen_ch0(cb.y), cen_ch0(cb.z), cen_ch0(cb.w));
    const float4 c1 = make_float4(normalise_cost(v1.x, 1), normalise_cost(v1.y, 1), normalise_cost(v1.z, 1),
                                  normalise_cost(v1.w, 1));
    const float4 c2 = make_float4(normalise_cost(v2.x, 2), normalise_cost(v2.y, 2), normalise_cost(v2.z, 2),
                                  normalise_cost(v2.w, 2));
    const float4 c3 = make_float4(normalise_cost(v3.x, 3), normalise_cost(v3.y, 3), normalise_cost(v3.z, 3),
                                  normalise_cost(v3.w, 3));
    float* o = orow + (size_t)(a.out_d0 + d) * plane;
    if (vec) {
      store_quads<true>(o, chan, nlive, c0, c1, c2, c3);
      // parked raw costs are read again by slab_phase_b/c: plain (cached) stores
      *reinterpret_cast<float4*>(o + 4 * chan) = v0;
      *reinterpret_cast<float4*>(o + 5 * chan) = v1;
      *reinterpret_cast<float4*>(o + 6 * chan) = v2;
      *reinterpret_cast<float4*>(o + 7 * chan) = v3;
    } else {
      store_quads<false>(o, chan, nlive, c0, c1, c2, c3);
      const float rr[4][4] = {{v0.x, v0.y, v0.z, v0.w}, {v1.x, v1.y, v1.z, v1.w}, {v2.x, v2.y, v2.z, v2.w},
                              {v3.x, v3.y, v3.z, v3.w}};
#pragma unroll
      for (int ch = 0; ch < 4; ++ch)
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (i < nlive) o[(4 + ch) * chan + i] = rr[ch][i];
    }
  }
}

// ---- one CTA per tile (fallback: any D up to 448, with or without TMA) ----------------------
//   phase 1  thread = (pixel, d-group): 8 warps split D (phase1_tile)
//   phase 2  thread = (pixel quad, d): channels 0-3 stored, costs -> AML exponentials in place
//   phase 2b one thread per (pixel, matcher): sequential denominator
//   phase 3  thread = (pixel quad, d): channels 4-7 = exponential / den
// kTma: right-image rows and the SAD-of-Sobel tile arrive through cp.async.bulk /
// cp.async.bulk.tensor (D <= 256: box limit); otherwise through LDGSTS.  The tensor copy's
// inner coordinate must be a multiple of 16 bytes (measured: anything else raises an
// illegal-instruction fault), which is why the scratch is stored with column offset sxo.
// kMode: kModeFull the whole volume; kModeSlabA stop after phase 1 and emit what slab.cu's phase A emits
// (tile_slab_a); kModeXchg a rank's disparity slab, minima and denominators traded inside the tile.
template <int DMAX, bool kTma, int kMode>
__device__ __forceinline__ void fused_tile(const FusedArgs& a, const CUtensorMap& sad_map, long long tile, int sub) {
  using L = Lay<DMAX, kSlack>;
  constexpr int NT = 256;
  constexpr int PS = L::PS;
  extern __shared__ __align__(128) unsigned char smem_raw[];  // TMA destinations need 128 B
  const FusedGeom& g = a.g;
  const int D = g.D;
  unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(smem_raw + L::off_bar);  // [0] rows, [1] sadsob tile
  float* s_red = reinterpret_cast<float*>(smem_raw + L::off_red);    // [8][4][32]
  float* s_min = reinterpret_cast<float*>(smem_raw + L::off_min);
  float* s_inv = reinterpret_cast<float*>(smem_raw + L::off_inv);
  float* s_lut = reinterpret_cast<float*>(smem_raw + L::off_lut);
  float* s_lutn = reinterpret_cast<float*>(smem_raw + L::off_lutn);
  float* s_par = reinterpret_cast<float*>(smem_raw + L::off_par);    // [3][DS][32]
  uint8_t* s_cen = smem_raw + L::off_par + L::pk_cen;                // [DS][32]
  const int tid = threadIdx.x;
  const int px = tid % kTile;             // phase 1: this thread's pixel ...
  const int grp = tid / kTile;            // ... and d-group
  const TileId t = decode_tile((int)tile, a, sub);
  const int d_lo = grp * a.DC;
  const int d_end = min(D, d_lo + a.DC);  // real disparities of this thread: [d_lo, d_end)
  if (kMode == kModeRight) {
    // The right view: left-image rows through bulk copies (any D: no tensor box), this thread's own SAD-of-Sobel
    // costs -- right(xr, d) = scratch(d, y, xr + d), a diagonal no box describes -- through LDGSTS, only where
    // the cost exists (finish_right fills the rest).
    if (tid == 0) {
      mbar_init(&s_bar[0], 1);
      mbar_init_fence();
      stage_rows_tma<L, true>(a, t, smem_raw, &s_bar[0]);
    }
    if (tid < 128) s_lut[tid] = __ldg(a.luts + tid);
    s_lutn[tid] = __ldg(a.luts + 128 + tid);
    {
      const int Xr = t.x0 + px + g.bwl, Y = t.y + g.bh;
      const int dcrop = (g.w - 1 - (t.x0 + px)) - t.d0;
      const int dmax_sad = min(min(D - 1, dcrop), ((Y >= 2 && Y < g.H - 3 && Xr >= 2) ? g.W - 4 - Xr : -1) - t.d0);
      const size_t splane = g.d_inner ? (size_t)g.Ws : (size_t)g.H * g.Ws;
      const size_t row0 = g.d_inner ? (((size_t)t.n * g.H + (t.y + g.bh)) * g.Dl + t.sub0) * g.Ws
                                    : (((size_t)t.n * g.Dl + t.sub0) * g.H + (t.y + g.bh)) * g.Ws;
      const float* src = a.sadsob + row0 + (Xr + t.d0 + g.sxo) + (size_t)d_lo * (splane + 1);
      float* dst = s_par + PS + d_lo * kTile + px;
      const int dl = min(d_end, dmax_sad + 1);
      for (int d = d_lo; d < dl; ++d, src += splane + 1, dst += kTile) cp_async4(dst, src);
    }
    LeftRegs rr;
    load_left<true>(a, t, px, rr);
    __syncthreads();
    mbar_wait(&s_bar[0], 0);
    const Phase1RightOut ro = phase1_tile_right<L>(a, t, smem_raw, s_par, s_cen, rr, px, d_lo);
    cp_async_wait_all();
    finish_right<L>(s_par, s_cen, s_red, ro, a.first4 + 4 * t.n, px, grp, d_lo, d_end);
    __syncthreads();
    tile_back_half<L, false>(a, t, tile, tid, s_par, s_cen, s_red, s_min, s_inv, s_lut);
    return;
  }
  if (kTma) {
    if (tid == 0) {
      mbar_init(&s_bar[0], 1);
      mbar_init(&s_bar[1], 1);
      mbar_init_fence();
      // rows first: phase 1 waits for them; the SAD-of-Sobel box is only needed after phase 1
      stage_rows_tma<L>(a, t, smem_raw, &s_bar[0]);
      stage_sad_tma(a, &sad_map, t, s_par + PS, &s_bar[1]);
    }
  } else {
    // sadsob costs of this thread's own disparities: async global -> parked plane 1
    const size_t splane = g.d_inner ? (size_t)g.Ws : (size_t)g.H * g.Ws;
    const size_t row0 = g.d_inner ? (((size_t)t.n * g.H + (t.y + g.bh)) * g.Dl + t.sub0) * g.Ws
                                  : (((size_t)t.n * g.Dl + t.sub0) * g.H + (t.y + g.bh)) * g.Ws;
    const float* src = a.sadsob + row0 + (t.x0 + px + g.bwl + g.sxo) + (size_t)d_lo * splane;
    float* dst = s_par + PS + d_lo * kTile + px;
    for (int d = d_lo; d < d_end; ++d, src += splane, dst += kTile) cp_async4(dst, src);
    stage_right<L, NT>(a, t, smem_raw);
  }
  if (tid < 128) s_lut[tid] = __ldg(a.luts + tid);
  s_lutn[tid] = __ldg(a.luts + 128 + tid);
  LeftRegs lr;
  load_left(a, t, px, lr);
  if (!kTma) cp_async_wait_all();
  __syncthreads();                       // barrier init, LUTs (and LDGSTS data) visible to everyone
  if (kTma) mbar_wait(&s_bar[0], 0);

  const Phase1Out o = phase1_tile<L>(a, t, smem_raw, s_par, s_cen, lr, px, d_lo);
  if (kTma) mbar_wait(&s_bar[1], 0);
  finish_phase1<L>(s_par, s_red, o, px, grp, d_lo, d_end);
  __syncthreads();
  if (kMode == kModeFull || kMode == kModeExact) {
    // both views requested: the raw costs of cropped voxel (0, 0, 0) are what get_right_cost fills with
    if (a.first4_out && tid < 4 && t.yl == 0 && g.y0 == 0 && t.x0 == 0 && t.d0 == 0) {
      const float v = (tid == 0) ? ((s_cen[0] == 255) ? kFill : (float)s_cen[0]) : s_par[(tid - 1) * PS];
      a.first4_out[4 * t.n + tid] = v;
    }
  }
  if (kMode == kModeSlabA) tile_slab_a<L>(a, t, tid, s_par, s_cen, s_red);
  else if (kMode == kModeExact) tile_back_half<L, false, float, true>(a, t, tile, tid, s_par, s_cen, s_red, s_min, s_inv, s_lut);
  else if (kMode == kModeBf16) tile_back_half<L, false, __nv_bfloat16>(a, t, tile, tid, s_par, s_cen, s_red, s_min, s_inv, s_lut);
  else if (kMode == kModeXchg) tile_back_half<L, true>(a, t, tile, tid, s_par, s_cen, s_red, s_min, s_inv, s_lut);
  else tile_back_half<L, false>(a, t, tile, tid, s_par, s_cen, s_red, s_min, s_inv, s_lut);
}

template <int DMAX, bool kTma, int kMode>
__global__ void __launch_bounds__(256, 2)
ms_fused_kernel(const FusedArgs a, const __grid_constant__ CUtensorMap sad_map) {
  if (kMode == kModeXchg) {
    // CTA = (tile, sub-slab), sub-slab fastest: the CTAs that wait for each other's minima are dispatched
    // together.  A sub-slab is a virtual rank: its own disparity offset, its own row in the exchange tables.
    fused_tile<DMAX, kTma, kMode>(a, sad_map, blockIdx.x / (unsigned)a.subs, (int)(blockIdx.x % (unsigned)a.subs));
  } else {
    fused_tile<DMAX, kTma, kMode>(a, sad_map, blockIdx.x, 0);
  }
}

// Optional per-kernel timing (msn_profile_enable): CUDA events recorded on the launch
// stream between the kernels of the fused sequence, read back by msn_profile_read.
struct ProfRec { cudaEvent_t ev[4]; };
std::mutex g_prof_mu;
bool g_prof_on = false;
std::vector<ProfRec> g_prof;
constexpr size_t kProfMaxPending = 4096;   // records kept when nobody calls msn_profile_read

// cuTensorMapEncodeTiled results, keyed by what they describe (a launch sequence repeats the same map)
struct MapKey {
  const void* base;
  int Ws, H, ND, D, inner;
  bool operator==(const MapKey& o) const { return base == o.base && Ws == o.Ws && H == o.H && ND == o.ND && D == o.D && inner == o.inner; }
};
std::mutex g_map_mu;
std::vector<std::pair<MapKey, CUtensorMap>> g_maps;

}  // namespace

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
// cuTensorMapEncodeTiled through the runtime's driver entry-point lookup (no libcuda link)
static PFN_encodeTiled get_encode_fn() {
  static PFN_encodeTiled fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return (PFN_encodeTiled)p;
  }();
  return fn;
}
static bool tma_disabled() {
  const char* e = getenv("MSNETS_NO_TMA");
  return e && e[0] == '1';
}

// 3-D tensor map over the SAD-of-Sobel scratch: [N*D][H][Ws], box 32 x 1 x D -- or, d_inner, [N*H][D][Ws], box 32 x D x 1
static bool sad_tensor_map(const FusedGeom& g, int H, int N, const float* base, CUtensorMap* out) {
  const MapKey key{base, g.Ws, H, N * g.Dl, g.D, g.d_inner};
  {
    std::lock_guard<std::mutex> lk(g_map_mu);
    for (auto& kv : g_maps)
      if (kv.first == key) {
        *out = kv.second;
        return true;
      }
  }
  PFN_encodeTiled enc = get_encode_fn();
  if (!enc) return false;
  cuuint64_t gdim[3] = {(cuuint64_t)g.Ws, (cuuint64_t)H, (cuuint64_t)N * g.Dl};
  cuuint64_t gstr[2] = {(cuuint64_t)g.Ws * 4, (cuuint64_t)H * g.Ws * 4};
  cuuint32_t box[3] = {(cuuint32_t)kTile, 1u, (cuuint32_t)g.D};
  if (g.d_inner) {
    gdim[1] = (cuuint64_t)g.Dl; gdim[2] = (cuuint64_t)N * H;
    gstr[1] = (cuuint64_t)g.Dl * g.Ws * 4;
    box[1] = (cuuint32_t)g.D; box[2] = 1u;
  }
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  if (enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), gdim, gstr, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  std::lock_guard<std::mutex> lk(g_map_mu);
  if (g_maps.size() >= 64) g_maps.erase(g_maps.begin());
  g_maps.emplace_back(key, *out);
  return true;
}

// One launch of an instantiation; the dynamic shared-memory opt-in is set once per instantiation
// and device, not per launch.
template <int DMAX, bool kTma, int kMode>
static int launch_inst(const FusedArgs& a, const CUtensorMap& map, long long tiles, cudaStream_t s) {
  auto kern = ms_fused_kernel<DMAX, kTma, kMode>;
  constexpr size_t smem = Lay<DMAX, kSlack>::bytes;
  static std::mutex mu;
  static unsigned long long done_mask = 0;   // bit per device ordinal (< 64)
  int dev = 0;
  MSN_CUDA_OK(cudaGetDevice(&dev));
  {
    std::lock_guard<std::mutex> lk(mu);
    if (dev >= 64 || !((done_mask >> dev) & 1ull)) {
      MSN_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      if (dev < 64) done_mask |= 1ull << dev;
    }
  }
  kern<<<(unsigned)(tiles * (kMode == kModeXchg ? a.subs : 1)), 256, smem, s>>>(a, map);
  return 0;
}

int profile_enable(int on) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  g_prof_on = on != 0;
  if (!g_prof_on) {   // switching off drops whatever was never read
    for (ProfRec& r : g_prof)
      for (int i = 0; i < 4; ++i) cudaEventDestroy(r.ev[i]);
    g_prof.clear();
  }
  return 0;
}

int profile_read(double* prep_ms, double* sadsob_ms, double* fused_ms, int* calls) {
  std::lock_guard<std::mutex> lk(g_prof_mu);
  double t[3] = {0, 0, 0};
  for (ProfRec& r : g_prof) {
    MSN_CUDA_OK(cudaEventSynchronize(r.ev[3]));
    for (int i = 0; i < 3; ++i) {
      float ms = 0.f;
      MSN_CUDA_OK(cudaEventElapsedTime(&ms, r.ev[i], r.ev[i + 1]));
      t[i] += ms;
    }
    for (int i = 0; i < 4; ++i) cudaEventDestroy(r.ev[i]);
  }
  if (prep_ms) *prep_ms = t[0];
  if (sadsob_ms) *sadsob_ms = t[1];
  if (fused_ms) *fused_ms = t[2];
  if (calls) *calls = (int)g_prof.size();
  g_prof.clear();
  return 0;
}

size_t fused_exchange_bytes(int N, int H, int W, const msn_ms_params* p, int sources) {
  FusedGeom g = make_geom(N, H, W, p);
  const long long tiles = (long long)N * g.h * ((g.w + kTile - 1) / kTile);
  return (size_t)2 * 2 * tiles * sources * kXLines * kXLineWords * sizeof(unsigned);   // [half][round][tile][source][5][32]
}

bool fused_supported(const msn_ms_params* p, int Dn) {
  // cens_sigma < 1e7: the back half lets "no cost" underflow the census AML term to 0 (cen_bytes_as_biased_floats)
  return p->censw == kCensW && p->nccw == kNccW && p->sadw == kSadW && p->sobelw == kSadW &&
         p->cens_sigma < 1.0e7f && Dn <= kMaxFusedD;  // (image width is checked at launch; p->lr: the caller adds the right view)
}

size_t fused_workspace_bytes(int N, int H, int W, int Dn, const msn_ms_params* p) {
  (void)Dn;
  FusedGeom g = make_geom(N, H, W, p);
  FusedWs ws;
  ws.carve(nullptr, g);
  return ws.total;
}

// d_mins == nullptr: the whole feature volume (p describes all disparities).  Otherwise phase A of
// the slab path for disparities [p->d_begin, p->d_begin + p->d_count): the output tensor holds
// out_D disparities per channel and the slab starts at out_d0 in it (a rank's own slab tensor:
// out_D = d_count, out_d0 = 0; slabs of one big volume on one GPU: out_D = ndisp, out_d0 = d_begin,
// accumulate != 0 from the second slab on).
int launch_ms_fused(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W, const msn_ms_params* p,
                    float* d_out, float* d_mins, char* workspace, cudaStream_t s, int out_D, int out_d0,
                    int accumulate, const msn_slab_exchange* xchg, const FusedWta* wta, bool out_bf16) {
  MSN_REQUIRE(!out_bf16 || (!xchg && !d_mins), "ms_features: the bf16 volume is written by the one-pass kernel only");
  const bool exact = g_aml_exact != 0 && !d_mins;   // (the phase-A form computes no AML: phases B/C follow the mode)
  MSN_REQUIRE(!exact || (!xchg && !out_bf16), "ms_features: the exact AML mode is not served by the slab exchange / bf16 forms");
  if (N == 0) return 0;
  FusedGeom g = make_geom(N, H, W, p);
  FusedWs ws;
  ws.carve(workspace, g);
  MSN_REQUIRE(2 * N <= 65535 && g.Hp <= 65535, "ms_features: batch or image too large for one launch");
  const int subs = (xchg && xchg->subs > 1) ? xchg->subs : 1;
  MSN_REQUIRE(g.Dl % subs == 0, "ms_slab_fused: %d disparities do not split into %d equal sub-slabs", g.Dl, subs);

  bool prof;
  ProfRec rec;
  {
    std::lock_guard<std::mutex> lk(g_prof_mu);
    prof = g_prof_on;
  }
  if (prof) {
    for (int i = 0; i < 4; ++i) MSN_CUDA_OK(cudaEventCreate(&rec.ev[i]));
    MSN_CUDA_OK(cudaEventRecord(rec.ev[0], s));
  }
  // zero the row padding of the Sobel images (the scan reads up to 31 rows past H)
  for (int i = 0; i < 2; ++i)
    MSN_CUDA_OK(cudaMemsetAsync(ws.sob[i], 0, (size_t)N * (H + kSadRowPad) * g.Ws * sizeof(float), s));
  dim3 pgrid(div_up(g.Wp, 128), g.Hp, 2 * N);
  ms_prep_kernel<<<pgrid, 128, 0, s>>>(d_left, d_right, g, ws.desc[0], ws.desc[1], ws.stat[0], ws.stat[1],
                                       ws.fimg[0], ws.fimg[1], ws.sob[0], ws.sob[1], ws.meanR, ws.AR, ws.CR,
                                       ws.meanL, ws.AL, ws.CL, ws.luts, aml_scale(p->cens_sigma));
  MSN_LAUNCH_OK();
  if (prof) MSN_CUDA_OK(cudaEventRecord(rec.ev[1], s));
  g.d_inner = subs > 1 ? 1 : 0;   // several sub-slabs in flight: keep a tile's scratch rows on one page
  if (launch_sadsob5_padded(ws.sob[0], ws.sob[1], N, H, W, g.Dl, g.d0, ws.sadsob + g.sxo, ws.sad_ws, s, g.d_inner != 0,
                            g.y0 + g.bh, g.y0 + g.bh + g.h, xchg == nullptr))
    return 1;
  if (prof) MSN_CUDA_OK(cudaEventRecord(rec.ev[2], s));

  g.D = g.Dl / subs;   // what one CTA handles (the scan above covered the launch's whole slab)
  FusedArgs a;
  a.g = g;
  a.descL = ws.desc[0]; a.descR = ws.desc[1];
  a.statL = ws.stat[0]; a.statR = ws.stat[1];
  a.fL = ws.fimg[0]; a.fR = ws.fimg[1];
  a.meanR = ws.meanR; a.AR = ws.AR; a.CR = ws.CR;
  a.meanL = ws.meanL; a.AL = ws.AL; a.CL = ws.CL;
  // both views in one call (p->lr, no minima buffer): this launch writes channels 0-7 and leaves the raw costs of
  // cropped voxel (0,0,0) for the right-view launch below, which writes channels 8-15
  const bool both_views = p->lr && !d_mins;
  MSN_REQUIRE(!both_views || (!exact && !xchg && !out_bf16 && g.d0 == 0 && !(wta && wta->idx)),
              "ms_features: both views come from the one-pass kernels in the fast AML mode only (no slab, bf16 or WTA form)");
  a.first4 = nullptr;
  a.first4_out = both_views ? ws.first4 : nullptr;
  a.out_ch0 = 0;
  a.luts = ws.luts;
  a.sadsob = ws.sadsob;
  a.out = d_out;
  a.mins = d_mins;
  a.out_channels = p->lr ? 16 : 8;
  a.mins_planes = p->lr ? 8 : 4;
  a.out_D = out_D > 0 ? out_D : g.D;
  a.out_d0 = out_d0;
  a.mins_accumulate = accumulate;
  a.k_cen = aml_scale(p->cens_sigma);
  a.k_ncc = aml_scale(p->ncc_sigma);
  a.k_sad = aml_scale(p->sad_sigma);
  a.tiles_x = (g.w + kTile - 1) / kTile;
  a.wta_idx = nullptr; a.wta_min1 = a.wta_min2 = nullptr;
  if (wta && wta->idx) {
    MSN_REQUIRE(!d_mins && wta->min1 && wta->min2, "ms_features: the WTA by-product needs all three planes and the one-pass path");
    a.wta_idx = wta->idx; a.wta_min1 = wta->min1; a.wta_min2 = wta->min2;
  }
  memset(&a.xchg, 0, sizeof(a.xchg));
  if (xchg) {
    MSN_REQUIRE(!d_mins, "ms_slab_fused: the exchange path takes no minima buffer");
    MSN_REQUIRE(xchg->world >= 1 && xchg->world <= kMaxRanks && xchg->rank >= 0 && xchg->rank < xchg->world,
                "ms_slab_fused: rank %d / world %d out of range (at most %d ranks)", xchg->rank, xchg->world, kMaxRanks);
    MSN_REQUIRE(xchg->epoch != 0, "ms_slab_fused: epoch must be > 0");
    for (int r = 0; r < xchg->world; ++r) {
      MSN_REQUIRE(xchg->tables[r] != nullptr, "ms_slab_fused: exchange table of rank %d is null", r);
      a.xchg.peer[r] = reinterpret_cast<unsigned*>(xchg->tables[r]);
    }
    a.xchg.G = xchg->world; a.xchg.rank = xchg->rank; a.xchg.epoch = xchg->epoch;
    a.xchg.V = xchg->world * subs; a.xchg.v = xchg->rank * subs;
  }
  a.subs = subs;
  const long long tiles = (long long)N * g.h * a.tiles_x;
  a.n_tiles = tiles;
  MSN_REQUIRE(tiles * subs <= 2147483647LL, "ms_features: too many tiles for one launch");
  CUtensorMap sad_map;
  memset(&sad_map, 0, sizeof(sad_map));
  bool use_tma = g.D <= 256 && !tma_disabled();
  if (use_tma) use_tma = sad_tensor_map(g, H, N, ws.sadsob, &sad_map);
  a.DC = 2 * (((g.D + kGroups - 1) / kGroups + 1) / 2);   // phase 1 walks disparity pairs
#define MSN_FUSED_LAUNCH(DMAX, TMA)                                                \
  {                                                                                \
    if (exact) { if (launch_inst<DMAX, TMA, kModeExact>(a, sad_map, tiles, s)) return 1; } \
    else if (out_bf16) { if (launch_inst<DMAX, TMA, kModeBf16>(a, sad_map, tiles, s)) return 1; } \
    else if (xchg) { if (launch_inst<DMAX, TMA, kModeXchg>(a, sad_map, tiles, s)) return 1; } \
    else if (d_mins) { if (launch_inst<DMAX, TMA, kModeSlabA>(a, sad_map, tiles, s)) return 1; } \
    else { if (launch_inst<DMAX, TMA, kModeFull>(a, sad_map, tiles, s)) return 1; }    \
  }
#define MSN_FUSED_CASE(DMAX)                                                       \
  if (g.D <= DMAX) {                                                               \
    if (use_tma && DMAX <= 256) MSN_FUSED_LAUNCH(DMAX <= 256 ? DMAX : 256, true)   \
    else MSN_FUSED_LAUNCH(DMAX, false)                                             \
  } else
  MSN_FUSED_CASE(64)
  MSN_FUSED_CASE(128)
  MSN_FUSED_CASE(192)
  MSN_FUSED_CASE(256)
  MSN_FUSED_CASE(384)
  MSN_FUSED_CASE(448) { return fail("ms_features: D=%d exceeds the fused kernel's limit", g.D); }
#undef MSN_FUSED_CASE
#undef MSN_FUSED_LAUNCH
  MSN_LAUNCH_OK();
  if (both_views) {
    a.first4 = ws.first4;
    a.first4_out = nullptr;
    a.out_ch0 = 8;
#define MSN_RIGHT_CASE(DMAX) \
  if (g.D <= DMAX) { if (launch_inst<DMAX, true, kModeRight>(a, sad_map, tiles, s)) return 1; } else
    MSN_RIGHT_CASE(64)
    MSN_RIGHT_CASE(128)
    MSN_RIGHT_CASE(192)
    MSN_RIGHT_CASE(256)
    MSN_RIGHT_CASE(384)
    MSN_RIGHT_CASE(448) { return fail("ms_features: D=%d exceeds the fused kernel's limit", g.D); }
#undef MSN_RIGHT_CASE
    MSN_LAUNCH_OK();
  }
  if (prof) {
    MSN_CUDA_OK(cudaEventRecord(rec.ev[3], s));
    std::lock_guard<std::mutex> lk(g_prof_mu);
    if (g_prof.size() >= kProfMaxPending) {   // nobody reads: recycle the oldest record instead of growing
      for (int i = 0; i < 4; ++i) cudaEventDestroy(g_prof.front().ev[i]);
      g_prof.erase(g_prof.begin());
    }
    g_prof.push_back(rec);
  }
  return 0;
}

}  // namespace msn
