// sadsob.cu -- SAD over Sobel images through an fp32 summed-area table whose
// ROUNDING IS PART OF THE RESULT (matchers.cpp:356-438).
//
// The reference builds, for every disparity, S = horizontal-prefix(vertical-
// prefix(|L(i,j) - R(i,j-d)|)) with sequential fp32 adds and evaluates the box as
// ((br - bl) - tr) + tl.  On a 560x980 pair the running sums pass 2^24, so S is
// NOT the exact integer sum (SURVEY.md section 7): a bit-exact result needs the same
// add order.  Both prefix passes are therefore replayed as sequential chains --
// there are D*(W+1) independent vertical chains and D*(H+1) independent
// horizontal chains, plenty of parallelism -- organised so that every global
// access is coalesced:
//
//   1. vband kernel: one thread per (d, column) walks down the image and records
//      the vertical prefix at the first row of every 32-row band  -> Vb[d][band][j].
//   2. scan kernel: one warp per (d, band) sweeps left to right in 32x32 tiles.
//      Lanes first own COLUMNS (finish the vertical prefix inside the band from
//      Vb, coalesced image reads), the tile is transposed through shared memory,
//      lanes then own ROWS (continue the horizontal chain, carry in a register),
//      and finally own columns again to evaluate the boxes and store one
//      coalesced 128-byte row segment per output row.
//
// A band holds 32 table rows, i.e. 32 - wsize output rows (the box needs rows i
// and i + wsize), so bands overlap by wsize rows.
#include <stdlib.h>

#include "common.cuh"

namespace msn {

constexpr int kSadTile = 32;
constexpr int kSadMaxW = 16;                       // wsize <= 16
constexpr int kSadVStride = kSadTile + 1;          // tV[32][33]
constexpr int kSadSStride = kSadTile + kSadMaxW + 1;  // tS[32][49]: halo(wsize) + 32 columns
constexpr int kSadWarps = 4;

__device__ __forceinline__ float absdiff_rn(float a, float b) { return fabsf(__fsub_rn(a, b)); }

// Band-prefix pre-pass.  grid: (ceil(W/128), Dn, N); thread i owns table column j = i + 1, i.e.
// image column i: the warp's loads of L start on a 128-byte line.  Table column 0 is identically
// zero; thread 0 writes it as well.  The thread walks down the image band by band (RB rows each),
// records the vertical prefix at the first row of every band and keeps adding: pointers advance
// by the pitch, nine rows of loads are in flight (27 = 3 x 9 rows per band for the default window:
// no remainder loop; measured 3 % faster than 4 or 8 rows), the adds stay strictly sequential.
// pitch: row pitch of L/R in floats (>= W).  Only rows below (NB-1)*RB < H - wsize are read.
// SP > 0: the pitch is a compile-time constant (the fused path's padded Sobel images), so the nine row offsets of
// a step are immediates instead of two ALU-pipe instructions per load (the generic form spent 41 % of its
// instructions on them).
template <int SP>
__global__ void __launch_bounds__(128)
sadsob_vband_kernel(const float* __restrict__ L, const float* __restrict__ R, int /*H*/, int W, int pitch_rt,
                    int d_begin, int RB, int NB, size_t img_stride, float* __restrict__ Vb) {
  const int pitch = SP > 0 ? SP : pitch_rt;
  const int IW = W + 1;
  const int j = blockIdx.x * blockDim.x + threadIdx.x + 1;
  const int dd = blockIdx.y, d = d_begin + dd, n = blockIdx.z;
  if (j >= IW) return;
  float* vb = Vb + (((size_t)n * gridDim.y + dd) * NB) * IW + j;
  if (j == 1)
    for (int b = 0; b < NB; ++b) vb[(size_t)b * IW - 1] = 0.f;
  const int jc = j - 1;
  if (jc < d) {   // the column lies left of the disparity: every prefix is zero
    for (int b = 0; b < NB; ++b) vb[(size_t)b * IW] = 0.f;
    return;
  }
  const float* l = L + n * img_stride + jc;
  const float* r = R + n * img_stride + (jc - d);
  float v = 0.f;
  for (int b = 0; b < NB; ++b, vb += IW) {
    *vb = v;
    if (b == NB - 1) break;             // nothing reads the prefix below the last band's first row
    int q0 = 0;
    for (; q0 + 9 <= RB; q0 += 9, l += 9 * (size_t)pitch, r += 9 * (size_t)pitch) {
      float av[9];
#pragma unroll
      for (int q = 0; q < 9; ++q)
        av[q] = absdiff_rn(__ldg(l + q * (size_t)pitch), __ldg(r + q * (size_t)pitch));
#pragma unroll
      for (int q = 0; q < 9; ++q) v = __fadd_rn(v, av[q]);
    }
    for (; q0 < RB; ++q0, l += pitch, r += pitch)
      v = __fadd_rn(v, absdiff_rn(__ldg(l), __ldg(r)));
  }
}

// The same pre-pass for the fused path (compile-time pitch, zero-padded Sobel images), FOUR disparities per thread:
// the column's L value is loaded once for the four, so a row costs 5 loads instead of 8 (the kernel is bound by
// L1/L2 load throughput: every Sobel row is read once per disparity).  grid: (ceil(W/128), ceil(Dn/4), N).
template <int SP>
__global__ void __launch_bounds__(128)
sadsob_vbandg_kernel(const float* __restrict__ L, const float* __restrict__ R, int W, int d_begin, int Dn, int RB,
                     int NB, size_t img_stride, float* __restrict__ Vb) {
  const int IW = W + 1;
  const int j = blockIdx.x * blockDim.x + threadIdx.x + 1;
  const int dd0 = blockIdx.y * 4, n = blockIdx.z;
  if (j >= IW) return;
  const int jc = j - 1;
  const int nk = min(4, Dn - dd0);
  float* vb = Vb + (((size_t)n * Dn + dd0) * NB) * IW + j;       // disparity dd0 + k: + k * NB * IW
  const size_t kstride = (size_t)NB * IW;
  if (j == 1)
    for (int k = 0; k < nk; ++k)
      for (int b = 0; b < NB; ++b) vb[k * kstride + (size_t)b * IW - 1] = 0.f;
  bool val[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) val[k] = k < nk && jc >= d_begin + dd0 + k;   // else: left of the disparity, all zero
  if (!val[0]) {
    for (int k = 0; k < nk; ++k)
      for (int b = 0; b < NB; ++b) vb[k * kstride + (size_t)b * IW] = 0.f;
    return;
  }
  const float* l = L + n * img_stride + jc;
  const float* r = R + n * img_stride + (jc - d_begin - dd0);   // disparity dd0 + k reads r[-k] (r[0] where it has no column)
  int roff[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) roff[k] = val[k] ? -k : 0;
  float v[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) v[k] = 0.f;
  for (int b = 0; b < NB; ++b, vb += IW) {
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k < nk) vb[k * kstride] = v[k];
    if (b == NB - 1) break;
    int q0 = 0;
    for (; q0 + 3 <= RB; q0 += 3, l += 3 * SP, r += 3 * SP) {
      float lv[3], rv[3][4];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        lv[q] = __ldg(l + q * SP);
#pragma unroll
        for (int k = 0; k < 4; ++k) rv[q][k] = __ldg(r + q * SP + roff[k]);
      }
#pragma unroll
      for (int q = 0; q < 3; ++q)
#pragma unroll
        for (int k = 0; k < 4; ++k) v[k] = __fadd_rn(v[k], val[k] ? absdiff_rn(lv[q], rv[q][k]) : 0.f);
    }
    for (; q0 < RB; ++q0, l += SP, r += SP) {
      const float lq = __ldg(l);
#pragma unroll
      for (int k = 0; k < 4; ++k) v[k] = __fadd_rn(v[k], val[k] ? absdiff_rn(lq, __ldg(r + roff[k])) : 0.f);
    }
  }
}

// grid: (ceil(Dn*NB / kSadWarps), 1, N); one warp per (dd, band).
// WS > 0: window size known at compile time (shared strides and box offsets become
// immediates); WS == 0: runtime wsize (any 1..16).
template <int WS>
__global__ void __launch_bounds__(kSadWarps * 32)
sadsob_scan_kernel(const float* __restrict__ L, const float* __restrict__ R, int H, int W, int Dn,
                   int d_begin, int wsize_rt, int NB, size_t img_stride,
                   const float* __restrict__ Vb, float* __restrict__ out, size_t out_stride, int out_pitch) {
  constexpr int SS = (WS > 0) ? (kSadTile + WS + ((WS & 1) ? 0 : 1)) : kSadSStride;  // odd stride
  __shared__ float sV[kSadWarps][kSadTile * kSadVStride];
  __shared__ float sS[kSadWarps][kSadTile * SS];
  const int wsize = (WS > 0) ? WS : wsize_rt;
  const int RB = kSadTile - wsize;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int job = blockIdx.x * kSadWarps + warp;
  if (job >= Dn * NB) return;  // whole warp exits together
  const int dd = job / NB, b = job % NB, n = blockIdx.z;
  const int d = d_begin + dd;
  const int IW = W + 1, wc = wsize / 2;
  const int i0 = b * RB;
  float* tV = sV[warp];
  float* tS = sS[warp];
  const float* Ln = L + n * img_stride;
  const float* Rn = R + n * img_stride;
  const float* vb = Vb + (((size_t)n * Dn + dd) * NB + b) * IW;
  float* o = out + n * out_stride + (size_t)dd * H * out_pitch;  // rows of out_pitch floats
  const int rows_live = min(kSadTile - 1, H - i0);      // image rows i0 .. i0+rows_live-1 exist
  const int rmax = min(RB, H - wsize - i0);             // origin rows produced by this band

  // table columns <= d are zero, so the sweep starts at the tile holding column d
  const int t0 = d / kSadTile, t1 = (W - 1) / kSadTile;
  float s = 0.f;  // horizontal carry of table row i0 + lane
  float* srow = tS + lane * SS;
#pragma unroll 1
  for (int k = 0; k < wsize; ++k) srow[kSadTile + k] = 0.f;
  for (int t = t0; t <= t1; ++t) {
    // (a) lanes own table columns: finish the vertical prefix inside the band.
    // All loads of the tile column are issued before the dependent add chain starts.
    const int j = t * kSadTile + lane;
    const int jc = j - 1;
    const bool active = (j < IW) && (jc >= d);
    float v = (j < IW) ? __ldg(vb + j) : 0.f;
    float av[kSadTile - 1];
    {
      const float* lp = Ln + (size_t)i0 * W + jc;
      const float* rp = lp + (Rn - Ln) - d;
#pragma unroll
      for (int r = 0; r < kSadTile - 1; ++r) {
        av[r] = (active && r < rows_live) ? absdiff_rn(__ldg(lp), __ldg(rp)) : 0.f;
        lp += W; rp += W;
      }
    }
    tV[lane] = v;
#pragma unroll
    for (int r = 1; r < kSadTile; ++r) {
      v = __fadd_rn(v, av[r - 1]);  // + 0.0f on inactive entries is exact
      tV[r * kSadVStride + lane] = v;
    }
    __syncwarp();
    // (b) lanes own table rows: slide the halo, continue the horizontal chain
#pragma unroll
    for (int k = 0; k < (WS > 0 ? WS : kSadMaxW); ++k)
      if (k < wsize) srow[k] = srow[kSadTile + k];
    {
      const float* vrow = tV + lane * kSadVStride;
      float* dst = srow + wsize;
#pragma unroll
      for (int c = 0; c < kSadTile; ++c) {
        s = __fadd_rn(s, vrow[c]);
        dst[c] = s;
      }
    }
    __syncwarp();
    // (c) lanes own origin columns again: boxes ((br - bl) - tr) + tl
    const int jo = t * kSadTile - wsize + lane;  // window origin column
    if (jo >= d && jo < W - wsize) {
      const float* top = tS + lane;
      const float* bot = top + wsize * SS;
      float* op = o + (size_t)(i0 + wc) * out_pitch + (jo + wc);
#pragma unroll 9
      for (int r = 0; r < rmax; ++r) {
        const float val = __fadd_rn(__fsub_rn(__fsub_rn(bot[wsize], bot[0]), top[wsize]), top[0]);
        st_stream(op, val);
        top += SS; bot += SS; op += out_pitch;
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// Specialised sweep for the reference's default window (sobelw = 5) used by the fused
// path, whose Sobel images carry >= 31 ZERO rows below row H-1 (kSadRowPad), so the 62
// loads of a tile column need no row guards (|0 - 0| adds an exact 0).  One shared tile
// T[32][37] per warp serves in turn the vertical prefixes (written column-wise, read
// row-wise), the horizontal prefixes (in place) and the boxes (read column-wise); the five
// halo columns travel in registers between tiles, and the box stage reads every table
// element once, keeping the five rows a window spans in registers.
constexpr int kS5W = 5;
constexpr int kS5Stride = kSadTile + kS5W;  // 37: odd, conflict-free both ways
constexpr int kS5Warps = 4;

template <bool kMask, int SP>
__device__ __forceinline__ void s5_vertical(const float* __restrict__ lp, const float* __restrict__ rp,
                                            bool active, float v, float* __restrict__ T, int lane) {
  float av[kSadTile - 1];
#pragma unroll
  for (int r = 0; r < kSadTile - 1; ++r) {   // row offsets r*SP are immediates: no address math
    const float x = absdiff_rn(__ldg(lp + r * SP), __ldg(rp + r * SP));
    av[r] = (!kMask || active) ? x : 0.f;
  }
  T[kS5W + lane] = v;
#pragma unroll
  for (int r = 1; r < kSadTile; ++r) {
    v = __fadd_rn(v, av[r - 1]);  // + 0.0f on masked / padded entries is exact
    T[r * kS5Stride + kS5W + lane] = v;
  }
}

// SP: row pitch in floats of BOTH the Sobel images and the output volume (compile-time so
// that every row offset is an immediate); W <= SP.
template <int SP, bool kDInner>
__global__ void __launch_bounds__(kS5Warps * 32, 4)
sadsob_scan5_kernel(const float* __restrict__ L, const float* __restrict__ R, int H, int W, int Dn, int d_begin,
                    int NB, int b_min, size_t img_stride, const float* __restrict__ Vb, float* __restrict__ out,
                    size_t out_stride) {
  // kDInner: the output is [N][H][Dn][SP] -- the Dn rows of one image row lie side by side, so the fused
  // kernel's tile (one row y, all disparities) reads ONE contiguous Dn x 4 KB span instead of Dn rows megabytes
  // apart: a Middlebury-sized volume cut into sub-slabs of one launch (12+ GB of scratch) otherwise falls off
  // the TLB (measured 1.5x slower); jobs are then numbered disparity-fastest, so neighbouring warps write
  // neighbouring rows.  Otherwise [N][Dn][H][SP] with compile-time row offsets (5 % faster at config B).
  __shared__ float sT[kS5Warps][kSadTile * kS5Stride];
  constexpr int RB = kSadTile - kS5W;  // 27 origin rows per band
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int job = blockIdx.x * kS5Warps + warp;
  const int nbs = NB - b_min;     // bands b_min .. NB-1 are scanned (all of them unless the caller wants a row range)
  if (job >= Dn * nbs) return;  // whole warp exits together
  const int dd = kDInner ? job % Dn : job / nbs, b = b_min + (kDInner ? job / Dn : job % nbs), n = blockIdx.z;
  const int d = d_begin + dd;
  const int IW = W + 1;
  const int i0 = b * RB;
  float* T = sT[warp];
  const float* Ln = L + n * img_stride + (size_t)i0 * SP;
  const float* Rn = R + n * img_stride + (size_t)i0 * SP - d;
  const float* vb = Vb + (((size_t)n * Dn + dd) * NB + b) * IW;
  const size_t row_stride = kDInner ? (size_t)Dn * SP : (size_t)SP;
  float* o = kDInner ? out + n * out_stride + ((size_t)(i0 + 2) * Dn + dd) * SP + 2
                     : out + n * out_stride + (size_t)dd * H * SP + (size_t)(i0 + 2) * SP + 2;
  const int rmax = min(RB, H - kS5W - i0);          // origin rows produced by this band

  const int t0 = d / kSadTile, t1 = (W - 1) / kSadTile;
  float s = 0.f;                                  // horizontal carry of table row i0 + lane
  float h0 = 0.f, h1 = 0.f, h2 = 0.f, h3 = 0.f, h4 = 0.f;  // this row's last five S values
  float* trow = T + lane * kS5Stride;
  for (int t = t0; t <= t1; ++t) {
    // (a) lanes own table columns: vertical prefix inside the band (loads first, then chain)
    // tile t holds table columns j = 32t+1 .. 32t+32, i.e. image columns jc = 32t .. 32t+31: the
    // warp's loads of L start on a 128-byte line, and so do its stores of the 27 output rows when
    // the caller's output pointer is offset by 2 columns modulo 32 (the fused path's scratch is)
    const int j = t * kSadTile + lane + 1;
    const int jc = j - 1;
    const float v = (j < IW) ? __ldg(vb + j) : 0.f;
    if (t == t0 || t == t1) {
      const bool active = (j < IW) && (jc >= d);
      const int jsafe = min(max(jc, d), W - 1);      // masked lanes load a valid address
      s5_vertical<true, SP>(Ln + jsafe, Rn + jsafe, active, v, T, lane);
    } else {
      s5_vertical<false, SP>(Ln + jc, Rn + jc, true, v, T, lane);
    }
    __syncwarp();
    // (b) lanes own table rows: halo from registers, horizontal chain in place
    trow[0] = h0; trow[1] = h1; trow[2] = h2; trow[3] = h3; trow[4] = h4;
#pragma unroll
    for (int c = 0; c < kSadTile; ++c) {
      s = __fadd_rn(s, trow[kS5W + c]);
      trow[kS5W + c] = s;
      if (c == kSadTile - 5) h0 = s;
      if (c == kSadTile - 4) h1 = s;
      if (c == kSadTile - 3) h2 = s;
      if (c == kSadTile - 2) h3 = s;
      if (c == kSadTile - 1) h4 = s;
    }
    __syncwarp();
    // (c) lanes own origin columns: out(r) = ((S[r+5][j+5] - S[r+5][j]) - S[r][j+5]) + S[r][j]
    const int jo = t * kSadTile + 1 - kS5W + lane;  // window origin column
    if (jo >= d && jo < W - kS5W) {
      float lo[kS5W], hi[kS5W];  // table rows r .. r+4 at columns jo and jo+5
#pragma unroll
      for (int r = 0; r < kS5W; ++r) {
        lo[r] = T[r * kS5Stride + lane];
        hi[r] = T[r * kS5Stride + lane + kS5W];
      }
      float* op = o + jo;
#pragma unroll
      for (int r = 0; r < RB; ++r) {
        const float bl = T[(r + kS5W) * kS5Stride + lane];
        const float br = T[(r + kS5W) * kS5Stride + lane + kS5W];
        const float val = __fadd_rn(__fsub_rn(__fsub_rn(br, bl), hi[r % kS5W]), lo[r % kS5W]);
        if (r < rmax) st_stream(kDInner ? op + r * row_stride : op + r * SP, val);
        lo[r % kS5W] = bl;
        hi[r % kS5W] = br;
      }
    }
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------
// The same sweep over bands of 64 table rows = 59 origin rows: neighbouring bands still share five table rows, but
// that is 8 % of a band instead of 16 %, and a lane owns TWO rows in the horizontal step (two independent chains).
// By wavefront count (the kernel is bound by the L1 data pipe) a tile of 59 x 32 costs 127 global-load, 59
// global-store and 330 shared wavefronts = 8.75 per output row against 9.44.  A band whose second half holds no
// origin row (the last band of an image, a row range) is processed as a 32-row band.
constexpr int kS5Rows2 = 2 * kSadTile;          // 64 table rows
constexpr int kS5RB2 = kS5Rows2 - kS5W;          // 59 origin rows per band

template <int SP, bool kDInner>
__global__ void __launch_bounds__(kS5Warps * 32, 4)
sadsob_scan5x2_kernel(const float* __restrict__ L, const float* __restrict__ R, int H, int W, int Dn, int d_begin,
                      int NB, int b_min, size_t img_stride, const float* __restrict__ Vb, float* __restrict__ out,
                      size_t out_stride) {
  __shared__ float sT[kS5Warps][kS5Rows2 * kS5Stride];
  constexpr int RB = kS5RB2;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int job = blockIdx.x * kS5Warps + warp;
  const int nbs = NB - b_min;
  if (job >= Dn * nbs) return;
  const int dd = kDInner ? job % Dn : job / nbs, b = b_min + (kDInner ? job / Dn : job % nbs), n = blockIdx.z;
  const int d = d_begin + dd;
  const int IW = W + 1;
  const int i0 = b * RB;
  float* T = sT[warp];
  const float* Ln = L + n * img_stride + (size_t)i0 * SP;
  const float* Rn = R + n * img_stride + (size_t)i0 * SP - d;
  const float* vb = Vb + (((size_t)n * Dn + dd) * NB + b) * IW;
  const size_t row_stride = kDInner ? (size_t)Dn * SP : (size_t)SP;
  float* o = kDInner ? out + n * out_stride + ((size_t)(i0 + 2) * Dn + dd) * SP + 2
                     : out + n * out_stride + (size_t)dd * H * SP + (size_t)(i0 + 2) * SP + 2;
  const int rmax = min(RB, H - kS5W - i0);          // origin rows produced by this band
  const bool two = rmax > kSadTile - kS5W;          // the second half holds origin rows (else: a 32-row band)

  const int t0 = d / kSadTile, t1 = (W - 1) / kSadTile;
  float s0 = 0.f, s1 = 0.f;                         // horizontal carries of table rows i0 + lane, i0 + 32 + lane
  float h0[kS5W] = {0.f, 0.f, 0.f, 0.f, 0.f}, h1[kS5W] = {0.f, 0.f, 0.f, 0.f, 0.f};   // their last five S values
  float* trow0 = T + lane * kS5Stride;
  float* trow1 = trow0 + kSadTile * kS5Stride;
  for (int t = t0; t <= t1; ++t) {
    // (a) lanes own table columns: vertical prefix, 31 (+ 32) image rows, loads first, then the chain
    const int j = t * kSadTile + lane + 1;
    const int jc = j - 1;
    float v = (j < IW) ? __ldg(vb + j) : 0.f;
    const bool edge = (t == t0 || t == t1);
    const bool active = (j < IW) && (jc >= d);
    const int jsafe = edge ? min(max(jc, d), W - 1) : jc;      // masked lanes load a valid address
    const float* lp = Ln + jsafe;
    const float* rp = Rn + jsafe;
    {
      float av[kSadTile - 1];
#pragma unroll
      for (int r = 0; r < kSadTile - 1; ++r) {
        const float x = absdiff_rn(__ldg(lp + r * SP), __ldg(rp + r * SP));
        av[r] = (!edge || active) ? x : 0.f;
      }
      T[kS5W + lane] = v;
#pragma unroll
      for (int r = 1; r < kSadTile; ++r) {
        v = __fadd_rn(v, av[r - 1]);
        T[r * kS5Stride + kS5W + lane] = v;
      }
    }
    if (two) {
      float av[kSadTile];
#pragma unroll
      for (int r = 0; r < kSadTile; ++r) {
        const float x = absdiff_rn(__ldg(lp + (kSadTile - 1 + r) * SP), __ldg(rp + (kSadTile - 1 + r) * SP));
        av[r] = (!edge || active) ? x : 0.f;
      }
#pragma unroll
      for (int r = 0; r < kSadTile; ++r) {
        v = __fadd_rn(v, av[r]);
        T[(kSadTile + r) * kS5Stride + kS5W + lane] = v;
      }
    }
    __syncwarp();
    // (b) lanes own table rows lane and 32 + lane: halo from registers, two horizontal chains in place
#pragma unroll
    for (int k = 0; k < kS5W; ++k) trow0[k] = h0[k];
    if (two) {
#pragma unroll
      for (int k = 0; k < kS5W; ++k) trow1[k] = h1[k];
#pragma unroll
      for (int c = 0; c < kSadTile; ++c) {
        s0 = __fadd_rn(s0, trow0[kS5W + c]);
        s1 = __fadd_rn(s1, trow1[kS5W + c]);
        trow0[kS5W + c] = s0;
        trow1[kS5W + c] = s1;
        if (c >= kSadTile - kS5W) { h0[c - (kSadTile - kS5W)] = s0; h1[c - (kSadTile - kS5W)] = s1; }
      }
    } else {
#pragma unroll
      for (int c = 0; c < kSadTile; ++c) {
        s0 = __fadd_rn(s0, trow0[kS5W + c]);
        trow0[kS5W + c] = s0;
        if (c >= kSadTile - kS5W) h0[c - (kSadTile - kS5W)] = s0;
      }
    }
    __syncwarp();
    // (c) lanes own origin columns: out(r) = ((S[r+5][j+5] - S[r+5][j]) - S[r][j+5]) + S[r][j]
    const int jo = t * kSadTile + 1 - kS5W + lane;
    if (jo >= d && jo < W - kS5W) {
      float lo[kS5W], hi[kS5W];
#pragma unroll
      for (int r = 0; r < kS5W; ++r) {
        lo[r] = T[r * kS5Stride + lane];
        hi[r] = T[r * kS5Stride + lane + kS5W];
      }
      float* op = o + jo;
#pragma unroll
      for (int r = 0; r < kSadTile - kS5W; ++r) {
        const float bl = T[(r + kS5W) * kS5Stride + lane];
        const float br = T[(r + kS5W) * kS5Stride + lane + kS5W];
        const float val = __fadd_rn(__fsub_rn(__fsub_rn(br, bl), hi[r % kS5W]), lo[r % kS5W]);
        if (r < rmax) st_stream(kDInner ? op + r * row_stride : op + r * SP, val);
        lo[r % kS5W] = bl;
        hi[r % kS5W] = br;
      }
      if (two) {
#pragma unroll
        for (int r = kSadTile - kS5W; r < RB; ++r) {
          const float bl = T[(r + kS5W) * kS5Stride + lane];
          const float br = T[(r + kS5W) * kS5Stride + lane + kS5W];
          const float val = __fadd_rn(__fsub_rn(__fsub_rn(br, bl), hi[r % kS5W]), lo[r % kS5W]);
          if (r < rmax) st_stream(kDInner ? op + r * row_stride : op + r * SP, val);
          lo[r % kS5W] = bl;
          hi[r % kS5W] = br;
        }
      }
    }
    __syncwarp();
  }
}

static inline void sadsob_geom(int H, int wsize, int* RB, int* NB) {
  *RB = kSadTile - wsize;
  const int rows = H - wsize;  // origin rows i in [0, H - wsize)
  *NB = rows > 0 ? (rows + *RB - 1) / *RB : 0;
}

size_t sadsob_workspace_bytes_n(int N, int H, int W, int Dn, int wsize) {
  int RB, NB;
  sadsob_geom(H, wsize, &RB, &NB);
  return (size_t)N * Dn * (NB > 0 ? NB : 1) * (W + 1) * sizeof(float);
}
size_t sadsob_workspace_bytes(int H, int W, int D, int wsize) {
  return sadsob_workspace_bytes_n(1, H, W, D, wsize);
}

// N pairs; L/R are float [N][H][W]; out is [N][Dn][H][out_pitch] (out_pitch >= W; the caller may
// pre-offset `out` by a few columns) with stride out_stride floats per pair.
// Generic form: L/R are [N][H][W] (pitch W); out is [N][Dn][H][out_pitch] (out_pitch >= W) with
// stride out_stride floats per pair.
int launch_sadsob_n(const float* L, const float* R, int N, int H, int W, int Dn, int d_begin, int wsize,
                    float* out, size_t out_stride, int out_pitch, bool write_fill, void* workspace,
                    cudaStream_t s) {
  MSN_REQUIRE(wsize >= 1 && wsize <= kSadMaxW, "sadsob: wsize %d unsupported (1..%d)", wsize, kSadMaxW);
  if (write_fill) {
    for (int n = 0; n < N; ++n)
      if (launch_fill(out + n * out_stride, (size_t)Dn * H * out_pitch, kFill, s)) return 1;
  }
  int RB, NB;
  sadsob_geom(H, wsize, &RB, &NB);
  if (NB <= 0 || W - wsize <= 0 || Dn <= 0) return 0;
  float* Vb = static_cast<float*>(workspace);
  const size_t img_stride = (size_t)H * W;
  dim3 g1(div_up(W, 128), Dn, N);
  sadsob_vband_kernel<0><<<g1, 128, 0, s>>>(L, R, H, W, W, d_begin, RB, NB, img_stride, Vb);
  MSN_LAUNCH_OK();
  dim3 g2(div_up((long long)Dn * NB, kSadWarps), 1, N);
  if (wsize == 5)  // the reference's default sobelw (cbmv_generator.py:440)
    sadsob_scan_kernel<5><<<g2, kSadWarps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, wsize, NB, img_stride, Vb, out,
                                                        out_stride, out_pitch);
  else
    sadsob_scan_kernel<0><<<g2, kSadWarps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, wsize, NB, img_stride, Vb, out,
                                                        out_stride, out_pitch);
  MSN_LAUNCH_OK();
  return 0;
}

// Fast form for the fused path (window 5): L/R are [N][H + kSadRowPad][SP] with ZERO padding
// rows/columns, out is [N][Dn][H][SP] (d_inner: [N][H][Dn][SP]); SP = sadsob_fast_pitch(W) is one of 1024/2048/4096.
int sadsob_fast_pitch(int W) { return W <= 1024 ? 1024 : W <= 2048 ? 2048 : W <= 4096 ? 4096 : 0; }

int launch_sadsob5_padded(const float* L, const float* R, int N, int H, int W, int Dn, int d_begin, float* out,
                          void* workspace, cudaStream_t s, bool d_inner, int row_lo, int row_hi, bool tall_ok) {
  const int SP = sadsob_fast_pitch(W);
  MSN_REQUIRE(SP > 0, "sadsob: W=%d too wide for the padded window-5 scan", W);
  int RB, NB;
  sadsob_geom(H, kS5W, &RB, &NB);
  if (NB <= 0 || W - kS5W <= 0 || Dn <= 0) return 0;
  // bands of 64 table rows (sadsob_scan5x2_kernel) unless MSNETS_SCAN32=1 asks for the 32-row form
  // (tall_ok = false: launches of the slab exchange.  Their tiles WAIT for other ranks; when those ranks are other
  // streams of the same GPU -- the virtual-rank tests -- a waiting kernel's CTAs leave 27 KB of shared memory per SM,
  // which the 32-row form's blocks fit into and the 64-row form's 38 KB do not: the peers' scans would never run.)
  const char* e32 = getenv("MSNETS_SCAN32");
  const bool tall_env = !(e32 && e32[0] == '1');
  // ... and only when the taller (half as many, twice as long) jobs still fill the machine: a single small pair is
  // faster in 32-row bands (config A: 0.358 vs 0.364 ms per step; two config-B pairs: 0.313 vs 0.318 ms)
  // (at two waves of jobs and up; MSNETS_SCAN64=1 forces it for the tests)
  const long long jobs64 = (long long)Dn * ((H - kS5W + kS5RB2 - 1) / kS5RB2) * N;
  const char* force = getenv("MSNETS_SCAN64");
  const bool tall = tall_env && tall_ok && (jobs64 >= 4736 || (force && force[0] == '1'));
  if (tall) {
    RB = kS5RB2;
    NB = (H - kS5W + RB - 1) / RB;
  }
  // band b holds output rows [b*RB + 2, b*RB + 2 + RB): the bands a row range needs
  int b_min = 0;
  if (row_hi >= 0) {
    b_min = (row_lo - 2 < 0 ? 0 : row_lo - 2) / RB;
    const int b_max = (row_hi - 1 - 2 < 0 ? 0 : row_hi - 1 - 2) / RB;
    if (b_min >= NB) return 0;
    NB = (b_max + 1 < NB) ? b_max + 1 : NB;      // prefixes below the last needed band are never read
  }
  float* Vb = static_cast<float*>(workspace);
  const size_t img_stride = (size_t)(H + kSadRowPad) * SP;
  const size_t out_stride = (size_t)Dn * H * SP;
  dim3 g1(div_up(W, 128), Dn, N);
  (void)g1;
  dim3 g4(div_up(W, 128), div_up(Dn, 4), N);
  if (SP == 1024) sadsob_vbandg_kernel<1024><<<g4, 128, 0, s>>>(L, R, W, d_begin, Dn, RB, NB, img_stride, Vb);
  else if (SP == 2048) sadsob_vbandg_kernel<2048><<<g4, 128, 0, s>>>(L, R, W, d_begin, Dn, RB, NB, img_stride, Vb);
  else sadsob_vbandg_kernel<4096><<<g4, 128, 0, s>>>(L, R, W, d_begin, Dn, RB, NB, img_stride, Vb);
  MSN_LAUNCH_OK();
  const int nbs = NB - b_min;
  dim3 g5(div_up((long long)Dn * nbs, kS5Warps), 1, N);
#define MSN_SCAN5(P)                                                                                             \
  {                                                                                                              \
    if (tall) {                                                                                                  \
      if (d_inner) sadsob_scan5x2_kernel<P, true><<<g5, kS5Warps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, NB, b_min, img_stride, Vb, out, out_stride); \
      else sadsob_scan5x2_kernel<P, false><<<g5, kS5Warps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, NB, b_min, img_stride, Vb, out, out_stride);        \
    } else if (d_inner) sadsob_scan5_kernel<P, true><<<g5, kS5Warps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, NB, b_min, img_stride, Vb, out, out_stride); \
    else sadsob_scan5_kernel<P, false><<<g5, kS5Warps * 32, 0, s>>>(L, R, H, W, Dn, d_begin, NB, b_min, img_stride, Vb, out, out_stride);        \
  }
  if (SP == 1024) MSN_SCAN5(1024)
  else if (SP == 2048) MSN_SCAN5(2048)
  else MSN_SCAN5(4096)
#undef MSN_SCAN5
  MSN_LAUNCH_OK();
  return 0;
}

int launch_sadsob(const float* L, const float* R, int H, int W, int D, int d_begin, int wsize, float* out,
                  bool write_fill, void* workspace, cudaStream_t s) {
  return launch_sadsob_n(L, R, 1, H, W, D, d_begin, wsize, out, (size_t)D * H * W, W, write_fill, workspace, s);
}

}  // namespace msn
