// regress.cu -- soft-argmin disparity regression and the 4D volume builders.
//
// soft-argmin replaces F.softmax(out,1) + disparityregression
// (gcnet_3dcnn.py:127-141): the reference makes >= 4 passes over the [N,D,H,W]
// volume and materialises arange(D).repeat(N,1,H,W); here one thread streams the D
// column of 1 or 4 neighbouring pixels once, with an online-softmax (running max,
// rescaled sums) so the volume is read exactly once: 4 B/voxel in, 4 B/pixel out.
// HBM-bound; 8 independent 128-bit loads are kept in flight per thread.
#include "common.cuh"
#include "feature_math.cuh"

namespace msn {

constexpr float kLog2e = 1.4426950408889634f;
constexpr int kSaChunk = 8;

template <int V>
struct Vec;
template <>
struct Vec<1> {
  using T = float;
  __device__ static void get(const T& v, float* f) { f[0] = v; }
};
template <>
struct Vec<4> {
  using T = float4;
  __device__ static void get(const T& v, float* f) { f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w; }
};

// MODE 0: write disp; MODE 1: write partial (max, sum e, sum d*e) planes [N][3][HW];
// MODE 2: input already holds probabilities -> plain expectation sum_d d*p_d
// (the body of the reference's disparityregression, gcnet_3dcnn.py:136-139).
// The float4 form is held to 3 CTAs (24 warps) per SM, the occupancy its loads in flight were measured at: left
// alone, ptxas gives it 87 registers, which fits only 2.  The scalar form fits 6 CTAs in 40 registers.
template <int V, int MODE>
__global__ void __launch_bounds__(256, V == 4 ? 3 : 6)
soft_argmin_kernel(const float* __restrict__ logits, int N, int D, long long HW, int d_begin,
                   float* __restrict__ out) {
  using VT = typename Vec<V>::T;
  const long long groups = HW / V;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (g >= groups) return;
  const VT* src = reinterpret_cast<const VT*>(logits + (size_t)n * D * HW) + g;
  float m[V], s[V], t[V];
#pragma unroll
  for (int i = 0; i < V; ++i) { m[i] = -INFINITY; s[i] = 0.f; t[i] = 0.f; }
  for (int d0 = 0; d0 < D; d0 += kSaChunk) {
    VT raw[kSaChunk];
#pragma unroll
    for (int j = 0; j < kSaChunk; ++j)
      if (d0 + j < D) raw[j] = __ldcs(src + (size_t)(d0 + j) * groups);
    float x[kSaChunk][V];
#pragma unroll
    for (int j = 0; j < kSaChunk; ++j) Vec<V>::get(raw[j], x[j]);
    if (MODE == 2) {
#pragma unroll
      for (int i = 0; i < V; ++i)
#pragma unroll
        for (int j = 0; j < kSaChunk; ++j)
          if (d0 + j < D) t[i] = fmaf(x[j][i], (float)(d_begin + d0 + j), t[i]);
      continue;
    }
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float cm = m[i];
#pragma unroll
      for (int j = 0; j < kSaChunk; ++j)
        if (d0 + j < D) cm = fmaxf(cm, x[j][i]);
      // While every logit so far is -inf (masked), subtract 0 so that (m, s, t) stays (-inf, 0, 0)
      // instead of turning into 2^(-inf - -inf) = NaN.
      const float cs = (cm == -INFINITY) ? 0.f : cm;
      const float sc = ex2_approx((m[i] - cs) * kLog2e);  // first chunk: 2^-inf = 0
      float ss = s[i] * sc, tt = t[i] * sc;
#pragma unroll
      for (int j = 0; j < kSaChunk; ++j)
        if (d0 + j < D) {
          // x - max first: exact near the maximum (Sterbenz), so the weights do not depend on |max|.  Folding the
          // shift into fma(x, log2e, -fl(max * log2e)) adds the rounding of that product, which grows with |max|
          // and differs from chunk to chunk.
          const float e = ex2_approx((x[j][i] - cs) * kLog2e);
          ss += e;
          tt = fmaf(e, (float)(d_begin + d0 + j), tt);
        }
      m[i] = cm; s[i] = ss; t[i] = tt;
    }
  }
  if (MODE == 0 || MODE == 2) {
    float* o = out + (size_t)n * HW + g * V;
#pragma unroll
    for (int i = 0; i < V; ++i) o[i] = (MODE == 2) ? t[i] : t[i] / s[i];
  } else {
    float* o = out + (size_t)n * 3 * HW + g * V;
#pragma unroll
    for (int i = 0; i < V; ++i) { o[i] = m[i]; o[HW + i] = s[i]; o[2 * HW + i] = t[i]; }
  }
}

// mode: 0 soft-argmin, 1 slab partials, 2 expectation of given probabilities
int launch_soft_argmin(const float* logits, int N, int D, int H, int W, int d_begin, int mode,
                       float* out, cudaStream_t s) {
  MSN_REQUIRE(N >= 0 && D >= 1 && H >= 0 && W >= 0, "soft_argmin: bad shape N=%d D=%d H=%d W=%d", N, D, H, W);
  const long long HW = (long long)H * W;
  if (N == 0 || HW == 0) return 0;
  MSN_REQUIRE(N <= 65535, "soft_argmin: N=%d too large", N);
  const bool vec = (HW % 4 == 0) && ((reinterpret_cast<uintptr_t>(logits) & 15) == 0);
  if (vec) {
    dim3 grid(div_up(HW / 4, 256), N);
    if (mode == 1) soft_argmin_kernel<4, 1><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
    else if (mode == 2) soft_argmin_kernel<4, 2><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
    else soft_argmin_kernel<4, 0><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
  } else {
    dim3 grid(div_up(HW, 256), N);
    if (mode == 1) soft_argmin_kernel<1, 1><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
    else if (mode == 2) soft_argmin_kernel<1, 2><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
    else soft_argmin_kernel<1, 0><<<grid, 256, 0, s>>>(logits, N, D, HW, d_begin, out);
  }
  MSN_LAUNCH_OK();
  return 0;
}

// Backward of soft-argmin for training (the reference trains through F.softmax + disparityregression,
// gcnet_3dcnn.py:127-141; psmnet_3dcnn.py:149-176):  d disp / d x_d = p_d * (d - disp), so
// grad_x[n][d][p] = grad_out[n][p] * p_d * (d - disp[n][p]).  Two sweeps over the column: (max, sum)
// online, then the gradient; thread = pixel, coalesced along W.
__global__ void __launch_bounds__(256)
soft_argmin_bwd_kernel(const float* __restrict__ logits, const float* __restrict__ disp,
                       const float* __restrict__ gout, int D, long long HW, float* __restrict__ gin) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int n = blockIdx.y;
  if (p >= HW) return;
  const float* x = logits + (size_t)n * D * HW + p;
  float m = -INFINITY, s = 0.f;
  for (int d = 0; d < D; ++d) {
    const float v = x[(size_t)d * HW];
    const float cm = fmaxf(m, v);
    const float cs = (cm == -INFINITY) ? 0.f : cm;  // leading -inf logits: s stays 0, not NaN
    s = s * ex2_approx((m - cs) * kLog2e) + ex2_approx((v - cs) * kLog2e);
    m = cm;
  }
  const float go = gout[(size_t)n * HW + p] / s, dv = disp[(size_t)n * HW + p];
  float* g = gin + (size_t)n * D * HW + p;
  for (int d = 0; d < D; ++d) {
    const float e = ex2_approx((x[(size_t)d * HW] - m) * kLog2e);
    g[(size_t)d * HW] = go * e * ((float)d - dv);
  }
}

int launch_soft_argmin_bwd(const float* logits, const float* disp, const float* gout, int N, int D, int H, int W,
                           float* gin, cudaStream_t s) {
  MSN_REQUIRE(N >= 0 && D >= 1 && H >= 0 && W >= 0, "soft_argmin_backward: bad shape");
  const long long HW = (long long)H * W;
  if (N == 0 || HW == 0) return 0;
  MSN_REQUIRE(N <= 65535, "soft_argmin_backward: N=%d too large", N);
  dim3 grid(div_up(HW, 256), N);
  soft_argmin_bwd_kernel<<<grid, 256, 0, s>>>(logits, disp, gout, D, HW, gin);
  MSN_LAUNCH_OK();
  return 0;
}

// parts: [P][N][3][HW] gathered slab partials -> disp [N][HW]
__global__ void soft_argmin_merge_kernel(const float* __restrict__ parts, int P, long long NHW3, long long HW,
                                         long long total, float* __restrict__ disp) {
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= total) return;
  const long long n = q / HW, p = q % HW;
  const float* base = parts + n * 3 * HW + p;
  float M = -INFINITY;
  for (int r = 0; r < P; ++r) M = fmaxf(M, base[(size_t)r * NHW3]);
  float S = 0.f, T = 0.f;
  for (int r = 0; r < P; ++r) {
    const float* b = base + (size_t)r * NHW3;
    const float sc = ex2_approx((b[0] - M) * kLog2e);
    S = fmaf(b[HW], sc, S);
    T = fmaf(b[2 * HW], sc, T);
  }
  disp[q] = T / S;
}

int launch_soft_argmin_merge(const float* parts, int P, int N, int H, int W, float* disp, cudaStream_t s) {
  const long long HW = (long long)H * W, total = HW * N;
  if (total == 0) return 0;
  MSN_REQUIRE(P >= 1, "soft_argmin_merge: parts must be >= 1");
  soft_argmin_merge_kernel<<<div_up(total, 256), 256, 0, s>>>(parts, P, 3 * total, HW, total, disp);
  MSN_LAUNCH_OK();
  return 0;
}

// ------------------------------------------------------------ 4D volumes --
// concat: vol[n][c][d][y][x]   = x >= d ? fl[n][c][y][x]   : 0      (c <  C)
//         vol[n][C+c][d][y][x] = x >= d ? fr[n][c][y][x-d] : 0
// diff  : vol[n][c][d][y][x]   = x >= d ? fl[n][c][y][x] - fr[n][c][y][x-d] : 0
// Pure data movement, D-fold write amplification: HBM-write bound.  One thread owns 4
// consecutive x of one input channel row and walks ALL disparities: the left quad stays in
// registers, the right quad slides one column per disparity (one scalar load per step), and
// every step emits one (diff) or two (concat) 128-bit streaming stores.  blockIdx.y splits D
// into chunks so small inputs still fill the machine.
template <bool kDiff>
__global__ void __launch_bounds__(256)
shift_volume_kernel(const float* __restrict__ fl, const float* __restrict__ fr, int C, int H, int W, int D,
                    int d_chunk, float* __restrict__ vol) {
  const int Wq = (W + 3) >> 2;
  const long long row_groups = (long long)H * Wq;
  const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= row_groups) return;
  const int nc = blockIdx.z;  // n * C + ci
  const int n = nc / C, ci = nc % C;
  const int y = (int)(g / Wq), x0 = (int)(g % Wq) * 4;
  const int d_lo = blockIdx.y * d_chunk, d_hi = min(D, d_lo + d_chunk);
  const float* lrow = fl + (((size_t)n * C + ci) * H + y) * W;
  const float* rrow = fr + (((size_t)n * C + ci) * H + y) * W;
  const int Cout = kDiff ? C : 2 * C;
  const size_t plane = (size_t)H * W;
  float* o_l = vol + ((((size_t)n * Cout + ci) * D + d_lo) * H + y) * W + x0;            // left copy / difference
  float* o_r = kDiff ? nullptr : o_l + (size_t)C * D * plane;                            // shifted right copy
  float l[4], r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int x = x0 + i;
    l[i] = (x < W) ? lrow[x] : 0.f;
    const int xr = x - d_lo;
    r[i] = (x < W && xr >= 0) ? rrow[xr] : 0.f;
  }
  const bool vec = (W & 3) == 0 && (reinterpret_cast<uintptr_t>(vol) & 15) == 0;   // 128-bit stores: aligned rows
  for (int d = d_lo; d < d_hi; ++d) {
    float a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const bool in = (x0 + i >= d) && (x0 + i < W);
      if (kDiff) a[i] = in ? __fsub_rn(l[i], r[i]) : 0.f;
      else {
        a[i] = in ? l[i] : 0.f;
        b[i] = in ? r[i] : 0.f;
      }
    }
    if (vec) {
      st_stream4(o_l, make_float4(a[0], a[1], a[2], a[3]));
      if (!kDiff) st_stream4(o_r, make_float4(b[0], b[1], b[2], b[3]));
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (x0 + i < W) {
          st_stream(o_l + i, a[i]);
          if (!kDiff) st_stream(o_r + i, b[i]);
        }
    }
    o_l += plane;
    if (!kDiff) o_r += plane;
    // next disparity: the right quad moves one column to the left
    r[3] = r[2]; r[2] = r[1]; r[1] = r[0];
    const int xn = x0 - (d + 1);
    r[0] = (xn >= 0 && x0 < W) ? rrow[xn] : 0.f;
  }
}

int launch_shift_volume(const float* fl, const float* fr, int N, int C, int H, int W, int D, bool diff,
                        float* vol, cudaStream_t s) {
  MSN_REQUIRE(N >= 0 && C >= 1 && H >= 0 && W >= 0 && D >= 1, "volume: bad shape");
  if (N == 0 || H == 0 || W == 0) return 0;
  MSN_REQUIRE((long long)N * C <= 65535, "volume: N*C too large for one launch");
  const unsigned gx = div_up((long long)H * ((W + 3) / 4), 256);
  // enough CTAs for a few waves of 148 SMs x 8 CTAs; otherwise one thread walks all of D
  int chunks = 1;
  while (chunks < D && (long long)gx * N * C * chunks < 4 * 148 * 8) chunks *= 2;
  const int d_chunk = (D + chunks - 1) / chunks;
  dim3 grid(gx, (D + d_chunk - 1) / d_chunk, N * C);
  if (diff) shift_volume_kernel<true><<<grid, 256, 0, s>>>(fl, fr, C, H, W, D, d_chunk, vol);
  else shift_volume_kernel<false><<<grid, 256, 0, s>>>(fl, fr, C, H, W, D, d_chunk, vol);
  MSN_LAUNCH_OK();
  return 0;
}

// Backward of the volumes above, G = d loss / d vol:
// concat: gfl[n][c][y][x]  =   sum_{d=0..min(x, D-1)}     G[n][c][d][y][x]
//         gfr[n][c][y][x'] =   sum_{d=0..min(W-1-x', D-1)} G[n][C+c][d][y][x'+d]
// diff  : gfl as concat from G[n][c], gfr = -(the concat sum, taken over G[n][c] as well)
// Every sum is in fp32, one rounding per add, d ascending from 0.0f, in one thread: no atomics and no split
// of a sum across threads, so the result is deterministic and equals the NumPy restatement bit for bit.
// A masked voxel (x < d, which covers every d >= W) never enters a sum, whatever it holds (NaN included);
// the forward wrote 0 there.  diff negates the finished sum (the same bits as adding negated terms).
//
// One thread owns 4 consecutive columns x0..x0+3 of one (n, c, y) row, of gfl and of gfr, and walks d
// kBwdChunk disparities at a time with every load of the chunk issued before the adds.  gfl: the aligned
// quad at x0 of each plane, streamed once from HBM (__ldcs) in the concat form.  gfr needs columns x0+d ..
// x0+d+3, the aligned quads k = d/4 and k+1 of the plane shifted by r = d % 4; d0 is a multiple of
// kBwdChunk, so r is a compile-time constant in the unrolled chunk.  Those quads are what the neighbouring
// threads of the warp (or the next warp) read at the same d, so across the grid every line of the
// gradient volume is fetched from DRAM once and the diagonal re-reads come from L1 / L2.
// The scalar form (W % 4 != 0 or a base pointer off 16 bytes) loads only the voxels it adds.
constexpr int kBwdChunk = 4;

template <bool kDiff, bool kVec>
__global__ void __launch_bounds__(256)
shift_volume_bwd_kernel(const float* __restrict__ g, int C, int H, int W, int D, float* __restrict__ gfl,
                        float* __restrict__ gfr) {
  static_assert(kBwdChunk % 4 == 0, "the gfr shift d % 4 must be a compile-time constant");
  const int Wq = (W + 3) >> 2;
  const long long row_groups = (long long)H * Wq;
  const long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= row_groups) return;
  const int nc = blockIdx.y;  // n * C + ci
  const int n = nc / C, ci = nc % C;
  const int y = (int)(q / Wq), x0 = (int)(q % Wq) * 4;
  const size_t plane = (size_t)H * W;
  const int Cg = kDiff ? C : 2 * C;
  const float* gl = g + ((size_t)n * Cg + ci) * D * plane + (size_t)y * W;   // plane 0 of G[n][c], row y
  const float* gr = kDiff ? gl : gl + (size_t)C * D * plane;                 // plane 0 of G[n][C+c] (concat)
  // sums of gfl run over d <= x (x <= x0+3), those of gfr over d <= W-1-x' (x' >= x0)
  const int dl_end = gfl ? min(D, x0 + 4) : 0;
  const int dr_end = gfr ? min(D, W - x0) : 0;
  const int d_end = max(dl_end, dr_end);
  float al[4] = {0.f, 0.f, 0.f, 0.f}, ar[4] = {0.f, 0.f, 0.f, 0.f};
  for (int d0 = 0; d0 < d_end; d0 += kBwdChunk) {
    float a[kBwdChunk][4], b[kBwdChunk][4];
#pragma unroll
    for (int j = 0; j < kBwdChunk; ++j) {
      const int d = d0 + j;
      const float* pl = gl + (size_t)d * plane;
      const float* pr = gr + (size_t)d * plane;
#pragma unroll
      for (int i = 0; i < 4; ++i) a[j][i] = b[j][i] = 0.f;
      if (kVec) {
        if (d < dl_end) {
          const float4 v = kDiff ? __ldg(reinterpret_cast<const float4*>(pl + x0))
                                 : __ldcs(reinterpret_cast<const float4*>(pl + x0));
          a[j][0] = v.x; a[j][1] = v.y; a[j][2] = v.z; a[j][3] = v.w;
        }
        if (d < dr_end) {  // x0 + d < W: quad k holds column x0+d, so it lies inside the row
          const int r = j & 3;
          const int xk = x0 + (d - r);
          const float4 u = __ldg(reinterpret_cast<const float4*>(pr + xk));
          float w[8] = {u.x, u.y, u.z, u.w, 0.f, 0.f, 0.f, 0.f};
          if (r != 0 && xk + 4 < W) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(pr + xk + 4));
            w[4] = t.x; w[5] = t.y; w[6] = t.z; w[7] = t.w;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i) b[j][i] = w[r + i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int x = x0 + i;
          if (d < dl_end && x >= d && x < W) a[j][i] = pl[x];
          if (d < dr_end && x + d < W) b[j][i] = pr[x + d];
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kBwdChunk; ++j) {
      const int d = d0 + j;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int x = x0 + i;
        if (d < dl_end && x >= d && x < W) al[i] += a[j][i];
        if (d < dr_end && x + d < W) ar[i] += b[j][i];
      }
    }
  }
  const size_t o = ((size_t)nc * H + y) * W + x0;
  if (kDiff) {
#pragma unroll
    for (int i = 0; i < 4; ++i) ar[i] = -ar[i];
  }
  if (kVec) {
    if (gfl) *reinterpret_cast<float4*>(gfl + o) = make_float4(al[0], al[1], al[2], al[3]);
    if (gfr) *reinterpret_cast<float4*>(gfr + o) = make_float4(ar[0], ar[1], ar[2], ar[3]);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if (x0 + i < W) {
        if (gfl) gfl[o + i] = al[i];
        if (gfr) gfr[o + i] = ar[i];
      }
  }
}

int launch_shift_volume_bwd(const float* grad, int N, int C, int H, int W, int D, bool diff, float* gfl,
                            float* gfr, cudaStream_t s) {
  MSN_REQUIRE(N >= 0 && C >= 1 && H >= 0 && W >= 0 && D >= 1, "volume_backward: bad shape");
  if (N == 0 || H == 0 || W == 0) return 0;
  MSN_REQUIRE((long long)N * C <= 65535, "volume_backward: N*C too large for one launch");
  auto aligned = [](const float* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  const bool vec = (W & 3) == 0 && aligned(grad) && aligned(gfl) && aligned(gfr);   // NULL is aligned
  // one thread per 4-column quad and all of its disparities: config P has 4.2 M quads per gradient
  dim3 grid(div_up((long long)H * ((W + 3) / 4), 256), N * C);
  if (diff) {
    if (vec) shift_volume_bwd_kernel<true, true><<<grid, 256, 0, s>>>(grad, C, H, W, D, gfl, gfr);
    else shift_volume_bwd_kernel<true, false><<<grid, 256, 0, s>>>(grad, C, H, W, D, gfl, gfr);
  } else {
    if (vec) shift_volume_bwd_kernel<false, true><<<grid, 256, 0, s>>>(grad, C, H, W, D, gfl, gfr);
    else shift_volume_bwd_kernel<false, false><<<grid, 256, 0, s>>>(grad, C, H, W, D, gfl, gfr);
  }
  MSN_LAUNCH_OK();
  return 0;
}

}  // namespace msn
