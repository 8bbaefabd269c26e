// common.cuh -- shared helpers for the msnets_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/msnets_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "msnets_b200 is written for sm_100a (B200) only"
#endif

namespace msn {

constexpr float kFill = MSN_FILL_VALUE;  // float(RAND_MAX), matchers.cpp:65
constexpr int kMaxCensusWords = 8;       // census window up to 16x16 bits

// thread-local error text behind msn_last_error()
void set_error(const char* fmt, ...);
int fail(const char* fmt, ...);  // sets the error, returns 1

#define MSN_CUDA_OK(expr)                                                              \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess)                                                             \
      return ::msn::fail("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
  } while (0)

#define MSN_LAUNCH_OK()                                                                \
  do {                                                                                 \
    cudaError_t _e = cudaGetLastError();                                               \
    if (_e != cudaSuccess)                                                             \
      return ::msn::fail("%s:%d kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
  } while (0)

#define MSN_REQUIRE(cond, ...)                      \
  do {                                              \
    if (!(cond)) return ::msn::fail(__VA_ARGS__);   \
  } while (0)

static inline unsigned div_up(long long a, long long b) { return (unsigned)((a + b - 1) / b); }
static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

// Valid window-origin geometry shared by every matcher (matchers.cpp loops run
// i < H-wsize, j < W-wsize; results land on the window centre (i+wc, j+wc)).
struct Win {
  int w, wc;
  __host__ __device__ Win(int wsize) : w(wsize), wc(wsize / 2) {}
  __host__ __device__ bool row_ok(int y, int H) const { return y >= wc && y < H - w + wc; }
  __host__ __device__ bool col_ok(int x, int W) const { return x >= wc && x < W - w + wc; }
  // cost (y, x, d) is written iff row_ok, col_ok and the origin column j = x-wc >= d
  __host__ __device__ bool ok(int y, int x, int d, int H, int W) const {
    return row_ok(y, H) && col_ok(x, W) && (x - wc) >= d;
  }
};

// streaming (evict-first) stores for the write-once cost volumes
__device__ __forceinline__ void st_stream(float* p, float v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream4(float* p, float4 v) { __stcs(reinterpret_cast<float4*>(p), v); }
// bf16 volume (SURVEY.md 8f-4): the same values rounded to nearest even, four pixels per 64-bit store
__device__ __forceinline__ void st_stream4(__nv_bfloat16* p, const float4& v) {
  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const unsigned*>(&lo);
  u.y = *reinterpret_cast<const unsigned*>(&hi);
  __stcs(reinterpret_cast<uint2*>(p), u);
}
__device__ __forceinline__ void st_stream(__nv_bfloat16* p, float v) { *p = __float2bfloat16_rn(v); }


// ---- host-side launchers (each returns 0 or sets the error and returns 1) ---
// prep.cu
int launch_census_transform(const uint8_t* img, int H, int W, int wsize, uint32_t* desc, cudaStream_t s);
int launch_window_mean(const uint8_t* img, int H, int W, int wsize, float* mean, cudaStream_t s);
int launch_ncc_stats(const uint8_t* img, int H, int W, int wsize, unsigned long long* A, double* C,
                     cudaStream_t s);
int launch_sobel(const uint8_t* img, int H, int W, float* out, cudaStream_t s);
int launch_fill(float* p, size_t n, float v, cudaStream_t s);
int launch_rescale(const uint8_t* in, int N, int H, int W, int oh, int ow, const double* w_rows, int r_rows,
                   const double* w_cols, int r_cols, double zoom_rows, double zoom_cols, uint8_t* out, float* tmp,
                   int* minmax, cudaStream_t s);
// matchers.cu
int launch_census_cost_hwd(const uint32_t* dl, const uint32_t* dr, int H, int W, int D, int wsize,
                           float* out, cudaStream_t s);
int launch_census_cost_dhw(const uint32_t* dl, const uint32_t* dr, int H, int W, int d_begin, int Dn,
                           int wsize, float* out, cudaStream_t s);
int launch_ncc_cost(const uint8_t* L, const uint8_t* R, const unsigned long long* Al,
                    const unsigned long long* Ar, const double* Cl, const double* Cr, int H, int W,
                    int d_begin, int Dn, int wsize, float* out, cudaStream_t s);
int launch_zsad_cost(const uint8_t* L, const uint8_t* R, const float* ml, const float* mr, int H, int W,
                     int d_begin, int Dn, int wsize, float* out, cudaStream_t s);
// sadsob.cu
size_t sadsob_workspace_bytes(int H, int W, int D, int wsize);
size_t sadsob_workspace_bytes_n(int N, int H, int W, int Dn, int wsize);
int launch_sadsob(const float* L, const float* R, int H, int W, int D, int d_begin, int wsize, float* out,
                  bool write_fill, void* workspace, cudaStream_t s);
int launch_sadsob_n(const float* L, const float* R, int N, int H, int W, int Dn, int d_begin, int wsize,
                    float* out, size_t out_stride, int out_pitch, bool write_fill, void* workspace,
                    cudaStream_t s);
constexpr int kSadRowPad = 32;  // zero rows below an image that enable the unguarded window-5 scan
int sadsob_fast_pitch(int W);    // 1024 / 2048 / 4096, or 0 when W is too wide
int launch_sadsob5_padded(const float* L, const float* R, int N, int H, int W, int Dn, int d_begin, float* out,
                          void* workspace, cudaStream_t s, bool d_inner = false, int row_lo = 0, int row_hi = -1,
                          bool tall_ok = true);
// row_lo / row_hi: only output rows [row_lo, row_hi) of the (bordered) image are needed (a row band of a frame
// sharded by rows): the band prefixes still start at row 0 -- the table of a row depends on every row above it --
// but only the bands that hold those rows are scanned.
// fte.cu
int launch_transpose2d(const float* in, long long A, long long B, float* out, cudaStream_t s);
int launch_reindex_cost(const float* c, int H, int W, int D, bool right, float* out, cudaStream_t s);
int launch_aml_rows(const float* cost, long long n, int D, float sigma, float* out, cudaStream_t s);
int launch_pkrn_rows(const float* cost, long long n, int D, float e, float* out, cudaStream_t s);
int launch_wta(const float* cost, long long n, int D, int layout, int d_begin, int32_t* amin, float* m1,
               float* m2, long long* keys, cudaStream_t s);
int launch_wta_unpack(const long long* keys, long long n, int32_t* amin, float* m1, cudaStream_t s);
int launch_wta_merge(const int32_t* idx_p, const float* m1_p, const float* m2_p, int parts, long long n, int32_t* idx,
                     float* m1, float* m2, cudaStream_t s);
int launch_pkrn_conf(const float* m1, const float* m2, long long n, float e, float* conf, cudaStream_t s);
int launch_lrc(const float* c, int H, int W, int D, int thresh, int32_t* dl, int32_t* dr, uint8_t* mask,
               cudaStream_t s);
// features.cu
int launch_features_from_costs(const float* census, const float* ncc, const float* sobel, const float* sad,
                               int h, int w, int D, float cens_sigma, float ncc_sigma, float sad_sigma, int lr,
                               float* out, cudaStream_t s);
// slab.cu
int launch_slab_phase_a(const float* census, const float* ncc, const float* sob, const float* sad, int H, int W,
                        int y0, int x0, int h, int w, int Dn, int d_begin, int lr, const float* d_first4,
                        float* out, float* mins, cudaStream_t s);
int launch_slab_right_view(float* out, int h, int w, int Dn, int d_begin, const float* d_first4, float* mins,
                           cudaStream_t s);
int launch_slab_phase_b(const float* out, const float* gmin, long long n, int Dn, int lr, float cens_sigma,
                        float ncc_sigma, float sad_sigma, float* den, cudaStream_t s);
int launch_slab_phase_c(float* out, const float* gmin, const float* gden, long long n, int Dn, int lr,
                        float cens_sigma, float ncc_sigma, float sad_sigma, cudaStream_t s);
// regress.cu
int launch_soft_argmin(const float* logits, int N, int D, int H, int W, int d_begin, int mode,
                       float* out, cudaStream_t s);
int launch_soft_argmin_bwd(const float* logits, const float* disp, const float* gout, int N, int D, int H, int W,
                           float* gin, cudaStream_t s);
int launch_soft_argmin_merge(const float* parts, int P, int N, int H, int W, float* disp, cudaStream_t s);
int launch_shift_volume(const float* fl, const float* fr, int N, int C, int H, int W, int D, bool diff,
                        float* vol, cudaStream_t s);
int launch_shift_volume_bwd(const float* grad, int N, int C, int H, int W, int D, bool diff, float* gfl,
                            float* gfr, cudaStream_t s);

}  // namespace msn
