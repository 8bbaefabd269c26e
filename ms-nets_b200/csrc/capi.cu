// capi.cu -- the extern "C" boundary declared in include/msnets_b200.h.
//
// Host entry points stage through stream-ordered device allocations
// (cudaMallocAsync) on a private per-thread stream; device entry points only
// enqueue on the caller's stream.  Nothing here computes on the CPU: without a
// device every entry point fails with a message.
#include <stdarg.h>
#include <stdlib.h>

#include <mutex>
#include <thread>
#include <vector>

#include "common.cuh"
#include "ms_fused.cuh"

namespace msn {
int g_aml_exact = 0;   // msn_set_aml_exact: AML in the reference's own fp32 operations (feature_math.cuh)

static thread_local char g_err[768] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
int fail(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return 1;
}

// ---- per-thread host-call context: one non-blocking stream + async allocations
struct HostCtx {
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  int init() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
      cudaGetLastError();
      return fail("no CUDA device available (%s); msnets_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    }
    MSN_CUDA_OK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    return 0;
  }
  int alloc(void** p, size_t bytes) {
    *p = nullptr;
    if (bytes == 0) bytes = 16;
    MSN_CUDA_OK(cudaMallocAsync(p, bytes, stream));
    allocs.push_back(*p);
    return 0;
  }
  template <class T>
  int upload(T** d, const T* h, size_t count) {
    if (alloc(reinterpret_cast<void**>(d), count * sizeof(T))) return 1;
    if (count) MSN_CUDA_OK(cudaMemcpyAsync(*d, h, count * sizeof(T), cudaMemcpyHostToDevice, stream));
    return 0;
  }
  // Results go back to PAGEABLE NumPy memory.  A plain cudaMemcpyAsync of gigabytes into pageable pages crawls
  // (measured 2.5 GB/s for the 3.2 GB volume of one config-B pair), so large results are staged: 32 MB chunks
  // alternate between two pinned buffers (kept for the life of the process); while chunk i+1 crosses PCIe, four
  // host threads copy chunk i out of its pinned buffer.
  template <class T>
  int download(T* h, const T* d, size_t count) {
    const size_t bytes = count * sizeof(T);
    if (bytes == 0) return 0;
    if (bytes < 2 * kStageBytes) {
      MSN_CUDA_OK(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, stream));
      return 0;
    }
    static std::mutex mu;                     // the two staging buffers are shared by every caller
    std::lock_guard<std::mutex> lk(mu);
    static char* pinned[2] = {nullptr, nullptr};
    for (int i = 0; i < 2; ++i)
      if (!pinned[i]) MSN_CUDA_OK(cudaHostAlloc(reinterpret_cast<void**>(&pinned[i]), kStageBytes, cudaHostAllocDefault));
    cudaEvent_t ev[2];
    for (int i = 0; i < 2; ++i) MSN_CUDA_OK(cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming));
    const char* src = reinterpret_cast<const char*>(d);
    char* dst = reinterpret_cast<char*>(h);
    const size_t chunks = (bytes + kStageBytes - 1) / kStageBytes;
    auto chunk_bytes = [&](size_t c) { return c + 1 < chunks ? kStageBytes : bytes - c * kStageBytes; };
    int rc = 0;
    for (size_t c = 0; c <= chunks && rc == 0; ++c) {
      if (c < chunks) {
        if (cudaMemcpyAsync(pinned[c & 1], src + c * kStageBytes, chunk_bytes(c), cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
            cudaEventRecord(ev[c & 1], stream) != cudaSuccess)
          rc = fail("download: staged copy failed");
      }
      if (c > 0 && rc == 0) {
        const size_t p = c - 1, nb = chunk_bytes(p);
        if (cudaEventSynchronize(ev[p & 1]) != cudaSuccess) { rc = fail("download: staged copy failed"); break; }
        constexpr int kThreads = 4;
        std::thread th[kThreads];
        const size_t slice = (nb + kThreads - 1) / kThreads;
        for (int t = 0; t < kThreads; ++t) {
          const size_t o = t * slice, n = o < nb ? (nb - o < slice ? nb - o : slice) : 0;
          th[t] = std::thread([=] { if (n) memcpy(dst + p * kStageBytes + o, pinned[p & 1] + o, n); });
        }
        for (int t = 0; t < kThreads; ++t) th[t].join();
      }
    }
    for (int i = 0; i < 2; ++i) cudaEventDestroy(ev[i]);
    return rc;
  }
  static constexpr size_t kStageBytes = 32u << 20;
  int finish() {
    for (void* p : allocs) cudaFreeAsync(p, stream);
    allocs.clear();
    MSN_CUDA_OK(cudaStreamSynchronize(stream));
    return 0;
  }
  ~HostCtx() {
    if (stream) {
      for (void* p : allocs) cudaFreeAsync(p, stream);
      cudaStreamSynchronize(stream);
      cudaStreamDestroy(stream);
    }
  }
};

#define HOST_BEGIN()  \
  ::msn::HostCtx ctx; \
  if (ctx.init()) return 1
#define TRY(expr)          \
  do {                     \
    if ((expr)) return 1;  \
  } while (0)

static int check_image_args(const void* l, const void* r, int H, int W, int ndisp, int wsize, const void* out,
                            const char* who, int max_w) {
  MSN_REQUIRE(l && r && out, "%s: null pointer argument", who);
  MSN_REQUIRE(H >= 1 && W >= 1, "%s: bad image shape %dx%d", who, H, W);
  MSN_REQUIRE(ndisp >= 1, "%s: ndisp must be >= 1 (got %d)", who, ndisp);
  MSN_REQUIRE(wsize >= 1 && wsize <= max_w, "%s: wsize %d unsupported (1..%d)", who, wsize, max_w);
  MSN_REQUIRE(H <= 65535 && ndisp <= 65535, "%s: H and ndisp must be <= 65535", who);
  return 0;
}

// ---------------------------------------------------------------- matchers --
static int census_dev(const uint8_t* dl, const uint8_t* dr, int H, int W, int D, int wsize, float* out,
                      uint32_t* descl, uint32_t* descr, cudaStream_t s) {
  TRY(launch_census_transform(dl, H, W, wsize, descl, s));
  TRY(launch_census_transform(dr, H, W, wsize, descr, s));
  return launch_census_cost_hwd(descl, descr, H, W, D, wsize, out, s);
}

struct StreamScratch {  // scratch for *_dev calls that need temporaries
  cudaStream_t s;
  std::vector<void*> ptrs;
  explicit StreamScratch(cudaStream_t st) : s(st) {}
  int get(void** p, size_t bytes) {
    MSN_CUDA_OK(cudaMallocAsync(p, bytes ? bytes : 16, s));
    ptrs.push_back(*p);
    return 0;
  }
  ~StreamScratch() {
    for (void* p : ptrs) cudaFreeAsync(p, s);
  }
};

}  // namespace msn

using namespace msn;

extern "C" {

const char* msn_last_error(void) { return g_err; }
int msn_abi_version(void) { return MSN_ABI_VERSION; }

int msn_device_count(int* count) {
  MSN_REQUIRE(count, "msn_device_count: null argument");
  *count = 0;
  cudaError_t e = cudaGetDeviceCount(count);
  if (e != cudaSuccess) {
    cudaGetLastError();
    *count = 0;
  }
  return 0;
}

int msn_set_device(int device) {
  MSN_CUDA_OK(cudaSetDevice(device));
  return 0;
}

int msn_initthreads(int* count) {
  MSN_REQUIRE(count, "msn_initthreads: null argument");
  int dev = 0, sms = 0;
  MSN_CUDA_OK(cudaGetDevice(&dev));
  MSN_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  *count = sms;
  return 0;
}

void msn_ms_params_default(msn_ms_params* p) {
  if (!p) return;
  p->ndisp = 192;
  p->censw = 11; p->nccw = 3; p->sadw = 5; p->sobelw = 5;   // cbmv_generator.py:437-440
  p->board_h = 10; p->board_w_left = 10; p->board_w_right = 0;  // get_costs defaults, :27
  p->cens_sigma = 128.0f; p->ncc_sigma = 0.02f; p->sad_sigma = 20000.0f;  // :441-444
  p->lr = 0;
  p->d_begin = 0; p->d_count = 0;
  p->row_begin = 0; p->row_count = 0;
}

// ------------------------------------------------------- device matchers --
int msn_census_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                   float* d_out_hwd, void* stream) {
  TRY(check_image_args(d_left, d_right, H, W, ndisp, wsize, d_out_hwd, "census", 16));
  cudaStream_t s = as_stream(stream);
  StreamScratch sc(s);
  const size_t nw = (wsize * wsize + 31) / 32;
  uint32_t *dl, *dr;
  TRY(sc.get((void**)&dl, (size_t)H * W * nw * 4));
  TRY(sc.get((void**)&dr, (size_t)H * W * nw * 4));
  return census_dev(d_left, d_right, H, W, ndisp, wsize, d_out_hwd, dl, dr, s);
}

int msn_ncc_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                float* d_out_dhw, void* stream) {
  TRY(check_image_args(d_left, d_right, H, W, ndisp, wsize, d_out_dhw, "nccNister", 255));
  cudaStream_t s = as_stream(stream);
  StreamScratch sc(s);
  unsigned long long *al, *ar;
  double *cl, *cr;
  const size_t n = (size_t)H * W;
  TRY(sc.get((void**)&al, n * 8)); TRY(sc.get((void**)&ar, n * 8));
  TRY(sc.get((void**)&cl, n * 8)); TRY(sc.get((void**)&cr, n * 8));
  TRY(launch_ncc_stats(d_left, H, W, wsize, al, cl, s));
  TRY(launch_ncc_stats(d_right, H, W, wsize, ar, cr, s));
  return launch_ncc_cost(d_left, d_right, al, ar, cl, cr, H, W, 0, ndisp, wsize, d_out_dhw, s);
}

int msn_zsad_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                 float* d_out_dhw, void* stream) {
  TRY(check_image_args(d_left, d_right, H, W, ndisp, wsize, d_out_dhw, "zsad", 255));
  cudaStream_t s = as_stream(stream);
  StreamScratch sc(s);
  float *ml, *mr;
  const size_t n = (size_t)H * W;
  TRY(sc.get((void**)&ml, n * 4)); TRY(sc.get((void**)&mr, n * 4));
  TRY(launch_window_mean(d_left, H, W, wsize, ml, s));
  TRY(launch_window_mean(d_right, H, W, wsize, mr, s));
  return launch_zsad_cost(d_left, d_right, ml, mr, H, W, 0, ndisp, wsize, d_out_dhw, s);
}

int msn_sobel_dev(const uint8_t* d_img, int H, int W, float* d_out_hw, void* stream) {
  MSN_REQUIRE(d_img && d_out_hw, "sobel: null pointer argument");
  MSN_REQUIRE(H >= 1 && W >= 1 && H <= 65535, "sobel: bad image shape %dx%d", H, W);
  return launch_sobel(d_img, H, W, d_out_hw, as_stream(stream));
}

size_t msn_rescale_workspace_bytes(int N, int H, int W) {
  return (size_t)N * H * W * sizeof(float) + (size_t)N * 2 * sizeof(int) + 512;
}

int msn_rescale_dev(const uint8_t* d_in, int N, int H, int W, int out_h, int out_w, const double* w_rows, int r_rows,
                    const double* w_cols, int r_cols, double zoom_rows, double zoom_cols, uint8_t* d_out,
                    void* d_workspace, size_t workspace_bytes, void* stream) {
  MSN_REQUIRE(d_in && d_out && d_workspace, "rescale: null pointer argument");
  MSN_REQUIRE(N >= 0 && H >= 1 && W >= 1 && out_h >= 1 && out_w >= 1, "rescale: bad shape");
  MSN_REQUIRE((r_rows < 0 || w_rows) && (r_cols < 0 || w_cols), "rescale: filter weights missing");
  MSN_REQUIRE(workspace_bytes >= msn_rescale_workspace_bytes(N, H, W), "rescale: workspace too small");
  if (N == 0) return 0;
  char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
  float* tmp = reinterpret_cast<float*>(base);
  int* mm = reinterpret_cast<int*>(base + (size_t)N * H * W * sizeof(float));
  return launch_rescale(d_in, N, H, W, out_h, out_w, w_rows, r_rows, w_cols, r_cols, zoom_rows, zoom_cols, d_out, tmp, mm,
                        as_stream(stream));
}

int msn_rescale_host(const uint8_t* in, int N, int H, int W, int out_h, int out_w, const double* w_rows, int r_rows,
                     const double* w_cols, int r_cols, double zoom_rows, double zoom_cols, uint8_t* out) {
  MSN_REQUIRE(in && out, "rescale: null pointer argument");
  MSN_REQUIRE(N >= 0 && H >= 1 && W >= 1 && out_h >= 1 && out_w >= 1, "rescale: bad shape");
  HOST_BEGIN();
  uint8_t *di, *dout;
  void* ws;
  TRY(ctx.upload(&di, in, (size_t)N * H * W));
  TRY(ctx.alloc((void**)&dout, (size_t)N * out_h * out_w));
  TRY(ctx.alloc(&ws, msn_rescale_workspace_bytes(N, H, W)));
  TRY(msn_rescale_dev(di, N, H, W, out_h, out_w, w_rows, r_rows, w_cols, r_cols, zoom_rows, zoom_cols, dout, ws,
                      msn_rescale_workspace_bytes(N, H, W), ctx.stream));
  TRY(ctx.download(out, dout, (size_t)N * out_h * out_w));
  return ctx.finish();
}

int msn_sadsob_dev(const float* d_left, const float* d_right, int H, int W, int ndisp, int wsize,
                   float* d_out_dhw, void* stream) {
  TRY(check_image_args(d_left, d_right, H, W, ndisp, wsize, d_out_dhw, "sadsob", 16));
  cudaStream_t s = as_stream(stream);
  StreamScratch sc(s);
  void* ws;
  TRY(sc.get(&ws, sadsob_workspace_bytes(H, W, ndisp, wsize)));
  return launch_sadsob(d_left, d_right, H, W, ndisp, 0, wsize, d_out_dhw, true, ws, s);
}

int msn_aml_dev(const float* d_cost_nd, long long n, int D, float sigma, float* d_out_nd, void* stream) {
  MSN_REQUIRE(d_cost_nd && d_out_nd, "extract_likelihood: null pointer argument");
  MSN_REQUIRE(n >= 0 && D >= 1, "extract_likelihood: bad shape [%lld][%d]", n, D);
  MSN_REQUIRE(sigma > 0.f, "extract_likelihood: sigma must be > 0");
  return launch_aml_rows(d_cost_nd, n, D, sigma, d_out_nd, as_stream(stream));
}

int msn_pkrn_dev(const float* d_cost_nd, long long n, int D, float e, float* d_out_nd, void* stream) {
  MSN_REQUIRE(d_cost_nd && d_out_nd, "extract_ratio: null pointer argument");
  MSN_REQUIRE(n >= 0 && D >= 1, "extract_ratio: bad shape [%lld][%d]", n, D);
  return launch_pkrn_rows(d_cost_nd, n, D, e, d_out_nd, as_stream(stream));
}

// --------------------------------------------------------- host matchers --
int msn_census_host(const uint8_t* left, const uint8_t* right, int H, int W, int ndisp, int wsize,
                    float* out_hwd) {
  TRY(check_image_args(left, right, H, W, ndisp, wsize, out_hwd, "census", 16));
  HOST_BEGIN();
  const size_t n = (size_t)H * W;
  uint8_t *dl, *dr;
  float* dout;
  TRY(ctx.upload(&dl, left, n)); TRY(ctx.upload(&dr, right, n));
  TRY(ctx.alloc((void**)&dout, n * ndisp * 4));
  TRY(msn_census_dev(dl, dr, H, W, ndisp, wsize, dout, ctx.stream));
  TRY(ctx.download(out_hwd, dout, n * ndisp));
  return ctx.finish();
}

#define HOST_U8_MATCHER(NAME, DEVFN, WHO, MAXW)                                                     \
  int NAME(const uint8_t* left, const uint8_t* right, int H, int W, int ndisp, int wsize,           \
           float* out_dhw) {                                                                        \
    TRY(check_image_args(left, right, H, W, ndisp, wsize, out_dhw, WHO, MAXW));                     \
    HOST_BEGIN();                                                                                   \
    const size_t n = (size_t)H * W;                                                                 \
    uint8_t *dl, *dr;                                                                               \
    float* dout;                                                                                    \
    TRY(ctx.upload(&dl, left, n)); TRY(ctx.upload(&dr, right, n));                                  \
    TRY(ctx.alloc((void**)&dout, n * ndisp * 4));                                                   \
    TRY(DEVFN(dl, dr, H, W, ndisp, wsize, dout, ctx.stream));                                       \
    TRY(ctx.download(out_dhw, dout, n * ndisp));                                                    \
    return ctx.finish();                                                                            \
  }
HOST_U8_MATCHER(msn_ncc_host, msn_ncc_dev, "nccNister", 255)
HOST_U8_MATCHER(msn_zsad_host, msn_zsad_dev, "zsad", 255)

int msn_sobel_host(const uint8_t* img, int H, int W, float* out_hw) {
  MSN_REQUIRE(img && out_hw, "sobel: null pointer argument");
  MSN_REQUIRE(H >= 1 && W >= 1 && H <= 65535, "sobel: bad image shape %dx%d", H, W);
  HOST_BEGIN();
  const size_t n = (size_t)H * W;
  uint8_t* di;
  float* dout;
  TRY(ctx.upload(&di, img, n));
  TRY(ctx.alloc((void**)&dout, n * 4));
  TRY(msn_sobel_dev(di, H, W, dout, ctx.stream));
  TRY(ctx.download(out_hw, dout, n));
  return ctx.finish();
}

int msn_sadsob_host(const float* left, const float* right, int H, int W, int ndisp, int wsize,
                    float* out_dhw) {
  TRY(check_image_args(left, right, H, W, ndisp, wsize, out_dhw, "sadsob", 16));
  HOST_BEGIN();
  const size_t n = (size_t)H * W;
  float *dl, *dr, *dout;
  TRY(ctx.upload(&dl, left, n)); TRY(ctx.upload(&dr, right, n));
  TRY(ctx.alloc((void**)&dout, n * ndisp * 4));
  TRY(msn_sadsob_dev(dl, dr, H, W, ndisp, wsize, dout, ctx.stream));
  TRY(ctx.download(out_dhw, dout, n * ndisp));
  return ctx.finish();
}

// ----------------------------------------------------- host featextract --
static int host_unary(const float* in, size_t count, float* out, const char* who,
                      int (*run)(const float*, float*, cudaStream_t, void*), void* arg) {
  MSN_REQUIRE(in && out, "%s: null pointer argument", who);
  HOST_BEGIN();
  float *din, *dout;
  TRY(ctx.upload(&din, in, count));
  TRY(ctx.alloc((void**)&dout, count * 4));
  TRY(run(din, dout, ctx.stream, arg));
  TRY(ctx.download(out, dout, count));
  return ctx.finish();
}

struct Shape3 { long long a, b, c; float f; };

int msn_swap_axes_host(const float* in_dhw, int D, int H, int W, float* out_hwd) {
  MSN_REQUIRE(D >= 1 && H >= 1 && W >= 1, "swap_axes: bad shape [%d][%d][%d]", D, H, W);
  Shape3 sh{D, (long long)H * W, 0, 0.f};
  return host_unary(in_dhw, (size_t)D * H * W, out_hwd, "swap_axes",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_transpose2d(i, q->a, q->b, o, s);
                    }, &sh);
}

int msn_swap_axes_back_host(const float* in_hwd, int H, int W, int D, float* out_dhw) {
  MSN_REQUIRE(D >= 1 && H >= 1 && W >= 1, "swap_axes_back: bad shape [%d][%d][%d]", H, W, D);
  Shape3 sh{(long long)H * W, D, 0, 0.f};
  MSN_REQUIRE((sh.a + 31) / 32 <= 65535, "swap_axes_back: H*W too large");
  return host_unary(in_hwd, (size_t)D * H * W, out_dhw, "swap_axes_back",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_transpose2d(i, q->a, q->b, o, s);
                    }, &sh);
}

int msn_right_cost_host(const float* cost_hwd, int H, int W, int D, float* out_hwd) {
  MSN_REQUIRE(D >= 1 && H >= 1 && W >= 1, "get_right_cost: bad shape [%d][%d][%d]", H, W, D);
  Shape3 sh{H, W, D, 0.f};
  return host_unary(cost_hwd, (size_t)D * H * W, out_hwd, "get_right_cost",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_reindex_cost(i, (int)q->a, (int)q->b, (int)q->c, true, o, s);
                    }, &sh);
}

int msn_left_cost_host(const float* cost_hwd, int H, int W, int D, float* out_hwd) {
  MSN_REQUIRE(D >= 1 && H >= 1 && W >= 1, "get_left_cost: bad shape [%d][%d][%d]", H, W, D);
  Shape3 sh{H, W, D, 0.f};
  return host_unary(cost_hwd, (size_t)D * H * W, out_hwd, "get_left_cost",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_reindex_cost(i, (int)q->a, (int)q->b, (int)q->c, false, o, s);
                    }, &sh);
}

int msn_aml_host(const float* cost_nd, long long n, int D, float sigma, float* out_nd) {
  MSN_REQUIRE(n >= 0 && D >= 1, "extract_likelihood: bad shape [%lld][%d]", n, D);
  MSN_REQUIRE(sigma > 0.f, "extract_likelihood: sigma must be > 0");
  Shape3 sh{n, D, 0, sigma};
  return host_unary(cost_nd, (size_t)n * D, out_nd, "extract_likelihood",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_aml_rows(i, q->a, (int)q->b, q->f, o, s);
                    }, &sh);
}

int msn_pkrn_host(const float* cost_nd, long long n, int D, float e, float* out_nd) {
  MSN_REQUIRE(n >= 0 && D >= 1, "extract_ratio: bad shape [%lld][%d]", n, D);
  Shape3 sh{n, D, 0, e};
  return host_unary(cost_nd, (size_t)n * D, out_nd, "extract_ratio",
                    [](const float* i, float* o, cudaStream_t s, void* a) {
                      Shape3* q = (Shape3*)a;
                      return launch_pkrn_rows(i, q->a, (int)q->b, q->f, o, s);
                    }, &sh);
}

int msn_features_from_costs_host(const float* census_hwd, const float* ncc_hwd, const float* sobel_hwd,
                                 const float* sad_hwd, int h, int w, int D, float cens_sigma, float ncc_sigma,
                                 float sad_sigma, int lr, float* out_cdhw) {
  MSN_REQUIRE(census_hwd && ncc_hwd && sobel_hwd && sad_hwd && out_cdhw, "extract_features: null pointer argument");
  MSN_REQUIRE(h >= 1 && w >= 1 && D >= 1, "extract_features: bad shape [%d][%d][%d]", h, w, D);
  MSN_REQUIRE(cens_sigma > 0 && ncc_sigma > 0 && sad_sigma > 0, "extract_features: sigmas must be > 0");
  HOST_BEGIN();
  const size_t n = (size_t)h * w * D;
  float *c0, *c1, *c2, *c3, *dout;
  TRY(ctx.upload(&c0, census_hwd, n)); TRY(ctx.upload(&c1, ncc_hwd, n));
  TRY(ctx.upload(&c2, sobel_hwd, n)); TRY(ctx.upload(&c3, sad_hwd, n));
  const size_t C = lr ? 16 : 8;
  TRY(ctx.alloc((void**)&dout, C * n * 4));
  TRY(launch_features_from_costs(c0, c1, c2, c3, h, w, D, cens_sigma, ncc_sigma, sad_sigma, lr, dout, ctx.stream));
  TRY(ctx.download(out_cdhw, dout, C * n));
  return ctx.finish();
}

// ------------------------------------------------ MS feature pipeline --
namespace {

struct Geometry {
  int H, W, h, w, D, d_begin, Dn, C;   // h: output rows (the row band's when one is requested)
  bool band;
};

int resolve(const msn_ms_params* p, int N, int H, int W, Geometry* g, const char* who) {
  MSN_REQUIRE(p, "%s: null params", who);
  MSN_REQUIRE(N >= 0 && H >= 1 && W >= 1 && H <= 65535, "%s: bad input shape N=%d H=%d W=%d", who, N, H, W);
  MSN_REQUIRE(p->ndisp >= 1 && p->ndisp <= 65535, "%s: ndisp %d out of range", who, p->ndisp);
  MSN_REQUIRE(p->censw >= 1 && p->censw <= 16, "%s: censw %d unsupported (1..16)", who, p->censw);
  MSN_REQUIRE(p->sobelw >= 1 && p->sobelw <= 16, "%s: sobelw %d unsupported (1..16)", who, p->sobelw);
  MSN_REQUIRE(p->nccw >= 1 && p->nccw <= 255 && p->sadw >= 1 && p->sadw <= 255, "%s: bad nccw/sadw", who);
  MSN_REQUIRE(p->board_h >= 0 && p->board_w_left >= 0 && p->board_w_right >= 0, "%s: negative border", who);
  MSN_REQUIRE(p->cens_sigma > 0 && p->ncc_sigma > 0 && p->sad_sigma > 0, "%s: sigmas must be > 0", who);
  g->H = H; g->W = W;
  g->h = H - 2 * p->board_h;
  g->w = W - p->board_w_left - p->board_w_right;
  MSN_REQUIRE(g->h >= 1 && g->w >= 1, "%s: borders (%d,%d,%d) leave nothing of a %dx%d image", who, p->board_h,
              p->board_w_left, p->board_w_right, H, W);
  g->band = p->row_count > 0;
  if (g->band) {
    MSN_REQUIRE(p->row_begin >= 0 && p->row_begin + p->row_count <= g->h, "%s: row band [%d,%d) outside [0,%d)", who,
                p->row_begin, p->row_begin + p->row_count, g->h);
    g->h = p->row_count;
  }
  g->D = p->ndisp;
  g->d_begin = p->d_count > 0 ? p->d_begin : 0;
  g->Dn = p->d_count > 0 ? p->d_count : p->ndisp;
  MSN_REQUIRE(g->d_begin >= 0 && g->d_begin + g->Dn <= g->D, "%s: slab [%d,%d) outside [0,%d)", who, g->d_begin,
              g->d_begin + g->Dn, g->D);
  g->C = p->lr ? 16 : 8;
  return 0;
}

size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// workspace carve-up of the generic (three-phase) path, one pair at a time
struct GenericWs {
  uint32_t *descl, *descr;
  float *ml, *mr, *sobl, *sobr;
  unsigned long long *al, *ar;
  double *cl, *cr;
  float* raw[4];
  void* sad_ws;
  float *mins, *den;
  size_t total;
  void carve(char* base, const Geometry& g, const msn_ms_params* p) {
    size_t off = 0;
    auto take = [&](size_t bytes) { char* q = base ? base + off : nullptr; off += align256(bytes); return q; };
    const size_t n = (size_t)g.H * g.W, nw = (p->censw * p->censw + 31) / 32;
    descl = (uint32_t*)take(n * nw * 4); descr = (uint32_t*)take(n * nw * 4);
    ml = (float*)take(n * 4); mr = (float*)take(n * 4);
    sobl = (float*)take(n * 4); sobr = (float*)take(n * 4);
    al = (unsigned long long*)take(n * 8); ar = (unsigned long long*)take(n * 8);
    cl = (double*)take(n * 8); cr = (double*)take(n * 8);
    for (int m = 0; m < 4; ++m) raw[m] = (float*)take(n * g.Dn * 4);
    sad_ws = take(sadsob_workspace_bytes(g.H, g.W, g.Dn, p->sobelw));
    mins = (float*)take((size_t)8 * g.h * g.w * 4);
    den = (float*)take((size_t)8 * g.h * g.w * 4);
    total = off;
  }
};

// prep + four matchers for the slab + phase A, for pair `n`
int generic_phase_a(const uint8_t* dl, const uint8_t* dr, const Geometry& g, const msn_ms_params* p, GenericWs& ws,
                    const float* d_first4, float* out, float* mins, cudaStream_t s) {
  TRY(launch_census_transform(dl, g.H, g.W, p->censw, ws.descl, s));
  TRY(launch_census_transform(dr, g.H, g.W, p->censw, ws.descr, s));
  TRY(launch_census_cost_dhw(ws.descl, ws.descr, g.H, g.W, g.d_begin, g.Dn, p->censw, ws.raw[0], s));
  TRY(launch_ncc_stats(dl, g.H, g.W, p->nccw, ws.al, ws.cl, s));
  TRY(launch_ncc_stats(dr, g.H, g.W, p->nccw, ws.ar, ws.cr, s));
  TRY(launch_ncc_cost(dl, dr, ws.al, ws.ar, ws.cl, ws.cr, g.H, g.W, g.d_begin, g.Dn, p->nccw, ws.raw[1], s));
  TRY(launch_sobel(dl, g.H, g.W, ws.sobl, s));
  TRY(launch_sobel(dr, g.H, g.W, ws.sobr, s));
  TRY(launch_sadsob(ws.sobl, ws.sobr, g.H, g.W, g.Dn, g.d_begin, p->sobelw, ws.raw[2], true, ws.sad_ws, s));
  TRY(launch_window_mean(dl, g.H, g.W, p->sadw, ws.ml, s));
  TRY(launch_window_mean(dr, g.H, g.W, p->sadw, ws.mr, s));
  TRY(launch_zsad_cost(dl, dr, ws.ml, ws.mr, g.H, g.W, g.d_begin, g.Dn, p->sadw, ws.raw[3], s));
  return launch_slab_phase_a(ws.raw[0], ws.raw[1], ws.raw[2], ws.raw[3], g.H, g.W, p->board_h, p->board_w_left,
                             g.h, g.w, g.Dn, g.d_begin, p->lr, d_first4, out, mins, s);
}

bool force_generic() {
  const char* e = getenv("MSNETS_FORCE_GENERIC");
  return e && e[0] == '1';
}

}  // namespace

// The fused kernel serves the default windows.  Left view only (lr = 0): one launch writes the
// final volume.  Both views (lr = 1): the fused kernel runs in its phase-A form (channels 0-3
// final, raw costs parked in 4-7, minima), slab.cu derives channels 8-15 from the parked costs and
// phases B/C finish all eight AML channels; mins/den [N][8][h][w] follow the fused workspace.
static bool use_fused(const msn_ms_params* p, const Geometry& g, int W) {
  return fused_supported(p, g.Dn) && sadsob_fast_pitch(W + 35) > 0 && !force_generic();
}
// More disparities than one fused launch parks in shared memory (left view, default windows): the
// volume is cut into slabs of kFusedSlabD disparities, each through the fused kernel's phase-A
// form, then phases B/C over all disparities -- the slab-sharding scheme of SURVEY.md 8e on one GPU.
static bool use_fused_slabs(const msn_ms_params* p, const Geometry& g, int W) {
  return !p->lr && g.Dn == g.D && !fused_supported(p, g.Dn) && fused_supported(p, kFusedSlabD) &&
         sadsob_fast_pitch(W + 35) > 0 && !force_generic();
}
// ... and when those slabs can be EQUAL (D divisible by their number), they run as sub-slabs of ONE launch of
// the fused kernel's exchange form instead (one rank, `subs` virtual ranks): the tiles of a pixel trade their
// minima / denominators through a table in the workspace and the volume is written once -- no parked costs,
// no phases B/C (2.5x less DRAM traffic).
// Opt-in (MSNETS_ONE_GPU_EXCHANGE=1): measured on config M (1984x2880, D = 640, one B200) the two routes are
// within 4 % of each other (78.8 vs 81.6 ms) -- with four sub-slabs in flight the 117 GB of scattered output
// rows, not the parked-cost traffic, sets the pace -- and the exchange route needs the SAD-of-Sobel scratch of
// all 640 disparities at once (21 GB instead of 6 GB).
static int exchange_subs(const msn_ms_params* p, const Geometry& g, int W) {
  const char* e = getenv("MSNETS_ONE_GPU_EXCHANGE");
  if (!(e && e[0] == '1') || !use_fused_slabs(p, g, W)) return 0;
  const int subs = (g.D + kFusedSlabD - 1) / kFusedSlabD;
  return (g.D % subs == 0) ? subs : 0;
}
static msn_ms_params slab_params(const msn_ms_params* p, int d0, int dn) {
  msn_ms_params q = *p;
  q.d_begin = d0;
  q.d_count = dn;
  return q;
}


size_t msn_ms_features_workspace_bytes(int N, int H, int W, const msn_ms_params* p) {
  Geometry g;
  if (resolve(p, N, H, W, &g, "ms_features_workspace_bytes")) return 0;
  if (use_fused(p, g, W)) {
    size_t need = align256(fused_workspace_bytes(N, H, W, g.Dn, p));
    if (p->lr) need += 2 * align256((size_t)N * 8 * g.h * g.w * sizeof(float));
    return need + 256;
  }
  if (const int subs = exchange_subs(p, g, W))
    return align256(fused_workspace_bytes(N, H, W, g.D, p)) + align256(fused_exchange_bytes(N, H, W, p, subs)) + 256;
  if (use_fused_slabs(p, g, W)) {
    // sized for the slab with the largest disparity offset (widest left padding) and a full count
    const msn_ms_params q = slab_params(p, g.D - kFusedSlabD, kFusedSlabD);
    return align256(fused_workspace_bytes(N, H, W, kFusedSlabD, &q)) +
           2 * align256((size_t)N * 4 * g.h * g.w * sizeof(float)) + 256;
  }
  GenericWs ws;
  ws.carve(nullptr, g, p);
  return ws.total + 256;
}

int msn_ms_features_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                        const msn_ms_params* p, float* d_out, void* d_workspace, size_t workspace_bytes,
                        void* stream) {
  return msn_ms_features_wta_dev(d_left, d_right, N, H, W, p, d_out, nullptr, nullptr, nullptr, d_workspace,
                                 workspace_bytes, stream);
}

int msn_ms_features_wta_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                            const msn_ms_params* p, float* d_out, int32_t* d_wta_idx, float* d_wta_min1,
                            float* d_wta_min2, void* d_workspace, size_t workspace_bytes, void* stream) {
  Geometry g;
  TRY(resolve(p, N, H, W, &g, "ms_features"));
  const bool want_wta = d_wta_idx || d_wta_min1 || d_wta_min2;
  MSN_REQUIRE(!want_wta || (d_wta_idx && d_wta_min1 && d_wta_min2), "ms_features: pass all three WTA planes or none");
  MSN_REQUIRE(!want_wta || (use_fused(p, g, W) && !p->lr),
              "ms_features: the WTA by-product comes from the fused kernel (default windows, left view, D <= 448); "
              "use msn_wta_dev on the volume otherwise");
  const FusedWta wta{d_wta_idx, d_wta_min1, d_wta_min2};
  MSN_REQUIRE(d_left && d_right && d_out && d_workspace, "ms_features: null pointer argument");
  MSN_REQUIRE(workspace_bytes >= msn_ms_features_workspace_bytes(N, H, W, p),
              "ms_features: workspace too small (%zu < %zu)", workspace_bytes,
              msn_ms_features_workspace_bytes(N, H, W, p));
  MSN_REQUIRE(g.d_begin == 0 && g.Dn == g.D, "ms_features: slabs go through msn_ms_slab_phase_*_dev");
  MSN_REQUIRE(!g.band || (use_fused(p, g, W) && !p->lr), "ms_features: a row band needs the fused path (default windows, left view, D <= 448)");
  cudaStream_t s = as_stream(stream);
  char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
  const size_t n = (size_t)g.h * g.w;
  if (use_fused(p, g, W)) {
    if (!p->lr) return launch_ms_fused(d_left, d_right, N, H, W, p, d_out, nullptr, base, s, 0, 0, 0, nullptr, &wta);
    // both views, fast AML mode: two one-pass launches -- the left view as above into channels 0-7, then the right
    // view (channels 8-15) recomputed from the images with the roles swapped (ms_fused.cu: phase1_tile_right); the
    // volume is written once and never re-read.  The exact AML mode keeps the three-phase route below.
    if (!g_aml_exact) return launch_ms_fused(d_left, d_right, N, H, W, p, d_out, nullptr, base, s);
    const size_t stat_bytes = align256((size_t)N * 8 * n * sizeof(float));
    float* mins = reinterpret_cast<float*>(base + align256(fused_workspace_bytes(N, H, W, g.Dn, p)));
    float* den = reinterpret_cast<float*>(reinterpret_cast<char*>(mins) + stat_bytes);
    TRY(launch_ms_fused(d_left, d_right, N, H, W, p, d_out, mins, base, s));
    for (int i = 0; i < N; ++i) {
      float* out = d_out + (size_t)i * 16 * g.Dn * n;
      TRY(launch_slab_right_view(out, g.h, g.w, g.Dn, 0, nullptr, mins + (size_t)i * 8 * n, s));
      TRY(launch_slab_phase_b(out, mins + (size_t)i * 8 * n, (long long)n, g.Dn, 1, p->cens_sigma, p->ncc_sigma,
                              p->sad_sigma, den + (size_t)i * 8 * n, s));
      TRY(launch_slab_phase_c(out, mins + (size_t)i * 8 * n, den + (size_t)i * 8 * n, (long long)n, g.Dn, 1,
                              p->cens_sigma, p->ncc_sigma, p->sad_sigma, s));
    }
    return 0;
  }
  if (const int subs = exchange_subs(p, g, W)) {
    char* table = base + align256(fused_workspace_bytes(N, H, W, g.D, p));
    const size_t tb = fused_exchange_bytes(N, H, W, p, subs);
    msn_slab_exchange x;
    memset(&x, 0, sizeof(x));
    x.tables[0] = table; x.world = 1; x.rank = 0; x.epoch = 1; x.subs = subs;
    MSN_CUDA_OK(cudaMemsetAsync(table + tb / 2, 0, tb / 2, s));   // epoch 1 lives in the table's second half
    return launch_ms_fused(d_left, d_right, N, H, W, p, d_out, nullptr, base, s, g.D, 0, 0, &x);
  }
  if (use_fused_slabs(p, g, W)) {
    const msn_ms_params q0 = slab_params(p, g.D - kFusedSlabD, kFusedSlabD);
    const size_t stat_bytes = align256((size_t)N * 4 * n * sizeof(float));
    float* mins = reinterpret_cast<float*>(base + align256(fused_workspace_bytes(N, H, W, kFusedSlabD, &q0)));
    float* den = reinterpret_cast<float*>(reinterpret_cast<char*>(mins) + stat_bytes);
    for (int d0 = 0; d0 < g.D; d0 += kFusedSlabD) {
      const msn_ms_params q = slab_params(p, d0, g.D - d0 < kFusedSlabD ? g.D - d0 : kFusedSlabD);
      TRY(launch_ms_fused(d_left, d_right, N, H, W, &q, d_out, mins, base, s, g.D, d0, d0 > 0));
    }
    for (int i = 0; i < N; ++i) {
      float* out = d_out + (size_t)i * 8 * g.D * n;
      TRY(launch_slab_phase_b(out, mins + (size_t)i * 4 * n, (long long)n, g.D, 0, p->cens_sigma, p->ncc_sigma,
                              p->sad_sigma, den + (size_t)i * 4 * n, s));
      TRY(launch_slab_phase_c(out, mins + (size_t)i * 4 * n, den + (size_t)i * 4 * n, (long long)n, g.D, 0,
                              p->cens_sigma, p->ncc_sigma, p->sad_sigma, s));
    }
    return 0;
  }
  GenericWs ws;
  ws.carve(base, g, p);
  for (int i = 0; i < N; ++i) {
    float* out = d_out + (size_t)i * g.C * g.Dn * n;
    TRY(generic_phase_a(d_left + (size_t)i * H * W, d_right + (size_t)i * H * W, g, p, ws, nullptr, out, ws.mins, s));
    TRY(launch_slab_phase_b(out, ws.mins, (long long)n, g.Dn, p->lr, p->cens_sigma, p->ncc_sigma, p->sad_sigma,
                            ws.den, s));
    TRY(launch_slab_phase_c(out, ws.mins, ws.den, (long long)n, g.Dn, p->lr, p->cens_sigma, p->ncc_sigma,
                            p->sad_sigma, s));
  }
  return 0;
}

int msn_ms_features_bf16_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W, const msn_ms_params* p,
                             void* d_out_bf16, void* d_workspace, size_t workspace_bytes, void* stream) {
  Geometry g;
  TRY(resolve(p, N, H, W, &g, "ms_features_bf16"));
  MSN_REQUIRE(d_left && d_right && d_out_bf16 && d_workspace, "ms_features_bf16: null pointer argument");
  MSN_REQUIRE(use_fused(p, g, W) && !p->lr && g.d_begin == 0 && g.Dn == g.D,
              "ms_features_bf16: the bf16 volume comes from the fused kernel (default windows, left view, D <= 448)");
  MSN_REQUIRE(workspace_bytes >= msn_ms_features_workspace_bytes(N, H, W, p), "ms_features_bf16: workspace too small");
  char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
  return launch_ms_fused(d_left, d_right, N, H, W, p, reinterpret_cast<float*>(d_out_bf16), nullptr, base,
                         as_stream(stream), 0, 0, 0, nullptr, nullptr, true);
}

int msn_ms_features_host(const uint8_t* left, const uint8_t* right, int N, int H, int W, const msn_ms_params* p,
                         float* out_ncdhw) {
  Geometry g;
  TRY(resolve(p, N, H, W, &g, "ms_features"));
  MSN_REQUIRE(left && right && out_ncdhw, "ms_features: null pointer argument");
  HOST_BEGIN();
  const size_t npx = (size_t)N * H * W, nout = (size_t)N * g.C * g.Dn * g.h * g.w;
  uint8_t *dl, *dr;
  float* dout;
  void* ws;
  const size_t wsb = msn_ms_features_workspace_bytes(N, H, W, p);
  TRY(ctx.upload(&dl, left, npx)); TRY(ctx.upload(&dr, right, npx));
  TRY(ctx.alloc((void**)&dout, nout * 4));
  TRY(ctx.alloc(&ws, wsb));
  TRY(msn_ms_features_dev(dl, dr, N, H, W, p, dout, ws, wsb, ctx.stream));
  TRY(ctx.download(out_ncdhw, dout, nout));
  return ctx.finish();
}

int msn_profile_enable(int on) { return profile_enable(on); }
int msn_profile_read(double* prep_ms, double* sadsob_ms, double* fused_ms, int* calls) {
  return profile_read(prep_ms, sadsob_ms, fused_ms, calls);
}

// slab phases (multi-GPU disparity sharding); workspace sized by
// msn_ms_slab_workspace_bytes for the slab in p.
static bool slab_fused(const msn_ms_params* p, const Geometry& g, int W) {
  return !p->lr && use_fused(p, g, W);   // (the slab path provides the left view only)
}

size_t msn_ms_slab_workspace_bytes(int N, int H, int W, const msn_ms_params* p) {
  Geometry g;
  if (resolve(p, N, H, W, &g, "ms_slab_workspace_bytes")) return 0;
  if (slab_fused(p, g, W)) {
    // sized for the sub-slab with the largest disparity offset and a full count (see phase A)
    const int dn = g.Dn < kFusedSlabD ? g.Dn : kFusedSlabD;
    const msn_ms_params q = slab_params(p, g.d_begin + g.Dn - dn, dn);
    return fused_workspace_bytes(N, H, W, dn, &q) + 256;
  }
  GenericWs ws;
  ws.carve(nullptr, g, p);
  return ws.total + 256;
}

int msn_ms_slab_phase_a_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                            const msn_ms_params* p, const float* d_first4, float* d_out, float* d_min,
                            void* d_workspace, size_t workspace_bytes, void* stream) {
  Geometry g;
  TRY(resolve(p, N, H, W, &g, "ms_slab_phase_a"));
  MSN_REQUIRE(!g.band, "ms_slab_phase_a: row bands are served by msn_ms_slab_fused_dev");
  MSN_REQUIRE(d_left && d_right && d_out && d_min && d_workspace, "ms_slab_phase_a: null pointer argument");
  MSN_REQUIRE(workspace_bytes >= msn_ms_slab_workspace_bytes(N, H, W, p), "ms_slab_phase_a: workspace too small");
  cudaStream_t s = as_stream(stream);
  char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
  // default windows, left view: phase 1 of the fused kernel computes the slab's costs on chip
  if (slab_fused(p, g, W)) {
    // sub-slabs of at most kFusedSlabD disparities keep the launch on the TMA instantiations
    for (int o = 0; o < g.Dn; o += kFusedSlabD) {
      const msn_ms_params q = slab_params(p, g.d_begin + o, g.Dn - o < kFusedSlabD ? g.Dn - o : kFusedSlabD);
      TRY(launch_ms_fused(d_left, d_right, N, H, W, &q, d_out, d_min, base, s, g.Dn, o, o > 0));
    }
    return 0;
  }
  GenericWs ws;
  ws.carve(base, g, p);
  const size_t n = (size_t)g.h * g.w;
  const int nm = p->lr ? 8 : 4;
  for (int i = 0; i < N; ++i)
    TRY(generic_phase_a(d_left + (size_t)i * H * W, d_right + (size_t)i * H * W, g, p, ws,
                        d_first4 ? d_first4 + (size_t)i * 4 : nullptr, d_out + (size_t)i * g.C * g.Dn * n,
                        d_min + (size_t)i * nm * n, s));
  return 0;
}

// the fused exchange serves the default windows, the left view and sub-slabs the fused kernel can park
static bool exchange_ok(const msn_ms_params* p, const Geometry& g, int W, int subs) {
  if (p->lr || subs < 1 || g.Dn % subs != 0) return false;
  const int ds = g.Dn / subs;
  return fused_supported(p, ds) && sadsob_fast_pitch(W + 35) > 0 && !force_generic();
}

size_t msn_ms_slab_exchange_bytes(int N, int H, int W, const msn_ms_params* p, int world, int subs) {
  Geometry g;
  if (resolve(p, N, H, W, &g, "ms_slab_exchange_bytes")) return 0;
  if (subs < 1) subs = 1;
  if (world < 1 || world > 8) { set_error("ms_slab_exchange_bytes: world %d not in 1..8", world); return 0; }
  if (!exchange_ok(p, g, W, subs)) {
    set_error("ms_slab_exchange_bytes: the fused exchange needs the default windows, the left view and %d equal "
              "sub-slabs of at most 448 disparities (slab: %d)", subs, g.Dn);
    return 0;
  }
  return fused_exchange_bytes(N, H, W, p, world * subs);
}

size_t msn_ms_slab_fused_workspace_bytes(int N, int H, int W, const msn_ms_params* p) {
  Geometry g;
  if (resolve(p, N, H, W, &g, "ms_slab_fused_workspace_bytes")) return 0;
  return fused_workspace_bytes(N, H, W, g.Dn, p) + 256;
}

int msn_ms_slab_fused_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W, const msn_ms_params* p,
                          const msn_slab_exchange* xchg, float* d_out, int32_t* d_wta_idx, float* d_wta_min1,
                          float* d_wta_min2, void* d_workspace, size_t workspace_bytes, void* stream) {
  Geometry g;
  TRY(resolve(p, N, H, W, &g, "ms_slab_fused"));
  MSN_REQUIRE(d_left && d_right && d_out && d_workspace && xchg, "ms_slab_fused: null pointer argument");
  MSN_REQUIRE(exchange_ok(p, g, W, xchg->subs > 1 ? xchg->subs : 1),
              "ms_slab_fused: needs the default windows, the left view and equal sub-slabs of at most 448 disparities "
              "(use msn_ms_slab_phase_*_dev otherwise)");
  const size_t need = fused_workspace_bytes(N, H, W, g.Dn, p) + 256;
  MSN_REQUIRE(workspace_bytes >= need, "ms_slab_fused: workspace too small (%zu < %zu)", workspace_bytes, need);
  char* base = (char*)(((uintptr_t)d_workspace + 255) & ~(uintptr_t)255);
  const bool want_wta = d_wta_idx || d_wta_min1 || d_wta_min2;
  MSN_REQUIRE(!want_wta || (d_wta_idx && d_wta_min1 && d_wta_min2), "ms_slab_fused: pass all three WTA planes or none");
  const FusedWta wta{d_wta_idx, d_wta_min1, d_wta_min2};
  return launch_ms_fused(d_left, d_right, N, H, W, p, d_out, nullptr, base, as_stream(stream), g.Dn, 0, 0, xchg, &wta);
}

int msn_wta_merge_dev(const int32_t* d_idx_parts, const float* d_min1_parts, const float* d_min2_parts, int parts,
                      long long n, int32_t* d_idx, float* d_min1, float* d_min2, void* stream) {
  MSN_REQUIRE(d_idx_parts && d_min1_parts && d_min2_parts && d_idx && d_min1 && d_min2, "wta_merge: null pointer argument");
  MSN_REQUIRE(parts >= 1 && n >= 0, "wta_merge: bad shape");
  return launch_wta_merge(d_idx_parts, d_min1_parts, d_min2_parts, parts, n, d_idx, d_min1, d_min2, as_stream(stream));
}

int msn_set_aml_exact(int on) {
  g_aml_exact = on ? 1 : 0;
  return 0;
}
int msn_get_aml_exact(void) { return g_aml_exact; }

int msn_peer_alloc(size_t bytes, void** d_ptr) {
  MSN_REQUIRE(d_ptr && bytes > 0, "peer_alloc: bad argument");
  MSN_CUDA_OK(cudaMalloc(d_ptr, bytes));
  MSN_CUDA_OK(cudaMemset(*d_ptr, 0, bytes));
  MSN_CUDA_OK(cudaDeviceSynchronize());
  return 0;
}
int msn_peer_free(void* d_ptr) {
  if (d_ptr) MSN_CUDA_OK(cudaFree(d_ptr));
  return 0;
}
int msn_peer_export(void* d_ptr, unsigned char handle64[64]) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  MSN_REQUIRE(d_ptr && handle64, "peer_export: null pointer argument");
  cudaIpcMemHandle_t h;
  MSN_CUDA_OK(cudaIpcGetMemHandle(&h, d_ptr));
  memcpy(handle64, &h, 64);
  return 0;
}
int msn_peer_open(const unsigned char handle64[64], void** d_ptr) {
  MSN_REQUIRE(d_ptr && handle64, "peer_open: null pointer argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  MSN_CUDA_OK(cudaIpcOpenMemHandle(d_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
int msn_peer_close(void* d_ptr) {
  if (d_ptr) MSN_CUDA_OK(cudaIpcCloseMemHandle(d_ptr));
  return 0;
}

int msn_ms_slab_phase_b_dev(const float* d_out, const float* d_min, int N, int h, int w, const msn_ms_params* p,
                            float* d_den, void* stream) {
  MSN_REQUIRE(p && d_out && d_min && d_den, "ms_slab_phase_b: null pointer argument");
  MSN_REQUIRE(N >= 0 && h >= 1 && w >= 1, "ms_slab_phase_b: bad shape");
  const int Dn = p->d_count > 0 ? p->d_count : p->ndisp, C = p->lr ? 16 : 8, nm = p->lr ? 8 : 4;
  const size_t n = (size_t)h * w;
  for (int i = 0; i < N; ++i)
    TRY(launch_slab_phase_b(d_out + (size_t)i * C * Dn * n, d_min + (size_t)i * nm * n, (long long)n, Dn, p->lr,
                            p->cens_sigma, p->ncc_sigma, p->sad_sigma, d_den + (size_t)i * nm * n,
                            as_stream(stream)));
  return 0;
}

int msn_ms_slab_phase_c_dev(float* d_out, const float* d_min, const float* d_den, int N, int h, int w,
                            const msn_ms_params* p, void* stream) {
  MSN_REQUIRE(p && d_out && d_min && d_den, "ms_slab_phase_c: null pointer argument");
  MSN_REQUIRE(N >= 0 && h >= 1 && w >= 1, "ms_slab_phase_c: bad shape");
  const int Dn = p->d_count > 0 ? p->d_count : p->ndisp, C = p->lr ? 16 : 8, nm = p->lr ? 8 : 4;
  const size_t n = (size_t)h * w;
  for (int i = 0; i < N; ++i)
    TRY(launch_slab_phase_c(d_out + (size_t)i * C * Dn * n, d_min + (size_t)i * nm * n, d_den + (size_t)i * nm * n,
                            (long long)n, Dn, p->lr, p->cens_sigma, p->ncc_sigma, p->sad_sigma, as_stream(stream)));
  return 0;
}

// ------------------------------------------- soft-argmin / WTA / volumes --
int msn_soft_argmin_dev(const float* d_logits, int N, int D, int H, int W, float* d_disp, void* stream) {
  MSN_REQUIRE(d_logits && d_disp, "soft_argmin: null pointer argument");
  return launch_soft_argmin(d_logits, N, D, H, W, 0, 0, d_disp, as_stream(stream));
}

int msn_expect_disp_dev(const float* d_prob, int N, int D, int H, int W, float* d_disp, void* stream) {
  MSN_REQUIRE(d_prob && d_disp, "expect_disp: null pointer argument");
  return launch_soft_argmin(d_prob, N, D, H, W, 0, 2, d_disp, as_stream(stream));
}

int msn_soft_argmin_backward_dev(const float* d_logits, const float* d_disp, const float* d_grad_disp, int N, int D,
                                 int H, int W, float* d_grad_logits, void* stream) {
  MSN_REQUIRE(d_logits && d_disp && d_grad_disp && d_grad_logits, "soft_argmin_backward: null pointer argument");
  return launch_soft_argmin_bwd(d_logits, d_disp, d_grad_disp, N, D, H, W, d_grad_logits, as_stream(stream));
}

int msn_soft_argmin_host(const float* logits, int N, int D, int H, int W, float* disp) {
  MSN_REQUIRE(logits && disp, "soft_argmin: null pointer argument");
  MSN_REQUIRE(N >= 0 && D >= 1 && H >= 0 && W >= 0, "soft_argmin: bad shape");
  HOST_BEGIN();
  float *din, *dout;
  TRY(ctx.upload(&din, logits, (size_t)N * D * H * W));
  TRY(ctx.alloc((void**)&dout, (size_t)N * H * W * 4));
  TRY(msn_soft_argmin_dev(din, N, D, H, W, dout, ctx.stream));
  TRY(ctx.download(disp, dout, (size_t)N * H * W));
  return ctx.finish();
}

int msn_soft_argmin_partial_dev(const float* d_logits, int N, int D, int H, int W, int d_begin, float* d_part,
                                void* stream) {
  MSN_REQUIRE(d_logits && d_part, "soft_argmin_partial: null pointer argument");
  return launch_soft_argmin(d_logits, N, D, H, W, d_begin, 1, d_part, as_stream(stream));
}

int msn_soft_argmin_merge_dev(const float* d_parts, int parts, int N, int H, int W, float* d_disp, void* stream) {
  MSN_REQUIRE(d_parts && d_disp, "soft_argmin_merge: null pointer argument");
  return launch_soft_argmin_merge(d_parts, parts, N, H, W, d_disp, as_stream(stream));
}

int msn_wta_dev(const float* d_cost, long long n, int D, int layout, int32_t* d_argmin, float* d_min1,
                float* d_min2, void* stream) {
  MSN_REQUIRE(d_cost, "wta: null cost pointer");
  MSN_REQUIRE(n >= 0, "wta: bad pixel count");
  return launch_wta(d_cost, n, D, layout, 0, d_argmin, d_min1, d_min2, nullptr, as_stream(stream));
}

int msn_wta_host(const float* cost, long long n, int D, int layout, int32_t* argmin, float* min1, float* min2) {
  MSN_REQUIRE(cost, "wta: null cost pointer");
  MSN_REQUIRE(n >= 0 && D >= 1, "wta: bad shape");
  HOST_BEGIN();
  float *dc, *m1, *m2;
  int32_t* am;
  TRY(ctx.upload(&dc, cost, (size_t)n * D));
  TRY(ctx.alloc((void**)&am, (size_t)n * 4)); TRY(ctx.alloc((void**)&m1, (size_t)n * 4));
  TRY(ctx.alloc((void**)&m2, (size_t)n * 4));
  TRY(msn_wta_dev(dc, n, D, layout, am, m1, m2, ctx.stream));
  if (argmin) TRY(ctx.download(argmin, am, (size_t)n));
  if (min1) TRY(ctx.download(min1, m1, (size_t)n));
  if (min2) TRY(ctx.download(min2, m2, (size_t)n));
  return ctx.finish();
}

int msn_wta_keys_dev(const float* d_cost, long long n, int D, int layout, int d_begin, long long* d_keys,
                     void* stream) {
  MSN_REQUIRE(d_cost && d_keys, "wta_keys: null pointer argument");
  return launch_wta(d_cost, n, D, layout, d_begin, nullptr, nullptr, nullptr, d_keys, as_stream(stream));
}

int msn_wta_unpack_dev(const long long* d_keys, long long n, int32_t* d_argmin, float* d_min1, void* stream) {
  MSN_REQUIRE(d_keys, "wta_unpack: null pointer argument");
  return launch_wta_unpack(d_keys, n, d_argmin, d_min1, as_stream(stream));
}

int msn_pkrn_conf_dev(const float* d_min1, const float* d_min2, long long n, float e, float* d_conf, void* stream) {
  MSN_REQUIRE(d_min1 && d_min2 && d_conf, "pkrn_conf: null pointer argument");
  return launch_pkrn_conf(d_min1, d_min2, n, e, d_conf, as_stream(stream));
}

int msn_lrc_dev(const float* d_cost_hwd, int H, int W, int D, int thresh, int32_t* d_dl, int32_t* d_dr,
                uint8_t* d_mask, void* stream) {
  MSN_REQUIRE(d_cost_hwd && d_dl && d_dr && d_mask, "lrc: null pointer argument");
  MSN_REQUIRE(H >= 1 && W >= 1 && D >= 1, "lrc: bad shape");
  return launch_lrc(d_cost_hwd, H, W, D, thresh, d_dl, d_dr, d_mask, as_stream(stream));
}

int msn_lrc_host(const float* cost_hwd, int H, int W, int D, int thresh, int32_t* dl, int32_t* dr, uint8_t* mask) {
  MSN_REQUIRE(cost_hwd && dl && dr && mask, "lrc: null pointer argument");
  MSN_REQUIRE(H >= 1 && W >= 1 && D >= 1, "lrc: bad shape");
  HOST_BEGIN();
  const size_t n = (size_t)H * W;
  float* dc;
  int32_t *ddl, *ddr;
  uint8_t* dm;
  TRY(ctx.upload(&dc, cost_hwd, n * D));
  TRY(ctx.alloc((void**)&ddl, n * 4)); TRY(ctx.alloc((void**)&ddr, n * 4)); TRY(ctx.alloc((void**)&dm, n));
  TRY(msn_lrc_dev(dc, H, W, D, thresh, ddl, ddr, dm, ctx.stream));
  TRY(ctx.download(dl, ddl, n)); TRY(ctx.download(dr, ddr, n)); TRY(ctx.download(mask, dm, n));
  return ctx.finish();
}

int msn_concat_volume_dev(const float* d_fl, const float* d_fr, int N, int C, int H, int W, int D, float* d_vol,
                          void* stream) {
  MSN_REQUIRE(d_fl && d_fr && d_vol, "concat_volume: null pointer argument");
  return launch_shift_volume(d_fl, d_fr, N, C, H, W, D, false, d_vol, as_stream(stream));
}

int msn_diff_volume_dev(const float* d_fl, const float* d_fr, int N, int C, int H, int W, int D, float* d_vol,
                        void* stream) {
  MSN_REQUIRE(d_fl && d_fr && d_vol, "diff_volume: null pointer argument");
  return launch_shift_volume(d_fl, d_fr, N, C, H, W, D, true, d_vol, as_stream(stream));
}

int msn_concat_volume_backward_dev(const float* d_grad_vol, int N, int C, int H, int W, int D, float* d_grad_fl,
                                   float* d_grad_fr, void* stream) {
  MSN_REQUIRE(d_grad_vol, "concat_volume_backward: null pointer argument");
  MSN_REQUIRE(d_grad_fl || d_grad_fr, "concat_volume_backward: grad_fl and grad_fr are both NULL");
  return launch_shift_volume_bwd(d_grad_vol, N, C, H, W, D, false, d_grad_fl, d_grad_fr, as_stream(stream));
}

int msn_diff_volume_backward_dev(const float* d_grad_vol, int N, int C, int H, int W, int D, float* d_grad_fl,
                                 float* d_grad_fr, void* stream) {
  MSN_REQUIRE(d_grad_vol, "diff_volume_backward: null pointer argument");
  MSN_REQUIRE(d_grad_fl || d_grad_fr, "diff_volume_backward: grad_fl and grad_fr are both NULL");
  return launch_shift_volume_bwd(d_grad_vol, N, C, H, W, D, true, d_grad_fl, d_grad_fr, as_stream(stream));
}

}  // extern "C"
