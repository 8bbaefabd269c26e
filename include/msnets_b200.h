/* msnets_b200.h -- C ABI of libmsnets_b200.so (hand-written sm_100a CUDA kernels).
 *
 * Drop-in boundary for the matching-space (MS) hot path of ccj5351/MS-Nets.
 * Each entry point names the reference interface it replaces (paths relative to
 * the reference checkout).  Plain pointers and sizes only; no torch / numpy /
 * Boost types.  INTEGRATION.md shows the reference-side stubs that bind these.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from msn_last_error() (thread-local, never NULL).  The reference
 *     functions never validate and never raise (SURVEY.md 8b); this ABI checks
 *     shapes/arguments and fails loudly instead of misreading memory.
 *   - "*_host" entry points take HOST buffers (what the reference's Boost.Python
 *     exports receive from NumPy): inputs are borrowed, outputs are caller-
 *     allocated, the call is synchronous, and all host<->device copies happen
 *     inside it on the device selected by msn_set_device().
 *   - "*_dev" entry points take DEVICE buffers and a cudaStream_t (passed as
 *     void*; NULL = legacy default stream).  They only enqueue work.
 *   - images are uint8, row-major, contiguous [H][W] (pitch == W) unless a pitch
 *     argument says otherwise.  Cost volumes are float32.  "fill" is
 *     2147483648.0f == float(RAND_MAX) (matchers.cpp:65,251,377,462).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point
 *     returns an error.
 */
#ifndef MSNETS_B200_H_
#define MSNETS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MSN_API __attribute__((visibility("default")))
#else
#define MSN_API
#endif

#define MSN_FILL_VALUE 2147483648.0f
#define MSN_ABI_VERSION 1

/* ---------------------------------------------------------------- runtime -- */
MSN_API const char* msn_last_error(void);
MSN_API int msn_abi_version(void);
MSN_API int msn_device_count(int* count);
MSN_API int msn_set_device(int device);
/* replaces initthreads() (matchers.cpp:556-563): the reference returns its
 * OpenMP team size (THREADS_NUM_USED = 8, paramSetting.hpp:11); this returns the
 * SM count of the current device. */
MSN_API int msn_initthreads(int* count);

/* ------------------------------------------------- libmatchers (host API) -- */
/* census(left,right,ndisp,wsize) -> float32 [H][W][D]      matchers.cpp:232-353 */
MSN_API int msn_census_host(const uint8_t* left, const uint8_t* right, int H, int W, int ndisp,
                    int wsize, float* out_hwd);
/* nccNister(left,right,ndisp,wsize) -> float32 [D][H][W]   matchers.cpp:47-228 */
MSN_API int msn_ncc_host(const uint8_t* left, const uint8_t* right, int H, int W, int ndisp, int wsize,
                 float* out_dhw);
/* zsad(left,right,ndisp,wsize) -> float32 [D][H][W]        matchers.cpp:442-512 */
MSN_API int msn_zsad_host(const uint8_t* left, const uint8_t* right, int H, int W, int ndisp, int wsize,
                  float* out_dhw);
/* sobel(img) -> float32 [H][W]                             matchers.cpp:515-554 */
MSN_API int msn_sobel_host(const uint8_t* img, int H, int W, float* out_hw);
/* sadsob(left_f32,right_f32,ndisp,wsize) -> float32 [D][H][W]   matchers.cpp:356-438 */
MSN_API int msn_sadsob_host(const float* left, const float* right, int H, int W, int ndisp, int wsize,
                    float* out_dhw);

/* ---------------------------------------------- libfeatextract (host API) -- */
/* swap_axes: [D][H][W] -> [H][W][D]                        featextract.cpp:49-76 */
MSN_API int msn_swap_axes_host(const float* in_dhw, int D, int H, int W, float* out_hwd);
/* swap_axes_back: [H][W][D] -> [D][H][W]                   featextract.cpp:78-105 */
MSN_API int msn_swap_axes_back_host(const float* in_hwd, int H, int W, int D, float* out_dhw);
/* get_right_cost: res[y][x][d] = c[y][x+d][d] (x < W-d), else c[0]   featextract.cpp:136-172 */
MSN_API int msn_right_cost_host(const float* cost_hwd, int H, int W, int D, float* out_hwd);
/* get_left_cost:  res[y][x][d] = c[y][x-d][d] (x >= d), else c[0]    featextract.cpp:464-499 */
MSN_API int msn_left_cost_host(const float* cost_hwd, int H, int W, int D, float* out_hwd);
/* extract_likelihood(vol[n][D], sigma) -> AML [n][D]       featextract.cpp:415-462 */
MSN_API int msn_aml_host(const float* cost_nd, long long n, int D, float sigma, float* out_nd);
/* extract_ratio(vol[n][D], e) -> (min+e)/(c+e) [n][D]      featextract.cpp:320-356 */
MSN_API int msn_pkrn_host(const float* cost_nd, long long n, int D, float e, float* out_nd);

/* ------------------------------------ cbmv_generator glue (host + device) -- */
/* Parameters of get_costs + extract_features_{left,lr}
 * (cbmv_generator.py:27-79, :258-308, :84-254; defaults :434-462). */
typedef struct msn_ms_params {
  int ndisp;          /* maxdisp handed to the matchers                         */
  int censw, nccw, sadw, sobelw;   /* window sizes (defaults 11, 3, 5, 5)       */
  int board_h;        /* rows cropped top AND bottom      (cbmv_generator.py:73-79) */
  int board_w_left;   /* columns cropped on the left                            */
  int board_w_right;  /* columns cropped on the right (0 = none)                */
  float cens_sigma, ncc_sigma, sad_sigma;  /* AML sigmas 128, 0.02, 20000;      *
                       * the sobel channel uses sad_sigma (cbmv_generator.py:298) */
  int lr;             /* 0: 8 channels (extract_features_left); 1: 16 (.._lr)   */
  int d_begin, d_count; /* disparity slab [d_begin, d_begin+d_count) to produce; *
                       * d_count = 0 means the whole range (single-GPU case)    */
  int row_begin, row_count; /* row band [row_begin, row_begin+row_count) of the CROPPED image to produce  *
                       * (output [N][C][Dp][row_count][w]); row_count = 0 means all rows.  A frame sharded by  *
                       * rows needs no exchange: every matcher is a window, and the SAD-of-Sobel table of a   *
                       * row -- which depends on every row above it -- is still built from row 0.  Served by  *
                       * the fused paths (msn_ms_features_dev with the default windows, msn_ms_slab_fused_dev). */
} msn_ms_params;
MSN_API void msn_ms_params_default(msn_ms_params* p);

/* extract_features_left / _lr from four already cropped [h][w][D] volumes
 * (census, ncc, sobel, sad) -> float32 [8 or 16][D][h][w]   cbmv_generator.py:258-308, :84-254 */
MSN_API int msn_features_from_costs_host(const float* census_hwd, const float* ncc_hwd,
                                 const float* sobel_hwd, const float* sad_hwd, int h, int w, int D,
                                 float cens_sigma, float ncc_sigma, float sad_sigma, int lr,
                                 float* out_cdhw);

/* get_costs + extract_features_* in one call (what generate_test_cbmv chains,
 * cbmv_generator.py:826-843) for N bordered pairs [N][H][W] uint8.
 * Output [N][C][Dp][h][w] float32, C = 8 or 16, h = H-2*board_h,
 * w = W-board_w_left-board_w_right, Dp = d_count (or ndisp). */
MSN_API int msn_ms_features_host(const uint8_t* left, const uint8_t* right, int N, int H, int W,
                         const msn_ms_params* p, float* out_ncdhw);
MSN_API size_t msn_ms_features_workspace_bytes(int N, int H, int W, const msn_ms_params* p);
MSN_API int msn_ms_features_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                        const msn_ms_params* p, float* d_out_ncdhw, void* d_workspace,
                        size_t workspace_bytes, void* stream);

/* The same with the confidence by-products of the fused kernel (default windows, left view, D <= 448): for
 * each of channels 0-3 the winner-take-all disparity with np.argmin's tie rule -- what main_msnet.py:443-448
 * computes on the host from a copy of the whole volume -- plus the smallest and second smallest channel value
 * (second-min / peak-ratio, SURVEY.md 8a row 14), as [N][4][h][w] planes taken from the costs while they
 * are still in shared memory: no extra pass over the volume.  All three pointers or none (NULL). */
MSN_API int msn_ms_features_wta_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                            const msn_ms_params* p, float* d_out_ncdhw, int32_t* d_wta_idx_n4hw,
                            float* d_wta_min1_n4hw, float* d_wta_min2_n4hw, void* d_workspace,
                            size_t workspace_bytes, void* stream);

/* bf16 volume (SURVEY.md 8f-4): the same [N][8][D][h][w] volume with every value rounded to nearest-even
 * bfloat16 inside the fused kernel (default windows, left view, D <= 448) -- half the bytes for a consumer
 * that runs its first Conv3d under bf16 autocast.  Identical to converting the fp32 volume afterwards. */
MSN_API int msn_ms_features_bf16_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                             const msn_ms_params* p, void* d_out_bf16_ncdhw, void* d_workspace,
                             size_t workspace_bytes, void* stream);

/* AML arithmetic mode, process-wide.  0 (default): SFU exponential and reciprocal multiply -- within 2e-6 of the
 * reference (1.2e-5 on rare degenerate rows).  1: the reference's own fp32 operations with glibc's expf replayed
 * bit for bit (featextract.cpp:435-453) -- extract_likelihood and feature channels 4-7 / 12-15 BIT-EXACT, about
 * 6x slower on the fused path (0.78 -> 4.7 ms per config-B pair: the fp64 pipe).  Served by every entry point except msn_ms_slab_fused_dev and
 * msn_ms_features_bf16_dev. */
MSN_API int msn_set_aml_exact(int on);
MSN_API int msn_get_aml_exact(void);

/* Measurement aid for bench.py: when enabled, msn_ms_features_dev brackets the kernels of
 * the fused sequence (prep | sadsob scan | fused volume) with CUDA events on the launch
 * stream; msn_profile_read synchronises, returns the summed milliseconds and the number
 * of calls since the last read, and clears the records. */
MSN_API int msn_profile_enable(int on);
MSN_API int msn_profile_read(double* prep_ms, double* sadsob_ms, double* fused_ms, int* calls);

/* Disparity-slab sharding (SURVEY.md 8e): the AML of a pixel needs min and
 * sum over ALL disparities.  Phase A writes channels 0-3 for the slab, parks
 * the raw costs in channels 4-7 and emits per-pixel slab minima [N][4][h][w];
 * after an all-reduce(min) over ranks, phase B emits partial denominators
 * [N][4][h][w]; after an all-reduce(sum), phase C turns the parked costs into
 * AML values in place.  With one rank the three phases reproduce
 * msn_ms_features_dev. */
MSN_API size_t msn_ms_slab_workspace_bytes(int N, int H, int W, const msn_ms_params* p);
/* d_first4: NULL, or (lr && d_begin > 0 only) device [N][4] floats holding voxel
 * (d=0, y=board_h, x=board_w_left) of the four raw volumes -- the c[0] fill of
 * get_right_cost (featextract.cpp:151), which lives on the rank that owns d = 0. */
MSN_API int msn_ms_slab_phase_a_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                            const msn_ms_params* p, const float* d_first4, float* d_out_ncdhw,
                            float* d_min_n4hw, void* d_workspace, size_t workspace_bytes, void* stream);
MSN_API int msn_ms_slab_phase_b_dev(const float* d_out_ncdhw, const float* d_min_n4hw, int N, int h, int w,
                            const msn_ms_params* p, float* d_den_n4hw, void* stream);
MSN_API int msn_ms_slab_phase_c_dev(float* d_out_ncdhw, const float* d_min_n4hw, const float* d_den_n4hw,
                            int N, int h, int w, const msn_ms_params* p, void* stream);

/* Disparity-slab sharding, fused with its exchange (SURVEY.md 8e; replaces phases A/B/C and the two
 * NCCL all-reduces between them when the slab fits the fused kernel: default windows, left view,
 * d_count / subs <= 448).  Every rank calls this for the SAME pair(s) with its own slab in p->d_begin / d_count;
 * the kernel keeps a tile's costs in shared memory and trades the per-pixel AML minima and partial
 * denominators with the other ranks through their exchange tables -- peer-mapped device memory written
 * over NVLink / NVSwitch -- so the volume is written once (32 B per voxel) and never re-read.
 *   tables[r]  device pointer, valid on THIS device, to rank r's exchange table (tables[rank] = own):
 *              msn_ms_slab_exchange_bytes bytes, zeroed once at allocation, same size on every rank
 *   epoch      > 0, the same on every rank, incremented for every frame (call) by every rank
 * A rank whose peers never arrive traps after ~2 s instead of hanging. */
typedef struct msn_slab_exchange {
  void* tables[8];
  int world;
  int rank;
  unsigned epoch;
  int subs;   /* 0 or 1: none.  > 1: every rank's slab is cut into `subs` equal sub-slabs that run as CTAs of the
               * same launch and trade through the same tables (virtual ranks): slabs wider than the 256
               * disparities a tile can park, on any number of GPUs including one.  Same value on every rank. */
} msn_slab_exchange;
MSN_API size_t msn_ms_slab_exchange_bytes(int N, int H, int W, const msn_ms_params* p, int world, int subs);
MSN_API size_t msn_ms_slab_fused_workspace_bytes(int N, int H, int W, const msn_ms_params* p);
MSN_API int msn_ms_slab_fused_dev(const uint8_t* d_left, const uint8_t* d_right, int N, int H, int W,
                          const msn_ms_params* p, const msn_slab_exchange* xchg, float* d_out_ncdhw,
                          int32_t* d_wta_idx, float* d_wta_min1, float* d_wta_min2, void* d_workspace,
                          size_t workspace_bytes, void* stream);
/* d_wta_*: NULL, or the slab's WTA by-product as [subs][N][4][h][w] planes (absolute disparity indices), to be
 * merged over ranks (all-gather, ranks ascending) and sub-slabs by msn_wta_merge_dev: parts [P][n] ordered by
 * ascending disparity range -> the global (argmin, min, second min) of every pixel. */
MSN_API int msn_wta_merge_dev(const int32_t* d_idx_parts, const float* d_min1_parts, const float* d_min2_parts,
                      int parts, long long n, int32_t* d_idx, float* d_min1, float* d_min2, void* stream);
/* Peer memory for the exchange tables: a zeroed cudaMalloc allocation on the current device, its 64-byte
 * CUDA IPC handle (to be all-gathered by the host side), and the mapping of another process's handle into
 * this one (peer access is enabled by the mapping).  One node only. */
MSN_API int msn_peer_alloc(size_t bytes, void** d_ptr);
MSN_API int msn_peer_free(void* d_ptr);
MSN_API int msn_peer_export(void* d_ptr, unsigned char handle64[64]);
MSN_API int msn_peer_open(const unsigned char handle64[64], void** d_ptr);
MSN_API int msn_peer_close(void* d_ptr);

/* Pre-matching image op on the device (SURVEY.md 8f-2): down_sampling_input (cbmv_generator.py:465-482) =
 * uint8 / 255 -> skimage.transform.rescale(anti_aliasing=True, order 1, mode='constant') -> * 255 -> uint8, i.e.
 * (skimage >= 0.19) scipy.ndimage.gaussian_filter + scipy.ndimage.zoom(grid_mode) + range clip, replayed in
 * scipy's arithmetic so the truncated uint8 result is identical.  N images [N][H][W] -> [N][out_h][out_w].
 * w_rows / w_cols: HOST arrays of 2r+1 normalised Gaussian weights per axis (r < 0: no filtering along that
 * axis), zoom_* = input extent / output extent; the Python mirror evaluates them with NumPy as scipy does. */
MSN_API size_t msn_rescale_workspace_bytes(int N, int H, int W);
MSN_API int msn_rescale_dev(const uint8_t* d_in, int N, int H, int W, int out_h, int out_w, const double* w_rows,
                    int r_rows, const double* w_cols, int r_cols, double zoom_rows, double zoom_cols,
                    uint8_t* d_out, void* d_workspace, size_t workspace_bytes, void* stream);
MSN_API int msn_rescale_host(const uint8_t* in, int N, int H, int W, int out_h, int out_w, const double* w_rows,
                     int r_rows, const double* w_cols, int r_cols, double zoom_rows, double zoom_cols,
                     uint8_t* out);

/* ----------------------------------------------------- device-level pieces -- */
MSN_API int msn_census_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                   float* d_out_hwd, void* stream);
MSN_API int msn_ncc_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                float* d_out_dhw, void* stream);
MSN_API int msn_zsad_dev(const uint8_t* d_left, const uint8_t* d_right, int H, int W, int ndisp, int wsize,
                 float* d_out_dhw, void* stream);
MSN_API int msn_sobel_dev(const uint8_t* d_img, int H, int W, float* d_out_hw, void* stream);
MSN_API int msn_sadsob_dev(const float* d_left, const float* d_right, int H, int W, int ndisp, int wsize,
                   float* d_out_dhw, void* stream);
MSN_API int msn_aml_dev(const float* d_cost_nd, long long n, int D, float sigma, float* d_out_nd, void* stream);
MSN_API int msn_pkrn_dev(const float* d_cost_nd, long long n, int D, float e, float* d_out_nd, void* stream);

/* ---------------------------------------- soft-argmin / WTA / confidence -- */
/* softmax over D + expectation of d: replaces F.softmax + disparityregression
 * (gcnet_3dcnn.py:127-141; duplicates psmnet_3dcnn.py:28-37, basic_convs.py:279-287).
 * logits [N][D][H][W] float32 -> disp [N][H][W] float32. */
MSN_API int msn_soft_argmin_dev(const float* d_logits, int N, int D, int H, int W, float* d_disp, void* stream);
/* disparityregression alone (gcnet_3dcnn.py:132-141): prob [N][D][H][W] already
 * normalised -> sum_d d * prob_d. */
MSN_API int msn_expect_disp_dev(const float* d_prob, int N, int D, int H, int W, float* d_disp, void* stream);
MSN_API int msn_soft_argmin_host(const float* logits, int N, int D, int H, int W, float* disp);
/* Backward of msn_soft_argmin_dev for training through the regression (the reference back-propagates
 * through F.softmax + disparityregression, gcnet_3dcnn.py:127-141):
 * grad_logits[n][d][p] = grad_disp[n][p] * softmax(logits)[n][d][p] * (d - disp[n][p]). */
MSN_API int msn_soft_argmin_backward_dev(const float* d_logits, const float* d_disp, const float* d_grad_disp, int N,
                                 int D, int H, int W, float* d_grad_logits, void* stream);
/* Slab-sharded soft-argmin: per-pixel partial (max, sum e, sum d*e) over the
 * local D slab whose first disparity is d_begin -> [N][3][H][W]; merged by
 * msn_soft_argmin_merge_dev over `parts` gathered partials [parts][N][3][H][W]. */
MSN_API int msn_soft_argmin_partial_dev(const float* d_logits, int N, int D, int H, int W, int d_begin,
                                float* d_part_n3hw, void* stream);
MSN_API int msn_soft_argmin_merge_dev(const float* d_parts, int parts, int N, int H, int W, float* d_disp,
                              void* stream);

/* Winner-take-all over D (np.argmin semantics of main_msnet.py:444-448: first
 * minimal index wins) plus second minimum.  layout: 0 = [n][D] rows (D innermost,
 * the reference's [H][W][D] volumes flattened; warp-shuffle reduction), 1 =
 * [D][n] planes (the [C][D][h][w] feature layout; one thread per pixel).
 * Outputs (any may be NULL): argmin int32 [n], min float [n], second-min float [n]. */
MSN_API int msn_wta_dev(const float* d_cost, long long n, int D, int layout, int32_t* d_argmin, float* d_min1,
                float* d_min2, void* stream);
MSN_API int msn_wta_host(const float* cost, long long n, int D, int layout, int32_t* argmin, float* min1,
                 float* min2);
/* Slab merge key for WTA across ranks: order-preserving 64-bit key
 * (float bits made monotonic) << 32 | (d_begin + d); all-reduce(min) over
 * int64 then msn_wta_unpack_dev. */
MSN_API int msn_wta_keys_dev(const float* d_cost, long long n, int D, int layout, int d_begin,
                     long long* d_keys, void* stream);
MSN_API int msn_wta_unpack_dev(const long long* d_keys, long long n, int32_t* d_argmin, float* d_min1,
                       void* stream);
/* peak-ratio confidence (min1+e)/(min2+e), 0 where min1 is fill (same algebra as
 * featextract.cpp:349 evaluated at the runner-up; no reference caller). */
MSN_API int msn_pkrn_conf_dev(const float* d_min1, const float* d_min2, long long n, float e, float* d_conf,
                      void* stream);
/* Left-right consistency on an [H][W][D] volume (no reference code; definition
 * in oracle/ms_oracle.py:lr_consistency): dL, dR int32 [H][W], mask uint8 [H][W]. */
MSN_API int msn_lrc_dev(const float* d_cost_hwd, int H, int W, int D, int thresh, int32_t* d_dl, int32_t* d_dr,
                uint8_t* d_mask, void* stream);
MSN_API int msn_lrc_host(const float* cost_hwd, int H, int W, int D, int thresh, int32_t* dl, int32_t* dr,
                 uint8_t* mask);

/* -------------------------------------------------- 4D cost-volume builder -- */
/* GC-Net / PSMNet concat volume (the 64-channel input psmnet_3dcnn.py:96 expects;
 * the reference has no builder, SURVEY.md 0.3): fl, fr [N][C][H][W] ->
 * [N][2C][D][H][W]; x < d is zero.  diff: [N][C][D][H][W] = fl - fr(x-d). */
MSN_API int msn_concat_volume_dev(const float* d_fl, const float* d_fr, int N, int C, int H, int W, int D,
                          float* d_vol, void* stream);
MSN_API int msn_diff_volume_dev(const float* d_fl, const float* d_fr, int N, int C, int H, int W, int D,
                        float* d_vol, void* stream);
/* Backward of msn_concat_volume_dev: grad_vol [N][2C][D][H][W] -> grad_fl, grad_fr [N][C][H][W]:
 *   grad_fl[n][c][y][x]  = sum over d = 0 .. min(x, D-1)      of grad_vol[n][c][d][y][x]
 *   grad_fr[n][c][y][x'] = sum over d = 0 .. min(W-1-x', D-1) of grad_vol[n][C+c][d][y][x'+d]
 * Each sum in fp32, d ascending from 0.0f, in one thread (deterministic, no atomics); masked voxels
 * (x < d) never enter a sum, whatever they hold.  Either output may be NULL (not computed); not both.
 * The concat form reads only the half of grad_vol that a non-NULL output needs. */
MSN_API int msn_concat_volume_backward_dev(const float* d_grad_vol, int N, int C, int H, int W, int D,
                                           float* d_grad_fl, float* d_grad_fr, void* stream);
/* Backward of msn_diff_volume_dev: grad_vol [N][C][D][H][W] -> grad_fl, grad_fr [N][C][H][W], the concat
 * sums taken over grad_vol[n][c] for both, grad_fr negated (same rules). */
MSN_API int msn_diff_volume_backward_dev(const float* d_grad_vol, int N, int C, int H, int W, int D,
                                         float* d_grad_fl, float* d_grad_fr, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MSNETS_B200_H_ */
