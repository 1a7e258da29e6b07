/*
 * fdn_b200.h -- C ABI of libfdn_b200.so: the B200 (sm_100a) implementation of FlowDenoising's hot path,
 * the optical-flow-driven separable Gaussian filter (filter_along_Z/Y/X).
 *
 * Every entry point is extern "C", takes plain pointers/sizes (device pointers are raw CUdeviceptr-style
 * addresses; no torch or C++ types cross this boundary), returns an int status (0 = FDN_OK) and never
 * throws. fdn_last_error() returns a thread-local description of the last failure.
 * All device work is enqueued on the caller's stream (`stream` is a cudaStream_t passed as void*; NULL =
 * the legacy default stream) and is asynchronous with respect to the host unless stated otherwise.
 *
 * Reference interfaces these replace (file:line in /root/reference):
 *   fdn_filter_axis      <- GaussianDenoising.filter_along_{Z,Y,X}  src/flowdenoising.py:175-283 (whole pass:
 *                           _chunk :160-173, no-OF _slice :133-158, OF _slice :306-373)
 *   fdn_farneback        <- get_flow_with_prev_flow / get_flow_without_prev_flow  :65-114
 *                           (= cv2.calcOpticalFlowFarneback call sites :69-79, :98-108)
 *   fdn_warp_accumulate  <- warp_slice :55-63 (= cv2.remap :60-62) fused with `tmp_slice += ... * kernel[i]` :316
 *   fdn_gaussian_kernel  <- get_gaussian_kernel :34-45
 *   stage entry points (fdn_pyramid_level, fdn_polyexp, fdn_flow_iteration, ...) expose the four north-star
 *   stages one by one so that parity tests can address them (SURVEY.md §8b).
 *
 * Data layouts (all float32 unless noted):
 *   volume view   : element (s, y, x) at base[s*slice_stride + y*row_stride + x]; strides in ELEMENTS; x is
 *                   always contiguous. Z pass on [Z][Y][X]: slice_stride=Y*X,row_stride=X; Y pass:
 *                   slice_stride=X,row_stride=Y*X; X pass runs on the [Z][X][Y] transpose (fdn_transpose_yx).
 *   image         : dense row-major (h, w)
 *   flow          : dense (h, w, 2), x component first  (same as OpenCV CV_32FC2)
 *   R (polyexp)   : per image [h*w] float4 holding channels 0-3 followed by [h*w] float holding channel 4 (padded
 *                   to 16 bytes; fdn_polyexp_floats(h, w) floats in total), channel order as OpenCV
 *                   (R0=d/dy, R1=d/dx, R2=yy, R3=xx, R4=xy)  -- NOT OpenCV's interleaved (h, w, 5)
 */
#ifndef FDN_B200_H
#define FDN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FDN_OK 0
#define FDN_ERR_INVALID 1   /* bad argument */
#define FDN_ERR_CUDA 2      /* a CUDA runtime call or kernel launch failed */
#define FDN_ERR_WORKSPACE 3 /* workspace too small */

#define FDN_MAX_LEVELS 16

/* fdn_of_params.flags: OpenCV's OPTFLOW_FARNEBACK_GAUSSIAN (same value). The matrices of the displacement update are
 * smoothed by a separable Gaussian window (2m+1 taps, m = winsize/2, sigma = 0.3 m) instead of the winsize x winsize
 * box mean: a different, usually more accurate flow estimate, not a speed switch. winsize 2m and 2m+1 are the same
 * window in this mode. */
#define FDN_OF_FARNEBACK_GAUSSIAN 256

/* Farneback parameters (reference constants src/flowdenoising.py:47-53; pyr_scale is fixed at 0.5 like :73) */
typedef struct fdn_of_params {
    int levels;          /* -l  (OF_LEVELS = 3): EXTRA pyramid levels, cropped while min(W,H)*0.5^k >= 32 */
    int winsize;         /* -w  (OF_WINDOW_SIZE = 5) */
    int iterations;      /* OF_ITERS = 3 */
    int poly_n;          /* OF_POLY_N = 5 (5 or 7 as in OpenCV) */
    double poly_sigma;   /* OF_POLY_SIGMA = 1.2 */
    int use_prev_flow;   /* 1: chain flows (get_flow_with_prev_flow), 0: --recompute_flow */
    int flags;           /* 0 (box window) or FDN_OF_FARNEBACK_GAUSSIAN; any other bit is rejected */
} fdn_of_params;

/* Geometry of one volume view of a pass. The view holds n_in slices of (H, W). Output slice s (0..n_out-1)
 * is centred on input slice s+halo; its neighbours are input slices s+halo+d, d in [-r, r]. If periodic != 0
 * every input index wraps modulo n_in exactly like `% self.vol.shape[0]` in src/flowdenoising.py:312 (whole axis
 * resident: halo = 0, n_out = n_in; a WINDOW of the axis: halo = first output slice, n_out <= n_in, d_out pointing at
 * that slice -- the plugin runs the first / last slices of a pass as their own call so that the upload / download
 * of the rest overlaps them); otherwise the caller guarantees halo >= r slices on both sides (multi-GPU slabs carry
 * the periodic halo explicitly). */
typedef struct fdn_view {
    int n_in, n_out, halo, periodic;
    int H, W;
    int64_t in_slice_stride, in_row_stride;    /* input view strides (elements) */
    int64_t out_slice_stride, out_row_stride;  /* output view strides; out index s is the OUTPUT slice number */
} fdn_view;

/* ---- library / error handling ---- */
int fdn_version(void);
const char* fdn_last_error(void);
/* Number of this library's kernel launches since the last reset (bench.py "gpu_launches"). */
int64_t fdn_launch_count(void);
void fdn_reset_launch_count(void);
/* Launch log (tests): while enabled, the name of every kernel this library launches is recorded in order, so that a
 * test can assert which specialisation a pyramid level / window size actually runs. Enabling clears the log. */
void fdn_launch_log_enable(int on);
int fdn_launch_log_count(void);
const char* fdn_launch_log_name(int i);
/* Progress feedback for the reference's feedback() thread (src/flowdenoising.py:139-140, :292-295): thousandths of
 * output slices the device has finished since the last reset, all passes of this process together. A pass advances it
 * after every chain step (host functions in the stream), so it follows execution, not enqueueing. fdn_gauss_rows
 * (slices are not its unit) does not touch it. */
int64_t fdn_progress_milli(void);
void fdn_progress_reset(void);

/* Optional per-kernel timing: when enabled every kernel launch is bracketed by CUDA events on the launching
 * stream. fdn_profile_read(id) synchronises on them and returns, for kernel `id` (0 <= id <
 * fdn_profile_kernel_count()), the summed device time, the number of launches and the summed ALGORITHMIC bytes
 * (SURVEY.md §8d: what the stage must read + write once) since fdn_profile_reset(). */
void fdn_profile_enable(int on);
void fdn_profile_reset(void);
int fdn_profile_kernel_count(void);
const char* fdn_profile_kernel_name(int id);
int fdn_profile_read(int id, double* total_ms, int64_t* launches, double* algorithmic_bytes);
/* The individual launches behind fdn_profile_read, in launch order: kernel id, batch size and image size of the
 * launch (0 where a launcher does not record them), device time, algorithmic bytes. Any output may be NULL. */
int fdn_profile_record_count(void);
int fdn_profile_record(int i, int* id, int* n, int* h, int* w, double* ms, double* algorithmic_bytes);

/* ---- host-side helpers ---- */
/* get_gaussian_kernel (src/flowdenoising.py:34-45): writes 2*int(4*sigma+0.5)+1 float64 taps, returns the
 * count (or -needed if cap is too small). */
int fdn_gaussian_kernel(double sigma, double* taps, int cap);
/* Pyramid geometry (OpenCV level cropping, SURVEY App. A.0): returns the number of EXTRA levels run (nl) and
 * fills hs/ws/ksz/sigma[0..nl]. Any output pointer may be NULL. */
int fdn_level_geometry(int H, int W, int levels, int* hs, int* ws, int* ksz, double* sigma);

/* ---- whole pass (the hot path) ---- */
/* Bytes of device workspace fdn_filter_axis needs for this view when it processes `chunk` output slices at a
 * time (chunk <= 0: all n_out at once). */
size_t fdn_workspace_bytes(const fdn_view* view, int klen, const fdn_of_params* of, int chunk);
/* One pass along the view's slice axis: out[s] = sum_i kernel[i] * warp(in[s+halo+i-r], flow_i) with the
 * reference's chain order and per-tap float32 rounding (src/flowdenoising.py:306-327); `of == NULL` selects
 * the no-OF path (:133-140). d_in and d_out must not overlap. kernel: klen float64 taps on the HOST. */
int fdn_filter_axis(const float* d_in, float* d_out, const fdn_view* view, const double* kernel, int klen,
                    const fdn_of_params* of, int chunk, void* d_workspace, size_t workspace_bytes, void* stream);

/* No-OF pass only, selectable arithmetic: exact != 0 reproduces NumPy's per-tap
 * float32(float64(acc) + float64(v)*k) bit for bit; exact == 0 uses float32 FMA (<= ~2 ulp, HBM-bound). */
int fdn_gauss_axis(const float* d_in, float* d_out, const fdn_view* view, const double* kernel, int klen,
                   int exact, void* stream);
/* Plain separable Gaussian along the contiguous x axis of a dense [n][W] array (X pass without transposes),
 * periodic wrap. */
int fdn_gauss_rows(const float* d_in, float* d_out, int64_t n_rows, int W, const double* kernel, int klen,
                   int exact, void* stream);
/* Batched 2-D transpose of the last two axes: in [n][A][B] -> out [n][B][A]. */
int fdn_transpose_yx(const float* d_in, float* d_out, int n, int A, int B, void* stream);

/* ---- typed volumes: the reference's integer semantics (SURVEY App. B Q3) ----
 * An integer volume keeps its dtype through a pass in the reference: cv2.remap of an integer neighbour returns an
 * integer image (OpenCV's integer rounding: fixed point for 8U, float32 weights + rint + saturation for 16U/16S), the
 * taps accumulate in float32 exactly as for float32 volumes, and the store into the integer result truncates toward
 * zero. These entry points run that on device volumes of the given element type (d_in / d_out: T elements, strides
 * in elements). FDN_DTYPE_F32 forwards to the float32 entry points above. Rejected with FDN_ERR_INVALID: an unknown
 * dtype, int8 with optical flow (cv2.remap rejects int8), and exact == 0 for an integer dtype. */
#define FDN_DTYPE_F32 0
#define FDN_DTYPE_U8 1
#define FDN_DTYPE_I8 2
#define FDN_DTYPE_U16 3
#define FDN_DTYPE_I16 4
/* workspace of fdn_filter_axis_typed (0 on error, and for of == NULL) */
size_t fdn_workspace_bytes_typed(const fdn_view* view, int klen, const fdn_of_params* of, int chunk, int dtype);
/* fdn_filter_axis on a typed volume; of == NULL: the exact no-OF pass */
int fdn_filter_axis_typed(const void* d_in, void* d_out, int dtype, const fdn_view* view, const double* kernel, int klen,
                          const fdn_of_params* of, int chunk, void* d_workspace, size_t workspace_bytes, void* stream);
int fdn_gauss_axis_typed(const void* d_in, void* d_out, int dtype, const fdn_view* view, const double* kernel, int klen,
                         int exact, void* stream);
int fdn_gauss_rows_typed(const void* d_in, void* d_out, int dtype, int64_t n_rows, int W, const double* kernel, int klen,
                         int exact, void* stream);
int fdn_transpose_yx_typed(const void* d_in, void* d_out, int dtype, int n, int A, int B, void* stream);
/* Stage entry point: cv2.remap(src, flow + grid, INTER_LINEAR, BORDER_REPLICATE) of n dense (H, W) images of the
 * dtype; flow (n, H, W, 2) float32. */
int fdn_remap_typed(const void* d_src, const float* d_flow, void* d_dst, int dtype, int n, int H, int W, void* stream);

/* Strided variants used by the multi-GPU re-slab (flowdenoising_b200/dist.py):
 *   fdn_transpose_strided: out[n*out_sn + b*out_sb + a] = in[n*in_sn + a*in_sa + b]           (a < A, b < B)
 *   fdn_copy3d           : out[a*out_sa + b*out_sb + c] = in[a*in_sa + ((b0+b) mod b_wrap)*in_sb + ((c0+c) mod c_wrap)]
 * (the periodic offsets pack a slab together with its wrap-around halo, src/flowdenoising.py:312 `% shape`). */
int fdn_transpose_strided(const float* d_in, int64_t in_sn, int64_t in_sa, float* d_out, int64_t out_sn, int64_t out_sb,
                          int n, int A, int B, void* stream);
int fdn_copy3d(const float* d_in, int64_t in_sa, int64_t in_sb, int b0, int b_wrap, int c0, int c_wrap, float* d_out,
               int64_t out_sa, int64_t out_sb, int A, int B, int C, void* stream);
/* The same two on elements of any FDN_DTYPE_* (strides and offsets in elements): they move bits, so the signed types
 * share the kernel of their size, and FDN_DTYPE_F32 forwards to the float32 entry points. A re-slab of a typed volume
 * moves 1 or 2 B/voxel. An unknown dtype is rejected with FDN_ERR_INVALID. */
int fdn_transpose_strided_typed(const void* d_in, int dtype, int64_t in_sn, int64_t in_sa, void* d_out, int64_t out_sn,
                                int64_t out_sb, int n, int A, int B, void* stream);
int fdn_copy3d_typed(const void* d_in, int dtype, int64_t in_sa, int64_t in_sb, int b0, int b_wrap, int c0, int c_wrap,
                     void* d_out, int64_t out_sa, int64_t out_sb, int A, int B, int C, void* stream);

/* Pitched copy on a stream (cudaMemcpy2DAsync): `rows` rows of `width_bytes`, direction 0 = host to device, 1 = device
 * to host, 2 = device to device. Plumbing of the plugin's staging: a range of columns of the result volume goes home
 * while the rest of the X pass still runs (the reference's classes own HOST arrays, src/flowdenoising.py:122-127,
 * :285-290). Host memory should be page-locked, otherwise the copy is staged by the driver. */
int fdn_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
                     int direction, void* stream);

/* ---- stage entry points (parity tests; all operate on a batch of `n` dense images) ---- */
/* Stage 1: Gaussian pyramid level: GaussianBlur(full-res, ksz, sigma) then bilinear resize to (h, w).
 * d_tmp: scratch of 2*n*H*W floats. Input images: view-strided (slice_stride/row_stride as in fdn_view). */
int fdn_pyramid_level(const float* d_img, int n, int H, int W, int64_t slice_stride, int64_t row_stride,
                      int ksz, double sigma, int h, int w, float* d_tmp, float* d_out, void* stream);
/* Stage 2: polynomial expansion (h, w) -> R. One R image occupies fdn_polyexp_floats(h, w) floats. */
size_t fdn_polyexp_floats(int h, int w);
int fdn_polyexp(const float* d_img, int n, int h, int w, int poly_n, double poly_sigma, float* d_R, void* stream);
/* Stage 3: one displacement-update iteration: M = UpdateMatrices(R0, R1, flow_in); flow_out =
 * BlurSolve(M, winsize). R0/R1: n images each (fdn_polyexp_floats layout), R1 - R0 a whole number of images;
 * flow_in/out: (n, h, w, 2), must not alias. d_scratch: fdn_flow_iteration_scratch_bytes(n, h, w) bytes (the
 * inter-strip carries of the exact horizontal running sum). */
size_t fdn_flow_iteration_scratch_bytes(int n, int h, int w);
int fdn_flow_iteration(const float* d_R0, const float* d_R1, const float* d_flow_in, float* d_flow_out, int n,
                       int h, int w, int winsize, void* d_scratch, size_t scratch_bytes, void* stream);
/* `iterations` consecutive displacement-update iterations of one level (the `for i < iterations` loop of
 * cv2.calcOpticalFlowFarneback, reached from src/flowdenoising.py:69-79). Iteration i reads rotation buffer i % 3 and
 * writes buffer (i + 1) % 3 of {d_flow, d_tmp1, d_tmp2} (each (n, h, w, 2), distinct); *d_result is the buffer that
 * holds the last output. Up to three iterations run as ONE launch of the warp-specialised kernel. */
int fdn_flow_iterations(const float* d_R0, const float* d_R1, float* d_flow, float* d_tmp1, float* d_tmp2, int n,
                        int h, int w, int winsize, int iterations, void* d_scratch, size_t scratch_bytes,
                        void* stream, float** d_result);
/* The same iterations with the Gaussian window (FDN_OF_FARNEBACK_GAUSSIAN): one launch per iteration, blocks without
 * dependencies on each other, so no scratch. winsize 1..31. */
int fdn_flow_iterations_gaussian(const float* d_R0, const float* d_R1, float* d_flow, float* d_tmp1, float* d_tmp2,
                                 int n, int h, int w, int winsize, int iterations, void* stream, float** d_result);
/* Development / test switch: 1 (default) = warp-specialised k_flow_iter_ws where it applies, 0 = the strip kernel
 * k_flow_iter everywhere (the two are compared bit for bit by tests/test_gpu_stages.py). With the Gaussian window,
 * 1 = the register-ring kernel for winsize 4, 5, 8, 9 and 0 = the shared-memory-ring kernel everywhere (compared bit for
 * bit by tests/test_gpu_gaussian_window.py). Process-wide. */
void fdn_set_flow_iter_variant(int variant);
/* Flow resampling between levels: INTER_AREA down-scale * scale (initial flow, coarsest level) and
 * INTER_LINEAR up-scale * 2 (next finer level). */
int fdn_flow_area_down(const float* d_flow, int n, int H, int W, float* d_out, int h, int w, float scale,
                       void* stream);
int fdn_flow_upsample(const float* d_flow, int n, int h_in, int w_in, float* d_out, int h, int w, void* stream);
/* Whole Farneback for n independent image pairs (prev = target/centre, next = reference/neighbour; dense
 * (n, H, W)); flow (n, H, W, 2) is read as the initial flow when use_prev_flow != 0 and overwritten.
 * Workspace: fdn_farneback_workspace_bytes. (= cv2.calcOpticalFlowFarneback(prev, next, flow, 0.5, ...)) */
size_t fdn_farneback_workspace_bytes(int n, int H, int W, const fdn_of_params* of);
int fdn_farneback(const float* d_prev, const float* d_next, float* d_flow, int n, int H, int W,
                  const fdn_of_params* of, void* d_workspace, size_t workspace_bytes, void* stream);
/* Stage 4: acc = float32(float64(acc) + float64(remap(neigh, flow)) * weight)  for n images; d_flow == NULL
 * means identity warp (the centre tap, src/flowdenoising.py:317). neigh/acc are view-strided. */
int fdn_warp_accumulate(const float* d_neigh, int64_t neigh_slice_stride, int64_t neigh_row_stride,
                        const float* d_flow, double weight, float* d_acc, int64_t acc_slice_stride,
                        int64_t acc_row_stride, int n, int H, int W, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FDN_B200_H */
