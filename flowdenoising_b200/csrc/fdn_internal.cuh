// Internal declarations shared by the translation units of libfdn_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>
#include <stdio.h>
#include <type_traits>

#include "fdn_b200.h"

namespace fdn {

// ---- error plumbing (no exceptions across the C ABI) ----
void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;   // (engines on several host threads may launch concurrently)
extern std::atomic<bool> g_launch_log_on;
void launch_log_add(const char* name);    // records the kernel name while the launch log is enabled (tests)

#define FDN_CHECK_ARG(cond, ...)                 \
    do {                                         \
        if (!(cond)) {                           \
            fdn::set_error(__VA_ARGS__);         \
            return FDN_ERR_INVALID;              \
        }                                        \
    } while (0)

#define FDN_CUDA(call)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (call);                                                                \
        if (e_ != cudaSuccess) {                                                                \
            fdn::set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,                 \
                           cudaGetErrorString(e_));                                             \
            return FDN_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

// after every kernel launch
#define FDN_LAUNCHED(name)                                                                      \
    do {                                                                                        \
        ++fdn::g_launches;                                                                      \
        if (fdn::g_launch_log_on.load(std::memory_order_relaxed)) fdn::launch_log_add(name);    \
        cudaError_t e_ = cudaGetLastError();                                                    \
        if (e_ != cudaSuccess) {                                                                \
            fdn::set_error("launch of %s failed at %s:%d: %s", name, __FILE__, __LINE__,        \
                           cudaGetErrorString(e_));                                             \
            return FDN_ERR_CUDA;                                                                \
        }                                                                                       \
    } while (0)

static inline int64_t cdiv(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- optional per-kernel timing with CUDA events on the launching stream (bench.py roofline) ----
enum KernelId {
    K_BLUR_ROWS = 0, K_BLUR_COLS, K_RESIZE_IMG, K_POLYEXP, K_FLOW_ITER, K_FLOW_AREA, K_FLOW_UP, K_WARP_ACC,
    K_GAUSS_AXIS, K_GAUSS_ROWS, K_TRANSPOSE, K_COPY3D, K_FLOW_GAUSS, K_COUNT
};
extern bool g_prof_on;
int prof_begin(int id, double algorithmic_bytes, cudaStream_t st, int n = 0, int h = 0, int w = 0);   // -> record index
void prof_end(int record, cudaStream_t st);
struct ProfScope {
    cudaStream_t st;
    int rec;
    ProfScope(int id, double bytes, cudaStream_t s, int n = 0, int h = 0, int w = 0) : st(s), rec(-1)
    {
        if (g_prof_on) rec = prof_begin(id, bytes, s, n, h, w);
    }
    ~ProfScope() { if (rec >= 0) prof_end(rec, st); }
};

// ---- constants passed by value to kernels ----
struct PolyConsts {
    int n;
    float g[8], xg[8], xxg[8];  // taps k = 0..n (n <= 7)
    double gd[8], xxgd[8];      // (double)g[k], (double)xxg[k]: the horizontal pass multiplies them in float64
    double ig11, ig03, ig33, ig55;
};
void prepare_poly_consts(int n, double sigma, PolyConsts* pc);

#define FDN_MAX_KSZ 159  // Gaussian pyramid smoothing kernel (levels <= 6 -> 159 taps)
struct BlurTaps {
    int ksz;
    float k[FDN_MAX_KSZ];
};
int prepare_blur_taps(int ksz, double sigma, BlurTaps* bt);

// ---- borders along a pass's axis (FDN_BORDER_*, include/fdn_b200.h) ----
// fdn_view.periodic -> the border its periodic indices take (every nonzero value but the three named modes wraps)
static inline int view_border(int periodic)
{
    return (periodic == FDN_BORDER_REFLECT || periodic == FDN_BORDER_MIRROR || periodic == FDN_BORDER_NEAREST)
               ? periodic : FDN_BORDER_WRAP;
}
// slice of an axis of n (1 <= n <= 2^30) that index i maps to under `border`; an index inside [0, n) maps to itself
__host__ __device__ __forceinline__ int border_index(int i, int n, int border)
{
    if ((unsigned)i < (unsigned)n) return i;
    if (border == FDN_BORDER_NEAREST) return i < 0 ? 0 : n - 1;
    if (border == FDN_BORDER_REFLECT || border == FDN_BORDER_MIRROR) {
        if (n == 1) return 0;
        const int p = border == FDN_BORDER_REFLECT ? 2 * n : 2 * n - 2;
        int j = i % p;
        if (j < 0) j += p;
        return j < n ? j : (border == FDN_BORDER_REFLECT ? p - 1 - j : p - j);
    }
    int j = i % n;
    if (j < 0) j += n;
    return j;
}

// Batch addressing of cached per-slice data: image b of a launch lives in slot
//   s = base + b                          (wrap == 0)
//   s = (base + b) mod wrap               (wrap  > 0, border == FDN_BORDER_WRAP)
//   s = border_index(base + b, wrap, border) (wrap > 0, another border)
// A batch may be the concatenation of two runs (the backward and the forward chain of a pass advance together):
// images b >= split continue at base2 + (b - split).
// A run may span several volumes of a batch (fdn_filter_axis_batch): image j of a run belongs to volume j / per, and
// the slot above is taken with the volume-local index j % per; the volume adds vstride to the offset. One volume:
// per = 0x7fffffff, so every index is local. b0 shifts a launch's images (launchers that split over blockIdx.z).
struct SlotMap {
    int base, wrap;
    int split = 0x7fffffff, base2 = 0;
    int per = 0x7fffffff;
    int64_t vstride = 0;
    int b0 = 0;
    int border = FDN_BORDER_WRAP;
    // element (or float) offset of image b's data: slot * stride + volume * vstride
    __host__ __device__ inline int64_t offset(int b, int64_t stride) const
    {
        b += b0;
        const bool first = b < split;
        int j = first ? b : b - split;
        const int g = j / per;
        j -= g * per;
        int s = (first ? base : base2) + j;
        if (wrap > 0) {
            if (border == FDN_BORDER_WRAP) {
                s %= wrap;
                if (s < 0) s += wrap;
            } else {
                s = border_index(s, wrap, border);
            }
        }
        return (int64_t)s * stride + (int64_t)g * vstride;
    }
};

// ---- launchers (each returns an FDN_* status) ----
// Stage 1
// T: float, or an integer element type of a typed volume (each value read as float32, like OpenCV's convertTo)
template <typename T>
int launch_blur_rows(const T* in, int64_t in_ss, int64_t in_rs, SlotMap in_map, float* out, int n, int H, int W,
                     const BlurTaps& bt, cudaStream_t st);
int launch_blur_cols(const float* in, float* out, int n, int H, int W, const BlurTaps& bt, cudaStream_t st);
int launch_resize_linear_img(const float* in, int n, int H, int W, float* out, int64_t out_stride, int h, int w,
                             cudaStream_t st);
// Stage 2
int launch_polyexp(const float* img, int64_t img_stride, float* R, int64_t R_stride, SlotMap R_map, int n, int h,
                   int w, const PolyConsts& pc, cudaStream_t st);
// Stage 3
// floats one polynomial-expansion image occupies: [h*w] float4 (channels 0-3) + [h*w] float (channel 4), padded to 16 B
static inline size_t R_image_floats(int h, int w) { size_t p = (size_t)h * w; return 4 * p + ((p + 3) / 4) * 4; }
// Scratch of the flow iteration (counters, strip-to-strip carries). Every offset depends only on the CAPACITY the
// scratch was sized for (pairs, and the largest strip count and strips x rows over the levels it serves), never on
// the size of an individual launch.
struct FlowScratch {
    char* base;
    size_t bytes;
    int cap_n, H, W;                    // largest level height and width
    int flag_strips;                    // k_flow_iter strips per pair
    int64_t packet_rows, carry_rows;    // strips x rows per pair: k_flow_iter_ws packets, k_flow_iter carries
    size_t off_done, off_flags, off_packets, off_carry;
};
// levels k < nlev of hs[k] x ws[k] pixels (one level: nlev = 1)
size_t flow_iter_scratch_bytes(int cap_n, int nlev, const int* hs, const int* ws);
int flow_scratch_make(void* scratch, size_t bytes, int cap_n, int nlev, const int* hs, const int* ws,
                      FlowScratch* fs);                                                           // layout only
int flow_iter_scratch_init(const FlowScratch& fs, cudaStream_t st);                              // zero-fill
// `iters` Farneback iterations of one pyramid level for n image pairs: cur -> ... rotating through {cur, a, b}
// (iteration i reads bufs[i % 3] and writes bufs[(i + 1) % 3]); *result = the buffer holding the last output.
int launch_flow_level(const float* R, int64_t R_stride, SlotMap map0, SlotMap map1, float* cur, float* a, float* b,
                      int n, int h, int w, int winsize, int iters, const FlowScratch& fs, cudaStream_t st,
                      float** result);
// The same with the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN): one launch per iteration, no scratch.
int launch_flow_level_gauss(const float* R, int64_t R_stride, SlotMap map0, SlotMap map1, float* cur, float* a,
                            float* b, int n, int h, int w, int winsize, int iters, cudaStream_t st, float** result);
// 0: strip kernel k_flow_iter everywhere, 1 (default): warp-specialised k_flow_iter_ws where it applies; with the
// Gaussian window 0 selects the shared-memory-ring kernel for every winsize
void set_flow_iter_variant(int v);
int launch_flow_area_down(const float* flow, int n, int H, int W, float* out, int h, int w, float scale,
                          cudaStream_t st);
int launch_flow_upsample(const float* flow, int n, int hin, int win, float* out, int h, int w, cudaStream_t st);
// Stage 4
int launch_warp_acc(const float* neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float* flow, double weight,
                    float* acc, int64_t a_ss, int64_t a_rs, int n, int H, int W, int first, cudaStream_t st);
// One chain step of both directions: images [0, n) (backward neighbours, flows flow[0..n)) are remapped and
// accumulated into acc (image b at a_map.offset(b, a_ss)) with `weight`; images [n, 2n) (forward neighbours, flows flow[n..2n)) are remapped into
// stash (dense [n][H][W]) for launch_acc_finish. T: element type of the volume and the stash (integer T: OpenCV's
// integer remap, the accumulator stays float32).
template <typename T>
int launch_warp_pair(const T* neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float* flow, double weight,
                     float* acc, int64_t a_ss, int64_t a_rs, SlotMap a_map, T* stash, int n, int H, int W, int first,
                     cudaStream_t st);
// acc = fold over [centre * k[0], stash[0] * k[1], ..., stash[r-1] * k[r]] of f32(f64(acc) + f64(v) * k), in that
// order; have_acc == 0 starts from 0 (no backward taps). float: the result stays in acc (out unused); integer T: the
// float32 result is truncated into out (the reference's `int_vol[z] = tmp_slice`).
template <typename T>
int launch_acc_finish(const T* centre, int64_t c_ss, int64_t c_rs, SlotMap c_map, const T* stash, int r, const double* k,
                      float* acc, int64_t a_ss, int64_t a_rs, SlotMap a_map, T* out, int64_t o_ss, int64_t o_rs,
                      SlotMap o_map, int n, int H, int W, int have_acc, cudaStream_t st);
// cv2.remap of n dense T images (FDN_DTYPE_* other than int8)
template <typename T>
int launch_remap(const T* src, const float* flow, T* dst, int n, int H, int W, cudaStream_t st);
// no-OF
// batch volumes of view v, volume g at in + g * in_bs / out + g * out_bs (elements); v.periodic selects the border
int launch_gauss_axis(const float* in, float* out, const fdn_view& v, const double* k, int klen, int exact,
                      cudaStream_t st, int batch = 1, int64_t in_bs = 0, int64_t out_bs = 0);
// border: FDN_BORDER_* at both ends of every row
int launch_gauss_rows(const float* in, float* out, int64_t rows, int W, const double* k, int klen, int exact,
                      cudaStream_t st, int border = FDN_BORDER_WRAP);
// typed no-OF passes: T in, T out, exact arithmetic only, truncated store
template <typename T>
int launch_gauss_axis_typed(const T* in, T* out, const fdn_view& v, const double* k, int klen, cudaStream_t st);
template <typename T>
int launch_gauss_rows_typed(const T* in, T* out, int64_t rows, int W, const double* k, int klen, cudaStream_t st,
                            int border);
template <typename T>
int launch_transpose(const T* in, T* out, int n, int A, int B, cudaStream_t st);
template <typename T>
int launch_transpose_strided(const T* in, int64_t in_sn, int64_t in_sa, T* out, int64_t out_sn, int64_t out_sb, int n,
                             int A, int B, cudaStream_t st);
template <typename T>
int launch_copy3d(const T* in, int64_t in_sa, int64_t in_sb, int b0, int bw, int c0, int cw, T* out,
                  int64_t out_sa, int64_t out_sb, int A, int B, int C, cudaStream_t st);

#ifdef __CUDACC__
// ---- typed volumes (FDN_DTYPE_*): element range and the reference's truncating store `int_vol[z] = float32_tmp` ----
template <typename T> struct TypeRange;
template <> struct TypeRange<uint8_t> { static constexpr int lo = 0, hi = 255; };
template <> struct TypeRange<int8_t> { static constexpr int lo = -128, hi = 127; };
template <> struct TypeRange<uint16_t> { static constexpr int lo = 0, hi = 65535; };
template <> struct TypeRange<int16_t> { static constexpr int lo = -32768, hi = 32767; };
// float32 -> T toward zero (NumPy's cast; the accumulated values lie in T's range, the clamp only guards rounding)
template <typename T>
__device__ __forceinline__ T store_cast(float a)
{
    if constexpr (std::is_same<T, float>::value) return a;
    else return (T)min(max(__float2int_rz(a), TypeRange<T>::lo), TypeRange<T>::hi);
}
// four consecutive elements (one 4-, 8- or 16-byte access; p aligned to 4 * sizeof(T))
template <typename T> struct __align__(4 * sizeof(T)) Vec4T { T e[4]; };
template <typename T>
__device__ __forceinline__ void load4(const T* p, float* d)
{
    if constexpr (std::is_same<T, float>::value) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(p));
        d[0] = q.x; d[1] = q.y; d[2] = q.z; d[3] = q.w;
    } else {
        const Vec4T<T> q = *reinterpret_cast<const Vec4T<T>*>(p);
#pragma unroll
        for (int i = 0; i < 4; i++) d[i] = (float)q.e[i];
    }
}
template <typename T>
__device__ __forceinline__ void store4(T* p, float a, float b, float c, float d)
{
    if constexpr (std::is_same<T, float>::value) {
        *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
    } else {
        Vec4T<T> q;
        q.e[0] = store_cast<T>(a); q.e[1] = store_cast<T>(b); q.e[2] = store_cast<T>(c); q.e[3] = store_cast<T>(d);
        *reinterpret_cast<Vec4T<T>*>(p) = q;
    }
}

// ---- shared-memory barrier helpers (mbarrier: waiting threads sleep in hardware instead of polling) ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(bar) : "memory");
}
// try_wait, then sleep NS nanoseconds between retries: a waiting warp stays out of the issue arbitration
template <int NS>
__device__ __forceinline__ void mbar_wait_sleep(uint32_t bar, uint32_t parity)
{
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
        if (done) break;
        if (NS > 0) __nanosleep(NS);
    }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    }
}
#endif

}  // namespace fdn
