// Stage 4: bilinear remap of a neighbour slice fused with the Gaussian-weighted accumulation; plus the
// no-OF wrap-around 1-D Gaussian and the batched transpose used by the X pass. sm_100a.
//
// Reference behaviour:
//   warp_slice                  /root/reference/src/flowdenoising.py:55-63  (cv2.remap INTER_LINEAR,
//                               BORDER_REPLICATE, float32 map -> OpenCV's 1/32-pixel quantiser, SURVEY App. A.1)
//   tmp_slice += warped*k[i]    :316, :317, :323  (NumPy >= 2: float64 product and sum, rounded to float32
//                               once per tap, SURVEY App. B Q9)
//   GaussianDenoising slices    :133-158 (no-OF path)
// Compiled with -fmad=false.
#include "fdn_internal.cuh"

namespace fdn {

// ------------------------------------------------------------------------------------------------
// K4: acc = f32(f64(acc) + f64(remap(neigh, flow)) * weight)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_warp_acc(const float* __restrict__ neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float2* __restrict__ flow,
           double weight, float* __restrict__ acc, int64_t a_ss, int64_t a_rs, int H, int W, int first)
{
    const int x = blockIdx.x * 128 + threadIdx.x;
    const int y = blockIdx.y;
    const int b = blockIdx.z;
    if (x >= W) return;
    const float* src = neigh + n_map.offset(b, n_ss);
    float v;
    if (flow) {
        const float2 f = flow[((int64_t)b * H + y) * W + x];
        // map = (flow + grid).astype(float32): one rounding of the exact sum
        const float mx = __fadd_rn(f.x, (float)x), my = __fadd_rn(f.y, (float)y);
        // cvRound(map * INTER_TAB_SIZE): round half to even
        const int sx = __float2int_rn(__fmul_rn(mx, 32.f)), sy = __float2int_rn(__fmul_rn(my, 32.f));
        const int ax = sx & 31, ay = sy & 31;
        int ix = sx >> 5, iy = sy >> 5;
        ix = min(max(ix, -32768), 32767);  // saturate_cast<short>
        iy = min(max(iy, -32768), 32767);
        const float tx1 = __fmul_rn((float)ax, 0.03125f), tx0 = __fsub_rn(1.f, tx1);
        const float ty1 = __fmul_rn((float)ay, 0.03125f), ty0 = __fsub_rn(1.f, ty1);
        const float w0 = __fmul_rn(ty0, tx0), w1 = __fmul_rn(ty0, tx1), w2 = __fmul_rn(ty1, tx0),
                    w3 = __fmul_rn(ty1, tx1);
        const int x0 = min(max(ix, 0), W - 1), x1 = min(max(ix + 1, 0), W - 1);
        const int y0 = min(max(iy, 0), H - 1), y1 = min(max(iy + 1, 0), H - 1);
        const float* r0 = src + (int64_t)y0 * n_rs;
        const float* r1 = src + (int64_t)y1 * n_rs;
        const float v0 = r0[x0], v1 = r0[x1], v2 = r1[x0], v3 = r1[x1];
        v = __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(v0, w0), __fmul_rn(v1, w1)), __fmul_rn(v2, w2)),
                      __fmul_rn(v3, w3));
    } else {
        v = src[(int64_t)y * n_rs + x];
    }
    float* ap = acc + (int64_t)b * a_ss + (int64_t)y * a_rs + x;
    const double prod = __dmul_rn((double)v, weight);
    *ap = (float)__dadd_rn(first ? 0.0 : (double)*ap, prod);   // tmp = zeros; tmp += v * k (:308, :316)
}

// Four consecutive pixels per thread (128-bit flow / accumulator accesses, four independent gathers in flight).
// Same arithmetic as k_warp_acc. Needs W % 4 == 0 and 16-byte aligned rows.
//
// remap_px<T> is cv2.remap of a T image with the same quantised map (SURVEY App. B Q3), returned as a float:
//   float      the float path above;
//   uint8      OpenCV's fixed point: weights rint(wy * wx * 2^15) of the 1/32-px table, (sum + 2^14) >> 15, saturated.
//              wy, wx are multiples of 1/32, so every entry is the exact integer (32 - ay or ay) * (32 - ax or ax) * 32:
//              it is computed in registers instead of read from a table (no per-lane divergent lookups). The one entry
//              OpenCV saturates to 32767 (ax = ay = 0) gives the same result for every 8-bit value;
//              tests/test_integer_volume_oracle.py pins all 1024 entries against cv2.
//   16U / 16S  the float32 weights and tap order of the float path, then rint and saturate (Cast<float, T>).
template <typename T>
__device__ __forceinline__ float remap_px(const T* __restrict__ src, int64_t n_rs, float fx, float fy, int x, int y, int H,
                                          int W)
{
    const float mx = __fadd_rn(fx, (float)x), my = __fadd_rn(fy, (float)y);
    const int sx = __float2int_rn(__fmul_rn(mx, 32.f)), sy = __float2int_rn(__fmul_rn(my, 32.f));
    const int ax = sx & 31, ay = sy & 31;
    int ix = sx >> 5, iy = sy >> 5;
    ix = min(max(ix, -32768), 32767);
    iy = min(max(iy, -32768), 32767);
    const int x0 = min(max(ix, 0), W - 1), x1 = min(max(ix + 1, 0), W - 1);
    const int y0 = min(max(iy, 0), H - 1), y1 = min(max(iy + 1, 0), H - 1);
    const T* r0 = src + (int64_t)y0 * n_rs;
    const T* r1 = src + (int64_t)y1 * n_rs;
    if constexpr (std::is_same<T, uint8_t>::value) {
        const int v0 = __ldg(r0 + x0), v1 = __ldg(r0 + x1), v2 = __ldg(r1 + x0), v3 = __ldg(r1 + x1);
        const int s = v0 * (((32 - ay) * (32 - ax)) << 5) + v1 * (((32 - ay) * ax) << 5) + v2 * ((ay * (32 - ax)) << 5) +
                      v3 * ((ay * ax) << 5);
        return (float)min(max((s + (1 << 14)) >> 15, 0), 255);
    } else {
        const float tx1 = __fmul_rn((float)ax, 0.03125f), tx0 = __fsub_rn(1.f, tx1);
        const float ty1 = __fmul_rn((float)ay, 0.03125f), ty0 = __fsub_rn(1.f, ty1);
        const float w0 = __fmul_rn(ty0, tx0), w1 = __fmul_rn(ty0, tx1), w2 = __fmul_rn(ty1, tx0), w3 = __fmul_rn(ty1, tx1);
        const float v0 = (float)__ldg(r0 + x0), v1 = (float)__ldg(r0 + x1), v2 = (float)__ldg(r1 + x0),
                    v3 = (float)__ldg(r1 + x1);
        const float s =
            __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(v0, w0), __fmul_rn(v1, w1)), __fmul_rn(v2, w2)), __fmul_rn(v3, w3));
        if constexpr (std::is_same<T, float>::value) return s;
        else return (float)min(max(__float2int_rn(s), (int)TypeRange<T>::lo), (int)TypeRange<T>::hi);
    }
}

__global__ void __launch_bounds__(128)
k_warp_acc4(const float* __restrict__ neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float4* __restrict__ flow,
            double weight, float* __restrict__ acc, int64_t a_ss, int64_t a_rs, int H, int W, int first)
{
    const int x = (blockIdx.x * 128 + threadIdx.x) * 4;
    const int y = blockIdx.y;
    const int b = blockIdx.z;
    if (x >= W) return;
    const float* src = neigh + n_map.offset(b, n_ss);
    float v[4];
    if (flow) {
        const float4* fp = flow + (((int64_t)b * H + y) * W + x) / 2;   // two float2 flows per float4
        const float4 f01 = __ldg(fp), f23 = __ldg(fp + 1);
        v[0] = remap_px(src, n_rs, f01.x, f01.y, x, y, H, W);
        v[1] = remap_px(src, n_rs, f01.z, f01.w, x + 1, y, H, W);
        v[2] = remap_px(src, n_rs, f23.x, f23.y, x + 2, y, H, W);
        v[3] = remap_px(src, n_rs, f23.z, f23.w, x + 3, y, H, W);
    } else {
        const float4 c = __ldg(reinterpret_cast<const float4*>(src + (int64_t)y * n_rs + x));
        v[0] = c.x; v[1] = c.y; v[2] = c.z; v[3] = c.w;
    }
    float4* ap = reinterpret_cast<float4*>(acc + (int64_t)b * a_ss + (int64_t)y * a_rs + x);
    float o[4];
    if (first) {
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = (float)__dadd_rn(0.0, __dmul_rn((double)v[i], weight));   // tmp = zeros; tmp += v * k
    } else {
        const float4 a = *ap;
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int i = 0; i < 4; i++) o[i] = (float)__dadd_rn((double)av[i], __dmul_rn((double)v[i], weight));
    }
    *ap = make_float4(o[0], o[1], o[2], o[3]);
}

int launch_warp_acc(const float* neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float* flow, double weight,
                    float* acc, int64_t a_ss, int64_t a_rs, int n, int H, int W, int first, cudaStream_t st)
{
    const bool vec4 = W % 4 == 0 && n_ss % 4 == 0 && n_rs % 4 == 0 && a_ss % 4 == 0 && a_rs % 4 == 0 &&
                      (reinterpret_cast<uintptr_t>(neigh) & 15) == 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(flow) & 15) == 0;
    if (vec4) {
        for (int b0 = 0; b0 < n; b0 += 65535) {
            const int nb = n - b0 < 65535 ? n - b0 : 65535;
            SlotMap m = n_map;
            m.b0 += b0;
            dim3 grid((unsigned)cdiv(W, 512), (unsigned)H, (unsigned)nb);
            ProfScope ps(K_WARP_ACC, (double)nb * H * W * (4.0 + (flow ? 8.0 : 0.0) + (first ? 4.0 : 8.0)), st);
            k_warp_acc4<<<grid, 128, 0, st>>>(neigh, n_ss, n_rs, m,
                                              flow ? reinterpret_cast<const float4*>(flow + (int64_t)b0 * H * W * 2) : nullptr,
                                              weight, acc + (int64_t)b0 * a_ss, a_ss, a_rs, H, W, first);
            FDN_LAUNCHED("k_warp_acc4");
        }
        return FDN_OK;
    }
    for (int b0 = 0; b0 < n; b0 += 65535) {
        const int nb = n - b0 < 65535 ? n - b0 : 65535;
        SlotMap m = n_map;
        m.b0 += b0;
        dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)nb);
        ProfScope ps(K_WARP_ACC, (double)nb * H * W * (4.0 + (flow ? 8.0 : 0.0) + (first ? 4.0 : 8.0)), st);
        k_warp_acc<<<grid, 128, 0, st>>>(neigh, n_ss, n_rs, m,
                                         flow ? reinterpret_cast<const float2*>(flow) + (int64_t)b0 * H * W : nullptr,
                                         weight, acc + (int64_t)b0 * a_ss, a_ss, a_rs, H, W, first);
        FDN_LAUNCHED("k_warp_acc");
    }
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Both chain directions in one launch (the two chains of src/flowdenoising.py:311-316 and :319-324 advance together):
// images [0, n) are the backward neighbours -- remapped and accumulated in place, the reference's order -- and images
// [n, 2n) the forward neighbours, whose remapped values wait in `stash` until the backward chain and the centre tap
// are in the accumulator (k_acc_finish applies them in the reference's order: centre, +1, ..., +r).
// T is the element type of the volume and of the stash (a remapped integer image is an integer image); the
// accumulator is float32 for every T.
// ------------------------------------------------------------------------------------------------
template <typename T, int VEC>
__global__ void __launch_bounds__(128)
k_warp_pair(const T* __restrict__ neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float* __restrict__ flow,
            double weight, float* __restrict__ acc, int64_t a_ss, int64_t a_rs, SlotMap a_map, T* __restrict__ stash,
            int n, int b0, int H, int W, int first)
{
    const int x = (blockIdx.x * 128 + threadIdx.x) * VEC;
    const int y = blockIdx.y;
    const int b = b0 + blockIdx.z;   // 0 .. 2n-1
    if (x >= W) return;
    const T* src = neigh + n_map.offset(b, n_ss);
    const int64_t fpx = ((int64_t)b * H + y) * W + x;
    float v[VEC];
    if (VEC == 4) {
        const float4* fp = reinterpret_cast<const float4*>(flow) + fpx / 2;   // two float2 flows per float4
        const float4 f01 = __ldg(fp), f23 = __ldg(fp + 1);
        v[0] = remap_px(src, n_rs, f01.x, f01.y, x, y, H, W);
        v[1 % VEC] = remap_px(src, n_rs, f01.z, f01.w, x + 1, y, H, W);
        v[2 % VEC] = remap_px(src, n_rs, f23.x, f23.y, x + 2, y, H, W);
        v[3 % VEC] = remap_px(src, n_rs, f23.z, f23.w, x + 3, y, H, W);
    } else {
        const float2 f = __ldg(reinterpret_cast<const float2*>(flow) + fpx);
        v[0] = remap_px(src, n_rs, f.x, f.y, x, y, H, W);
    }
    if (b < n) {
        float* ap = acc + a_map.offset(b, a_ss) + (int64_t)y * a_rs + x;
        if (VEC == 4) {
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            if (!first) a = *reinterpret_cast<float4*>(ap);
            const float av[4] = {a.x, a.y, a.z, a.w};
            float o[4];
#pragma unroll
            for (int i = 0; i < 4; i++)
                o[i] = (float)__dadd_rn(first ? 0.0 : (double)av[i], __dmul_rn((double)v[i % VEC], weight));
            *reinterpret_cast<float4*>(ap) = make_float4(o[0], o[1], o[2], o[3]);
        } else {
            *ap = (float)__dadd_rn(first ? 0.0 : (double)*ap, __dmul_rn((double)v[0], weight));
        }
    } else {
        T* sp = stash + ((int64_t)(b - n) * H + y) * W + x;
        if (VEC == 4) store4(sp, v[0], v[1 % VEC], v[2 % VEC], v[3 % VEC]);
        else *sp = store_cast<T>(v[0]);
    }
}

template <typename T>
int launch_warp_pair(const T* neigh, int64_t n_ss, int64_t n_rs, SlotMap n_map, const float* flow, double weight,
                     float* acc, int64_t a_ss, int64_t a_rs, SlotMap a_map, T* stash, int n, int H, int W, int first,
                     cudaStream_t st)
{
    // (the volume strides of a batch move every image's base: they must keep the 16-byte alignment too)
    const bool vec4 = W % 4 == 0 && n_ss % 4 == 0 && n_rs % 4 == 0 && a_ss % 4 == 0 && a_rs % 4 == 0 &&
                      n_map.vstride % 4 == 0 && a_map.vstride % 4 == 0 &&
                      (reinterpret_cast<uintptr_t>(neigh) & 15) == 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(flow) & 15) == 0 &&
                      (reinterpret_cast<uintptr_t>(stash) & (4 * sizeof(T) - 1)) == 0;
    FDN_CHECK_ARG(H <= 65535, "image too tall for one launch");
    const double es = (double)sizeof(T);
    for (int b0 = 0; b0 < 2 * n; b0 += 65535) {
        const int nb = 2 * n - b0 < 65535 ? 2 * n - b0 : 65535;
        // remap: flow 8 + neighbour; backward half: float32 accumulator 4 (+4 unless first), forward half: stash
        ProfScope ps(K_WARP_ACC, (double)nb * H * W * (8.0 + es + (first ? 4.0 + es : 8.0 + es) / 2), st);
        if (vec4) {
            dim3 grid((unsigned)cdiv(W, 512), (unsigned)H, (unsigned)nb);
            k_warp_pair<T, 4><<<grid, 128, 0, st>>>(neigh, n_ss, n_rs, n_map, flow, weight, acc, a_ss, a_rs, a_map, stash, n,
                                                    b0, H, W, first);
        } else {
            dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)nb);
            k_warp_pair<T, 1><<<grid, 128, 0, st>>>(neigh, n_ss, n_rs, n_map, flow, weight, acc, a_ss, a_rs, a_map, stash, n,
                                                    b0, H, W, first);
        }
        FDN_LAUNCHED("k_warp_pair");
    }
    return FDN_OK;
}

#define FDN_MAX_R 128
static_assert(2 * FDN_MAX_R + 1 == FDN_MAX_KLEN, "k_acc_finish must take every kernel make_plan accepts");
struct FinishTaps {
    double k[FDN_MAX_R + 1];   // centre, +1, ..., +r
};

template <typename T, int VEC>
__global__ void __launch_bounds__(128)
k_acc_finish(const T* __restrict__ centre, int64_t c_ss, int64_t c_rs, SlotMap c_map, const T* __restrict__ stash,
             int64_t stash_stride, int r, FinishTaps taps, float* __restrict__ acc, int64_t a_ss, int64_t a_rs,
             SlotMap a_map, T* __restrict__ out, int64_t o_ss, int64_t o_rs, SlotMap o_map, int b0, int H, int W,
             int have_acc)
{
    const int x = (blockIdx.x * 128 + threadIdx.x) * VEC;
    const int y = blockIdx.y;
    const int b = b0 + blockIdx.z;
    if (x >= W) return;
    const T* cp = centre + c_map.offset(b, c_ss) + (int64_t)y * c_rs + x;
    float* ap = acc + a_map.offset(b, a_ss) + (int64_t)y * a_rs + x;
    const T* sp = stash + ((int64_t)b * H + y) * W + x;
    float a[VEC], v[VEC];
    auto load = [&](const T* p, float* dst) {
        if (VEC == 4) {
            float q[4];
            load4(p, q);
            dst[0] = q[0]; dst[1 % VEC] = q[1]; dst[2 % VEC] = q[2]; dst[3 % VEC] = q[3];
        } else {
            dst[0] = (float)__ldg(p);
        }
    };
#pragma unroll
    for (int i = 0; i < VEC; i++) a[i] = 0.f;
    if (have_acc) {
        if (VEC == 4) {
            const float4 q = *reinterpret_cast<const float4*>(ap);
            a[0] = q.x; a[1 % VEC] = q.y; a[2 % VEC] = q.z; a[3 % VEC] = q.w;
        } else {
            a[0] = *ap;
        }
    }
    load(cp, v);   // tmp_slice += vol[z] * kernel[ks2]  (src/flowdenoising.py:317)
#pragma unroll
    for (int i = 0; i < VEC; i++) a[i] = (float)__dadd_rn((double)a[i], __dmul_rn((double)v[i], taps.k[0]));
    for (int d = 0; d < r; d++) {   // forward chain, nearest neighbour first (:319-324)
        load(sp + (int64_t)d * stash_stride, v);
#pragma unroll
        for (int i = 0; i < VEC; i++) a[i] = (float)__dadd_rn((double)a[i], __dmul_rn((double)v[i], taps.k[d + 1]));
    }
    if constexpr (std::is_same<T, float>::value) {
        if (VEC == 4) *reinterpret_cast<float4*>(ap) = make_float4(a[0], a[1 % VEC], a[2 % VEC], a[3 % VEC]);
        else *ap = a[0];
    } else {   // filtered_vol[z] = tmp_slice (:325): truncation toward zero
        T* op = out + o_map.offset(b, o_ss) + (int64_t)y * o_rs + x;
        if (VEC == 4) store4(op, a[0], a[1 % VEC], a[2 % VEC], a[3 % VEC]);
        else *op = store_cast<T>(a[0]);
    }
}

template <typename T>
int launch_acc_finish(const T* centre, int64_t c_ss, int64_t c_rs, SlotMap c_map, const T* stash, int r, const double* k,
                      float* acc, int64_t a_ss, int64_t a_rs, SlotMap a_map, T* out, int64_t o_ss, int64_t o_rs,
                      SlotMap o_map, int n, int H, int W, int have_acc, cudaStream_t st)
{
    FDN_CHECK_ARG(r >= 0 && r <= FDN_MAX_R, "kernel radius %d unsupported (<= %d)", r, FDN_MAX_R);
    FDN_CHECK_ARG(H <= 65535, "image too tall for one launch");
    constexpr bool typed = !std::is_same<T, float>::value;
    constexpr uintptr_t al = 4 * sizeof(T) - 1;
    FinishTaps taps;
    for (int i = 0; i <= r; i++) taps.k[i] = k[i];
    bool vec4 = W % 4 == 0 && c_ss % 4 == 0 && c_rs % 4 == 0 && a_ss % 4 == 0 && a_rs % 4 == 0 &&
                c_map.vstride % 4 == 0 && a_map.vstride % 4 == 0 &&
                (reinterpret_cast<uintptr_t>(centre) & al) == 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0 &&
                (reinterpret_cast<uintptr_t>(stash) & al) == 0;
    if (typed)
        vec4 = vec4 && o_ss % 4 == 0 && o_rs % 4 == 0 && o_map.vstride % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & al) == 0;
    const int64_t stash_stride = (int64_t)n * H * W;
    const double es = (double)sizeof(T);
    for (int b0 = 0; b0 < n; b0 += 65535) {
        const int nb = n - b0 < 65535 ? n - b0 : 65535;
        // centre + r stash images + the result (in T), the float32 accumulator read when there are backward taps
        ProfScope ps(K_WARP_ACC, (double)nb * H * W * (es * (r + 2) + (have_acc ? 4.0 : 0.0)), st);
        if (vec4) {
            dim3 grid((unsigned)cdiv(W, 512), (unsigned)H, (unsigned)nb);
            k_acc_finish<T, 4><<<grid, 128, 0, st>>>(centre, c_ss, c_rs, c_map, stash, stash_stride, r, taps, acc, a_ss, a_rs,
                                                     a_map, out, o_ss, o_rs, o_map, b0, H, W, have_acc);
        } else {
            dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)nb);
            k_acc_finish<T, 1><<<grid, 128, 0, st>>>(centre, c_ss, c_rs, c_map, stash, stash_stride, r, taps, acc, a_ss, a_rs,
                                                     a_map, out, o_ss, o_rs, o_map, b0, H, W, have_acc);
        }
        FDN_LAUNCHED("k_acc_finish");
    }
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// cv2.remap of dense T images alone (stage entry point fdn_remap_typed: pins the integer remap)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128)
k_remap(const T* __restrict__ src, const float2* __restrict__ flow, T* __restrict__ dst, int H, int W)
{
    const int x = blockIdx.x * 128 + threadIdx.x;
    const int y = blockIdx.y;
    const int64_t b = blockIdx.z;
    if (x >= W) return;
    const float2 f = flow[(b * H + y) * W + x];
    dst[(b * H + y) * W + x] = store_cast<T>(remap_px(src + b * H * W, W, f.x, f.y, x, y, H, W));
}

template <typename T>
int launch_remap(const T* src, const float* flow, T* dst, int n, int H, int W, cudaStream_t st)
{
    FDN_CHECK_ARG(H <= 65535 && n <= 65535, "batch or image too large for one launch");
    dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)n);
    k_remap<T><<<grid, 128, 0, st>>>(src, reinterpret_cast<const float2*>(flow), dst, H, W);
    FDN_LAUNCHED("k_remap");
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Batched transpose of the last two axes with arbitrary outer/row strides (32x32 shared-memory tiles):
//   out[n*out_sn + b*out_sb + a] = in[n*in_sn + a*in_sa + b],  a < A, b < B
// Dense case ([n][A][B] -> [n][B][A]): in_sn = out_sn = A*B, in_sa = B, out_sb = A. The strided form is the
// transposing unpack of the multi-GPU re-slab (flowdenoising_b200/dist.py).
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
k_transpose(const T* __restrict__ in, int64_t in_sn, int64_t in_sa, T* __restrict__ out, int64_t out_sn, int64_t out_sb,
            int A, int B)
{
    __shared__ T tile[32][33];
    const int64_t img = blockIdx.z;
    const int b0 = blockIdx.x * 32, a0 = blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const T* src = in + img * in_sn;
    T* dst = out + img * out_sn;
    for (int i = ty; i < 32; i += 8) {
        int a = a0 + i, b = b0 + tx;
        if (a < A && b < B) tile[i][tx] = src[(int64_t)a * in_sa + b];
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        int b = b0 + i, a = a0 + tx;
        if (a < A && b < B) dst[(int64_t)b * out_sb + a] = tile[tx][i];
    }
}

template <typename T>
int launch_transpose_strided(const T* in, int64_t in_sn, int64_t in_sa, T* out, int64_t out_sn, int64_t out_sb, int n,
                             int A, int B, cudaStream_t st)
{
    FDN_CHECK_ARG(cdiv(A, 32) <= 65535, "transpose: A too large");
    for (int b0 = 0; b0 < n; b0 += 65535) {
        const int nb = n - b0 < 65535 ? n - b0 : 65535;
        dim3 grid((unsigned)cdiv(B, 32), (unsigned)cdiv(A, 32), (unsigned)nb);
        ProfScope ps(K_TRANSPOSE, 2.0 * sizeof(T) * nb * A * B, st);
        k_transpose<T><<<grid, 256, 0, st>>>(in + (int64_t)b0 * in_sn, in_sn, in_sa, out + (int64_t)b0 * out_sn, out_sn,
                                          out_sb, A, B);
        FDN_LAUNCHED("k_transpose");
    }
    return FDN_OK;
}

template <typename T>
int launch_transpose(const T* in, T* out, int n, int A, int B, cudaStream_t st)
{
    return launch_transpose_strided(in, (int64_t)A * B, B, out, (int64_t)A * B, A, n, A, B, st);
}

// ------------------------------------------------------------------------------------------------
// Strided 3-D copy with periodic index offsets (the packing side of the re-slab / halo exchange):
//   out[a*out_sa + b*out_sb + c] = in[a*in_sa + ((b0 + b) mod bw)*in_sb + ((c0 + c) mod cw)]
// A copy moves bits: one kernel per element size (1, 2, 4 bytes). 4-byte elements take one per thread. Narrower ones
// take a run of 4 bytes of consecutive c per thread (4 uint8 / 2 uint16), so that a warp's stores cover 128 contiguous
// bytes instead of 32 / 64; the run is stored as one 32-bit word where the destination is 4-byte aligned and does not
// end inside it. Reads follow the periodic index element by element; a run that crosses the wrap takes the guarded
// loop.
// ------------------------------------------------------------------------------------------------
template <typename T>
__host__ __device__ constexpr int copy3d_run() { return sizeof(T) >= 4 ? 1 : (int)(4 / sizeof(T)); }

template <typename T>
__global__ void __launch_bounds__(256)
k_copy3d(const T* __restrict__ in, int64_t in_sa, int64_t in_sb, int b0, int bw, int c0, int cw,
         T* __restrict__ out, int64_t out_sa, int64_t out_sb, int B, int C)
{
    constexpr int R = copy3d_run<T>();
    const int c = (blockIdx.x * 256 + threadIdx.x) * R;
    const int b = blockIdx.y;
    const int64_t a = blockIdx.z;
    if (c >= C) return;
    int bi = (b0 + b) % bw;
    if (bi < 0) bi += bw;
    int ci = (c0 + c) % cw;
    if (ci < 0) ci += cw;
    (void)B;
    if constexpr (R == 1) {
        out[a * out_sa + (int64_t)b * out_sb + c] = in[a * in_sa + (int64_t)bi * in_sb + ci];
    } else {
        const T* src = in + a * in_sa + (int64_t)bi * in_sb;
        T* dst = out + a * out_sa + (int64_t)b * out_sb + c;
        const int n = C - c < R ? C - c : R;
        union { uint32_t w; T e[R]; } v;
        v.w = 0;
        if (ci + n <= cw) {
#pragma unroll
            for (int j = 0; j < R; j++)
                if (j < n) v.e[j] = src[ci + j];
        } else {                                    // the run crosses the wrap (possibly more than once: cw < R)
#pragma unroll
            for (int j = 0; j < R; j++)
                if (j < n) v.e[j] = src[(ci + j) % cw];
        }
        if (n == R && (reinterpret_cast<uintptr_t>(dst) & 3) == 0) {
            *reinterpret_cast<uint32_t*>(dst) = v.w;
        } else {
#pragma unroll
            for (int j = 0; j < R; j++)
                if (j < n) dst[j] = v.e[j];
        }
    }
}

template <typename T>
int launch_copy3d(const T* in, int64_t in_sa, int64_t in_sb, int b0, int bw, int c0, int cw, T* out,
                  int64_t out_sa, int64_t out_sb, int A, int B, int C, cudaStream_t st)
{
    FDN_CHECK_ARG(B <= 65535, "copy3d: B too large");
    FDN_CHECK_ARG(bw >= 1 && cw >= 1, "copy3d: wrap lengths must be >= 1");
    constexpr int R = copy3d_run<T>();
    for (int a0 = 0; a0 < A; a0 += 65535) {
        const int na = A - a0 < 65535 ? A - a0 : 65535;
        dim3 grid((unsigned)cdiv(C, 256 * R), (unsigned)B, (unsigned)na);
        ProfScope ps(K_COPY3D, 2.0 * sizeof(T) * na * B * C, st);
        k_copy3d<T><<<grid, 256, 0, st>>>(in + (int64_t)a0 * in_sa, in_sa, in_sb, b0, bw, c0, cw,
                                          out + (int64_t)a0 * out_sa, out_sa, out_sb, B, C);
        FDN_LAUNCHED("k_copy3d");
    }
    return FDN_OK;
}

#define FDN_INST_WARP(T)                                                                                              \
    template int launch_warp_pair<T>(const T*, int64_t, int64_t, SlotMap, const float*, double, float*, int64_t, int64_t, \
                                     SlotMap, T*, int, int, int, int, cudaStream_t);                                      \
    template int launch_acc_finish<T>(const T*, int64_t, int64_t, SlotMap, const T*, int, const double*, float*, int64_t, \
                                      int64_t, SlotMap, T*, int64_t, int64_t, SlotMap, int, int, int, int, cudaStream_t);
FDN_INST_WARP(float)
FDN_INST_WARP(uint8_t)
FDN_INST_WARP(uint16_t)
FDN_INST_WARP(int16_t)
template int launch_remap<uint8_t>(const uint8_t*, const float*, uint8_t*, int, int, int, cudaStream_t);
template int launch_remap<uint16_t>(const uint16_t*, const float*, uint16_t*, int, int, int, cudaStream_t);
template int launch_remap<int16_t>(const int16_t*, const float*, int16_t*, int, int, int, cudaStream_t);
#define FDN_INST_TRANSPOSE(T)                                                                                         \
    template int launch_transpose<T>(const T*, T*, int, int, int, cudaStream_t);                                      \
    template int launch_transpose_strided<T>(const T*, int64_t, int64_t, T*, int64_t, int64_t, int, int, int, cudaStream_t); \
    template int launch_copy3d<T>(const T*, int64_t, int64_t, int, int, int, int, T*, int64_t, int64_t, int, int, int,      \
                                  cudaStream_t);
FDN_INST_TRANSPOSE(float)
FDN_INST_TRANSPOSE(uint8_t)
FDN_INST_TRANSPOSE(uint16_t)
}  // namespace fdn
