// Stage 1 (Gaussian pyramid) and stage 2 (Farneback polynomial expansion) kernels, sm_100a.
//
// Reference behaviour: cv2.calcOpticalFlowFarneback internals reached from
// /root/reference/src/flowdenoising.py:69-79 (OpenCV 4.13 optflowgf.cpp: GaussianBlur + resize per level,
// FarnebackPolyExp), specified in SURVEY.md App. A.0-A.2. Arithmetic (operation order, which products are
// fused, float32 vs float64) follows OpenCV so that results are bit-identical to the CPU reference on
// AVX2 hosts; this file is compiled with -fmad=false and fuses only where fmaf() is written.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <cuda.h>

#include "fdn_internal.cuh"

namespace fdn {

// ------------------------------------------------------------------------------------------------
// host-side constant preparation
// ------------------------------------------------------------------------------------------------
int prepare_blur_taps(int ksz, double sigma, BlurTaps* bt)
{
    if (ksz < 1 || ksz > FDN_MAX_KSZ || (ksz & 1) == 0) {
        set_error("pyramid smoothing kernel size %d unsupported (odd, <= %d)", ksz, FDN_MAX_KSZ);
        return FDN_ERR_INVALID;
    }
    bt->ksz = ksz;
    if (sigma <= 0 && ksz == 3) {  // cv::getGaussianKernel small fixed kernel (level 0)
        bt->k[0] = 0.25f; bt->k[1] = 0.5f; bt->k[2] = 0.25f;
        return FDN_OK;
    }
    double sx = sigma > 0 ? sigma : ((ksz - 1) * 0.5 - 1) * 0.3 + 0.8;
    double scale2x = -0.5 / (sx * sx);
    double t[FDN_MAX_KSZ];
    double sum = 0;
    for (int i = 0; i < ksz; i++) {
        double x = i - (ksz - 1) * 0.5;
        t[i] = exp(scale2x * x * x);
        sum += t[i];
    }
    sum = 1. / sum;
    for (int i = 0; i < ksz; i++) bt->k[i] = (float)(t[i] * sum);
    return FDN_OK;
}

void prepare_poly_consts(int n, double sigma, PolyConsts* pc)
{
    // FarnebackPrepareGaussian: float taps, float64 Gram matrix, closed-form inverse of its block structure
    if (sigma < 1.1920928955078125e-07) sigma = n * 0.3;
    float g[16], xg[16], xxg[16];
    double s = 0.;
    for (int x = -n; x <= n; x++) {
        g[x + n] = (float)exp(-x * x / (2 * sigma * sigma));
        s += g[x + n];
    }
    s = 1. / s;
    for (int x = -n; x <= n; x++) {
        g[x + n] = (float)(g[x + n] * s);
        xg[x + n] = (float)(x * g[x + n]);
        xxg[x + n] = (float)(x * x * g[x + n]);
    }
    double G00 = 0, G11 = 0, G33 = 0, G55 = 0;
    for (int y = -n; y <= n; y++)
        for (int x = -n; x <= n; x++) {
            float gg = g[y + n] * g[x + n];
            G00 += gg;
            G11 += gg * x * x;
            G33 += gg * x * x * x * x;
            G55 += gg * x * x * y * y;
        }
    // cv::invert(G, DECOMP_CHOLESKY): OpenCV's CholImpl on an identity right-hand side, operation by operation
    // (a closed-form inverse differs in the last bit of ig03/ig33 and flips ~1 float32 rounding of R in 1e7)
    enum { m = 6 };
    double L[6][6], inv[6][6];
    memset(L, 0, sizeof L);
    L[0][0] = G00; L[1][1] = G11; L[3][3] = G33; L[5][5] = G55;
    L[2][2] = L[0][3] = L[0][4] = L[3][0] = L[4][0] = L[1][1];
    L[4][4] = L[3][3];
    L[3][4] = L[4][3] = L[5][5];
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) inv[i][j] = i == j ? 1. : 0.;
    for (int i = 0; i < m; i++) {
        double t;
        for (int j = 0; j < i; j++) {
            t = L[i][j];
            for (int k = 0; k < j; k++) t -= L[i][k] * L[j][k];
            L[i][j] = t * L[j][j];
        }
        t = L[i][i];
        for (int k = 0; k < i; k++) { double u = L[i][k]; t -= u * u; }
        L[i][i] = 1. / sqrt(t);
    }
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) {
            double t = inv[i][j];
            for (int k = 0; k < i; k++) t -= L[i][k] * inv[k][j];
            inv[i][j] = t * L[i][i];
        }
    for (int i = m - 1; i >= 0; i--)
        for (int j = 0; j < m; j++) {
            double t = inv[i][j];
            for (int k = m - 1; k > i; k--) t -= L[k][i] * inv[k][j];
            inv[i][j] = t * L[i][i];
        }
    pc->n = n;
    pc->ig11 = inv[1][1];
    pc->ig03 = inv[0][3];
    pc->ig33 = inv[3][3];
    pc->ig55 = inv[5][5];
    for (int k = 0; k < 8; k++) { pc->g[k] = pc->xg[k] = pc->xxg[k] = 0.f; }
    for (int k = 0; k <= n; k++) { pc->g[k] = g[n + k]; pc->xg[k] = xg[n + k]; pc->xxg[k] = xxg[n + k]; }
    for (int k = 0; k < 8; k++) { pc->gd[k] = (double)pc->g[k]; pc->xxgd[k] = (double)pc->xxg[k]; }
}

// ------------------------------------------------------------------------------------------------
// GaussianBlur: row filter then column filter, BORDER_REFLECT_101
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * (len - 1) - p;
    return p;
}

// One thread per output pixel; the taps of neighbouring threads overlap in L1. The input is float32 or the integer
// element type of a typed volume: calcOpticalFlowFarneback converts its images with convertTo(CV_32F) before this
// blur, so every value is read and converted here and no float32 copy of the volume exists.
template <typename T>
__global__ void __launch_bounds__(128)
k_blur_rows(const T* __restrict__ in_, int64_t in_ss, int64_t in_rs, SlotMap in_map, float* __restrict__ out, int H,
            int W, BlurTaps bt)
{
    const int x = blockIdx.x * 128 + threadIdx.x;
    const int y = blockIdx.y;
    const int b = blockIdx.z;
    if (x >= W) return;
    const T* s_ = in_ + (int64_t)in_map.slot(b) * in_ss + (int64_t)y * in_rs;
    auto s = [&](int i) { return (float)s_[i]; };
    const int ksz = bt.ksz, r = ksz >> 1;
    float acc;
    if (ksz == 3) {
        // SymmRowSmallVec_32f: fma(centre, k1, (l + r) * k0); a last odd column is OpenCV's scalar tail
        float lr = __fadd_rn(s(reflect101(x - 1, W)), s(reflect101(x + 1, W)));
        acc = x < (W & ~1) ? fmaf(s(x), bt.k[1], __fmul_rn(lr, bt.k[0])) : fmaf(lr, bt.k[0], __fmul_rn(s(x), bt.k[1]));
    } else if (x >= r && x + r < W) {
        const int p0 = x - r;
        acc = __fmul_rn(s(p0), bt.k[0]);
        if (x < (W & ~3)) {
            for (int i = 1; i < ksz; i++) acc = fmaf(s(p0 + i), bt.k[i], acc);
        } else {
            for (int i = 1; i < ksz; i++) acc = __fadd_rn(acc, __fmul_rn(s(p0 + i), bt.k[i]));
        }
    } else {
        acc = __fmul_rn(s(reflect101(x - r, W)), bt.k[0]);
        if (x < (W & ~3)) {
            for (int i = 1; i < ksz; i++) acc = fmaf(s(reflect101(x - r + i, W)), bt.k[i], acc);
        } else {
            for (int i = 1; i < ksz; i++) acc = __fadd_rn(acc, __fmul_rn(s(reflect101(x - r + i, W)), bt.k[i]));
        }
    }
    out[((int64_t)b * H + y) * W + x] = acc;
}

__global__ void __launch_bounds__(128)
k_blur_cols(const float* __restrict__ in, float* __restrict__ out, int H, int W, BlurTaps bt)
{
    const int x = blockIdx.x * 128 + threadIdx.x;
    const int y = blockIdx.y;
    const int b = blockIdx.z;
    if (x >= W) return;
    const float* s = in + (int64_t)b * H * W + x;
    const int ksz = bt.ksz, r = ksz >> 1;
    float acc = __fmul_rn(s[(int64_t)y * W], bt.k[r]);
    const bool fused = (ksz == 3) || x < (W & ~7);  // SymmColumnVec_32f covers multiples of 8 lanes
    for (int i = 1; i <= r; i++) {
        float a = s[(int64_t)reflect101(y + i, H) * W];
        float c = s[(int64_t)reflect101(y - i, H) * W];
        float ac = __fadd_rn(a, c);
        acc = fused ? fmaf(ac, bt.k[r + i], acc) : __fadd_rn(acc, __fmul_rn(ac, bt.k[r + i]));
    }
    out[((int64_t)b * H + y) * W + x] = acc;
}

// Register-window variants for the tap counts the Farneback pyramid actually uses: ksz = max(rint(5 sigma_k) | 1, 3)
// with sigma_k = (2^k - 1) / 2 -> 3, 3, 9, 19, 39, 79 taps for levels 0..5 (half widths 1, 4, 9, 19, 39; SURVEY.md
// App. A.0). Same arithmetic per output as k_blur_rows / k_blur_cols; each thread produces 4 outputs from one window of
// 4 + 2R inputs instead of 4 * (2R + 1) loads with their address arithmetic.
template <typename T, int R>
__global__ void __launch_bounds__(128)
k_blur_rows4(const T* __restrict__ in, int64_t in_ss, int64_t in_rs, SlotMap in_map, float* __restrict__ out, int H,
             int W, BlurTaps bt)
{
    constexpr int KS = 2 * R + 1;
    const int x0 = (blockIdx.x * 128 + threadIdx.x) * 4;   // W % 4 == 0
    const int y = blockIdx.y;
    const int b = blockIdx.z;
    if (x0 >= W) return;
    const T* s = in + (int64_t)in_map.slot(b) * in_ss + (int64_t)y * in_rs;
    float v[4 + 2 * R];
    if (x0 >= R && x0 + 3 + R < W) {
#pragma unroll
        for (int i = 0; i < 4 + 2 * R; i++) v[i] = (float)__ldg(s + x0 - R + i);
    } else {
#pragma unroll
        for (int i = 0; i < 4 + 2 * R; i++) v[i] = (float)__ldg(s + reflect101(x0 - R + i, W));
    }
    float o[4];
#pragma unroll
    for (int j = 0; j < 4; j++) {
        const int x = x0 + j;
        float acc;
        if (KS == 3) {
            // SymmRowSmallVec_32f: fma(centre, k1, (l + r) * k0); a last odd column is OpenCV's scalar tail
            const float lr = __fadd_rn(v[j], v[j + 2]);
            acc = x < (W & ~1) ? fmaf(v[j + 1], bt.k[1], __fmul_rn(lr, bt.k[0])) : fmaf(lr, bt.k[0], __fmul_rn(v[j + 1], bt.k[1]));
        } else {
            // x0 is a multiple of 4 and W % 4 == 0 here: every output lies in the vectorised part (x < (W & ~3))
            acc = __fmul_rn(v[j], bt.k[0]);
#pragma unroll
            for (int i = 1; i < KS; i++) acc = fmaf(v[j + i], bt.k[i], acc);
        }
        o[j] = acc;
    }
    *reinterpret_cast<float4*>(out + ((int64_t)b * H + y) * W + x0) = make_float4(o[0], o[1], o[2], o[3]);
}

template <int R>
__global__ void __launch_bounds__(128)
k_blur_cols4(const float* __restrict__ in, float* __restrict__ out, int H, int W, BlurTaps bt)
{
    constexpr int KS = 2 * R + 1;
    const int x = blockIdx.x * 128 + threadIdx.x;
    const int y0 = blockIdx.y * 4;
    const int b = blockIdx.z;
    if (x >= W) return;
    const float* s = in + (int64_t)b * H * W + x;
    float v[4 + 2 * R];
    if (y0 >= R && y0 + 3 + R < H) {
#pragma unroll
        for (int i = 0; i < 4 + 2 * R; i++) v[i] = __ldg(s + (int64_t)(y0 - R + i) * W);
    } else {
#pragma unroll
        for (int i = 0; i < 4 + 2 * R; i++) v[i] = __ldg(s + (int64_t)reflect101(y0 - R + i, H) * W);
    }
    const bool fused = (KS == 3) || x < (W & ~7);  // SymmColumnVec_32f covers multiples of 8 lanes
#pragma unroll
    for (int j = 0; j < 4; j++) {
        if (y0 + j >= H) break;
        float acc = __fmul_rn(v[j + R], bt.k[R]);
#pragma unroll
        for (int i = 1; i <= R; i++) {
            const float ac = __fadd_rn(v[j + R + i], v[j + R - i]);
            acc = fused ? fmaf(ac, bt.k[R + i], acc) : __fadd_rn(acc, __fmul_rn(ac, bt.k[R + i]));
        }
        out[((int64_t)b * H + y0 + j) * W + x] = acc;
    }
}

template <typename T>
int launch_blur_rows(const T* in, int64_t in_ss, int64_t in_rs, SlotMap in_map, float* out, int n, int H, int W,
                     const BlurTaps& bt, cudaStream_t st)
{
    const bool win4 = (bt.ksz == 3 || bt.ksz == 9 || bt.ksz == 19 || bt.ksz == 39 || bt.ksz == 79) && W % 4 == 0 &&
                      W >= 4 + bt.ksz && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && H <= 65535;
    for (int b0 = 0; b0 < n; b0 += 65535) {
        int nb = n - b0 < 65535 ? n - b0 : 65535;
        SlotMap m = in_map;
        m.base += b0;
        ProfScope ps(K_BLUR_ROWS, (4.0 + sizeof(T)) * nb * H * W, st);
        if (win4) {
            dim3 grid((unsigned)cdiv(W, 512), (unsigned)H, (unsigned)nb);
            float* o = out + (int64_t)b0 * H * W;
            if (bt.ksz == 3) k_blur_rows4<T, 1><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, o, H, W, bt);
            else if (bt.ksz == 9) k_blur_rows4<T, 4><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, o, H, W, bt);
            else if (bt.ksz == 19) k_blur_rows4<T, 9><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, o, H, W, bt);
            else if (bt.ksz == 39) k_blur_rows4<T, 19><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, o, H, W, bt);
            else k_blur_rows4<T, 39><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, o, H, W, bt);
            FDN_LAUNCHED("k_blur_rows4");
            continue;
        }
        dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)nb);
        k_blur_rows<T><<<grid, 128, 0, st>>>(in, in_ss, in_rs, m, out + (int64_t)b0 * H * W, H, W, bt);
        FDN_LAUNCHED("k_blur_rows");
    }
    return FDN_OK;
}

template int launch_blur_rows<float>(const float*, int64_t, int64_t, SlotMap, float*, int, int, int, const BlurTaps&,
                                     cudaStream_t);
template int launch_blur_rows<uint8_t>(const uint8_t*, int64_t, int64_t, SlotMap, float*, int, int, int, const BlurTaps&,
                                       cudaStream_t);
template int launch_blur_rows<uint16_t>(const uint16_t*, int64_t, int64_t, SlotMap, float*, int, int, int,
                                        const BlurTaps&, cudaStream_t);
template int launch_blur_rows<int16_t>(const int16_t*, int64_t, int64_t, SlotMap, float*, int, int, int, const BlurTaps&,
                                       cudaStream_t);

int launch_blur_cols(const float* in, float* out, int n, int H, int W, const BlurTaps& bt, cudaStream_t st)
{
    const bool win4 = (bt.ksz == 3 || bt.ksz == 9 || bt.ksz == 19 || bt.ksz == 39 || bt.ksz == 79) && H >= 4 + bt.ksz;
    for (int b0 = 0; b0 < n; b0 += 65535) {
        int nb = n - b0 < 65535 ? n - b0 : 65535;
        ProfScope ps(K_BLUR_COLS, 8.0 * nb * H * W, st);
        const float* i_ = in + (int64_t)b0 * H * W;
        float* o_ = out + (int64_t)b0 * H * W;
        if (win4) {
            dim3 grid((unsigned)cdiv(W, 128), (unsigned)cdiv(H, 4), (unsigned)nb);
            if (bt.ksz == 3) k_blur_cols4<1><<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
            else if (bt.ksz == 9) k_blur_cols4<4><<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
            else if (bt.ksz == 19) k_blur_cols4<9><<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
            else if (bt.ksz == 39) k_blur_cols4<19><<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
            else k_blur_cols4<39><<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
            FDN_LAUNCHED("k_blur_cols4");
            continue;
        }
        dim3 grid((unsigned)cdiv(W, 128), (unsigned)H, (unsigned)nb);
        k_blur_cols<<<grid, 128, 0, st>>>(i_, o_, H, W, bt);
        FDN_LAUNCHED("k_blur_cols");
    }
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// resize INTER_LINEAR of the (1-channel) pyramid image, Intel-IPP arithmetic (what the x86 cv2 wheel executes):
// coord = (d + 0.5) * (S / D) - 0.5 in float64, frac = float(coord - floor(coord)), out = fma(b - a, frac, a),
// horizontal first, then vertical (SURVEY App. A.1; probe: bit-exact vs cv2.resize).
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void linear_coord_ipp(int d, int S, int D, int& s0, float& f)
{
    double c = __dsub_rn(__dmul_rn((double)d + 0.5, (double)S / (double)D), 0.5);
    double fl = floor(c);
    s0 = (int)fl;
    f = (float)__dsub_rn(c, fl);
    if (s0 < 0) { f = 0.f; s0 = 0; }
    if (s0 >= S - 1) { f = 0.f; s0 = S - 1; }
}

__global__ void __launch_bounds__(128)
k_resize_linear_img(const float* __restrict__ in, int H, int W, float* __restrict__ out, int64_t out_stride, int h, int w)
{
    const int dx = blockIdx.x * 128 + threadIdx.x;
    const int dy = blockIdx.y;
    const int b = blockIdx.z;
    if (dx >= w) return;
    int sx0, sy0;
    float fx, fy;
    linear_coord_ipp(dx, W, w, sx0, fx);
    linear_coord_ipp(dy, H, h, sy0, fy);
    const int sx1 = min(sx0 + 1, W - 1), sy1 = min(sy0 + 1, H - 1);
    const float* S0 = in + ((int64_t)b * H + sy0) * W;
    const float* S1 = in + ((int64_t)b * H + sy1) * W;
    float r0 = fmaf(__fsub_rn(S0[sx1], S0[sx0]), fx, S0[sx0]);
    float r1 = fmaf(__fsub_rn(S1[sx1], S1[sx0]), fx, S1[sx0]);
    out[(int64_t)b * out_stride + (int64_t)dy * w + dx] = fmaf(__fsub_rn(r1, r0), fy, r0);
}

int launch_resize_linear_img(const float* in, int n, int H, int W, float* out, int64_t out_stride, int h, int w,
                             cudaStream_t st)
{
    for (int b0 = 0; b0 < n; b0 += 65535) {
        int nb = n - b0 < 65535 ? n - b0 : 65535;
        dim3 grid((unsigned)cdiv(w, 128), (unsigned)h, (unsigned)nb);
        ProfScope ps(K_RESIZE_IMG, 4.0 * nb * ((double)H * W + (double)h * w), st);
        k_resize_linear_img<<<grid, 128, 0, st>>>(in + (int64_t)b0 * H * W, H, W, out + (int64_t)b0 * out_stride,
                                                  out_stride, h, w);
        FDN_LAUNCHED("k_resize_linear_img");
    }
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Stage 2: FarnebackPolyExp. Tile of PT x PT outputs per block, input tile with a poly_n halo staged in shared
// memory (replicate border = clamped loads), float32 vertical moments for PT + 2n columns, float64 horizontal
// pass. Output layout: [h*w] float4 (channels 0-3) followed by [h*w] float (channel 4).
// ------------------------------------------------------------------------------------------------
#define PT 32
#define PN_MAX 7

__global__ void __launch_bounds__(256)
k_polyexp(const float* __restrict__ img, int64_t img_stride, float* __restrict__ R, int64_t R_stride, SlotMap R_map,
          int h, int w, PolyConsts pc)
{
    __shared__ float s_in[(PT + 2 * PN_MAX) * (PT + 2 * PN_MAX)];
    __shared__ float s_row[3][PT][PT + 2 * PN_MAX + 1];
    const int n = pc.n;
    const int TW = PT + 2 * n;  // staged tile is TW x TW
    const int x0 = blockIdx.x * PT, y0 = blockIdx.y * PT, b = blockIdx.z;
    const float* src = img + (int64_t)b * img_stride;
    for (int i = threadIdx.x; i < TW * TW; i += 256) {
        int ty = i / TW, tx = i - ty * TW;
        int gy = min(max(y0 - n + ty, 0), h - 1), gx = min(max(x0 - n + tx, 0), w - 1);
        s_in[i] = src[(int64_t)gy * w + gx];
    }
    __syncthreads();
    // vertical pass: PT rows x TW columns
    for (int i = threadIdx.x; i < PT * TW; i += 256) {
        int ty = i / TW, tx = i - ty * TW;
        const float* c = s_in + (ty + n) * TW + tx;
        float t0 = __fmul_rn(c[0], pc.g[0]), t1 = 0.f, t2 = 0.f;
        for (int k = 1; k <= n; k++) {
            float a0 = c[-k * TW], a1 = c[k * TW];
            float p = __fadd_rn(a0, a1);
            t0 = __fadd_rn(t0, __fmul_rn(pc.g[k], p));
            t1 = __fadd_rn(t1, __fmul_rn(pc.xg[k], __fsub_rn(a1, a0)));
            t2 = __fadd_rn(t2, __fmul_rn(pc.xxg[k], p));
        }
        s_row[0][ty][tx] = t0; s_row[1][ty][tx] = t1; s_row[2][ty][tx] = t2;
    }
    __syncthreads();
    // horizontal pass (float64 accumulators; products of two floats stay float exactly as in OpenCV's C++)
    for (int i = threadIdx.x; i < PT * PT; i += 256) {
        int ty = i / PT, tx = i - ty * PT;
        int gy = y0 + ty, gx = x0 + tx;
        if (gy >= h || gx >= w) continue;
        const float* r0 = &s_row[0][ty][tx + n];
        const float* r1 = &s_row[1][ty][tx + n];
        const float* r2 = &s_row[2][ty][tx + n];
        float g0 = pc.g[0];
        double b1 = (double)__fmul_rn(r0[0], g0), b2 = 0, b3 = (double)__fmul_rn(r1[0], g0), b4 = 0,
               b5 = (double)__fmul_rn(r2[0], g0), b6 = 0;
        for (int k = 1; k <= n; k++) {
            double tg = (double)__fadd_rn(r0[k], r0[-k]);
            g0 = pc.g[k];
            b1 = __dadd_rn(b1, __dmul_rn(tg, pc.gd[k]));
            b4 = __dadd_rn(b4, __dmul_rn(tg, pc.xxgd[k]));
            b2 = __dadd_rn(b2, (double)__fmul_rn(__fsub_rn(r0[k], r0[-k]), pc.xg[k]));
            b3 = __dadd_rn(b3, (double)__fmul_rn(__fadd_rn(r1[k], r1[-k]), g0));
            b6 = __dadd_rn(b6, (double)__fmul_rn(__fsub_rn(r1[k], r1[-k]), pc.xg[k]));
            b5 = __dadd_rn(b5, (double)__fmul_rn(__fadd_rn(r2[k], r2[-k]), g0));
        }
        float* dst = R + (int64_t)R_map.slot(b) * R_stride;
        float4 o;
        o.x = (float)__dmul_rn(b3, pc.ig11);
        o.y = (float)__dmul_rn(b2, pc.ig11);
        o.z = (float)__dadd_rn(__dmul_rn(b1, pc.ig03), __dmul_rn(b5, pc.ig33));
        o.w = (float)__dadd_rn(__dmul_rn(b1, pc.ig03), __dmul_rn(b4, pc.ig33));
        reinterpret_cast<float4*>(dst)[(int64_t)gy * w + gx] = o;
        dst[(int64_t)4 * h * w + (int64_t)gy * w + gx] = (float)__dmul_rn(b6, pc.ig55);
    }
}

// ------------------------------------------------------------------------------------------------
// Stage 2 with TMA: the same arithmetic, input tiles brought in by the Tensor Memory Accelerator.
// A block walks along one row of 32x32 output tiles; while it computes tile i, the (32+2n)^2 input box of tile
// i+1 is already in flight (cp.async.bulk.tensor into the other shared-memory buffer, completion on an mbarrier).
// TMA zero-fills out-of-image elements; the replicate border OpenCV uses is applied when the tile is read (clamped
// tile coordinates -- the clamped source always lies inside the same box).
// Needs w % 4 == 0 (16-byte global strides); other widths use k_polyexp.
// ------------------------------------------------------------------------------------------------
// TMA needs the box's innermost start coordinate 16-byte aligned (4 floats) [probe: unaligned starts fault]: the box
// begins PL = 8 columns left of the tile (>= poly_n) instead of poly_n columns.
#define PL 8
#define PBX_MAX ((PL + PT + PN_MAX + 3) & ~3)
#define PBY_MAX (PT + 2 * PN_MAX)

// one thread arms the mbarrier with the byte count and starts the 3-D bulk tensor copy (box -> shared memory)
__device__ __forceinline__ void tma_load_box(uint64_t tmap_addr, uint32_t dst, uint32_t bar, uint32_t bytes, int cx,
                                             int cy, int cz)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        :: "r"(dst), "l"(tmap_addr), "r"(cx), "r"(cy), "r"(cz), "r"(bar) : "memory");
}

// NC > 0: poly_n known at compile time (5, the reference's constant): tile pitches, the divisions by them and the tap
// loops fold; NC == 0: generic.
template <int NC>
__global__ void __launch_bounds__(256)
k_polyexp_tma(const __grid_constant__ CUtensorMap tmap, float* __restrict__ R, int64_t R_stride, SlotMap R_map, int h,
              int w, PolyConsts pc)
{
    __shared__ __align__(128) float s_in[2][PBY_MAX * PBX_MAX];
    __shared__ float s_row[3][PT][PT + 2 * PN_MAX + 1];
    __shared__ __align__(8) unsigned long long s_bar[2];
    const int n = NC > 0 ? NC : pc.n;
    const int TW = PT + 2 * n;           // columns / rows actually used
    const int BX = (PL + PT + n + 3) & ~3;   // box width (multiple of 4 floats = 16 bytes), the tile's row pitch
    const int y0 = blockIdx.y * PT, b = blockIdx.z;
    const int ntiles = (w + PT - 1) / PT;
    const uint32_t box_bytes = (uint32_t)(BX * TW * sizeof(float));
    const uint32_t bar0 = smem_u32(&s_bar[0]), bar1 = smem_u32(&s_bar[1]);

    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar0));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar1));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // the descriptor must be addressed in the kernel-parameter (constant) space: take the address here, not through
    // a by-reference capture (a local copy of the 128-byte map would make the bulk copy fault)
    const uint64_t tmap_addr = reinterpret_cast<uint64_t>(&tmap);
    const uint32_t dst0 = smem_u32(&s_in[0][0]), dst1 = smem_u32(&s_in[1][0]);
    if (threadIdx.x == 0) tma_load_box(tmap_addr, dst0, bar0, box_bytes, -PL, y0 - n, b);

    float* dstR = R + (int64_t)R_map.slot(b) * R_stride;
    for (int tile = 0; tile < ntiles; tile++) {
        const int buf = tile & 1;
        if (threadIdx.x == 0 && tile + 1 < ntiles)   // prefetch the next tile into the other buffer
            tma_load_box(tmap_addr, buf ? dst0 : dst1, buf ? bar0 : bar1, box_bytes, (tile + 1) * PT - PL, y0 - n, b);
        mbar_wait(buf ? bar1 : bar0, (uint32_t)((tile >> 1) & 1));
        const float* tin = s_in[buf];
        const int x0 = tile * PT;
        const int gx0 = x0 - PL, gy0 = y0 - n;   // global coordinates of the box origin
        const bool border = x0 - n < 0 || gy0 < 0 || x0 + PT + n > w || gy0 + TW > h;
        // vertical pass: PT rows x TW columns
        for (int i = threadIdx.x; i < PT * TW; i += 256) {
            const int ty = i / TW, tx = i - ty * TW;
            float t0, t1 = 0.f, t2 = 0.f;
            if (!border) {
                const float* c = tin + (ty + n) * BX + tx + (PL - n);
                t0 = __fmul_rn(c[0], pc.g[0]);
#pragma unroll
    #pragma unroll
            for (int k = 1; k <= n; k++) {
                    const float a0 = c[-k * BX], a1 = c[k * BX];
                    const float p = __fadd_rn(a0, a1);
                    t0 = __fadd_rn(t0, __fmul_rn(pc.g[k], p));
                    t1 = __fadd_rn(t1, __fmul_rn(pc.xg[k], __fsub_rn(a1, a0)));
                    t2 = __fadd_rn(t2, __fmul_rn(pc.xxg[k], p));
                }
            } else {  // replicate: clamp the GLOBAL coordinate, then address the box
                const int cx = min(max(x0 - n + tx, 0), w - 1) - gx0;
                const int gy = gy0 + ty + n;
                const float* col = tin + cx;
                t0 = __fmul_rn(col[(min(max(gy, 0), h - 1) - gy0) * BX], pc.g[0]);
#pragma unroll
    #pragma unroll
            for (int k = 1; k <= n; k++) {
                    const float a0 = col[(min(max(gy - k, 0), h - 1) - gy0) * BX];
                    const float a1 = col[(min(max(gy + k, 0), h - 1) - gy0) * BX];
                    const float p = __fadd_rn(a0, a1);
                    t0 = __fadd_rn(t0, __fmul_rn(pc.g[k], p));
                    t1 = __fadd_rn(t1, __fmul_rn(pc.xg[k], __fsub_rn(a1, a0)));
                    t2 = __fadd_rn(t2, __fmul_rn(pc.xxg[k], p));
                }
            }
            s_row[0][ty][tx] = t0; s_row[1][ty][tx] = t1; s_row[2][ty][tx] = t2;
        }
        __syncthreads();
        // horizontal pass (identical to k_polyexp)
        for (int i = threadIdx.x; i < PT * PT; i += 256) {
            const int ty = i / PT, tx = i - ty * PT;
            const int gy = y0 + ty, gx = x0 + tx;
            if (gy >= h || gx >= w) continue;
            const float* r0 = &s_row[0][ty][tx + n];
            const float* r1 = &s_row[1][ty][tx + n];
            const float* r2 = &s_row[2][ty][tx + n];
            float g0 = pc.g[0];
            double b1 = (double)__fmul_rn(r0[0], g0), b2 = 0, b3 = (double)__fmul_rn(r1[0], g0), b4 = 0,
                   b5 = (double)__fmul_rn(r2[0], g0), b6 = 0;
#pragma unroll
            for (int k = 1; k <= n; k++) {
                const double tg = (double)__fadd_rn(r0[k], r0[-k]);
                g0 = pc.g[k];
                b1 = __dadd_rn(b1, __dmul_rn(tg, pc.gd[k]));
                b4 = __dadd_rn(b4, __dmul_rn(tg, pc.xxgd[k]));
                b2 = __dadd_rn(b2, (double)__fmul_rn(__fsub_rn(r0[k], r0[-k]), pc.xg[k]));
                b3 = __dadd_rn(b3, (double)__fmul_rn(__fadd_rn(r1[k], r1[-k]), g0));
                b6 = __dadd_rn(b6, (double)__fmul_rn(__fsub_rn(r1[k], r1[-k]), pc.xg[k]));
                b5 = __dadd_rn(b5, (double)__fmul_rn(__fadd_rn(r2[k], r2[-k]), g0));
            }
            float4 o;
            o.x = (float)__dmul_rn(b3, pc.ig11);
            o.y = (float)__dmul_rn(b2, pc.ig11);
            o.z = (float)__dadd_rn(__dmul_rn(b1, pc.ig03), __dmul_rn(b5, pc.ig33));
            o.w = (float)__dadd_rn(__dmul_rn(b1, pc.ig03), __dmul_rn(b4, pc.ig33));
            reinterpret_cast<float4*>(dstR)[(int64_t)gy * w + gx] = o;
            dstR[(int64_t)4 * h * w + (int64_t)gy * w + gx] = (float)__dmul_rn(b6, pc.ig55);
        }
        __syncthreads();   // s_row and s_in[buf] are free again (the copy issued two tiles later reuses s_in[buf])
    }
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link-time dependency on libcuda)
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode_tiled()
{
    static PFN_encodeTiled fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

static bool g_polyexp_use_tma = true;   // FDN_POLYEXP_TMA=0 disables (A/B timing, tests exercise both)

int launch_polyexp(const float* img, int64_t img_stride, float* R, int64_t R_stride, SlotMap R_map, int n, int h,
                   int w, const PolyConsts& pc, cudaStream_t st)
{
    if (pc.n < 1 || pc.n > PN_MAX) {
        set_error("poly_n %d unsupported (1..%d)", pc.n, PN_MAX);
        return FDN_ERR_INVALID;
    }
    static bool env_read = false;
    if (!env_read) {
        env_read = true;
        const char* e = getenv("FDN_POLYEXP_TMA");
        if (e && atoi(e) == 0) g_polyexp_use_tma = false;
    }
    PFN_encodeTiled enc = g_polyexp_use_tma ? get_encode_tiled() : nullptr;
    const bool tma_ok = enc && w % 4 == 0 && img_stride == (int64_t)h * w && w >= 4 &&
                        (reinterpret_cast<uintptr_t>(img) & 15) == 0 && n <= 65535 && cdiv(h, PT) <= 65535;
    if (tma_ok) {
        const int TW = PT + 2 * pc.n;
        CUtensorMap tmap;
        const cuuint64_t gdim[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
        const cuuint64_t gstr[2] = {(cuuint64_t)w * 4, (cuuint64_t)h * w * 4};
        const cuuint32_t box[3] = {(cuuint32_t)((PL + PT + pc.n + 3) & ~3), (cuuint32_t)TW, 1};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult cr = enc(&tmap, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(img), gdim, gstr, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (cr == CUDA_SUCCESS) {
            dim3 grid(1, (unsigned)cdiv(h, PT), (unsigned)n);
            ProfScope ps(K_POLYEXP, 24.0 * n * h * w, st);
            if (pc.n == 5) k_polyexp_tma<5><<<grid, 256, 0, st>>>(tmap, R, R_stride, R_map, h, w, pc);
            else k_polyexp_tma<0><<<grid, 256, 0, st>>>(tmap, R, R_stride, R_map, h, w, pc);
            FDN_LAUNCHED("k_polyexp_tma");
            return FDN_OK;
        }
    }
    for (int b0 = 0; b0 < n; b0 += 65535) {
        int nb = n - b0 < 65535 ? n - b0 : 65535;
        SlotMap m = R_map;
        m.base += b0;
        dim3 grid((unsigned)cdiv(w, PT), (unsigned)cdiv(h, PT), (unsigned)nb);
        ProfScope ps(K_POLYEXP, 24.0 * nb * h * w, st);
        k_polyexp<<<grid, 256, 0, st>>>(img + (int64_t)b0 * img_stride, img_stride, R, R_stride, m, h, w, pc);
        FDN_LAUNCHED("k_polyexp");
    }
    return FDN_OK;
}

}  // namespace fdn
