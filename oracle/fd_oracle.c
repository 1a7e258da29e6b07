/*
 * fd_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE ONLY, never shipped, never on the product path).
 *
 * Plain-C restatement of the hot path of microscopy-processing/FlowDenoising
 * (src/flowdenoising.py) and of the third-party numerics it calls:
 *
 *   - OpenCV 4.13.0 (opencv-python-headless 4.13.0.92; NOT vendored in /root/reference and
 *     unpinned by src/requirements.txt:2):
 *       cv2.calcOpticalFlowFarneback   (call sites src/flowdenoising.py:69-79, :98-108)
 *       cv2.remap                      (call site  src/flowdenoising.py:60-62)
 *     restated from OpenCV's published algorithm (modules/video/src/optflowgf.cpp,
 *     modules/imgproc/src/{imgwarp,resize,smooth}.cpp) as specified in SURVEY.md App. A.
 *   - SciPy 1.18.1 scipy.ndimage.gaussian_filter1d (call site src/flowdenoising.py:41).
 *
 * Parity pinning: the reference has NO tests/golden vectors for this path (SURVEY.md §4), so
 * this oracle is pinned against (a) outputs of the unmodified reference run in the build
 * container (tests/golden/*.npz, made by oracle/gen_golden.py) and (b) live cv2 calls
 * (tests/test_oracle_*.py).
 *
 * Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may
 * load this file's library.
 *
 * Build: see oracle/Makefile (gcc -O2 -ffp-contract=off -fopenmp -shared -fPIC).
 * -ffp-contract=off matters: the baseline OpenCV code is built for SSE3 without FMA, the few
 * places where OpenCV's AVX2 dispatch does use FMA call fmaf() explicitly below.
 *
 * Layouts: images are dense row-major float32; R and M are (H, W, 5) interleaved exactly like
 * OpenCV's CV_32FC(5); flow is (H, W, 2) with the x component first.
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#include <float.h>

#define FDO_API __attribute__((visibility("default")))

static inline int imin(int a, int b) { return a < b ? a : b; }
static inline int imax(int a, int b) { return a > b ? a : b; }
static inline int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
/* cvRound: round half to even (SSE cvtsd2si under the default rounding mode). */
static inline int cv_round(double v) { return (int)lrint(v); }
static inline int cv_floor(double v) { int i = (int)v; return i - (i > v); }
static inline int cv_ceil(double v) { int i = (int)v; return i + (i < v); }
/* BORDER_REFLECT_101 index */
static inline int reflect101(int p, int len)
{
    if (len == 1) return 0;
    while (p < 0 || p >= len) {
        if (p < 0) p = -p;
        else p = 2 * (len - 1) - p;
    }
    return p;
}

/* (a1, get_gaussian_kernel, is the reference's own SciPy loop in fd_oracle.py: NumPy's exp is not the C
 * library's in the last bit, so a C restatement of the taps would not be the reference's taps.) */

/* ------------------------------------------------------------------------------------------
 * cv::getGaussianKernel(ksz, sigma, CV_32F): double taps, normalised, stored as float.
 * sigma <= 0 -> the fixed small kernels ([0.25, 0.5, 0.25] for ksz == 3) (SURVEY App. A.1).
 * ------------------------------------------------------------------------------------------ */
static void cv_gaussian_kernel_f32(int n, double sigma, float* k)
{
    static const float small3[3] = {0.25f, 0.5f, 0.25f};
    if (sigma <= 0 && n == 3) { memcpy(k, small3, sizeof small3); return; }
    double sx = sigma > 0 ? sigma : ((n - 1) * 0.5 - 1) * 0.3 + 0.8;
    double scale2x = -0.5 / (sx * sx);
    double sum = 0;
    double* t = (double*)malloc(sizeof(double) * n);
    for (int i = 0; i < n; i++) {
        double x = i - (n - 1) * 0.5;
        t[i] = exp(scale2x * x * x);
        sum += t[i];
    }
    sum = 1. / sum;
    for (int i = 0; i < n; i++) k[i] = (float)(t[i] * sum);
    free(t);
}

/* ------------------------------------------------------------------------------------------
 * cv::GaussianBlur(f32, (ksz,ksz), sigma), BORDER_REFLECT_101 (SURVEY App. A.1).
 * Separable: row (horizontal) filter then column (vertical) filter, both float32.
 * Arithmetic order follows what OpenCV's AVX2-dispatched filters produce on x86 [probe, round
 * 1, bit-exact vs cv2 4.13.0 on widths that are multiples of 8]: the row filter accumulates
 * taps left to right with fused multiply-add (ksz > 5; ksz == 3 uses fma(c,k0,(l+r)*k1)), the
 * column filter uses the symmetric form k0*c + sum_i k_i*(a_{+i} + a_{-i}) with fused
 * multiply-add. cv2 itself differs in the last ulp between its own SIMD and scalar paths
 * (cv2.setUseOptimized), so for other widths/hosts this is "the same maths to 1 ulp".
 * ------------------------------------------------------------------------------------------ */
FDO_API void fdo_gauss_blur(const float* src, int H, int W, int ksz, double sigma, float* dst)
{
    int r = ksz / 2;
    float* k = (float*)malloc(sizeof(float) * ksz);
    cv_gaussian_kernel_f32(ksz, sigma, k);
    float* tmp = (float*)malloc(sizeof(float) * (size_t)H * W);
    /* Vector loops fuse multiply-add, OpenCV's scalar tails do not. The row filter's vector loops
       (8 + 4 lanes under AVX2) cover columns < W&~3, the column filter's cover columns < W&~7
       [probe: widths 77, 90, 300, 333 bit-exact vs cv2 4.13.0 on an AVX2 host]. */
    int wrow = W & ~3, wcol = W & ~7;
    for (int y = 0; y < H; y++) {
        const float* s = src + (size_t)y * W;
        float* d = tmp + (size_t)y * W;
        for (int x = 0; x < W; x++) {
            float acc;
            if (ksz == 3) {
                /* SymmRowSmallVec_32f: fma(centre, k0, (left + right) * k1); the scalar tail is
                   contracted the other way round: fma(left + right, k1, centre * k0); for ksz == 3 only
                   a last odd column is scalar */
                float lr = s[reflect101(x - 1, W)] + s[reflect101(x + 1, W)];
                acc = x < (W & ~1) ? fmaf(s[x], k[1], lr * k[0]) : fmaf(lr, k[0], s[x] * k[1]);
            } else if (x < wrow) {
                acc = s[reflect101(x - r, W)] * k[0];
                for (int i = 1; i < ksz; i++)
                    acc = fmaf(s[reflect101(x - r + i, W)], k[i], acc);
            } else {
                acc = s[reflect101(x - r, W)] * k[0];
                for (int i = 1; i < ksz; i++)
                    acc = acc + s[reflect101(x - r + i, W)] * k[i];
            }
            d[x] = acc;
        }
    }
    for (int y = 0; y < H; y++) {
        float* d = dst + (size_t)y * W;
        const float* c = tmp + (size_t)y * W;
        for (int x = 0; x < W; x++) {
            float acc = c[x] * k[r];
            for (int i = 1; i <= r; i++) {
                float a = tmp[(size_t)reflect101(y + i, H) * W + x];
                float b = tmp[(size_t)reflect101(y - i, H) * W + x];
                if (ksz == 3 || x < wcol) acc = fmaf(a + b, k[r + i], acc);
                else acc = acc + (a + b) * k[r + i];
            }
            d[x] = acc;
        }
    }
    free(tmp);
    free(k);
}

/* ------------------------------------------------------------------------------------------
 * cv::resize(..., INTER_LINEAR) for float32 with cn interleaved channels (SURVEY App. A.1).
 * Half-pixel centres, source index clamped with the fractional weight zeroed at the borders;
 * horizontal pass first, then vertical, float32 throughout.
 *
 * Two arithmetic variants exist inside the cv2 wheel the reference runs on [probe, round 1]:
 *   ipp = 0  OpenCV's own resizeGeneric_: frac = (float)coord - floor, out = a*(1-f) + b*f.
 *            Bit-exact vs cv2 with cv2.ipp.setUseIPP(False), and vs cv2 (IPP on) for 2-channel
 *            images (the flow up-sampling, which IPP does not take).
 *   ipp = 1  the Intel IPP HAL that the x86 wheel uses for 1-channel float images (the pyramid
 *            images): frac = (float)(coord - floor(coord)) with coord in float64,
 *            out = fma(b - a, f, a). Bit-exact vs cv2 with IPP on (its default).
 * ------------------------------------------------------------------------------------------ */
static void linear_tab(int ssize, int dsize, int* ofs, float* frac, int ipp, int vertical)
{
    double inv_scale = (double)dsize / ssize;
    double scale = ipp ? (double)ssize / dsize : 1. / inv_scale;
    for (int d = 0; d < dsize; d++) {
        double c = (d + 0.5) * scale - 0.5;
        int s;
        float f;
        if (ipp) {
            double fl = floor(c);
            s = (int)fl;
            f = (float)(c - fl);
        } else {
            f = (float)c;
            s = cv_floor(f);
            f -= s;
        }
        /* OpenCV's own code zeroes the fraction at the borders only horizontally; vertically it
           keeps (1-f, f) and clips each of the two row indices (so a border row is S*(1-f) + S*f). */
        if (ipp || !vertical) {
            if (s < 0) { f = 0; s = 0; }
            if (s >= ssize - 1) { f = 0; s = ssize - 1; }
        }
        ofs[d] = s;
        frac[d] = f;
    }
}

FDO_API void fdo_resize_linear(const float* src, int H, int W, int cn, float* dst, int h, int w,
                               int ipp)
{
    if (h == H && w == W) { memcpy(dst, src, sizeof(float) * (size_t)H * W * cn); return; }
    int* xo = (int*)malloc(sizeof(int) * w);
    float* xf = (float*)malloc(sizeof(float) * w);
    int* yo = (int*)malloc(sizeof(int) * h);
    float* yf = (float*)malloc(sizeof(float) * h);
    linear_tab(W, w, xo, xf, ipp, 0);
    linear_tab(H, h, yo, yf, ipp, 1);
    float* r0 = (float*)malloc(sizeof(float) * (size_t)w * cn);
    float* r1 = (float*)malloc(sizeof(float) * (size_t)w * cn);
    for (int dy = 0; dy < h; dy++) {
        int sy0 = clampi(yo[dy], 0, H - 1), sy1 = clampi(yo[dy] + 1, 0, H - 1);
        const float* S0 = src + (size_t)sy0 * W * cn;
        const float* S1 = src + (size_t)sy1 * W * cn;
        for (int dx = 0; dx < w; dx++) {
            int sx0 = xo[dx], sx1 = imin(sx0 + 1, W - 1);
            float a1 = xf[dx], a0 = 1.f - a1;
            for (int c = 0; c < cn; c++) {
                if (ipp) {
                    r0[dx * cn + c] = fmaf(S0[sx1 * cn + c] - S0[sx0 * cn + c], a1, S0[sx0 * cn + c]);
                    r1[dx * cn + c] = fmaf(S1[sx1 * cn + c] - S1[sx0 * cn + c], a1, S1[sx0 * cn + c]);
                } else {
                    r0[dx * cn + c] = S0[sx0 * cn + c] * a0 + S0[sx1 * cn + c] * a1;
                    r1[dx * cn + c] = S1[sx0 * cn + c] * a0 + S1[sx1 * cn + c] * a1;
                }
            }
        }
        float b1 = yf[dy], b0 = 1.f - b1;
        float* D = dst + (size_t)dy * w * cn;
        if (ipp)
            for (int i = 0; i < w * cn; i++) D[i] = fmaf(r1[i] - r0[i], b1, r0[i]);
        else
            for (int i = 0; i < w * cn; i++) D[i] = r0[i] * b0 + r1[i] * b1;
    }
    free(r0); free(r1); free(xo); free(xf); free(yo); free(yf);
}

/* ------------------------------------------------------------------------------------------
 * cv::resize(..., INTER_AREA) for float32, cn interleaved channels, downscale or same size
 * (used only for the initial flow, SURVEY App. A.0-3).
 * Integer ratios: plain block sum (row-major order) times 1/area in float32.
 * Other ratios: fractional-coverage tables (computeResizeAreaTab), horizontal accumulation per
 * source row, then beta-weighted accumulation over source rows.
 * ------------------------------------------------------------------------------------------ */
typedef struct { int si, di; float alpha; } area_tab_t;

static int area_tab(int ssize, int dsize, double scale, area_tab_t* tab)
{
    int k = 0;
    for (int dx = 0; dx < dsize; dx++) {
        double fsx1 = dx * scale;
        double fsx2 = fsx1 + scale;
        double cellWidth = fmin(scale, ssize - fsx1);
        int sx1 = cv_ceil(fsx1), sx2 = cv_floor(fsx2);
        sx2 = imin(sx2, ssize - 1);
        sx1 = imin(sx1, sx2);
        if (sx1 - fsx1 > 1e-3) {
            tab[k].di = dx; tab[k].si = sx1 - 1;
            tab[k++].alpha = (float)((sx1 - fsx1) / cellWidth);
        }
        for (int sx = sx1; sx < sx2; sx++) {
            tab[k].di = dx; tab[k].si = sx;
            tab[k++].alpha = (float)(1.0 / cellWidth);
        }
        if (fsx2 - sx2 > 1e-3) {
            tab[k].di = dx; tab[k].si = sx2;
            tab[k++].alpha = (float)(fmin(fmin(fsx2 - sx2, 1.), cellWidth) / cellWidth);
        }
    }
    return k;
}

FDO_API void fdo_resize_area(const float* src, int H, int W, int cn, float* dst, int h, int w)
{
    if (h == H && w == W) { memcpy(dst, src, sizeof(float) * (size_t)H * W * cn); return; }
    double scale_x = 1. / ((double)w / W), scale_y = 1. / ((double)h / H);
    int isx = cv_round(scale_x), isy = cv_round(scale_y); /* saturate_cast<int>(double) */
    int fast = fabs(scale_x - isx) < DBL_EPSILON && fabs(scale_y - isy) < DBL_EPSILON;
    if (fast) {
        int area = isx * isy;
        float scale = 1.f / area;
        float* v = (float*)malloc(sizeof(float) * (size_t)area);
        for (int dy = 0; dy < h; dy++)
            for (int dx = 0; dx < w; dx++)
                for (int c = 0; c < cn; c++) {
                    float sum = 0;
                    {
                        int k = 0;
                        for (int sy = 0; sy < isy; sy++)
                            for (int sx = 0; sx < isx; sx++)
                                v[k++] = src[((size_t)(dy * isy + sy) * W + dx * isx + sx) * cn + c];
                        /* OpenCV's generic loop is unrolled by four (CV_ENABLE_UNROLLED) */
                        for (k = 0; k <= area - 4; k += 4) sum += v[k] + v[k + 1] + v[k + 2] + v[k + 3];
                        for (; k < area; k++) sum += v[k];
                    }
                    dst[((size_t)dy * w + dx) * cn + c] = sum * scale;
                }
        free(v);
        return;
    }
    area_tab_t* xt = (area_tab_t*)malloc(sizeof(area_tab_t) * (size_t)(W * 2 + 2));
    area_tab_t* yt = (area_tab_t*)malloc(sizeof(area_tab_t) * (size_t)(H * 2 + 2));
    int nx = area_tab(W, w, scale_x, xt);
    int ny = area_tab(H, h, scale_y, yt);
    float* buf = (float*)malloc(sizeof(float) * (size_t)w * cn);
    float* sum = (float*)calloc((size_t)w * cn, sizeof(float));
    int prev_dy = yt[0].di;
    for (int j = 0; j < ny; j++) {
        float beta = yt[j].alpha;
        int dy = yt[j].di, sy = yt[j].si;
        const float* S = src + (size_t)sy * W * cn;
        for (int i = 0; i < w * cn; i++) buf[i] = 0.f;
        for (int k = 0; k < nx; k++) {
            float alpha = xt[k].alpha;
            for (int c = 0; c < cn; c++)
                buf[xt[k].di * cn + c] = buf[xt[k].di * cn + c] + S[xt[k].si * cn + c] * alpha;
        }
        if (dy != prev_dy) {
            float* D = dst + (size_t)prev_dy * w * cn;
            for (int i = 0; i < w * cn; i++) { D[i] = sum[i]; sum[i] = beta * buf[i]; }
            prev_dy = dy;
        } else {
            for (int i = 0; i < w * cn; i++) sum[i] += beta * buf[i];
        }
    }
    {
        float* D = dst + (size_t)prev_dy * w * cn;
        for (int i = 0; i < w * cn; i++) D[i] = sum[i];
    }
    free(buf); free(sum); free(xt); free(yt);
}

/* ------------------------------------------------------------------------------------------
 * FarnebackPrepareGaussian + FarnebackPolyExp (SURVEY App. A.2).
 * ------------------------------------------------------------------------------------------ */
typedef struct {
    int n;
    float g[32], xg[32], xxg[32]; /* index k = 0..n (symmetric / antisymmetric) */
    double ig11, ig03, ig33, ig55;
} polyexp_consts_t;

/* cv::invert(G, DECOMP_CHOLESKY) for the 6x6 float64 Gram matrix: OpenCV's own CholImpl (hal::Cholesky64f falls
   through to it for small matrices) applied to an identity right-hand side. Reproduced operation by operation:
   a closed-form inverse differs in the last bit of ig03 / ig33, which flips the float32 rounding of one R value
   in ~1e7 (enough to show up against cv2 on large images) [probe, round 1]. */
static void chol_inv6(const double G[6][6], double inv[6][6])
{
    enum { m = 6 };
    double L[6][6], b[6][6];
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) { L[i][j] = G[i][j]; b[i][j] = i == j ? 1. : 0.; }
    for (int i = 0; i < m; i++) {
        double s;
        for (int j = 0; j < i; j++) {
            s = L[i][j];
            for (int k = 0; k < j; k++) s -= L[i][k] * L[j][k];
            L[i][j] = s * L[j][j];
        }
        s = L[i][i];
        for (int k = 0; k < i; k++) { double t = L[i][k]; s -= t * t; }
        L[i][i] = 1. / sqrt(s);
    }
    for (int i = 0; i < m; i++)
        for (int j = 0; j < m; j++) {
            double s = b[i][j];
            for (int k = 0; k < i; k++) s -= L[i][k] * b[k][j];
            b[i][j] = s * L[i][i];
        }
    for (int i = m - 1; i >= 0; i--)
        for (int j = 0; j < m; j++) {
            double s = b[i][j];
            for (int k = m - 1; k > i; k--) s -= L[k][i] * b[k][j];
            b[i][j] = s * L[i][i];
        }
    memcpy(inv, b, sizeof b);
}

static void polyexp_prepare(int n, double sigma, polyexp_consts_t* pc)
{
    if (sigma < FLT_EPSILON) sigma = n * 0.3;
    float g[65], xg[65], xxg[65];
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
            G11 += gg * x * x;             /* float*int*int evaluated left to right in float */
            G33 += gg * x * x * x * x;
            G55 += gg * x * x * y * y;
        }
    double G[6][6], inv[6][6];
    memset(G, 0, sizeof G);
    G[0][0] = G00; G[1][1] = G11; G[3][3] = G33; G[5][5] = G55;
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    chol_inv6(G, inv);
    pc->ig11 = inv[1][1];
    pc->ig03 = inv[0][3];
    pc->ig33 = inv[3][3];
    pc->ig55 = inv[5][5];
    pc->n = n;
    for (int k = 0; k <= n; k++) { pc->g[k] = g[n + k]; pc->xg[k] = xg[n + k]; pc->xxg[k] = xxg[n + k]; }
}

FDO_API void fdo_polyexp_consts(int n, double sigma, float* g, float* xg, float* xxg, double* ig)
{
    polyexp_consts_t pc;
    polyexp_prepare(n, sigma, &pc);
    for (int k = 0; k <= n; k++) { g[k] = pc.g[k]; xg[k] = pc.xg[k]; xxg[k] = pc.xxg[k]; }
    ig[0] = pc.ig11; ig[1] = pc.ig03; ig[2] = pc.ig33; ig[3] = pc.ig55;
}

FDO_API void fdo_polyexp(const float* src, int H, int W, int n, double sigma, float* dst)
{
    polyexp_consts_t pc;
    polyexp_prepare(n, sigma, &pc);
    float* rowbuf = (float*)malloc(sizeof(float) * (size_t)(W + n * 2) * 3);
    float* row = rowbuf + n * 3;
    for (int y = 0; y < H; y++) {
        float g0 = pc.g[0], g1, g2;
        const float* srow0 = src + (size_t)y * W;
        const float* srow1;
        float* drow = dst + (size_t)y * W * 5;
        for (int x = 0; x < W; x++) {
            row[x * 3] = srow0[x] * g0;
            row[x * 3 + 1] = row[x * 3 + 2] = 0.f;
        }
        for (int k = 1; k <= n; k++) {
            g0 = pc.g[k]; g1 = pc.xg[k]; g2 = pc.xxg[k];
            srow0 = src + (size_t)imax(y - k, 0) * W;
            srow1 = src + (size_t)imin(y + k, H - 1) * W;
            for (int x = 0; x < W; x++) {
                float p = srow0[x] + srow1[x];
                float t0 = row[x * 3] + g0 * p;
                float t1 = row[x * 3 + 1] + g1 * (srow1[x] - srow0[x]);
                float t2 = row[x * 3 + 2] + g2 * p;
                row[x * 3] = t0; row[x * 3 + 1] = t1; row[x * 3 + 2] = t2;
            }
        }
        for (int x = 0; x < n * 3; x++) {
            row[-1 - x] = row[2 - x];
            row[W * 3 + x] = row[W * 3 + x - 3];
        }
        for (int x = 0; x < W; x++) {
            g0 = pc.g[0];
            double b1 = row[x * 3] * g0, b2 = 0, b3 = row[x * 3 + 1] * g0,
                   b4 = 0, b5 = row[x * 3 + 2] * g0, b6 = 0;
            for (int k = 1; k <= n; k++) {
                double tg = row[(x + k) * 3] + row[(x - k) * 3];
                g0 = pc.g[k];
                b1 += tg * g0;
                b4 += tg * pc.xxg[k];
                b2 += (row[(x + k) * 3] - row[(x - k) * 3]) * pc.xg[k];
                b3 += (row[(x + k) * 3 + 1] + row[(x - k) * 3 + 1]) * g0;
                b6 += (row[(x + k) * 3 + 1] - row[(x - k) * 3 + 1]) * pc.xg[k];
                b5 += (row[(x + k) * 3 + 2] + row[(x - k) * 3 + 2]) * g0;
            }
            drow[x * 5 + 1] = (float)(b2 * pc.ig11);
            drow[x * 5] = (float)(b3 * pc.ig11);
            drow[x * 5 + 3] = (float)(b1 * pc.ig03 + b4 * pc.ig33);
            drow[x * 5 + 2] = (float)(b1 * pc.ig03 + b5 * pc.ig33);
            drow[x * 5 + 4] = (float)(b6 * pc.ig55);
        }
    }
    free(rowbuf);
}

/* ------------------------------------------------------------------------------------------
 * FarnebackUpdateMatrices (SURVEY App. A.3), rows [y0, y1).
 * ------------------------------------------------------------------------------------------ */
FDO_API void fdo_update_matrices(const float* R0a, const float* R1, const float* flowa,
                                 int H, int W, float* Ma, int y0, int y1)
{
    static const float border[5] = {0.14f, 0.14f, 0.4472f, 0.4472f, 0.4472f};
    const int BORDER = 5;
    size_t step1 = (size_t)W * 5;
    for (int y = y0; y < y1; y++) {
        const float* flow = flowa + (size_t)y * W * 2;
        const float* R0 = R0a + (size_t)y * W * 5;
        float* M = Ma + (size_t)y * W * 5;
        for (int x = 0; x < W; x++) {
            float dx = flow[x * 2], dy = flow[x * 2 + 1];
            float fx = x + dx, fy = y + dy;
            int x1 = cv_floor(fx), yy1 = cv_floor(fy);
            float r2, r3, r4, r5, r6;
            fx -= x1; fy -= yy1;
            if ((unsigned)x1 < (unsigned)(W - 1) && (unsigned)yy1 < (unsigned)(H - 1)) {
                const float* ptr = R1 + (size_t)yy1 * step1 + (size_t)x1 * 5;
                float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy),
                      a10 = (1.f - fx) * fy, a11 = fx * fy;
                r2 = a00 * ptr[0] + a01 * ptr[5] + a10 * ptr[step1] + a11 * ptr[step1 + 5];
                r3 = a00 * ptr[1] + a01 * ptr[6] + a10 * ptr[step1 + 1] + a11 * ptr[step1 + 6];
                r4 = a00 * ptr[2] + a01 * ptr[7] + a10 * ptr[step1 + 2] + a11 * ptr[step1 + 7];
                r5 = a00 * ptr[3] + a01 * ptr[8] + a10 * ptr[step1 + 3] + a11 * ptr[step1 + 8];
                r6 = a00 * ptr[4] + a01 * ptr[9] + a10 * ptr[step1 + 4] + a11 * ptr[step1 + 9];
                r4 = (R0[x * 5 + 2] + r4) * 0.5f;
                r5 = (R0[x * 5 + 3] + r5) * 0.5f;
                r6 = (R0[x * 5 + 4] + r6) * 0.25f;
            } else {
                r2 = r3 = 0.f;
                r4 = R0[x * 5 + 2];
                r5 = R0[x * 5 + 3];
                r6 = R0[x * 5 + 4] * 0.5f;
            }
            r2 = (R0[x * 5] - r2) * 0.5f;
            r3 = (R0[x * 5 + 1] - r3) * 0.5f;
            r2 += r4 * dy + r6 * dx;
            r3 += r6 * dy + r5 * dx;
            if ((unsigned)(x - BORDER) >= (unsigned)(W - BORDER * 2) ||
                (unsigned)(y - BORDER) >= (unsigned)(H - BORDER * 2)) {
                float scale = (x < BORDER ? border[x] : 1.f) *
                              (x >= W - BORDER ? border[W - x - 1] : 1.f) *
                              (y < BORDER ? border[y] : 1.f) *
                              (y >= H - BORDER ? border[H - y - 1] : 1.f);
                r2 *= scale; r3 *= scale; r4 *= scale; r5 *= scale; r6 *= scale;
            }
            M[x * 5] = r4 * r4 + r6 * r6;
            M[x * 5 + 1] = (r4 + r5) * r6;
            M[x * 5 + 2] = r5 * r5 + r6 * r6;
            M[x * 5 + 3] = r4 * r2 + r6 * r3;
            M[x * 5 + 4] = r6 * r2 + r5 * r3;
        }
    }
}

/* ------------------------------------------------------------------------------------------
 * FarnebackUpdateFlow_Blur (SURVEY App. A.4): (2m+1)^2 box mean of M with replicate borders,
 * float64 sliding sums (the vertical slide adds the float32 difference of two rows), then the
 * regularised 2x2 solve. M is NOT refreshed here (the caller does full sweeps; OpenCV's
 * striped refresh is equivalent, SURVEY App. A.0-5).
 * ------------------------------------------------------------------------------------------ */
FDO_API void fdo_blur_solve(const float* Ma, int H, int W, int win, float* flowa)
{
    int m = win / 2;
    double scale = 1. / (win * win);
    double* vbuf = (double*)malloc(sizeof(double) * (size_t)(W + m * 2 + 2) * 5);
    double* vsum = vbuf + (m + 1) * 5;
    const float* srow0 = Ma;
    for (int x = 0; x < W * 5; x++) vsum[x] = srow0[x] * (m + 2);
    for (int y = 1; y < m; y++) {
        srow0 = Ma + (size_t)imin(y, H - 1) * W * 5;
        for (int x = 0; x < W * 5; x++) vsum[x] += srow0[x];
    }
    for (int y = 0; y < H; y++) {
        double g11, g12, g22, h1, h2;
        float* flow = flowa + (size_t)y * W * 2;
        srow0 = Ma + (size_t)imax(y - m - 1, 0) * W * 5;
        const float* srow1 = Ma + (size_t)imin(y + m, H - 1) * W * 5;
        for (int x = 0; x < W * 5; x++) vsum[x] += srow1[x] - srow0[x];
        for (int x = 0; x < (m + 1) * 5; x++) {
            vsum[-1 - x] = vsum[4 - x];
            vsum[W * 5 + x] = vsum[W * 5 + x - 5];
        }
        g11 = vsum[0] * (m + 2);
        g12 = vsum[1] * (m + 2);
        g22 = vsum[2] * (m + 2);
        h1 = vsum[3] * (m + 2);
        h2 = vsum[4] * (m + 2);
        for (int x = 1; x < m; x++) {
            g11 += vsum[x * 5];
            g12 += vsum[x * 5 + 1];
            g22 += vsum[x * 5 + 2];
            h1 += vsum[x * 5 + 3];
            h2 += vsum[x * 5 + 4];
        }
        for (int x = 0; x < W; x++) {
            g11 += vsum[(x + m) * 5] - vsum[(x - m) * 5 - 5];
            g12 += vsum[(x + m) * 5 + 1] - vsum[(x - m) * 5 - 4];
            g22 += vsum[(x + m) * 5 + 2] - vsum[(x - m) * 5 - 3];
            h1 += vsum[(x + m) * 5 + 3] - vsum[(x - m) * 5 - 2];
            h2 += vsum[(x + m) * 5 + 4] - vsum[(x - m) * 5 - 1];
            double g11_ = g11 * scale, g12_ = g12 * scale, g22_ = g22 * scale;
            double h1_ = h1 * scale, h2_ = h2 * scale;
            double idet = 1. / (g11_ * g22_ - g12_ * g12_ + 1e-3);
            flow[x * 2] = (float)((g11_ * h2_ - g12_ * h1_) * idet);
            flow[x * 2 + 1] = (float)((g22_ * h1_ - g12_ * h2_) * idet);
        }
    }
    free(vbuf);
}

/* ------------------------------------------------------------------------------------------
 * Level geometry (SURVEY App. A.0-1/2). Returns the number of EXTRA levels actually run
 * (so levels+1 images); fills per-level width/height/ksz/sigma for k = 0..ret.
 * ------------------------------------------------------------------------------------------ */
FDO_API int fdo_level_geometry(int H, int W, int levels, int* hs, int* ws, int* ksz, double* sig)
{
    int k;
    double scale;
    for (k = 0, scale = 1; k < levels; k++) {
        scale *= 0.5;
        if (W * scale < 32 || H * scale < 32) break;
    }
    int nl = k;
    for (k = 0; k <= nl; k++) {
        scale = 1;
        for (int i = 0; i < k; i++) scale *= 0.5;
        double sigma = (1. / scale - 1) * 0.5;
        int s = cv_round(sigma * 5) | 1;
        s = imax(s, 3);
        if (ksz) ksz[k] = s;
        if (sig) sig[k] = sigma;
        if (ws) ws[k] = cv_round(W * scale);
        if (hs) hs[k] = cv_round(H * scale);
    }
    return nl;
}

/* Stage access for parity tests: pyramid image of level k (blur of the full-res image, resize). */
FDO_API void fdo_pyramid_level(const float* img, int H, int W, int ksz, double sigma,
                               int h, int w, float* out)
{
    float* f = (float*)malloc(sizeof(float) * (size_t)H * W);
    fdo_gauss_blur(img, H, W, ksz, sigma, f);
    fdo_resize_linear(f, H, W, 1, out, h, w, 1);
    free(f);
}

/* ------------------------------------------------------------------------------------------
 * a7: cv2.calcOpticalFlowFarneback(prev, next, flow, 0.5, levels, winsize, iters, poly_n,
 *     poly_sigma, flags)  (SURVEY App. A.0). flags & 4 = OPTFLOW_USE_INITIAL_FLOW; flow is
 *     updated in place.  Returns 0.
 * ------------------------------------------------------------------------------------------ */
FDO_API int fdo_farneback(const float* prev, const float* next, float* flow0, int H, int W,
                          int levels, int winsize, int iters, int poly_n, double poly_sigma,
                          int flags)
{
    int hs[32], ws[32], ksz[32];
    double sig[32];
    if (levels > 30) levels = 30;
    int nl = fdo_level_geometry(H, W, levels, hs, ws, ksz, sig);
    float* prevFlow = NULL;
    int ph = 0, pw = 0;
    float* fimg = (float*)malloc(sizeof(float) * (size_t)H * W);
    const float* img[2] = {prev, next};
    for (int k = nl; k >= 0; k--) {
        int h = hs[k], w = ws[k];
        double scale = 1;
        for (int i = 0; i < k; i++) scale *= 0.5;
        float* flow = (k > 0) ? (float*)malloc(sizeof(float) * (size_t)h * w * 2) : flow0;
        if (!prevFlow) {
            if (flags & 4) {
                if (k > 0) {
                    fdo_resize_area(flow0, H, W, 2, flow, h, w);
                    float fs = (float)scale;
                    for (size_t i = 0; i < (size_t)h * w * 2; i++) flow[i] *= fs;
                } /* k == 0: same-size resize onto itself, times 1 */
            } else {
                memset(flow, 0, sizeof(float) * (size_t)h * w * 2);
            }
        } else {
            fdo_resize_linear(prevFlow, ph, pw, 2, flow, h, w, 0);
            for (size_t i = 0; i < (size_t)h * w * 2; i++) flow[i] *= 2.f;
        }
        float* R[2];
        float* I = (float*)malloc(sizeof(float) * (size_t)h * w);
        for (int i = 0; i < 2; i++) {
            R[i] = (float*)malloc(sizeof(float) * (size_t)h * w * 5);
            fdo_gauss_blur(img[i], H, W, ksz[k], sig[k], fimg);
            fdo_resize_linear(fimg, H, W, 1, I, h, w, 1);
            fdo_polyexp(I, h, w, poly_n, poly_sigma, R[i]);
        }
        free(I);
        float* M = (float*)malloc(sizeof(float) * (size_t)h * w * 5);
        fdo_update_matrices(R[0], R[1], flow, h, w, M, 0, h);
        for (int i = 0; i < iters; i++) {
            fdo_blur_solve(M, h, w, winsize, flow);
            if (i < iters - 1) fdo_update_matrices(R[0], R[1], flow, h, w, M, 0, h);
        }
        free(M); free(R[0]); free(R[1]);
        if (prevFlow) free(prevFlow);
        prevFlow = (k > 0) ? flow : NULL;
        ph = h; pw = w;
    }
    free(fimg);
    return 0;
}

/* ------------------------------------------------------------------------------------------
 * a8: warp_slice(reference, flow)  (src/flowdenoising.py:55-63) = cv2.remap(reference,
 * flow + grid, INTER_LINEAR, BORDER_REPLICATE) with OpenCV's 1/32-px map quantiser
 * (SURVEY App. A.1 "remap").
 * ------------------------------------------------------------------------------------------ */
FDO_API void fdo_warp_slice(const float* src, int H, int W, const float* flow, float* dst)
{
    for (int y = 0; y < H; y++)
        for (int x = 0; x < W; x++) {
            /* map = (flow + grid).astype(float32): float64 sum rounded once to float32 */
            float mx = (float)((double)flow[((size_t)y * W + x) * 2] + (double)x);
            float my = (float)((double)flow[((size_t)y * W + x) * 2 + 1] + (double)y);
            int sx = cv_round(mx * 32.f), sy = cv_round(my * 32.f);
            int ax = sx & 31, ay = sy & 31;
            int ix = sx >> 5, iy = sy >> 5;
            /* saturate_cast<short> of the integer coordinates */
            ix = clampi(ix, -32768, 32767); iy = clampi(iy, -32768, 32767);
            float tx1 = ax * (1.f / 32), tx0 = 1.f - tx1;
            float ty1 = ay * (1.f / 32), ty0 = 1.f - ty1;
            float w0 = ty0 * tx0, w1 = ty0 * tx1, w2 = ty1 * tx0, w3 = ty1 * tx1;
            int x0 = clampi(ix, 0, W - 1), x1 = clampi(ix + 1, 0, W - 1);
            int y0 = clampi(iy, 0, H - 1), y1 = clampi(iy + 1, 0, H - 1);
            float v0 = src[(size_t)y0 * W + x0], v1 = src[(size_t)y0 * W + x1];
            float v2 = src[(size_t)y1 * W + x0], v3 = src[(size_t)y1 * W + x1];
            dst[(size_t)y * W + x] = v0 * w0 + v1 * w1 + v2 * w2 + v3 * w3;
        }
}

/* tmp_slice += slice * kernel[i]  (src/flowdenoising.py:138, :316-317): float32 array times
 * np.float64 scalar is a float64 product (NumPy >= 2), the in-place add rounds to float32
 * once per tap (SURVEY App. B Q9). */
FDO_API void fdo_accumulate(float* acc, const float* v, double k, size_t n)
{
    for (size_t i = 0; i < n; i++) acc[i] = (float)((double)acc[i] + (double)v[i] * k);
}

/* ------------------------------------------------------------------------------------------
 * a5: GaussianDenoising.filter_along_{Z,Y,X}_slice  (src/flowdenoising.py:133-158), whole pass.
 * vol and out are dense [Z][Y][X]; axis 0/1/2 = Z/Y/X; periodic wrap along the axis.
 * ------------------------------------------------------------------------------------------ */
FDO_API void fdo_gauss_axis(const float* vol, float* out, int Z, int Y, int X, int axis,
                            const double* kernel, int klen)
{
    int ks2 = klen / 2;
    int dims[3] = {Z, Y, X};
    size_t strides[3] = {(size_t)Y * X, (size_t)X, 1};
    int n = dims[axis];
    size_t sa = strides[axis];
    int a1 = axis == 0 ? 1 : 0, a2 = axis == 2 ? 1 : 2;
#pragma omp parallel for schedule(static)
    for (int s = 0; s < n; s++)
        for (int p = 0; p < dims[a1]; p++)
            for (int q = 0; q < dims[a2]; q++) {
                size_t base = (size_t)p * strides[a1] + (size_t)q * strides[a2];
                float acc = 0.f;
                for (int i = 0; i < klen; i++) {
                    int j = ((s + i - ks2) % n + n) % n;
                    acc = (float)((double)acc + (double)vol[base + (size_t)j * sa] * kernel[i]);
                }
                out[base + (size_t)s * sa] = acc;
            }
}

/* ------------------------------------------------------------------------------------------
 * a6: FlowDenoising.filter_along_{Z,Y,X}_slice  (src/flowdenoising.py:306-373), whole pass,
 * with this file's Farneback / remap restatement. Slices [s0, s1) only (for bounded timing
 * samples); OpenMP over slices like the reference's thread pool (src/flowdenoising.py:187-206).
 * use_prev_flow = 0 reproduces --recompute_flow (get_flow_without_prev_flow, :89-114).
 * ------------------------------------------------------------------------------------------ */
static void gather_slice(const float* vol, int Z, int Y, int X, int axis, int s, float* img)
{
    if (axis == 0) {
        memcpy(img, vol + (size_t)s * Y * X, sizeof(float) * (size_t)Y * X);
    } else if (axis == 1) {
        for (int z = 0; z < Z; z++)
            memcpy(img + (size_t)z * X, vol + ((size_t)z * Y + s) * X, sizeof(float) * X);
    } else {
        for (int z = 0; z < Z; z++)
            for (int y = 0; y < Y; y++) img[(size_t)z * Y + y] = vol[((size_t)z * Y + y) * X + s];
    }
}

static void scatter_slice(float* vol, int Z, int Y, int X, int axis, int s, const float* img)
{
    if (axis == 0) {
        memcpy(vol + (size_t)s * Y * X, img, sizeof(float) * (size_t)Y * X);
    } else if (axis == 1) {
        for (int z = 0; z < Z; z++)
            memcpy(vol + ((size_t)z * Y + s) * X, img + (size_t)z * X, sizeof(float) * X);
    } else {
        for (int z = 0; z < Z; z++)
            for (int y = 0; y < Y; y++) vol[((size_t)z * Y + y) * X + s] = img[(size_t)z * Y + y];
    }
}

FDO_API void fdo_flow_axis(const float* vol, float* out, int Z, int Y, int X, int axis,
                           const double* kernel, int klen, int levels, int winsize, int iters,
                           int poly_n, double poly_sigma, int use_prev_flow, int s0, int s1)
{
    int ks2 = klen / 2;
    int dims[3] = {Z, Y, X};
    int n = dims[axis];
    int H = axis == 0 ? Y : Z;
    int W = axis == 2 ? Y : X;
    size_t P = (size_t)H * W;
#pragma omp parallel
    {
        float* centre = (float*)malloc(sizeof(float) * P);
        float* neigh = (float*)malloc(sizeof(float) * P);
        float* warped = (float*)malloc(sizeof(float) * P);
        float* acc = (float*)malloc(sizeof(float) * P);
        float* flow = (float*)malloc(sizeof(float) * P * 2);
#pragma omp for schedule(dynamic, 1)
        for (int s = s0; s < s1; s++) {
            gather_slice(vol, Z, Y, X, axis, s, centre);
            memset(acc, 0, sizeof(float) * P);
            for (int dir = 0; dir < 2; dir++) {
                memset(flow, 0, sizeof(float) * P * 2);
                if (dir == 1) fdo_accumulate(acc, centre, kernel[ks2], P);
                for (int d = 1; d <= ks2; d++) {
                    int i = dir == 0 ? ks2 - d : ks2 + d;
                    int j = ((s + i - ks2) % n + n) % n;
                    gather_slice(vol, Z, Y, X, axis, j, neigh);
                    if (!use_prev_flow) memset(flow, 0, sizeof(float) * P * 2);
                    fdo_farneback(centre, neigh, flow, H, W, levels, winsize, iters, poly_n,
                                  poly_sigma, use_prev_flow ? 4 : 0);
                    fdo_warp_slice(neigh, H, W, flow, warped);
                    fdo_accumulate(acc, warped, kernel[i], P);
                }
            }
            scatter_slice(out, Z, Y, X, axis, s, acc);
        }
        free(centre); free(neigh); free(warped); free(acc); free(flow);
    }
}
