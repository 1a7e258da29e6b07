/* CPU oracle of OpenCV's Farneback with the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN = 256) -- test
 * infrastructure only, like fd_oracle.c, whose restatement it extends without changing it: the whole of fd_oracle.c is
 * compiled into this library, plus
 *   fdo_gauss_blur_solve  FarnebackUpdateFlow_GaussianBlur: separable Gaussian of M with 2m+1 float32 taps
 *                         (m = win/2, sigma = m*0.3, built as OpenCV builds them), vertical pass then horizontal pass
 *                         in float32 with replicate borders, then the regularised 2x2 solve in float64 without the
 *                         1/winsize^2 scale of the box path. M is not refreshed here (the caller does full sweeps).
 *   fdo_farneback_gw      fdo_farneback with flags & 256 selecting the Gaussian window (same pyramid, polyexp,
 *                         UpdateMatrices, level transfer and initial flow).
 *   fdo_flow_axis_gw      fdo_flow_axis with a flags argument (256: Gaussian window).
 * Bit-exact vs cv2.calcOpticalFlowFarneback 4.13.0 with the same build flags as fd_oracle.c (-O2 -ffp-contract=off):
 * tests/test_gaussian_window_oracle.py.
 */
#include "fd_oracle.c"

FDO_API void fdo_gauss_blur_solve(const float* Ma, int H, int W, int win, float* flowa)
{
    int m = win / 2;
    double sigma = m * 0.3, s = 1;
    float k[64];
    k[0] = (float)s;
    for (int i = 1; i <= m; i++) { float t = (float)exp(-i * i / (2 * sigma * sigma)); k[i] = t; s += t * 2; }
    s = 1. / s;
    for (int i = 0; i <= m; i++) k[i] = (float)(k[i] * s);
    float* vbuf = (float*)malloc(sizeof(float) * (size_t)(W + 2 * m) * 5);
    float* vsum = vbuf + m * 5;
    for (int y = 0; y < H; y++) {
        for (int x = 0; x < W * 5; x++) {
            float s0 = Ma[(size_t)y * W * 5 + x] * k[0];
            for (int i = 1; i <= m; i++)
                s0 += (Ma[(size_t)imin(y + i, H - 1) * W * 5 + x] + Ma[(size_t)imax(y - i, 0) * W * 5 + x]) * k[i];
            vsum[x] = s0;
        }
        for (int p = 1; p <= m; p++) for (int c = 0; c < 5; c++) {
            vsum[-p * 5 + c] = vsum[c];
            vsum[(W - 1 + p) * 5 + c] = vsum[(W - 1) * 5 + c];
        }
        float* flow = flowa + (size_t)y * W * 2;
        for (int x = 0; x < W; x++) {
            float hs[5];
            for (int c = 0; c < 5; c++) {
                float s0 = vsum[x * 5 + c] * k[0];
                for (int i = 1; i <= m; i++) s0 += (vsum[(x + i) * 5 + c] + vsum[(x - i) * 5 + c]) * k[i];
                hs[c] = s0;
            }
            double g11 = hs[0], g12 = hs[1], g22 = hs[2], h1 = hs[3], h2 = hs[4];
            double idet = 1. / (g11 * g22 - g12 * g12 + 1e-3);
            flow[x * 2] = (float)((g11 * h2 - g12 * h1) * idet);
            flow[x * 2 + 1] = (float)((g22 * h1 - g12 * h2) * idet);
        }
    }
    free(vbuf);
}
FDO_API int fdo_farneback_gw(const float* prev, const float* next, float* flow0, int H, int W,
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
            if (flags & 256) fdo_gauss_blur_solve(M, h, w, winsize, flow);
            else fdo_blur_solve(M, h, w, winsize, flow);
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

FDO_API void fdo_flow_axis_gw(const float* vol, float* out, int Z, int Y, int X, int axis,
                           const double* kernel, int klen, int levels, int winsize, int iters,
                           int poly_n, double poly_sigma, int use_prev_flow, int s0, int s1, int flags)
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
                    fdo_farneback_gw(centre, neigh, flow, H, W, levels, winsize, iters, poly_n,
                                     poly_sigma, (use_prev_flow ? 4 : 0) | (flags & 256));
                    fdo_warp_slice(neigh, H, W, flow, warped);
                    fdo_accumulate(acc, warped, kernel[i], P);
                }
            }
            scatter_slice(out, Z, Y, X, axis, s, acc);
        }
        free(centre); free(neigh); free(warped); free(acc); free(flow);
    }
}
