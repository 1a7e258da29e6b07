// Stage 3 kernels: displacement update (FarnebackUpdateMatrices) fused with the flow blur + 2x2 solve
// (FarnebackUpdateFlow_Blur), and the flow resampling between pyramid levels. sm_100a.
//
// Reference behaviour: the inner loop of cv2.calcOpticalFlowFarneback as called from
// /root/reference/src/flowdenoising.py:69-79 (SURVEY.md App. A.0, A.3, A.4).
//
// k_flow_iter design (one launch = one Farneback iteration of one level for a batch of image pairs).
// OpenCV's box filter is two RUNNING sums, and both are history dependent in the last bits:
//   vertical   vsum(y)   = vsum(y-1) + float32(M[y+m] - M[y-m-1])          (float64 accumulator, float32 difference)
//   horizontal g(x)      = g(x-1)    + (vsum[x+m] - vsum[x-m-1])           (float64, rounding errors persist along x)
// so a tiled box filter cannot reproduce the reference bit for bit. This kernel reproduces both scans exactly:
//   * a block owns a strip of CW columns of one image pair and MARCHES down the rows in tiles of TR rows;
//   * phase V (thread per column, incl. an (m+1 | m)-column halo): M for the new row from R0, flow and a bilinear
//     gather of R1 (M never touches HBM), ring of the last 2m+2 rows in shared memory, float64 column sums updated
//     exactly like OpenCV, published to a shared-memory tile;
//   * phase H (thread per (row, channel) of the tile): the horizontal running sum walks the strip's columns
//     sequentially, starting from the carry of the strip to the left (same row). Carries travel between the
//     strips' blocks through global memory with release/acquire flags (blocks of one image are dispatched left
//     to right, a strip only ever waits on its left neighbour: the decoupled look-back argument);
//   * phase S (thread per column): regularised 2x2 solve, flow written once.
//   Every R0 / flow row is read once (no vertical halo), R1 gathers mostly hit L1/L2.
//   Algorithmic HBM bytes per pixel: R0 20 + R1 20 + flow in 8 + flow out 8 = 56 (SURVEY.md §8d).
// Compiled with -fmad=false: OpenCV's scalar code has no fused multiply-adds here.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>

#include "fdn_internal.cuh"

namespace fdn {

struct FlowIterArgs {
    const float* R;     // level base inside slot 0: [h*w] float4 (channels 0-3) then [h*w] float (channel 4)
    int64_t R_stride;   // floats per slot
    SlotMap map0, map1;
    const float* flow_in;
    float* flow_out;
    int h, w, m;
    int n;              // image pairs (grid = n * strips blocks)
    int LS;             // shared tile line stride in doubles (== 1 mod 16)
    int strips;
    double scale;       // 1 / winsize^2
    double* carry;      // [n][strips][h][5]
    unsigned long long* flags;  // [n][strips]
    unsigned long long epoch;
    unsigned* ctl;      // [0] tickets taken, [1] blocks finished (both 0 between launches)
};

// ROWCHK = false: the caller guarantees 5 <= y < h - 5, so the border weight reduces to the column factor `sx`
// (= border[x] * border[w-1-x], the first product OpenCV forms; the two row factors are exactly 1).
template <bool ROWCHK = true>
__device__ __forceinline__ void update_matrices_px(const float4* __restrict__ R0a, const float* __restrict__ R0b,
                                                   const float4* __restrict__ R1a, const float* __restrict__ R1b,
                                                   const float2 f, int x, int y, int h, int w, float M[5],
                                                   bool colb = false, float sx = 1.f)
{
    const int idx = y * w + x;
    const float dx = f.x, dy = f.y;
    float fx = __fadd_rn((float)x, dx), fy = __fadd_rn((float)y, dy);
    const int x1 = (int)floorf(fx), y1 = (int)floorf(fy);
    fx = __fsub_rn(fx, (float)x1);
    fy = __fsub_rn(fy, (float)y1);
    const float4 c03 = __ldg(R0a + idx);
    const float c4 = __ldg(R0b + idx);
    float r2, r3, r4, r5, r6;
    if ((unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1)) {
        const float ofx = __fsub_rn(1.f, fx), ofy = __fsub_rn(1.f, fy);
        const float a00 = __fmul_rn(ofx, ofy), a01 = __fmul_rn(fx, ofy), a10 = __fmul_rn(ofx, fy),
                    a11 = __fmul_rn(fx, fy);
        const int g = y1 * w + x1;
        const float4 p00 = __ldg(R1a + g), p01 = __ldg(R1a + g + 1), p10 = __ldg(R1a + g + w),
                     p11 = __ldg(R1a + g + w + 1);
        const float q00 = __ldg(R1b + g), q01 = __ldg(R1b + g + 1), q10 = __ldg(R1b + g + w),
                    q11 = __ldg(R1b + g + w + 1);
#define FDN_BILIN(v00, v01, v10, v11) \
    __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a00, v00), __fmul_rn(a01, v01)), __fmul_rn(a10, v10)), __fmul_rn(a11, v11))
        r2 = FDN_BILIN(p00.x, p01.x, p10.x, p11.x);
        r3 = FDN_BILIN(p00.y, p01.y, p10.y, p11.y);
        r4 = FDN_BILIN(p00.z, p01.z, p10.z, p11.z);
        r5 = FDN_BILIN(p00.w, p01.w, p10.w, p11.w);
        r6 = FDN_BILIN(q00, q01, q10, q11);
#undef FDN_BILIN
        r4 = __fmul_rn(__fadd_rn(c03.z, r4), 0.5f);
        r5 = __fmul_rn(__fadd_rn(c03.w, r5), 0.5f);
        r6 = __fmul_rn(__fadd_rn(c4, r6), 0.25f);
    } else {
        r2 = r3 = 0.f;
        r4 = c03.z;
        r5 = c03.w;
        r6 = __fmul_rn(c4, 0.5f);
    }
    r2 = __fmul_rn(__fsub_rn(c03.x, r2), 0.5f);
    r3 = __fmul_rn(__fsub_rn(c03.y, r3), 0.5f);
    r2 = __fadd_rn(r2, __fadd_rn(__fmul_rn(r4, dy), __fmul_rn(r6, dx)));
    r3 = __fadd_rn(r3, __fadd_rn(__fmul_rn(r6, dy), __fmul_rn(r5, dx)));
    if (ROWCHK) {
        if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
            // border[5] = {0.14, 0.14, 0.4472, 0.4472, 0.4472}
            float s = x < 5 ? (x < 2 ? 0.14f : 0.4472f) : 1.f;
            const int xr = w - x - 1, yr = h - y - 1;
            s = __fmul_rn(s, x >= w - 5 ? (xr < 2 ? 0.14f : 0.4472f) : 1.f);
            s = __fmul_rn(s, y < 5 ? (y < 2 ? 0.14f : 0.4472f) : 1.f);
            s = __fmul_rn(s, y >= h - 5 ? (yr < 2 ? 0.14f : 0.4472f) : 1.f);
            r2 = __fmul_rn(r2, s); r3 = __fmul_rn(r3, s); r4 = __fmul_rn(r4, s);
            r5 = __fmul_rn(r5, s); r6 = __fmul_rn(r6, s);
        }
    } else if (colb) {
        r2 = __fmul_rn(r2, sx); r3 = __fmul_rn(r3, sx); r4 = __fmul_rn(r4, sx);
        r5 = __fmul_rn(r5, sx); r6 = __fmul_rn(r6, sx);
    }
    M[0] = __fadd_rn(__fmul_rn(r4, r4), __fmul_rn(r6, r6));
    M[1] = __fmul_rn(__fadd_rn(r4, r5), r6);
    M[2] = __fadd_rn(__fmul_rn(r5, r5), __fmul_rn(r6, r6));
    M[3] = __fadd_rn(__fmul_rn(r4, r2), __fmul_rn(r6, r3));
    M[4] = __fadd_rn(__fmul_rn(r6, r2), __fmul_rn(r5, r3));
}

constexpr int tile_line_stride(int cw, int m)
{
    int ls = cw + 2 * m + 2;
    while (ls % 16 != 1) ls++;
    return ls;
}

// MT > 0: half window m = MT known at compile time (winsize 5 -> MT 2, winsize 9 -> MT 4): ring / tile strides fold
// into immediates. MT == 0: generic m from the arguments.
template <int CW, int TR, int MT, int MINB>
__global__ void __launch_bounds__(CW + 32, MINB)
k_flow_iter(FlowIterArgs a)
{
    constexpr int NT = CW + 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int m = MT > 0 ? MT : a.m;
    const int LS = MT > 0 ? tile_line_stride(CW, MT) : a.LS;
    const int RR = 2 * m + 2;
    const int h = a.h, w = a.w;
    double* tile = reinterpret_cast<double*>(smem_raw);                               // [TR*5][LS]
    float* ring = reinterpret_cast<float*>(smem_raw + sizeof(double) * TR * 5 * LS);  // [RR][5][NT]

    const int t = threadIdx.x;
    // (pair, strip) from a ticket, strip fastest: a strip spin-waits on the strip to its left, which therefore must
    // already be running whatever order the hardware dispatches blocks in
    __shared__ int s_ticket;
    if (t == 0) s_ticket = (int)atomicAdd(a.ctl, 1u);
    __syncthreads();
    const int k = s_ticket % a.strips;  // strip
    const int b = s_ticket / a.strips;  // image pair
    const int x0 = k * CW;
    // tile position q <-> column x0 - m - 1 + q, q in [0, CW + 2m + 1)
    int q;
    bool active = true;
    if (t < CW) {
        q = t + m + 1;
    } else {
        const int hd = t - CW;
        if (hd < m + 1) q = hd;
        else if (hd < 2 * m + 1) q = CW + hd;
        else { q = 0; active = false; }
    }
    const int xcl = min(max(x0 - m - 1 + q, 0), w - 1);
    const bool core = (t < CW) && (x0 + t < w);
    const int ncols = min(CW, w - x0);
    // column part of the border weight (steady tiles): (x < 5 ? border[x] : 1) * (x >= w-5 ? border[w-1-x] : 1)
    const bool colb = (unsigned)(xcl - 5) >= (unsigned)(w - 10);
    const float sxc = __fmul_rn(xcl < 5 ? (xcl < 2 ? 0.14f : 0.4472f) : 1.f,
                                xcl >= w - 5 ? (w - xcl - 1 < 2 ? 0.14f : 0.4472f) : 1.f);

    const float* R0 = a.R + (int64_t)a.map0.slot(b) * a.R_stride;
    const float* R1 = a.R + (int64_t)a.map1.slot(b) * a.R_stride;
    const float4* R0a = reinterpret_cast<const float4*>(R0);
    const float4* R1a = reinterpret_cast<const float4*>(R1);
    const float* R0b = R0 + (int64_t)4 * h * w;
    const float* R1b = R1 + (int64_t)4 * h * w;
    const float2* fin = reinterpret_cast<const float2*>(a.flow_in) + (int64_t)b * h * w;
    float2* fout = reinterpret_cast<float2*>(a.flow_out) + (int64_t)b * h * w;
    double* carry_out = a.carry + ((int64_t)b * a.strips + k) * h * 5;
    const double* carry_in = a.carry + ((int64_t)b * a.strips + max(k - 1, 0)) * h * 5;
    volatile unsigned long long* flag_in = a.flags + (int64_t)b * a.strips + max(k - 1, 0);
    volatile unsigned long long* flag_out = a.flags + (int64_t)b * a.strips + k;

    double vs[5] = {0, 0, 0, 0, 0};
    int next_row = 0;       // next M row to compute
    float* ring_new = ring + t;   // ring slot of next_row      (slot stride 5*NT, channel stride NT)
    float* ring_old = ring + t;   // ring slot of row max(y-m-1, 0)
    float* const ring_end = ring + RR * 5 * NT;
    float Mv[5];

    if (active) {
        // rows 0 .. m-1 (clamped to h-1) seed the column sums: vsum = M[0]*(m+2) + sum_{y=1}^{m-1} M[min(y,h-1)]
        const int last_init = min(max(m - 1, 0), h - 1);
        for (; next_row <= last_init; next_row++) {
            update_matrices_px(R0a, R0b, R1a, R1b, __ldg(fin + next_row * w + xcl), xcl, next_row, h, w, Mv);
#pragma unroll
            for (int c = 0; c < 5; c++) ring_new[c * NT] = Mv[c];
            ring_new += 5 * NT;
            if (ring_new >= ring_end) ring_new -= RR * 5 * NT;
        }
        const float mp2 = (float)(m + 2);
#pragma unroll
        for (int c = 0; c < 5; c++) vs[c] = (double)__fmul_rn(ring[c * NT + t], mp2);
        for (int y = 1; y < m; y++) {
            const int sl = min(y, h - 1);  // < RR always
#pragma unroll
            for (int c = 0; c < 5; c++) vs[c] = __dadd_rn(vs[c], (double)ring[(sl * 5 + c) * NT + t]);
        }
    }

    // Step y of the march consumes the new row y + m. The flow of a tile's TR new rows is fetched one tile ahead
    // (issued before the block waits for the horizontal scan), so phase V exposes one memory latency per row (the R1
    // gather) instead of two dependent ones.
    float2 fl[TR];
#pragma unroll
    for (int r = 0; r < TR; r++) {
        fl[r] = make_float2(0.f, 0.f);
        if (active && r + m < h) fl[r] = __ldg(fin + (r + m) * w + xcl);
    }

    int tile_idx = 0;
    for (int y0 = 0; y0 < h; y0 += TR, tile_idx++) {
        // ---------------- phase V: column sums of TR rows ----------------
        // Steady tiles (every step brings a new row, no top/bottom border involved): with TR == ring rows the ring
        // slots of a tile are compile-time constants -- row r is written to slot (m + r) % RR and the row leaving
        // the window sits in slot (m + 1 + r) % RR -- and all bookkeeping branches disappear.
        constexpr bool kStatic = MT > 0 && TR == 2 * MT + 2;
        const bool steady = kStatic && y0 >= TR && y0 + TR - 1 + m <= h - 1 && y0 + m >= 5 && y0 + TR - 1 + m < h - 5;
        if (active && steady) {
            if constexpr (kStatic) {
                constexpr int RRs = 2 * MT + 2;
                double* tq = tile + q;
                float* rg = ring + t;
#pragma unroll
                for (int r = 0; r < TR; r++) {
                    update_matrices_px<false>(R0a, R0b, R1a, R1b, fl[r], xcl, y0 + r + MT, h, w, Mv, colb, sxc);
#pragma unroll
                    for (int c = 0; c < 5; c++) {
                        rg[(((MT + r) % RRs) * 5 + c) * NT] = Mv[c];
                        const float d = __fsub_rn(Mv[c], rg[(((MT + 1 + r) % RRs) * 5 + c) * NT]);
                        vs[c] = __dadd_rn(vs[c], (double)d);
                        tq[(r * 5 + c) * LS] = vs[c];
                    }
                }
                next_row += TR;   // ring_new / ring_old come back to the same slots after TR == RR advances
            }
        } else if (active) {
            double* tq = tile + q;
#pragma unroll
            for (int r = 0; r < TR; r++) {
                const int y = y0 + r;
                if (y < h) {
                    if (next_row <= min(y + m, h - 1)) {  // exactly one new row per step while y + m < h
                        update_matrices_px(R0a, R0b, R1a, R1b, fl[r], xcl, next_row, h, w, Mv);  // next_row == y + m
#pragma unroll
                        for (int c = 0; c < 5; c++) ring_new[c * NT] = Mv[c];
                        ring_new += 5 * NT;
                        if (ring_new >= ring_end) ring_new -= RR * 5 * NT;
                        next_row++;
                    } else {  // bottom border: row h-1 again (the last slot written)
                        const float* last = (ring_new == ring + t ? ring_end + t : ring_new) - 5 * NT;
#pragma unroll
                        for (int c = 0; c < 5; c++) Mv[c] = last[c * NT];
                    }
#pragma unroll
                    for (int c = 0; c < 5; c++) {
                        const float d = __fsub_rn(Mv[c], ring_old[c * NT]);
                        vs[c] = __dadd_rn(vs[c], (double)d);
                        tq[(r * 5 + c) * LS] = vs[c];
                    }
                    if (y >= m + 1) {  // row max(y-m, 0) next
                        ring_old += 5 * NT;
                        if (ring_old >= ring_end) ring_old -= RR * 5 * NT;
                    }
                }
            }
        }
        if (t == 0 && k > 0) {  // the left strip must have published this tile's carries
            const unsigned long long want = a.epoch + (unsigned long long)tile_idx + 1ull;
            while (*flag_in < want) __nanosleep(20);
            __threadfence();
        }
        __syncthreads();
        if (active) {  // flows of the next tile's new rows: in flight while the scan and the solve run
#pragma unroll
            for (int r = 0; r < TR; r++) {
                const int row = y0 + TR + r + m;
                if (row < h) fl[r] = __ldg(fin + row * w + xcl);
            }
        }
        // ---------------- phase H: sequential horizontal running sums ----------------
        if (t < 5 * TR) {
            const int r = t / 5, c = t - r * 5;
            const int y = y0 + r;
            if (y < h) {
                double* line = tile + (r * 5 + c) * LS;
                double S;
                if (k == 0) {
                    // g = vsum[0]*(m+2) + vsum[1] + ... + vsum[m-1]   (columns clamp to the replicated border)
                    S = __dmul_rn(line[m + 1], (double)(m + 2));
                    for (int x = 1; x < m; x++) S = __dadd_rn(S, line[m + 1 + x]);
                } else {
                    S = __ldcg(carry_in + (int64_t)y * 5 + c);
                }
                // S(i) = S(i-1) + (vs[i+m] - vs[i-m-1]); S(i) overwrites the dead slot of column i-m-1. The differences
                // of the next batch are formed before this batch's stores, so only the add chain is serial.
                const int off = 2 * m + 1;
                constexpr int HB = 8;
                int i = 0;
                if (ncols >= HB) {
                    double d[HB];
#pragma unroll
                    for (int u = 0; u < HB; u++) d[u] = __dsub_rn(line[u + off], line[u]);
                    for (; i + 2 * HB <= ncols; i += HB) {
                        double d2[HB];
#pragma unroll
                        for (int u = 0; u < HB; u++) d2[u] = __dsub_rn(line[i + HB + u + off], line[i + HB + u]);
#pragma unroll
                        for (int u = 0; u < HB; u++) {
                            S = __dadd_rn(S, d[u]);
                            line[i + u] = S;
                        }
#pragma unroll
                        for (int u = 0; u < HB; u++) d[u] = d2[u];
                    }
#pragma unroll
                    for (int u = 0; u < HB; u++) {
                        S = __dadd_rn(S, d[u]);
                        line[i + u] = S;
                    }
                    i += HB;
                }
                for (; i < ncols; i++) {
                    S = __dadd_rn(S, __dsub_rn(line[i + off], line[i]));
                    line[i] = S;
                }
                if (k + 1 < a.strips) {
                    __stcg(carry_out + (int64_t)y * 5 + c, S);
                    __threadfence();
                }
            }
        }
        __syncthreads();
        if (t == 0 && k + 1 < a.strips) *flag_out = a.epoch + (unsigned long long)tile_idx + 1ull;
        // ---------------- phase S: solve ----------------
        if (core) {
            const double* tt = tile + t;
#pragma unroll
            for (int r = 0; r < TR; r++) {
                const int y = y0 + r;
                if (y < h) {
                    double g[5];
#pragma unroll
                    for (int c = 0; c < 5; c++) g[c] = __dmul_rn(tt[(r * 5 + c) * LS], a.scale);
                    const double det = __dadd_rn(__dsub_rn(__dmul_rn(g[0], g[2]), __dmul_rn(g[1], g[1])), 1e-3);
                    const double idet = __drcp_rn(det);  // == 1./det correctly rounded, like the IEEE division
                    float2 o;
                    o.x = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[0], g[4]), __dmul_rn(g[1], g[3])), idet);
                    o.y = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[2], g[3]), __dmul_rn(g[1], g[4])), idet);
                    fout[y * w + x0 + t] = o;
                }
            }
        }
        __syncthreads();
    }
    if (t == 0) {   // the last block to finish re-arms the ticket counters for the next launch
        __threadfence();
        if (atomicAdd(a.ctl + 1, 1u) == gridDim.x - 1) { a.ctl[0] = 0; a.ctl[1] = 0; }
    }
}


// ------------------------------------------------------------------------------------------------
// k_flow_iter_ws: the same march as k_flow_iter, rebuilt as a warp-specialised pipeline (default for winsize 5).
//   * 256 threads = two warpgroups. The "column" warpgroup (128 threads: one strip of CW <= 120 core columns plus
//     its (m+1 | m) halo columns, thread t <-> image column x0 - m - 1 + t) runs phase V only. In the second
//     warpgroup one "scan" warp runs phase H and three "solve" warps run phase S. The column sums of a tile go into
//     one of TWO shared-memory tiles, so the scan / solve of tile j overlap phase V of tiles j+1 and j+2. Registers
//     are moved between the warpgroups with setmaxnreg (176 per column thread, 80 per scan / solve thread, 2 blocks
//     per SM); hand-offs are hardware barriers only -- named barriers (bar.arrive / bar.sync) between the column
//     warps and the scan / solve warps, and one mbarrier per 32-column chunk of a tile on which the solve warps
//     sleep until the scan has passed (round 1 polled a shared-memory counter here: a fifth of all issued
//     instructions and of the L1 / shared-memory pipe's wavefronts were that poll);
//   * the ring of the last 2m+2 rows of M lives in REGISTERS: a tile is one ring period (TR = 2m+2 rows), so every
//     ring slot is a compile-time constant of the unrolled row loop;
//   * phase V is branch-free (selects, clamped gather addresses): the m+1 rows of half a tile form one straight-line
//     block whose dependency chains the compiler interleaves. The bilinear gather reads R1 through L1 -- the
//     kernel's shared memory is small (62 KB per block), so about 100 KB of L1 remain per SM; every gather also
//     prefetches (prefetch.global.L1) the R1 line the same column will need FDN_WS_PF rows further down, and the
//     R0 / flow rows, read once, bypass L1 and are register-prefetched a tile ahead;
//   * carries between strips travel as self-validating packets {32 data bits, 32-bit launch tag} (two per double,
//     one 16-byte store): no fences, no flag, only the 5*TR scanning lanes ever wait for the left strip;
//   * phase H reads a line once, 128 bits at a time, through a sliding register window, forms the differences of
//     the next 8 columns while the dependent DADD chain of the current 8 runs, and stores 128 bits at a time;
//   * phase S follows the scan through the tile in chunks of 32 columns (a full tile is one straight-line block);
//   * ONE launch runs up to three consecutive Farneback iterations of a level: a block's work item
//     (iteration, pair, strip) comes from a ticket counter (iteration slowest, strip fastest). A strip waits for the
//     strip to its left, and an iteration of a pair for all strips of its previous iteration (a counter per
//     (iteration, pair)); both are always held by blocks with EARLIER tickets, which are resident or finished --
//     forward progress does not depend on the order the hardware dispatches blocks in. Three iterations rotate
//     through three flow buffers, so no buffer is read after it was written in the same launch by another SM
//     except through L2 (flow loads are ld.global.cg). The last warp to leave re-arms all counters.
// Same arithmetic, same order of operations, same bits as k_flow_iter. Needs w % 4 == 0.
// ------------------------------------------------------------------------------------------------
struct RowIn {
    float2 f;
    float4 c03;
    float c4;
};

template <int MT, int NT_>
struct WsCfg {
    static constexpr int NT = NT_;
    static constexpr int RR = 2 * MT + 2;   // ring period: rows of M a column keeps
    // tile rows: one ring period when its 5 * RR lines fit the lanes of the one scan warp (winsize 5: 6 rows), else half
    // a period (winsize 9: 5 rows, the two tiles of a period are the two shared-memory tiles)
    static constexpr int TR = 5 * RR <= 32 ? RR : RR / 2;
    static constexpr int TPP = RR / TR;     // tiles per ring period
#ifndef FDN_WS_SR4
#define FDN_WS_SR4 2
#endif
    static constexpr int SR = MT == 4 ? FDN_WS_SR4 : 3;   // rows per straight-line block of phase V
    static constexpr int NB = (TR + SR - 1) / SR;
    static constexpr int HALO = 2 * MT + 1;
    static constexpr int CWMAX = (NT - HALO) & ~3;
    static constexpr int NCH = (CWMAX + 31) / 32;   // 32-column chunks of a strip (scan -> solve hand-off)
    static constexpr int LS = NT + 2;       // tile line stride in doubles (even: every line is 16-byte aligned)
#ifndef FDN_WS_NBUF
#define FDN_WS_NBUF 2
#endif
    static constexpr int NBUF = FDN_WS_NBUF;   // shared-memory tiles: phase V may run NBUF tiles ahead of the solve
    static constexpr size_t tiles_bytes = NBUF * sizeof(double) * TR * 5 * LS + 128;   // (+ the scan's read-ahead past the last line)
    static constexpr size_t smem_bytes = tiles_bytes + 8 * NBUF * NCH + 16;      // + the chunk mbarriers, the ticket
    static_assert(5 * TR <= 32, "phase H runs in one warp");
    static_assert(TR * TPP == RR && (TPP == 1 || TPP == 2), "a ring period is one tile or the two shared-memory tiles");
    static_assert(HALO + 8 <= 17, "the scan's register window spans two 8-column sets and one more column");
};

// The eight bilinear taps of one pixel (R1 at the displaced position), read at clamped -- always valid -- positions.
struct Taps {
    float4 p00, p01, p10, p11;
    float q00, q01, q10, q11;
};

template <int PF>
__device__ __forceinline__ Taps ws_gather(const float2 f, const float4* __restrict__ R1a, const float* __restrict__ R1b,
                                          int x, int y, int h, int w)
{
    const int x1 = (int)floorf(__fadd_rn((float)x, f.x)), y1 = (int)floorf(__fadd_rn((float)y, f.y));
    const int yc = min(max(y1, 0), h - 2), xc = min(max(x1, 0), w - 2);
    const int g = yc * w + xc;
    if (PF > 0) {
        // warm L1 with the R1 rows this column will gather from PF rows further down (the flow is smooth)
        const int gp = min(yc + PF + 1, h - 1) * w + xc;
        asm volatile("prefetch.global.L1 [%0];" :: "l"(R1a + gp));
        asm volatile("prefetch.global.L1 [%0];" :: "l"(R1b + gp));
    }
    Taps t;
    t.p00 = __ldg(R1a + g); t.p01 = __ldg(R1a + g + 1); t.p10 = __ldg(R1a + g + w); t.p11 = __ldg(R1a + g + w + 1);
    t.q00 = __ldg(R1b + g); t.q01 = __ldg(R1b + g + 1); t.q10 = __ldg(R1b + g + w); t.q11 = __ldg(R1b + g + w + 1);
    return t;
}

// M of one pixel, branch-free: the taps are discarded by a select when the displaced position lies outside the
// image, exactly as the branch of update_matrices_px would.
__device__ __forceinline__ void ws_matrices_px(const RowIn& in, const Taps& tp, int x, int y, int h, int w, float sxc,
                                               float M[5])
{
    const float dx = in.f.x, dy = in.f.y;
    float fx = __fadd_rn((float)x, dx), fy = __fadd_rn((float)y, dy);
    const int x1 = (int)floorf(fx), y1 = (int)floorf(fy);
    fx = __fsub_rn(fx, (float)x1);
    fy = __fsub_rn(fy, (float)y1);
    const float4 c03 = in.c03;
    const float c4 = in.c4;
    const bool in_img = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
    const float ofx = __fsub_rn(1.f, fx), ofy = __fsub_rn(1.f, fy);
    const float a00 = __fmul_rn(ofx, ofy), a01 = __fmul_rn(fx, ofy), a10 = __fmul_rn(ofx, fy), a11 = __fmul_rn(fx, fy);
#define FDN_BILIN(v00, v01, v10, v11) \
    __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(a00, v00), __fmul_rn(a01, v01)), __fmul_rn(a10, v10)), __fmul_rn(a11, v11))
    float r2 = FDN_BILIN(tp.p00.x, tp.p01.x, tp.p10.x, tp.p11.x);
    float r3 = FDN_BILIN(tp.p00.y, tp.p01.y, tp.p10.y, tp.p11.y);
    float r4 = FDN_BILIN(tp.p00.z, tp.p01.z, tp.p10.z, tp.p11.z);
    float r5 = FDN_BILIN(tp.p00.w, tp.p01.w, tp.p10.w, tp.p11.w);
    float r6 = FDN_BILIN(tp.q00, tp.q01, tp.q10, tp.q11);
#undef FDN_BILIN
    r4 = __fmul_rn(__fadd_rn(c03.z, r4), 0.5f);
    r5 = __fmul_rn(__fadd_rn(c03.w, r5), 0.5f);
    r6 = __fmul_rn(__fadd_rn(c4, r6), 0.25f);
    r2 = in_img ? r2 : 0.f;
    r3 = in_img ? r3 : 0.f;
    r4 = in_img ? r4 : c03.z;
    r5 = in_img ? r5 : c03.w;
    r6 = in_img ? r6 : __fmul_rn(c4, 0.5f);
    r2 = __fmul_rn(__fsub_rn(c03.x, r2), 0.5f);
    r3 = __fmul_rn(__fsub_rn(c03.y, r3), 0.5f);
    r2 = __fadd_rn(r2, __fadd_rn(__fmul_rn(r4, dy), __fmul_rn(r6, dx)));
    r3 = __fadd_rn(r3, __fadd_rn(__fmul_rn(r6, dy), __fmul_rn(r5, dx)));
    // border weight ((border_x_left * border_x_right) * border_y_top) * border_y_bottom; every factor is 1 away from
    // the borders and x * 1.f == x bit for bit, so the product is applied unconditionally
    float s = sxc;
    s = __fmul_rn(s, y < 5 ? (y < 2 ? 0.14f : 0.4472f) : 1.f);
    s = __fmul_rn(s, y >= h - 5 ? (h - y - 1 < 2 ? 0.14f : 0.4472f) : 1.f);
    r2 = __fmul_rn(r2, s); r3 = __fmul_rn(r3, s); r4 = __fmul_rn(r4, s);
    r5 = __fmul_rn(r5, s); r6 = __fmul_rn(r6, s);
    M[0] = __fadd_rn(__fmul_rn(r4, r4), __fmul_rn(r6, r6));
    M[1] = __fmul_rn(__fadd_rn(r4, r5), r6);
    M[2] = __fadd_rn(__fmul_rn(r5, r5), __fmul_rn(r6, r6));
    M[3] = __fadd_rn(__fmul_rn(r4, r2), __fmul_rn(r6, r3));
    M[4] = __fadd_rn(__fmul_rn(r6, r2), __fmul_rn(r5, r3));
}

// Phase H keeps a register window of 17 tile positions: two 8-column sets (four 128-bit loads each) and the first pair
// of the set after them. `idx` is a compile-time constant after unrolling.
__device__ __forceinline__ double ws_win(const double2 (&W0)[4], const double2 (&W1)[4], const double2& X, int idx)
{
    return idx < 8 ? ((idx & 1) ? W0[idx >> 1].y : W0[idx >> 1].x)
                   : idx < 16 ? ((idx & 1) ? W1[(idx - 8) >> 1].y : W1[(idx - 8) >> 1].x) : X.x;
}
// D[u] = pos[8k + u + OFF] - pos[8k + u] for the 8 columns of chunk k (W0 = set k, W1 = set k+1, X = first pair of set k+2)
template <int OFF>
__device__ __forceinline__ void ws_diffs(double (&D)[8], const double2 (&W0)[4], const double2 (&W1)[4], const double2& X)
{
#pragma unroll
    for (int u = 0; u < 8; u++) D[u] = __dsub_rn(ws_win(W0, W1, X, u + OFF), ws_win(W0, W1, X, u));
}

// phase-removal experiments exist only in -DFDN_WS_EXPERIMENTS builds: in product builds the tests fold to constants
// (no branches inside the straight-line blocks of phase V)
#ifdef FDN_WS_EXPERIMENTS
#define FDN_WS_EXP(bit) (wa.exp & (bit))
#else
#define FDN_WS_EXP(bit) (0)
#endif
#ifndef FDN_WS_HC
#define FDN_WS_HC 8
#endif
#ifndef FDN_WS_PF
#define FDN_WS_PF 6
#endif
#ifndef FDN_WS_L2PF
#define FDN_WS_L2PF 0
#endif
#ifndef FDN_WS_SOLVE_SLEEP
// The solve warps sleep this many nanoseconds between two tries of a chunk mbarrier. A bare try_wait loop retries every
// ~40 cycles: measured, a sixth of all warp instructions the kernel issued were that spin. Pauses of 20 .. 400 ns leave
// the launch time unchanged (2.197 .. 2.200 ms per iteration, 128 pairs of 1024 x 1024) and take the spin out of the
// issue arbitration and the power budget.
#define FDN_WS_SOLVE_SLEEP 100
#endif
#define FDN_WS_MAX_ITERS 3   // iterations per launch: one flow buffer per iteration, none read after being rewritten

struct WsArgs {
    const float* R;         // level base inside slot 0
    int64_t R_stride;       // floats per slot
    SlotMap map0, map1;
    const float* fin[FDN_WS_MAX_ITERS];    // flow read / written by iteration i of this launch
    float* fout[FDN_WS_MAX_ITERS];
    int n, iters;           // image pairs, iterations in this launch
    int h, w, CW, strips;
    double scale;           // 1 / winsize^2
    int exp;                // 0 in product builds; phase-removal timing experiments with -DFDN_WS_EXPERIMENTS (FDN_EXP)
    unsigned tag;           // iteration i tags its carry packets with tag + i (never 0)
    ulonglong2* packets;    // [n][strips][h][5]: {lo32 | tag << 32, hi32 | tag << 32}
    unsigned* ctl;          // [0] tickets taken, [1] warps that have finished (both 0 between launches)
    unsigned* done;         // [iters][n]: strips of (iteration, pair) that have written all their flow (0 between launches)
};

// named barriers (id 0 is __syncthreads)
__device__ __forceinline__ void nbar_sync(int id, int count)
{
    asm volatile("bar.sync %0, %1;" :: "r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void nbar_arrive(int id, int count)
{
    asm volatile("bar.arrive %0, %1;" :: "r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// Roles and hand-offs:
//   column warps:  [wait FREE[j&1]] -> V(j) -> arrive FULL[j&1] -> V(j+1) ...
//   scan warp:     wait FULL[j&1] -> H(j) in place, arriving on CHUNK[j&1][q] every 32 columns
//   solve warps:   wait CHUNK[j&1][q] -> S(j) for chunk q -> ... -> arrive FREE[j&1]
// Registers: the kernel is compiled for (65536 / 2 blocks / 256 threads) = 128 per thread; the column warpgroup then
// takes 176 (setmaxnreg.inc) and the scan warpgroup keeps 80 (setmaxnreg.dec).
template <int MT, int NT_>
__global__ void __launch_bounds__(NT_ + 128, 2)
k_flow_iter_ws(WsArgs wa)
{
    using C = WsCfg<MT, NT_>;
    constexpr int NT = C::NT, TR = C::TR, SR = C::SR, RR = C::RR, TPP = C::TPP, NB = C::NB, LS = C::LS, NCH = C::NCH, m = MT;
    constexpr int NBUF = C::NBUF, BAR_FULL = 1, BAR_FREE = 1 + NBUF, BAR_SOLVED = 1 + 2 * NBUF;
    constexpr unsigned WARPS = (NT + 128) / 32;
    extern __shared__ __align__(128) unsigned char smem_ws[];
    double* tiles = reinterpret_cast<double*>(smem_ws);                       // [2][TR*5][LS]
    unsigned long long* chunk_bar = reinterpret_cast<unsigned long long*>(smem_ws + C::tiles_bytes);   // [NBUF][NCH]
    volatile int* sh = reinterpret_cast<volatile int*>(smem_ws + C::tiles_bytes + 8 * NBUF * NCH);
    const int h = wa.h, w = wa.w;
    const int t = threadIdx.x;
    const unsigned per_it = (unsigned)wa.n * (unsigned)wa.strips;
    if (t == 0) {
        const unsigned tk = atomicAdd(wa.ctl, 1u);
        sh[0] = (int)tk;
        const unsigned it0 = tk / per_it;
        if (it0 > 0) {   // every strip of this pair's previous iteration must have written its flow
            const unsigned b0 = (tk - it0 * per_it) / (unsigned)wa.strips;
            const unsigned* dn = wa.done + (size_t)(it0 - 1) * wa.n + b0;
            while (ld_acquire_u32(dn) < (unsigned)wa.strips) __nanosleep(200);
        }
    }
    if (t < NBUF * NCH) mbar_init(smem_u32(chunk_bar + t), 1);
    __syncthreads();
    const unsigned ticket = (unsigned)sh[0];
    const int it = (int)(ticket / per_it);
    const unsigned rem = ticket - (unsigned)it * per_it;
    const int b = (int)(rem / (unsigned)wa.strips);   // image pair
    const int k = (int)(rem - (unsigned)b * wa.strips);   // strip
    const unsigned tag = wa.tag + (unsigned)it;
    const int CW = wa.CW;
    const int x0 = k * CW;
    const int ncols = min(CW, w - x0);   // multiple of 4
    const int ntiles = (h + TR - 1) / TR;

    // every warp reports when it leaves; the last one of the grid re-arms the counters for the next launch
    auto warp_exit = [&]() {
        __syncwarp();
        unsigned last = 0;
        if ((t & 31) == 0) {
            __threadfence();
            last = atomicAdd(wa.ctl + 1, 1u) == gridDim.x * WARPS - 1u;
        }
        last = __shfl_sync(0xffffffffu, last, 0);
        if (last) {
            for (int i = t & 31; i < wa.iters * wa.n; i += 32) wa.done[i] = 0;
            if ((t & 31) == 0) { wa.ctl[0] = 0; wa.ctl[1] = 0; }
        }
    };

    if (t >= NT) {
#ifndef FDN_WS_RC4
#define FDN_WS_RC4 168
#define FDN_WS_RS4 88
#endif
        if (MT == 4) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" :: "n"(FDN_WS_RS4));
        else asm volatile("setmaxnreg.dec.sync.aligned.u32 80;");
        if (t >= NT + 32) {
            // =============================== solve warps: phase S ===============================
            // regularised 2x2 solve in float64, flow written once. Full tiles run as one straight-line block (the
            // rows are independent: the compiler interleaves their dependency chains).
            constexpr int NS = 96;   // solving lanes
            const int sl = t - (NT + 32);
            float2* fout = reinterpret_cast<float2*>(wa.fout[it]) + (int64_t)b * h * w;
            auto solve_px = [&](const double* tt, int r, float2* dst) {
                double g[5];
#pragma unroll
                for (int c = 0; c < 5; c++) g[c] = __dmul_rn(tt[(r * 5 + c) * LS], wa.scale);
                const double det = __dadd_rn(__dsub_rn(__dmul_rn(g[0], g[2]), __dmul_rn(g[1], g[1])), 1e-3);
                const double idet = __drcp_rn(det);  // == 1./det correctly rounded, like the IEEE division
                float2 o;
                o.x = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[0], g[4]), __dmul_rn(g[1], g[3])), idet);
                o.y = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[2], g[3]), __dmul_rn(g[1], g[4])), idet);
                *dst = o;
            };
            const int sw = sl >> 5, sln = sl & 31;
            const int qlast = (ncols - 1) >> 5;
            for (int j = 0; j < ntiles; j++) {
                const int y0 = j * TR;
                const int buf = j % NBUF;
                const uint32_t bars = smem_u32(chunk_bar + buf * NCH);
                const uint32_t parity = (uint32_t)((j / NBUF) & 1);
                // the solve follows the scan through the tile: 32-column chunk q goes to solve warp q % 3 as soon as the
                // scan warp has passed it
                for (int q = sw; q <= qlast; q += NS / 32) {
                    mbar_wait_sleep<FDN_WS_SOLVE_SLEEP>(bars + 8 * q, parity);
                    const int col = q * 32 + sln;
                    if (col < ncols && !FDN_WS_EXP(8)) {
                        const double* tt = tiles + buf * TR * 5 * LS + col;
                        float2* dst = fout + (int64_t)y0 * w + x0 + col;
                        if (y0 + TR <= h) {
#pragma unroll
                            for (int r = 0; r < TR; r++) solve_px(tt, r, dst + r * w);
                        } else {
                            for (int r = 0; r < h - y0; r++) solve_px(tt, r, dst + r * w);
                        }
                    }
                }
                // a warp without a chunk in this strip (narrow strips) must not run ahead of the tile either: its
                // arrival below has to count for THIS tile's phase of the FREE barrier
                mbar_wait_sleep<FDN_WS_SOLVE_SLEEP>(bars + 8 * qlast, parity);
                nbar_arrive(BAR_FREE + buf, NS + NT);     // this warp is done with the tile (phase V of tile j+NBUF may overwrite it)
            }
            if (it + 1 < wa.iters) {   // publish: this strip's flow of iteration `it` is in memory
                nbar_sync(BAR_SOLVED, NS);
                if (sl == 0) {
                    __threadfence();
                    atomicAdd(wa.done + (size_t)it * wa.n + b, 1u);
                }
            }
            warp_exit();
            return;
        }
        // =============================== scan warp: phase H ===============================
        const int lane = t - NT;
        const int r = lane / 5, c = lane - r * 5;
        ulonglong2* pk_out = wa.packets + ((int64_t)b * wa.strips + k) * h * 5;
        const ulonglong2* pk_in = wa.packets + ((int64_t)b * wa.strips + max(k - 1, 0)) * h * 5;
        constexpr int off = 2 * m + 1;
        static_assert(FDN_WS_HC == 8, "the sliding window below is written for 8-column chunks");
        for (int j = 0; j < ntiles; j++) {
            const int y = j * TR + r;
            const int buf = j % NBUF;
            const uint32_t bars = smem_u32(chunk_bar + buf * NCH);
            nbar_sync(BAR_FULL + buf, NT + 32);
            const unsigned hmask = __ballot_sync(0xffffffffu, lane < 5 * TR && y < h);   // the scanning lanes
            if (lane < 5 * TR && y < h) {
                double* line = tiles + (buf * TR * 5 + r * 5 + c) * LS;
                double2* l2 = reinterpret_cast<double2*>(line);   // 16-byte aligned (LS is even)
                // S(i) = S(i-1) + (vs[i+m] - vs[i-m-1]); S(i) overwrites the dead slot of column i-m-1.
                // The line is read ONCE, 128 bits at a time, through a sliding window of two 8-column sets (plus, for
                // winsize 9, the first pair of the third): while the chain of chunk k runs (8 dependent DADDs, then four
                // 128-bit stores) the set after next is in flight and the differences of chunk k+1 are formed from the
                // sets in registers. positions 8k .. 8k+7 = set k; d_k[u] = pos[8k + u + off] - pos[8k + u].
#define FDN_LOADSET(W, kk)                                                        \
    { W[0] = l2[4 * (kk)]; W[1] = l2[4 * (kk) + 1]; W[2] = l2[4 * (kk) + 2]; W[3] = l2[4 * (kk) + 3];   \
      if (off > 7) xx_ = l2[4 * (kk) + 4]; }
#define FDN_CHAIN8(D, kk)                                                          \
    {                                                                              \
        double2 s0, s1, s2, s3;                                                    \
        S = __dadd_rn(S, D[0]); s0.x = S; S = __dadd_rn(S, D[1]); s0.y = S;        \
        S = __dadd_rn(S, D[2]); s1.x = S; S = __dadd_rn(S, D[3]); s1.y = S;        \
        S = __dadd_rn(S, D[4]); s2.x = S; S = __dadd_rn(S, D[5]); s2.y = S;        \
        S = __dadd_rn(S, D[6]); s3.x = S; S = __dadd_rn(S, D[7]); s3.y = S;        \
        l2[4 * (kk)] = s0; l2[4 * (kk) + 1] = s1; l2[4 * (kk) + 2] = s2; l2[4 * (kk) + 3] = s3; \
    }
                // every 32 columns: wake the solve warp that owns the chunk (the last chunk is announced after the loop)
#define FDN_CHUNK_DONE(kk)                                                         \
    if (((kk) & 3) == 0 && 8 * (kk) < ncols) {                                     \
        __syncwarp(hmask);                                                         \
        if (lane == 0) mbar_arrive(bars + 8 * (((kk) >> 2) - 1));                  \
    }
                const int n8 = ncols >> 3;   // full chunks; ncols % 8 is 0 or 4
                double2 wa_[4], wb_[4], xx_ = make_double2(0., 0.);   // xx_: first pair of the set after the newest one
                double d[8];
                FDN_LOADSET(wa_, 0);
                FDN_LOADSET(wb_, 1);   // (a line has LS >= ncols + 2m + 1 + 8 readable positions)
                double S;
                if (k == 0) {
                    // g = vsum[0]*(m+2) + vsum[1] + ... + vsum[m-1]   (columns clamp to the replicated border)
                    S = __dmul_rn(line[m + 1], (double)(m + 2));
#pragma unroll
                    for (int x = 1; x < m; x++) S = __dadd_rn(S, line[m + 1 + x]);
                } else if (FDN_WS_EXP(2)) {
                    S = 0.;
                } else {
                    const ulonglong2* src = pk_in + (int64_t)y * 5 + c;
                    ulonglong2 v = __ldcv(src);
                    while ((unsigned)(v.x >> 32) != tag || (unsigned)(v.y >> 32) != tag) {
                        __nanosleep(32);
                        v = __ldcv(src);
                    }
                    S = __hiloint2double((int)(unsigned)v.y, (int)(unsigned)v.x);
                }
                __syncwarp(hmask);   // the lanes leave their polling loops one by one: scan in lockstep from here on
                if (!FDN_WS_EXP(1)) {
                    ws_diffs<off>(d, wa_, wb_, xx_);
                    int kk = 0;
                    while (kk < n8) {
                        // sets: wa_ = kk, wb_ = kk+1; d = differences of chunk kk
                        FDN_LOADSET(wa_, kk + 2);
                        FDN_CHAIN8(d, kk);
                        ws_diffs<off>(d, wb_, wa_, xx_);
                        ++kk;
                        FDN_CHUNK_DONE(kk);
                        if (kk == n8) break;
                        // sets: wb_ = kk, wa_ = kk+1
                        FDN_LOADSET(wb_, kk + 2);
                        FDN_CHAIN8(d, kk);
                        ws_diffs<off>(d, wa_, wb_, xx_);
                        ++kk;
                        FDN_CHUNK_DONE(kk);
                    }
                    if (ncols & 4) {   // d[0..3] are the differences of the last 4 columns
                        double2 s0, s1;
                        S = __dadd_rn(S, d[0]); s0.x = S; S = __dadd_rn(S, d[1]); s0.y = S;
                        S = __dadd_rn(S, d[2]); s1.x = S; S = __dadd_rn(S, d[3]); s1.y = S;
                        l2[4 * n8] = s0; l2[4 * n8 + 1] = s1;
                    }
                }
#undef FDN_LOADSET
#undef FDN_CHAIN8
#undef FDN_CHUNK_DONE
                if (k + 1 < wa.strips) {
                    ulonglong2 o;
                    const unsigned long long tg = (unsigned long long)tag << 32;
                    o.x = tg | (unsigned)__double2loint(S);
                    o.y = tg | (unsigned)__double2hiint(S);
                    __stcg(pk_out + (int64_t)y * 5 + c, o);
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bars + 8 * ((ncols - 1) >> 5));   // the last chunk: the whole tile is scanned
        }
        warp_exit();
        return;
    }

    // =============================== column warps: phase V ===============================
    if (MT == 4) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" :: "n"(FDN_WS_RC4));
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 176;");
    // thread t <-> tile position t <-> image column x0 - m - 1 + t (clamped: replicated border); threads beyond the
    // strip's halo work on a clamped column too, their results are never read
    const int xcl = min(max(x0 - m - 1 + t, 0), w - 1);
    const float sxc = __fmul_rn(xcl < 5 ? (xcl < 2 ? 0.14f : 0.4472f) : 1.f,
                                xcl >= w - 5 ? (w - xcl - 1 < 2 ? 0.14f : 0.4472f) : 1.f);

    const float* R0 = wa.R + (int64_t)wa.map0.slot(b) * wa.R_stride;
    const float* R1 = wa.R + (int64_t)wa.map1.slot(b) * wa.R_stride;
    const float4* R0a = reinterpret_cast<const float4*>(R0);
    const float* R0b = R0 + (int64_t)4 * h * w;
    const float4* R1a = reinterpret_cast<const float4*>(R1);
    const float* R1b = R1 + (int64_t)4 * h * w;
    const float2* fin = reinterpret_cast<const float2*>(wa.fin[it]) + (int64_t)b * h * w;

    // R0 / flow of one row of this thread's column: read once, streamed past L1's resident R1 rows. The flow may
    // have been written by another SM earlier in this launch (previous iteration): L2 is the point of coherence.
    auto load_row = [&](int y) {
        RowIn in;
        const int idx = min(y, h - 1) * w + xcl;
        asm volatile("ld.global.cg.v2.f32 {%0, %1}, [%2];" : "=f"(in.f.x), "=f"(in.f.y) : "l"(fin + idx));
        asm("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                     : "=f"(in.c03.x), "=f"(in.c03.y), "=f"(in.c03.z), "=f"(in.c03.w) : "l"(R0a + idx));
        asm("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(in.c4) : "l"(R0b + idx));
#if FDN_WS_L2PF
        // The six scoreboard slots of a warp are shared between these loads and the R1 gathers: a gather's first use
        // also waits for every streaming load in flight on the same slot. Bring the row into L2 FDN_WS_L2PF tiles
        // before it is loaded (prefetches take no scoreboard slot), so that what a gather may wait for is an L2 hit.
        const int idp = min(y + (FDN_WS_L2PF > 0 ? FDN_WS_L2PF : -FDN_WS_L2PF) * TR, h - 1) * w + xcl;
#if FDN_WS_L2PF > 0
        asm volatile("prefetch.global.L2 [%0];" :: "l"(fin + idp));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(R0a + idp));
        asm volatile("prefetch.global.L2 [%0];" :: "l"(R0b + idp));
#else
        asm volatile("prefetch.global.L1 [%0];" :: "l"(fin + idp));
        asm volatile("prefetch.global.L1 [%0];" :: "l"(R0a + idp));
        asm volatile("prefetch.global.L1 [%0];" :: "l"(R0b + idp));
#endif
#endif
        return in;
    };

    float Mring[RR][5];
    double vs[5];
    RowIn cur[TR];
    {
        // rows 0 .. m-1 seed the column sums: vsum = M[0]*(m+2) + sum_{y=1}^{m-1} M[min(y,h-1)]
#pragma unroll
        for (int y = 0; y < m; y++) {
            const RowIn in = load_row(y);
            const Taps tp = ws_gather<0>(in.f, R1a, R1b, xcl, min(y, h - 1), h, w);
            ws_matrices_px(in, tp, xcl, min(y, h - 1), h, w, sxc, Mring[y]);
        }
        const float mp2 = (float)(m + 2);
#pragma unroll
        for (int c = 0; c < 5; c++) vs[c] = (double)__fmul_rn(Mring[0][c], mp2);
#pragma unroll
        for (int y = 1; y < m; y++)
#pragma unroll
            for (int c = 0; c < 5; c++) vs[c] = __dadd_rn(vs[c], (double)Mring[y][c]);
        // steps y = 0 .. m of the first tile subtract row max(y-m-1, 0) = row 0: park copies of it in the slots those
        // steps read (slot (y+m+1) % RR), so that tile 0 runs the same code as every other tile
#pragma unroll
        for (int s = m; s < RR; s++)
#pragma unroll
            for (int c = 0; c < 5; c++) Mring[s][c] = Mring[0][c];
#pragma unroll
        for (int r = 0; r < TR; r++) cur[r] = load_row(r + m);
    }

    // One trip of the outer loop = one ring period = TPP tiles: every ring slot below is a compile-time constant.
    for (int jp = 0; jp < ntiles; jp += TPP) {
#pragma unroll
        for (int tp = 0; tp < TPP; tp++) {
            const int j = jp + tp;
            if (TPP > 1 && j >= ntiles) break;
            const int y0 = j * TR;
            const int buf = (TPP == 2 && NBUF == 2) ? tp : j % NBUF;   // (jp is even when a period is two tiles)
            double* tq = tiles + buf * TR * 5 * LS + t;
            if (j >= NBUF) nbar_sync(BAR_FREE + buf, 96 + NT);   // tile j-NBUF has been solved: its shared-memory tile is free
            // ---------------- phase V ----------------
#pragma unroll
            for (int blk = 0; blk < NB; blk++) {
                // the (up to) SR rows of a block are independent up to the column sums: one straight-line block (all the
                // gathers first, then the arithmetic of the rows interleaved by the compiler).
                Taps tps[SR];
#pragma unroll
                for (int rr = 0; rr < SR; rr++) {
                    const int r = blk * SR + rr;
                    if (r < TR) tps[rr] = ws_gather<FDN_WS_PF>(cur[r].f, R1a, R1b, xcl, min(y0 + r + m, h - 1), h, w);
                }
                float Mv[SR][5];
#pragma unroll
                for (int rr = 0; rr < SR; rr++) {
                    const int r = blk * SR + rr;
                    if (r < TR) ws_matrices_px(cur[r], tps[rr], xcl, min(y0 + r + m, h - 1), h, w, sxc, Mv[rr]);
                }
                // The column-sum update sits behind a branch the compiler cannot fold (the packet tag is never 0): it
                // keeps the blocks of a tile apart for the scheduler. Merged into one basic block, ptxas hoists the
                // gathers of all rows, the register allocation collapses and the launch is 20 % slower (measured: 10.3
                // instead of 8.5 ms for 512 pairs).
                if (wa.tag != 0 && !FDN_WS_EXP(4)) {
#pragma unroll
                    for (int rr = 0; rr < SR; rr++) {
                        const int r = blk * SR + rr;
                        if (r < TR) {
                            const int snew = (tp * TR + r + m) % RR, sold = (tp * TR + r + m + 1) % RR;
#pragma unroll
                            for (int c = 0; c < 5; c++) {
                                const float d = __fsub_rn(Mv[rr][c], Mring[sold][c]);
                                Mring[snew][c] = Mv[rr][c];
                                vs[c] = __dadd_rn(vs[c], (double)d);
                                tq[(r * 5 + c) * LS] = vs[c];
                            }
                        }
                    }
                }
                // R0 / flow of the same rows of the NEXT tile: in flight for a whole tile period
#pragma unroll
                for (int rr = 0; rr < SR; rr++) {
                    const int r = blk * SR + rr;
                    if (r < TR) cur[r] = load_row(y0 + TR + r + m);
                }
            }
#ifndef FDN_WS_NOFENCE
            __threadfence_block();
#endif
            nbar_arrive(BAR_FULL + buf, NT + 32);          // the scan warp may start on tile j
        }
    }
    warp_exit();
}

static std::atomic<unsigned long long> g_flow_epoch{1};
static std::atomic<int> g_flow_variant{1};
void set_flow_iter_variant(int v) { g_flow_variant.store(v ? 1 : 0); }

static int strip_width(int w) { return w > 96 ? 128 : 32; }   // k_flow_iter

// packet tags of one k_flow_iter_ws launch: cnt consecutive 32-bit values, none of them 0
static unsigned next_packet_tags(int cnt)
{
    for (;;) {
        const unsigned lo = (unsigned)g_flow_epoch.fetch_add((unsigned long long)cnt);
        if (lo != 0 && lo <= 0xffffffffu - (unsigned)cnt) return lo;
    }
}

// strips of k_flow_iter_ws: CW = multiple of 4, <= WsCfg::CWMAX
static int ws_strip_width(int w, int cwmax)
{
    const int strips = (int)cdiv(w, cwmax);
    return (int)((cdiv(w, strips) + 3) / 4 * 4);
}
#define FDN_WS_NT 128
typedef WsCfg<2, FDN_WS_NT> WsCfg2;   // winsize 5
typedef WsCfg<4, FDN_WS_NT> WsCfg4;   // winsize 9
static int ws_strips_max(int w)   // strips of the narrower configuration: what the packet area is sized for
{
    const int a = (int)cdiv(w, ws_strip_width(w, WsCfg2::CWMAX)), b = (int)cdiv(w, ws_strip_width(w, WsCfg4::CWMAX));
    return a > b ? a : b;
}

static size_t align256(size_t v) { return (v + 255) / 256 * 256; }

// Scratch layout (offsets depend on the capacity only, see FlowScratch):
//   [ctl: tickets taken, warps / blocks finished]                                    256 B, zero between launches
//   [done: FDN_WS_MAX_ITERS x cap_n counters of k_flow_iter_ws]                       zero between launches
//   [flags: cap_n x strips epochs of k_flow_iter]                                     only ever grow
//   [packets of k_flow_iter_ws: cap_n x strips x h x 5 tagged 16-byte pairs]
//   [carries of k_flow_iter:    cap_n x strips x h x 5 doubles]
// Each area holds the largest of the nlev levels (hs[k] x ws[k]) it may serve. That is not always level 0: a
// narrower level can need more strips (97..128 px: 1 strip of k_flow_iter, 48..64 px: 2), and cvRound rounds an odd
// height up (67 rows -> 34). The two carry areas are disjoint, so a level run by one kernel never writes where the
// other kernel polls at another level (a plain double must never be mistaken for a tagged packet). A smaller launch
// (coarser level, last chunk of a pass) uses a prefix of each area.
int flow_scratch_make(void* scratch, size_t bytes, int cap_n, int nlev, const int* hs, const int* ws, FlowScratch* fs)
{
    fs->base = static_cast<char*>(scratch);
    fs->bytes = bytes;
    fs->cap_n = cap_n; fs->H = 0; fs->W = 0;
    fs->flag_strips = 0; fs->packet_rows = 0; fs->carry_rows = 0;
    for (int k = 0; k < nlev; k++) {
        const int h = hs[k], w = ws[k];
        const int strips = (int)cdiv(w, strip_width(w));
        if (h > fs->H) fs->H = h;
        if (w > fs->W) fs->W = w;
        if (strips > fs->flag_strips) fs->flag_strips = strips;
        if ((int64_t)ws_strips_max(w) * h > fs->packet_rows) fs->packet_rows = (int64_t)ws_strips_max(w) * h;
        if ((int64_t)strips * h > fs->carry_rows) fs->carry_rows = (int64_t)strips * h;
    }
    size_t off = 256;
    fs->off_done = off;    off += align256(sizeof(unsigned) * FDN_WS_MAX_ITERS * (size_t)cap_n);
    fs->off_flags = off;   off += align256(sizeof(unsigned long long) * (size_t)cap_n * fs->flag_strips);
    fs->off_packets = off; off += align256(sizeof(ulonglong2) * 5 * (size_t)cap_n * (size_t)fs->packet_rows);
    fs->off_carry = off;   off += align256(sizeof(double) * 5 * (size_t)cap_n * (size_t)fs->carry_rows);
    if (scratch && bytes < off) {
        set_error("flow iteration scratch too small: need %zu bytes, got %zu", off, bytes);
        return FDN_ERR_WORKSPACE;
    }
    fs->bytes = off;
    return FDN_OK;
}

size_t flow_iter_scratch_bytes(int cap_n, int nlev, const int* hs, const int* ws)
{
    FlowScratch fs;
    flow_scratch_make(nullptr, 0, cap_n, nlev, hs, ws, &fs);
    return fs.bytes;
}

int flow_iter_scratch_init(const FlowScratch& fs, cudaStream_t st)
{
    // counters and flags must start at zero; carries / packets need no initialisation but a stale bit pattern must
    // not look like a packet of a future launch: zero everything once per pass
    FDN_CUDA(cudaMemsetAsync(fs.base, 0, fs.bytes, st));
    return FDN_OK;
}

// function attributes are per device: remember which devices of this process have them
static bool first_use_on_device(std::atomic<bool> (&seen)[64])
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return true;
    return !seen[dev].exchange(true);
}

template <int CW, int TR, int MT, int MINB>
static int launch_flow_variant(const FlowIterArgs& a, unsigned blocks, size_t smem, cudaStream_t st)
{
    static std::atomic<bool> seen[64];
    if (first_use_on_device(seen))
        FDN_CUDA(cudaFuncSetAttribute(k_flow_iter<CW, TR, MT, MINB>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      200 * 1024));
    k_flow_iter<CW, TR, MT, MINB><<<blocks, CW + 32, smem, st>>>(a);
    return FDN_OK;
}

// one iteration with the strip kernel
static int launch_flow_iter_strip(const float* R, int64_t R_stride, SlotMap map0, SlotMap map1, const float* flow_in,
                                  float* flow_out, int n, int h, int w, int winsize, const FlowScratch& fs,
                                  cudaStream_t st)
{
    FlowIterArgs a;
    a.R = R; a.R_stride = R_stride;
    a.h = h; a.w = w; a.m = winsize / 2;
    a.n = n;
    a.scale = 1. / ((double)winsize * winsize);
    const int m = a.m;
    const int RR = 2 * m + 2;
    const bool wide = w > 96;
    const int CW = strip_width(w);
    const int NT = CW + 32;
    // tile rows per step: 6 when the compile-time m = 2 kernel applies (ring rows = tile rows), else 4
    const int TR = (wide && m == 2) ? 6 : 4;
    a.strips = (int)cdiv(w, CW);
    a.LS = tile_line_stride(CW, m);
    FDN_CHECK_ARG(a.strips <= fs.flag_strips && (int64_t)a.strips * h <= fs.carry_rows,
                  "flow iteration scratch was not sized for a %d x %d level", h, w);
    FDN_CHECK_ARG((int64_t)n * a.strips < (1ll << 31), "too many image pairs in one launch");
    a.ctl = reinterpret_cast<unsigned*>(fs.base);
    a.flags = reinterpret_cast<unsigned long long*>(fs.base + fs.off_flags);
    a.carry = reinterpret_cast<double*>(fs.base + fs.off_carry);
    const size_t smem = sizeof(double) * TR * 5 * a.LS + sizeof(float) * RR * 5 * NT;
    const unsigned long long tiles = (unsigned long long)cdiv(h, TR);
    a.map0 = map0; a.map1 = map1;
    a.flow_in = flow_in; a.flow_out = flow_out;
    a.epoch = g_flow_epoch.fetch_add(tiles + 1);
    ProfScope ps(K_FLOW_ITER, 56.0 * n * h * w, st, n, h, w);
    const unsigned blocks = (unsigned)a.strips * (unsigned)n;
    int rc;
    if (wide) {
        if (m == 2) rc = launch_flow_variant<128, 6, 2, 4>(a, blocks, smem, st);
        else if (m == 4) rc = launch_flow_variant<128, 4, 4, 4>(a, blocks, smem, st);
        else rc = launch_flow_variant<128, 4, 0, 4>(a, blocks, smem, st);
    } else {
        if (m == 2) rc = launch_flow_variant<32, 4, 2, 8>(a, blocks, smem, st);
        else rc = launch_flow_variant<32, 4, 0, 8>(a, blocks, smem, st);
    }
    if (rc) return rc;
    FDN_LAUNCHED("k_flow_iter");
    return FDN_OK;
}

template <int MT>
static int launch_ws(const WsArgs& wa, unsigned blocks, cudaStream_t st)
{
    using C = WsCfg<MT, FDN_WS_NT>;
    static std::atomic<bool> seen[64];
    if (first_use_on_device(seen)) {
        FDN_CUDA(cudaFuncSetAttribute(k_flow_iter_ws<MT, FDN_WS_NT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)C::smem_bytes));
        // leave the rest of the SM's L1/shared array to L1: the R1 rows a strip walks over live there
        FDN_CUDA(cudaFuncSetAttribute(k_flow_iter_ws<MT, FDN_WS_NT>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                      (int)((2 * (C::smem_bytes + 1024) * 100 + 228 * 1024 - 1) / (228 * 1024))));
        if (getenv("FDN_DEBUG")) {
            int nb = 0;
            cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_flow_iter_ws<MT, FDN_WS_NT>, FDN_WS_NT + 128, C::smem_bytes);
            fprintf(stderr, "[fdn] k_flow_iter_ws<%d>: %d blocks/SM, %zu B shared memory per block\n", MT, nb,
                    (size_t)C::smem_bytes);
        }
    }
    k_flow_iter_ws<MT, FDN_WS_NT><<<blocks, FDN_WS_NT + 128, C::smem_bytes, st>>>(wa);
    return FDN_OK;
}

int launch_flow_level(const float* R, int64_t R_stride, SlotMap map0, SlotMap map1, float* cur, float* bufa, float* bufb,
                      int n, int h, int w, int winsize, int iters, const FlowScratch& fs, cudaStream_t st,
                      float** result)
{
    FDN_CHECK_ARG(winsize >= 1 && winsize <= 31, "winsize %d unsupported (1..31)", winsize);
    FDN_CHECK_ARG(cur != bufa && cur != bufb && bufa != bufb, "the three flow buffers must be distinct");
    FDN_CHECK_ARG((int64_t)h * w < (1ll << 28), "level image too large");
    FDN_CHECK_ARG(n >= 1 && n <= fs.cap_n && h <= fs.H && w <= fs.W, "flow iteration scratch was sized for %d pairs of %d x %d",
                  fs.cap_n, fs.H, fs.W);
    float* bufs[3] = {cur, bufa, bufb};
    const int m = winsize / 2;
    // warp-specialised variant (default for winsize 5 on images that are not tiny)
    const bool win = g_flow_variant.load() == 1 && (m == 2 || m == 4) && w % 4 == 0 && w >= 64 && h >= 16 &&
                     (reinterpret_cast<uintptr_t>(R) & 15) == 0 && R_stride % 4 == 0;
    if (!win) {
        for (int i = 0; i < iters; i++) {
            int rc = launch_flow_iter_strip(R, R_stride, map0, map1, bufs[i % 3], bufs[(i + 1) % 3], n, h, w, winsize, fs,
                                            st);
            if (rc) return rc;
        }
        *result = bufs[iters % 3];
        return FDN_OK;
    }
    WsArgs wa;
    wa.R = R; wa.R_stride = R_stride;
    wa.map0 = map0; wa.map1 = map1;
    wa.n = n; wa.h = h; wa.w = w;
    wa.scale = 1. / ((double)winsize * winsize);
    wa.CW = ws_strip_width(w, m == 2 ? WsCfg2::CWMAX : WsCfg4::CWMAX);
    wa.strips = (int)cdiv(w, wa.CW);
    FDN_CHECK_ARG((int64_t)wa.strips * h <= fs.packet_rows, "flow iteration scratch was not sized for a %d x %d level",
                  h, w);
    FDN_CHECK_ARG((int64_t)n * wa.strips * FDN_WS_MAX_ITERS < (1ll << 31), "too many image pairs in one launch");
    wa.ctl = reinterpret_cast<unsigned*>(fs.base);
    wa.done = reinterpret_cast<unsigned*>(fs.base + fs.off_done);
    wa.packets = reinterpret_cast<ulonglong2*>(fs.base + fs.off_packets);
    wa.exp = 0;
#ifdef FDN_WS_EXPERIMENTS   // phase-removal timing experiments of tools/flow_iter_lab.py (FDN_EXP bit mask): wrong results
    { const char* e = getenv("FDN_EXP"); wa.exp = e ? atoi(e) : 0; }
#endif
#ifdef FDN_WS_ITERS_PER_LAUNCH
    const int per_launch = FDN_WS_ITERS_PER_LAUNCH;
#else
    const int per_launch = FDN_WS_MAX_ITERS;
#endif
    for (int i0 = 0; i0 < iters; i0 += per_launch) {
        const int cnt = iters - i0 < per_launch ? iters - i0 : per_launch;
        for (int i = 0; i < cnt; i++) {
            wa.fin[i] = bufs[(i0 + i) % 3];
            wa.fout[i] = bufs[(i0 + i + 1) % 3];
        }
        for (int i = cnt; i < FDN_WS_MAX_ITERS; i++) { wa.fin[i] = nullptr; wa.fout[i] = nullptr; }
        wa.iters = cnt;
        wa.tag = next_packet_tags(cnt);
        ProfScope ps(K_FLOW_ITER, 56.0 * cnt * n * h * w, st, n, h, w);
        const unsigned blocks = (unsigned)cnt * (unsigned)n * (unsigned)wa.strips;
        int rc = m == 2 ? launch_ws<2>(wa, blocks, st) : launch_ws<4>(wa, blocks, st);
        if (rc) return rc;
        FDN_LAUNCHED("k_flow_iter_ws");
    }
    *result = bufs[iters % 3];
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN, FarnebackUpdateFlow_GaussianBlur): M is smoothed by a separable
// Gaussian of 2m+1 float32 taps (sigma = 0.3 m) instead of the box mean, then the same regularised solve without the
// 1/winsize^2 scale. OpenCV's order, no FMA:
//   vertical   v(y, x)  = M[y]*k0 + sum_{i=1..m} (M[min(y+i, h-1)] + M[max(y-i, 0)]) * k[i]     (float32)
//   horizontal g(y, x)  = v[x]*k0 + sum_{i=1..m} (v[min(x+i, w-1)] + v[max(x-i, 0)]) * k[i]     (float32)
// Nothing runs along a row or a column, so the filter is tile local and still bit exact: a block owns a strip of CW
// output columns of one image pair plus an m-column halo on each side (128 threads, thread t <-> image column
// x0 - m + t, clamped: the replicated border), and marches down the rows. Per row a thread computes M of the new row
// y + m from R0, flow_in and the R1 gather (update_matrices_px, the arithmetic of phase V of k_flow_iter), keeps the
// last 2m+1 rows of M in a ring, and writes the vertical sums of its column to a shared-memory tile; after a barrier
// the CW core threads run the horizontal sums and the solve of the tile's rows. No carries, no tickets, no scratch:
// blocks are independent. Rows past the bottom are recomputed at row h-1 and the m rows above the top hold M of
// row 0, so every step of the march is the same. Algorithmic HBM bytes per pixel: 56, as for the box kernels.
//   k_flow_gauss_iter       (MT = 2, 4: winsize 4/5, 8/9): the ring lives in registers, a tile is one ring period
//                           (2m+1 rows) so every ring slot is a compile-time constant of the unrolled row loop;
//   k_flow_gauss_iter_smem  (any m <= 15): the ring lives in shared memory, tiles of GW_TR rows.
// ------------------------------------------------------------------------------------------------
#define GW_NT 128
#define GW_TR 8
#define GW_MAX_M 15

struct GaussIterArgs {
    const float* R;      // level base inside slot 0 (layout as FlowIterArgs)
    int64_t R_stride;
    SlotMap map0, map1;
    const float* flow_in;
    float* flow_out;
    int h, w, m;
    int CW, strips;      // core columns per strip (GW_NT - 2m), strips per image
    float k[GW_MAX_M + 1];
};

// taps as OpenCV builds them (float, normalised through a double sum)
static void gauss_window_taps(int m, float* k)
{
    const double sigma = m * 0.3;
    double s = 1;
    k[0] = (float)s;
    for (int i = 1; i <= m; i++) {
        const float t = (float)exp(-i * i / (2 * sigma * sigma));
        k[i] = t;
        s += t * 2;
    }
    s = 1. / s;
    for (int i = 0; i <= m; i++) k[i] = (float)(k[i] * s);
}

template <int MT>
__global__ void __launch_bounds__(GW_NT, 4)
k_flow_gauss_iter(GaussIterArgs a)
{
    constexpr bool kReg = MT > 0;
    extern __shared__ __align__(16) float gw_smem[];
    const int m = kReg ? MT : a.m;
    const int RR = 2 * m + 1;
    const int TR = kReg ? 2 * MT + 1 : GW_TR;
    const int h = a.h, w = a.w;
    float* tile = gw_smem;                       // [TR][5][GW_NT] vertical sums
    float* ring = gw_smem + TR * 5 * GW_NT + threadIdx.x;   // [RR][5][GW_NT] rows of M (shared-memory variant)

    const int t = threadIdx.x;
    const int b = blockIdx.x / a.strips, k = blockIdx.x - b * a.strips;
    const int x0 = k * a.CW;
    const int xcol = x0 - m + t;
    const bool active = xcol <= w - 1 + m;       // columns past the right halo of a narrow image are not needed
    const int xcl = min(max(xcol, 0), w - 1);
    const bool core = t < a.CW && x0 + t < w;

    const float* R0 = a.R + (int64_t)a.map0.slot(b) * a.R_stride;
    const float* R1 = a.R + (int64_t)a.map1.slot(b) * a.R_stride;
    const float4* R0a = reinterpret_cast<const float4*>(R0);
    const float4* R1a = reinterpret_cast<const float4*>(R1);
    const float* R0b = R0 + (int64_t)4 * h * w;
    const float* R1b = R1 + (int64_t)4 * h * w;
    const float2* fin = reinterpret_cast<const float2*>(a.flow_in) + (int64_t)b * h * w;
    float2* fout = reinterpret_cast<float2*>(a.flow_out) + (int64_t)b * h * w;

    auto matrices = [&](int row, float M[5]) {
        update_matrices_px(R0a, R0b, R1a, R1b, __ldg(fin + row * w + xcl), xcl, row, h, w, M);
    };
    // horizontal sums + solve of tile row r (image row y), core threads
    auto solve_row = [&](int r, int y) {
        const float* tl = tile + r * 5 * GW_NT + t + m;
        double g[5];
#pragma unroll
        for (int c = 0; c < 5; c++) {
            const float* v = tl + c * GW_NT;
            float s = __fmul_rn(v[0], a.k[0]);
            if (kReg) {
#pragma unroll
                for (int i = 1; i <= MT; i++) s = __fadd_rn(s, __fmul_rn(__fadd_rn(v[i], v[-i]), a.k[i]));
            } else {
                for (int i = 1; i <= m; i++) s = __fadd_rn(s, __fmul_rn(__fadd_rn(v[i], v[-i]), a.k[i]));
            }
            g[c] = (double)s;
        }
        const double det = __dadd_rn(__dsub_rn(__dmul_rn(g[0], g[2]), __dmul_rn(g[1], g[1])), 1e-3);
        const double idet = __drcp_rn(det);   // == 1./det correctly rounded
        float2 o;
        o.x = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[0], g[4]), __dmul_rn(g[1], g[3])), idet);
        o.y = (float)__dmul_rn(__dsub_rn(__dmul_rn(g[2], g[3]), __dmul_rn(g[1], g[4])), idet);
        fout[y * w + x0 + t] = o;
    };

    if constexpr (kReg) {
        constexpr int RRc = 2 * MT + 1;
        float rg[RRc][5];   // row j of M in slot j mod RR (rows -m..-1 hold row 0)
        if (active) {
            float M0[5];
            matrices(0, M0);
#pragma unroll
            for (int j = -MT; j <= 0; j++)
#pragma unroll
                for (int c = 0; c < 5; c++) rg[(j + RRc) % RRc][c] = M0[c];
#pragma unroll
            for (int j = 1; j < MT; j++) matrices(min(j, h - 1), rg[j]);
        }
        for (int y0 = 0; y0 < h; y0 += RRc) {   // y0 = 0 mod RR: row y0 + r + i sits in slot (r + i) mod RR
            if (active) {
#pragma unroll
                for (int r = 0; r < RRc; r++) {
                    const int y = y0 + r;
                    if (y < h) {
                        matrices(min(y + MT, h - 1), rg[(r + MT) % RRc]);
#pragma unroll
                        for (int c = 0; c < 5; c++) {
                            float s = __fmul_rn(rg[r][c], a.k[0]);
#pragma unroll
                            for (int i = 1; i <= MT; i++)
                                s = __fadd_rn(s, __fmul_rn(__fadd_rn(rg[(r + i) % RRc][c], rg[(r - i + RRc) % RRc][c]),
                                                          a.k[i]));
                            tile[(r * 5 + c) * GW_NT + t] = s;
                        }
                    }
                }
            }
            __syncthreads();
            if (core) {
#pragma unroll
                for (int r = 0; r < RRc; r++)
                    if (y0 + r < h) solve_row(r, y0 + r);
            }
            __syncthreads();
        }
    } else {
        // ring slot of row j: (j + m) mod RR, kept as a running index (rows -m..-1 hold row 0)
        if (active) {
            float M0[5];
            matrices(0, M0);
            for (int j = -m; j <= 0; j++)
#pragma unroll
                for (int c = 0; c < 5; c++) ring[((j + m) * 5 + c) * GW_NT] = M0[c];
            for (int j = 1; j < m; j++) {
                float Mv[5];
                matrices(min(j, h - 1), Mv);
#pragma unroll
                for (int c = 0; c < 5; c++) ring[((j + m) * 5 + c) * GW_NT] = Mv[c];
            }
        }
        int sy = m;   // slot of row y
        for (int y0 = 0; y0 < h; y0 += GW_TR) {
            if (active) {
                for (int r = 0; r < GW_TR && y0 + r < h; r++) {
                    const int y = y0 + r;
                    int sn = sy + m;   // slot of the new row y + m
                    if (sn >= RR) sn -= RR;
                    float Mv[5];
                    matrices(min(y + m, h - 1), Mv);
#pragma unroll
                    for (int c = 0; c < 5; c++) ring[(sn * 5 + c) * GW_NT] = Mv[c];
#pragma unroll
                    for (int c = 0; c < 5; c++) {
                        const float* rc = ring + c * GW_NT;
                        float s = __fmul_rn(rc[sy * 5 * GW_NT], a.k[0]);
                        int sd = sy, su = sy;
                        for (int i = 1; i <= m; i++) {
                            if (++sd == RR) sd = 0;
                            if (--su < 0) su = RR - 1;
                            s = __fadd_rn(s, __fmul_rn(__fadd_rn(rc[sd * 5 * GW_NT], rc[su * 5 * GW_NT]), a.k[i]));
                        }
                        tile[(r * 5 + c) * GW_NT + t] = s;
                    }
                    if (++sy == RR) sy = 0;
                }
            }
            __syncthreads();
            if (core) {
                for (int r = 0; r < GW_TR && y0 + r < h; r++) solve_row(r, y0 + r);
            }
            __syncthreads();
        }
    }
}

static size_t gauss_smem_bytes(int MT, int m)
{
    const int TR = MT > 0 ? 2 * MT + 1 : GW_TR;
    return sizeof(float) * 5 * GW_NT * (size_t)(TR + (MT > 0 ? 0 : 2 * m + 1));
}

template <int MT>
static int launch_gauss_variant(const GaussIterArgs& a, unsigned blocks, cudaStream_t st)
{
    static std::atomic<bool> seen[64];
    if (first_use_on_device(seen))
        FDN_CUDA(cudaFuncSetAttribute(k_flow_gauss_iter<MT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)gauss_smem_bytes(MT, GW_MAX_M)));
    k_flow_gauss_iter<MT><<<blocks, GW_NT, gauss_smem_bytes(MT, a.m), st>>>(a);
    return FDN_OK;
}

int launch_flow_level_gauss(const float* R, int64_t R_stride, SlotMap map0, SlotMap map1, float* cur, float* bufa,
                            float* bufb, int n, int h, int w, int winsize, int iters, cudaStream_t st, float** result)
{
    FDN_CHECK_ARG(winsize >= 1 && winsize <= 31, "winsize %d unsupported (1..31)", winsize);
    FDN_CHECK_ARG(cur != bufa && cur != bufb && bufa != bufb, "the three flow buffers must be distinct");
    FDN_CHECK_ARG((int64_t)h * w < (1ll << 28), "level image too large");
    GaussIterArgs a;
    a.R = R; a.R_stride = R_stride;
    a.map0 = map0; a.map1 = map1;
    a.h = h; a.w = w; a.m = winsize / 2;
    a.CW = GW_NT - 2 * a.m;
    a.strips = (int)cdiv(w, a.CW);
    FDN_CHECK_ARG((int64_t)n * a.strips < (1ll << 31), "too many image pairs in one launch");
    gauss_window_taps(a.m, a.k);
    const unsigned blocks = (unsigned)n * (unsigned)a.strips;
    const bool reg = g_flow_variant.load() == 1 && (a.m == 2 || a.m == 4);
    float* bufs[3] = {cur, bufa, bufb};
    for (int i = 0; i < iters; i++) {
        a.flow_in = bufs[i % 3];
        a.flow_out = bufs[(i + 1) % 3];
        ProfScope ps(K_FLOW_GAUSS, 56.0 * n * h * w, st, n, h, w);
        int rc;
        if (reg) {
            rc = a.m == 2 ? launch_gauss_variant<2>(a, blocks, st) : launch_gauss_variant<4>(a, blocks, st);
            if (rc) return rc;
            FDN_LAUNCHED("k_flow_gauss_iter");
        } else {
            if ((rc = launch_gauss_variant<0>(a, blocks, st))) return rc;
            FDN_LAUNCHED("k_flow_gauss_iter_smem");
        }
    }
    *result = bufs[iters % 3];
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Initial flow of the coarsest level: resize(flow0, INTER_AREA) * scale  (SURVEY App. A.0-3)
// ------------------------------------------------------------------------------------------------
struct AreaAxis {
    int S, D, iscale, fast;
    double scale;
};

// fractional-coverage taps of destination index d (OpenCV computeResizeAreaTab): [first, last] source range with
// alpha weights; returns count and fills si/alpha (at most 3 + interior entries; interior alpha = 1/cellWidth)
__device__ __forceinline__ void area_entry_range(const AreaAxis& ax, int d, int& sx1, int& sx2, float& a_first,
                                                 float& a_mid, float& a_last, bool& has_first, bool& has_last)
{
    const double fsx1 = __dmul_rn((double)d, ax.scale);
    const double fsx2 = __dadd_rn(fsx1, ax.scale);
    const double cell = fmin(ax.scale, __dsub_rn((double)ax.S, fsx1));
    sx1 = (int)ceil(fsx1);
    sx2 = (int)floor(fsx2);
    sx2 = min(sx2, ax.S - 1);
    sx1 = min(sx1, sx2);
    has_first = __dsub_rn((double)sx1, fsx1) > 1e-3;
    a_first = (float)__ddiv_rn(__dsub_rn((double)sx1, fsx1), cell);
    a_mid = (float)__ddiv_rn(1.0, cell);
    has_last = __dsub_rn(fsx2, (double)sx2) > 1e-3;
    a_last = (float)__ddiv_rn(fmin(fmin(__dsub_rn(fsx2, (double)sx2), 1.), cell), cell);
}

__global__ void __launch_bounds__(128)
k_flow_area_down(const float2* __restrict__ in, int H, int W, float2* __restrict__ out, int h, int w, AreaAxis ax,
                 AreaAxis ay, float scale)
{
    const int dx = blockIdx.x * 128 + threadIdx.x;
    const int dy = blockIdx.y;
    const int b = blockIdx.z;
    if (dx >= w) return;
    const float2* src = in + (int64_t)b * H * W;
    float rx, ry;
    if (ax.fast && ay.fast && (ax.iscale & 3) == 0 && (W & 1) == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0) {
        // the same sum when a block row is a whole number of groups of four (every power-of-two pyramid): a group is two
        // 16-byte loads, the accumulation order is unchanged (s += ((v0 + v1) + v2) + v3, groups in row-major order)
        float sx_ = 0.f, sy_ = 0.f;
        for (int sy = 0; sy < ay.iscale; sy++) {
            const float4* row = reinterpret_cast<const float4*>(src + (int64_t)(dy * ay.iscale + sy) * W + dx * ax.iscale);
            for (int g = 0; g < ax.iscale / 4; g++) {
                const float4 q0 = __ldg(row + 2 * g), q1 = __ldg(row + 2 * g + 1);
                sx_ = __fadd_rn(sx_, __fadd_rn(__fadd_rn(__fadd_rn(q0.x, q0.z), q1.x), q1.z));
                sy_ = __fadd_rn(sy_, __fadd_rn(__fadd_rn(__fadd_rn(q0.y, q0.w), q1.y), q1.w));
            }
        }
        const float inv = __fdiv_rn(1.f, (float)(ax.iscale * ay.iscale));
        rx = __fmul_rn(sx_, inv);
        ry = __fmul_rn(sy_, inv);
    } else if (ax.fast && ay.fast) {
        // resizeAreaFast_: block sum in row-major order, unrolled by four, times 1/area (float32)
        const int area = ax.iscale * ay.iscale;
        float sx_ = 0.f, sy_ = 0.f;
        int k = 0;
        float vx[4], vy[4];
        for (int sy = 0; sy < ay.iscale; sy++) {
            const float2* row = src + (int64_t)(dy * ay.iscale + sy) * W + dx * ax.iscale;
            for (int sx = 0; sx < ax.iscale; sx++) {
                const float2 v = row[sx];
                if (k < (area & ~3)) {
                    vx[k & 3] = v.x; vy[k & 3] = v.y;
                    if ((k & 3) == 3) {
                        sx_ = __fadd_rn(sx_, __fadd_rn(__fadd_rn(__fadd_rn(vx[0], vx[1]), vx[2]), vx[3]));
                        sy_ = __fadd_rn(sy_, __fadd_rn(__fadd_rn(__fadd_rn(vy[0], vy[1]), vy[2]), vy[3]));
                    }
                } else {
                    sx_ = __fadd_rn(sx_, v.x);
                    sy_ = __fadd_rn(sy_, v.y);
                }
                k++;
            }
        }
        const float inv = __fdiv_rn(1.f, (float)area);
        rx = __fmul_rn(sx_, inv);
        ry = __fmul_rn(sy_, inv);
    } else {
        // resizeArea_: per source row, horizontal weighted sum in table order; rows combined with beta weights
        int x1, x2, y1, y2;
        float axf, axm, axl, ayf, aym, ayl;
        bool hxf, hxl, hyf, hyl;
        area_entry_range(ax, dx, x1, x2, axf, axm, axl, hxf, hxl);
        area_entry_range(ay, dy, y1, y2, ayf, aym, ayl, hyf, hyl);
        float sumx = 0.f, sumy = 0.f;
        bool firstrow = true;
        const int ya = hyf ? y1 - 1 : y1, yb = hyl ? y2 : y2 - 1;
        for (int sy = ya; sy <= yb; sy++) {
            const float beta = (sy == y1 - 1) ? ayf : ((sy == y2 && hyl) ? ayl : aym);
            const float2* row = src + (int64_t)sy * W;
            float bx = 0.f, by = 0.f;
            if (hxf) {
                const float2 v = row[x1 - 1];
                bx = __fadd_rn(bx, __fmul_rn(v.x, axf)); by = __fadd_rn(by, __fmul_rn(v.y, axf));
            }
            for (int sx = x1; sx < x2; sx++) {
                const float2 v = row[sx];
                bx = __fadd_rn(bx, __fmul_rn(v.x, axm)); by = __fadd_rn(by, __fmul_rn(v.y, axm));
            }
            if (hxl) {
                const float2 v = row[x2];
                bx = __fadd_rn(bx, __fmul_rn(v.x, axl)); by = __fadd_rn(by, __fmul_rn(v.y, axl));
            }
            if (firstrow) {
                sumx = __fmul_rn(beta, bx); sumy = __fmul_rn(beta, by);
                firstrow = false;
            } else {
                sumx = __fadd_rn(sumx, __fmul_rn(beta, bx)); sumy = __fadd_rn(sumy, __fmul_rn(beta, by));
            }
        }
        rx = sumx; ry = sumy;
    }
    float2 o;
    o.x = __fmul_rn(rx, scale);
    o.y = __fmul_rn(ry, scale);
    out[((int64_t)b * h + dy) * w + dx] = o;
}

static AreaAxis make_area_axis(int S, int D)
{
    AreaAxis a;
    a.S = S; a.D = D;
    a.scale = 1. / ((double)D / S);
    a.iscale = (int)lrint(a.scale);
    a.fast = fabs(a.scale - a.iscale) < 2.220446049250313e-16;
    return a;
}

int launch_flow_area_down(const float* flow, int n, int H, int W, float* out, int h, int w, float scale,
                          cudaStream_t st)
{
    AreaAxis ax = make_area_axis(W, w), ay = make_area_axis(H, h);
    FDN_CHECK_ARG(h <= H && w <= W, "area resize only shrinks");
    for (int b0 = 0; b0 < n; b0 += 65535) {
        const int nb = n - b0 < 65535 ? n - b0 : 65535;
        dim3 grid((unsigned)cdiv(w, 128), (unsigned)h, (unsigned)nb);
        ProfScope ps(K_FLOW_AREA, 8.0 * nb * ((double)H * W + (double)h * w), st);
        k_flow_area_down<<<grid, 128, 0, st>>>(reinterpret_cast<const float2*>(flow) + (int64_t)b0 * H * W, H, W,
                                               reinterpret_cast<float2*>(out) + (int64_t)b0 * h * w, h, w, ax, ay,
                                               scale);
        FDN_LAUNCHED("k_flow_area_down");
    }
    return FDN_OK;
}

// ------------------------------------------------------------------------------------------------
// Flow to the next finer level: resize(prevFlow, INTER_LINEAR) * 2  (OpenCV's own 2-channel code path:
// frac = float(coord) - floor, out = a*(1-f) + b*f, fractions zeroed at the borders horizontally only)
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
k_flow_upsample(const float2* __restrict__ in, int hin, int win, float2* __restrict__ out, int h, int w,
                double scale_x, double scale_y)
{
    const int dx = blockIdx.x * 128 + threadIdx.x;
    const int dy = blockIdx.y;
    const int b = blockIdx.z;
    if (dx >= w) return;
    float fx = (float)__dsub_rn(__dmul_rn((double)dx + 0.5, scale_x), 0.5);
    int sx = (int)floorf(fx);
    fx = __fsub_rn(fx, (float)sx);
    if (sx < 0) { fx = 0.f; sx = 0; }
    if (sx >= win - 1) { fx = 0.f; sx = win - 1; }
    float fy = (float)__dsub_rn(__dmul_rn((double)dy + 0.5, scale_y), 0.5);
    const int sy = (int)floorf(fy);
    fy = __fsub_rn(fy, (float)sy);
    const int sy0 = min(max(sy, 0), hin - 1), sy1 = min(max(sy + 1, 0), hin - 1);
    const int sx1 = min(sx + 1, win - 1);
    const float2* S0 = in + ((int64_t)b * hin + sy0) * win;
    const float2* S1 = in + ((int64_t)b * hin + sy1) * win;
    const float a1 = fx, a0 = __fsub_rn(1.f, fx), b1 = fy, b0 = __fsub_rn(1.f, fy);
    const float2 p00 = S0[sx], p01 = S0[sx1], p10 = S1[sx], p11 = S1[sx1];
    const float r0x = __fadd_rn(__fmul_rn(p00.x, a0), __fmul_rn(p01.x, a1));
    const float r0y = __fadd_rn(__fmul_rn(p00.y, a0), __fmul_rn(p01.y, a1));
    const float r1x = __fadd_rn(__fmul_rn(p10.x, a0), __fmul_rn(p11.x, a1));
    const float r1y = __fadd_rn(__fmul_rn(p10.y, a0), __fmul_rn(p11.y, a1));
    float2 o;
    o.x = __fmul_rn(__fadd_rn(__fmul_rn(r0x, b0), __fmul_rn(r1x, b1)), 2.f);
    o.y = __fmul_rn(__fadd_rn(__fmul_rn(r0y, b0), __fmul_rn(r1y, b1)), 2.f);
    out[((int64_t)b * h + dy) * w + dx] = o;
}

// Two consecutive outputs per thread (one 16-byte store); same arithmetic. Needs an even output width.
__device__ __forceinline__ float2 upsample_px(const float2* __restrict__ S0, const float2* __restrict__ S1, int win,
                                              int dx, double scale_x, float b0, float b1)
{
    float fx = (float)__dsub_rn(__dmul_rn((double)dx + 0.5, scale_x), 0.5);
    int sx = (int)floorf(fx);
    fx = __fsub_rn(fx, (float)sx);
    if (sx < 0) { fx = 0.f; sx = 0; }
    if (sx >= win - 1) { fx = 0.f; sx = win - 1; }
    const int sx1 = min(sx + 1, win - 1);
    const float a1 = fx, a0 = __fsub_rn(1.f, fx);
    const float2 p00 = __ldg(S0 + sx), p01 = __ldg(S0 + sx1), p10 = __ldg(S1 + sx), p11 = __ldg(S1 + sx1);
    const float r0x = __fadd_rn(__fmul_rn(p00.x, a0), __fmul_rn(p01.x, a1));
    const float r0y = __fadd_rn(__fmul_rn(p00.y, a0), __fmul_rn(p01.y, a1));
    const float r1x = __fadd_rn(__fmul_rn(p10.x, a0), __fmul_rn(p11.x, a1));
    const float r1y = __fadd_rn(__fmul_rn(p10.y, a0), __fmul_rn(p11.y, a1));
    float2 o;
    o.x = __fmul_rn(__fadd_rn(__fmul_rn(r0x, b0), __fmul_rn(r1x, b1)), 2.f);
    o.y = __fmul_rn(__fadd_rn(__fmul_rn(r0y, b0), __fmul_rn(r1y, b1)), 2.f);
    return o;
}

__global__ void __launch_bounds__(128)
k_flow_upsample2(const float2* __restrict__ in, int hin, int win, float4* __restrict__ out, int h, int w, double scale_x,
                 double scale_y)
{
    const int dx = (blockIdx.x * 128 + threadIdx.x) * 2;
    const int dy = blockIdx.y;
    const int b = blockIdx.z;
    if (dx >= w) return;
    float fy = (float)__dsub_rn(__dmul_rn((double)dy + 0.5, scale_y), 0.5);
    const int sy = (int)floorf(fy);
    fy = __fsub_rn(fy, (float)sy);
    const int sy0 = min(max(sy, 0), hin - 1), sy1 = min(max(sy + 1, 0), hin - 1);
    const float2* S0 = in + ((int64_t)b * hin + sy0) * win;
    const float2* S1 = in + ((int64_t)b * hin + sy1) * win;
    const float b1 = fy, b0 = __fsub_rn(1.f, fy);
    const float2 o0 = upsample_px(S0, S1, win, dx, scale_x, b0, b1);
    const float2 o1 = upsample_px(S0, S1, win, dx + 1, scale_x, b0, b1);
    out[(((int64_t)b * h + dy) * w + dx) / 2] = make_float4(o0.x, o0.y, o1.x, o1.y);
}

// Exact factor 2 in both directions (every level of an even-sized pyramid): the source coordinate of output 2k is
// k - 0.25 and of 2k+1 is k + 0.25, so floor / fraction are constants (fraction 0.75 and 0.25, exact in float32) and the
// float64 coordinate arithmetic of k_flow_upsample2 folds away; the interpolation itself is the same sequence of
// float32 operations. One thread = the 2 x 2 outputs (rows 2j, 2j+1, columns 2k, 2k+1) from the 3 x 3 source
// neighbourhood of (j, k).
__global__ void __launch_bounds__(128)
k_flow_upsample_x2(const float2* __restrict__ in, int hin, int win, float4* __restrict__ out, int h, int w)
{
    const int k = blockIdx.x * 128 + threadIdx.x;   // source column
    const int j = blockIdx.y;                       // source row: output rows 2j and 2j + 1
    const int b = blockIdx.z;
    if (k >= win) return;
    // rows: dy = 2j -> sy = j - 1, fy = 0.75; dy = 2j + 1 -> sy = j, fy = 0.25 (no clamping of the fraction vertically,
    // the row indices are clamped)
    const float2* Sm = in + ((int64_t)b * hin + max(j - 1, 0)) * win;
    const float2* Sc = in + ((int64_t)b * hin + j) * win;
    const float2* Sp = in + ((int64_t)b * hin + min(j + 1, hin - 1)) * win;
    const int km = max(k - 1, 0), kp = min(k + 1, win - 1);
    float2 v[3][3];
    v[0][0] = __ldg(Sm + km); v[0][1] = __ldg(Sm + k); v[0][2] = __ldg(Sm + kp);
    v[1][0] = __ldg(Sc + km); v[1][1] = __ldg(Sc + k); v[1][2] = __ldg(Sc + kp);
    v[2][0] = __ldg(Sp + km); v[2][1] = __ldg(Sp + k); v[2][2] = __ldg(Sp + kp);
    // columns: output 2k: sx = k - 1, fx = 0.75 (k = 0: sx = 0, fx = 0 -> taps S[0], S[min(1, win-1)]);
    //          output 2k+1: sx = k, fx = 0.25 (k = win-1: fx = 0 -> taps S[win-1], S[win-1])
    const float ea1 = k >= 1 ? 0.75f : 0.f, ea0 = __fsub_rn(1.f, ea1);
    const float oa1 = k >= win - 1 ? 0.f : 0.25f, oa0 = __fsub_rn(1.f, oa1);
    const int e0 = k >= 1 ? 0 : 1, e1 = k >= 1 ? 1 : 2;   // tap columns of the even output inside v[.][0..2]
    float2 he[3], ho[3];   // horizontally interpolated rows (even / odd output column)
#pragma unroll
    for (int r = 0; r < 3; r++) {
        const float2 p0 = e0 == 0 ? v[r][0] : v[r][1], p1 = e1 == 1 ? v[r][1] : v[r][2];
        he[r].x = __fadd_rn(__fmul_rn(p0.x, ea0), __fmul_rn(p1.x, ea1));
        he[r].y = __fadd_rn(__fmul_rn(p0.y, ea0), __fmul_rn(p1.y, ea1));
        ho[r].x = __fadd_rn(__fmul_rn(v[r][1].x, oa0), __fmul_rn(v[r][2].x, oa1));
        ho[r].y = __fadd_rn(__fmul_rn(v[r][1].y, oa0), __fmul_rn(v[r][2].y, oa1));
    }
#pragma unroll
    for (int half = 0; half < 2; half++) {
        const int dy = 2 * j + half;
        if (dy >= h) break;
        // dy even: rows (j-1, j) with b1 = 0.75; dy odd: rows (j, j+1) with b1 = 0.25
        const float b1 = half ? 0.25f : 0.75f, b0 = __fsub_rn(1.f, b1);
        const float2 re0 = he[half], re1 = he[half + 1], ro0 = ho[half], ro1 = ho[half + 1];
        float4 o;
        o.x = __fmul_rn(__fadd_rn(__fmul_rn(re0.x, b0), __fmul_rn(re1.x, b1)), 2.f);
        o.y = __fmul_rn(__fadd_rn(__fmul_rn(re0.y, b0), __fmul_rn(re1.y, b1)), 2.f);
        o.z = __fmul_rn(__fadd_rn(__fmul_rn(ro0.x, b0), __fmul_rn(ro1.x, b1)), 2.f);
        o.w = __fmul_rn(__fadd_rn(__fmul_rn(ro0.y, b0), __fmul_rn(ro1.y, b1)), 2.f);
        out[(((int64_t)b * h + dy) * w) / 2 + k] = o;
    }
}

int launch_flow_upsample(const float* flow, int n, int hin, int win, float* out, int h, int w, cudaStream_t st)
{
    const double scale_x = 1. / ((double)w / win), scale_y = 1. / ((double)h / hin);
    if (w == 2 * win && h == 2 * hin && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        for (int b0 = 0; b0 < n; b0 += 65535) {
            const int nb = n - b0 < 65535 ? n - b0 : 65535;
            dim3 grid((unsigned)cdiv(win, 128), (unsigned)hin, (unsigned)nb);
            ProfScope ps(K_FLOW_UP, 8.0 * nb * ((double)hin * win + (double)h * w), st);
            k_flow_upsample_x2<<<grid, 128, 0, st>>>(reinterpret_cast<const float2*>(flow) + (int64_t)b0 * hin * win, hin, win,
                                                     reinterpret_cast<float4*>(out + (int64_t)b0 * h * w * 2), h, w);
            FDN_LAUNCHED("k_flow_upsample_x2");
        }
        return FDN_OK;
    }
    if (w % 2 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        for (int b0 = 0; b0 < n; b0 += 65535) {
            const int nb = n - b0 < 65535 ? n - b0 : 65535;
            dim3 grid((unsigned)cdiv(w, 256), (unsigned)h, (unsigned)nb);
            ProfScope ps(K_FLOW_UP, 8.0 * nb * ((double)hin * win + (double)h * w), st);
            k_flow_upsample2<<<grid, 128, 0, st>>>(reinterpret_cast<const float2*>(flow) + (int64_t)b0 * hin * win, hin, win,
                                                   reinterpret_cast<float4*>(out + (int64_t)b0 * h * w * 2), h, w, scale_x,
                                                   scale_y);
            FDN_LAUNCHED("k_flow_upsample2");
        }
        return FDN_OK;
    }
    for (int b0 = 0; b0 < n; b0 += 65535) {
        const int nb = n - b0 < 65535 ? n - b0 : 65535;
        dim3 grid((unsigned)cdiv(w, 128), (unsigned)h, (unsigned)nb);
        ProfScope ps(K_FLOW_UP, 8.0 * nb * ((double)hin * win + (double)h * w), st);
        k_flow_upsample<<<grid, 128, 0, st>>>(reinterpret_cast<const float2*>(flow) + (int64_t)b0 * hin * win, hin,
                                              win, reinterpret_cast<float2*>(out) + (int64_t)b0 * h * w, h, w,
                                              scale_x, scale_y);
        FDN_LAUNCHED("k_flow_upsample");
    }
    return FDN_OK;
}

}  // namespace fdn
