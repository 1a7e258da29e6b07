// No-OF path (the reference's --disable_OF switch, BASELINE.json configs[2]): plain separable Gaussian, one pass per axis,
//   out[s] = fold_i f32(f64(acc) + f64(in[(s + i - r) wrap]) * k[i])          (src/flowdenoising.py:133-158)
// Two arithmetic modes:
//   exact (default): NumPy's arithmetic for `tmp_slice(f32) += slice(f32) * kernel[i](f64)` -- float64 product, float64
//                    sum, rounded to float32 after EVERY tap (SURVEY.md App. B, Q9). Bit-identical to the reference.
//   fast:            float32 FMA chain (<= 4 ulp from the exact mode), HBM-bound.
// HBM-bound by design: 4 B read + 4 B written per voxel and pass. sm_100a.
//
// k_gauss_axis_ring  filter along a strided axis (Z and Y passes; x is contiguous). A thread owns VEC consecutive x of
//                    one row and marches along the slice axis with the last KLEN inputs in registers (static rotation:
//                    the loop is unrolled KLEN times). New inputs arrive through a PER-THREAD ring of cp.async copies
//                    (global -> shared, 16 or 8 bytes per thread and slot, GA_DEPTH slices ahead): no thread ever waits
//                    for a load it has just issued, nobody reads anybody else's slot, so there is no block-level
//                    synchronisation at all.
// k_gauss_rows_direct filter along contiguous rows (X pass, fast mode): four consecutive outputs per thread from a register
//                    window of aligned 128-bit loads (neighbouring threads overlap in L1), periodic wrap per 16-byte group.
// k_gauss_rows_tile  the same pass in exact mode: a block stages its inputs in shared memory so that every value is
//                    loaded and range-checked once, then four outputs per thread from a float64 register window.
//
// The exact mode is an instruction-throughput problem, not a bandwidth problem: per tap it needs a float64 multiply, a
// float64 add and a rounding of the sum to float32 precision. Written naively (float<->double conversions) that is
// three XU-pipe operations per tap at 16 lanes / clock / SM, and the pass ran at 9 % of the HBM roofline (round 1). Here
//   * every input is converted to float64 ONCE, when it enters the register window (1/KLEN conversions per tap);
//   * the accumulator stays in float64 registers; "round to float32" is Veltkamp's splitting with the constant
//     2^29 + 1 (three float64 operations on the FP64 pipe) for three taps out of four and the conversion pair
//     (double -> float -> double, XU pipe) for the fourth. Measured on B200 (512x1024x1024, 17 taps, ms per pass along
//     Z / X): conversions only 4.6 / 5.0, integer rounding of the bit pattern only 4.6 / 3.8, Veltkamp only 3.26 / 2.93,
//     this 3:1 mix 2.99 / 2.63. The FP64 pipe (64 lanes / clock / SM) is the bound: 2 + 3 operations per tap, 17
//     taps -> >= 2.3 ms per pass on 148 SMs at 1.85 GHz, i.e. the exact mode cannot exceed ~0.28 of the HBM roofline;
//   * Veltkamp's form is exact whenever the sum is zero or a normal float32 number. A thread (a block, for the row
//     kernel) uses it only while every input it has seen is 0 or has a magnitude in [2^-30, 2^90) and the taps are in
//     [2^-30, 2] (checked on the host): then every partial sum is 0 or at least 2^-112 in magnitude (a cancellation
//     between an accumulator and a product of similar size leaves a multiple of the product's ulp, >= 2^-60-52) and
//     below 2^127. Anything else -- subnormals, huge values, Inf / NaN -- takes the conversion path.
#include <type_traits>

#include "fdn_internal.cuh"

namespace fdn {

struct Taps64 {   // FDN_MAX_KLEN: include/fdn_b200.h
    int klen;
    double k[FDN_MAX_KLEN];
};
struct Taps32 {
    int klen;
    float k[FDN_MAX_KLEN];
};
template <int KLEN>
struct TapsW {
    double k64[KLEN];
    float k32[KLEN];
};

// ------------------------------------------------------------------------------------------------
// exact-mode arithmetic
// ------------------------------------------------------------------------------------------------
// s rounded to float32 precision (round to nearest even), as a double
__device__ __forceinline__ double round_f32_grid_cvt(double s) { return (double)__double2float_rn(s); }
// Veltkamp splitting: the high part of s with 53 - 29 = 24 significant bits. With round-to-nearest-even float64
// arithmetic it IS s rounded to nearest even on 24 bits (checked against the conversion on 5 M values, 2.3 M of them
// exact ties, carries into the exponent included, tests/test_oracle_golden.py); s must be 0 or a normal float32 magnitude.
__device__ __forceinline__ double round_f32_grid_f64(double s)
{
    const double p = __dmul_rn(s, 536870913.0);
    return __dadd_rn(__dsub_rn(s, p), p);
}
// the form tap i uses while the fast form is allowed (i is a compile-time constant: the tap loops are fully unrolled)
__device__ __forceinline__ double round_f32_grid(double s, int i)
{
    return (i % 4) == 0 ? round_f32_grid_cvt(s) : round_f32_grid_f64(s);
}

// 1 unless v is 0 or has a magnitude in [2^-30, 2^90) (accumulated with |: no short-circuit chains)
__device__ __forceinline__ unsigned not_benign_f32(float v)
{
    const unsigned u = __float_as_uint(v) & 0x7fffffffu;
    return (unsigned)(u != 0u) & (unsigned)((u - 0x30800000u) >= 0x3C000000u);   // [2^-30, 2^90) <-> [0x30800000, 0x6C800000)
}

static bool taps_benign(const double* k, int n)
{
    for (int i = 0; i < n; i++) {
        const double a = k[i] < 0 ? -k[i] : k[i];
        if (!(a >= 9.313225746154785e-10 && a <= 2.0)) return false;   // 2^-30
    }
    return true;
}

// ------------------------------------------------------------------------------------------------
// generic fallbacks (any odd kernel length): one thread per output, neighbours re-read through L1 / L2. They also run
// the typed volumes (T = uint8 / int8 / uint16 / int16, exact mode only): every input is converted to float32 as
// NumPy does for `int_slice * kernel[i]`, the float32 sum is truncated toward zero into T once, at the store.
// ------------------------------------------------------------------------------------------------
// BORDERED: the view's indices take the border v.periodic (FDN_BORDER_REFLECT, _MIRROR or _NEAREST) instead of the wrap
// (the wrap instantiations are the kernels of the periodic pass, unchanged)
template <typename T, bool EXACT, bool BORDERED>
__global__ void __launch_bounds__(256)
k_gauss_axis(const T* __restrict__ in, T* __restrict__ out, fdn_view v, Taps64 t64, Taps32 t32, int64_t in_bs,
             int64_t out_bs)
{
    const int x = blockIdx.x * 256 + threadIdx.x;
    const int y = blockIdx.y;
    const int g = blockIdx.z / v.n_out;   // volume of a batch (blockIdx.z = volume * n_out + slice)
    const int s = blockIdx.z - g * v.n_out;
    if (x >= v.W) return;
    in += g * in_bs;
    out += g * out_bs;
    const int klen = EXACT ? t64.klen : t32.klen;
    const int r = klen >> 1;
    const int64_t off = (int64_t)y * v.in_row_stride + x;
    float acc = 0.f;
    for (int i = 0; i < klen; i++) {
        int j = s + v.halo + i - r;
        if (BORDERED) {
            j = border_index(j, v.n_in, v.periodic);
        } else if (v.periodic) {
            j %= v.n_in;
            if (j < 0) j += v.n_in;
        }
        const float val = (float)in[(int64_t)j * v.in_slice_stride + off];
        if (EXACT) acc = (float)__dadd_rn((double)acc, __dmul_rn((double)val, t64.k[i]));
        else acc = fmaf(val, t32.k[i], acc);
    }
    out[(int64_t)s * v.out_slice_stride + (int64_t)y * v.out_row_stride + x] = store_cast<T>(acc);
}

#define GR_TILE 512
// BORDERED: both row ends take `border` (FDN_BORDER_REFLECT, _MIRROR or _NEAREST) instead of the wrap
template <typename T, bool EXACT, bool BORDERED>
__global__ void __launch_bounds__(256)
k_gauss_rows(const T* __restrict__ in, T* __restrict__ out, int W, Taps64 t64, Taps32 t32, int border)
{
    extern __shared__ float s_seg[];  // GR_TILE + klen - 1
    const int klen = EXACT ? t64.klen : t32.klen;
    const int r = klen >> 1;
    const int64_t row = blockIdx.y;
    const int x0 = blockIdx.x * GR_TILE;
    const T* src = in + row * W;
    const int nload = min(GR_TILE, W - x0) + 2 * r;
    for (int i = threadIdx.x; i < nload; i += 256) {
        int j;
        if (BORDERED) {
            j = border_index(x0 - r + i, W, border);
        } else {
            j = (x0 - r + i) % W;
            if (j < 0) j += W;
        }
        s_seg[i] = (float)src[j];
    }
    __syncthreads();
    for (int i = threadIdx.x; i < GR_TILE && x0 + i < W; i += 256) {
        float acc = 0.f;
        for (int t = 0; t < klen; t++) {
            const float val = s_seg[i + t];
            if (EXACT) acc = (float)__dadd_rn((double)acc, __dmul_rn((double)val, t64.k[t]));
            else acc = fmaf(val, t32.k[t], acc);
        }
        out[row * W + x0 + i] = store_cast<T>(acc);
    }
}

// ------------------------------------------------------------------------------------------------
// k_gauss_axis_ring
// ------------------------------------------------------------------------------------------------
#define GA_SEG 128      // output slices per thread (the window is filled with KLEN - 1 extra loads per segment)
#define GA_DEPTH 8      // cp.async slots per thread (slices in flight)

template <int BYTES>
__device__ __forceinline__ void cp_async_thread(void* smem_dst, const void* gsrc)
{
    const uint32_t d = smem_u32(smem_dst);
    if (BYTES == 16) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(d), "l"(gsrc) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" :: "r"(d), "l"(gsrc), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

template <int KLEN, bool EXACT, int VEC, bool BORDERED>
__global__ void __launch_bounds__(128)
k_gauss_axis_ring(const float* __restrict__ in, float* __restrict__ out, fdn_view v, TapsW<KLEN> taps, int int_rounding,
                  int nseg, int64_t in_bs, int64_t out_bs)
{
    constexpr int R = KLEN / 2;
    typedef typename std::conditional<EXACT, double, float>::type W_t;   // window element
    struct __align__(4 * VEC) Slot { float e[VEC]; };
    __shared__ Slot ring[GA_DEPTH][128];
    const int t = threadIdx.x;
    const int x = (blockIdx.x * 128 + t) * VEC;
    const int y = blockIdx.y;
    const int g = blockIdx.z / nseg;   // volume of a batch (blockIdx.z = volume * nseg + segment)
    const int s0 = (blockIdx.z - g * nseg) * GA_SEG;
    if (x >= v.W) return;       // (no block-level synchronisation below)
    in += g * in_bs;
    out += g * out_bs;
    const int s_end = min(s0 + GA_SEG, v.n_out);
    const int n_in_seg = s_end - s0 + 2 * R;          // input slices this thread consumes: s0 - R .. s_end - 1 + R
    const float* src = in + (int64_t)y * v.in_row_stride + x;
    float* dst = out + (int64_t)y * v.out_row_stride + x;

    // q-th input of the segment (q = 0 .. n_in_seg - 1) <-> view slice s0 - R + q (+ halo, periodic wrap). The copies
    // are issued in order of q: the next slice index and its address advance incrementally (no division per copy).
    // BORDERED (v.periodic: FDN_BORDER_REFLECT, _MIRROR or _NEAREST): each copy maps its index, which costs a compare
    // inside the axis and a division only for the r slices beyond either end.
    int jn = s0 - R + v.halo;
    if (!BORDERED && v.periodic) {
        jn %= v.n_in;
        if (jn < 0) jn += v.n_in;
    }
    const int u0 = jn;
    const float* pn = src + (int64_t)jn * v.in_slice_stride;
    int qn = 0;
    auto issue = [&]() {
        if (qn < n_in_seg) {
            if (BORDERED) pn = src + (int64_t)border_index(u0 + qn, v.n_in, v.periodic) * v.in_slice_stride;
            cp_async_thread<4 * VEC>(&ring[qn % GA_DEPTH][t], pn);
            if (!BORDERED) {
                pn += v.in_slice_stride;
                if (++jn == v.n_in && v.periodic) { jn = 0; pn = src; }
            }
        }
        ++qn;
        cp_async_commit();      // one group per q, empty past the end: wait_group counts stay uniform
    };
    unsigned bad = int_rounding ? 0u : 1u;   // sticky: once set the thread rounds with conversions only
    struct Vec { W_t e[VEC]; };
    auto take = [&](int q) -> Vec {  // the oldest copy in flight has landed: read it, refill its slot
        cp_async_wait<GA_DEPTH - 1>();
        const Slot sl = ring[q % GA_DEPTH][t];
        issue();
        Vec r;
#pragma unroll
        for (int c = 0; c < VEC; c++) {
            if (EXACT) bad |= not_benign_f32(sl.e[c]);
            r.e[c] = (W_t)sl.e[c];
        }
        return r;
    };
#pragma unroll
    for (int q = 0; q < GA_DEPTH; q++) issue();

    Vec win[KLEN];
#pragma unroll
    for (int i = 0; i < KLEN - 1; i++) win[i] = take(i);
    int q = KLEN - 1;
    for (int s = s0; s < s_end; s += KLEN) {
        // Outputs are produced in PAIRS (s + u, s + u + 1): 2 * VEC independent accumulation chains per thread, advanced
        // tap by tap, hide the latency of a chain's add -> round -> add dependency. Window slot n % KLEN holds input
        // s0 - R + n; output u reads slots (u + i) % KLEN and receives its newest input in slot (u - 1) % KLEN; the
        // newest input of output u + 1 replaces slot u % KLEN, whose old value output u still needs for tap 0 (`old`).
#pragma unroll
        for (int u = 0; u < KLEN; u += 2) {
            if (s + u < s_end) {
                constexpr bool kNever = false;
                const bool pair = (u + 1 < KLEN) || kNever;      // compile-time per unrolled u
                win[(u + KLEN - 1) % KLEN] = take(q++);
                Vec old = win[u % KLEN];
                if (pair) win[u % KLEN] = take(q++);             // (past the segment's end: stale data, result unused)
                W_t a[2][VEC];
#pragma unroll
                for (int c = 0; c < VEC; c++) { a[0][c] = (W_t)0; a[1][c] = (W_t)0; }
                auto run = [&](auto rnd) {
#pragma unroll
                    for (int i = 0; i < KLEN; i++) {
#pragma unroll
                        for (int c = 0; c < VEC; c++) {
                            const W_t v0 = (i == 0) ? old.e[c] : win[(u + i) % KLEN].e[c];
                            a[0][c] = rnd(a[0][c], v0, i);
                            if (pair) a[1][c] = rnd(a[1][c], win[(u + 1 + i) % KLEN].e[c], i);
                        }
                    }
                };
                if (!EXACT) {
                    run([&](W_t acc, W_t val, int i) { return (W_t)fmaf((float)val, taps.k32[i], (float)acc); });
                } else if (!bad) {
                    run([&](W_t acc, W_t val, int i) {
                        return (W_t)round_f32_grid(__dadd_rn((double)acc, __dmul_rn((double)val, taps.k64[i])), i);
                    });
                } else {
                    run([&](W_t acc, W_t val, int i) {
                        return (W_t)round_f32_grid_cvt(__dadd_rn((double)acc, __dmul_rn((double)val, taps.k64[i])));
                    });
                }
#pragma unroll
                for (int o = 0; o < 2; o++) {
                    if (o == 1 && (!pair || s + u + 1 >= s_end)) break;
                    float* d = dst + (int64_t)(s + u + o) * v.out_slice_stride;
                    if (VEC == 4)
                        *reinterpret_cast<float4*>(d) = make_float4((float)a[o][0], (float)a[o][1 % VEC], (float)a[o][2 % VEC],
                                                                    (float)a[o][3 % VEC]);
                    else if (VEC == 2) *reinterpret_cast<float2*>(d) = make_float2((float)a[o][0], (float)a[o][1 % VEC]);
                    else d[0] = (float)a[o][0];
                }
            }
        }
    }
    cp_async_wait<0>();
}

template <int KLEN, bool BD>
static int launch_gauss_axis_ring(const float* in, float* out, const fdn_view& v, const double* k, int exact,
                                  cudaStream_t st, int batch, int64_t in_bs, int64_t out_bs)
{
    TapsW<KLEN> taps;
    for (int i = 0; i < KLEN; i++) { taps.k64[i] = k[i]; taps.k32[i] = (float)k[i]; }
    // widest vector every address of the view is aligned for; the exact mode keeps its window in float64 (2 columns)
    auto aligned = [&](int n) {
        return v.W % n == 0 && v.in_row_stride % n == 0 && v.in_slice_stride % n == 0 && v.out_row_stride % n == 0 &&
               v.out_slice_stride % n == 0 && (reinterpret_cast<uintptr_t>(in) % (4 * n)) == 0 &&
               (reinterpret_cast<uintptr_t>(out) % (4 * n)) == 0;
    };
    int vec = 1;
    if (aligned(2)) vec = 2;
    if (!exact && KLEN <= 17 && aligned(4)) vec = 4;
    const int ir = taps_benign(k, KLEN) ? 1 : 0;
    while (batch > 1 && vec > 1 && (in_bs % vec != 0 || out_bs % vec != 0)) vec /= 2;   // every volume stays aligned
    const int nseg = (int)cdiv(v.n_out, GA_SEG);
    const int per_launch = 65535 / nseg;   // volumes per launch: batch x segments in blockIdx.z
    for (int g0 = 0; g0 < batch; g0 += per_launch) {
        const int nb = batch - g0 < per_launch ? batch - g0 : per_launch;
        const float* i_ = in + g0 * in_bs;
        float* o_ = out + g0 * out_bs;
        dim3 grid((unsigned)cdiv(v.W, 128 * vec), (unsigned)v.H, (unsigned)(nb * nseg));
        ProfScope ps(K_GAUSS_AXIS, 8.0 * nb * v.n_out * v.H * v.W, st);
        if (exact) {
            if (vec == 2) k_gauss_axis_ring<KLEN, true, 2, BD><<<grid, 128, 0, st>>>(i_, o_, v, taps, ir, nseg, in_bs, out_bs);
            else k_gauss_axis_ring<KLEN, true, 1, BD><<<grid, 128, 0, st>>>(i_, o_, v, taps, ir, nseg, in_bs, out_bs);
        } else {
            if (vec == 4) k_gauss_axis_ring<KLEN, false, 4, BD><<<grid, 128, 0, st>>>(i_, o_, v, taps, ir, nseg, in_bs, out_bs);
            else if (vec == 2) k_gauss_axis_ring<KLEN, false, 2, BD><<<grid, 128, 0, st>>>(i_, o_, v, taps, ir, nseg, in_bs, out_bs);
            else k_gauss_axis_ring<KLEN, false, 1, BD><<<grid, 128, 0, st>>>(i_, o_, v, taps, ir, nseg, in_bs, out_bs);
        }
        FDN_LAUNCHED("k_gauss_axis_ring");
    }
    return FDN_OK;
}

template <bool BD>
static int launch_gauss_axis_border(const float* in, float* out, const fdn_view& v, const double* k, int klen,
                                    int exact, cudaStream_t st, int batch, int64_t in_bs, int64_t out_bs)
{
    switch (klen) {  // sigma = 0.5, 1, 1.5, 2, 2.5, 3, 4 (radius int(4 sigma + 0.5))
        case 5: return launch_gauss_axis_ring<5, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 9: return launch_gauss_axis_ring<9, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 13: return launch_gauss_axis_ring<13, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 17: return launch_gauss_axis_ring<17, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 21: return launch_gauss_axis_ring<21, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 25: return launch_gauss_axis_ring<25, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        case 33: return launch_gauss_axis_ring<33, BD>(in, out, v, k, exact, st, batch, in_bs, out_bs);
        default: break;
    }
    Taps64 t64;
    Taps32 t32;
    t64.klen = t32.klen = klen;
    for (int i = 0; i < klen; i++) { t64.k[i] = k[i]; t32.k[i] = (float)k[i]; }
    const int per_launch = 65535 / v.n_out;   // volumes per launch: batch x slices in blockIdx.z
    for (int g0 = 0; g0 < batch; g0 += per_launch) {
        const int nb = batch - g0 < per_launch ? batch - g0 : per_launch;
        dim3 grid((unsigned)cdiv(v.W, 256), (unsigned)v.H, (unsigned)(nb * v.n_out));
        ProfScope ps(K_GAUSS_AXIS, 8.0 * nb * v.n_out * v.H * v.W, st);
        if (exact) k_gauss_axis<float, true, BD><<<grid, 256, 0, st>>>(in + g0 * in_bs, out + g0 * out_bs, v, t64, t32, in_bs, out_bs);
        else k_gauss_axis<float, false, BD><<<grid, 256, 0, st>>>(in + g0 * in_bs, out + g0 * out_bs, v, t64, t32, in_bs, out_bs);
        FDN_LAUNCHED("k_gauss_axis");
    }
    return FDN_OK;
}

int launch_gauss_axis(const float* in, float* out, const fdn_view& v, const double* k, int klen, int exact,
                      cudaStream_t st, int batch, int64_t in_bs, int64_t out_bs)
{
    FDN_CHECK_ARG(klen >= 1 && klen <= FDN_MAX_KLEN && (klen & 1), "kernel length %d unsupported (odd, <= %d)", klen,
                  FDN_MAX_KLEN);
    FDN_CHECK_ARG(v.H <= 65535 && v.n_out <= 65535, "view too large for one launch");
    if (v.periodic && view_border(v.periodic) != FDN_BORDER_WRAP)
        return launch_gauss_axis_border<true>(in, out, v, k, klen, exact, st, batch, in_bs, out_bs);
    return launch_gauss_axis_border<false>(in, out, v, k, klen, exact, st, batch, in_bs, out_bs);
}

// ------------------------------------------------------------------------------------------------
// k_gauss_rows_direct
// ------------------------------------------------------------------------------------------------
// Four consecutive outputs x0 .. x0 + 3 of a row need inputs x0 - R .. x0 + 3 + R: the NV aligned 16-byte groups
// starting at x0 - PAD (PAD = R rounded up to a multiple of 4), each wrapped periodically as a whole (W % 4 == 0).
// All NV loads of a thread are independent and issued back to back; the groups a thread shares with its neighbours
// come from L1. BORDERED (`border`: FDN_BORDER_REFLECT, _MIRROR or _NEAREST): a group lies wholly inside or wholly
// outside the row (W % 4 == 0); one outside is reversed or repeated by the border, so it maps element by element.
template <int KLEN, bool BORDERED>
__global__ void __launch_bounds__(128)
k_gauss_rows_direct(const float* __restrict__ in, float* __restrict__ out, int W, int64_t rows, TapsW<KLEN> taps,
                    int border)
{
    constexpr int R = KLEN / 2;
    constexpr int PAD = (R + 3) / 4 * 4;
    constexpr int NV = (2 * PAD + 4) / 4;
    const int x0 = (blockIdx.x * 128 + threadIdx.x) * 4;
    const int64_t row = blockIdx.y + (int64_t)blockIdx.z * 65535;
    if (x0 >= W || row >= rows) return;
    const float* src = in + row * W;
    float win[4 * NV];
#pragma unroll
    for (int g = 0; g < NV; g++) {
        int j = x0 - PAD + 4 * g;
        if (BORDERED && (unsigned)j >= (unsigned)W) {
#pragma unroll
            for (int e = 0; e < 4; e++) win[4 * g + e] = __ldg(src + border_index(j + e, W, border));
            continue;
        }
        j %= W;
        if (j < 0) j += W;
        const float4 qv = __ldg(reinterpret_cast<const float4*>(src + j));
        win[4 * g] = qv.x; win[4 * g + 1] = qv.y; win[4 * g + 2] = qv.z; win[4 * g + 3] = qv.w;
    }
    float o[4];
#pragma unroll
    for (int e = 0; e < 4; e++) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < KLEN; i++) acc = fmaf(win[e + (PAD - R) + i], taps.k32[i], acc);
        o[e] = acc;
    }
    *reinterpret_cast<float4*>(out + row * W + x0) = make_float4(o[0], o[1], o[2], o[3]);
}

// Exact mode along rows: a block stages 512 outputs' inputs (+ wrapped halo) of one row in shared memory, every value
// loaded and range-checked ONCE (the check decides, for the whole block, whether the fast rounding forms are allowed),
// then each thread computes four consecutive outputs from a float64 register window.
template <int KLEN, bool BORDERED>
__global__ void __launch_bounds__(128)
k_gauss_rows_tile(const float* __restrict__ in, float* __restrict__ out, int W, int64_t rows, TapsW<KLEN> taps,
                  int int_rounding, int border)
{
    constexpr int R = KLEN / 2;
    constexpr int PAD = (R + 3) / 4 * 4;
    constexpr int NG = 128 + 2 * PAD / 4;       // 16-byte groups of the tile: [x0 - PAD, x0 + 512 + PAD)
    constexpr int NV = (2 * PAD + 4) / 4;
    __shared__ __align__(16) float tile[4 * NG];
    const int t = threadIdx.x;
    const int xb = blockIdx.x * 512;
    const int64_t row = blockIdx.y + (int64_t)blockIdx.z * 65535;
    if (row >= rows) return;                    // (uniform per block)
    const float* src = in + row * W;
    unsigned bad = int_rounding ? 0u : 1u;
    for (int g = t; g < NG; g += 128) {
        int j = xb - PAD + 4 * g;               // beyond the row's end (last, partial tile): wrapped, harmless
        float4 qv;
        if (BORDERED && (unsigned)j >= (unsigned)W) {     // (outside the row as a whole group, as in the direct kernel)
            qv = make_float4(__ldg(src + border_index(j, W, border)), __ldg(src + border_index(j + 1, W, border)),
                             __ldg(src + border_index(j + 2, W, border)), __ldg(src + border_index(j + 3, W, border)));
        } else {
            j %= W;
            if (j < 0) j += W;
            qv = __ldg(reinterpret_cast<const float4*>(src + j));
        }
        bad |= not_benign_f32(qv.x) | not_benign_f32(qv.y) | not_benign_f32(qv.z) | not_benign_f32(qv.w);
        *reinterpret_cast<float4*>(tile + 4 * g) = qv;
    }
    const int any_bad = __syncthreads_or((int)bad);
    const int x0 = xb + 4 * t;
    if (x0 >= W) return;
    double wd[4 * NV];
#pragma unroll
    for (int g = 0; g < NV; g++) {
        const float4 qv = *reinterpret_cast<const float4*>(tile + 4 * (t + g));
        wd[4 * g] = (double)qv.x; wd[4 * g + 1] = (double)qv.y; wd[4 * g + 2] = (double)qv.z; wd[4 * g + 3] = (double)qv.w;
    }
    // the four outputs' chains advance together, tap by tap (independent dependency chains for the scheduler)
    double acc[4] = {0., 0., 0., 0.};
    if (!any_bad) {
#pragma unroll
        for (int i = 0; i < KLEN; i++)
#pragma unroll
            for (int e = 0; e < 4; e++)
                acc[e] = round_f32_grid(__dadd_rn(acc[e], __dmul_rn(wd[e + (PAD - R) + i], taps.k64[i])), i);
    } else {
#pragma unroll
        for (int i = 0; i < KLEN; i++)
#pragma unroll
            for (int e = 0; e < 4; e++)
                acc[e] = round_f32_grid_cvt(__dadd_rn(acc[e], __dmul_rn(wd[e + (PAD - R) + i], taps.k64[i])));
    }
    *reinterpret_cast<float4*>(out + row * W + x0) =
        make_float4((float)acc[0], (float)acc[1], (float)acc[2], (float)acc[3]);
}

template <int KLEN, bool BD>
static int launch_gauss_rows_direct(const float* in, float* out, int64_t rows, int W, const double* k, int exact,
                                    int border, cudaStream_t st)
{
    TapsW<KLEN> taps;
    for (int i = 0; i < KLEN; i++) { taps.k64[i] = k[i]; taps.k32[i] = (float)k[i]; }
    const int ir = taps_benign(k, KLEN) ? 1 : 0;
    const int64_t ny = rows < 65535 ? rows : 65535;
    dim3 grid((unsigned)cdiv(W, 512), (unsigned)ny, (unsigned)cdiv(rows, 65535));
    ProfScope ps(K_GAUSS_ROWS, 8.0 * rows * W, st);
    if (exact) {
        k_gauss_rows_tile<KLEN, BD><<<grid, 128, 0, st>>>(in, out, W, rows, taps, ir, border);
        FDN_LAUNCHED("k_gauss_rows_tile");
    } else {
        k_gauss_rows_direct<KLEN, BD><<<grid, 128, 0, st>>>(in, out, W, rows, taps, border);
        FDN_LAUNCHED("k_gauss_rows_direct");
    }
    return FDN_OK;
}

template <bool BD>
static int launch_gauss_rows_border(const float* in, float* out, int64_t rows, int W, const double* k, int klen,
                                    int exact, int border, cudaStream_t st)
{
    if (W % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0) {
        switch (klen) {
            case 5: return launch_gauss_rows_direct<5, BD>(in, out, rows, W, k, exact, border, st);
            case 9: return launch_gauss_rows_direct<9, BD>(in, out, rows, W, k, exact, border, st);
            case 13: return launch_gauss_rows_direct<13, BD>(in, out, rows, W, k, exact, border, st);
            case 17: return launch_gauss_rows_direct<17, BD>(in, out, rows, W, k, exact, border, st);
            case 21: return launch_gauss_rows_direct<21, BD>(in, out, rows, W, k, exact, border, st);
            case 25: return launch_gauss_rows_direct<25, BD>(in, out, rows, W, k, exact, border, st);
            case 33: return launch_gauss_rows_direct<33, BD>(in, out, rows, W, k, exact, border, st);
            default: break;
        }
    }
    Taps64 t64;
    Taps32 t32;
    t64.klen = t32.klen = klen;
    for (int i = 0; i < klen; i++) { t64.k[i] = k[i]; t32.k[i] = (float)k[i]; }
    const size_t smem = sizeof(float) * (GR_TILE + klen - 1);
    for (int64_t r0 = 0; r0 < rows; r0 += 65535) {
        const int64_t nr = rows - r0 < 65535 ? rows - r0 : 65535;
        dim3 grid((unsigned)cdiv(W, GR_TILE), (unsigned)nr);
        ProfScope ps(K_GAUSS_ROWS, 8.0 * nr * W, st);
        if (exact) k_gauss_rows<float, true, BD><<<grid, 256, smem, st>>>(in + r0 * W, out + r0 * W, W, t64, t32, border);
        else k_gauss_rows<float, false, BD><<<grid, 256, smem, st>>>(in + r0 * W, out + r0 * W, W, t64, t32, border);
        FDN_LAUNCHED("k_gauss_rows");
    }
    return FDN_OK;
}

int launch_gauss_rows(const float* in, float* out, int64_t rows, int W, const double* k, int klen, int exact,
                      cudaStream_t st, int border)
{
    FDN_CHECK_ARG(klen >= 1 && klen <= FDN_MAX_KLEN && (klen & 1), "kernel length %d unsupported (odd, <= %d)", klen,
                  FDN_MAX_KLEN);
    if (border != FDN_BORDER_WRAP) return launch_gauss_rows_border<true>(in, out, rows, W, k, klen, exact, border, st);
    return launch_gauss_rows_border<false>(in, out, rows, W, k, klen, exact, border, st);
}

// ------------------------------------------------------------------------------------------------
// typed volumes: the generic kernels in exact mode (the fast FMA mode would move the truncation boundaries)
// ------------------------------------------------------------------------------------------------
template <typename T>
int launch_gauss_axis_typed(const T* in, T* out, const fdn_view& v, const double* k, int klen, cudaStream_t st)
{
    FDN_CHECK_ARG(klen >= 1 && klen <= FDN_MAX_KLEN && (klen & 1), "kernel length %d unsupported (odd, <= %d)", klen,
                  FDN_MAX_KLEN);
    FDN_CHECK_ARG(v.H <= 65535 && v.n_out <= 65535, "view too large for one launch");
    Taps64 t64;
    Taps32 t32;
    t64.klen = t32.klen = klen;
    for (int i = 0; i < klen; i++) { t64.k[i] = k[i]; t32.k[i] = (float)k[i]; }
    dim3 grid((unsigned)cdiv(v.W, 256), (unsigned)v.H, (unsigned)v.n_out);
    ProfScope ps(K_GAUSS_AXIS, 2.0 * sizeof(T) * v.n_out * v.H * v.W, st);
    if (v.periodic && view_border(v.periodic) != FDN_BORDER_WRAP)
        k_gauss_axis<T, true, true><<<grid, 256, 0, st>>>(in, out, v, t64, t32, 0, 0);
    else
        k_gauss_axis<T, true, false><<<grid, 256, 0, st>>>(in, out, v, t64, t32, 0, 0);
    FDN_LAUNCHED("k_gauss_axis");
    return FDN_OK;
}

template <typename T>
int launch_gauss_rows_typed(const T* in, T* out, int64_t rows, int W, const double* k, int klen, cudaStream_t st,
                            int border)
{
    FDN_CHECK_ARG(klen >= 1 && klen <= FDN_MAX_KLEN && (klen & 1), "kernel length %d unsupported (odd, <= %d)", klen,
                  FDN_MAX_KLEN);
    Taps64 t64;
    Taps32 t32;
    t64.klen = t32.klen = klen;
    for (int i = 0; i < klen; i++) { t64.k[i] = k[i]; t32.k[i] = (float)k[i]; }
    const size_t smem = sizeof(float) * (GR_TILE + klen - 1);
    for (int64_t r0 = 0; r0 < rows; r0 += 65535) {
        const int64_t nr = rows - r0 < 65535 ? rows - r0 : 65535;
        dim3 grid((unsigned)cdiv(W, GR_TILE), (unsigned)nr);
        ProfScope ps(K_GAUSS_ROWS, 2.0 * sizeof(T) * nr * W, st);
        if (border != FDN_BORDER_WRAP)
            k_gauss_rows<T, true, true><<<grid, 256, smem, st>>>(in + r0 * W, out + r0 * W, W, t64, t32, border);
        else
            k_gauss_rows<T, true, false><<<grid, 256, smem, st>>>(in + r0 * W, out + r0 * W, W, t64, t32, border);
        FDN_LAUNCHED("k_gauss_rows");
    }
    return FDN_OK;
}

#define FDN_INST_NOOF(T)                                                                                              \
    template int launch_gauss_axis_typed<T>(const T*, T*, const fdn_view&, const double*, int, cudaStream_t);         \
    template int launch_gauss_rows_typed<T>(const T*, T*, int64_t, int, const double*, int, cudaStream_t, int);
FDN_INST_NOOF(uint8_t)
FDN_INST_NOOF(int8_t)
FDN_INST_NOOF(uint16_t)
FDN_INST_NOOF(int16_t)

}  // namespace fdn
