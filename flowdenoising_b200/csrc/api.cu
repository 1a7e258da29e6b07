// C ABI of libfdn_b200.so (see include/fdn_b200.h) and the host-side pass engine.
//
// The pass engine restates, as batched GPU work, the reference's per-slice loops
// (/root/reference/src/flowdenoising.py:306-327 and the Y/X twins :329-373):
//   for every output slice s: two chains (backward d = 1..r, then the centre tap, then forward d = 1..r), each
//   chain seeding the flow of neighbour d+1 with neighbour d's flow, tmp += warp(neigh, flow) * kernel[i].
// Here all output slices of a chunk advance through the chain together (one launch per stage per chain step),
// and the per-slice work that depends on one image only (pyramid levels and polynomial expansions) is computed
// once per slice per pass and cached in HBM instead of once per pair as the reference does.
#include <math.h>
#include <stdarg.h>
#include <string.h>

#include <atomic>
#include <mutex>
#include <vector>

#include "fdn_internal.cuh"

namespace fdn {

static thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

// launch log: the names of the kernels launched while it is enabled (tests assert which specialisation a level uses)
std::atomic<bool> g_launch_log_on{false};
static std::mutex g_launch_log_mutex;
static std::vector<const char*> g_launch_log;
void launch_log_add(const char* name)
{
    std::lock_guard<std::mutex> lock(g_launch_log_mutex);
    if (g_launch_log.size() < (1u << 20)) g_launch_log.push_back(name);
}

void set_error(const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
}

// ---- per-kernel event timing ----
bool g_prof_on = false;
struct ProfRec {
    cudaEvent_t a, b;
    int id;
    double bytes;
    int n, h, w;   // batch and image size of the launch (0 where the launcher does not say)
};
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_event_pool;
static std::mutex g_prof_mutex;   // the record list is shared by every host thread that launches with profiling on
static const char* const g_kernel_names[K_COUNT] = {
    "k_blur_rows", "k_blur_cols", "k_resize_linear_img", "k_polyexp", "k_flow_iter", "k_flow_area_down",
    "k_flow_upsample", "k_warp_acc", "k_gauss_axis", "k_gauss_rows", "k_transpose", "k_copy3d",
    "k_flow_gauss_iter"};

static cudaEvent_t get_event()
{
    if (!g_event_pool.empty()) {
        cudaEvent_t e = g_event_pool.back();
        g_event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}

int prof_begin(int id, double bytes, cudaStream_t st, int n, int h, int w)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    ProfRec r;
    r.a = get_event();
    r.b = get_event();
    r.id = id;
    r.bytes = bytes;
    r.n = n; r.h = h; r.w = w;
    cudaEventRecord(r.a, st);
    g_prof.push_back(r);
    return (int)g_prof.size() - 1;
}

void prof_end(int rec, cudaStream_t st)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    if (rec >= 0 && rec < (int)g_prof.size()) cudaEventRecord(g_prof[rec].b, st);
}

static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---- progress feedback (src/flowdenoising.py:139-140, :292-295: the reference counts finished slices) ----
// Thousandths of a slice, advanced by host functions placed in the stream after every chain step: the count follows
// what the device has EXECUTED, not what the host has enqueued.
static std::atomic<long long> g_progress_milli{0};
static void CUDART_CB progress_cb(void* data) { g_progress_milli.fetch_add((long long)(intptr_t)data); }
static void progress_add(cudaStream_t st, long long milli)
{
    if (milli > 0) cudaLaunchHostFunc(st, progress_cb, (void*)(intptr_t)milli);
}

struct Geometry {
    int nl;  // extra levels
    int hs[FDN_MAX_LEVELS + 1], ws[FDN_MAX_LEVELS + 1], ksz[FDN_MAX_LEVELS + 1];
    double sigma[FDN_MAX_LEVELS + 1];
    size_t R_off[FDN_MAX_LEVELS + 1];  // float offset of level k inside one slot
    size_t R_slot;                     // floats per slot
};

static int make_geometry(int H, int W, int levels, Geometry* g)
{
    if (levels > FDN_MAX_LEVELS) levels = FDN_MAX_LEVELS;
    if (levels < 0) levels = 0;
    g->nl = fdn_level_geometry(H, W, levels, g->hs, g->ws, g->ksz, g->sigma);
    size_t off = 0;
    for (int k = 0; k <= g->nl; k++) {
        g->R_off[k] = off;
        off += R_image_floats(g->hs[k], g->ws[k]);
    }
    g->R_slot = off;
    for (int k = 0; k <= g->nl; k++)
        if (g->ksz[k] > FDN_MAX_KSZ) {
            set_error("pyramid level %d needs a %d-tap smoothing kernel (max %d)", k, g->ksz[k], FDN_MAX_KSZ);
            return FDN_ERR_INVALID;
        }
    return FDN_OK;
}

// the border arithmetic (border_index: periods up to 2 n) stays inside int
static int check_border_extent(int periodic, int64_t n)
{
    FDN_CHECK_ARG(view_border(periodic) == FDN_BORDER_WRAP || n <= (1 << 30),
                  "border %d needs an axis of at most 2^30 slices (%lld)", periodic, (long long)n);
    return FDN_OK;
}

static int check_of(const fdn_of_params* of)
{
    FDN_CHECK_ARG(of->winsize >= 1 && of->winsize <= 31, "winsize %d unsupported (1..31)", of->winsize);
    FDN_CHECK_ARG(of->iterations >= 1, "iterations must be >= 1");
    FDN_CHECK_ARG(of->poly_n >= 1 && of->poly_n <= 7, "poly_n %d unsupported (1..7)", of->poly_n);
    FDN_CHECK_ARG(of->levels >= 0, "levels must be >= 0");
    FDN_CHECK_ARG((of->flags & ~FDN_OF_FARNEBACK_GAUSSIAN) == 0, "unsupported flags 0x%x (only FDN_OF_FARNEBACK_GAUSSIAN)",
                  (unsigned)of->flags);
    return FDN_OK;
}

// Pyramid + polynomial expansion of `n` images (view-strided input, image b = input slice in_map.slot(b)) into
// R slots R_map.slot(b). tmpA/tmpB/img: scratch of n*H*W floats each. T: element type of the input view.
template <typename T>
static int build_R(const T* in, int64_t in_ss, int64_t in_rs, SlotMap in_map, int n, int H, int W,
                   const Geometry& g, const PolyConsts& pc, float* R, SlotMap R_map, float* tmpA, float* tmpB,
                   float* img, cudaStream_t st)
{
    int rc;
    for (int k = 0; k <= g.nl; k++) {
        BlurTaps bt;
        if ((rc = prepare_blur_taps(g.ksz[k], g.sigma[k], &bt))) return rc;
        const int h = g.hs[k], w = g.ws[k];
        if ((rc = launch_blur_rows(in, in_ss, in_rs, in_map, tmpA, n, H, W, bt, st))) return rc;
        const float* level_img;
        if (h == H && w == W) {
            if ((rc = launch_blur_cols(tmpA, img, n, H, W, bt, st))) return rc;
            level_img = img;
        } else {
            if ((rc = launch_blur_cols(tmpA, tmpB, n, H, W, bt, st))) return rc;
            if ((rc = launch_resize_linear_img(tmpB, n, H, W, img, (int64_t)h * w, h, w, st))) return rc;
            level_img = img;
        }
        if ((rc = launch_polyexp(level_img, (int64_t)h * w, R + g.R_off[k], (int64_t)g.R_slot, R_map, n, h, w, pc,
                                 st)))
            return rc;
    }
    return FDN_OK;
}

// Farneback for a batch of n pairs whose polynomial expansions are cached in R (pair b: prev = map0.slot(b),
// next = map1.slot(b)). P: (n, H, W, 2) initial flow in / final flow out. S1, S2: scratch of the same size.
// The iterations of a level rotate through the three buffers (launch_flow_level); the level transfers are placed
// so that, for the usual iteration counts, the last iteration of level 0 writes P itself.
static int farneback_batch(const float* R, const Geometry& g, SlotMap map0, SlotMap map1, float* P, float* S1,
                           float* S2, int n, int H, int W, const fdn_of_params& of, const FlowScratch& fs,
                           cudaStream_t st)
{
    int rc;
    float* cur = nullptr;
    int ch = 0, cw = 0;
    const int iters = of.iterations;
    for (int k = g.nl; k >= 0; k--) {
        const int h = g.hs[k], w = g.ws[k];
        const size_t fbytes = sizeof(float) * 2 * (size_t)n * h * w;
        // where this level's input flow should live so that its result ends up where the next step wants it:
        // the result of `iters` iterations lands in rotation slot iters % 3 of {cur, a, b}
        //   level 0: result in P      -> iters % 3 == 0: cur = P;  else cur != P and P in slot iters % 3
        //   level k > 0: result != P  -> (the next upsample can then write P if it has to)
        float* want_cur;
        if (k == 0) want_cur = (iters % 3 == 0) ? P : nullptr;   // nullptr: anything but P
        else want_cur = nullptr;
        if (k == g.nl) {
            if (of.use_prev_flow) {
                if (k == 0) {
                    cur = P;  // same-size INTER_AREA resize times 1
                } else {
                    if ((rc = launch_flow_area_down(P, n, H, W, S1, h, w, (float)ldexp(1.0, -k), st))) return rc;
                    cur = S1;
                }
            } else {
                cur = (k == 0) ? P : S1;
                FDN_CUDA(cudaMemsetAsync(cur, 0, fbytes, st));
            }
        } else {
            float* dst = want_cur ? want_cur : (cur == S1 ? S2 : S1);   // cur != P here (see below)
            if ((rc = launch_flow_upsample(cur, n, ch, cw, dst, h, w, st))) return rc;
            cur = dst;
        }
        // order the other two buffers: the rotation slot of the result (iters % 3: 0 -> cur, 1 -> a, 2 -> b) must be P at
        // level 0 and should not be P above it (so that the next upsample may write P)
        float* others[2];
        int no = 0;
        float* const all3[3] = {P, S1, S2};
        for (int q = 0; q < 3; q++)
            if (all3[q] != cur) others[no++] = all3[q];
        float* a = others[0];
        float* b = others[1];
        const int slot = iters % 3;
        const bool want_P = (k == 0);
        if ((slot == 1 && (a == P) != want_P) || (slot == 2 && (b == P) != want_P)) { float* t = a; a = b; b = t; }
        float* res = nullptr;
        if (of.flags & FDN_OF_FARNEBACK_GAUSSIAN)
            rc = launch_flow_level_gauss(R + g.R_off[k], (int64_t)g.R_slot, map0, map1, cur, a, b, n, h, w, of.winsize,
                                         iters, st, &res);
        else
            rc = launch_flow_level(R + g.R_off[k], (int64_t)g.R_slot, map0, map1, cur, a, b, n, h, w, of.winsize, iters,
                                   fs, st, &res);
        if (rc) return rc;
        cur = res;
        ch = h; cw = w;
    }
    if (cur != P) FDN_CUDA(cudaMemcpyAsync(P, cur, sizeof(float) * 2 * (size_t)n * H * W, cudaMemcpyDeviceToDevice, st));
    return FDN_OK;
}

struct PassPlan {
    int chunk, r, slots, full_wrap;   // slots: R-cache slots per volume (the cache holds batch * slots)
    int batch;
    Geometry g;
    size_t off_R, off_P, off_S1, off_S2, off_stash, off_scratch, scratch_bytes, off_acc, total;
};

// esize: bytes per element of the volume (4: float32, whose accumulator is the output itself; 1 or 2: a typed volume,
// whose stash holds T and whose float32 accumulator for one chunk follows the other buffers)
// batch > 1: volumes of one whole periodic axis each (fdn_filter_axis_batch), every per-chunk buffer holds batch chunks
static int make_plan(const fdn_view& v, int klen, const fdn_of_params& of, int chunk, size_t esize, PassPlan* p,
                     int batch = 1)
{
    int rc;
    FDN_CHECK_ARG(klen >= 1 && (klen & 1), "kernel length must be odd (src/flowdenoising.py:309)");
    // checked here, before the first launch of the pass: the centre / forward taps (launch_acc_finish) take r <= 128
    FDN_CHECK_ARG(klen <= FDN_MAX_KLEN, "kernel length %d unsupported (<= %d, sigma < 32.125)", klen, FDN_MAX_KLEN);
    FDN_CHECK_ARG(v.n_in >= 1 && v.n_out >= 1 && v.H >= 1 && v.W >= 1, "empty view");
    p->r = klen / 2;
    if (v.periodic) {
        FDN_CHECK_ARG(v.halo >= 0 && v.halo < v.n_in && v.n_out <= v.n_in,
                      "periodic views need 0 <= halo < n_in and n_out <= n_in (halo=%d, n_in=%d, n_out=%d)", v.halo,
                      v.n_in, v.n_out);
    } else {
        FDN_CHECK_ARG(v.halo >= p->r && v.n_in >= v.n_out + v.halo + p->r,
                      "non-periodic view needs >= r halo slices on both sides (r=%d, halo=%d, n_in=%d, n_out=%d)",
                      p->r, v.halo, v.n_in, v.n_out);
    }
    if ((rc = check_border_extent(v.periodic, v.n_in))) return rc;
    if ((rc = check_of(&of))) return rc;
    if ((rc = make_geometry(v.H, v.W, of.levels, &p->g))) return rc;
    FDN_CHECK_ARG(batch >= 1, "batch must be >= 1");
    FDN_CHECK_ARG(batch == 1 || (v.periodic && v.halo == 0 && v.n_out == v.n_in),
                  "a batch member must be a whole periodic axis (periodic = 1, halo = 0, n_out = n_in)");
    // image pairs of one launch: 2 * batch * chunk (kept inside int, like every image index of the kernels)
    FDN_CHECK_ARG(2ll * batch * v.n_out < (1ll << 31), "too many image pairs in one batch");
    p->batch = batch;
    if (chunk <= 0 || chunk > v.n_out || batch > 1) chunk = v.n_out;
    p->chunk = chunk;
    p->full_wrap = v.periodic && (chunk + 2 * p->r >= v.n_in);
    p->slots = p->full_wrap ? v.n_in : chunk + 2 * p->r;
    // both chain directions advance together: 2 * chunk image pairs per launch
    const size_t px = (size_t)batch * chunk * v.H * v.W;
    const size_t fl = sizeof(float) * 2 * 2 * px;
    size_t off = 0;
    p->off_R = off;  off += align_up(sizeof(float) * p->g.R_slot * (size_t)p->slots * batch, 256);
    p->off_P = off;  off += align_up(fl, 256);
    p->off_S1 = off; off += align_up(fl, 256);
    p->off_S2 = off; off += align_up(fl, 256);
    p->off_stash = off; off += align_up(esize * px * (size_t)p->r, 256);   // remapped forward neighbours
    p->scratch_bytes = flow_iter_scratch_bytes(2 * batch * chunk, p->g.nl + 1, p->g.hs, p->g.ws);   // every level
    p->off_scratch = off; off += align_up(p->scratch_bytes, 256);
    p->off_acc = off;
    if (esize != sizeof(float)) off += align_up(sizeof(float) * px, 256);
    p->total = off;
    return FDN_OK;
}

// T = float: the accumulator is d_out itself. Integer T: a float32 accumulator of one chunk in the workspace; the last
// tap truncates it into d_out (the reference's `filtered_vol[z] = tmp_slice` into an integer volume).
// batch > 1 (make_plan: whole periodic axes, one chunk): volume g reads d_in + g * in_bs and writes d_out + g * out_bs.
// A launch's images are ordered [chain][volume][slice]: pairs [0, B*C) are the backward neighbours, [B*C, 2*B*C) the
// forward ones, and the SlotMaps resolve image j of a chain to volume j / C, slice j % C.
template <typename T>
static int filter_axis_of(const T* d_in, T* d_out, const fdn_view& v, const double* kernel, int klen,
                          const fdn_of_params& of, int chunk, void* ws, size_t ws_bytes, cudaStream_t st,
                          int batch = 1, int64_t in_bs = 0, int64_t out_bs = 0)
{
    constexpr bool typed = !std::is_same<T, float>::value;
    int rc;
    PassPlan p;
    if ((rc = make_plan(v, klen, of, chunk, sizeof(T), &p, batch))) return rc;
    if (ws_bytes < p.total || ws == nullptr) {
        set_error("workspace too small: need %zu bytes, got %zu", p.total, ws_bytes);
        return FDN_ERR_WORKSPACE;
    }
    const int r = p.r, H = v.H, W = v.W;
    char* base = static_cast<char*>(ws);
    float* R = reinterpret_cast<float*>(base + p.off_R);
    float* P = reinterpret_cast<float*>(base + p.off_P);
    float* S1 = reinterpret_cast<float*>(base + p.off_S1);
    float* S2 = reinterpret_cast<float*>(base + p.off_S2);
    T* stash = reinterpret_cast<T*>(base + p.off_stash);
    FlowScratch fs;
    if ((rc = flow_scratch_make(base + p.off_scratch, p.scratch_bytes, 2 * batch * p.chunk, p.g.nl + 1, p.g.hs, p.g.ws,
                                &fs)))
        return rc;
    if ((rc = flow_iter_scratch_init(fs, st))) return rc;
    PolyConsts pc;
    prepare_poly_consts(of.poly_n, of.poly_sigma, &pc);
    const int wrap_in = v.periodic ? v.n_in : 0;
    const int border = view_border(v.periodic);   // of every map below that wraps (input slices, full_wrap R slots)
    const int64_t R_vs = (int64_t)p.slots * p.g.R_slot;   // R-cache floats per volume
    bool cache_full = false;

    for (int c0 = 0; c0 < v.n_out; c0 += p.chunk) {
        const int C = v.n_out - c0 < p.chunk ? v.n_out - c0 : p.chunk;
        const int ubase = c0 + v.halo - r;  // first (unwrapped) input slice this chunk touches
        // ---- stages 1+2 for every slice the chunk needs (S1/S2 double as image scratch) ----
        if (!(p.full_wrap && cache_full)) {
            const int need = p.full_wrap ? v.n_in : C + 2 * r;
            float* tmpA = S1;
            float* tmpB = S1 + (size_t)batch * p.chunk * H * W;
            float* img = S2;
            // batch > 1: one sub-batch of every slice of every volume (need == chunk); R slot b = volume * n_in + slice
            for (int sb = 0; sb < batch * need; sb += batch * p.chunk) {
                const int nb = batch * need - sb < batch * p.chunk ? batch * need - sb : batch * p.chunk;
                SlotMap in_map{p.full_wrap ? sb : ubase + sb, wrap_in};
                in_map.border = border;
                in_map.per = need;
                in_map.vstride = in_bs;
                SlotMap R_map{sb, 0};
                if ((rc = build_R(d_in, v.in_slice_stride, v.in_row_stride, in_map, nb, H, W, p.g, pc, R, R_map, tmpA,
                                  tmpB, img, st)))
                    return rc;
            }
            cache_full = p.full_wrap;
        }
        // ---- the two chains (src/flowdenoising.py:311-316 backward, :319-324 forward) advance together: image
        //      pairs [0, C) = (slice, slice - d), pairs [C, 2C) = (slice, slice + d) ----
        const int cbase = p.full_wrap ? c0 + v.halo : r;             // R slot of the chunk's first centre slice
        const int swrap = p.full_wrap ? v.n_in : 0;
        const int BC = batch * C;                                    // pairs of one chain
        // every map below resolves image j of a chain to volume j / C, slice j % C (one volume: always volume 0)
        auto vmap = [&](int b1, int wrap, int split, int b2, int64_t vstride) {
            SlotMap m{b1, wrap, split, b2};
            m.border = border;
            m.per = C;
            m.vstride = vstride;
            return m;
        };
        const SlotMap map0 = vmap(cbase, swrap, BC, cbase, R_vs);
        T* out = d_out + (int64_t)c0 * v.out_slice_stride;
        float* acc = typed ? reinterpret_cast<float*>(base + p.off_acc) : reinterpret_cast<float*>(out);
        const int64_t a_ss = typed ? (int64_t)H * W : v.out_slice_stride, a_rs = typed ? (int64_t)W : v.out_row_stride;
        const SlotMap amap = vmap(0, 0, 0x7fffffff, 0, typed ? 0 : out_bs);   // (typed: batch == 1)
        const SlotMap omap = vmap(0, 0, 0x7fffffff, 0, out_bs);
        const size_t fbytes = sizeof(float) * 2 * 2 * (size_t)BC * H * W;
        if (r > 0) FDN_CUDA(cudaMemsetAsync(P, 0, fbytes, st));  // prev_flow = zeros (:310, :318)
        for (int d = 1; d <= r; d++) {
            const SlotMap map1 = vmap(cbase - d, swrap, BC, cbase + d, R_vs);
            if ((rc = farneback_batch(R, p.g, map0, map1, P, S1, S2, 2 * BC, H, W, of, fs, st))) return rc;
            // backward neighbour: tap r-d accumulated now (reference order -1, -2, ..., -r); forward neighbour:
            // remapped now, applied by launch_acc_finish after the centre tap (order 0, +1, ..., +r)
            const SlotMap nmap = vmap(c0 + v.halo - d, wrap_in, BC, c0 + v.halo + d, in_bs);
            if ((rc = launch_warp_pair(d_in, v.in_slice_stride, v.in_row_stride, nmap, P, kernel[r - d], acc, a_ss, a_rs,
                                       amap, stash + (size_t)(d - 1) * BC * H * W, BC, H, W, d == 1 ? 1 : 0, st)))
                return rc;
            progress_add(st, 1000ll * BC / (r + 1));
        }
        const SlotMap cmap = vmap(c0 + v.halo, wrap_in, 0x7fffffff, 0, in_bs);
        if ((rc = launch_acc_finish(d_in, v.in_slice_stride, v.in_row_stride, cmap, stash, r, kernel + r, acc, a_ss, a_rs,
                                    amap, out, v.out_slice_stride, v.out_row_stride, omap, BC, H, W, r > 0 ? 1 : 0, st)))
            return rc;
        progress_add(st, 1000ll * BC - (long long)r * (1000ll * BC / (r + 1)));
    }
    return FDN_OK;
}

// ---- typed volumes (FDN_DTYPE_*) ----
static size_t dtype_size(int dtype)
{
    switch (dtype) {
        case FDN_DTYPE_F32: return 4;
        case FDN_DTYPE_U8: case FDN_DTYPE_I8: return 1;
        case FDN_DTYPE_U16: case FDN_DTYPE_I16: return 2;
        default: return 0;
    }
}

static int check_dtype(int dtype, bool with_of)
{
    FDN_CHECK_ARG(dtype_size(dtype) != 0, "unknown dtype %d (FDN_DTYPE_F32, _U8, _I8, _U16 or _I16)", dtype);
    FDN_CHECK_ARG(!(with_of && dtype == FDN_DTYPE_I8),
                  "int8 volumes are supported without optical flow only (cv2.remap rejects int8 images)");
    return FDN_OK;
}

}  // namespace fdn

using namespace fdn;

#pragma GCC visibility push(default)
extern "C" {

int fdn_version(void) { return 101; }
const char* fdn_last_error(void) { return g_err; }
int64_t fdn_launch_count(void) { return g_launches.load(); }
int64_t fdn_progress_milli(void) { return (int64_t)g_progress_milli.load(); }
void fdn_progress_reset(void) { g_progress_milli.store(0); }
void fdn_reset_launch_count(void) { g_launches.store(0); }

void fdn_launch_log_enable(int on)
{
    std::lock_guard<std::mutex> lock(g_launch_log_mutex);
    if (on) g_launch_log.clear();
    g_launch_log_on.store(on != 0);
}
int fdn_launch_log_count(void)
{
    std::lock_guard<std::mutex> lock(g_launch_log_mutex);
    return (int)g_launch_log.size();
}
const char* fdn_launch_log_name(int i)
{
    std::lock_guard<std::mutex> lock(g_launch_log_mutex);
    return (i >= 0 && i < (int)g_launch_log.size()) ? g_launch_log[i] : "";
}

void fdn_profile_enable(int on) { g_prof_on = on != 0; }

void fdn_profile_reset(void)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    for (auto& r : g_prof) { g_event_pool.push_back(r.a); g_event_pool.push_back(r.b); }
    g_prof.clear();
}

int fdn_profile_kernel_count(void) { return K_COUNT; }
const char* fdn_profile_kernel_name(int id) { return (id >= 0 && id < K_COUNT) ? g_kernel_names[id] : ""; }

int fdn_profile_read(int id, double* total_ms, int64_t* launches, double* algorithmic_bytes)
{
    FDN_CHECK_ARG(id >= 0 && id < K_COUNT, "bad kernel id %d", id);
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    double ms = 0, bytes = 0;
    int64_t n = 0;
    for (auto& r : g_prof) {
        if (r.id != id) continue;
        FDN_CUDA(cudaEventSynchronize(r.b));
        float t = 0;
        FDN_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
        ms += t; bytes += r.bytes; n++;
    }
    if (total_ms) *total_ms = ms;
    if (launches) *launches = n;
    if (algorithmic_bytes) *algorithmic_bytes = bytes;
    return FDN_OK;
}

int fdn_profile_record_count(void)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    return (int)g_prof.size();
}

int fdn_profile_record(int i, int* id, int* n, int* h, int* w, double* ms, double* algorithmic_bytes)
{
    std::lock_guard<std::mutex> lock(g_prof_mutex);
    FDN_CHECK_ARG(i >= 0 && i < (int)g_prof.size(), "bad record index %d", i);
    ProfRec& r = g_prof[i];
    FDN_CUDA(cudaEventSynchronize(r.b));
    float t = 0;
    FDN_CUDA(cudaEventElapsedTime(&t, r.a, r.b));
    if (id) *id = r.id;
    if (n) *n = r.n;
    if (h) *h = r.h;
    if (w) *w = r.w;
    if (ms) *ms = t;
    if (algorithmic_bytes) *algorithmic_bytes = r.bytes;
    return FDN_OK;
}

// NumPy's pairwise summation (numpy/_core/src/umath/loops_utils.h.src, pairwise_sum): what ndarray.sum() computes
// for a contiguous float64 vector. SciPy normalises the taps with it, so the order of the additions is part of the
// reference's result.
static double numpy_pairwise_sum(const double* a, int n)
{
    if (n < 8) {
        double res = 0.;
        for (int i = 0; i < n; i++) res += a[i];
        return res;
    }
    if (n <= 128) {
        double r[8];
        for (int j = 0; j < 8; j++) r[j] = a[j];
        int i;
        for (i = 8; i < n - (n % 8); i += 8)
            for (int j = 0; j < 8; j++) r[j] += a[i + j];
        double res = ((r[0] + r[1]) + (r[2] + r[3])) + ((r[4] + r[5]) + (r[6] + r[7]));
        for (; i < n; i++) res += a[i];
        return res;
    }
    int n2 = n / 2;
    n2 -= n2 % 8;
    return numpy_pairwise_sum(a, n2) + numpy_pairwise_sum(a + n2, n - n2);
}

int fdn_gaussian_kernel(double sigma, double* taps, int cap)
{
    // scipy.ndimage._filters._gaussian_kernel1d(sigma, 0, radius=int(4*sigma+0.5)), which is what the reference's
    // delta-response loop (src/flowdenoising.py:34-45) returns after trimming the two exact zeros:
    // phi = exp(-0.5 / sigma^2 * x^2); phi / phi.sum()
    // with the C library's exp, which differs from NumPy's in the last bit for some arguments (include/fdn_b200.h); the
    // Python package computes the taps with NumPy instead (engine.gaussian_kernel)
    // (the upper bound keeps int(4 * sigma + 0.5) and the tap count inside int: infinity used to reach that cast)
    if (!(sigma > 0 && sigma <= 1e8)) { set_error("sigma must be > 0 and at most 1e8"); return 0; }
    const int r = (int)(4.0 * sigma + 0.5);
    const int n = 2 * r + 1;
    if (n > cap || !taps) return -n;
    const double sigma2 = sigma * sigma;
    for (int j = -r; j <= r; j++) {
        const double x = (double)j;
        taps[j + r] = exp(-0.5 / sigma2 * (x * x));
    }
    const double s = numpy_pairwise_sum(taps, n);
    for (int j = 0; j < n; j++) taps[j] /= s;
    return n;
}

int fdn_level_geometry(int H, int W, int levels, int* hs, int* ws, int* ksz, double* sigma)
{
    int k;
    double scale;
    if (levels > FDN_MAX_LEVELS) levels = FDN_MAX_LEVELS;
    for (k = 0, scale = 1; k < levels; k++) {
        scale *= 0.5;
        if (W * scale < 32 || H * scale < 32) break;
    }
    const int nl = k;
    for (k = 0; k <= nl; k++) {
        scale = ldexp(1.0, -k);
        const double sg = (1. / scale - 1) * 0.5;
        int s = (int)lrint(sg * 5) | 1;
        if (s < 3) s = 3;
        if (ksz) ksz[k] = s;
        if (sigma) sigma[k] = sg;
        if (ws) ws[k] = (int)lrint(W * scale);
        if (hs) hs[k] = (int)lrint(H * scale);
    }
    return nl;
}

size_t fdn_workspace_bytes(const fdn_view* view, int klen, const fdn_of_params* of, int chunk)
{
    if (!view) { set_error("null view"); return 0; }
    if (!of) return 0;  // the no-OF path needs no workspace
    PassPlan p;
    if (make_plan(*view, klen, *of, chunk, sizeof(float), &p)) return 0;
    return p.total;
}

int fdn_filter_axis(const float* d_in, float* d_out, const fdn_view* view, const double* kernel, int klen,
                    const fdn_of_params* of, int chunk, void* d_workspace, size_t workspace_bytes, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (!of) return fdn_gauss_axis(d_in, d_out, view, kernel, klen, 1, stream);
    return filter_axis_of(d_in, d_out, *view, kernel, klen, *of, chunk, d_workspace, workspace_bytes, st);
}

size_t fdn_workspace_bytes_batch(const fdn_view* view, int batch, int klen, const fdn_of_params* of)
{
    if (!view || !of) { set_error("null argument"); return 0; }
    PassPlan p;
    if (make_plan(*view, klen, *of, 0, sizeof(float), &p, batch)) return 0;
    return p.total;
}

int fdn_filter_axis_batch(const float* d_in, float* d_out, const fdn_view* view, int batch, int64_t in_batch_stride,
                          int64_t out_batch_stride, const double* kernel, int klen, const fdn_of_params* of,
                          void* d_workspace, size_t workspace_bytes, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    if (!of) return fdn_gauss_axis_batch(d_in, d_out, view, batch, in_batch_stride, out_batch_stride, kernel, klen, 1,
                                         stream);
    return filter_axis_of(d_in, d_out, *view, kernel, klen, *of, 0, d_workspace, workspace_bytes,
                          static_cast<cudaStream_t>(stream), batch, in_batch_stride, out_batch_stride);
}

int fdn_gauss_axis_batch(const float* d_in, float* d_out, const fdn_view* view, int batch, int64_t in_batch_stride,
                         int64_t out_batch_stride, const double* kernel, int klen, int exact, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    const fdn_view& v = *view;
    FDN_CHECK_ARG(batch >= 1, "batch must be >= 1");
    FDN_CHECK_ARG(klen >= 1 && (klen & 1), "kernel length must be odd");
    FDN_CHECK_ARG(klen <= FDN_MAX_KLEN, "kernel length %d unsupported (<= %d, sigma < 32.125)", klen, FDN_MAX_KLEN);
    FDN_CHECK_ARG(v.n_in >= 1 && v.H >= 1 && v.W >= 1, "empty view");
    FDN_CHECK_ARG(v.periodic && v.halo == 0 && v.n_out == v.n_in,
                  "a batch member must be a whole periodic axis (periodic = 1, halo = 0, n_out = n_in)");
    int rc0;
    if ((rc0 = check_border_extent(v.periodic, v.n_in))) return rc0;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const int rc = launch_gauss_axis(d_in, d_out, v, kernel, klen, exact, st, batch, in_batch_stride, out_batch_stride);
    if (rc == FDN_OK) progress_add(st, 1000ll * batch * v.n_out);
    return rc;
}

size_t fdn_workspace_bytes_typed(const fdn_view* view, int klen, const fdn_of_params* of, int chunk, int dtype)
{
    if (!view) { set_error("null view"); return 0; }
    if (check_dtype(dtype, of != nullptr)) return 0;
    if (!of) return 0;
    PassPlan p;
    if (make_plan(*view, klen, *of, chunk, dtype_size(dtype), &p)) return 0;
    return p.total;
}

int fdn_filter_axis_typed(const void* d_in, void* d_out, int dtype, const fdn_view* view, const double* kernel, int klen,
                          const fdn_of_params* of, int chunk, void* d_workspace, size_t workspace_bytes, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    int rc;
    if ((rc = check_dtype(dtype, of != nullptr))) return rc;
    if (!of) return fdn_gauss_axis_typed(d_in, d_out, dtype, view, kernel, klen, 1, stream);
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype) {
        case FDN_DTYPE_U8:
            return filter_axis_of(static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), *view, kernel, klen, *of,
                                  chunk, d_workspace, workspace_bytes, st);
        case FDN_DTYPE_U16:
            return filter_axis_of(static_cast<const uint16_t*>(d_in), static_cast<uint16_t*>(d_out), *view, kernel, klen,
                                  *of, chunk, d_workspace, workspace_bytes, st);
        case FDN_DTYPE_I16:
            return filter_axis_of(static_cast<const int16_t*>(d_in), static_cast<int16_t*>(d_out), *view, kernel, klen, *of,
                                  chunk, d_workspace, workspace_bytes, st);
        default:
            return fdn_filter_axis(static_cast<const float*>(d_in), static_cast<float*>(d_out), view, kernel, klen, of,
                                   chunk, d_workspace, workspace_bytes, stream);
    }
}

int fdn_gauss_axis_typed(const void* d_in, void* d_out, int dtype, const fdn_view* view, const double* kernel, int klen,
                         int exact, void* stream)
{
    int rc;
    if ((rc = check_dtype(dtype, false))) return rc;
    if (dtype == FDN_DTYPE_F32)
        return fdn_gauss_axis(static_cast<const float*>(d_in), static_cast<float*>(d_out), view, kernel, klen, exact,
                              stream);
    FDN_CHECK_ARG(exact, "typed volumes run the exact no-OF arithmetic only (the fast mode moves truncation boundaries)");
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    const fdn_view& v = *view;
    FDN_CHECK_ARG(klen >= 1 && (klen & 1), "kernel length must be odd");
    FDN_CHECK_ARG(v.n_in >= 1 && v.n_out >= 1 && v.H >= 1 && v.W >= 1, "empty view");
    if (v.periodic) FDN_CHECK_ARG(v.halo >= 0 && v.halo < v.n_in && v.n_out <= v.n_in,
                                  "periodic views need 0 <= halo < n_in and n_out <= n_in");
    else FDN_CHECK_ARG(v.halo >= klen / 2 && v.n_in >= v.n_out + v.halo + klen / 2, "halo too small");
    if ((rc = check_border_extent(v.periodic, v.n_in))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype) {
        case FDN_DTYPE_U8:
            rc = launch_gauss_axis_typed(static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), v, kernel, klen, st);
            break;
        case FDN_DTYPE_I8:
            rc = launch_gauss_axis_typed(static_cast<const int8_t*>(d_in), static_cast<int8_t*>(d_out), v, kernel, klen, st);
            break;
        case FDN_DTYPE_U16:
            rc = launch_gauss_axis_typed(static_cast<const uint16_t*>(d_in), static_cast<uint16_t*>(d_out), v, kernel, klen,
                                         st);
            break;
        default:
            rc = launch_gauss_axis_typed(static_cast<const int16_t*>(d_in), static_cast<int16_t*>(d_out), v, kernel, klen, st);
            break;
    }
    if (rc == FDN_OK) progress_add(st, 1000ll * v.n_out);
    return rc;
}

int fdn_gauss_rows_typed(const void* d_in, void* d_out, int dtype, int64_t n_rows, int W, const double* kernel, int klen,
                         int exact, void* stream)
{
    return fdn_gauss_rows_border(d_in, d_out, dtype, n_rows, W, kernel, klen, exact, FDN_BORDER_WRAP, stream);
}

int fdn_gauss_rows_border(const void* d_in, void* d_out, int dtype, int64_t n_rows, int W, const double* kernel,
                          int klen, int exact, int border, void* stream)
{
    int rc;
    FDN_CHECK_ARG(border >= FDN_BORDER_WRAP && border <= FDN_BORDER_NEAREST,
                  "unknown border %d (FDN_BORDER_WRAP, _REFLECT, _MIRROR or _NEAREST)", border);
    if ((rc = check_border_extent(border, W))) return rc;
    if ((rc = check_dtype(dtype, false))) return rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    if (dtype == FDN_DTYPE_F32) {
        FDN_CHECK_ARG(d_in && d_out && kernel && n_rows >= 1 && W >= 1, "bad argument");
        return launch_gauss_rows(static_cast<const float*>(d_in), static_cast<float*>(d_out), n_rows, W, kernel, klen,
                                 exact, st, border);
    }
    FDN_CHECK_ARG(exact, "typed volumes run the exact no-OF arithmetic only (the fast mode moves truncation boundaries)");
    FDN_CHECK_ARG(d_in && d_out && kernel && n_rows >= 1 && W >= 1, "bad argument");
    switch (dtype) {
        case FDN_DTYPE_U8:
            return launch_gauss_rows_typed(static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), n_rows, W, kernel,
                                           klen, st, border);
        case FDN_DTYPE_I8:
            return launch_gauss_rows_typed(static_cast<const int8_t*>(d_in), static_cast<int8_t*>(d_out), n_rows, W, kernel,
                                           klen, st, border);
        case FDN_DTYPE_U16:
            return launch_gauss_rows_typed(static_cast<const uint16_t*>(d_in), static_cast<uint16_t*>(d_out), n_rows, W,
                                           kernel, klen, st, border);
        default:
            return launch_gauss_rows_typed(static_cast<const int16_t*>(d_in), static_cast<int16_t*>(d_out), n_rows, W, kernel,
                                           klen, st, border);
    }
}

int fdn_transpose_yx_typed(const void* d_in, void* d_out, int dtype, int n, int A, int B, void* stream)
{
    int rc;
    if ((rc = check_dtype(dtype, false))) return rc;
    FDN_CHECK_ARG(d_in && d_out && n >= 1 && A >= 1 && B >= 1, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype_size(dtype)) {   // a transpose moves bits: one kernel per element size
        case 1: return launch_transpose(static_cast<const uint8_t*>(d_in), static_cast<uint8_t*>(d_out), n, A, B, st);
        case 2: return launch_transpose(static_cast<const uint16_t*>(d_in), static_cast<uint16_t*>(d_out), n, A, B, st);
        default: return launch_transpose(static_cast<const float*>(d_in), static_cast<float*>(d_out), n, A, B, st);
    }
}

int fdn_remap_typed(const void* d_src, const float* d_flow, void* d_dst, int dtype, int n, int H, int W, void* stream)
{
    int rc;
    if ((rc = check_dtype(dtype, true))) return rc;
    FDN_CHECK_ARG(d_src && d_flow && d_dst && n >= 1 && H >= 1 && W >= 1, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype) {
        case FDN_DTYPE_U8:
            return launch_remap(static_cast<const uint8_t*>(d_src), d_flow, static_cast<uint8_t*>(d_dst), n, H, W, st);
        case FDN_DTYPE_U16:
            return launch_remap(static_cast<const uint16_t*>(d_src), d_flow, static_cast<uint16_t*>(d_dst), n, H, W, st);
        case FDN_DTYPE_I16:
            return launch_remap(static_cast<const int16_t*>(d_src), d_flow, static_cast<int16_t*>(d_dst), n, H, W, st);
        default: {   // float32: the float path's remap (f32(0 + f64(v) * 1) == v)
            float* dst = static_cast<float*>(d_dst);
            return launch_warp_acc(static_cast<const float*>(d_src), (int64_t)H * W, W, SlotMap{0, 0}, d_flow, 1.0, dst,
                                   (int64_t)H * W, W, n, H, W, 1, st);
        }
    }
}

int fdn_gauss_axis(const float* d_in, float* d_out, const fdn_view* view, const double* kernel, int klen, int exact,
                   void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && view && kernel, "null argument");
    const fdn_view& v = *view;
    FDN_CHECK_ARG(klen >= 1 && (klen & 1), "kernel length must be odd");
    FDN_CHECK_ARG(v.n_in >= 1 && v.n_out >= 1 && v.H >= 1 && v.W >= 1, "empty view");
    if (v.periodic) FDN_CHECK_ARG(v.halo >= 0 && v.halo < v.n_in && v.n_out <= v.n_in,
                                  "periodic views need 0 <= halo < n_in and n_out <= n_in");
    else FDN_CHECK_ARG(v.halo >= klen / 2 && v.n_in >= v.n_out + v.halo + klen / 2, "halo too small");
    int rc;
    if ((rc = check_border_extent(v.periodic, v.n_in))) return rc;
    rc = launch_gauss_axis(d_in, d_out, v, kernel, klen, exact, static_cast<cudaStream_t>(stream));
    if (rc == FDN_OK) progress_add(static_cast<cudaStream_t>(stream), 1000ll * v.n_out);
    return rc;
}

int fdn_gauss_rows(const float* d_in, float* d_out, int64_t n_rows, int W, const double* kernel, int klen, int exact,
                   void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && kernel && n_rows >= 1 && W >= 1, "bad argument");
    return launch_gauss_rows(d_in, d_out, n_rows, W, kernel, klen, exact, static_cast<cudaStream_t>(stream));
}

int fdn_transpose_yx(const float* d_in, float* d_out, int n, int A, int B, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && n >= 1 && A >= 1 && B >= 1, "bad argument");
    return launch_transpose(d_in, d_out, n, A, B, static_cast<cudaStream_t>(stream));
}

int fdn_transpose_strided(const float* d_in, int64_t in_sn, int64_t in_sa, float* d_out, int64_t out_sn, int64_t out_sb,
                          int n, int A, int B, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && n >= 1 && A >= 1 && B >= 1, "bad argument");
    return launch_transpose_strided(d_in, in_sn, in_sa, d_out, out_sn, out_sb, n, A, B,
                                    static_cast<cudaStream_t>(stream));
}

int fdn_copy3d(const float* d_in, int64_t in_sa, int64_t in_sb, int b0, int b_wrap, int c0, int c_wrap, float* d_out,
               int64_t out_sa, int64_t out_sb, int A, int B, int C, void* stream)
{
    FDN_CHECK_ARG(d_in && d_out && A >= 1 && B >= 1 && C >= 1, "bad argument");
    return launch_copy3d(d_in, in_sa, in_sb, b0, b_wrap, c0, c_wrap, d_out, out_sa, out_sb, A, B, C,
                         static_cast<cudaStream_t>(stream));
}

int fdn_transpose_strided_typed(const void* d_in, int dtype, int64_t in_sn, int64_t in_sa, void* d_out, int64_t out_sn,
                                int64_t out_sb, int n, int A, int B, void* stream)
{
    int rc;
    if ((rc = check_dtype(dtype, false))) return rc;
    FDN_CHECK_ARG(d_in && d_out && n >= 1 && A >= 1 && B >= 1, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype_size(dtype)) {   // a transpose moves bits: one kernel per element size
        case 1:
            return launch_transpose_strided(static_cast<const uint8_t*>(d_in), in_sn, in_sa, static_cast<uint8_t*>(d_out),
                                            out_sn, out_sb, n, A, B, st);
        case 2:
            return launch_transpose_strided(static_cast<const uint16_t*>(d_in), in_sn, in_sa,
                                            static_cast<uint16_t*>(d_out), out_sn, out_sb, n, A, B, st);
        default:
            return fdn_transpose_strided(static_cast<const float*>(d_in), in_sn, in_sa, static_cast<float*>(d_out), out_sn,
                                         out_sb, n, A, B, stream);
    }
}

int fdn_copy3d_typed(const void* d_in, int dtype, int64_t in_sa, int64_t in_sb, int b0, int b_wrap, int c0, int c_wrap,
                     void* d_out, int64_t out_sa, int64_t out_sb, int A, int B, int C, void* stream)
{
    int rc;
    if ((rc = check_dtype(dtype, false))) return rc;
    FDN_CHECK_ARG(d_in && d_out && A >= 1 && B >= 1 && C >= 1, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    switch (dtype_size(dtype)) {   // a copy moves bits: one kernel per element size
        case 1:
            return launch_copy3d(static_cast<const uint8_t*>(d_in), in_sa, in_sb, b0, b_wrap, c0, c_wrap,
                                 static_cast<uint8_t*>(d_out), out_sa, out_sb, A, B, C, st);
        case 2:
            return launch_copy3d(static_cast<const uint16_t*>(d_in), in_sa, in_sb, b0, b_wrap, c0, c_wrap,
                                 static_cast<uint16_t*>(d_out), out_sa, out_sb, A, B, C, st);
        default:
            return fdn_copy3d(static_cast<const float*>(d_in), in_sa, in_sb, b0, b_wrap, c0, c_wrap,
                              static_cast<float*>(d_out), out_sa, out_sb, A, B, C, stream);
    }
}

int fdn_copy2d_async(void* dst, size_t dst_pitch, const void* src, size_t src_pitch, size_t width_bytes, size_t rows,
                     int direction, void* stream)
{
    FDN_CHECK_ARG(dst && src && width_bytes >= 1 && rows >= 1 && dst_pitch >= width_bytes && src_pitch >= width_bytes,
                  "bad argument");
    FDN_CHECK_ARG(direction >= 0 && direction <= 2, "direction must be 0 (host to device), 1 (device to host) or 2");
    const cudaMemcpyKind kind = direction == 0 ? cudaMemcpyHostToDevice
                              : direction == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    FDN_CUDA(cudaMemcpy2DAsync(dst, dst_pitch, src, src_pitch, width_bytes, rows, kind,
                               static_cast<cudaStream_t>(stream)));
    return FDN_OK;
}

int fdn_pyramid_level(const float* d_img, int n, int H, int W, int64_t slice_stride, int64_t row_stride, int ksz,
                      double sigma, int h, int w, float* d_tmp, float* d_out, void* stream)
{
    FDN_CHECK_ARG(d_img && d_tmp && d_out && n >= 1, "bad argument");
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    int rc;
    BlurTaps bt;
    if ((rc = prepare_blur_taps(ksz, sigma, &bt))) return rc;
    float* tmpA = d_tmp;
    float* tmpB = d_tmp + (size_t)n * H * W;
    if ((rc = launch_blur_rows(d_img, slice_stride, row_stride, SlotMap{0, 0}, tmpA, n, H, W, bt, st))) return rc;
    if (h == H && w == W) return launch_blur_cols(tmpA, d_out, n, H, W, bt, st);
    if ((rc = launch_blur_cols(tmpA, tmpB, n, H, W, bt, st))) return rc;
    return launch_resize_linear_img(tmpB, n, H, W, d_out, (int64_t)h * w, h, w, st);
}

int fdn_polyexp(const float* d_img, int n, int h, int w, int poly_n, double poly_sigma, float* d_R, void* stream)
{
    FDN_CHECK_ARG(d_img && d_R && n >= 1, "bad argument");
    FDN_CHECK_ARG(poly_n >= 1 && poly_n <= 7, "poly_n %d unsupported (1..7)", poly_n);
    PolyConsts pc;
    prepare_poly_consts(poly_n, poly_sigma, &pc);
    return launch_polyexp(d_img, (int64_t)h * w, d_R, (int64_t)R_image_floats(h, w), SlotMap{0, 0}, n, h, w, pc,
                          static_cast<cudaStream_t>(stream));
}

size_t fdn_polyexp_floats(int h, int w) { return R_image_floats(h, w); }

size_t fdn_flow_iteration_scratch_bytes(int n, int h, int w) { return flow_iter_scratch_bytes(n, 1, &h, &w); }

void fdn_set_flow_iter_variant(int variant) { set_flow_iter_variant(variant); }

int fdn_flow_iterations(const float* d_R0, const float* d_R1, float* d_flow, float* d_tmp1, float* d_tmp2, int n, int h,
                        int w, int winsize, int iterations, void* d_scratch, size_t scratch_bytes, void* stream,
                        float** d_result)
{
    FDN_CHECK_ARG(d_R0 && d_R1 && d_flow && d_tmp1 && d_tmp2 && n >= 1 && iterations >= 1 && d_result, "bad argument");
    // R0 and R1 are separate dense batches: address both relative to R0 with a slot stride of one image
    const int64_t stride = (int64_t)R_image_floats(h, w);
    int rc;
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    FlowScratch fs;
    if ((rc = flow_scratch_make(d_scratch, scratch_bytes, n, 1, &h, &w, &fs))) return rc;
    if ((rc = flow_iter_scratch_init(fs, st))) return rc;
    const ptrdiff_t delta = d_R1 - d_R0;
    FDN_CHECK_ARG(delta % stride == 0, "R1 - R0 must be a multiple of one image (fdn_polyexp_floats(h, w))");
    return launch_flow_level(d_R0, stride, SlotMap{0, 0}, SlotMap{(int)(delta / stride), 0}, d_flow, d_tmp1, d_tmp2, n, h,
                             w, winsize, iterations, fs, st, d_result);
}

int fdn_flow_iterations_gaussian(const float* d_R0, const float* d_R1, float* d_flow, float* d_tmp1, float* d_tmp2, int n,
                                 int h, int w, int winsize, int iterations, void* stream, float** d_result)
{
    FDN_CHECK_ARG(d_R0 && d_R1 && d_flow && d_tmp1 && d_tmp2 && n >= 1 && iterations >= 1 && d_result, "bad argument");
    const int64_t stride = (int64_t)R_image_floats(h, w);
    const ptrdiff_t delta = d_R1 - d_R0;
    FDN_CHECK_ARG(delta % stride == 0, "R1 - R0 must be a multiple of one image (fdn_polyexp_floats(h, w))");
    return launch_flow_level_gauss(d_R0, stride, SlotMap{0, 0}, SlotMap{(int)(delta / stride), 0}, d_flow, d_tmp1, d_tmp2,
                                   n, h, w, winsize, iterations, static_cast<cudaStream_t>(stream), d_result);
}

int fdn_flow_iteration(const float* d_R0, const float* d_R1, const float* d_flow_in, float* d_flow_out, int n, int h,
                       int w, int winsize, void* d_scratch, size_t scratch_bytes, void* stream)
{
    FDN_CHECK_ARG(d_R0 && d_R1 && d_flow_in && d_flow_out && n >= 1, "bad argument");
    FDN_CHECK_ARG(d_flow_in != d_flow_out, "flow_in and flow_out must not alias");
    // a single iteration touches two of the three rotation buffers: the third is never dereferenced
    float* res = nullptr;
    float* in = const_cast<float*>(d_flow_in);
    float* dummy = reinterpret_cast<float*>(static_cast<char*>(d_scratch));   // distinct address, unused with 1 iteration
    int rc = fdn_flow_iterations(d_R0, d_R1, in, d_flow_out, dummy, n, h, w, winsize, 1, d_scratch, scratch_bytes, stream,
                                 &res);
    if (rc) return rc;
    if (res != d_flow_out) { set_error("internal: unexpected result buffer"); return FDN_ERR_INVALID; }
    return FDN_OK;
}

int fdn_flow_area_down(const float* d_flow, int n, int H, int W, float* d_out, int h, int w, float scale, void* stream)
{
    FDN_CHECK_ARG(d_flow && d_out && n >= 1, "bad argument");
    return launch_flow_area_down(d_flow, n, H, W, d_out, h, w, scale, static_cast<cudaStream_t>(stream));
}

int fdn_flow_upsample(const float* d_flow, int n, int h_in, int w_in, float* d_out, int h, int w, void* stream)
{
    FDN_CHECK_ARG(d_flow && d_out && n >= 1, "bad argument");
    return launch_flow_upsample(d_flow, n, h_in, w_in, d_out, h, w, static_cast<cudaStream_t>(stream));
}

size_t fdn_farneback_workspace_bytes(int n, int H, int W, const fdn_of_params* of)
{
    if (!of || n < 1) { set_error("bad argument"); return 0; }
    Geometry g;
    if (make_geometry(H, W, of->levels, &g)) return 0;
    const size_t fl = align_up(sizeof(float) * 2 * (size_t)n * H * W, 256);
    return align_up(sizeof(float) * g.R_slot * 2 * (size_t)n, 256) + 2 * fl +
           align_up(flow_iter_scratch_bytes(n, g.nl + 1, g.hs, g.ws), 256);
}

int fdn_farneback(const float* d_prev, const float* d_next, float* d_flow, int n, int H, int W,
                  const fdn_of_params* of, void* d_workspace, size_t workspace_bytes, void* stream)
{
    FDN_CHECK_ARG(d_prev && d_next && d_flow && of && n >= 1, "bad argument");
    int rc;
    if ((rc = check_of(of))) return rc;
    Geometry g;
    if ((rc = make_geometry(H, W, of->levels, &g))) return rc;
    const size_t need = fdn_farneback_workspace_bytes(n, H, W, of);
    if (!d_workspace || workspace_bytes < need) {
        set_error("workspace too small: need %zu bytes, got %zu", need, workspace_bytes);
        return FDN_ERR_WORKSPACE;
    }
    cudaStream_t st = static_cast<cudaStream_t>(stream);
    const size_t fl = align_up(sizeof(float) * 2 * (size_t)n * H * W, 256);
    char* base = static_cast<char*>(d_workspace);
    float* R = reinterpret_cast<float*>(base);
    float* S1 = reinterpret_cast<float*>(base + align_up(sizeof(float) * g.R_slot * 2 * (size_t)n, 256));
    float* S2 = reinterpret_cast<float*>(reinterpret_cast<char*>(S1) + fl);
    FlowScratch fs;
    if ((rc = flow_scratch_make(reinterpret_cast<char*>(S2) + fl, flow_iter_scratch_bytes(n, g.nl + 1, g.hs, g.ws), n,
                                g.nl + 1, g.hs, g.ws, &fs)))
        return rc;
    if ((rc = flow_iter_scratch_init(fs, st))) return rc;
    PolyConsts pc;
    prepare_poly_consts(of->poly_n, of->poly_sigma, &pc);
    // slots [0, n): prev images, [n, 2n): next images. S1/S2 double as image scratch (3*n*H*W floats needed).
    float* tmpA = S1;
    float* tmpB = S1 + (size_t)n * H * W;
    float* img = S2;
    if ((rc = build_R(d_prev, (int64_t)H * W, W, SlotMap{0, 0}, n, H, W, g, pc, R, SlotMap{0, 0}, tmpA, tmpB, img, st)))
        return rc;
    if ((rc = build_R(d_next, (int64_t)H * W, W, SlotMap{0, 0}, n, H, W, g, pc, R, SlotMap{n, 0}, tmpA, tmpB, img, st)))
        return rc;
    return farneback_batch(R, g, SlotMap{0, 0}, SlotMap{n, 0}, d_flow, S1, S2, n, H, W, *of, fs, st);
}

int fdn_warp_accumulate(const float* d_neigh, int64_t neigh_slice_stride, int64_t neigh_row_stride,
                        const float* d_flow, double weight, float* d_acc, int64_t acc_slice_stride,
                        int64_t acc_row_stride, int n, int H, int W, void* stream)
{
    FDN_CHECK_ARG(d_neigh && d_acc && n >= 1, "bad argument");
    return launch_warp_acc(d_neigh, neigh_slice_stride, neigh_row_stride, SlotMap{0, 0}, d_flow, weight, d_acc,
                           acc_slice_stride, acc_row_stride, n, H, W, 0, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
#pragma GCC visibility pop
