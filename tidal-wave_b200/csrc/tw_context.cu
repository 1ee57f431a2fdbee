// tw_context.cu -- host side of the C ABI: context, per-shape plan (pyramid schedule + tables), the launch
// sequence, result fetch, measurement hooks.  Mirrors OpticalFlow::calculate / calculateInternal
// (/root/reference/src/opticalflow.cpp:20-119) and the sampling of Consumer::run (src/consumer.cpp:59-88).
#include "../../include/tidalwave_b200.h"
#include "tw_kernels.cuh"

#include <nvtx3/nvToolsExt.h> // header-only NVTX v3: one range per launch, named after the kernel family (SURVEY section 5, tracing)

#include <atomic>
#include <cfloat>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace tw;

namespace {

enum Family { F_LEVEL = 0, F_POLY, F_FIRST, F_GITER, F_GLAST, F_BVSUM, F_BITER, F_BLAST, F_BUPD, F_SAMPLE, F_PAINT, F_MASK, F_REGIONS, F_INTENSITY, F_COUNT };
const char *kFamilyNames[F_COUNT] = {"level_image", "polyexp", "first_update", "gauss_iter", "gauss_last",
                                     "box_vsum", "box_hscan", "box_hscan_last", "box_update", "sample", "ignore_paint",
                                     "mask_paint", "change_regions", "intensity"};

struct Scale {
    int k, ksize;
    double sigma;
    LevelDims d;
    // device tables
    int *img_xi = nullptr, *img_yi = nullptr, *up_xi = nullptr, *up_yi = nullptr;
    float *img_xf = nullptr, *img_yf = nullptr, *up_xf = nullptr, *up_yf = nullptr;
    float *taps = nullptr;
    int tile_w = 32, tile_h = 8, smem_w = 0, smem_h = 0, identity = 0;
    int int_scale = 0;            // S if the level is an exact integer down-scale with 0.5/0.5 taps (fast path), else 0
    std::vector<float> host_taps;
    // buffers (alias the shared work buffers unless keep_levels)
    float *I = nullptr, *R = nullptr, *M0 = nullptr, *M1 = nullptr, *flow = nullptr;
    StripMaps maps[2] = {}; // tensor maps of the strip window kernel reading M0 / M1 (and R) at this scale
    TileMap imap = {};      // tensor map of the level images (poly-exp input tiles by TMA)
};

// The run-time switches that change the launch sequence of a plan without rebuilding it: part of the graph key.
struct LaunchOptions {
    int arith = 1;        // 0 = faithful (App. A operation order), 1 = relaxed where validated (relaxed_in_effect)
    int sparse_last = 0;  // 1: last iteration of the finest scale only at the span-grid points (no dense flow field)
    int window_tiles = 1; // 1 (default): the tile-per-CTA window kernel (gauss_iter2_kernel); 0: the persistent TMA-fed strip kernel (tw_window.cu),
                          // bit-identical and measured 1-7 % slower (DESIGN.md section 4.2)
    int box_unfused = 0;  // 1: the three-launch box iteration (V plane through HBM), kept for the parity tests
    int level_generic = 0, level_unfused = 0;
    int change_regions = 0; // 1: the change-region kernel runs after the sample kernel
    int intensity = 0;      // "intensity_threshold" t (1 .. 255): the intensity-cell kernels run after the sample kernel; 0: off
    bool operator==(const LaunchOptions &o) const
    {
        return arith == o.arith && sparse_last == o.sparse_last && window_tiles == o.window_tiles && box_unfused == o.box_unfused &&
               level_generic == o.level_generic && level_unfused == o.level_unfused && change_regions == o.change_regions &&
               intensity == o.intensity;
    }
};

// A plan's CUDA graph of the launch sequence (enqueue) is captured for one (n, threshold, span, options, result buffer, ignore,
// mask) key.  `ignore`: the batch has ignore regions (paint launch first, the ignore form of the sample kernel).  `mask`: the batch
// has ignore masks (mask paint launch first, the mask form of the sample kernel, which also tests the regions if `ignore`).  The
// graph reads the regions from the context's region buffer and the masks from the plan's mask plane at fixed addresses, so new
// lists and new masks replay the same graph.
struct GraphKey {
    int n = 0; double thr = 0; int span = 0; LaunchOptions opt; const void *vectors = nullptr; int dev_cap = 0; bool ignore = false;
    bool mask = false;
    bool operator==(const GraphKey &o) const
    {
        return n == o.n && thr == o.thr && span == o.span && opt == o.opt && vectors == o.vectors && dev_cap == o.dev_cap &&
               ignore == o.ignore && mask == o.mask;
    }
};

struct Plan {
    bool valid = false;
    int W = 0, H = 0, batch = 0, keep = 0;
    tw_flow_param p{};
    std::vector<Scale> scales; // coarse -> fine
    PolyTables poly{};
    WinTaps win{};
    std::vector<void *> allocs;
    uint8_t *src = nullptr; // [B][2][H][spitch]
    int spitch = 0;
    double *V = nullptr; // box only
    float *T = nullptr;  // long pre-blur levels only: row-pass intermediate of launch_level_image_big
    bool fused_levels = false;
    // ignore masks ([B][H][spitch] u8, nonzero = ignore) and their per-pair flags ([B] int): allocated on the plan's first masked batch
    uint8_t *mask = nullptr;
    int *mask_has = nullptr;
    // captured launch sequence (run_sequence): graph_exec replays graph_key; seen_key is the key of the last eager run
    GraphKey graph_key, seen_key;
    cudaGraphExec_t graph_exec = nullptr;
    long long graph_launches = 0;
    unsigned long long last_use = 0; // in the plan cache: the least recently used plan is evicted first
};

} // namespace

struct tw_ctx {
    int device = 0;
    int max_w = 0, max_h = 0, max_batch = 1;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_r0 = nullptr, ev_r1 = nullptr;
    Plan plan;
    int keep_levels = 0;
    bool last_sparse = false; // the previous run left no dense field
    LaunchOptions opt;
    int opt_graph = 1;  // replay the launch sequence of a batch from a captured CUDA graph
    // options that change how plans are built: setting one rebuilds the plan
    int opt_tight_pitch = 0;
    int opt_poly_no_tma = 1;  // 0 ("polyexp_tma" = 1, TW_POLY_TMA=1): interior input tiles of the relaxed poly-exp staged by one TMA tile copy --
                              // bit-identical, measured 5 % slower than the per-thread loads (0.697 vs 0.662 ms per step), hence opt-in
    // Plans (all device buffers, tables and tensor maps of one (size, parameters)) that are not the current one, each with its
    // captured graph: screenshot directories mix page sizes, and rebuilding a plan costs tens of cudaMalloc / cudaFree calls.
    std::vector<Plan> plan_cache;
    unsigned long long use_tick = 0;
    int plan_cache_max = 3; // + the current plan (TW_PLAN_CACHE)
    // results
    int *d_counts = nullptr;
    int *h_counts = nullptr; // pinned
    // ignore regions of the batch being run: [max_batch][kMaxIgnore] int4 clipped bounds, then [max_batch] counts (ignore_bytes);
    // h_ignore is the page-locked mirror the synchronous entry points copy from
    void *d_ignore = nullptr, *h_ignore = nullptr;
    int *h_mask_has = nullptr; // page-locked [max_batch]: which pairs of the batch have a mask (the plan holds the planes)
    void *d_vectors = nullptr;
    int dev_cap = 0;
    // change regions ("change_regions"): scratch [max_batch][2][reg_cap] int, sized with d_vectors (reg_cap == dev_cap when in use),
    // the region counts [max_batch] and the regions [max_batch][kMaxChangeRegions] with their page-locked mirrors
    int *d_reg_scratch = nullptr;
    int reg_cap = 0;
    int *d_nreg = nullptr, *h_nreg = nullptr;
    tw_change_region *d_regions = nullptr, *h_regions = nullptr;
    int reg_pairs = -1; // pairs of the last answered batch whose regions the mirror holds; -1: that batch ran without the option
    // intensity cells ("intensity_threshold"): per-cell totals [max_batch][int_cap] u64 S, then [max_batch][int_cap] u32 n, then
    // [max_batch][int_chunks] per-chunk counts, sized with d_vectors like the region scratch; the cell counts [max_batch] and the
    // cells [max_batch][kMaxIntensityCells] with their page-locked mirrors.  The totals are zero between runs (the compaction clears
    // them); int_dirty: a run that launched the sums may not have reached the compaction, so they are cleared before the next one
    void *d_int_acc = nullptr;
    int int_cap = 0, int_chunks = 0;
    bool int_dirty = false;
    int *d_ncell = nullptr, *h_ncell = nullptr;
    tw_intensity_cell *d_cells = nullptr, *h_cells = nullptr;
    int cell_pairs = -1; // pairs of the last answered batch whose cells the mirror holds; -1: that batch ran without the option
    int last_n = 0, last_w = 0, last_h = 0, last_span = 0;
    bool last_regions = false; // the last run had "change_regions" on
    bool last_intensity = false; // the last run had "intensity_threshold" on
    bool ran = false;
    // profiling
    bool profiling = false;
    struct Rec { int fam; cudaEvent_t a, b; };
    std::vector<Rec> recs;
    std::vector<cudaEvent_t> ev_pool;
    float fam_ms[F_COUNT] = {0};
    int fam_launches[F_COUNT] = {0};
    double fam_bytes[F_COUNT] = {0};
    long long launches = 0;
    // pipelined batches (tw_pipe_*): upload of batch k + 1 on `copy` into `stage` while batch k runs on `stream`; the results of
    // a finished batch are snapshot on the device so that the host reads them (on `fetch`) while the next batch runs
    struct PipeSlot {
        cudaEvent_t done = nullptr, r0 = nullptr, r1 = nullptr;
        int *d_counts = nullptr, *h_counts = nullptr;
        void *d_vec = nullptr;
        void *h_ignore = nullptr; // page-locked: this batch's region lists, copied into the staging buffer behind its images
        int *h_mask_has = nullptr; // page-locked [max_batch]: which pairs of this batch have a mask
        size_t vec_bytes = 0;
        int n = 0, w = 0, h = 0, dev_cap = 0;
        // change regions of this batch (regions: it ran with the option): device snapshot of the counts and regions, counts on the host
        bool regions = false;
        int *d_nreg = nullptr, *h_nreg = nullptr;
        tw_change_region *d_regions = nullptr;
        // intensity cells of this batch (intensity: it ran with the option), snapshot likewise
        bool intensity = false;
        int *d_ncell = nullptr, *h_ncell = nullptr;
        tw_intensity_cell *d_cells = nullptr;
    };
    struct Pipe {
        cudaStream_t copy = nullptr, fetch = nullptr;
        uint8_t *stage = nullptr;
        size_t stage_bytes = 0;
        cudaEvent_t ev_up = nullptr, ev_stage_free = nullptr;
        bool stage_used = false;
        PipeSlot slot[2];
        int head = 0, count = 0;
    } pipe;
    void *rs_buf = nullptr; // +-5 px resize path: raw target + coefficient tables
    size_t rs_cap = 0;
    void *flush_buf = nullptr;
    int flush_val = 0;
    std::string err;
};

namespace {

int cv_round(double v) { return (int)nearbyint(v); }

bool set_err(tw_ctx *c, const char *what, cudaError_t e)
{
    char buf[256];
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    c->err = buf;
    cudaGetLastError(); // clear the runtime's last-error slot: the next request's first launch must not inherit this failure
    return false;
}

#define CK(call)                                                         \
    do {                                                                 \
        cudaError_t e_ = (call);                                         \
        if (e_ != cudaSuccess) { set_err(ctx, #call, e_); return false; } \
    } while (0)

void drop_graph(Plan &pl)
{
    if (pl.graph_exec) { cudaGraphExecDestroy(pl.graph_exec); pl.graph_exec = nullptr; }
    pl.graph_key = GraphKey();
    pl.seen_key = GraphKey();
}

// Frees the plan's device buffers and its graph (stream idle).
void free_plan(Plan &pl)
{
    drop_graph(pl);
    for (void *p : pl.allocs) cudaFree(p);
    pl = Plan();
}

// Frees every cached plan (stream idle): options that change how plans are built, out-of-memory, destruction.
void flush_plan_cache(tw_ctx *ctx)
{
    for (Plan &pl : ctx->plan_cache) free_plan(pl);
    ctx->plan_cache.clear();
}

// The current plan (valid or not) leaves ctx->plan: into the cache with its graph, or freed.  Stream idle.
void stash_plan(tw_ctx *ctx)
{
    if (!ctx->plan.valid || ctx->plan_cache_max < 1) { free_plan(ctx->plan); return; }
    while ((int)ctx->plan_cache.size() >= ctx->plan_cache_max) { // evict the least recently used
        size_t lru = 0;
        for (size_t i = 1; i < ctx->plan_cache.size(); i++)
            if (ctx->plan_cache[i].last_use < ctx->plan_cache[lru].last_use) lru = i;
        free_plan(ctx->plan_cache[lru]);
        ctx->plan_cache.erase(ctx->plan_cache.begin() + lru);
    }
    ctx->plan.last_use = ++ctx->use_tick;
    ctx->plan_cache.push_back(std::move(ctx->plan));
    ctx->plan = Plan();
}

template <typename T>
bool dev_alloc(tw_ctx *ctx, T **out, size_t count)
{
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, count * sizeof(T) + 256);
    if (e == cudaErrorMemoryAllocation && !ctx->plan_cache.empty()) { // out of memory: the cached plans go first (the stream is idle here)
        cudaGetLastError();
        flush_plan_cache(ctx);
        e = cudaMalloc(&p, count * sizeof(T) + 256);
    }
    if (e != cudaSuccess) return set_err(ctx, "cudaMalloc", e);
    ctx->plan.allocs.push_back(p);
    *out = reinterpret_cast<T *>(p);
    return true;
}

template <typename T>
bool dev_upload(tw_ctx *ctx, T **out, const std::vector<T> &v)
{
    if (!dev_alloc(ctx, out, v.size())) return false;
    CK(cudaMemcpyAsync(*out, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream)); // v is a temporary
    return true;
}

// SURVEY App. A.2b: per-axis bilinear coefficients (double expression, one cast).  OpenCV clamps an out-of-range
// tap along x (index clamped, fraction zeroed) but along y keeps the fraction and only clips the two row indices;
// the two rules differ in the first / last output row of an up-scale (the flow up-sample, the +-5 px target resize).
void resize_coeffs(int N, int n, std::vector<int> &idx, std::vector<float> &frac, bool clamp_fraction = true)
{
    idx.resize(n); frac.resize(n);
    double s = 1.0 / (n / (double)N);
    for (int d = 0; d < n; d++) {
        float f = (float)((d + 0.5) * s - 0.5);
        int i = (int)floorf(f);
        f = f - (float)i;
        if (clamp_fraction) {
            if (i < 0) { f = 0; i = 0; }
            if (i >= N - 1) { f = 0; i = N - 1; }
        }
        idx[d] = i; frac[d] = f;
    }
}

// OpenCV 8-bit bilinear coefficients: the float fractions scaled by 2048 and rounded half-to-even (saturate_cast<short>).
void resize_coeffs_u8(int N, int n, std::vector<int> &idx, std::vector<short> &alpha, bool clamp_fraction)
{
    std::vector<float> frac;
    resize_coeffs(N, n, idx, frac, clamp_fraction);
    alpha.resize(2 * (size_t)n);
    for (int d = 0; d < n; d++) {
        alpha[2 * d] = (short)nearbyintf((1.f - frac[d]) * 2048.f);
        alpha[2 * d + 1] = (short)nearbyintf(frac[d] * 2048.f);
    }
}

// SURVEY App. A.2a: cv::getGaussianKernel(ksize, sigma, CV_32F).
std::vector<float> gauss_taps(int ksize, double sigma)
{
    std::vector<float> k(ksize);
    if (sigma <= 0 && ksize == 3) { k[0] = 0.25f; k[1] = 0.5f; k[2] = 0.25f; return k; }
    double sx = sigma > 0 ? sigma : ((ksize - 1) * 0.5 - 1) * 0.3 + 0.8;
    double scale2x = -0.5 / (sx * sx), sum = 0;
    std::vector<double> t(ksize);
    for (int i = 0; i < ksize; i++) {
        double x = i - (ksize - 1) * 0.5;
        t[i] = std::exp(scale2x * x * x);
        sum += t[i];
    }
    sum = 1. / sum;
    for (int i = 0; i < ksize; i++) k[i] = (float)(t[i] * sum);
    return k;
}

void invert6(double A[6][6], double inv[6][6])
{
    double a[6][12];
    for (int i = 0; i < 6; i++)
        for (int j = 0; j < 6; j++) { a[i][j] = A[i][j]; a[i][j + 6] = (i == j); }
    for (int c = 0; c < 6; c++) {
        int p = c;
        for (int r = c + 1; r < 6; r++) if (std::fabs(a[r][c]) > std::fabs(a[p][c])) p = r;
        if (p != c) for (int j = 0; j < 12; j++) std::swap(a[c][j], a[p][j]);
        double d = a[c][c];
        for (int j = 0; j < 12; j++) a[c][j] /= d;
        for (int r = 0; r < 6; r++) if (r != c) {
            double f = a[r][c];
            if (f != 0) for (int j = 0; j < 12; j++) a[r][j] -= f * a[c][j];
        }
    }
    for (int i = 0; i < 6; i++) for (int j = 0; j < 6; j++) inv[i][j] = a[i][j + 6];
}

// SURVEY App. A.3 tables (FarnebackPrepareGaussian).
void poly_tables(int n, double sigma, PolyTables &t)
{
    if (sigma < FLT_EPSILON) sigma = n * 0.3;
    std::vector<float> gb(2 * n + 1), xgb(2 * n + 1), xxgb(2 * n + 1);
    float *g = gb.data() + n, *xg = xgb.data() + n, *xxg = xxgb.data() + n;
    double s = 0.;
    for (int x = -n; x <= n; x++) { g[x] = (float)std::exp(-x * x / (2 * sigma * sigma)); s += g[x]; }
    s = 1. / s;
    for (int x = -n; x <= n; x++) {
        g[x] = (float)(g[x] * s);
        xg[x] = (float)(x * g[x]);
        xxg[x] = (float)(x * x * g[x]);
    }
    double G[6][6] = {{0}}, inv[6][6];
    for (int y = -n; y <= n; y++)
        for (int x = -n; x <= n; x++) {
            float wgt = g[y] * g[x], fx = (float)x, fy = (float)y;
            G[0][0] += wgt;
            G[1][1] += wgt * fx * fx;
            G[3][3] += wgt * fx * fx * fx * fx;
            G[5][5] += wgt * fx * fx * fy * fy;
        }
    G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
    G[4][4] = G[3][3];
    G[3][4] = G[4][3] = G[5][5];
    invert6(G, inv);
    t.n = n;
    t.ig11 = inv[1][1]; t.ig03 = inv[0][3]; t.ig33 = inv[3][3]; t.ig55 = inv[5][5];
    t.fig11 = (float)t.ig11; t.fig55 = (float)t.ig55;
    t.one = 1.0f;
    for (int x = 0; x <= n; x++) {
        t.g[x] = g[x]; t.xg[x] = xg[x]; t.xxg[x] = xxg[x];
        t.gd[x] = (double)g[x]; t.xxgd[x] = (double)xxg[x];
    }
}

// SURVEY App. A.5 window taps.
void window_taps(int winSize, WinTaps &t)
{
    int m = winSize / 2;
    double sigma = m * 0.3, s = 1.;
    t.m = m;
    t.one = 1.0f;
    t.k[0] = 1.f;
    for (int i = 1; i <= m; i++) {
        float v = (float)std::exp(-i * i / (2 * sigma * sigma));
        t.k[i] = v;
        s += v * 2;
    }
    s = 1. / s;
    for (int i = 0; i <= m; i++) t.k[i] = (float)(t.k[i] * s);
}

int validate_param(const tw_flow_param *p)
{
    if (!p) return TW_BAD_PARAMETER;
    if (!(p->pyrScale > 0 && p->pyrScale < 1)) return TW_BAD_PARAMETER;
    if (p->pyrLevels < 0 || p->pyrLevels > 14) return TW_BAD_PARAMETER;
    if (p->polyN < 1 || p->polyN > kMaxPolyN) return TW_BAD_PARAMETER;
    if (p->flags != 0 && p->flags != 256) return TW_BAD_PARAMETER;
    if (p->winSize < 2 || p->winSize / 2 > kMaxWinRadius) return TW_BAD_PARAMETER;
    if (p->pyrIterations < 0 || p->pyrIterations > 100) return TW_BAD_PARAMETER;
    if (!(p->polySigma >= 0)) return TW_BAD_PARAMETER;
    return TW_OK;
}

bool same_param(const tw_flow_param &a, const tw_flow_param &b)
{
    return a.pyrScale == b.pyrScale && a.pyrLevels == b.pyrLevels && a.winSize == b.winSize &&
           a.pyrIterations == b.pyrIterations && a.polyN == b.polyN && a.polySigma == b.polySigma && a.flags == b.flags;
}

// Whether pl is a valid plan for W x H frames, parameters p and the context's batch size and keep_levels.
bool plan_fits(const tw_ctx *ctx, const Plan &pl, int W, int H, const tw_flow_param &p)
{
    return pl.valid && pl.W == W && pl.H == H && pl.batch == ctx->max_batch && pl.keep == ctx->keep_levels && same_param(pl.p, p);
}

bool build_plan(tw_ctx *ctx, int W, int H, const tw_flow_param &p)
{
    Plan &pl = ctx->plan;
    if (plan_fits(ctx, pl, W, H, p)) return true;
    CK(cudaStreamSynchronize(ctx->stream));
    stash_plan(ctx);
    for (size_t i = 0; i < ctx->plan_cache.size(); i++) { // a plan of this size and these parameters from before?
        if (plan_fits(ctx, ctx->plan_cache[i], W, H, p)) {
            pl = std::move(ctx->plan_cache[i]);
            ctx->plan_cache.erase(ctx->plan_cache.begin() + i);
            return true;
        }
    }
    pl.W = W; pl.H = H; pl.p = p; pl.batch = ctx->max_batch; pl.keep = ctx->keep_levels;
    const int B = pl.batch;

    // A.1 schedule
    int k; double scale = 1.0;
    for (k = 0; k < p.pyrLevels; k++) {
        scale *= p.pyrScale;
        if (W * scale < 32 || H * scale < 32) break;
    }
    const int L = k;
    for (k = L; k >= 0; k--) {
        Scale s;
        scale = 1.0;
        for (int i = 0; i < k; i++) scale *= p.pyrScale;
        s.k = k;
        s.sigma = (1. / scale - 1) * 0.5;
        s.ksize = std::max(cv_round(s.sigma * 5) | 1, 3);
        s.d.w = cv_round(W * scale); s.d.h = cv_round(H * scale);
        // one row pitch for every level of the plan, a compile-time constant inside the hot kernels (2048 / 4096):
        // unrolled row addresses become load immediates.  Costs address space, not traffic.
        s.d.pitch = ctx->opt_tight_pitch ? ((s.d.w + 31) & ~31) : (W <= 2048 ? 2048 : (W <= 4096 ? 4096 : ((W + 31) & ~31)));
        s.d.plane = (size_t)s.d.h * s.d.pitch;
        if (s.ksize > 1023 || s.d.w < 1 || s.d.h < 1) { ctx->err = "unsupported pyramid geometry"; return false; }
        pl.scales.push_back(s);
    }
    poly_tables(p.polyN, p.polySigma, pl.poly);
    window_taps(p.winSize, pl.win);

    pl.spitch = (W + 15) & ~15;
    if (!dev_alloc(ctx, &pl.src, (size_t)B * 2 * H * pl.spitch)) return false;

    // tables + tile geometry
    for (size_t si = 0; si < pl.scales.size(); si++) {
        Scale &s = pl.scales[si];
        std::vector<int> xi, yi; std::vector<float> xf, yf;
        resize_coeffs(W, s.d.w, xi, xf);
        resize_coeffs(H, s.d.h, yi, yf);
        s.identity = (s.d.w == W && s.d.h == H);
        const int c = s.ksize / 2;
        // choose an output tile whose float source tile + row-pass buffer leave room for >= 2 CTAs per SM (<= 64 KB); with
        // very long pre-blur kernels (79 taps at 1/32 scale) such a tile would hold only a handful of outputs behind a huge
        // halo, so fall back to the largest tile that fits one CTA per SM (<= 160 KB)
        int tw_ = s.identity ? 128 : 64, th_ = 16;
        int big_tw = 0, big_th = 0, big_sw = 0, big_sh = 0;
        for (;;) {
            int sw = 0, sh = 0;
            for (int d0 = 0; d0 < s.d.w; d0 += tw_) {
                int d1 = std::min(d0 + tw_, s.d.w) - 1;
                sw = std::max(sw, std::min(xi[d1] + 1, W - 1) + c - ((xi[d0] - c) & ~3) + 1);
            }
            for (int e0 = 0; e0 < s.d.h; e0 += th_) {
                int e1 = std::min(e0 + th_, s.d.h) - 1;
                sh = std::max(sh, std::min(yi[e1] + 1, H - 1) + c - (yi[e0] - c) + 1);
            }
            sw = (sw + 3 + 4) & ~3; // the staging loop writes whole 4-column words
            size_t bytes = level_image_smem_bytes(sw, sh, tw_, s.ksize, s.identity);
            if (!big_tw && bytes <= 160 * 1024) { big_tw = tw_; big_th = th_; big_sw = sw; big_sh = sh; }
            if (bytes <= 64 * 1024 || (tw_ == 1 && th_ == 1)) {
                if (bytes > 200 * 1024) { ctx->err = "pre-blur kernel too large for shared memory"; return false; }
                s.smem_w = sw; s.smem_h = sh;
                if (tw_ * th_ < 32 && big_tw * big_th > tw_ * th_) { tw_ = big_tw; th_ = big_th; s.smem_w = big_sw; s.smem_h = big_sh; }
                break;
            }
            if (tw_ >= th_ * 2 && tw_ > 1) tw_ /= 2; else if (th_ > 1) th_ /= 2; else tw_ /= 2;
        }
        s.tile_w = tw_; s.tile_h = th_;
        if (!dev_upload(ctx, &s.img_xi, xi) || !dev_upload(ctx, &s.img_xf, xf) || !dev_upload(ctx, &s.img_yi, yi) ||
            !dev_upload(ctx, &s.img_yf, yf))
            return false;
        s.host_taps = gauss_taps(s.ksize, s.sigma);
        if (!dev_upload(ctx, &s.taps, s.host_taps)) return false;
        // exact integer down-scale?  (tables xi/xf/yi/yf still hold the image-resize coefficients here)
        s.int_scale = 0;
        if (!s.identity && s.d.w > 0 && W % s.d.w == 0 && H % s.d.h == 0 && W / s.d.w == H / s.d.h) {
            const int S = W / s.d.w;
            bool ok = (S % 2 == 0);
            for (int d = 0; ok && d < s.d.w; d++) ok = (xi[d] == S * d + S / 2 - 1) && (xf[d] == 0.5f);
            for (int e = 0; ok && e < s.d.h; e++) ok = (yi[e] == S * e + S / 2 - 1) && (yf[e] == 0.5f);
            if (ok) s.int_scale = S;
        }
        if (si > 0) {
            const Scale &cs = pl.scales[si - 1];
            resize_coeffs(cs.d.w, s.d.w, xi, xf);
            resize_coeffs(cs.d.h, s.d.h, yi, yf, false); // rows: fraction kept, indices clipped by the kernel
            if (!dev_upload(ctx, &s.up_xi, xi) || !dev_upload(ctx, &s.up_xf, xf) || !dev_upload(ctx, &s.up_yi, yi) ||
                !dev_upload(ctx, &s.up_yf, yf))
                return false;
        }
        if (!dev_alloc(ctx, &s.flow, (size_t)B * 2 * s.d.plane)) return false;
    }
    // work buffers: shared across scales (sized for the finest) unless keep_levels
    const Scale &fine = pl.scales.back();
    float *R = nullptr, *M0 = nullptr, *M1 = nullptr;
    if (!ctx->keep_levels) {
        if (!dev_alloc(ctx, &R, (size_t)B * 10 * fine.d.plane) ||
            !dev_alloc(ctx, &M0, (size_t)B * 5 * fine.d.plane) || !dev_alloc(ctx, &M1, (size_t)B * 5 * fine.d.plane))
            return false;
    }
    for (Scale &s : pl.scales) {
        // level images are small (2 planes) and, on the fused path, all written up front: one buffer per scale
        if (!dev_alloc(ctx, &s.I, (size_t)B * 2 * s.d.plane)) return false;
        if (ctx->keep_levels) {
            if (!dev_alloc(ctx, &s.R, (size_t)B * 10 * s.d.plane) ||
                !dev_alloc(ctx, &s.M0, (size_t)B * 5 * s.d.plane) || !dev_alloc(ctx, &s.M1, (size_t)B * 5 * s.d.plane))
                return false;
        } else {
            s.R = R; s.M0 = M0; s.M1 = M1;
        }
        s.maps[0].valid = s.maps[1].valid = 0;
        s.imap.valid = 0;
        if (!ctx->opt_poly_no_tma) make_polyexp_map(s.I, s.d, 2 * B, p.polyN, &s.imap);
        if ((p.flags & 256) && pl.win.m == 15) { // no tensor maps (old driver?): the tile kernel runs instead
            make_strip_maps(s.M0, s.R, s.d, B, &s.maps[0]);
            make_strip_maps(s.M1, s.R, s.d, B, &s.maps[1]);
        }
    }
    // the default pyramid (full resolution + exact 2x / 4x / 8x with 3 / 9 / 19-tap pre-blurs) takes the fused level kernel
    // (the FINEST four scales; deeper pyramids keep their coarser scales on the per-level kernels)
    {
        const size_t nsc = pl.scales.size();
        pl.fused_levels = nsc >= 4 && pl.scales[nsc - 1].identity && pl.scales[nsc - 1].ksize == 3 && pl.scales[nsc - 2].int_scale == 2 &&
                          pl.scales[nsc - 2].ksize == 3 && pl.scales[nsc - 3].int_scale == 4 && pl.scales[nsc - 3].ksize == 9 &&
                          pl.scales[nsc - 4].int_scale == 8 && pl.scales[nsc - 4].ksize == 19 && (9 + 2 < std::min(W, H));
    }
    {   // row-pass intermediate for levels behind a long pre-blur that no exact-integer fast path takes (deep pyramids)
        size_t nT = 0;
        for (const Scale &s : pl.scales)
            if (!s.identity && s.ksize >= 31 && !(s.int_scale == 16 && s.ksize == 39)) nT = std::max(nT, level_image_big_floats(H, s.d.w, 2 * B));
        if (nT && !dev_alloc(ctx, &pl.T, nT)) return false;
    }
    if (p.flags == 0) { // box window: V planes of the three-launch form, or the band checkpoints of the fused form ([B][ceil(h/32)][5 * pitch])
        size_t nV = (size_t)B * 5 * (size_t)(fine.d.w + 32) * (size_t)(fine.d.h + 32);
        for (const Scale &s : pl.scales) nV = std::max(nV, (size_t)B * (size_t)((s.d.h + box_band_height() - 1) / box_band_height()) * 5 * (size_t)s.d.pitch);
        if (!dev_alloc(ctx, &pl.V, nV)) return false;
    }
    pl.valid = true;
    return true;
}

cudaEvent_t get_event(tw_ctx *ctx)
{
    if (!ctx->ev_pool.empty()) { cudaEvent_t e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); return e; }
    cudaEvent_t e; cudaEventCreate(&e); return e;
}

struct LaunchScope {
    tw_ctx *ctx; int fam; cudaEvent_t a = nullptr, b = nullptr;
    LaunchScope(tw_ctx *c, int f, double bytes) : ctx(c), fam(f)
    {
        nvtxRangePushA(kFamilyNames[f]);
        ctx->launches++;
        if (ctx->profiling) {
            a = get_event(ctx); b = get_event(ctx);
            cudaEventRecord(a, ctx->stream);
            ctx->fam_bytes[fam] += bytes;
            ctx->fam_launches[fam]++;
        }
    }
    ~LaunchScope()
    {
        if (ctx->profiling) { cudaEventRecord(b, ctx->stream); ctx->recs.push_back({fam, a, b}); }
        nvtxRangePop();
    }
};

void drain_profile(tw_ctx *ctx)
{
    for (auto &r : ctx->recs) {
        float ms = 0;
        if (cudaEventSynchronize(r.b) == cudaSuccess && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) ctx->fam_ms[r.fam] += ms;
        ctx->ev_pool.push_back(r.a); ctx->ev_pool.push_back(r.b);
    }
    ctx->recs.clear();
}

#define LAUNCH(fam, bytes, expr)                                          \
    do {                                                                  \
        LaunchScope ls_(ctx, fam, bytes);                                 \
        cudaError_t e_ = (expr);                                          \
        if (e_ != cudaSuccess) { set_err(ctx, #expr, e_); return false; } \
    } while (0)

bool ensure_results(tw_ctx *ctx, int cap)
{
    if (ctx->d_vectors && ctx->dev_cap >= cap) return true;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->d_vectors) cudaFree(ctx->d_vectors);
    ctx->d_vectors = nullptr;
    CK(cudaMalloc(&ctx->d_vectors, (size_t)ctx->max_batch * cap * sizeof(tw_vector)));
    ctx->dev_cap = cap;
    return true;
}

static_assert(kMaxChangeRegions == TW_MAX_CHANGE_REGIONS && sizeof(tw_change_region) == 48, "tw_change_region as the kernel writes it");

// The region counts and regions of the context (tw_ctx::d_nreg, d_regions) and their page-locked mirrors: allocated on first use,
// at a fixed size, and kept until the context goes.
bool ensure_region_mirrors(tw_ctx *ctx)
{
    if (ctx->h_regions) return true;
    const size_t bytes = (size_t)ctx->max_batch * kMaxChangeRegions * sizeof(tw_change_region);
    CK(cudaMalloc(&ctx->d_nreg, sizeof(int) * ctx->max_batch));
    CK(cudaMallocHost(&ctx->h_nreg, sizeof(int) * ctx->max_batch));
    CK(cudaMalloc(&ctx->d_regions, bytes));
    CK(cudaMallocHost(&ctx->h_regions, bytes));
    return true;
}

// Those and the scratch of the region kernel, for dev_cap.  The scratch follows the result buffer: it is reallocated only when
// dev_cap changes, which changes the graph key as well, so no captured graph keeps a freed scratch.
bool ensure_region_buffers(tw_ctx *ctx)
{
    if (!ensure_region_mirrors(ctx)) return false;
    if (ctx->d_reg_scratch && ctx->reg_cap == ctx->dev_cap) return true;
    CK(cudaStreamSynchronize(ctx->stream));
    if (ctx->d_reg_scratch) cudaFree(ctx->d_reg_scratch);
    ctx->d_reg_scratch = nullptr;
    CK(cudaMalloc(&ctx->d_reg_scratch, (size_t)ctx->max_batch * 2 * ctx->dev_cap * sizeof(int)));
    ctx->reg_cap = ctx->dev_cap;
    return true;
}

// The host mirror now answers for a batch of n pairs: with 0 regions each if `on`, else for no pair (tw_change_regions refuses).
void answer_regions(tw_ctx *ctx, int n, bool on)
{
    n = std::max(0, std::min(n, ctx->max_batch));
    ctx->reg_pairs = on && ensure_region_mirrors(ctx) ? n : -1;
    if (ctx->reg_pairs > 0) memset(ctx->h_nreg, 0, sizeof(int) * n);
}

static_assert(kMaxIntensityCells == TW_MAX_INTENSITY_CELLS && sizeof(tw_intensity_cell) == 16, "tw_intensity_cell as the kernel writes it");

// The cell counts and cells of the context (tw_ctx::d_ncell, d_cells) and their page-locked mirrors: allocated on first use, at a
// fixed size, and kept until the context goes.
bool ensure_cell_mirrors(tw_ctx *ctx)
{
    if (ctx->h_cells) return true;
    const size_t bytes = (size_t)ctx->max_batch * kMaxIntensityCells * sizeof(tw_intensity_cell);
    CK(cudaMalloc(&ctx->d_ncell, sizeof(int) * ctx->max_batch));
    CK(cudaMallocHost(&ctx->h_ncell, sizeof(int) * ctx->max_batch));
    CK(cudaMalloc(&ctx->d_cells, bytes));
    CK(cudaMallocHost(&ctx->h_cells, bytes));
    return true;
}

size_t intensity_acc_bytes(const tw_ctx *ctx)
{
    return (size_t)ctx->max_batch * ((size_t)ctx->int_cap * (sizeof(unsigned long long) + sizeof(unsigned)) + ctx->int_chunks * sizeof(int));
}

// Those and the per-cell totals, for dev_cap (>= the cells of the grid, one vector per sample point).  Like the region scratch, the
// totals are reallocated only when dev_cap changes, which changes the graph key as well; they are cleared when allocated and
// after a run that may have left them set.
bool ensure_intensity_buffers(tw_ctx *ctx)
{
    if (!ensure_cell_mirrors(ctx)) return false;
    if (!ctx->d_int_acc || ctx->int_cap != ctx->dev_cap) {
        CK(cudaStreamSynchronize(ctx->stream));
        if (ctx->d_int_acc) cudaFree(ctx->d_int_acc);
        ctx->d_int_acc = nullptr;
        ctx->int_cap = ctx->dev_cap;
        ctx->int_chunks = (ctx->dev_cap + kIntChunk - 1) / kIntChunk;
        CK(cudaMalloc(&ctx->d_int_acc, intensity_acc_bytes(ctx)));
        ctx->int_dirty = true;
    }
    if (ctx->int_dirty) {
        CK(cudaMemsetAsync(ctx->d_int_acc, 0, intensity_acc_bytes(ctx), ctx->stream));
        ctx->int_dirty = false;
    }
    return true;
}

// The host mirror now answers for a batch of n pairs: with 0 cells each if `on`, else for no pair (tw_intensity_cells refuses).
void answer_cells(tw_ctx *ctx, int n, bool on)
{
    n = std::max(0, std::min(n, ctx->max_batch));
    ctx->cell_pairs = on && ensure_cell_mirrors(ctx) ? n : -1;
    if (ctx->cell_pairs > 0) memset(ctx->h_ncell, 0, sizeof(int) * n);
}

// Region buffer (tw_ctx::d_ignore, h_ignore, the pipe's staging tail): [max_batch][kMaxIgnore] int4, then [max_batch] int.
size_t ignore_bytes(int max_batch) { return (size_t)max_batch * (kMaxIgnore * sizeof(int4) + sizeof(int)); }

IgnoreRegions ignore_regions(const void *base, int max_batch)
{
    IgnoreRegions g;
    g.rects = reinterpret_cast<const int4 *>(base);
    g.n = reinterpret_cast<const int *>(g.rects + (size_t)max_batch * kMaxIgnore);
    return g;
}

// Checks the region lists of n pairs (n_ignore == NULL: none) and writes them, clipped to the W x H frame, into `mirror` (layout of
// ignore_bytes).  Returns 1 if some pair keeps a region, 0 if none does, -1 for a bad list (ctx->err says why).
int pack_ignore(tw_ctx *ctx, int n, const tw_rect *const *ignore, const int *n_ignore, int W, int H, void *mirror)
{
    if (!n_ignore) return 0;
    for (int i = 0; i < n; i++) {
        const int k = n_ignore[i];
        if (k < 0 || k > kMaxIgnore) { ctx->err = "bad ignore region: 0 to " + std::to_string(kMaxIgnore) + " regions per pair"; return -1; }
        if (k > 0 && (!ignore || !ignore[i])) { ctx->err = "bad ignore region: NULL list with a count > 0"; return -1; }
        for (int j = 0; j < k; j++)
            if (ignore[i][j].width < 1 || ignore[i][j].height < 1) { ctx->err = "bad ignore region: width and height must be >= 1"; return -1; }
    }
    int4 *rects = reinterpret_cast<int4 *>(mirror);
    int *cnt = reinterpret_cast<int *>(rects + (size_t)ctx->max_batch * kMaxIgnore);
    int any = 0;
    for (int i = 0; i < n; i++) {
        int kept = 0;
        for (int j = 0; j < n_ignore[i]; j++) {
            const tw_rect &r = ignore[i][j];
            const long long x0 = std::max<long long>(r.x, 0), y0 = std::max<long long>(r.y, 0);
            const long long x1 = std::min<long long>((long long)r.x + r.width, W), y1 = std::min<long long>((long long)r.y + r.height, H);
            if (x0 < x1 && y0 < y1) rects[(size_t)i * kMaxIgnore + kept++] = make_int4((int)x0, (int)y0, (int)x1, (int)y1);
        }
        cnt[i] = kept;
        any |= kept > 0;
    }
    return any;
}

// The plan's ignore-mask plane and flags (Plan::mask, mask_has), allocated on its first masked batch and freed with it.
bool ensure_mask_plane(tw_ctx *ctx)
{
    Plan &pl = ctx->plan;
    if (pl.mask) return true;
    return dev_alloc(ctx, &pl.mask, (size_t)pl.batch * pl.H * pl.spitch) && dev_alloc(ctx, &pl.mask_has, (size_t)pl.batch);
}

IgnoreMasks ignore_masks(const Plan &pl) { return IgnoreMasks{pl.mask, pl.mask_has, pl.W, pl.H, pl.spitch}; }

// Pipe staging buffer behind the images and the region lists (tw_pipe_submit_mask): [max_batch] int flags, then the planes.
size_t mask_flag_bytes(int max_batch) { return ((size_t)max_batch * sizeof(int) + 255) & ~(size_t)255; }

// Relaxed arithmetic (fmaf in the Gaussian window taps, mixed double / float horizontal pass of the polynomial
// expansion) is used only for the option family it was validated on against the faithful oracle and cv2
// (tools/relax_study.py, tests/test_gpu_parity.py): Gaussian window of the reference's default size or larger and
// polyN = 7.  Smaller windows and the box window are measured to be chaotic under ANY reordering (SURVEY App. B) and
// always run the faithful kernels.
bool relaxed_in_effect(const tw_ctx *ctx, const tw_flow_param &p)
{
    return ctx->opt.arith == 1 && (p.flags & 256) && p.winSize >= 30 && p.polyN == 7;
}

// Whether a run with this span ends in the sparse last iteration (K5s): then no dense flow field exists afterwards.
bool sparse_in_effect(const tw_ctx *ctx, int span)
{
    const Plan &pl = ctx->plan;
    const tw_flow_param &p = pl.p;
    if (!(span > 0 && ctx->opt.sparse_last && (p.flags & 256) && p.pyrIterations > 0 && (pl.win.m == 15 || pl.win.m == 7))) return false;
    IterArgs ia{};
    ia.span = span;
    return gauss_last_sparse_ok(ia, pl.win);
}

// The launch sequence for n pairs already resident in plan.src.  SURVEY App. A.1 / A.7.  ignore: the batch has ignore regions
// (in ctx->d_ignore): the target is painted first and the sample kernel leaves the points inside the regions out.  mask: the batch
// has ignore masks (in plan.mask / mask_has): the same for the pixels and points under the masks.
bool enqueue(tw_ctx *ctx, int n, double threshold, int span, bool ignore, bool mask)
{
    Plan &pl = ctx->plan;
    const tw_flow_param &p = pl.p;
    const bool relaxed = relaxed_in_effect(ctx, p);
    const int W = pl.W, H = pl.H;
    const double P0 = (double)W * H;
    const size_t ns = pl.scales.size();
    // sampling is fused into the last Gaussian iteration of the finest scale when that kernel runs (radius 15 / 7)
    const bool fused_count = span > 0 && (p.flags & 256) && p.pyrIterations > 0 && (pl.win.m == 15 || pl.win.m == 7);
    if (mask) // expected pixels over the target under the masks, before anything reads the target
        LAUNCH(F_MASK, 0.0, launch_mask_paint(ctx->stream, pl.src, ignore_masks(pl), n));
    if (ignore) // expected pixels over the target inside the regions, before anything reads the target
        LAUNCH(F_PAINT, 0.0, launch_ignore_paint(ctx->stream, pl.src, H, pl.spitch, ignore_regions(ctx->d_ignore, ctx->max_batch), n));
    if (fused_count) {
        cudaError_t e = cudaMemsetAsync(ctx->d_counts, 0, sizeof(int) * n, ctx->stream);
        if (e != cudaSuccess) { set_err(ctx, "memset counts", e); return false; }
    }
    const bool fused_levels = pl.fused_levels && !ctx->opt.level_generic && !ctx->opt.level_unfused;
    const size_t fbase = ns >= 4 ? ns - 4 : 0; // first scale produced by the fused kernel
    if (fused_levels) {
        float *dst[4]; LevelDims dd[4];
        double bytes = 0;
        for (int i = 0; i < 4; i++) {
            dst[i] = pl.scales[fbase + i].I; dd[i] = pl.scales[fbase + i].d;
            bytes += n * 8.0 * dd[i].w * dd[i].h;
        }
        bytes += n * 2 * P0; // what this kernel moves: the u8 source ONCE for all four levels (SURVEY 8(d) charges it once per level)
        LAUNCH(F_LEVEL, bytes, launch_level_fused(ctx->stream, pl.src, W, H, pl.spitch, dst, dd, pl.scales[fbase].host_taps.data(),
                                                   pl.scales[fbase + 1].host_taps.data(), pl.scales[fbase + 2].host_taps.data(),
                                                   pl.scales[fbase + 3].host_taps.data(), 2 * n));
    }
    for (size_t si = 0; si < ns; si++) {
        Scale &s = pl.scales[si];
        const double Pl = (double)s.d.w * s.d.h;
        LevelImageArgs la{};
        la.src = pl.src; la.W = W; la.H = H; la.spitch = pl.spitch; la.dst = s.I; la.d = s.d;
        la.xi = s.img_xi; la.xf = s.img_xf; la.yi = s.img_yi; la.yf = s.img_yf; la.taps = s.taps; la.ksize = s.ksize;
        la.nimg = 2 * n; la.tile_w = s.tile_w; la.tile_h = s.tile_h; la.smem_w = s.smem_w; la.smem_h = s.smem_h;
        la.identity = s.identity;
        la.small = (s.ksize / 2 + 2 >= std::min(W, H));
        // I planes of a batch are laid out [B][2]: the u8 source is [B][2] too, so image index = blockIdx.z.
        if (!fused_levels || si < fbase) {
            LaunchScope ls_(ctx, F_LEVEL, n * (2 * P0 + 8 * Pl));
            cudaError_t e_ = ctx->opt.level_generic ? cudaErrorNotSupported : launch_level_image_fast(ctx->stream, la, s.host_taps.data(), s.int_scale);
            if (e_ == cudaErrorNotSupported && !ctx->opt.level_generic && pl.T && level_image_big_ok(la)) e_ = launch_level_image_big(ctx->stream, la, pl.T);
            if (e_ == cudaErrorNotSupported) e_ = launch_level_image(ctx->stream, la);
            if (e_ != cudaSuccess) { set_err(ctx, "launch_level_image", e_); return false; }
        }
        LAUNCH(F_POLY, n * 48 * Pl, launch_polyexp(ctx->stream, s.I, s.R, s.d, 2 * n, pl.poly, relaxed ? 1 : 0, &s.imap));

        FirstUpdateArgs fa{};
        if (si > 0) {
            const Scale &cs = pl.scales[si - 1];
            fa.coarse = cs.flow; fa.cd = cs.d; fa.xi = s.up_xi; fa.xf = s.up_xf; fa.yi = s.up_yi; fa.yf = s.up_yf;
        }
        fa.inv_scale = (float)(1. / p.pyrScale);
        fa.R = s.R; fa.d = s.d; fa.batch = n;
        fa.M = p.pyrIterations > 0 ? s.M0 : nullptr;
        fa.flow_out = p.pyrIterations > 0 ? nullptr : s.flow;
        double cbytes = si > 0 ? 8.0 * pl.scales[si - 1].d.w * pl.scales[si - 1].d.h : 0.0;
        LAUNCH(F_FIRST, n * (cbytes + 60 * Pl), launch_first_update(ctx->stream, fa));

        float *Min = s.M0, *Mout = s.M1;
        for (int it = 0; it < p.pyrIterations; it++) {
            IterArgs ia{};
            ia.Min = Min; ia.Mout = Mout; ia.R = s.R; ia.flow = s.flow; ia.d = s.d; ia.batch = n;
            ia.last = (it == p.pyrIterations - 1);
            if (fused_count && ia.last && si + 1 == ns) { ia.span = span; ia.thr2 = threshold * threshold; ia.counts = ctx->d_counts; }
            ia.fma = relaxed ? 2 : 0;
            double bytes = n * (ia.last ? 28 : 80) * Pl;
            if (ia.span > 0 && sparse_in_effect(ctx, span)) {
                // classification only: blur + solve at the sampled positions (one pass over M, no flow plane written)
                LAUNCH(F_GLAST, n * 20.0 * Pl, launch_gauss_last_sparse(ctx->stream, ia, pl.win));
            } else if ((p.flags & 256) && ctx->opt.window_tiles == 0 && gauss_strip_ok(ia, pl.win) &&
                       s.maps[Min == s.M1 ? 1 : 0].valid) {
                LAUNCH(ia.last ? F_GLAST : F_GITER, bytes, launch_gauss_strip(ctx->stream, ia, pl.win, s.maps[Min == s.M1 ? 1 : 0]));
            } else if (p.flags & 256) {
                LAUNCH(ia.last ? F_GLAST : F_GITER, bytes, launch_gauss_iter(ctx->stream, ia, pl.win));
            } else if (!ctx->opt.box_unfused && box_fused_ok(s.d, p.winSize / 2)) {
                // fused box iteration: band checkpoints of the vertical running sums, then blur + solve + update in one kernel
                LAUNCH(F_BVSUM, n * 20.0 * Pl, launch_box_ckpt(ctx->stream, Min, pl.V, s.d, n, p.winSize / 2));
                LAUNCH(ia.last ? F_BLAST : F_BITER, n * (ia.last ? 28.0 : 80.0) * Pl - n * 20.0 * Pl,
                       launch_box_band(ctx->stream, Min, pl.V, s.R, Mout, s.flow, s.d, n, p.winSize / 2, p.winSize, ia.last));
            } else {
                LAUNCH(F_BVSUM, 0.0, launch_box_vsum(ctx->stream, Min, pl.V, s.d, n, p.winSize / 2));
                LAUNCH(ia.last ? F_BLAST : F_BITER, bytes, launch_box_hscan(ctx->stream, pl.V, s.flow, s.d, n, p.winSize / 2, p.winSize));
                if (!ia.last) {
                    FirstUpdateArgs ua{};
                    ua.flow_in = s.flow; ua.R = s.R; ua.M = Mout; ua.d = s.d; ua.batch = n; ua.inv_scale = 1.f;
                    LAUNCH(F_BUPD, 0.0, launch_first_update(ctx->stream, ua));
                }
            }
            if (!ia.last) std::swap(Min, Mout);
        }
    }
    if (span > 0) {
        Scale &f = pl.scales.back();
        int nsx = (f.d.w + span - 1) / span, nsy = (f.d.h + span - 1) / span;
        if (!ensure_results(ctx, nsx * nsy)) return false;
        SampleArgs sa{};
        sa.flow = f.flow; sa.d = f.d; sa.batch = n; sa.span = span; sa.thr2 = threshold * threshold;
        sa.counts = ctx->d_counts; sa.vectors = ctx->d_vectors; sa.cap = ctx->dev_cap; sa.counted = fused_count ? 1 : 0;
        if (mask)
            LAUNCH(F_SAMPLE, 0.0, launch_sample_mask(ctx->stream, sa, ignore ? ignore_regions(ctx->d_ignore, ctx->max_batch) : IgnoreRegions{},
                                                     ignore_masks(pl)));
        else if (ignore) LAUNCH(F_SAMPLE, 0.0, launch_sample_ignore(ctx->stream, sa, ignore_regions(ctx->d_ignore, ctx->max_batch)));
        else LAUNCH(F_SAMPLE, 0.0, launch_sample(ctx->stream, sa));
        if (ctx->opt.change_regions) {
            if (!ensure_region_buffers(ctx)) return false;
            ChangeRegionArgs ca{};
            ca.vectors = ctx->d_vectors; ca.counts = ctx->d_counts; ca.cap = ctx->dev_cap; ca.w = f.d.w; ca.h = f.d.h; ca.span = span;
            ca.scratch = ctx->d_reg_scratch; ca.n_regions = ctx->d_nreg; ca.regions = ctx->d_regions; ca.batch = n;
            LAUNCH(F_REGIONS, 0.0, launch_change_regions(ctx->stream, ca));
        }
        if (ctx->opt.intensity) {
            if (!ensure_intensity_buffers(ctx)) return false;
            IntensityArgs ta{};
            ta.src = pl.src; ta.spitch = pl.spitch; ta.flow = f.flow; ta.d = f.d; ta.span = span; ta.t = ctx->opt.intensity;
            if (ignore) ta.g = ignore_regions(ctx->d_ignore, ctx->max_batch);
            if (mask) ta.k = ignore_masks(pl);
            ta.sum = reinterpret_cast<unsigned long long *>(ctx->d_int_acc);
            ta.cnt = reinterpret_cast<unsigned *>(ta.sum + (size_t)ctx->max_batch * ctx->int_cap);
            ta.chunk_counts = reinterpret_cast<int *>(ta.cnt + (size_t)ctx->max_batch * ctx->int_cap);
            ta.cell_cap = ctx->int_cap; ta.max_chunks = ctx->int_chunks; ta.n_cells = ctx->d_ncell; ta.cells = ctx->d_cells; ta.batch = n;
            ctx->int_dirty = true;
            // what the sums read: E and T once (the 3 x 3 target taps are staged in shared memory)
            LAUNCH(F_INTENSITY, n * 2.0 * P0, launch_intensity_sum(ctx->stream, ta));
            LAUNCH(F_INTENSITY, 0.0, launch_intensity_count(ctx->stream, ta));
            LAUNCH(F_INTENSITY, 0.0, launch_intensity_compact(ctx->stream, ta));
            ctx->int_dirty = false;
        }
    }
    return true;
}

// enqueue() directly, or -- from the second run with an unchanged (plan, n, threshold, span, options) key on -- as ONE
// cudaGraphLaunch of the captured sequence (the step is ~22 short launches; at the coarse scales the kernels are
// shorter than their launch gaps).  The first run of a key is always eager: it configures the per-device kernel
// attributes and sizes the result buffers outside any capture.  Profiling (per-family events) runs eagerly.
bool run_sequence(tw_ctx *ctx, int n, double threshold, int span, bool ignore, bool mask)
{
    if (!ctx->opt_graph || ctx->profiling) return enqueue(ctx, n, threshold, span, ignore, mask);
    Plan &pl = ctx->plan;
    GraphKey key;
    key.n = n; key.thr = threshold; key.span = span; key.opt = ctx->opt; key.ignore = ignore; key.mask = mask;
    key.vectors = ctx->d_vectors; key.dev_cap = ctx->dev_cap; // the captured sample kernel bakes both in
    if (pl.graph_exec && key == pl.graph_key) {
        cudaError_t e = cudaGraphLaunch(pl.graph_exec, ctx->stream);
        if (e != cudaSuccess) { set_err(ctx, "cudaGraphLaunch", e); return false; }
        ctx->launches += pl.graph_launches;
        return true;
    }
    if (!(key == pl.seen_key)) { // first run of this key: eager
        if (!enqueue(ctx, n, threshold, span, ignore, mask)) return false;
        pl.seen_key = key;
        pl.seen_key.vectors = ctx->d_vectors; pl.seen_key.dev_cap = ctx->dev_cap; // enqueue may have (re)allocated the result buffer
        return true;
    }
    // second run: capture, instantiate, launch
    if (pl.graph_exec) { cudaGraphExecDestroy(pl.graph_exec); pl.graph_exec = nullptr; }
    const long long before = ctx->launches;
    cudaGraph_t graph = nullptr;
    cudaError_t e = cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) { // capture unavailable: stay eager
        cudaGetLastError();
        ctx->opt_graph = 0;
        return enqueue(ctx, n, threshold, span, ignore, mask);
    }
    const bool ok = enqueue(ctx, n, threshold, span, ignore, mask);
    e = cudaStreamEndCapture(ctx->stream, &graph);
    const long long captured = ctx->launches - before;
    ctx->launches = before;
    if (!ok || e != cudaSuccess || !graph) {
        if (graph) cudaGraphDestroy(graph);
        cudaGetLastError();
        ctx->opt_graph = 0; // never retry on this context; the eager path is the same launch sequence
        if (!ok) return false;
        return enqueue(ctx, n, threshold, span, ignore, mask);
    }
    e = cudaGraphInstantiate(&pl.graph_exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pl.graph_exec = nullptr;
        ctx->opt_graph = 0;
        return enqueue(ctx, n, threshold, span, ignore, mask);
    }
    pl.graph_key = key;
    pl.graph_launches = captured;
    e = cudaGraphLaunch(pl.graph_exec, ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "cudaGraphLaunch", e); return false; }
    ctx->launches += captured;
    return true;
}

void fill_error(tw_result *r, int code, const char *msg)
{
    memset(r, 0, sizeof *r);
    r->code = code;
    r->status = TW_STATUS_ERROR;
    snprintf(r->reason, sizeof r->reason, "%s", msg);
}

std::atomic<int> g_default_arith{-1}; // -1: not decided yet (TW_ARITHMETIC or 1)

int default_arith()
{
    int v = g_default_arith.load();
    if (v >= 0) return v;
    const char *env = getenv("TW_ARITHMETIC");
    v = (env && (!strcmp(env, "faithful") || !strcmp(env, "0"))) ? 0 : 1;
    g_default_arith.store(v);
    return v;
}

} // namespace

extern "C" {

void tw_default_param(tw_flow_param *p)
{
    p->pyrScale = 0.5; p->pyrLevels = 3; p->winSize = 30; p->pyrIterations = 3; p->polyN = 7; p->polySigma = 1.5; p->flags = 256;
}

const char *tw_version(void) { return "tidalwave_b200 0.1 sm_100a"; }

int tw_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

tw_ctx *tw_create(int device, int max_w, int max_h, int max_batch, char *err, int errlen)
{
    auto fail = [&](const std::string &m) -> tw_ctx * {
        if (err && errlen > 0) snprintf(err, errlen, "%s", m.c_str());
        return nullptr;
    };
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail("bad device index");
    if ((e = cudaSetDevice(device)) != cudaSuccess) return fail(cudaGetErrorString(e));
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail(cudaGetErrorString(e));
    if (prop.major != 10) {
        char b[160];
        snprintf(b, sizeof b, "device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
        return fail(b);
    }
    tw_ctx *ctx = new tw_ctx();
    ctx->device = device; ctx->max_w = max_w; ctx->max_h = max_h; ctx->max_batch = max_batch < 1 ? 1 : max_batch;
    ctx->opt.arith = default_arith();
    if (const char *g = getenv("TW_GRAPH")) ctx->opt_graph = atoi(g) ? 1 : 0; // TW_GRAPH=0: eager launches (profilers)
    if (const char *g = getenv("TW_PLAN_CACHE")) ctx->plan_cache_max = atoi(g) < 0 ? 0 : atoi(g);
    if (const char *g = getenv("TW_POLY_TMA")) ctx->opt_poly_no_tma = atoi(g) ? 0 : 1;
    if (const char *g = getenv("TW_WINDOW")) ctx->opt.window_tiles = !strcmp(g, "strip") ? 0 : 1; // TW_WINDOW=strip|tiles
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) { delete ctx; return fail(cudaGetErrorString(e)); }
    cudaEventCreate(&ctx->ev_t0); cudaEventCreate(&ctx->ev_t1); cudaEventCreate(&ctx->ev_r0); cudaEventCreate(&ctx->ev_r1);
    if ((e = cudaMalloc(&ctx->d_counts, sizeof(int) * ctx->max_batch)) != cudaSuccess ||
        (e = cudaMallocHost(&ctx->h_counts, sizeof(int) * ctx->max_batch)) != cudaSuccess ||
        (e = cudaMalloc(&ctx->d_ignore, ignore_bytes(ctx->max_batch))) != cudaSuccess ||
        (e = cudaMallocHost(&ctx->h_ignore, ignore_bytes(ctx->max_batch))) != cudaSuccess ||
        (e = cudaMallocHost(&ctx->h_mask_has, sizeof(int) * ctx->max_batch)) != cudaSuccess) {
        std::string m = cudaGetErrorString(e);
        tw_destroy(ctx);
        return fail(m);
    }
    return ctx;
}

void tw_destroy(tw_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    drain_profile(ctx);
    free_plan(ctx->plan);
    flush_plan_cache(ctx);
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    if (ctx->d_counts) cudaFree(ctx->d_counts);
    if (ctx->h_counts) cudaFreeHost(ctx->h_counts);
    if (ctx->d_ignore) cudaFree(ctx->d_ignore);
    if (ctx->h_ignore) cudaFreeHost(ctx->h_ignore);
    if (ctx->h_mask_has) cudaFreeHost(ctx->h_mask_has);
    if (ctx->d_vectors) cudaFree(ctx->d_vectors);
    if (ctx->d_reg_scratch) cudaFree(ctx->d_reg_scratch);
    if (ctx->d_nreg) cudaFree(ctx->d_nreg);
    if (ctx->h_nreg) cudaFreeHost(ctx->h_nreg);
    if (ctx->d_regions) cudaFree(ctx->d_regions);
    if (ctx->h_regions) cudaFreeHost(ctx->h_regions);
    if (ctx->d_int_acc) cudaFree(ctx->d_int_acc);
    if (ctx->d_ncell) cudaFree(ctx->d_ncell);
    if (ctx->h_ncell) cudaFreeHost(ctx->h_ncell);
    if (ctx->d_cells) cudaFree(ctx->d_cells);
    if (ctx->h_cells) cudaFreeHost(ctx->h_cells);
    if (ctx->flush_buf) cudaFree(ctx->flush_buf);
    if (ctx->rs_buf) cudaFree(ctx->rs_buf);
    {
        tw_ctx::Pipe &pp = ctx->pipe;
        if (pp.copy) { cudaStreamSynchronize(pp.copy); cudaStreamDestroy(pp.copy); }
        if (pp.fetch) { cudaStreamSynchronize(pp.fetch); cudaStreamDestroy(pp.fetch); }
        if (pp.stage) cudaFree(pp.stage);
        if (pp.ev_up) cudaEventDestroy(pp.ev_up);
        if (pp.ev_stage_free) cudaEventDestroy(pp.ev_stage_free);
        for (auto &s : pp.slot) {
            if (s.done) cudaEventDestroy(s.done);
            if (s.r0) cudaEventDestroy(s.r0);
            if (s.r1) cudaEventDestroy(s.r1);
            if (s.d_counts) cudaFree(s.d_counts);
            if (s.h_counts) cudaFreeHost(s.h_counts);
            if (s.h_ignore) cudaFreeHost(s.h_ignore);
            if (s.h_mask_has) cudaFreeHost(s.h_mask_has);
            if (s.d_vec) cudaFree(s.d_vec);
            if (s.d_nreg) cudaFree(s.d_nreg);
            if (s.h_nreg) cudaFreeHost(s.h_nreg);
            if (s.d_regions) cudaFree(s.d_regions);
            if (s.d_ncell) cudaFree(s.d_ncell);
            if (s.h_ncell) cudaFreeHost(s.h_ncell);
            if (s.d_cells) cudaFree(s.d_cells);
        }
    }
    if (ctx->ev_t0) cudaEventDestroy(ctx->ev_t0);
    if (ctx->ev_t1) cudaEventDestroy(ctx->ev_t1);
    if (ctx->ev_r0) cudaEventDestroy(ctx->ev_r0);
    if (ctx->ev_r1) cudaEventDestroy(ctx->ev_r1);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char *tw_last_error(tw_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

void *tw_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes) != cudaSuccess) return nullptr;
    return p;
}
void tw_host_free(void *p) { if (p) cudaFreeHost(p); }

int tw_sync(tw_ctx *ctx)
{
    if (!ctx) return TW_BAD_PARAMETER;
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "sync", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

// Upload of n pairs is shared by the batch entry points.  The plan must exist for (w, h): built lazily here
// with the last parameters (or defaults) and rebuilt by tw_batch_run if the parameters differ.
static int upload_impl(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h,
                       int stride, const tw_flow_param *param)
{
    if (!ctx) return TW_BAD_PARAMETER;
    if (n < 1 || n > ctx->max_batch || w < 1 || h < 1 || stride < w) { ctx->err = "bad batch/size"; return TW_BAD_PARAMETER; }
    if ((ctx->max_w > 0 && w > ctx->max_w) || (ctx->max_h > 0 && h > ctx->max_h)) { ctx->err = "image larger than the context's max_w x max_h"; return TW_BAD_PARAMETER; }
    cudaSetDevice(ctx->device);
    tw_flow_param p;
    if (param) p = *param; else if (ctx->plan.valid) p = ctx->plan.p; else tw_default_param(&p);
    if (validate_param(&p) != TW_OK) { ctx->err = "bad optical-flow parameter"; return TW_BAD_PARAMETER; }
    if (!build_plan(ctx, w, h, p)) return TW_CUDA_ERROR;
    Plan &pl = ctx->plan;
    for (int i = 0; i < n; i++) {
        if (!expect[i] || !target[i]) { ctx->err = "null image"; return TW_BAD_IMAGE_FORMAT; }
        uint8_t *d = pl.src + (size_t)i * 2 * h * pl.spitch;
        cudaError_t e = cudaMemcpy2DAsync(d, pl.spitch, expect[i], stride, w, h, cudaMemcpyHostToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(d + (size_t)h * pl.spitch, pl.spitch, target[i], stride, w, h, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) { set_err(ctx, "H2D", e); return TW_CUDA_ERROR; }
    }
    return TW_OK;
}

// Uploads a (tw x th) target and resizes it on the device into the target slot of pair 0 (plan already built).
static bool upload_resized_target(tw_ctx *ctx, const uint8_t *target, int tw_, int th_, int ew, int eh)
{
    Plan &pl = ctx->plan;
    const int tp = (tw_ + 15) & ~15;
    size_t need = (size_t)tp * th_ + sizeof(int) * (ew + eh) + sizeof(short) * 2 * (ew + eh) + 1024;
    if (ctx->rs_cap < need) {
        if (ctx->rs_buf) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->rs_buf); ctx->rs_buf = nullptr; }
        cudaError_t e = cudaMalloc(&ctx->rs_buf, need);
        if (e != cudaSuccess) return set_err(ctx, "cudaMalloc", e);
        ctx->rs_cap = need;
    }
    std::vector<int> xi, yi; std::vector<short> xa, ya;
    resize_coeffs_u8(tw_, ew, xi, xa, true);
    resize_coeffs_u8(th_, eh, yi, ya, false);
    uint8_t *base = reinterpret_cast<uint8_t *>(ctx->rs_buf);
    uint8_t *d_img = base;
    size_t off = ((size_t)tp * th_ + 255) & ~(size_t)255;
    int *d_xi = reinterpret_cast<int *>(base + off); off += sizeof(int) * ew;
    int *d_yi = reinterpret_cast<int *>(base + off); off += sizeof(int) * eh;
    short *d_xa = reinterpret_cast<short *>(base + off); off += sizeof(short) * 2 * ew;
    short *d_ya = reinterpret_cast<short *>(base + off);
    CK(cudaMemcpy2DAsync(d_img, tp, target, tw_, tw_, th_, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_xi, xi.data(), sizeof(int) * ew, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_yi, yi.data(), sizeof(int) * eh, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_xa, xa.data(), sizeof(short) * 2 * ew, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_ya, ya.data(), sizeof(short) * 2 * eh, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream)); // the tables are host temporaries
    ResizeU8Args ra{};
    ra.src = d_img; ra.W = tw_; ra.H = th_; ra.spitch = tp;
    ra.dst = pl.src + (size_t)eh * pl.spitch; ra.w = ew; ra.h = eh; ra.dpitch = pl.spitch;
    ra.xi = d_xi; ra.yi = d_yi; ra.xa = d_xa; ra.ya = d_ya;
    ctx->launches++;
    CK(launch_resize_u8(ctx->stream, ra));
    return true;
}

// Checks and clips the region lists of n pairs of w x h frames and copies them into the region buffer on the context's stream (the
// synchronous entry points: the page-locked mirror is free again once the call has fetched its results).  *any: some pair keeps a
// region.  Returns a tw_error_code.
static int upload_ignore(tw_ctx *ctx, int n, const tw_rect *const *ignore, const int *n_ignore, int w, int h, bool *any)
{
    const int r = pack_ignore(ctx, n, ignore, n_ignore, w, h, ctx->h_ignore);
    if (r < 0) return TW_BAD_PARAMETER;
    *any = r > 0;
    if (!*any) return TW_OK;
    cudaError_t e = cudaMemcpyAsync(ctx->d_ignore, ctx->h_ignore, ignore_bytes(ctx->max_batch), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "regions H2D", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

// Copies the ignore masks of n pairs of w x h frames (mask == NULL: none; mask[i] == NULL: pair i has none) into the plan's mask
// plane and flags on the context's stream (the synchronous entry points; plan already built).  *any: some pair has a mask.
static int upload_mask(tw_ctx *ctx, int n, const uint8_t *const *mask, int w, int h, int stride, bool *any)
{
    *any = false;
    if (!mask) return TW_OK;
    for (int i = 0; i < n; i++) *any |= (ctx->h_mask_has[i] = mask[i] ? 1 : 0) != 0;
    if (!*any) return TW_OK;
    if (!ensure_mask_plane(ctx)) return TW_CUDA_ERROR;
    Plan &pl = ctx->plan;
    cudaError_t e = cudaMemcpyAsync(pl.mask_has, ctx->h_mask_has, sizeof(int) * n, cudaMemcpyHostToDevice, ctx->stream);
    for (int i = 0; i < n && e == cudaSuccess; i++)
        if (mask[i])
            e = cudaMemcpy2DAsync(pl.mask + (size_t)i * h * pl.spitch, pl.spitch, mask[i], stride, w, h, cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "mask H2D", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_batch_upload(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride)
{
    return upload_impl(ctx, n, expect, target, w, h, stride, nullptr);
}

// tw_batch_run; ignore / mask: run the ignore / mask form with the regions / masks already in place
static int run_batch(tw_ctx *ctx, int n, int w, int h, const tw_flow_param *param, double threshold, int span, bool ignore, bool mask)
{
    if (!ctx) return TW_BAD_PARAMETER;
    if (n < 1 || n > ctx->max_batch) { ctx->err = "bad batch"; return TW_BAD_PARAMETER; }
    if (validate_param(param) != TW_OK) { ctx->err = "bad optical-flow parameter"; return TW_BAD_PARAMETER; }
    if (span < 0) { ctx->err = "bad span"; return TW_BAD_PARAMETER; }
    cudaSetDevice(ctx->device);
    Plan &pl = ctx->plan;
    if (!plan_fits(ctx, pl, w, h, pl.p)) { // images of this size resident (under whichever parameters)
        ctx->err = "tw_batch_run: no uploaded images of this size";
        return TW_BAD_PARAMETER;
    }
    if (!same_param(pl.p, *param)) {
        // parameters changed but the images are already resident: rebuild the plan around a copy of src
        uint8_t *tmp = nullptr;
        size_t bytes = (size_t)pl.batch * 2 * h * pl.spitch;
        cudaError_t e = cudaMalloc(&tmp, bytes);
        if (e != cudaSuccess) { set_err(ctx, "cudaMalloc", e); return TW_CUDA_ERROR; }
        cudaMemcpyAsync(tmp, pl.src, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
        bool ok = build_plan(ctx, w, h, *param);
        if (ok) cudaMemcpyAsync(ctx->plan.src, tmp, bytes, cudaMemcpyDeviceToDevice, ctx->stream);
        cudaStreamSynchronize(ctx->stream);
        cudaFree(tmp);
        if (!ok) return TW_CUDA_ERROR;
    }
    cudaEventRecord(ctx->ev_r0, ctx->stream);
    if (!run_sequence(ctx, n, threshold, span, ignore, mask)) return TW_CUDA_ERROR;
    cudaEventRecord(ctx->ev_r1, ctx->stream);
    ctx->last_n = n; ctx->last_w = w; ctx->last_h = h; ctx->ran = true;
    ctx->last_span = span; ctx->last_regions = ctx->opt.change_regions != 0; ctx->last_intensity = ctx->opt.intensity != 0;
    ctx->last_sparse = sparse_in_effect(ctx, span);
    return TW_OK;
}

int tw_batch_run(tw_ctx *ctx, int n, int w, int h, const tw_flow_param *param, double threshold, int span)
{
    return run_batch(ctx, n, w, h, param, threshold, span, false, false);
}

int tw_batch_fetch(tw_ctx *ctx, int n, tw_vector *out, int cap, tw_result *res)
{
    if (!ctx || !res) return TW_BAD_PARAMETER;
    if (!ctx->ran || n != ctx->last_n) { ctx->err = "tw_batch_fetch: nothing to fetch"; return TW_BAD_PARAMETER; }
    cudaSetDevice(ctx->device);
    answer_regions(ctx, n, ctx->last_regions);
    answer_cells(ctx, n, ctx->last_intensity);
    const bool labelled = ctx->last_regions && ctx->last_span > 0;
    const bool celled = ctx->last_intensity && ctx->last_span > 0 && ctx->cell_pairs >= 0;
    cudaError_t e = cudaMemcpyAsync(ctx->h_counts, ctx->d_counts, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && labelled) e = cudaMemcpyAsync(ctx->h_nreg, ctx->d_nreg, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && celled) e = cudaMemcpyAsync(ctx->h_ncell, ctx->d_ncell, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        answer_regions(ctx, n, ctx->last_regions);
        answer_cells(ctx, n, ctx->last_intensity);
        set_err(ctx, "fetch", e);
        for (int i = 0; i < n; i++) fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str());
        return TW_CUDA_ERROR;
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, ctx->ev_r0, ctx->ev_r1);
    for (int i = 0; i < n; i++) {
        int cnt = ctx->h_counts[i];
        const int ncell = celled ? ctx->h_ncell[i] : 0;
        memset(&res[i], 0, sizeof(tw_result));
        res[i].code = TW_OK;
        res[i].status = cnt == 0 && ncell == 0 ? TW_STATUS_OK : TW_STATUS_SUSPICIOUS;
        res[i].n_vectors = cnt;
        res[i].width = ctx->last_w; res[i].height = ctx->last_h;
        res[i].time = ms * 1e-3f / n;
        int ncopy = std::min(std::min(cnt, cap), ctx->dev_cap);
        if (ncopy > 0 && out) {
            e = cudaMemcpyAsync(out + (size_t)i * cap, (const tw_vector *)ctx->d_vectors + (size_t)i * ctx->dev_cap,
                                sizeof(tw_vector) * ncopy, cudaMemcpyDeviceToHost, ctx->stream);
            if (e != cudaSuccess) { set_err(ctx, "fetch vectors", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
        }
        const int nreg = labelled ? std::min(ctx->h_nreg[i], kMaxChangeRegions) : 0;
        if (nreg > 0 && res[i].code == TW_OK) {
            e = cudaMemcpyAsync(ctx->h_regions + (size_t)i * kMaxChangeRegions, ctx->d_regions + (size_t)i * kMaxChangeRegions,
                                sizeof(tw_change_region) * nreg, cudaMemcpyDeviceToHost, ctx->stream);
            if (e != cudaSuccess) { set_err(ctx, "fetch regions", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
        }
        const int kcell = std::min(ncell, kMaxIntensityCells);
        if (kcell > 0 && res[i].code == TW_OK) {
            e = cudaMemcpyAsync(ctx->h_cells + (size_t)i * kMaxIntensityCells, ctx->d_cells + (size_t)i * kMaxIntensityCells,
                                sizeof(tw_intensity_cell) * kcell, cudaMemcpyDeviceToHost, ctx->stream);
            if (e != cudaSuccess) { set_err(ctx, "fetch intensity cells", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
        }
        if (res[i].code != TW_OK && ctx->reg_pairs > 0) ctx->h_nreg[i] = 0;
        if (res[i].code != TW_OK && ctx->cell_pairs > 0) ctx->h_ncell[i] = 0;
    }
    e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "fetch sync", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_batch_flow(tw_ctx *ctx, int pair, float *flowx, float *flowy)
{
    if (!ctx || !ctx->ran || pair < 0 || pair >= ctx->last_n) return TW_BAD_PARAMETER;
    if (ctx->last_sparse) { ctx->err = "no dense flow: the last run used \"sparse_last\" (classification only)"; return TW_BAD_PARAMETER; }
    cudaSetDevice(ctx->device);
    const Scale &f = ctx->plan.scales.back();
    const float *base = f.flow + (size_t)pair * 2 * f.d.plane;
    cudaError_t e = cudaSuccess;
    if (flowx) e = cudaMemcpy2DAsync(flowx, sizeof(float) * f.d.w, base, sizeof(float) * f.d.pitch, sizeof(float) * f.d.w, f.d.h,
                                     cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && flowy)
        e = cudaMemcpy2DAsync(flowy, sizeof(float) * f.d.w, base + f.d.plane, sizeof(float) * f.d.pitch, sizeof(float) * f.d.w,
                              f.d.h, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "flow D2H", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_flow(tw_ctx *ctx, const uint8_t *expect, const uint8_t *target, int w, int h, int stride, const tw_flow_param *param,
            float *flowx, float *flowy, float *seconds)
{
    if (!ctx) return TW_BAD_PARAMETER;
    if (!expect || !target) { ctx->err = "null image"; return TW_BAD_IMAGE_FORMAT; }
    int rc = upload_impl(ctx, 1, &expect, &target, w, h, stride, param);
    if (rc != TW_OK) return rc;
    rc = tw_batch_run(ctx, 1, w, h, param, 0.0, 0);
    if (rc != TW_OK) return rc;
    rc = tw_batch_flow(ctx, 0, flowx, flowy);
    if (rc != TW_OK) return rc;
    if (seconds) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev_r0, ctx->ev_r1);
        *seconds = ms * 1e-3f;
    }
    return TW_OK;
}

int tw_compare_batch_mask(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                          const tw_flow_param *param, double threshold, int span, const tw_rect *const *ignore, const int *n_ignore,
                          const uint8_t *const *mask, tw_vector *out, int cap, tw_result *res)
{
    if (!ctx || !res) return TW_BAD_PARAMETER;
    answer_regions(ctx, n, ctx->opt.change_regions != 0); // what an ERROR answer leaves: 0 regions per pair
    answer_cells(ctx, n, ctx->opt.intensity != 0);        // and 0 intensity cells
    auto fail_all = [&](int code, const char *msg) {
        for (int i = 0; i < n; i++) fill_error(&res[i], code, msg);
        return code;
    };
    if (span < 1) return fail_all(TW_BAD_PARAMETER, "span must be >= 1");
    if (validate_param(param) != TW_OK) return fail_all(TW_BAD_PARAMETER, "bad optical-flow parameter");
    int rc = upload_impl(ctx, n, expect, target, w, h, stride, param);
    if (rc != TW_OK) return fail_all(rc, ctx->err.c_str());
    bool any = false, any_mask = false;
    rc = upload_ignore(ctx, n, ignore, n_ignore, w, h, &any);
    if (rc == TW_OK) rc = upload_mask(ctx, n, mask, w, h, stride, &any_mask);
    if (rc != TW_OK) return fail_all(rc, ctx->err.c_str());
    rc = run_batch(ctx, n, w, h, param, threshold, span, any, any_mask);
    if (rc != TW_OK) return fail_all(rc, ctx->err.c_str());
    return tw_batch_fetch(ctx, n, out, cap, res);
}

int tw_compare_batch_ignore(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                            const tw_flow_param *param, double threshold, int span, const tw_rect *const *ignore, const int *n_ignore,
                            tw_vector *out, int cap, tw_result *res)
{
    return tw_compare_batch_mask(ctx, n, expect, target, w, h, stride, param, threshold, span, ignore, n_ignore, nullptr, out, cap, res);
}

int tw_compare_batch(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                     const tw_flow_param *param, double threshold, int span, tw_vector *out, int cap, tw_result *res)
{
    return tw_compare_batch_ignore(ctx, n, expect, target, w, h, stride, param, threshold, span, nullptr, nullptr, out, cap, res);
}

// ---- pipelined form of tw_compare_batch: at most two batches in flight per context ----
// tw_pipe_submit returns as soon as everything is enqueued: the H2D copies of this batch go through a staging buffer on a copy
// stream (they overlap the previous batch's kernels), the compute stream takes them over with one device copy, runs the
// launch sequence and snapshots the compact results; tw_pipe_collect waits for the OLDEST batch and reads its snapshot on a third
// stream while the newer batch keeps running.  One host thread per GPU keeps the device busy this way (the reference: one
// Consumer thread per GPU, /root/reference/src/consumer.cpp:18-24, 42-94).
int tw_pipe_pending(tw_ctx *ctx) { return ctx ? ctx->pipe.count : 0; }

// 1 if the oldest batch in flight has finished on the device (tw_pipe_collect would not block), 0 if it is still running or nothing
// is in flight.
int tw_pipe_ready(tw_ctx *ctx)
{
    if (!ctx || ctx->pipe.count < 1) return 0;
    return cudaEventQuery(ctx->pipe.slot[ctx->pipe.head].done) == cudaSuccess ? 1 : 0;
}

int tw_pipe_submit_mask(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                        const tw_flow_param *param, double threshold, int span, const tw_rect *const *ignore, const int *n_ignore,
                        const uint8_t *const *mask)
{
    if (!ctx) return TW_BAD_PARAMETER;
    tw_ctx::Pipe &pp = ctx->pipe;
    if (pp.count >= 2) { ctx->err = "tw_pipe_submit: two batches in flight, collect one first"; return TW_BAD_PARAMETER; }
    if (n < 1 || n > ctx->max_batch || w < 1 || h < 1 || stride < w || span < 1) { ctx->err = "bad batch/size/span"; return TW_BAD_PARAMETER; }
    if ((ctx->max_w > 0 && w > ctx->max_w) || (ctx->max_h > 0 && h > ctx->max_h)) { ctx->err = "image larger than the context's max_w x max_h"; return TW_BAD_PARAMETER; }
    if (validate_param(param) != TW_OK) { ctx->err = "bad optical-flow parameter"; return TW_BAD_PARAMETER; }
    for (int i = 0; i < n; i++)
        if (!expect[i] || !target[i]) { ctx->err = "null image"; return TW_BAD_IMAGE_FORMAT; }
    cudaSetDevice(ctx->device);
    const bool same_plan = plan_fits(ctx, ctx->plan, w, h, *param);
    if (!same_plan && pp.count > 0) { ctx->err = "tw_pipe_submit: size / parameters changed, collect the pending batch first"; return TW_BAD_PARAMETER; }
    if (!build_plan(ctx, w, h, *param)) return TW_CUDA_ERROR;
    Plan &pl = ctx->plan;
    cudaError_t e = cudaSuccess;
    if (!pp.copy) {
        if ((e = cudaStreamCreateWithFlags(&pp.copy, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaStreamCreateWithFlags(&pp.fetch, cudaStreamNonBlocking)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&pp.ev_up, cudaEventDisableTiming)) != cudaSuccess ||
            (e = cudaEventCreateWithFlags(&pp.ev_stage_free, cudaEventDisableTiming)) != cudaSuccess) { set_err(ctx, "pipe setup", e); return TW_CUDA_ERROR; }
        for (auto &s : pp.slot) {
            if ((e = cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming)) != cudaSuccess || (e = cudaEventCreate(&s.r0)) != cudaSuccess ||
                (e = cudaEventCreate(&s.r1)) != cudaSuccess || (e = cudaMalloc(&s.d_counts, sizeof(int) * ctx->max_batch)) != cudaSuccess ||
                (e = cudaMallocHost(&s.h_counts, sizeof(int) * ctx->max_batch)) != cudaSuccess ||
                (e = cudaMallocHost(&s.h_ignore, ignore_bytes(ctx->max_batch))) != cudaSuccess ||
                (e = cudaMallocHost(&s.h_mask_has, sizeof(int) * ctx->max_batch)) != cudaSuccess) { set_err(ctx, "pipe setup", e); return TW_CUDA_ERROR; }
        }
    }
    // this batch's slot: free (at most one other batch in flight), its page-locked region mirror with it
    tw_ctx::PipeSlot &s = pp.slot[(pp.head + pp.count) & 1];
    const int packed = pack_ignore(ctx, n, ignore, n_ignore, w, h, s.h_ignore);
    if (packed < 0) return TW_BAD_PARAMETER;
    const bool any = packed > 0;
    bool any_mask = false;
    for (int i = 0; mask && i < n; i++) any_mask |= (s.h_mask_has[i] = mask[i] ? 1 : 0) != 0;
    if (any_mask && !ensure_mask_plane(ctx)) return TW_CUDA_ERROR;
    // staging buffer: the images of max_batch pairs, then the region lists (ignore_bytes); from the first masked batch on, then the
    // mask flags and the mask planes (at mask_at, 256-byte aligned)
    const size_t pair_bytes = (size_t)2 * h * pl.spitch, images = (size_t)ctx->max_batch * pair_bytes, plane = (size_t)h * pl.spitch;
    const size_t mask_at = (images + ignore_bytes(ctx->max_batch) + 255) & ~(size_t)255, mask_planes = mask_at + mask_flag_bytes(ctx->max_batch);
    const size_t need = any_mask ? mask_planes + ctx->max_batch * plane : images + ignore_bytes(ctx->max_batch);
    if (pp.stage_bytes < need) { // a new plan: nothing in flight (same_plan is false for a new size); the first masked batch: the batch
                                 // in flight, if any, must have taken its images over first
        cudaStreamSynchronize(pp.copy);
        if (pp.count > 0) cudaEventSynchronize(pp.ev_stage_free);
        else cudaStreamSynchronize(ctx->stream);
        if (pp.stage) cudaFree(pp.stage);
        pp.stage = nullptr; pp.stage_bytes = 0; pp.stage_used = false;
        if ((e = cudaMalloc(&pp.stage, need)) != cudaSuccess) { set_err(ctx, "cudaMalloc stage", e); return TW_CUDA_ERROR; }
        pp.stage_bytes = need;
    }
    // copy stream: the staging buffer is free once the previous batch's take-over copy has run
    if (pp.stage_used) cudaStreamWaitEvent(pp.copy, pp.ev_stage_free, 0);
    for (int i = 0; i < n; i++) {
        uint8_t *d = pp.stage + (size_t)i * pair_bytes;
        e = cudaMemcpy2DAsync(d, pl.spitch, expect[i], stride, w, h, cudaMemcpyHostToDevice, pp.copy);
        if (e == cudaSuccess) e = cudaMemcpy2DAsync(d + (size_t)h * pl.spitch, pl.spitch, target[i], stride, w, h, cudaMemcpyHostToDevice, pp.copy);
        if (e != cudaSuccess) { set_err(ctx, "H2D", e); return TW_CUDA_ERROR; }
    }
    if (any && (e = cudaMemcpyAsync(pp.stage + images, s.h_ignore, ignore_bytes(ctx->max_batch), cudaMemcpyHostToDevice, pp.copy)) != cudaSuccess) {
        set_err(ctx, "regions H2D", e);
        return TW_CUDA_ERROR;
    }
    if (any_mask) {
        e = cudaMemcpyAsync(pp.stage + mask_at, s.h_mask_has, sizeof(int) * n, cudaMemcpyHostToDevice, pp.copy);
        for (int i = 0; i < n && e == cudaSuccess; i++)
            if (mask[i]) e = cudaMemcpy2DAsync(pp.stage + mask_planes + i * plane, pl.spitch, mask[i], stride, w, h, cudaMemcpyHostToDevice, pp.copy);
        if (e != cudaSuccess) { set_err(ctx, "mask H2D", e); return TW_CUDA_ERROR; }
    }
    cudaEventRecord(pp.ev_up, pp.copy);
    // compute stream: the take-over copies run behind the previous batch's kernels, so its region lists and masks stay put while
    // they read them
    cudaStreamWaitEvent(ctx->stream, pp.ev_up, 0);
    e = cudaMemcpyAsync(pl.src, pp.stage, (size_t)n * pair_bytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess && any) e = cudaMemcpyAsync(ctx->d_ignore, pp.stage + images, ignore_bytes(ctx->max_batch), cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess && any_mask) e = cudaMemcpyAsync(pl.mask_has, pp.stage + mask_at, sizeof(int) * n, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess && any_mask) e = cudaMemcpyAsync(pl.mask, pp.stage + mask_planes, n * plane, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "stage -> src", e); return TW_CUDA_ERROR; }
    cudaEventRecord(pp.ev_stage_free, ctx->stream);
    pp.stage_used = true;
    cudaEventRecord(s.r0, ctx->stream);
    if (!run_sequence(ctx, n, threshold, span, any, any_mask)) return TW_CUDA_ERROR;
    cudaEventRecord(s.r1, ctx->stream);
    ctx->last_n = n; ctx->last_w = w; ctx->last_h = h; ctx->ran = true;
    ctx->last_span = span; ctx->last_regions = ctx->opt.change_regions != 0; ctx->last_intensity = ctx->opt.intensity != 0;
    ctx->last_sparse = sparse_in_effect(ctx, span);
    // snapshot of the compact results (counts + vectors), then the counts to the host
    const size_t vbytes = (size_t)n * ctx->dev_cap * sizeof(tw_vector);
    if (s.vec_bytes < vbytes) {
        if (s.d_vec) { cudaStreamSynchronize(pp.fetch); cudaFree(s.d_vec); s.d_vec = nullptr; s.vec_bytes = 0; }
        const size_t full = (size_t)ctx->max_batch * ctx->dev_cap * sizeof(tw_vector);
        if ((e = cudaMalloc(&s.d_vec, full)) != cudaSuccess) { set_err(ctx, "cudaMalloc snapshot", e); return TW_CUDA_ERROR; }
        s.vec_bytes = full;
    }
    e = cudaMemcpyAsync(s.d_counts, ctx->d_counts, sizeof(int) * n, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s.d_vec, ctx->d_vectors, vbytes, cudaMemcpyDeviceToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_counts, s.d_counts, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    s.regions = ctx->last_regions;
    if (e == cudaSuccess && s.regions) { // the change regions likewise: the host reads them on the fetch stream in tw_pipe_collect
        if ((!s.d_nreg && (e = cudaMalloc(&s.d_nreg, sizeof(int) * ctx->max_batch)) != cudaSuccess) ||
            (!s.h_nreg && (e = cudaMallocHost(&s.h_nreg, sizeof(int) * ctx->max_batch)) != cudaSuccess) ||
            (!s.d_regions && (e = cudaMalloc(&s.d_regions, sizeof(tw_change_region) * ctx->max_batch * kMaxChangeRegions)) != cudaSuccess)) {
            set_err(ctx, "cudaMalloc snapshot", e);
            return TW_CUDA_ERROR;
        }
        e = cudaMemcpyAsync(s.d_nreg, ctx->d_nreg, sizeof(int) * n, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s.d_regions, ctx->d_regions, sizeof(tw_change_region) * n * kMaxChangeRegions, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_nreg, s.d_nreg, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    }
    s.intensity = ctx->last_intensity;
    if (e == cudaSuccess && s.intensity) { // the intensity cells likewise
        if ((!s.d_ncell && (e = cudaMalloc(&s.d_ncell, sizeof(int) * ctx->max_batch)) != cudaSuccess) ||
            (!s.h_ncell && (e = cudaMallocHost(&s.h_ncell, sizeof(int) * ctx->max_batch)) != cudaSuccess) ||
            (!s.d_cells && (e = cudaMalloc(&s.d_cells, sizeof(tw_intensity_cell) * ctx->max_batch * kMaxIntensityCells)) != cudaSuccess)) {
            set_err(ctx, "cudaMalloc snapshot", e);
            return TW_CUDA_ERROR;
        }
        e = cudaMemcpyAsync(s.d_ncell, ctx->d_ncell, sizeof(int) * n, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(s.d_cells, ctx->d_cells, sizeof(tw_intensity_cell) * n * kMaxIntensityCells, cudaMemcpyDeviceToDevice, ctx->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(s.h_ncell, s.d_ncell, sizeof(int) * n, cudaMemcpyDeviceToHost, ctx->stream);
    }
    if (e != cudaSuccess) { set_err(ctx, "snapshot", e); return TW_CUDA_ERROR; }
    cudaEventRecord(s.done, ctx->stream);
    s.n = n; s.w = w; s.h = h; s.dev_cap = ctx->dev_cap;
    pp.count++;
    return TW_OK;
}

int tw_pipe_submit_ignore(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                          const tw_flow_param *param, double threshold, int span, const tw_rect *const *ignore, const int *n_ignore)
{
    return tw_pipe_submit_mask(ctx, n, expect, target, w, h, stride, param, threshold, span, ignore, n_ignore, nullptr);
}

int tw_pipe_submit(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                   const tw_flow_param *param, double threshold, int span)
{
    return tw_pipe_submit_ignore(ctx, n, expect, target, w, h, stride, param, threshold, span, nullptr, nullptr);
}

int tw_pipe_collect(tw_ctx *ctx, tw_vector *out, int cap, tw_result *res)
{
    if (!ctx || !res) return TW_BAD_PARAMETER;
    tw_ctx::Pipe &pp = ctx->pipe;
    if (pp.count < 1) { ctx->err = "tw_pipe_collect: nothing in flight"; return TW_BAD_PARAMETER; }
    cudaSetDevice(ctx->device);
    tw_ctx::PipeSlot &s = pp.slot[pp.head];
    pp.head ^= 1; pp.count--;
    const int n = s.n;
    answer_regions(ctx, n, s.regions);
    answer_cells(ctx, n, s.intensity);
    cudaError_t e = cudaEventSynchronize(s.done);
    if (e != cudaSuccess) {
        set_err(ctx, "collect", e);
        for (int i = 0; i < n; i++) fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str());
        return TW_CUDA_ERROR;
    }
    float ms = 0;
    cudaEventElapsedTime(&ms, s.r0, s.r1);
    bool copied = false;
    for (int i = 0; i < n; i++) {
        const int cnt = s.h_counts[i];
        const int ncell = s.intensity ? s.h_ncell[i] : 0;
        memset(&res[i], 0, sizeof(tw_result));
        res[i].code = TW_OK;
        res[i].status = cnt == 0 && ncell == 0 ? TW_STATUS_OK : TW_STATUS_SUSPICIOUS;
        res[i].n_vectors = cnt;
        res[i].width = s.w; res[i].height = s.h;
        res[i].time = ms * 1e-3f / n;
        const int ncopy = std::min(std::min(cnt, cap), s.dev_cap);
        if (ncopy > 0 && out) {
            e = cudaMemcpyAsync(out + (size_t)i * cap, (const tw_vector *)s.d_vec + (size_t)i * s.dev_cap, sizeof(tw_vector) * ncopy,
                                cudaMemcpyDeviceToHost, pp.fetch);
            if (e != cudaSuccess) { set_err(ctx, "collect vectors", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
            copied = true;
        }
        const int nreg = s.regions ? std::min(s.h_nreg[i], kMaxChangeRegions) : 0;
        if (nreg > 0 && res[i].code == TW_OK) {
            e = cudaMemcpyAsync(ctx->h_regions + (size_t)i * kMaxChangeRegions, s.d_regions + (size_t)i * kMaxChangeRegions,
                                sizeof(tw_change_region) * nreg, cudaMemcpyDeviceToHost, pp.fetch);
            if (e != cudaSuccess) { set_err(ctx, "collect regions", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
            copied = true;
        }
        if (s.regions) ctx->h_nreg[i] = res[i].code == TW_OK ? s.h_nreg[i] : 0;
        const int kcell = std::min(ncell, kMaxIntensityCells);
        if (kcell > 0 && res[i].code == TW_OK && ctx->cell_pairs > 0) {
            e = cudaMemcpyAsync(ctx->h_cells + (size_t)i * kMaxIntensityCells, s.d_cells + (size_t)i * kMaxIntensityCells,
                                sizeof(tw_intensity_cell) * kcell, cudaMemcpyDeviceToHost, pp.fetch);
            if (e != cudaSuccess) { set_err(ctx, "collect intensity cells", e); fill_error(&res[i], TW_CUDA_ERROR, ctx->err.c_str()); }
            copied = true;
        }
        if (ctx->cell_pairs > 0) ctx->h_ncell[i] = res[i].code == TW_OK ? ncell : 0;
    }
    if (copied && (e = cudaStreamSynchronize(pp.fetch)) != cudaSuccess) { set_err(ctx, "collect sync", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_compare_mask(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_,
                    const tw_flow_param *param, double threshold, int span, const tw_rect *ignore, int n_ignore, const uint8_t *mask,
                    tw_vector *out, int cap, tw_result *res)
{
    if (!res) return TW_BAD_PARAMETER;
    if (!ctx) { fill_error(res, TW_BAD_PARAMETER, "null context"); return res->code; }
    answer_regions(ctx, 1, ctx->opt.change_regions != 0); // what an ERROR answer leaves: 0 regions
    answer_cells(ctx, 1, ctx->opt.intensity != 0);        // and 0 intensity cells
    // src/opticalflow.cpp:37-49: an image that cannot be opened is BadImageFormat
    if (!expect || ew < 1 || eh < 1) { fill_error(res, TW_BAD_IMAGE_FORMAT, "Can't open expected image"); return res->code; }
    if (!target || tw_ < 1 || th_ < 1) { fill_error(res, TW_BAD_IMAGE_FORMAT, "Can't open target image"); return res->code; }
    // src/opticalflow.cpp:52-61
    if (abs(eh - th_) > 5 || abs(ew - tw_) > 5) { fill_error(res, TW_DONT_MATCH_SIZE, "Don't match image size"); return res->code; }
    if (eh != th_ || ew != tw_) {
        // src/opticalflow.cpp:64-68: sizes within 5 px -> the target is resized (bilinear) to the expected size
        if (span < 1) { fill_error(res, TW_BAD_PARAMETER, "span must be >= 1"); return res->code; }
        if (validate_param(param) != TW_OK) { fill_error(res, TW_BAD_PARAMETER, "bad optical-flow parameter"); return res->code; }
        int rc = upload_impl(ctx, 1, &expect, &expect, ew, eh, ew, param); // builds the plan, fills the expected slot
        if (rc == TW_OK && !upload_resized_target(ctx, target, tw_, th_, ew, eh)) rc = TW_CUDA_ERROR;
        // regions and masks are painted over the resized target (the paint kernels run first in the launch sequence)
        bool any = false, any_mask = false;
        if (rc == TW_OK) rc = upload_ignore(ctx, 1, &ignore, &n_ignore, ew, eh, &any);
        if (rc == TW_OK) rc = upload_mask(ctx, 1, &mask, ew, eh, ew, &any_mask);
        if (rc == TW_OK) rc = run_batch(ctx, 1, ew, eh, param, threshold, span, any, any_mask);
        if (rc != TW_OK) { fill_error(res, rc, ctx->err.c_str()); return res->code; }
        tw_batch_fetch(ctx, 1, out, cap, res);
        return res->code;
    }
    tw_compare_batch_mask(ctx, 1, &expect, &target, ew, eh, ew, param, threshold, span, &ignore, &n_ignore, &mask, out, cap, res);
    return res->code;
}

int tw_compare_ignore(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_,
                      const tw_flow_param *param, double threshold, int span, const tw_rect *ignore, int n_ignore,
                      tw_vector *out, int cap, tw_result *res)
{
    return tw_compare_mask(ctx, expect, ew, eh, target, tw_, th_, param, threshold, span, ignore, n_ignore, nullptr, out, cap, res);
}

int tw_compare(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw_, int th_,
               const tw_flow_param *param, double threshold, int span, tw_vector *out, int cap, tw_result *res)
{
    return tw_compare_ignore(ctx, expect, ew, eh, target, tw_, th_, param, threshold, span, nullptr, 0, out, cap, res);
}

int tw_l2_flush(tw_ctx *ctx)
{
    if (!ctx) return TW_BAD_PARAMETER;
    cudaSetDevice(ctx->device);
    const size_t bytes = (size_t)256 << 20;
    if (!ctx->flush_buf) {
        cudaError_t e = cudaMalloc(&ctx->flush_buf, bytes);
        if (e != cudaSuccess) { set_err(ctx, "flush alloc", e); return TW_CUDA_ERROR; }
    }
    ctx->flush_val ^= 1;
    cudaError_t e = cudaMemsetAsync(ctx->flush_buf, ctx->flush_val, bytes, ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "flush", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_resize_target(tw_ctx *ctx, const uint8_t *target, int tw_, int th_, uint8_t *out, int ew, int eh)
{
    if (!ctx || !target || !out || tw_ < 1 || th_ < 1 || ew < 1 || eh < 1) return TW_BAD_PARAMETER;
    cudaSetDevice(ctx->device);
    tw_flow_param p;
    if (ctx->plan.valid) p = ctx->plan.p; else tw_default_param(&p);
    if (!build_plan(ctx, ew, eh, p)) return TW_CUDA_ERROR;
    if (!upload_resized_target(ctx, target, tw_, th_, ew, eh)) return TW_CUDA_ERROR;
    Plan &pl = ctx->plan;
    cudaError_t e = cudaMemcpy2DAsync(out, ew, pl.src + (size_t)eh * pl.spitch, pl.spitch, ew, eh, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { set_err(ctx, "resize D2H", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_timer_start(tw_ctx *ctx)
{
    if (!ctx) return TW_BAD_PARAMETER;
    cudaSetDevice(ctx->device);
    return cudaEventRecord(ctx->ev_t0, ctx->stream) == cudaSuccess ? TW_OK : TW_CUDA_ERROR;
}

int tw_timer_stop(tw_ctx *ctx, float *ms)
{
    if (!ctx) return TW_BAD_PARAMETER;
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaEventRecord(ctx->ev_t1, ctx->stream);
    if (e == cudaSuccess) e = cudaEventSynchronize(ctx->ev_t1);
    if (e == cudaSuccess && ms) e = cudaEventElapsedTime(ms, ctx->ev_t0, ctx->ev_t1);
    if (e != cudaSuccess) { set_err(ctx, "timer", e); return TW_CUDA_ERROR; }
    return TW_OK;
}

int tw_profile_enable(tw_ctx *ctx, int on)
{
    if (!ctx) return TW_BAD_PARAMETER;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    drain_profile(ctx);
    ctx->profiling = on != 0;
    for (int i = 0; i < F_COUNT; i++) { ctx->fam_ms[i] = 0; ctx->fam_launches[i] = 0; ctx->fam_bytes[i] = 0; }
    return TW_OK;
}

int tw_profile_read(tw_ctx *ctx, int max_n, const char **names, float *ms, int *launches, double *alg_bytes)
{
    if (!ctx) return -1;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    drain_profile(ctx);
    int n = std::min(max_n, (int)F_COUNT);
    for (int i = 0; i < n; i++) {
        if (names) names[i] = kFamilyNames[i];
        if (ms) ms[i] = ctx->fam_ms[i];
        if (launches) launches[i] = ctx->fam_launches[i];
        if (alg_bytes) alg_bytes[i] = ctx->fam_bytes[i];
    }
    return F_COUNT;
}

long long tw_launch_count(tw_ctx *ctx) { return ctx ? ctx->launches : 0; }

int tw_change_regions(tw_ctx *ctx, int pair, tw_change_region *out, int cap, int *n_regions)
{
    if (!ctx) return TW_BAD_PARAMETER;
    if (ctx->reg_pairs < 0) { ctx->err = "tw_change_regions: the last answered batch ran without \"change_regions\""; return TW_BAD_PARAMETER; }
    if (pair < 0 || pair >= ctx->reg_pairs) { ctx->err = "tw_change_regions: pair out of range"; return TW_BAD_PARAMETER; }
    const int total = ctx->h_nreg[pair];
    const int k = std::min(std::min(cap, total), kMaxChangeRegions);
    if (out && k > 0) memcpy(out, ctx->h_regions + (size_t)pair * kMaxChangeRegions, sizeof(tw_change_region) * k);
    if (n_regions) *n_regions = total;
    return TW_OK;
}

int tw_intensity_cells(tw_ctx *ctx, int pair, tw_intensity_cell *out, int cap, int *n_cells)
{
    if (!ctx) return TW_BAD_PARAMETER;
    if (ctx->cell_pairs < 0) { ctx->err = "tw_intensity_cells: the last answered batch ran without \"intensity_threshold\""; return TW_BAD_PARAMETER; }
    if (pair < 0 || pair >= ctx->cell_pairs) { ctx->err = "tw_intensity_cells: pair out of range"; return TW_BAD_PARAMETER; }
    const int total = ctx->h_ncell[pair];
    const int k = std::min(std::min(cap, total), kMaxIntensityCells);
    if (out && k > 0) memcpy(out, ctx->h_cells + (size_t)pair * kMaxIntensityCells, sizeof(tw_intensity_cell) * k);
    if (n_cells) *n_cells = total;
    return TW_OK;
}

int tw_set_option(tw_ctx *ctx, const char *name, int value)
{
    if (!ctx || !name) return TW_BAD_PARAMETER;
    if (!strcmp(name, "arithmetic")) { ctx->opt.arith = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "graph")) { ctx->opt_graph = value ? 1 : 0; if (!value) drop_graph(ctx->plan); return TW_OK; }
    if (!strcmp(name, "gauss_fma") || !strcmp(name, "update_fma") || !strcmp(name, "gauss_scalar")) {
        // studied and rejected relaxations (oracle relax bits 0 / 6) and the scalar v1 window kernel: no longer in the library
        if (value) { ctx->err = std::string(name) + ": removed from the library (DESIGN.md section 2)"; return TW_UNSUPPORTED; }
        return TW_OK;
    }
    if (!strcmp(name, "sparse_last")) { ctx->opt.sparse_last = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "polyexp_tma")) { // takes effect when the next plan is built (the tensor maps are made with the plan)
        ctx->opt_poly_no_tma = value ? 0 : 1;
        ctx->plan.valid = false;
        cudaStreamSynchronize(ctx->stream);
        flush_plan_cache(ctx);
        return TW_OK;
    }
    if (!strcmp(name, "box_unfused")) { ctx->opt.box_unfused = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "window_tiles")) { ctx->opt.window_tiles = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "level_generic")) { ctx->opt.level_generic = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "level_unfused")) { ctx->opt.level_unfused = value ? 1 : 0; return TW_OK; }
    if (!strcmp(name, "change_regions")) { // the batches in flight were submitted with the other setting
        if (ctx->pipe.count > 0) { ctx->err = "change_regions: collect the pending pipe batches first"; return TW_BAD_PARAMETER; }
        ctx->opt.change_regions = value ? 1 : 0;
        return TW_OK;
    }
    if (!strcmp(name, "intensity_threshold")) {
        if (value < 0 || value > 255) { ctx->err = "intensity_threshold: 0 (off) or 1 .. 255 gray levels"; return TW_BAD_PARAMETER; }
        if (ctx->pipe.count > 0) { ctx->err = "intensity_threshold: collect the pending pipe batches first"; return TW_BAD_PARAMETER; }
        ctx->opt.intensity = value;
        return TW_OK;
    }
    if (!strcmp(name, "tight_pitch")) {
        ctx->opt_tight_pitch = value ? 1 : 0;
        ctx->plan.valid = false;
        cudaStreamSynchronize(ctx->stream);
        flush_plan_cache(ctx);
        return TW_OK;
    }
    if (!strcmp(name, "plan_cache")) { // how many plans besides the current one are kept (0: rebuild on every change of size / parameters)
        ctx->plan_cache_max = value < 0 ? 0 : value;
        cudaStreamSynchronize(ctx->stream);
        flush_plan_cache(ctx);
        return TW_OK;
    }
    ctx->err = std::string("unknown option ") + name;
    return TW_BAD_PARAMETER;
}

int tw_set_default_arithmetic(int relaxed)
{
    g_default_arith.store(relaxed ? 1 : 0);
    return TW_OK;
}

int tw_arithmetic_in_effect(tw_ctx *ctx, const tw_flow_param *param)
{
    if (!ctx || !param) return -1;
    return relaxed_in_effect(ctx, *param) ? 1 : 0;
}

int tw_debug_keep_levels(tw_ctx *ctx, int on)
{
    if (!ctx) return TW_BAD_PARAMETER;
    ctx->keep_levels = on ? 1 : 0;
    return TW_OK;
}

int tw_debug_read(tw_ctx *ctx, const char *name, int scale, int pair, float *out, int cap_floats, int *w, int *h)
{
    if (!ctx || !ctx->ran || !name || !out) return -1;
    Plan &pl = ctx->plan;
    if (scale < 0 || scale >= (int)pl.scales.size() || pair < 0 || pair >= ctx->last_n) return -1;
    cudaSetDevice(ctx->device);
    const Scale &s = pl.scales[scale];
    const float *base = nullptr;
    int cn = 0;
    if (!strcmp(name, "I0")) { base = s.I + (size_t)pair * 2 * s.d.plane; cn = 1; }
    else if (!strcmp(name, "I1")) { base = s.I + ((size_t)pair * 2 + 1) * s.d.plane; cn = 1; }
    else if (!strcmp(name, "R0")) { base = s.R + (size_t)pair * 10 * s.d.plane; cn = 5; }
    else if (!strcmp(name, "R1")) { base = s.R + ((size_t)pair * 10 + 5) * s.d.plane; cn = 5; }
    else if (!strcmp(name, "M")) {
        // the buffer the last iteration kernel of this scale read (its input M)
        int it = pl.p.pyrIterations;
        const float *m = (it <= 1 || ((it - 1) % 2 == 0)) ? s.M0 : s.M1;
        base = m + (size_t)pair * 5 * s.d.plane; cn = 5;
    }
    else if (!strcmp(name, "flow")) { base = s.flow + (size_t)pair * 2 * s.d.plane; cn = 2; }
    else return -1;
    if ((size_t)cn * s.d.w * s.d.h > (size_t)cap_floats) return -2;
    if (w) *w = s.d.w;
    if (h) *h = s.d.h;
    if (cn == 5) {
        // R and M are row-interleaved (tw_kernels.cu): (y, c, x) at (y*5 + c)*pitch + x; M additionally packs the
        // channel pairs (0,1) and (2,3) as float2.  De-interleave on the host.
        const bool isM = !strcmp(name, "M");
        std::vector<float> tmp(5 * s.d.plane);
        if (cudaMemcpyAsync(tmp.data(), base, sizeof(float) * 5 * s.d.plane, cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
            cudaStreamSynchronize(ctx->stream) != cudaSuccess)
            return -3;
        const size_t P = (size_t)s.d.w * s.d.h;
        const int pitch = s.d.pitch;
        for (int y = 0; y < s.d.h; y++)
            for (int x = 0; x < s.d.w; x++) {
                const float *row = tmp.data() + (size_t)y * 5 * pitch;
                const size_t q = (size_t)y * s.d.w + x;
                if (isM) {
                    out[q] = row[2 * x]; out[P + q] = row[2 * x + 1];
                    out[2 * P + q] = row[2 * pitch + 2 * x]; out[3 * P + q] = row[2 * pitch + 2 * x + 1];
                    out[4 * P + q] = row[4 * pitch + x];
                } else {
                    for (int c = 0; c < 5; c++) out[c * P + q] = row[c * pitch + x];
                }
            }
        return cn;
    }
    for (int c = 0; c < cn; c++) {
        cudaError_t e = cudaMemcpy2DAsync(out + (size_t)c * s.d.w * s.d.h, sizeof(float) * s.d.w, base + (size_t)c * s.d.plane,
                                          sizeof(float) * s.d.pitch, sizeof(float) * s.d.w, s.d.h, cudaMemcpyDeviceToHost, ctx->stream);
        if (e != cudaSuccess) { set_err(ctx, "debug read", e); return -3; }
    }
    if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -3;
    return cn;
}

} // extern "C"
