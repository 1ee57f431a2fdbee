// tw_kernels.cuh -- launch wrappers of the sm_100a kernel families (see DESIGN.md section 3).
// Device layout: every tensor is PLANAR float32 with a row pitch that is a multiple of 32 floats (128 B):
//   I    [B][2][h][pitch]        level images (expected, target)
//   R    [B][2][5][h][pitch]     polynomial expansion coefficients (R0 = expected, R1 = target)
//   M    [B][5][h][pitch]        (G11, G12, G22, h1, h2)
//   flow [B][2][h][pitch]        (dx, dy)
// A "plane" is h*pitch floats.  Batches are the outermost dimension; kernels index them with blockIdx.z.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace tw {

constexpr int kMaxPolyN = 15;    // radius of the polynomial expansion window
constexpr int kMaxWinRadius = 32; // winSize/2

struct PolyTables {
    float g[kMaxPolyN + 1], xg[kMaxPolyN + 1], xxg[kMaxPolyN + 1];
    double gd[kMaxPolyN + 1], xxgd[kMaxPolyN + 1]; // (double)g[k], (double)xxg[k]: no conversions in the tap loop
    double ig11, ig03, ig33, ig55;
    float fig11, fig55; // (float)ig11, (float)ig55: relaxed-arithmetic kernel
    float one;          // 1.0f, deliberately a runtime value (packed f32x2 accumulate: see tw_fma2 in tw_device.cuh)
    int n;
};

struct WinTaps {
    float k[kMaxWinRadius + 1];
    float one; // 1.0f, deliberately a runtime value (see tw_fma2 in tw_kernels.cu)
    int m;
};

struct LevelDims {
    int w, h, pitch;
    size_t plane; // h * pitch
};

// K1: u8 full-res frames -> float level image (pre-blur REFLECT_101 + bilinear downsample), SURVEY App. A.2.
struct LevelImageArgs {
    const uint8_t *src; // [nimg][H][spitch]
    int W, H, spitch;
    float *dst;         // [nimg][h][pitch]
    LevelDims d;
    const int *xi; const float *xf; const int *yi; const float *yf; // device tables, A.2b
    const float *taps;  // device, ksize floats
    int ksize;
    int nimg;
    int tile_w, tile_h; // output tile
    int smem_w, smem_h; // source tile bound (before clamping)
    int identity;       // w == W && h == H
    int small;          // ksize/2 >= min(W, H): multi-bounce reflect path
};
cudaError_t launch_level_image(cudaStream_t s, const LevelImageArgs &a);
// Fast paths (full-resolution level; exact integer down-scales 2/4/8/16).  int_scale = S if W == w*S, H == h*S and the
// resize tables are exactly (S*d + S/2 - 1, 0.5), else 0.  Returns cudaErrorNotSupported if none applies.
cudaError_t launch_level_image_fast(cudaStream_t s, const LevelImageArgs &a, const float *host_taps, int int_scale);
// Long pre-blur kernels (ksize >= 31, not an exact integer down-scale): separable blur through an intermediate T in global memory
// ([nimg][H][roundup(2w, 32)] floats, level_image_big_floats): two small launches instead of huge shared-memory tiles.
bool level_image_big_ok(const LevelImageArgs &a);
size_t level_image_big_floats(int H, int w, int nimg);
cudaError_t launch_level_image_big(cudaStream_t s, const LevelImageArgs &a, float *T);
// All four level images of the default pyramid (S = 8, 4, 2, 1 with 19/9/3/3-tap pre-blurs) from one staged source tile.
cudaError_t launch_level_fused(cudaStream_t s, const uint8_t *src, int W, int H, int spitch, float *const dst[4], const LevelDims d[4],
                               const float *k8, const float *k4, const float *k2, const float *k1, int nimg);
size_t level_image_smem_bytes(int smem_w, int smem_h, int tile_w, int ksize, int identity);

// K2: polynomial expansion I -> R (5 planes), SURVEY App. A.3.  nimg = 2*B images.
// relaxed = 1: the mixed double/float horizontal pass (polyN 5 / 7 only; otherwise the faithful kernels run).
// `imap` (optional): tensor map of I made by make_polyexp_map -- interior tiles of the relaxed kernel are then staged by ONE TMA tile copy
// (cp.async.bulk.tensor) instead of per-thread loads; border tiles (replicate clamp) keep the per-thread path.
struct TileMap {
    alignas(64) unsigned char opaque[128]; // one CUtensorMap
    int valid;
};
bool make_polyexp_map(const float *I, const LevelDims &d, int nimg, int polyN, TileMap *out);
cudaError_t launch_polyexp(cudaStream_t s, const float *I, float *R, const LevelDims &d, int nimg, const PolyTables &t, int relaxed,
                           const TileMap *imap = nullptr);

// K3: (coarse flow -> bilinear upsample * 1/pyrScale | zero) -> first update-matrices, App. A.1 + A.4.
struct FirstUpdateArgs {
    const float *flow_in; // [B][2] planes of THIS scale (box window path), or nullptr
    const float *coarse; // [B][2][ch][cpitch] or nullptr (coarsest scale: zero flow)
    LevelDims cd;
    const int *xi; const float *xf; const int *yi; const float *yf; // upsample tables
    float inv_scale;
    const float *R;  // [B][2][5] planes
    float *M;        // [B][5] planes (nullptr: skip)
    float *flow_out; // [B][2] planes (nullptr: skip; used when pyrIterations == 0)
    LevelDims d;
    int batch;
};
cudaError_t launch_first_update(cudaStream_t s, const FirstUpdateArgs &a);

// K4/K5: window blur of M + 2x2 solve, then (not last) next update-matrices or (last) flow write.
struct IterArgs {
    const float *Min; // [B][5] planes
    float *Mout;      // [B][5] planes (not last)
    const float *R;   // [B][2][5] planes
    float *flow;      // [B][2] planes (last)
    LevelDims d;
    int batch;
    int last;
    // span sampling fused into the last iteration of the finest scale (reference src/consumer.cpp:60-77): the
    // threshold test runs on the flow tile while it is still in shared memory; per-pair counts are reduced with
    // warp shuffles and one atomicAdd per warp.  span == 0: off.
    int span;
    double thr2;
    int *counts; // [B], zeroed by the host before the launch
    int fma; // Gaussian tap sums: 0 = oracle order (add, mul, add); 2 = the validated relaxation, direct form fmaf(a, k, t),
             // fmaf(b, k, t) (oracle relax bit 7).  Never set for the box window.
};
cudaError_t launch_gauss_iter(cudaStream_t s, const IterArgs &a, const WinTaps &t);
// K4/K5 for window radius 15: the persistent, warp-specialised strip kernel (tw_window.cu).  Its operands arrive through
// TMA tensor maps (cuTensorMapEncodeTiled) built once per (scale, M buffer): make_strip_maps.
struct StripMaps {
    alignas(64) unsigned char opaque[6 * 128]; // six CUtensorMap: M channel-pair / h2 rows (1-row and 8-row boxes), R0 tiles, R1 row chunks
    int valid;
};
bool make_strip_maps(const float *M, const float *R, const LevelDims &d, int batch, StripMaps *out);
bool gauss_strip_ok(const IterArgs &a, const WinTaps &t);
cudaError_t launch_gauss_strip(cudaStream_t s, const IterArgs &a, const WinTaps &t, const StripMaps &m);
// K5s: last iteration of the finest scale evaluated only at the span-grid points (needs a.span, a.thr2, a.counts; writes the
// sampled (dx, dy) at their positions of a.flow and nothing else).  gauss_last_sparse_ok: whether this geometry is supported.
bool gauss_last_sparse_ok(const IterArgs &a, const WinTaps &t);
cudaError_t launch_gauss_last_sparse(cudaStream_t s, const IterArgs &a, const WinTaps &t);
// Box window (flags == 0), App. A.6: vertical float-difference running sums in double (VT = V transposed,
// [B*5][w][roundup(h,32)] doubles), then the horizontal running sum + solve -> flow; the next update-matrices
// is launch_first_update with flow_in.
cudaError_t launch_box_vsum(cudaStream_t s, const float *Min, double *VT, const LevelDims &d, int batch, int m);
cudaError_t launch_box_hscan(cudaStream_t s, const double *VT, float *flow, const LevelDims &d, int batch, int m, int winSize);
// Fused form (m <= 16): launch_box_ckpt keeps only the vertical running sums at the top of every band of box_band_height() rows (CK: [B][bands]
// [5 * pitch] doubles); launch_box_band re-runs them inside each band from its checkpoint, continues the horizontal running sums
// across the band and goes straight on to the solve and the next update-matrices (or the flow store): no V plane in HBM.
bool box_fused_ok(const LevelDims &d, int m);
int box_band_height(); // rows per band: CK holds ceil(h / box_band_height()) checkpoints per pair
cudaError_t launch_box_ckpt(cudaStream_t s, const float *Min, double *CK, const LevelDims &d, int batch, int m);
cudaError_t launch_box_band(cudaStream_t s, const float *Min, const double *CK, const float *R, float *Mout, float *flow, const LevelDims &d,
                            int batch, int m, int winSize, int last);

// +-5 px size-tolerance path: OpenCV's 8-bit fixed-point bilinear resize of the target to the expected size.
struct ResizeU8Args {
    const uint8_t *src; int W, H, spitch;   // device, target as uploaded
    uint8_t *dst; int w, h, dpitch;         // device, target slot of the pair
    const int *xi, *yi;                     // device tables
    const short *xa, *ya;                   // device, 2 coefficients per output column / row (x2048)
};
cudaError_t launch_resize_u8(cudaStream_t s, const ResizeU8Args &a);

// Span sampling + threshold classification + ordered compaction, reference src/consumer.cpp:60-77.
struct SampleArgs {
    const float *flow; // [B][2] planes, full-res
    LevelDims d;
    int batch;
    int span;
    double thr2; // threshold * threshold in double
    int *counts;       // [B]
    int counted;       // counts[] already hold the totals (fused into K5): pairs with 0 vectors exit at once
    void *vectors;     // [B][cap] tw_vector {int x, int y, double dx, double dy}
    int cap;
};
cudaError_t launch_sample(cudaStream_t s, const SampleArgs &a);

// Ignore regions (tw_compare_ignore and the other *_ignore entry points): up to kMaxIgnore rectangles per pair, clipped to the
// frame on the host and stored as non-empty half-open bounds int4 (x0, y0, x1, y1).  Pairs without regions have n[b] = 0.
constexpr int kMaxIgnore = 32; // TW_MAX_IGNORE
struct IgnoreRegions {
    const int4 *rects; // [B][kMaxIgnore]
    const int *n;      // [B]
};
// Copies the expected pixels inside each region over the target slot of src ([B][2][H][spitch] u8): the flow is then the
// ordinary flow of (expected, painted target).  Grid (kMaxIgnore, batch), one CTA per (region, pair).
cudaError_t launch_ignore_paint(cudaStream_t s, uint8_t *src, int H, int spitch, const IgnoreRegions &g, int batch);
// sample_kernel with the point test of the regions: a sample point inside any region of its pair yields no vector and is not
// counted.  Same arguments as launch_sample (a.counted included: see the early exit of the kernel).
cudaError_t launch_sample_ignore(cudaStream_t s, const SampleArgs &a, const IgnoreRegions &g);

// Ignore masks (tw_compare_mask and the other *_mask entry points): one u8 plane per pair in expected-image pixels, nonzero =
// ignore, laid out like a slot of src ([B][H][spitch], 16-byte aligned rows; the bytes past column W are never read).  Pairs
// without a mask have has[b] = 0 and their plane is not read.
struct IgnoreMasks {
    const uint8_t *m; // [B][H][spitch]
    const int *has;   // [B]
    int W, H, spitch;
};
// Copies the expected pixels where the pair's mask is nonzero over the target slot of src (as launch_ignore_paint does inside
// regions).  One thread per 16 bytes of a row; grid (ceil(H * ceil(W / 16) / 256), batch).
cudaError_t launch_mask_paint(cudaStream_t s, uint8_t *src, const IgnoreMasks &k, int batch);
// sample_kernel with the point test of the pair's mask and then of its regions (g.n == NULL: no pair has regions).  Same
// arguments as launch_sample_ignore.
cudaError_t launch_sample_mask(cudaStream_t s, const SampleArgs &a, const IgnoreRegions &g, const IgnoreMasks &k);

// Change regions (tw_change_regions): the 8-connected components of each pair's sample points that yielded a vector, read from the
// compact vector list the sample kernel wrote (never from the flow).  Regions are stored in the order of their first vector; at
// most kMaxChangeRegions per pair, n_regions[b] is the full count.  One CTA per pair.
constexpr int kMaxChangeRegions = 1024; // TW_MAX_CHANGE_REGIONS
struct ChangeRegionArgs {
    const void *vectors; // [B][cap] tw_vector, as SampleArgs::vectors
    const int *counts;   // [B] vectors per pair (after the sample kernel)
    int cap;
    int w, h, span;      // frame (expected-image pixels) and sample spacing
    int *scratch;        // [B][2][cap] int: cell -> vector index map (never cleared: entries are checked against the vectors), then
                         // union-find parents
    int *n_regions;      // [B]
    void *regions;       // [B][kMaxChangeRegions] tw_change_region
    int batch;
};
cudaError_t launch_change_regions(cudaStream_t s, const ChangeRegionArgs &a);

// Intensity cells (tw_intensity_cells): the span cells whose pixels changed where the flow found no motion.  Cell (i, j) is
// [i * span, min(i * span + span, w)) x [j * span, min(j * span + span, h)); its shift is the rounded flow at its sample point.
// launch_intensity_sum sums, per cell, the residual r(p) = min over the 3 x 3 neighbours of the shifted target pixel of
// |E(p) - T| and the count of pixels not ignored (regions, mask); launch_intensity_count counts the cells with n > 0 and S > t * n
// per chunk of kIntChunk cells, and launch_intensity_compact writes them in scan order and clears the totals it read.  All
// arithmetic is integer, so the sums are exact whatever the order of the atomics.
constexpr int kMaxIntensityCells = 4096; // TW_MAX_INTENSITY_CELLS
constexpr int kIntChunk = 8192;          // cells per CTA of the count and compact steps
struct IntensityArgs {
    const uint8_t *src;       // [B][2][h][spitch]: expected, then the target as the flow saw it (resized, painted)
    int spitch;
    const float *flow;        // [B][2] planes of the finest scale: the flow at every sample point
    LevelDims d;
    int span;
    int t;                    // threshold in gray levels, 1 .. 255
    IgnoreRegions g;          // g.n == NULL: no pair has regions
    IgnoreMasks k;            // k.m == NULL: no pair has a mask
    unsigned long long *sum;  // [B][cell_cap] residual sums S: zero before launch_intensity_sum, zero again after the compaction
    unsigned int *cnt;        // [B][cell_cap] pixel counts n, likewise
    int cell_cap;             // >= ceil(w / span) * ceil(h / span)
    int *chunk_counts;        // [B][max_chunks] intensity cells per chunk
    int max_chunks;           // >= intensity_chunks(w, h, span)
    int *n_cells;             // [B] flagged cells (full count)
    void *cells;              // [B][kMaxIntensityCells] tw_intensity_cell
    int batch;
};
int intensity_chunks(int w, int h, int span);
cudaError_t launch_intensity_sum(cudaStream_t s, const IntensityArgs &a);
cudaError_t launch_intensity_count(cudaStream_t s, const IntensityArgs &a);
cudaError_t launch_intensity_compact(cudaStream_t s, const IntensityArgs &a);

} // namespace tw
