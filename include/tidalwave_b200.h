/*
 * tidalwave_b200.h -- C ABI of the B200-native hot path of arielnetworks/tidal-wave:
 * dense Farneback optical flow between an expected/target screenshot pair, span-strided
 * vector sampling and threshold classification into OK / SUSPICIOUS / ERROR.
 *
 * Every entry point cites the reference interface it replaces (paths relative to the
 * reference tree).  Plain pointers and sizes only; no exceptions cross this boundary
 * ("node-gyp can't use exceptions", src/opticalflow.h:16-19) -- errors are values.
 *
 * There is NO CPU fallback: every compute entry point fails with TW_CUDA_ERROR if no
 * sm_100-class device / kernel image is available.
 */
#ifndef TIDALWAVE_B200_H
#define TIDALWAVE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ErrorCode, src/opticalflow.h:9-14 (values 0..3 identical) + two additions. */
enum tw_error_code {
    TW_OK = 0,
    TW_BAD_PARAMETER = 1,
    TW_BAD_IMAGE_FORMAT = 2,
    TW_DONT_MATCH_SIZE = 3,
    TW_CUDA_ERROR = 4,   /* reason carries cudaGetErrorString */
    TW_UNSUPPORTED = 5   /* a documented gap (removed experimental options) */
};

/* Response.status, src/consumer.cpp:77,86 */
enum tw_status { TW_STATUS_OK = 0, TW_STATUS_SUSPICIOUS = 1, TW_STATUS_ERROR = 2 };

/* OpticalFlowParameter, src/opticalflow.h:28-36 -- field for field. */
typedef struct tw_flow_param {
    double pyrScale;
    int pyrLevels;
    int winSize;
    int pyrIterations;
    int polyN;
    double polySigma;
    int flags; /* 256 = OPTFLOW_FARNEBACK_GAUSSIAN, 0 = box window; anything else -> TW_BAD_PARAMETER */
} tw_flow_param;

/* Vector, src/message_queue.h:20-25 */
typedef struct tw_vector {
    int x;
    int y;
    double dx;
    double dy;
} tw_vector;

/* The value part of Response (src/message_queue.h:27-42) + OpticalFlowStatus (src/opticalflow.h:20-26). */
typedef struct tw_result {
    int code;       /* tw_error_code */
    int status;     /* tw_status */
    int n_vectors;  /* number of vectors that passed the threshold (may exceed the caller's cap) */
    int width;      /* of the expected image, src/opticalflow.cpp:72-73 */
    int height;
    float time;     /* seconds of device compute for this pair (src/opticalflow.cpp:82-93,112-118) */
    char reason[128];
} tw_result;

typedef struct tw_ctx tw_ctx;
typedef struct tw_pool tw_pool;

/* Fills *p with the defaults of Broker::createInstance (src/broker.cpp:106-117):
 * pyrScale .5, pyrLevels 3, winSize 30, pyrIterations 3, polyN 7, polySigma 1.5, flags 256. */
void tw_default_param(tw_flow_param *p);

/* Library / build information: "tidalwave_b200 <version> sm_100a". */
const char *tw_version(void);

/* Number of CUDA devices visible (cv::gpu::getCudaEnabledDeviceCount, src/consumer.cpp:19-20). */
int tw_device_count(void);

/* cv::imread(path, IMREAD_GRAYSCALE) on an in-memory file (src/opticalflow.cpp:37,44): PNG (every colour type and bit depth, Adam7
 * or not, critical-chunk CRCs checked; colour -> gray exactly as OpenCV/libpng: (9797 R + 19234 G + 3737 B) >> 15), JPEG (baseline / progressive Huffman, gray or YCbCr: the
 * luma plane through libjpeg's ISLOW inverse DCT, as OpenCV's JCS_GRAYSCALE request does; EXIF orientation ignored like
 * OpenCV 2.4.9) and binary PGM.  Host code, no device needed.  Call with out == NULL to query *w, *h.  Anything else ->
 * TW_BAD_IMAGE_FORMAT, reported by callers as "Can't open <path>". */
int tw_decode_gray(const uint8_t *bytes, size_t n, uint8_t *out, size_t cap, int *w, int *h);

/* ---- operator seam: OpticalFlow instance, one per consumer thread (src/consumer.cpp:27-35) ----
 * A context is thread-confined, bound to one device (cv::gpu::setDevice(id), src/consumer.cpp:22),
 * owns all device memory, pinned staging and its stream.  max_batch = pairs processed per launch
 * sequence by the batch entry points (>= 1).  Returns NULL and fills err on failure. */
tw_ctx *tw_create(int device, int max_w, int max_h, int max_batch, char *err, int errlen);
void tw_destroy(tw_ctx *ctx);

/* OpticalFlow::calculateInternal (src/opticalflow.h:49, src/opticalflow.cpp:78-119):
 * equal-size 8-bit gray images in, two float planes out (either may be NULL), *seconds = device
 * compute time (uploads/downloads excluded, as in src/opticalflow.cpp:112-116).  flowx/flowy are
 * w*h floats, row-major, tightly packed.  Returns a tw_error_code. */
int tw_flow(tw_ctx *ctx, const uint8_t *expect, const uint8_t *target, int w, int h, int stride,
            const tw_flow_param *param, float *flowx, float *flowy, float *seconds);

/* OpticalFlow::calculate (src/opticalflow.cpp:20-76) from decoded images + the sampling loop of
 * Consumer::run (src/consumer.cpp:59-88).  Size rule of src/opticalflow.cpp:52-68: |dw|>5 or |dh|>5 ->
 * TW_DONT_MATCH_SIZE; unequal within 5 px -> target bilinearly resized to the expected size.
 * Vectors are written in row-major scan order (y outer, x inner); at most cap are stored,
 * res->n_vectors is the full count.  NULL / empty images -> TW_BAD_IMAGE_FORMAT.  Returns res->code. */
int tw_compare(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw, int th,
               const tw_flow_param *param, double threshold, int span, tw_vector *out, int cap,
               tw_result *res);

/* The resize step of OpticalFlow::calculate alone (src/opticalflow.cpp:64-68, cv::resize INTER_LINEAR on 8-bit data), for
 * hosts that keep calculate() / calculateInternal() separate: target (tw x th) -> out (ew x eh), tightly packed. */
int tw_resize_target(tw_ctx *ctx, const uint8_t *target, int tw, int th, uint8_t *out, int ew, int eh);

/* n same-size pairs through one batched launch sequence (n <= max_batch).  out has n*cap entries
 * (pair i at out + i*cap), res has n entries.  Semantics per pair identical to tw_compare. */
int tw_compare_batch(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w,
                     int h, int stride, const tw_flow_param *param, double threshold, int span,
                     tw_vector *out, int cap, tw_result *res);

/* ---- pipelined form of tw_compare_batch (what a dispatcher consumer uses: ONE host thread keeps its GPU busy, as the
 * reference's Consumer does with its device, src/consumer.cpp:18-24, 42-94).  tw_pipe_submit enqueues a batch and returns:
 * the host -> device copies run on a copy stream through a staging buffer (overlapping the previous batch's kernels), the
 * compute stream takes them over, runs the launch sequence and snapshots the compact results.  tw_pipe_collect waits for the
 * OLDEST submitted batch and fills res[0..n) / out exactly as tw_compare_batch does (n = that batch's size).  At most two batches
 * are in flight (tw_pipe_pending); the images of a submitted batch must stay valid until it has been collected; a change of
 * size or parameters needs an empty pipe (TW_BAD_PARAMETER otherwise).  Not to be interleaved with the synchronous entry
 * points while batches are pending. */
int tw_pipe_submit(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h, int stride,
                   const tw_flow_param *param, double threshold, int span);
int tw_pipe_collect(tw_ctx *ctx, tw_vector *out, int cap, tw_result *res);
int tw_pipe_pending(tw_ctx *ctx);
/* 1 if the oldest pending batch has finished on the device (tw_pipe_collect would not block), else 0. */
int tw_pipe_ready(tw_ctx *ctx);

/* ---- ignore regions: leave chosen rectangles of a page out of a comparison (clocks, ads, carousels, avatars, build numbers) ----
 * A region is a rectangle in EXPECTED-image pixels, [x, x + width) x [y, y + height); a pair has 0 .. TW_MAX_IGNORE of them.
 * For a pair with regions:
 *   1. before any flow work, every target pixel inside a region is replaced by the expected pixel at the same position (after the
 *      +-5 px resize of the target); the flow is the ordinary flow of (expected, painted target), by the same kernels and arithmetic;
 *   2. a sample point (x, y) of the span grid inside any region yields no vector and does not count toward n_vectors or the status.
 * So the result equals the plain compare of (expected, painted target) minus the vectors inside the regions, bit for bit.
 * Regions are clipped to the frame (one entirely outside changes nothing); width < 1, height < 1, more than TW_MAX_IGNORE regions or
 * a NULL list with a count > 0 answer TW_BAD_PARAMETER with the reason "bad ignore region: ...".  With no regions on any pair the
 * *_ignore entry points are exactly their plain counterparts (same kernels, same results).  The result shapes do not change. */
#define TW_MAX_IGNORE 32
typedef struct tw_rect {
    int x, y, width, height; /* expected-image pixels */
} tw_rect;

/* tw_compare with ignore regions (ignore may be NULL when n_ignore == 0). */
int tw_compare_ignore(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw, int th,
                      const tw_flow_param *param, double threshold, int span, const tw_rect *ignore, int n_ignore,
                      tw_vector *out, int cap, tw_result *res);
/* tw_compare_batch with a region list per pair: pair i has n_ignore[i] regions at ignore[i].  n_ignore == NULL: no regions. */
int tw_compare_batch_ignore(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h,
                            int stride, const tw_flow_param *param, double threshold, int span,
                            const tw_rect *const *ignore, const int *n_ignore, tw_vector *out, int cap, tw_result *res);
/* tw_pipe_submit with a region list per pair (as tw_compare_batch_ignore).  The lists are copied before the call returns; they
 * travel with the batch, so the next batch's lists do not disturb one in flight.  Collect with tw_pipe_collect. */
int tw_pipe_submit_ignore(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h,
                          int stride, const tw_flow_param *param, double threshold, int span,
                          const tw_rect *const *ignore, const int *n_ignore);

/* ---- ignore masks: leave chosen pixels of a page out of a comparison (a timestamp on every row of a feed, round avatars, shapes
 * that are not rectangles, "dynamic element" masks rendered by the capture tool) ----
 * A mask is an 8-bit plane the size of the EXPECTED image, in expected-image pixels like a region; nonzero means ignore.
 * For a pair with a mask:
 *   1. after the +-5 px resize of the target and before any flow work, every target pixel whose mask byte is nonzero is replaced by
 *      the expected pixel at the same position;
 *   2. a sample point (x, y) of the span grid whose mask byte is nonzero yields no vector and does not count toward n_vectors or the
 *      status.
 * A pair can have a mask, regions, both or neither; with both, the ignored set is their union.  So the result equals the plain
 * compare of (expected, painted target) minus the vectors at ignored points, bit for bit.  A mask that is the rasterisation of a
 * region list gives exactly the result of that list; an all-zero mask gives exactly the plain result.  A mask whose size differs
 * from the expected image's (also when the target is resized: the mask follows the expected size) answers TW_BAD_PARAMETER with
 * the reason "bad ignore mask: <mw>x<mh> mask for a <ew>x<eh> expected image" where the size is known (the pool's mask files, the
 * Python binding); here the size is implied.  A NULL mask means "no mask".  With no mask on any pair the *_mask entry points are
 * exactly their *_ignore counterparts (same kernels, same results). */

/* tw_compare_ignore with an ignore mask: ew x eh bytes, tightly packed like expect; may be NULL. */
int tw_compare_mask(tw_ctx *ctx, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw, int th,
                    const tw_flow_param *param, double threshold, int span, const tw_rect *ignore, int n_ignore,
                    const uint8_t *mask, tw_vector *out, int cap, tw_result *res);
/* tw_compare_batch_ignore with a mask per pair: pair i's mask is mask[i] (w x h bytes, rows `stride` apart like the images).
 * mask == NULL: no masks; mask[i] == NULL: pair i has none. */
int tw_compare_batch_mask(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h,
                          int stride, const tw_flow_param *param, double threshold, int span,
                          const tw_rect *const *ignore, const int *n_ignore, const uint8_t *const *mask, tw_vector *out,
                          int cap, tw_result *res);
/* tw_pipe_submit_ignore with a mask per pair (as tw_compare_batch_mask).  The masks must stay valid until the batch has been
 * collected, like its images; they travel with the batch, so the next batch's masks do not disturb one in flight.  The staging
 * buffer grows to hold mask planes on the first masked batch (waiting for the batch in flight to take its images over); batches
 * with and without masks alternate freely. */
int tw_pipe_submit_mask(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w, int h,
                        int stride, const tw_flow_param *param, double threshold, int span,
                        const tw_rect *const *ignore, const int *n_ignore, const uint8_t *const *mask);

/* ---- change regions: where a page changed, as connected groups of its suspicious sample points (option "change_regions") ----
 * Grid: the sample points are (i * span, j * span) for 0 <= i < ceil(W / span), 0 <= j < ceil(H / span), in EXPECTED-image pixels
 * (after the +-5 px resize, as for vectors).  A point is suspicious when it yields a vector.  Points under ignore regions or masks
 * yield none, so they belong to no region and do not connect regions: a mask stripe through a changed area splits it in two.
 * Connectivity: two suspicious points are connected when their grid indices differ by at most 1 on each axis (8-connectivity); a
 * change region is a connected component.  Per region:
 *   rect       the bounding box of the span cells its points stand for: point (x, y) stands for [x, min(x + span, W)) x
 *              [y, min(y + span, H)), so rect = (min x, min y, min(max x + span, W) - min x, min(max y + span, H) - min y);
 *   n_vectors  the number of its points;
 *   peak       its vector (x, y, dx, dy as in the vector list) with the largest len = f32(f32(dx * dx) + f32(dy * dy)), the value
 *              the classification computes; a tie goes to the earlier point in scan order.
 * Order: by first point in row-major scan order (the order of their first vectors in the vector list), which is the label order of
 * scipy.ndimage.label(grid, structure=np.ones((3, 3))).  n_regions is always the full count; the first TW_MAX_CHANGE_REGIONS in
 * that order are stored.  Sum of n_vectors over the regions == tw_result.n_vectors whenever n_regions <= TW_MAX_CHANGE_REGIONS.
 * OK pairs, ERROR pairs and runs with span <= 0 have 0 regions.  Regions do not depend on the caller's vector cap: they are labelled
 * on the device from the full vector list.  The output is a function of the vector set alone: eager runs and graph replays, the
 * dense and sparse last iteration, the window kernels and both arithmetics (wherever their vectors agree) give identical bytes.
 * The rect is an ignore region's type: accepting a change for the next run is a copy of it into the pair's ignore list. */
#define TW_MAX_CHANGE_REGIONS 1024
typedef struct tw_change_region {
    tw_rect rect;      /* expected-image pixels, the same type as an ignore region */
    int n_vectors;
    tw_vector peak;    /* offset 24; sizeof 48 on LP64 */
} tw_change_region;

/* The change regions of pair `pair` of the batch that the last tw_compare*, tw_batch_fetch or tw_pipe_collect answered (those calls
 * copy them to the host when "change_regions" was 1 for that batch): min(cap, n_regions, TW_MAX_CHANGE_REGIONS) entries to out
 * (out may be NULL when cap is 0), the full count to *n_regions.  TW_BAD_PARAMETER if that batch ran without the option or pair is
 * out of range.  Set the option with tw_set_option(ctx, "change_regions", 1); it is refused while pipe batches are pending. */
int tw_change_regions(tw_ctx *ctx, int pair, tw_change_region *out, int cap, int *n_regions);

/* ---- intensity cells: where a page's pixels changed without moving, per span cell (option "intensity_threshold" = t) ----
 * The flow only sees structure that moves: a block darkened in place, a button re-coloured or a label erased leaves it at 0 and
 * the pair OK.  With t in 1 .. 255 gray levels, every run with span > 0 also tests each span cell for a change in place:
 *   cells      cell (i, j) has its sample point at (x, y) = (i * span, j * span) and covers [x, min(x + span, W)) x
 *              [y, min(y + span, H)) in EXPECTED-image pixels: the grid and cells of change regions.  E is the expected image,
 *              T the target after the +-5 px resize and after ignore painting -- the pair the flow was computed on;
 *   shift      (dx, dy) is the float flow at the cell's sample point (the value the classification reads);
 *              sx = rint(clamp(dx, -W, W)), sy = rint(clamp(dy, -H, H)), rounding half to even; a non-finite component is 0;
 *   residual   for a pixel p = (px, py) of the cell, r(p) = min over u, v in {-1, 0, 1} of
 *              |E(p) - T(clamp(px + sx + u, 0, W - 1), clamp(py + sy + v, 0, H - 1))|, an integer: the integer shift absorbs the
 *              motion the flow found, the 3 x 3 minimum its sub-pixel remainder and anti-aliasing;
 *   test       n = the cell's pixels not ignored (under no ignore region and no nonzero mask byte), S = the sum of r over them.
 *              The cell is an intensity cell when n > 0 and S > t * n (strict, as the vector rule).  Integer arithmetic
 *              throughout: exact and order-free.
 * A pair with at least one intensity cell is SUSPICIOUS even with 0 vectors; n_vectors, the vectors and the change regions do not
 * change (regions describe vectors only).  ERROR pairs and runs with span <= 0 have 0 cells.  n_cells is always the full count;
 * the first TW_MAX_INTENSITY_CELLS in row-major scan order are stored.  The output is a function of (E, T, the flow at the sample
 * points, the ignored set) alone: eager runs and graph replays, the dense and sparse last iteration and the tile and strip window
 * kernels (which write bit-identical sample-point flows) give identical bytes. */
#define TW_MAX_INTENSITY_CELLS 4096
typedef struct tw_intensity_cell {
    int x, y;       /* the cell's sample point, expected-image pixels */
    int n_pixels;   /* n */
    int residual;   /* S (the mean residual is S / n); saturates at INT_MAX, which only a cell of more than 8 421 504 pixels reaches */
} tw_intensity_cell;

/* The intensity cells of pair `pair` of the batch that the last tw_compare*, tw_batch_fetch or tw_pipe_collect answered (copied to
 * the host when "intensity_threshold" was on for that batch): min(cap, n_cells, TW_MAX_INTENSITY_CELLS) entries to out (out may be
 * NULL when cap is 0), the full count to *n_cells.  TW_BAD_PARAMETER if that batch ran without the option or pair is out of range. */
int tw_intensity_cells(tw_ctx *ctx, int pair, tw_intensity_cell *out, int cap, int *n_cells);

/* ---- split phases of tw_compare_batch (same stream; used by the dispatcher to overlap, and by the
 * benchmark to time the device-resident pass separately from the PCIe legs).  They take no ignore regions and no ignore masks:
 * painting changes the resident target, so only the whole-call entry points above apply them.  tw_batch_flow after a run with
 * regions or masks returns the flow of the painted pair. ---- */
int tw_batch_upload(tw_ctx *ctx, int n, const uint8_t *const *expect, const uint8_t *const *target, int w,
                    int h, int stride);                                     /* async H2D into the context */
int tw_batch_run(tw_ctx *ctx, int n, int w, int h, const tw_flow_param *param, double threshold,
                 int span);                                                  /* enqueue all kernels, no sync */
int tw_batch_fetch(tw_ctx *ctx, int n, tw_vector *out, int cap, tw_result *res); /* D2H compact results + sync */
int tw_sync(tw_ctx *ctx);
/* Copies the dense flow planes of pair `pair` of the last run back (either pointer may be NULL); TW_BAD_PARAMETER if that run
 * was classification-only ("sparse_last"). */
int tw_batch_flow(tw_ctx *ctx, int pair, float *flowx, float *flowy);
const char *tw_last_error(tw_ctx *ctx);
/* Per-context options.
 *   "arithmetic" = 0: every kernel keeps the oracle's operation order (SURVEY App. A): results bit-identical to
 *                     oracle/farneback_ref.c on every configuration.
 *                = 1 (default; TW_ARITHMETIC=faithful in the environment or tw_set_default_arithmetic(0) flips it):
 *                     relaxed arithmetic where it was validated -- Gaussian window (flags 256) with winSize >= 30 and
 *                     polyN 7, i.e. the reference's default option family: direct-form fmaf window taps and a mixed
 *                     double / float horizontal pass in the polynomial expansion (restated bit for bit in the oracle:
 *                     twref_set_relax(144)).  Measured against the faithful oracle and cv2: <= 1.5e-4 px at 1920x1080,
 *                     2.3e-3 px max / 1.3e-4 px RMS on the reference's fixture, identical status and vector sets (bar:
 *                     1e-2 px max, 1e-3 px RMS; tools/relax_cases.py, tools/parity_report.py).  Every other option set
 *                     (box window, smaller windows, polyN != 7) runs the faithful kernels.
 *   "sparse_last" = 1: classification only -- the last iteration of the finest scale evaluates the window blur and the solve
 *                     only at the positions src/consumer.cpp:60-77 samples (Gaussian window of radius 15 / 7, span > 0).  Status
 *                     and vectors (positions and the float dx, dy) are bit-identical to the dense path; the dense flow field
 *                     is not produced (tw_batch_flow fails after such a run; tw_flow is always dense).  Default 0 for
 *                     tw_create, 1 for the dispatcher's contexts (tw_pool_*; TW_SPARSE_LAST=0 turns it off there).
 *   "graph"      = 1 (default): repeated runs of one (size, batch, options) replay a captured CUDA graph.
 *   "gauss_fma", "update_fma", "gauss_scalar": removed in round 2 (studied and rejected relaxations -- oracle relax bits 0 / 6 --
 *                     and the scalar v1 window kernel); setting one to 1 answers TW_UNSUPPORTED.
 *   "window_tiles" = 1 (default) / 0: the Gaussian window iterations of radius 15 run the tile-per-CTA kernel / the persistent
 *                     warp-specialised strip kernel (tw_window.cu: TMA tensor-map rings, register-resident column walkers,
 *                     setmaxnreg).  Same arithmetic, bit-identical results; the strip kernel measures 1-7 % slower (DESIGN.md
 *                     section 4.2), so it is opt-in; TW_WINDOW=strip|tiles in the environment sets the default.
 *   "plan_cache" = n (default 3; TW_PLAN_CACHE): plans -- the device buffers, tables, tensor maps and the captured graph of one
 *                     (size, parameters) -- kept besides the current one, least recently used evicted first, all dropped when
 *                     memory runs out: a dispatcher that sees mixed page sizes does not rebuild a plan on every switch.
 *   "polyexp_tma" = 1: interior input tiles of the relaxed polynomial expansion are staged by one TMA tensor-map copy instead of
 *                     per-thread loads (bit-identical; measured 5 % slower, hence opt-in; TW_POLY_TMA=1 sets the default).
 *   "level_generic", "level_unfused", "tight_pitch", "box_unfused": alternative code paths (also the fall-backs of unusual
 *                     options) that the parity tests force.
 *   "change_regions" = 1: each run with span > 0 also groups every pair's vectors into change regions on the device (one more
 *                     launch, after the sample kernel; tw_change_regions reads them).  Default 0.  TW_BAD_PARAMETER while pipe
 *                     batches are pending.
 *   "intensity_threshold" = t: 0 (default) off; 1 .. 255: each run with span > 0 also finds every pair's intensity cells (three more
 *                     launches after the sample kernel; tw_intensity_cells reads them) and counts them toward the status.  Any
 *                     other value, or a change while pipe batches are pending, answers TW_BAD_PARAMETER. */
int tw_set_option(tw_ctx *ctx, const char *name, int value);
/* Process-wide default of "arithmetic" for contexts created afterwards (the dispatcher's consumers included). */
int tw_set_default_arithmetic(int relaxed);
/* 1 if `param` would run the relaxed kernels on this context, 0 if the faithful ones, <0 on bad arguments. */
int tw_arithmetic_in_effect(tw_ctx *ctx, const tw_flow_param *param);

/* Pinned (page-locked) host memory for image buffers: H2D copies from it are true async DMA. */
void *tw_host_alloc(size_t bytes);
void tw_host_free(void *p);

/* ---- measurement hooks (CUDA events on the context's own stream) ---- */
/* Enqueues a write of a >L2 (256 MB) scratch buffer on the context's stream, evicting L2 between timed steps. */
int tw_l2_flush(tw_ctx *ctx);
int tw_timer_start(tw_ctx *ctx);
int tw_timer_stop(tw_ctx *ctx, float *ms);       /* records, synchronises, returns elapsed ms */
/* Per-kernel-family event timing: enable, run, then read n families back.  names[i] points to a static
 * string; ms[i] is the summed device time, launches[i] the launch count and alg_bytes[i] the ALGORITHMIC HBM
 * bytes (DESIGN.md section 4: the family's term of B_alg) since enable/reset.  Returns the family count. */
int tw_profile_enable(tw_ctx *ctx, int on);
int tw_profile_read(tw_ctx *ctx, int max_n, const char **names, float *ms, int *launches, double *alg_bytes);
/* Number of kernel launches issued by this context since creation. */
long long tw_launch_count(tw_ctx *ctx);

/* ---- per-stage read-back for parity tests (planar float, c*h*w): name in
 * {"I","R0","R1","M","flow"}, scale = index in the coarse->fine schedule, pair < n of the last run.
 * Returns channel count written, <0 on error; *w,*h receive the plane size.  "M" holds whatever the last
 * kernel that wrote it left (run with pyrIterations = k to observe iteration k-1's input). ---- */
int tw_debug_read(tw_ctx *ctx, const char *name, int scale, int pair, float *out, int cap_floats, int *w, int *h);
int tw_debug_keep_levels(tw_ctx *ctx, int on); /* keep every scale's I/R/M (separate buffers) for read-back */

/* ---- dispatcher: Manager + Consumer pool (src/manager.cpp:40-98, src/consumer.cpp:12-94) ----
 * One host thread per entry of devices[] (consumer i binds GPU devices[i]), all blocking on one shared
 * request queue; options are fixed per pool (src/manager.cpp:72-73).  Images are caller-owned and must
 * stay valid until the result for that id has been taken.  No CPU fallback worker.
 * vector_cap > 0: at most that many vectors are kept per request (tw_result.n_vectors still holds the full count);
 * vector_cap == 0: all of them, whatever the image size (capacity = the request's own sampling grid).
 * max_w / max_h > 0 bound the image size a consumer accepts (larger requests answer TW_BAD_PARAMETER); 0 = no bound. */
tw_pool *tw_pool_create(const int *devices, int n_devices, int max_w, int max_h, int batch,
                        const tw_flow_param *param, double threshold, int span, int vector_cap,
                        char *err, int errlen);
/* Manager::request (src/manager.cpp:68-78): returns the request id (>= 0) or <0 if the pool is stopped. */
long long tw_pool_submit(tw_pool *pool, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw,
                         int th);
/* Manager::request exactly as the reference has it (src/manager.cpp:68-78, Request = two paths, src/message_queue.h:13-18): the
 * files are read and decoded -- cv::imread(IMREAD_GRAYSCALE), src/opticalflow.cpp:37,44 -> tw_decode_gray -- on the pool's decoder
 * threads (started on first use: one per host core, at most 32; tw_pool_set_decoders before the first call changes that), then join
 * the same request queue.  Empty path -> TW_BAD_PARAMETER, unreadable / undecodable file -> TW_BAD_IMAGE_FORMAT "Can't open <path>"
 * (src/opticalflow.cpp:20-49), sizes more than 5 px apart -> TW_DONT_MATCH_SIZE.  The pool owns the decoded images. */
long long tw_pool_submit_files(tw_pool *pool, const char *expect_path, const char *target_path);
/* The two submits with ignore regions (see tw_compare_ignore).  The list is copied at submit time.  A bad list answers that request
 * alone with TW_BAD_PARAMETER "bad ignore region: ..."; requests with and without regions share batches. */
long long tw_pool_submit_ignore(tw_pool *pool, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw, int th,
                                const tw_rect *ignore, int n_ignore);
long long tw_pool_submit_files_ignore(tw_pool *pool, const char *expect_path, const char *target_path,
                                      const tw_rect *ignore, int n_ignore);
/* The two submits with ignore regions and an ignore mask (see tw_compare_mask).  tw_pool_submit_mask: the mask (ew x eh bytes,
 * or NULL) is caller-owned and must stay valid until the result has been taken, like the images.  tw_pool_submit_files_mask: the
 * mask file (NULL or "": none) is read and decoded on the decoder threads with the two images, by tw_decode_gray, so it is a gray
 * value: colour is converted as for the images and alpha is dropped.  A mask file that cannot be read or decoded answers that
 * request alone with TW_BAD_IMAGE_FORMAT "Can't open <mask path>", one of another size than the expected image with
 * TW_BAD_PARAMETER "bad ignore mask: ...".  Requests with masks, regions, both or neither share batches. */
long long tw_pool_submit_mask(tw_pool *pool, const uint8_t *expect, int ew, int eh, const uint8_t *target, int tw, int th,
                              const tw_rect *ignore, int n_ignore, const uint8_t *mask);
long long tw_pool_submit_files_mask(tw_pool *pool, const char *expect_path, const char *target_path, const char *mask_path,
                                    const tw_rect *ignore, int n_ignore);
int tw_pool_set_decoders(tw_pool *pool, int n);
/* on = 1: every consumer runs with "change_regions" and keeps each request's regions (tw_pool_wait_regions), whatever vector_cap
 * is.  Valid before the first submit (TW_OK), TW_BAD_PARAMETER after. */
int tw_pool_set_change_regions(tw_pool *pool, int on);
/* t = 1 .. 255: every consumer runs with "intensity_threshold" = t and keeps each request's intensity cells
 * (tw_pool_wait_intensity); 0: off.  Valid before the first submit (TW_OK); TW_BAD_PARAMETER after, and for t outside 0 .. 255. */
int tw_pool_set_intensity(tw_pool *pool, int t);
/* Blocks until request `id` is answered; copies up to cap vectors.  Returns res->code, or <0 if dropped. */
int tw_pool_wait(tw_pool *pool, long long id, tw_vector *out, int cap, tw_result *res);
/* tw_pool_wait plus the request's change regions: up to region_cap of them to regions, the full count to *n_regions (0 for an
 * ERROR request and for a pool without change regions). */
int tw_pool_wait_regions(tw_pool *pool, long long id, tw_vector *out, int cap, tw_result *res, tw_change_region *regions,
                         int region_cap, int *n_regions);
/* tw_pool_wait_regions plus the request's intensity cells: up to cell_cap of them to cells, the full count to *n_cells (0 for an
 * ERROR request and for a pool without the option).  regions / n_regions may be NULL and region_cap 0. */
int tw_pool_wait_intensity(tw_pool *pool, long long id, tw_vector *out, int cap, tw_result *res, tw_change_region *regions,
                           int region_cap, int *n_regions, tw_intensity_cell *cells, int cell_cap, int *n_cells);
/* Blocks until request `id` is answered and copies its result WITHOUT taking it (res->n_vectors = the room tw_pool_wait needs).
 * Returns res->code, or <0 if dropped / unknown. */
int tw_pool_peek(tw_pool *pool, long long id, tw_result *res);
/* Non-blocking: 1 if answered (result copied), 0 if pending, <0 if dropped/unknown. */
int tw_pool_poll(tw_pool *pool, long long id, tw_vector *out, int cap, tw_result *res);
/* Report, src/message_queue.h:44-48: {request, data, error}. */
void tw_pool_report(tw_pool *pool, int *request_count, int *data_count, int *error_count);
/* Manager::stop (src/manager.cpp:63-66,93-97): drops pending requests, joins the consumers. */
void tw_pool_stop(tw_pool *pool);
void tw_pool_destroy(tw_pool *pool);

#ifdef __cplusplus
}
#endif
#endif /* TIDALWAVE_B200_H */
