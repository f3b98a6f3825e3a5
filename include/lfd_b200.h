/* lfd_b200.h - C ABI of the B200-native lfd.detecttrails per-frame detection library.
 *
 * The reference (DinoBektesevic/lfd) is pure Python and has no FFI for this path; its boundary
 * is the set of Python call signatures listed below.  Each entry point here replaces the device-
 * worthy part of one of them and is what a reference-side ctypes stub binds (INTEGRATION.md).
 * Paths are relative to /root/reference/.
 *
 *   lfd_submit + lfd_wait      replaces the body of process_field()
 *                                lfd/detecttrails/detecttrails.py:119-131
 *                              = remove_stars blot      lfd/detecttrails/removestars.py:231
 *                              + cv2.flip(img, 0)       lfd/detecttrails/detecttrails.py:124
 *                              + process_field_bright   lfd/detecttrails/processfield.py:291-388
 *                              + process_field_dim      lfd/detecttrails/processfield.py:391-506
 *   lfd_run_pass               one of process_field_bright / process_field_dim on an already
 *                              flipped frame (their public, directly callable form,
 *                              processfield.py:15 __all__), optional in-place write-back of the
 *                              clipped float image (processfield.py:342, :453-454)
 *   lfd_blot                   remove_stars' in-place square fill, removestars.py:231
 *   lfd_get_stage              the debug taps of processfield.py:349-378, :459-496 as raw arrays
 *   lfd_hough_lines            cv2.HoughLines(img, rho, theta, threshold) as called at
 *                              processfield.py:370-371, :488-489 (also the config-5 microbench)
 *   lfd_set_params             the params_bright / params_dim dicts,
 *                              lfd/detecttrails/detecttrails.py:202-230
 *
 * Conventions: every call returns 0 on success or a negative LFD_E_* code; lfd_last_error()
 * gives the text.  The caller owns all host buffers; the library owns all device memory and
 * streams.  A handle is bound to one GPU and is not thread-safe (one handle per host worker).
 * No C++ types and no exceptions cross this boundary.  There is no CPU fallback: without a
 * CUDA device lfd_create fails with LFD_E_CUDA.
 */
#ifndef LFD_B200_H
#define LFD_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFD_ABI_VERSION 1

/* error codes */
#define LFD_OK 0
#define LFD_E_ARG (-1)          /* bad argument */
#define LFD_E_CUDA (-2)         /* CUDA runtime error (text in lfd_last_error) */
#define LFD_E_UNSUPPORTED (-3)  /* legal reference parameter this build does not implement */
#define LFD_E_CAPACITY (-4)     /* a per-frame work list overflowed its configured capacity */
#define LFD_E_STATE (-5)        /* call order violated (e.g. wait without submit) */

/* per-frame status bits in lfd_result.status */
#define LFD_FRAME_OK 0
#define LFD_FRAME_OVERFLOW 1        /* run/component/peak list overflow: result invalid */
#define LFD_FRAME_NO_LINES_EQU 2    /* HoughLines(equ) returned no line: the reference raises TypeError */
#define LFD_FRAME_NO_LINES_BOX 4    /* HoughLines(box_img) returned no line: likewise */

/* passes */
#define LFD_PASS_BRIGHT 0
#define LFD_PASS_DIM 1

/* lfd_submit flags */
#define LFD_INPUT_NATIVE 0      /* host float32, native byte order (what fitsio.read returns) */
#define LFD_INPUT_BIGENDIAN 1   /* raw FITS payload: big-endian float32, byte-swapped on the device (lfd_submit,
                                   lfd_upload, lfd_run_resident; lfd_run_pass and lfd_submit_injected refuse it) */
#define LFD_KEEP_TAPS 2         /* materialise the uint8 stage images for lfd_get_stage */
#define LFD_FULL_LINES 4        /* sort and keep the full HoughLines lists (taps / parity) */
#define LFD_SERIAL_PASSES 8     /* run the dim pass after the bright pass on one stream (per-stage timings) */
#define LFD_KERNEL_TIMES 16     /* bracket the kernels that carry the step with CUDA events (lfd_get_kernel_times); the ~50
                                   extra event nodes cost about 5 % of a 64-frame step, so this is off by default */

/* stage ids for lfd_get_stage (uint8 H*W unless noted) */
enum lfd_stage {
    LFD_STAGE_MASK = 0,      /* star mask, 255 where blotted, in the flipped orientation */
    LFD_STAGE_GRAY = 1,      /* convertScaleAbs output          processfield.py:346,456 */
    LFD_STAGE_EQU = 2,       /* equalizeHist output             processfield.py:347,457 */
    LFD_STAGE_ERODED = 3,    /* erode output (dim only)         processfield.py:464     */
    LFD_STAGE_MORPH = 4,     /* dilate output = Canny/Hough input  processfield.py:354,471 */
    LFD_STAGE_CANNY = 5,     /* Canny(.,0,255)                  processfield.py:236     */
    LFD_STAGE_BOX = 6,       /* box_img                         processfield.py:235,261 */
    LFD_STAGE_HIST = 7,      /* uint32[256] histogram of GRAY */
    LFD_STAGE_LUT = 8,       /* uint8[256] equalisation LUT */
    LFD_STAGE_NMS = 9,       /* uint8 H*W: 0 none, 1 weak, 2 strong after non-maximum suppression */
    LFD_STAGE_FG_LABELS = 10,/* int32 H*W: raster-first pixel index of the 8-connected edge component, -1 elsewhere */
    LFD_STAGE_BG_LABELS = 11,/* int32 H*W: raster-first pixel index of the 4-connected hole, -2 outside background, -1 on edges */
    LFD_STAGE_RECTS = 12,    /* lfd_rect[n]; count via lfd_get_stage_count */
    LFD_STAGE_ACCUM_EQU = 13,/* int32 (numangle+2)*(numrho+2) Hough accumulator of MORPH */
    LFD_STAGE_ACCUM_BOX = 14,/* same for BOX */
    LFD_STAGE_LINES_EQU = 15,/* float32[n][2] (rho, theta) in cv2.HoughLines order; needs LFD_FULL_LINES; n via
                                lfd_get_stage_count: n_lines, capped at the handle's max_lines */
    LFD_STAGE_LINES_BOX = 16,
    LFD_STAGE_CLIPPED = 17,  /* float32 H*W: the frame after the pass's in-place clip (processfield.py:342,453-454) */
    LFD_STAGE_INPUT = 18,    /* float32 H*W: the un-flipped frame of a batch slot as the last whole-frame run read it, native
                                byte order (swapped back after an LFD_INPUT_BIGENDIAN run); needs no LFD_KEEP_TAPS; `pass` is
                                ignored.  LFD_E_STATE after lfd_run_pass / lfd_blot / a bare lfd_upload, which overwrite the slots */
    LFD_STAGE_RECT_SCREEN = 19 /* int32[n]: 1 where the aspect screen (DESIGN.md §7) rejected the contour, same order and
                                  count as LFD_STAGE_RECTS; recorded with and without LFD_KEEP_TAPS */
};

/* one pass's parameters: the keys of params_bright / params_dim (detecttrails.py:202-230) */
typedef struct lfd_pass_params {
    double lwTresh;
    double thetaTresh;
    double lineSetTresh;
    double dro;
    double minAreaRectMinLen;
    double houghMethod;         /* = rho of cv2.HoughLines (processfield.py:370) */
    double minFlux;             /* dim only */
    double addFlux;             /* dim only */
    int32_t nlinesInSet;        /* <= LFD_MAX_SET_LINES */
    int32_t contoursMode;       /* cv2.RETR_*: LIST(1), CCOMP(2), TREE(3) give the same contour set; EXTERNAL(0) = outermost outer borders only */
    int32_t contoursMethod;     /* cv2.CHAIN_APPROX_NONE(1) or SIMPLE(2) (same hulls); TC89_* unsupported */
    int32_t erode_h, erode_w;   /* 0,0 = no erosion (bright).  All-ones rectangles whose erode + dilate reach fits the
                                   rectangle kernels' halo (rows <= 16, columns <= 12 left / 11 right); any other
                                   element, up to 255 x 255: lfd_set_kernels. */
    int32_t dilate_h, dilate_w;
    int32_t reserved;
} lfd_pass_params;

typedef struct lfd_params {
    lfd_pass_params bright;
    lfd_pass_params dim;
} lfd_params;

#define LFD_MAX_SET_LINES 16

/* per-frame outcome of lfd_submit/lfd_wait or lfd_run_pass */
typedef struct lfd_result {
    int32_t detected;           /* 1 if a pass accepted a line */
    int32_t pass;               /* LFD_PASS_BRIGHT / LFD_PASS_DIM that detected, else -1 */
    int32_t status;             /* LFD_FRAME_* bits */
    int32_t rect_detection[2];  /* per pass: fit_minAreaRect's `detection` (processfield.py:258); -1 = pass not run */
    int32_t n_lines_equ[2];     /* per pass: len(HoughLines(equ)), -1 if Hough did not run */
    int32_t n_lines_box[2];
    int32_t rejected[2];        /* per pass: 1 if check_theta returned True (processfield.py:380,498) */
    float rho;                  /* equhough[0][0] of the detecting pass (processfield.py:384,502) */
    float theta;
    float top_equ[2][LFD_MAX_SET_LINES][2]; /* per pass: first nlinesInSet (rho,theta) of HoughLines(equ) */
    float top_box[2][LFD_MAX_SET_LINES][2];
} lfd_result;

/* a minimum-area rectangle as cv2.minAreaRect returns it (processfield.py:249) */
typedef struct lfd_rect {
    float cx, cy, w, h, angle;
    int32_t kind;               /* 0 = outer border of an edge component, 1 = hole border, 2 = not retrieved (RETR_EXTERNAL),
                                   3 = not fitted: its aspect bound (DESIGN.md §7) proves it cannot pass; only in runs without
                                   LFD_KEEP_TAPS, which fit every contour.  cx .. angle and box are 0, key is set */
    int32_t key;                /* raster-first pixel index (y*W+x) of the component / hole */
    int32_t passed;             /* 1 if it passed the length/width filter (processfield.py:256-257) */
    int32_t box[8];             /* int32(boxPoints(rect)) x0,y0..x3,y3 (processfield.py:259-260); valid if passed */
} lfd_rect;

/* optional capacities for lfd_create_ex (0 = default) */
typedef struct lfd_config {
    int32_t max_runs;           /* runs per frame, pass and mask kind (default 1<<19, at most height * ceil(width/2)) */
    int32_t max_components;     /* contours per frame, pass and kind (default 1<<16) */
    int32_t max_star_rects;     /* blot squares per frame (default 8192) */
    int32_t max_lines;          /* HoughLines entries kept per frame in LFD_FULL_LINES mode (default numangle*numrho) */
    int32_t reserved[4];
} lfd_config;

/* one synthetic trail for lfd_submit_injected: the Gaussian line segment of lfd_b200/synth.py::_add_trail.  Pixel (x, y)
 * gets peak * expf(-0.5f * (d / sigma)^2) added iff 0 <= t <= L and |d| <= ceil(5 * sigma) + 1, with, in float32,
 * t = (x - x0) * ux + (y - y0) * uy, d = -(x - x0) * uy + (y - y0) * ux and ux, uy, L computed in double from the end
 * points and rounded to float32 (oracle/inject_ref.py::render_trails).  A zero-length trail adds nothing; the frame
 * edges clip the footprint. */
typedef struct lfd_trail {
    float x0, y0, x1, y1;   /* end points, UN-flipped FITS orientation, x = column, y = row, pixel centres at integers */
    float sigma;            /* Gaussian cross-section sigma in px, finite and > 0 */
    float peak;             /* added flux at the centre line, frame units, finite (may be negative) */
} lfd_trail;

#define LFD_MAX_INJECT_TRAILS 16   /* trails per batch slot */

/* Tabulated trail shapes for lfd_submit_injected_shaped: a pool of float32 samples that the handle owns, and tables that
 * name n samples of it, evenly spaced on [lo, hi] (samples[offset + i] at lo + i * (hi - lo) / (n - 1)).
 * A cross-section profile's abscissa is the signed distance d of lfd_trail; with p = the profile's samples:
 *   footprint 0 <= t <= L and lo <= d <= hi (asymmetric profiles are allowed)
 *   u = (d - lo) * inv, inv = (float)((n - 1) / ((double)hi - (double)lo)), i = min(trunc(u), n - 2), f = u - i
 *   P = p[i] + f * (p[i+1] - p[i])
 * A light curve a of m samples spans the segment from (x0, y0) at t = 0 to (x1, y1) at t = L (its lo and hi are not
 * used): v = t * c, c = (float)((m - 1) / (double)L), j = min(trunc(v), m - 2), g = v - j, A = a[j] + g * (a[j+1] - a[j]).
 * The pixel gets (peak * P) * A added, or peak * P without a light curve; every operation is one float32 round-to-nearest
 * step (tests/inject_shapes_ref.py::render_trails(..., tables) is bit-identical).  Profile -1 is lfd_trail's Gaussian (P =
 * expf(...), footprint |d| <= ceil(5 sigma) + 1) and light curve -1 is A = 1, so shapes of all -1 give
 * lfd_submit_injected's frames bit for bit.  `peak` is the flux at a sample value of 1; a tabulated profile ignores
 * `sigma` (it is not validated). */
typedef struct lfd_table {
    int32_t offset, n;      /* samples[offset .. offset + n) of the pool, 2 <= n <= LFD_MAX_TABLE_SAMPLES */
    float lo, hi;           /* finite, lo < hi, max(|lo|, |hi|) <= 1024 */
} lfd_table;

typedef struct lfd_trail_shape {
    int32_t profile;        /* table index of the cross-section profile, -1 = Gaussian of lfd_trail.sigma */
    int32_t lightcurve;     /* table index of the light curve, -1 = constant 1 */
} lfd_trail_shape;

#define LFD_MAX_TABLE_SAMPLES 4096
#define LFD_MAX_TRAIL_TABLES 4096

typedef struct lfd_handle lfd_handle;

int lfd_abi_version(void);

/* Create a handle on CUDA device `device` for batches of up to `max_batch` frames of height x width. */
int lfd_create(int device, int max_batch, int height, int width, lfd_handle** out);
int lfd_create_ex(int device, int max_batch, int height, int width, const lfd_config* cfg, lfd_handle** out);
int lfd_destroy(lfd_handle* h);
const char* lfd_last_error(const lfd_handle* h);   /* h may be NULL: error of the last failed lfd_create */

int lfd_set_params(lfd_handle* h, const lfd_params* p);

/* Multi-GPU nodes: share a host->device copy slot with other processes.  `lock_path` names an advisory lock file; the
 * handle takes the lock (waiting at most 250 ms) before it enqueues a batch's H2D copy in lfd_submit / lfd_upload and a
 * stream callback releases it when the copy has completed, so at most one of the handles naming the same file copies at a
 * time.  With several GPUs behind one PCIe host bridge this makes the bridge's bandwidth shares equal (the Python driver
 * and bench.py name two slots per bridge when more than two ranks share one: lfd_b200/sharding.py::h2d_gate_path).
 * NULL or "" removes the gate.  The reference has no counterpart (its scale-out is one PBS job per run,
 * lfd/createjobs/createjobs.py:173-218). */
int lfd_set_h2d_gate(lfd_handle* h, const char* lock_path);

/* Flat structuring elements of any shape (cv2.getStructuringElement crosses / ellipses, rings, hand-made masks, and
 * all-ones rectangles past the rectangle kernels' halo), for one pass: row-major uint8 masks, non-zero = member, any
 * parity, cv2's default anchor (kw/2, kh/2) whether or not it is a member, sides 1..255 (larger: LFD_E_UNSUPPORTED; a
 * mask without a member: LFD_E_ARG).  Semantics of cv2.erode / cv2.dilate with the default border: out-of-frame samples
 * are ignored, also in frames smaller than the element; the erosion (dim pass only) runs first.  Evaluated by chord
 * decomposition (DESIGN.md §3): the cost per pixel grows with the element's rows and runs, not with its area.
 * Call after lfd_set_params (which resets both passes to the all-ones rectangles of lfd_pass_params).
 * erode_mask may be NULL (no erosion; always ignored for the bright pass, processfield.py:354). */
int lfd_set_kernels(lfd_handle* h, int pass, const uint8_t* erode_mask, int erode_h, int erode_w,
                    const uint8_t* dilate_mask, int dilate_h, int dilate_w);

/* Pinned host staging owned by the library (frames in, `max_batch` slots of height*width float32). */
int lfd_host_frames(lfd_handle* h, float** out);

/* Whole-frame path.  `frames`: n un-flipped float32 frames (FITS orientation), contiguous; pass NULL to use
 * the library's own pinned staging (lfd_host_frames).  `rects`: blot squares as (row_start,row_stop,col_start,
 * col_stop) half-open quadruples on the UN-flipped image, already resolved by the host to Python slice
 * semantics (removestars.py:231); rect_offsets[n+1] indexes them per frame.  Asynchronous. */
int lfd_submit(lfd_handle* h, const float* frames, int n, const int32_t* rects, const int32_t* rect_offsets, int flags);
int lfd_wait(lfd_handle* h, lfd_result* out /* n entries */);

/* Device-resident variant used by the benchmark's `value` leg: runs the same pipeline on the frames
 * uploaded by the previous lfd_submit/lfd_upload without any host<->device copy of pixel data. */
int lfd_upload(lfd_handle* h, const float* frames, int n, const int32_t* rects, const int32_t* rect_offsets, int flags);
/* After lfd_submit_injected it re-runs the injected frames (they stay in the batch slots). */
int lfd_run_resident(lfd_handle* h, int n, int flags);

/* Injection and recovery (measuring what fraction of synthetic trails the detector finds).
 * lfd_set_base uploads n_base native-order, un-flipped frames once into device memory the handle owns; their star
 * rectangles follow lfd_submit's convention and max_star_rects check and are kept on the host.  A second call replaces
 * the bases.  LFD_E_STATE while a batch is pending.
 * lfd_submit_injected runs slot f on base_index[f] plus trails[trail_offsets[f] .. trail_offsets[f+1]) (trails and
 * trail_offsets may both be NULL: no trails), with that base's rectangles: the trails are added on the device by
 * k_inject just before the pipeline, so no pixel data crosses the host link.  It takes lfd_submit's flags except
 * LFD_INPUT_BIGENDIAN; collect with lfd_wait.  LFD_E_ARG with nothing launched when n is outside 1..max_batch, a base
 * index is out of range, a slot has more than LFD_MAX_INJECT_TRAILS trails, or a trail value is not finite or
 * sigma <= 0; LFD_E_STATE when no base has been set.  k_inject's duration is lfd_get_kernel_times index 14. */
int lfd_set_base(lfd_handle* h, const float* frames, int n_base, const int32_t* rects, const int32_t* rect_offsets);
/* Make the n frames of the last collected whole-frame batch (lfd_submit, or lfd_upload + lfd_run_resident) the handle's
 * injection bases, without any host<->device copy: base b = batch slot b in native byte order (byte-swapped on the device
 * when that batch was LFD_INPUT_BIGENDIAN), with the star rectangles that batch was submitted with.  Replaces the bases
 * like lfd_set_base.  LFD_E_STATE, with nothing launched, while a batch is pending, before any whole-frame batch, and when
 * the slots no longer hold that batch's input (after lfd_run_pass, lfd_blot, lfd_submit_injected[_shaped], and
 * lfd_run_resident of injected frames).  Asynchronous: the copy, k_capture_bases, runs on the handle's stream ahead of the
 * next lfd_submit_injected; its duration is lfd_get_kernel_times index 15 of the next collected batch.  A drop-in run
 * can so measure completeness on every frame it reads, at the cost of one device copy per batch. */
int lfd_capture_bases(lfd_handle* h);
int lfd_submit_injected(lfd_handle* h, int n, const int32_t* base_index, const lfd_trail* trails,
                        const int32_t* trail_offsets, int flags);
/* lfd_set_trail_tables uploads the pool of tabulated shapes (lfd_table) once, synchronously; a second call replaces it.
 * LFD_E_STATE while a batch is pending; LFD_E_ARG when n_tables is outside 1..LFD_MAX_TRAIL_TABLES, a table's n is
 * outside 2..LFD_MAX_TABLE_SAMPLES or it lies outside samples[0 .. n_samples), a sample, lo or hi is not finite,
 * lo >= hi, or max(|lo|, |hi|) > 1024.
 * lfd_submit_injected_shaped is lfd_submit_injected with one shapes entry per trail (NULL = all -1, which is
 * lfd_submit_injected).  Beyond lfd_submit_injected's checks: LFD_E_ARG with nothing launched when a table index is
 * below -1 or not in the current pool, LFD_E_STATE when a trail names a table and no pool has been set; sigma is only
 * checked for Gaussian profiles. */
int lfd_set_trail_tables(lfd_handle* h, const float* samples, int n_samples, const lfd_table* tables, int n_tables);
int lfd_submit_injected_shaped(lfd_handle* h, int n, const int32_t* base_index, const lfd_trail* trails,
                               const lfd_trail_shape* shapes, const int32_t* trail_offsets, int flags);

/* One pass on one already flipped frame (process_field_bright / process_field_dim called directly).
 * If `writeback` != 0 the clipped float image is copied back into `img` (the reference mutates it).  `img` is native
 * float32 in and out: LFD_E_ARG with nothing launched when `flags` holds LFD_INPUT_BIGENDIAN. */
int lfd_run_pass(lfd_handle* h, int pass, float* img, int flags, int writeback, lfd_result* out);

/* remove_stars' blot on a host image, in place (UN-flipped orientation, same rect convention as lfd_submit). */
int lfd_blot(lfd_handle* h, float* img, const int32_t* rects, int nrects);

/* Stage taps of the last run; `frame` indexes the batch, `pass` is LFD_PASS_*. */
int lfd_get_stage(lfd_handle* h, int frame, int pass, int stage, void* host_out, size_t bytes);
int lfd_get_stage_count(lfd_handle* h, int frame, int pass, int stage, int* count);

/* cv2.HoughLines(img, rho, theta, threshold) on a host uint8 image of any size.
 * lines: float32[max_lines][2]; accum (optional): int32[(numangle+2)*(numrho+2)]; returns the total
 * number of lines in *n_lines (may exceed max_lines; only max_lines are written). */
int lfd_hough_dims(int height, int width, double rho, double theta, int* numangle, int* numrho);
int lfd_hough_lines(lfd_handle* h, const uint8_t* img, int height, int width, double rho, double theta,
                    int threshold, float* lines, int max_lines, int* n_lines, int32_t* accum);

/* cv2.Canny(img, low, high) (aperture 3, L2gradient=False) as called at processfield.py:236, on a host uint8 image
 * of the handle's frame size; edges_out: uint8 height*width, 0 / 255.  (Config-5 microbenchmark and parity.) */
int lfd_canny(lfd_handle* h, const uint8_t* img, int low, int high, uint8_t* edges_out);

/* Micro-benchmark: peak shared-memory atomicAdd rate of the device in G atomics/s (conflict-free, all SMs) - the
 * roofline the Hough vote kernel (shared-memory-privatised accumulators) is reported against. */
int lfd_smem_atomic_peak(lfd_handle* h, double* gops);

/* fit_minAreaRect(img, contoursMode, contoursMethod, minAreaRectMinLen, lwTresh) of processfield.py:201-263 on a host
 * uint8 image of the handle's frame size: Canny(0,255) -> findContours -> minAreaRect filter -> fillPoly.
 * box_out: uint8 height*width (0/255) = box_img; *detection = the function's first return value.
 * It runs as frame 0 of the bright pass: afterwards the CANNY, FG/BG_LABELS, RECTS and BOX taps of (0, LFD_PASS_BRIGHT)
 * and lfd_get_counters describe this call (the taps need a whole-frame run or lfd_run_pass earlier on the handle). */
int lfd_fit_min_area_rect(lfd_handle* h, const uint8_t* img, int contoursMode, int contoursMethod,
                          double minAreaRectMinLen, double lwTresh, uint8_t* box_out, int* detection);

/* Per-stage device times (ms, CUDA events) of the last lfd_wait / lfd_run_resident; names via lfd_stage_name. */
int lfd_get_timings(lfd_handle* h, float* ms, int max_entries, int* n_entries);
/* Bracketed kernels (the ones that carry the step: morphology, Sobel/NMS, the band CCL kernels, rectangles, Hough vote)
   of the last collected batch: CUDA events recorded on the launching stream on both sides of the launch - also inside
   the captured graph of the production path - so the durations are measured live, with the other streams running.
   index = 0 .. 13 (7 kernels x 2 passes); ms is summed over the batch parts, launches = number of parts.
   index 14 = k_inject of the last collected lfd_submit_injected batch (always bracketed; launches 0 otherwise).
   index 15 = k_capture_bases of an lfd_capture_bases call made before the last collected batch (launches 0 otherwise).
   Returns LFD_E_ARG past the last index. */
int lfd_get_kernel_times(lfd_handle* h, int index, const char** name, int* pass, float* ms, int* launches);
const char* lfd_timing_name(int i);
/* Developer aid: with LFD_KTIMING=1 in the environment at lfd_create time every launch is followed by a CUDA
 * event; returns (source line in lfd_b200.cu, ms) per launch of the last run. */
int lfd_get_ktimings(lfd_handle* h, int* lines, float* ms, int max_entries, int* n_entries);
/* Benchmark timing on the device: record a CUDA event (slot 0..3) on the handle's stream; elapsed ms between a
 * mark of `h` and a mark of `h_end` (may be the same handle; both must belong to the same GPU). */
int lfd_timer_mark(lfd_handle* h, int slot);
int lfd_timer_elapsed(lfd_handle* h, int slot_start, lfd_handle* h_end, int slot_end, float* ms);
/* Number of kernels this library launched since the handle was created. */
int64_t lfd_kernel_launches(const lfd_handle* h);

/* ---- host-side ingest (plain C++, no GPU needed; the GIL is released by ctypes for the whole call) -------------
 * lfd_fits_load_frame: fitsio.read + fitsio.read_header of a frame file (lfd/detecttrails/detecttrails.py:113-114).
 * The first HDU with data must be a 2-D BITPIX=-32 image of height x width without BSCALE/BZERO; its raw big-endian
 * payload is read into dest (height*width*4 bytes, e.g. a slot of lfd_host_frames; submit with
 * LFD_INPUT_BIGENDIAN) and the raw value text of the nkeys header cards keys[i] is copied to values + 72*i
 * (NUL-terminated).  LFD_E_UNSUPPORTED for any other layout or a missing card, LFD_E_ARG for I/O errors: the caller
 * then uses its general reader, which raises what the reference raises. */
int lfd_fits_load_frame(const char* path, void* dest, int height, int width, const char* const* keys, int nkeys,
                        char* values);
/* lfd_catalog_rects: read_photoObj + the object filter + the blot slices of remove_stars
 * (lfd/detecttrails/removestars.py:96-130, 212-231) for band (0..4 = ugriz) of one photoObj file: writes the
 * (row_start, row_stop, col_start, col_stop) rectangles lfd_submit takes, in catalog order.  cap = filter_caps[filter].
 * LFD_E_UNSUPPORTED when the table is not the plain photoObj layout (ROWC, COLC, PSFMAG, PETROTH90 as 5E, NOBSERVE,
 * NDETECT as J) or holds a non-finite value (the reference raises there), LFD_E_CAPACITY when max_rects is too small. */
int lfd_catalog_rects(const char* path, int band, int height, int width, double cap, double maxmagdiff,
                      double magcount, double pixscale, long long defaultxy, double maxxy, int32_t* rects,
                      int max_rects, int* n_rects);

/* lfd_ingest_batch: both readers for a whole GPU batch on a pool of `nthreads` native threads (0 = one per hardware
 * thread) - what the frame loop of DetectTrails.process does per frame before the pixel work
 * (lfd/detecttrails/detecttrails.py:73-117 and lfd/detecttrails/removestars.py:96-231), batched.  Frame i's raw payload
 * goes to staging + i * height * width * 4 (e.g. lfd_host_frames), its rectangles to rects + i * max_rects * 4 (count in
 * n_rects[i]), its header cards to values + (i * nkeys + k) * 72; bands[i] = 0..4 (ugriz) selects filter_caps[bands[i]].
 * status_frame[i] / status_cat[i] carry the per-item result of lfd_fits_load_frame / lfd_catalog_rects: an item that is
 * not LFD_OK is left to the caller's general reader, the others are ready for lfd_submit(..., LFD_INPUT_BIGENDIAN). */
int lfd_ingest_batch(void* staging, int height, int width, int n, const char* const* frame_paths,
                     const char* const* cat_paths, const int32_t* bands, const double* filter_caps, double maxmagdiff,
                     double magcount, double pixscale, long long defaultxy, double maxxy, const char* const* keys, int nkeys,
                     char* values, int32_t* rects, int max_rects, int32_t* n_rects, int32_t* status_frame,
                     int32_t* status_cat, int nthreads);
/* Work counters of the last run, summed over the batch: [0] nonzero px voted equ, [1] box, [2] votes,
 * [3] runs fg, [4] runs bg, [5] contours, [6] passing rects, [7] frames that ran dim, [8] frames that ran Hough,
 * [11] contours whose rectangle a whole warp computed, [12] of those, short contours handed over because their thread's hull stack was full,
 * [14] labelling bands whose run-id look-back gave up waiting (frame reported LFD_FRAME_OVERFLOW; expected 0),
 * [15] contours the aspect screen proved unable to pass (fitted anyway with LFD_KEEP_TAPS). */
int lfd_get_counters(lfd_handle* h, int64_t* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* LFD_B200_H */
