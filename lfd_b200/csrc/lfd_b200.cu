// lfd_b200.cu - handle, device memory layout, pipeline orchestration and the C ABI of include/lfd_b200.h.
//
// One handle = one GPU, one stream, buffers for `max_batch` frames.  A batch goes through
//   star mask -> prep (blot+flip+clip+u8+hist, both passes in one read of the float frame)
//   per pass: LUT -> morphology -> Sobel/NMS -> run-CCL (hysteresis + outer contours) -> run-CCL of the
//   background (hole contours) -> minAreaRect/filter/boxPoints -> box fill -> Hough x2 -> check_theta
// with every kernel gridded over (work, frame); frames a pass does not apply to exit at the first line
// (bright detected -> no dim; no rectangle passed -> no Hough), so there is no host round trip inside a batch.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <fcntl.h>
#include <sys/file.h>
#include <time.h>
#include <unistd.h>

#include <string>
#include <vector>

#include "common.cuh"
#include "geom.cuh"
#include "k_canny.cuh"
#include "k_ccl.cuh"
#include "k_hough.cuh"
#include "k_inject.cuh"
#include "k_morph.cuh"
#include "k_prep.cuh"
#include "k_rects.cuh"
#include "host_ingest.cuh"

static std::string g_create_error;

// dynamic shared-memory opt-in (cudaFuncSetAttribute) is per function AND per device: high-water marks per device
#define LFD_MAX_DEVICES 64
struct DevLimits { size_t band_max = 48 * 1024, rects_max = 48 * 1024, screen_max = 48 * 1024, anyk_max = 48 * 1024; };
static DevLimits g_dev_limits[LFD_MAX_DEVICES];

// with the two passes overlapped, a batch of >= 16 frames is cut in this many parts (1 / 2 / 3 / 4 parts measured
// 1.85 / 1.72 / 1.73 / 1.70 ms a step: DESIGN.md §3)
#define LFD_BATCH_PARTS 2

enum { T_PREP = 0, T_MORPH, T_CANNY, T_CCL_FG, T_CCL_BG, T_RECTS, T_HOUGH, T_CHECK, T_PER_PASS };
static const char* k_timing_names[] = {
    "setup(memset+star_mask)",
    "prep(blot+flip+clip+u8+hist)",
    "bright:lut+morph", "bright:sobel+nms", "bright:ccl_fg(hysteresis)", "bright:ccl_bg(holes)",
    "bright:rects+boxfill", "bright:hough", "bright:check_theta",
    "dim:lut+morph", "dim:sobel+nms", "dim:ccl_fg(hysteresis)", "dim:ccl_bg(holes)",
    "dim:rects+boxfill", "dim:hough", "dim:check_theta",
    "results_d2h"};
#define N_TIMINGS 17

// Brackets: a CUDA event on each side of the launches that carry the step (recorded on the launching stream, also
// inside the captured graph), so that bench.py can quote the average launch duration of the time-dominant kernel
// measured live in the timed region (lfd_get_kernel_times).
enum { KB_MORPH = 0, KB_NMS, KB_CCL_BAND_FG, KB_CCL_BAND_BG, KB_RECTS_SCREEN, KB_RECTS, KB_HOUGH_VOTE, KB_COUNT };
static const char* k_bracket_names[KB_COUNT] = {"k_morph_march", "k_nms_march", "k_ccl_band(fg)", "k_ccl_band(bg)",
                                                "k_rects_screen", "k_rects_warp", "k_hough_vote"};

struct HoughBufs {
    HoughCfg hc;
    float* tabSin = nullptr;   // device
    float* tabCos = nullptr;
    size_t accum_stride = 0, key_stride = 0, line_stride = 0;
    int max_lines = 0;
    int* accum = nullptr;      // [B][2][accum_stride]
    u64* keys = nullptr;       // [B][2][key_stride]
    float* lines = nullptr;    // [B][2][line_stride]  (allocated on first FULL_LINES use)
    size_t smem = 0;
};

// lfd_hough_lines' buffers, sized for the image of its last call
struct HoughScratch {
    int H = 0, W = 0;
    u8* img = nullptr; u32* mask = nullptr; uint2* segs = nullptr; FrameCtl* ctl = nullptr; lfd_result* res = nullptr;
    HoughBufs hb;
};

struct lfd_handle {
    int device = 0, B = 0, sm_count = 148;
    Dims d;
    lfd_config cfg;
    lfd_params params;
    bool have_params = false;
    cudaStream_t stream = nullptr;        // uploads, prep, bright pass, results
    // the batch is cut in `nsplit` parts; part k runs its bright pass on xs[k][0] and its dim pass on xs[k][1]
    // (xs[0][0] is `stream` itself); every extra stream joins `stream` through its own event
    cudaStream_t xs[LFD_BATCH_PARTS][2];
    cudaEvent_t xjoin[LFD_BATCH_PARTS][2];
    cudaEvent_t ev_fork = nullptr;
    // host->device copy gate (lfd_set_h2d_gate): an advisory file lock shared with the other ranks of the same host bridge
    // slot, held from the moment the batch copy is enqueued until it has completed (released by a stream host callback)
    int gate_fd = -1;
    int64_t gate_waits = 0, gate_timeouts = 0;
    std::string err;
    int64_t launches = 0;
    int last_n = 0, last_flags = 0;
    bool pending = false;
    // what h->in holds: the un-flipped frames the last whole-frame run read (LFD_STAGE_INPUT), in FITS byte order if in_be;
    // in_injected: they are base + trails written by lfd_submit_injected (until the next lfd_upload), not a submitted batch
    bool in_whole = false, in_be = false, in_injected = false;

    // device
    float* in = nullptr;              // [B][N]
    u32* starmask = nullptr;          // [B][NW]
    int4* rects_d = nullptr;          // [B*max_star_rects]
    int* rect_off_d = nullptr;        // [B+1]
    u8* gray[2] = {nullptr, nullptr}; // [B][N]
    u32* hist = nullptr;              // [2][B][256]
    u8* lut = nullptr;                // [2][B][256]
    u8* morph[2] = {nullptr, nullptr};
    u32* nz[2] = {nullptr, nullptr};  // [B][NW]
    u32* cand[2] = {nullptr, nullptr};
    u32* strong[2] = {nullptr, nullptr};
    u32* edges[2] = {nullptr, nullptr};
    u32* box[2] = {nullptr, nullptr};
    u8* tap_u8 = nullptr;             // [N] scratch for expanded taps
    u8* eroded_tap = nullptr;         // [B][N] lazily
    u8* nms_tap[2] = {nullptr, nullptr};
    float* clipped = nullptr;         // [N] lazily (run_pass writeback)
    int* labels_tap = nullptr;        // [N] lazily
    FrameCtl* ctl = nullptr;          // [2][B]: one bookkeeping block per pass (the passes run concurrently)
    unsigned* look = nullptr;         // [2][2][B][look_stride]: k_ccl_band's ticket + look-back words per pass, kind, frame
    int look_stride = 0;
    lfd_result* res_d = nullptr;      // [B]
    int64_t* counters_d = nullptr;    // [16]
    uint2* segs[2] = {nullptr, nullptr};     // per pass: [B][2][NW]
    CclBuf* ccl_d[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};   // [pass][kind] -> [B]
    CompBuf* comp_d[2] = {nullptr, nullptr}; // per pass: [B]
    RectBuf* rbuf_d[2] = {nullptr, nullptr}; // per pass: [B]
    int* rtasks[2] = {nullptr, nullptr};     // per pass: [B][2*max_components] k_rects_screen's survivors, a launch's from its first frame
    std::vector<CclBuf> ccl_h[2][2];
    std::vector<CompBuf> comp_h[2];
    std::vector<RectBuf> rbuf_h[2];
    std::vector<void*> allocs;
    HoughBufs hb[2];
    HoughScratch hs;                  // lfd_hough_lines, allocated on first use
    // injection campaigns (lfd_set_base / lfd_submit_injected): resident base frames and per-slot trails
    float* base_d = nullptr;          // [base_cap][N], replaced by lfd_set_base
    int n_base = 0, base_cap = 0;
    std::vector<int4> base_rects;     // star rectangles of the bases (host), base_rect_off[n_base + 1] indexes them
    std::vector<int> base_rect_off;
    InjTrail* inj_trails_d = nullptr; // [B * LFD_MAX_INJECT_TRAILS]
    int* inj_off_d = nullptr;         // [B + 1]
    int* inj_base_d = nullptr;        // [B]
    InjTrail* inj_trails_h = nullptr; // pinned staging of the three above
    int* inj_off_h = nullptr;
    int* inj_base_h = nullptr;
    float* tab_samples_d = nullptr;   // pool of tabulated trail shapes (lfd_set_trail_tables), [tab_cap] samples
    int tab_cap = 0;
    std::vector<lfd_table> tables;    // the pool's tables; empty: no pool set
    cudaEvent_t ev_inj[2] = {nullptr, nullptr};   // around k_inject; inj_recorded: the last run was lfd_submit_injected
    bool inj_recorded = false;
    float inj_ms = 0.f;
    cudaEvent_t ev_cap[2] = {nullptr, nullptr};   // around k_capture_bases; reported with the next collected batch
    bool cap_recorded = false;
    float cap_ms = 0.f;
    int cap_launches = 0;

    // host
    float* frames_h = nullptr;        // pinned [B][N]
    lfd_result* res_h = nullptr;      // pinned [B]
    int4* rects_h = nullptr;          // pinned
    int* rect_off_h = nullptr;        // pinned
    FrameCtl* ctl_h = nullptr;        // pinned [2][B]
    int64_t* counters_h = nullptr;    // pinned [16] (a pageable destination would make the D2H copy block the host)

    cudaEvent_t ev[N_TIMINGS + 1];
    bool ev_valid[N_TIMINGS + 1];
    float timings[N_TIMINGS];
    cudaEvent_t kb[LFD_BATCH_PARTS][2][KB_COUNT][2];  // [part][pass][kernel][begin / end], created on first use
    bool kb_used[LFD_BATCH_PARTS][2][KB_COUNT];       // recorded by the last run
    float kb_ms[2][KB_COUNT];                         // last run: per pass, summed over the parts
    int kb_launches[2][KB_COUNT];
    int cur_part = 0;                                 // part index of the run_pass_kernels call in progress
    // CUDA graph of the two passes + verdict + result copies (whole-frame path without taps): ~100 small launches
    // become one graph launch, which removes the per-launch gaps between the latency-bound kernels
    bool use_graphs = true;
    // one instantiated graph per (n, flags) in use, oldest first: a drop-in run with injections alternates its big-endian
    // batches with native injected steps, which would otherwise re-capture the graph twice per batch
    struct CachedGraph { cudaGraphExec_t exec; int n, flags; int64_t launches; };
    std::vector<CachedGraph> graphs;
    bool stage_timings_valid = true;
    // arbitrary structuring elements (lfd_set_kernels): [pass][0 erode / 1 dilate] chord lists (chords.cuh) in device
    // buffers sized by the element; kh == 0: no erosion.  anyk_on[pass] false: the all-ones rectangles of lfd_pass_params
    struct AnyElem { int kh = 0, kw = 0, nlev = 0; int* buf = nullptr; size_t cap = 0; } anyk[2][2];
    bool anyk_on[2] = {false, false};
    u8* anyk_eroded = nullptr;        // [B][N] the dim pass's erosion, allocated with its first erosion element
    int prep_grid[3] = {0, 0, 0};     // resident CTAs of k_prep<mode> on this device (one full wave)
    cudaEvent_t mark[4];              // caller-placed timestamps on the handle's stream (lfd_timer_mark)
    bool mark_valid[4];
    // developer aid (env LFD_KTIMING=1): one event after every launch, reported by source line
    bool ktiming = false;
    std::vector<cudaEvent_t> kev;
    std::vector<int> kline;
    int kn = 0;
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                           \
            return LFD_E_CUDA;                                                                     \
        }                                                                                          \
    } while (0)

#define LAUNCH_CHECK()                                                                             \
    do {                                                                                           \
        h->launches++;                                                                             \
        if (h->ktiming) ktime_mark(h, __LINE__);                                                   \
        cudaError_t e_ = cudaGetLastError();                                                       \
        if (e_ != cudaSuccess) {                                                                   \
            h->err = std::string("kernel launch: ") + cudaGetErrorString(e_) + " at line " + std::to_string(__LINE__); \
            return LFD_E_CUDA;                                                                     \
        }                                                                                          \
    } while (0)

// propagate an LFD_* error code
#define TRY(call) do { int rc_ = (call); if (rc_ != LFD_OK) return rc_; } while (0)

static void ktime_mark(lfd_handle* h, int line)
{
    if (h->kn >= (int)h->kev.size()) { cudaEvent_t e; cudaEventCreate(&e); h->kev.push_back(e); h->kline.push_back(0); }
    h->kline[h->kn] = line;
    cudaEventRecord(h->kev[h->kn], h->stream);
    h->kn++;
}

template <typename T>
static int dev_alloc(lfd_handle* h, T** p, size_t count)
{
    void* q = nullptr;
    size_t bytes = count * sizeof(T);
    if (bytes == 0) bytes = 16;
    CK(cudaMalloc(&q, bytes));
    h->allocs.push_back(q);
    *p = (T*)q;
    return LFD_OK;
}

static int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }

#define GRAPH_CACHE 4                 // instantiated graphs kept per handle (lfd_handle::graphs)

static void graphs_clear(lfd_handle* h)
{
    for (auto& g : h->graphs) cudaGraphExecDestroy(g.exec);
    h->graphs.clear();
}

// prologue of the entry points that enqueue work: the handle's device, and no batch in flight
static int enter(lfd_handle* h)
{
    cudaSetDevice(h->device);
    if (h->pending) { h->err = "previous batch not collected (call lfd_wait)"; return LFD_E_STATE; }
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// small bookkeeping kernels
// ------------------------------------------------------------------------------------------------
// ctl: [2][B] (one block per pass); block p only ever looks at active[p] / hough[p]
// look: k_ccl_band's tickets and look-back words, [2 pass][2 kind][B][lstride] (nullptr where no labelling follows)
__global__ void k_ctl_init(FrameCtl* ctl, int B, lfd_result* res, int n, int act0, int act1, unsigned* look, int lstride)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    if (look)
        for (int pk = 0; pk < 4; pk++)
            for (int i = 0; i < lstride; i++) look[((size_t)pk * B + f) * lstride + i] = 0u;
    FrameCtl c;
    memset(&c, 0, sizeof(c));
    c.active[0] = act0; c.active[1] = act1;
    ctl[f] = c;
    ctl[B + f] = c;
    lfd_result r;
    memset(&r, 0, sizeof(r));
    r.pass = -1;
    for (int p = 0; p < 2; p++) { r.rect_detection[p] = -1; r.n_lines_equ[p] = -1; r.n_lines_box[p] = -1; }
    res[f] = r;
}

// Verdict of the frame from the two passes' private results (detecttrails.py:125-131): bright wins; the dim
// pass counts only where bright neither detected nor failed, and is reported as "not run" elsewhere.
// mode 0: both passes ; 1: bright only ; 2: dim only
__global__ void k_finalize(const FrameCtl* __restrict__ ctl, int B, lfd_result* __restrict__ res, int n, int mode,
                           unsigned long long* counters)
{
    int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n) return;
    const FrameCtl& c0 = ctl[f];
    const FrameCtl& c1 = ctl[B + f];
    lfd_result* R = res + f;
    const int errbits = LFD_FRAME_NO_LINES_EQU | LFD_FRAME_NO_LINES_BOX | LFD_FRAME_OVERFLOW;
    const bool ran0 = mode != 2, ran1 = mode != 1;
    const bool use1 = ran1 && !(ran0 && (c0.detected || (c0.status & errbits)));
    int status = ran0 ? c0.status : 0;
    if (use1) status |= c1.status;
    R->status = status;
    int pass = -1;
    if (ran0 && c0.detected) pass = 0;
    else if (use1 && c1.detected) pass = 1;
    R->detected = pass >= 0;
    R->pass = pass;
    if (pass >= 0) { R->rho = R->top_equ[pass][0][0]; R->theta = R->top_equ[pass][0][1]; }
    if (ran1 && !use1) {      // what a run that skipped the dim pass reports
        R->rect_detection[1] = -1; R->n_lines_equ[1] = -1; R->n_lines_box[1] = -1; R->rejected[1] = 0;
        for (int i = 0; i < LFD_MAX_SET_LINES; i++) {
            R->top_equ[1][i][0] = R->top_equ[1][i][1] = 0.f;
            R->top_box[1][i][0] = R->top_box[1][i][1] = 0.f;
        }
    }
    if (mode == 0 && use1) atomicAdd(&counters[7], 1ull);
}

__global__ void k_pack_mask(const u8* __restrict__ img, u32* __restrict__ mask, Dims d)
{
    // one warp per 32 pixels
    int gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = gw; i < d.NW; i += nwarps) {
        int y = i / d.WW, w = i - y * d.WW;
        int x = (w << 5) + lane;
        bool nzp = x < d.W && img[(size_t)y * d.W + x] != 0;
        u32 b = __ballot_sync(FULLMASK, nzp);
        if (lane == 0) mask[i] = b;
    }
}

// ------------------------------------------------------------------------------------------------
// Hough configuration (host): OpenCV's numangle/numrho and float trig tables
// ------------------------------------------------------------------------------------------------
static void hough_dims_host(int H, int W, double rho_, double theta_, int* numangle, int* numrho)
{
    float rho = (float)rho_, theta = (float)theta_;
    int max_rho = W + H, min_rho = -max_rho;
    double min_theta = 0, max_theta = M_PI;
    int na = (int)floor((max_theta - min_theta) / theta) + 1;
    if (na > 1 && fabs(M_PI - (na - 1) * theta) < theta / 2) --na;
    *numangle = na;
    *numrho = (int)lrint(((max_rho - min_rho) + 1) / rho);
}

static void hough_free(HoughBufs& hb)
{
    cudaFree(hb.accum); cudaFree(hb.keys); cudaFree(hb.lines); cudaFree(hb.tabSin);   // tabCos lies in tabSin's block
    hb.accum = nullptr; hb.keys = nullptr; hb.lines = nullptr; hb.tabSin = hb.tabCos = nullptr;
}

static void hough_scratch_free(HoughScratch& hs)
{
    cudaFree(hs.img); cudaFree(hs.mask); cudaFree(hs.segs); cudaFree(hs.ctl); cudaFree(hs.res);
    hs.img = nullptr; hs.mask = nullptr; hs.segs = nullptr; hs.ctl = nullptr; hs.res = nullptr; hs.H = hs.W = 0;
    hough_free(hs.hb);
}

static int hough_setup(lfd_handle* h, HoughBufs* hb, int H, int W, double rho_, double theta_, int threshold,
                       int nframes, bool want_lines, int max_lines_cfg)
{
    if (!(rho_ > 0) || !(theta_ > 0)) { h->err = "HoughLines: rho and theta must be positive"; return LFD_E_ARG; }
    HoughCfg hc;
    hough_dims_host(H, W, rho_, theta_, &hc.numangle, &hc.numrho);
    if (hc.numangle < 1 || hc.numrho < 1 || (double)hc.numangle * hc.numrho > 2.0e8) {
        h->err = "HoughLines: accumulator size out of range";
        return LFD_E_ARG;
    }
    hc.RS = hc.numrho + 2;
    hc.rho = (float)rho_;
    hc.theta = (float)theta_;
    hc.threshold = threshold;
    const size_t smem_budget = 96 * 1024;
    int apc = (int)(smem_budget / ((size_t)hough_rss(hc.RS) * 4));
    if (apc > 32) apc = 32;
    if (apc < 1) { h->err = "HoughLines: rho too fine for the shared-memory accumulator (numrho too large)"; return LFD_E_UNSUPPORTED; }
    if (apc < 32) { int p = 1; while (p * 2 <= apc) p *= 2; apc = p; }   // power of two so sub-warps tile a warp
    if (apc > hc.numangle) apc = hc.numangle < 32 ? next_pow2(hc.numangle) : 32;
    hc.apc = apc;
    hc.ngroups = (hc.numangle + apc - 1) / apc;
    hb->smem = (size_t)apc * hough_rss(hc.RS) * 4;
    hb->hc = hc;
    // tables, exactly as OpenCV builds them (float accumulation of the angle)
    std::vector<float> ts(hc.numangle), tc(hc.numangle);
    float irho = 1 / hc.rho;
    float ang = 0.f;
    for (int n = 0; n < hc.numangle; ang += hc.theta, n++) {
        ts[n] = (float)(sin((double)ang) * irho);
        tc[n] = (float)(cos((double)ang) * irho);
    }
    size_t accum_stride = (size_t)(hc.numangle + 2) * hc.RS;
    size_t cells = (size_t)hc.numangle * hc.numrho;
    size_t key_stride = (size_t)next_pow2((int)cells);
    bool realloc_needed = (accum_stride != hb->accum_stride) || (key_stride != hb->key_stride) || !hb->accum;
    if (realloc_needed) {
        hough_free(*hb);
        CK(cudaMalloc((void**)&hb->accum, (size_t)nframes * 2 * accum_stride * sizeof(int)));
        CK(cudaMalloc((void**)&hb->keys, (size_t)nframes * 2 * key_stride * sizeof(u64)));
        CK(cudaMalloc((void**)&hb->tabSin, (size_t)2 * hc.numangle * sizeof(float)));
        hb->tabCos = hb->tabSin + hc.numangle;
        hb->accum_stride = accum_stride;
        hb->key_stride = key_stride;
    }
    hb->max_lines = (max_lines_cfg > 0 && (size_t)max_lines_cfg < cells) ? max_lines_cfg : (int)cells;
    hb->line_stride = (size_t)2 * hb->max_lines;
    if (want_lines && !hb->lines) CK(cudaMalloc((void**)&hb->lines, (size_t)nframes * 2 * hb->line_stride * sizeof(float)));
    CK(cudaMemcpyAsync(hb->tabSin, ts.data(), hc.numangle * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(hb->tabCos, tc.data(), hc.numangle * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    // the limit is per function, not per launch: both passes (and lfd_hough_lines) share k_hough_vote
    CK(cudaFuncSetAttribute(k_hough_vote<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_budget));
    CK(cudaFuncSetAttribute(k_hough_vote<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_budget));
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// create / destroy
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_abi_version(void) { return LFD_ABI_VERSION; }

extern "C" const char* lfd_last_error(const lfd_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

extern "C" int lfd_destroy(lfd_handle* h)
{
    if (!h) return LFD_E_ARG;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++)
            if (h->xs[k][p] && h->xs[k][p] != h->stream) cudaStreamSynchronize(h->xs[k][p]);
    if (h->gate_fd >= 0) { flock(h->gate_fd, LOCK_UN); close(h->gate_fd); h->gate_fd = -1; }
    for (void* p : h->allocs) cudaFree(p);
    for (int p = 0; p < 2; p++) hough_free(h->hb[p]);
    hough_scratch_free(h->hs);
    cudaFree(h->base_d); cudaFree(h->tab_samples_d);
    for (int p = 0; p < 2; p++) for (int k = 0; k < 2; k++) cudaFree(h->anyk[p][k].buf);
    for (void* p : {(void*)h->frames_h, (void*)h->res_h, (void*)h->rects_h, (void*)h->rect_off_h, (void*)h->ctl_h,
                    (void*)h->inj_trails_h, (void*)h->inj_off_h, (void*)h->inj_base_h, (void*)h->counters_h})
        cudaFreeHost(p);
    for (int i = 0; i < 2; i++) {
        if (h->ev_inj[i]) cudaEventDestroy(h->ev_inj[i]);
        if (h->ev_cap[i]) cudaEventDestroy(h->ev_cap[i]);
    }
    for (int i = 0; i <= N_TIMINGS; i++) if (h->ev_valid[i]) cudaEventDestroy(h->ev[i]);
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++)
            for (int b = 0; b < KB_COUNT; b++)
                for (int e = 0; e < 2; e++)
                    if (h->kb[k][p][b][e]) cudaEventDestroy(h->kb[k][p][b][e]);
    for (int i = 0; i < 4; i++) if (h->mark_valid[i]) cudaEventDestroy(h->mark[i]);
    graphs_clear(h);
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++) {
            if (h->xjoin[k][p]) cudaEventDestroy(h->xjoin[k][p]);
            if (h->xs[k][p] && h->xs[k][p] != h->stream) cudaStreamDestroy(h->xs[k][p]);
        }
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
    return LFD_OK;
}

static int create_impl(lfd_handle* h, int device, int max_batch, int H, int W, const lfd_config* cfg)
{
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { h->err = "no such CUDA device"; return LFD_E_CUDA; }
    CK(cudaSetDevice(device));
    h->device = device;
    { const char* kt = getenv("LFD_KTIMING"); h->ktiming = kt && kt[0] == '1'; }
    { const char* ng = getenv("LFD_NO_GRAPH"); h->use_graphs = !(ng && ng[0] == '1'); }
    if (max_batch < 1 || H < 8 || W < 8) { h->err = "bad batch or frame size"; return LFD_E_ARG; }
    if (W % 4 != 0) { h->err = "frame width must be a multiple of 4"; return LFD_E_UNSUPPORTED; }
    if (W > 4096 || H > 65535) { h->err = "frame too large (W <= 4096, H <= 65535)"; return LFD_E_UNSUPPORTED; }
    h->B = max_batch;
    h->d.H = H; h->d.W = W; h->d.WW = (W + 31) / 32; h->d.N = H * W; h->d.NW = H * h->d.WW;
    memset(&h->cfg, 0, sizeof(h->cfg));
    if (cfg) h->cfg = *cfg;
    if (h->cfg.max_runs <= 0) h->cfg.max_runs = 1 << 19;
    if (h->cfg.max_components <= 0) h->cfg.max_components = 1 << 16;
    if (h->cfg.max_star_rects <= 0) h->cfg.max_star_rects = 8192;
    // a frame cannot hold more runs than H * ceil(W/2)
    long long worst = (long long)H * ((W + 1) / 2);
    if (h->cfg.max_runs > worst) h->cfg.max_runs = (int)worst;
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++) {
            if (k == 0 && p == 0) { h->xs[0][0] = h->stream; continue; }
            CK(cudaStreamCreateWithFlags(&h->xs[k][p], cudaStreamNonBlocking));
            CK(cudaEventCreateWithFlags(&h->xjoin[k][p], cudaEventDisableTiming));
        }
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    {
        cudaDeviceProp prop;
        CK(cudaGetDeviceProperties(&prop, device));
        h->sm_count = prop.multiProcessorCount;
        int per_sm[3] = {0, 0, 0};
        // k_prep keeps its TMA rings in dynamic shared memory (above the 48 KB default limit)
#define PREP_ATTR(M, E) CK(cudaFuncSetAttribute(k_prep<M, E>, cudaFuncAttributeMaxDynamicSharedMemorySize, PR_SMEM))
        PREP_ATTR(0, false); PREP_ATTR(0, true); PREP_ATTR(1, false); PREP_ATTR(2, false);
#undef PREP_ATTR
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[0], k_prep<0, false>, PR_WARPS * 32, PR_SMEM));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[1], k_prep<1, false>, PR_WARPS * 32, PR_SMEM));
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm[2], k_prep<2, false>, PR_WARPS * 32, PR_SMEM));
        for (int m = 0; m < 3; m++) h->prep_grid[m] = prop.multiProcessorCount * (per_sm[m] > 0 ? per_sm[m] : 1);
    }
    // the dynamic shared-memory limit is a property of the FUNCTION on one DEVICE, shared by every handle of the process
    // on that device: only ever raise it, and keep the high-water mark per device
    {
        DevLimits& L = g_dev_limits[device % LFD_MAX_DEVICES];
        if (ccl_band_smem(h->d.WW) > L.band_max) {
            CK(cudaFuncSetAttribute(k_ccl_band, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ccl_band_smem(h->d.WW)));
            L.band_max = ccl_band_smem(h->d.WW);
        }
        if (rects_smem(max_batch) > L.rects_max) {
            CK(cudaFuncSetAttribute(k_rects_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rects_smem(max_batch)));
            L.rects_max = rects_smem(max_batch);
        }
        if (screen_smem(max_batch) > L.screen_max) {
            CK(cudaFuncSetAttribute(k_rects_screen, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)screen_smem(max_batch)));
            L.screen_max = screen_smem(max_batch);
        }
    }
    for (int i = 0; i <= N_TIMINGS; i++) { CK(cudaEventCreate(&h->ev[i])); h->ev_valid[i] = true; }
    for (int i = 0; i < 4; i++) { CK(cudaEventCreate(&h->mark[i])); h->mark_valid[i] = true; }
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++)
            for (int b = 0; b < KB_COUNT; b++)
                for (int e = 0; e < 2; e++) CK(cudaEventCreate(&h->kb[k][p][b][e]));

    const int B = h->B;
    const size_t N = h->d.N, NW = h->d.NW;
    int rc;
#define DA(ptr, count) if ((rc = dev_alloc(h, &(ptr), (count))) != LFD_OK) return rc
    DA(h->in, (size_t)B * N);
    DA(h->starmask, (size_t)B * NW);
    DA(h->rects_d, (size_t)B * h->cfg.max_star_rects);
    DA(h->rect_off_d, (size_t)B + 1);
    DA(h->hist, (size_t)2 * B * 256);
    DA(h->lut, (size_t)2 * B * 256);
    for (int p = 0; p < 2; p++) {
        DA(h->gray[p], (size_t)B * N);
        DA(h->morph[p], (size_t)B * N);
        DA(h->nz[p], (size_t)B * NW);
        DA(h->cand[p], (size_t)B * NW);
        DA(h->strong[p], (size_t)B * NW);
        DA(h->edges[p], (size_t)B * NW);
        DA(h->box[p], (size_t)B * NW);
    }
    DA(h->tap_u8, N);
    DA(h->ctl, (size_t)2 * B);
    DA(h->res_d, (size_t)B);
    DA(h->counters_d, 16);
    DA(h->segs[0], (size_t)B * 2 * NW);
    DA(h->segs[1], (size_t)B * 2 * NW);
    const int MR = h->cfg.max_runs, MC = h->cfg.max_components;
    h->look_stride = 1 + (H + CCL_BAND - 1) / CCL_BAND;
    DA(h->look, (size_t)4 * B * h->look_stride);
    const int slotcap = 2 * MR + 4 * MC, hullcap = 2 * slotcap + 4 * MC;
    // one slab per field, sliced per frame; everything the two passes touch exists once per pass
    for (int p = 0; p < 2; p++)
    for (int k = 0; k < 2; k++) {
        h->ccl_h[p][k].resize(B);
        Run* runs; int *parent, *flag, *ymax, *compidx, *rowbase;
        DA(runs, (size_t)B * MR); DA(parent, (size_t)B * MR); DA(flag, (size_t)B * MR); DA(ymax, (size_t)B * MR);
        DA(compidx, (size_t)B * MR); DA(rowbase, (size_t)B * (H + 1));
        for (int f = 0; f < B; f++) {
            CclBuf& c = h->ccl_h[p][k][f];
            c.runs = runs + (size_t)f * MR; c.parent = parent + (size_t)f * MR; c.flag = flag + (size_t)f * MR;
            c.ymax = ymax + (size_t)f * MR; c.compidx = compidx + (size_t)f * MR;
            c.rowbase = rowbase + (size_t)f * (H + 1);
            c.look = h->look + ((size_t)(p * 2 + k) * B + f) * h->look_stride;
        }
        DA(h->ccl_d[p][k], (size_t)B);
        CK(cudaMemcpy(h->ccl_d[p][k], h->ccl_h[p][k].data(), B * sizeof(CclBuf), cudaMemcpyHostToDevice));
    }
    for (int p = 0; p < 2; p++) {
        h->comp_h[p].resize(B);
        int *root, *y0, *hh, *slot, *hulloff, *rowmin, *rowmax;
        DA(root, (size_t)B * 2 * MC); DA(y0, (size_t)B * 2 * MC); DA(hh, (size_t)B * 2 * MC);
        DA(slot, (size_t)B * 2 * MC); DA(hulloff, (size_t)B * 2 * MC);
        DA(rowmin, (size_t)B * slotcap); DA(rowmax, (size_t)B * slotcap);
        for (int f = 0; f < B; f++) {
            CompBuf& c = h->comp_h[p][f];
            c.root = root + (size_t)f * 2 * MC; c.y0 = y0 + (size_t)f * 2 * MC; c.h = hh + (size_t)f * 2 * MC;
            c.slot = slot + (size_t)f * 2 * MC; c.hulloff = hulloff + (size_t)f * 2 * MC;
            c.rowmin = rowmin + (size_t)f * slotcap; c.rowmax = rowmax + (size_t)f * slotcap;
            c.slotcap = slotcap; c.hullcap = hullcap; c.maxcomp = MC;
        }
        DA(h->comp_d[p], (size_t)B);
        CK(cudaMemcpy(h->comp_d[p], h->comp_h[p].data(), B * sizeof(CompBuf), cudaMemcpyHostToDevice));
    }
    for (int p = 0; p < 2; p++) {
        h->rbuf_h[p].resize(B);
        lfdgeom::Pt* hulls; float* hullfs;
        DA(hulls, (size_t)B * hullcap); DA(hullfs, (size_t)B * 3 * hullcap);
        lfd_rect* rects; int *passing, *screened;
        DA(rects, (size_t)B * 2 * MC); DA(passing, (size_t)B * 2 * MC); DA(screened, (size_t)B * 2 * MC);
        DA(h->rtasks[p], (size_t)B * 2 * MC);
        for (int f = 0; f < B; f++) {
            RectBuf& r = h->rbuf_h[p][f];
            r.rects = rects + (size_t)f * 2 * MC; r.passing = passing + (size_t)f * 2 * MC; r.screened = screened + (size_t)f * 2 * MC;
            r.hull = hulls + (size_t)f * hullcap; r.hullf = hullfs + (size_t)f * 3 * hullcap;
        }
        DA(h->rbuf_d[p], (size_t)B);
        CK(cudaMemcpy(h->rbuf_d[p], h->rbuf_h[p].data(), B * sizeof(RectBuf), cudaMemcpyHostToDevice));
    }
#undef DA
    CK(cudaMallocHost((void**)&h->frames_h, (size_t)B * N * sizeof(float)));
    CK(cudaMallocHost((void**)&h->res_h, (size_t)B * sizeof(lfd_result)));
    CK(cudaMallocHost((void**)&h->rects_h, (size_t)B * h->cfg.max_star_rects * sizeof(int4)));
    CK(cudaMallocHost((void**)&h->rect_off_h, ((size_t)B + 1) * sizeof(int)));
    CK(cudaMallocHost((void**)&h->ctl_h, (size_t)2 * B * sizeof(FrameCtl)));
    CK(cudaMemset(h->counters_d, 0, 16 * sizeof(int64_t)));
    CK(cudaMallocHost((void**)&h->counters_h, 16 * sizeof(int64_t)));
    memset(h->counters_h, 0, 16 * sizeof(int64_t));
    memset(h->timings, 0, sizeof(h->timings));
    return LFD_OK;
}

extern "C" int lfd_create_ex(int device, int max_batch, int height, int width, const lfd_config* cfg, lfd_handle** out)
{
    if (!out) return LFD_E_ARG;
    *out = nullptr;
    lfd_handle* h = new lfd_handle();
    memset(h->ev_valid, 0, sizeof(h->ev_valid));
    memset(h->mark_valid, 0, sizeof(h->mark_valid));
    int rc = create_impl(h, device, max_batch, height, width, cfg);
    if (rc != LFD_OK) {
        g_create_error = h->err;
        lfd_destroy(h);
        return rc;
    }
    *out = h;
    return LFD_OK;
}

extern "C" int lfd_create(int device, int max_batch, int height, int width, lfd_handle** out)
{
    return lfd_create_ex(device, max_batch, height, width, nullptr, out);
}

extern "C" int lfd_host_frames(lfd_handle* h, float** out)
{
    if (!h || !out) return LFD_E_ARG;
    *out = h->frames_h;
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// parameters
// ------------------------------------------------------------------------------------------------
static int check_contours_args(lfd_handle* h, int mode, int method)
{
    if (mode < 0 || mode > 3) { h->err = "unknown contoursMode"; return LFD_E_ARG; }
    if (method != 1 && method != 2) { h->err = "contoursMethod CHAIN_APPROX_TC89_* is not implemented"; return LFD_E_UNSUPPORTED; }
    return LFD_OK;
}

static int check_pass_params(lfd_handle* h, const lfd_pass_params& p, bool dim)
{
    if (p.nlinesInSet < 1 || p.nlinesInSet > LFD_MAX_SET_LINES) { h->err = "nlinesInSet must be in 1..16"; return LFD_E_UNSUPPORTED; }
    TRY(check_contours_args(h, p.contoursMode, p.contoursMethod));
    if (p.dilate_h < 1 || p.dilate_w < 1) { h->err = "dilateKernel missing"; return LFD_E_ARG; }
    int eh = dim ? p.erode_h : 0, ew = dim ? p.erode_w : 0;
    if ((eh > 0) != (ew > 0)) { h->err = "bad erodeKernel"; return LFD_E_ARG; }
    // combined halo must fit the shared-memory tile padding of k_morph
    int e_t = eh / 2, e_b = eh > 0 ? eh - 1 - eh / 2 : 0, e_l = ew / 2, e_r = ew > 0 ? ew - 1 - ew / 2 : 0;
    int d_t = p.dilate_h / 2, d_b = p.dilate_h - 1 - p.dilate_h / 2, d_l = p.dilate_w / 2, d_r = p.dilate_w - 1 - p.dilate_w / 2;
    if (e_t + d_t > MORPH_PADH || e_b + d_b > MORPH_PADH || e_l + d_l > 12 || e_r + d_r > 11) {
        h->err = "erode+dilate kernel reach exceeds this build's tile halo (rows <= 16, cols <= 12 left / 11 right)";
        return LFD_E_UNSUPPORTED;
    }
    return LFD_OK;
}

extern "C" int lfd_set_params(lfd_handle* h, const lfd_params* p)
{
    if (!h || !p) return LFD_E_ARG;
    cudaSetDevice(h->device);
    TRY(check_pass_params(h, p->bright, false));
    TRY(check_pass_params(h, p->dim, true));
    CK(cudaStreamSynchronize(h->stream));
    for (int pass = 0; pass < 2; pass++) {
        const lfd_pass_params& pp = pass ? p->dim : p->bright;
        // theta = np.pi/180 and threshold = 1 are literals in the reference (processfield.py:370, :488)
        TRY(hough_setup(h, &h->hb[pass], h->d.H, h->d.W, pp.houghMethod, M_PI / 180, 1, h->B, false, h->cfg.max_lines));
    }
    h->params = *p;
    h->have_params = true;
    h->anyk_on[0] = h->anyk_on[1] = false;       // back to all-ones rectangles until lfd_set_kernels says otherwise
    graphs_clear(h);                             // kernel arguments changed
    return LFD_OK;
}

// The chord list of one element (chords.cuh) into its device buffer: rowoff[kh + 1], then the chord codes
static int fill_anykernel(lfd_handle* h, lfd_handle::AnyElem* k, const uint8_t* mask, int kh, int kw, const char* what)
{
    k->kh = k->kw = k->nlev = 0;
    if (!mask || kh == 0 || kw == 0) return LFD_OK;
    if (kh < 1 || kw < 1 || kh > CHORD_MAX_SIDE || kw > CHORD_MAX_SIDE) {
        h->err = std::string(what) + ": kernel side must be 1.." + std::to_string(CHORD_MAX_SIDE);
        return LFD_E_UNSUPPORTED;
    }
    std::vector<int> buf(kh + 1 + chord_capacity(kh, kw));
    int nlev = 0;
    const int n = chord_decompose(mask, kh, kw, buf.data(), reinterpret_cast<uint32_t*>(buf.data() + kh + 1), &nlev);
    if (n == 0) { h->err = std::string(what) + ": structuring element has no non-zero entry"; return LFD_E_ARG; }
    const size_t need = (size_t)(kh + 1 + n) * sizeof(int);
    if (need > k->cap) {
        cudaFree(k->buf);
        k->buf = nullptr; k->cap = 0;
        CK(cudaMalloc(&k->buf, need));
        k->cap = need;
    }
    CK(cudaMemcpy(k->buf, buf.data(), need, cudaMemcpyHostToDevice));
    k->kh = kh; k->kw = kw; k->nlev = nlev;
    return LFD_OK;
}

// Arbitrary structuring elements for one pass (row-major uint8 masks, non-zero = member, anchor at the centre like
// cv2.erode / cv2.dilate called with the default anchor: processfield.py:354, :464, :471).  erode_mask may be NULL.
extern "C" int lfd_set_kernels(lfd_handle* h, int pass, const uint8_t* erode_mask, int eh, int ew,
                               const uint8_t* dilate_mask, int dh, int dw)
{
    if (!h || (pass != 0 && pass != 1) || !dilate_mask) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    cudaSetDevice(h->device);
    if (!h->have_params) { h->err = "lfd_set_params has not been called"; return LFD_E_STATE; }
    CK(cudaStreamSynchronize(h->stream));
    h->anyk_on[pass] = false;                    // until both elements are in place
    TRY(fill_anykernel(h, &h->anyk[pass][0], pass == 1 ? erode_mask : nullptr, eh, ew, "erodeKernel"));
    TRY(fill_anykernel(h, &h->anyk[pass][1], dilate_mask, dh, dw, "dilateKernel"));
    if (h->anyk[pass][0].kh > 0 && !h->anyk_eroded) TRY(dev_alloc(h, &h->anyk_eroded, (size_t)h->B * h->d.N));
    h->anyk_on[pass] = true;
    graphs_clear(h);
    size_t need = 0;
    for (int k = 0; k < 2; k++) {
        const lfd_handle::AnyElem& e = h->anyk[pass][k];
        if (e.kh > 0) need = std::max(need, chord_smem(e.kh, e.kw, e.nlev));
    }
    DevLimits& L = g_dev_limits[h->device % LFD_MAX_DEVICES];
    if (need > L.anyk_max) {
        CK(cudaFuncSetAttribute(k_morph_any<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
        CK(cudaFuncSetAttribute(k_morph_any<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
        L.anyk_max = need;
    }
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// the pipeline
// ------------------------------------------------------------------------------------------------
// frames [f0, f0 + n) of one pass, launched on stream s: every per-frame array is entered at frame f0, kernels index
// frames from 0
struct PassView {
    lfd_handle* h;
    int f0, n, pass, flags;
    cudaStream_t s;
    FrameCtl* C;                      // this pass's bookkeeping block
    u8 *gray, *morph;
    u32 *nz, *cand, *strong, *edges, *box;
    CclBuf* ccl[2]; CompBuf* comp; RectBuf* rbuf;   // ccl: [kind]
};

static PassView pass_view(lfd_handle* h, int f0, int n, int pass, int flags, cudaStream_t s)
{
    const size_t fN = (size_t)f0 * h->d.N, fNW = (size_t)f0 * h->d.NW;
    return {h, f0, n, pass, flags, s, h->ctl + (size_t)pass * h->B + f0, h->gray[pass] + fN, h->morph[pass] + fN,
            h->nz[pass] + fNW, h->cand[pass] + fNW, h->strong[pass] + fNW, h->edges[pass] + fNW, h->box[pass] + fNW,
            {h->ccl_d[pass][0] + f0, h->ccl_d[pass][1] + f0}, h->comp_d[pass] + f0, h->rbuf_d[pass] + f0};
}

// One side (e = 0 begin, 1 end) of the bracket of kernel `id`, with LFD_KERNEL_TIMES only
static int kb_mark(const PassView& V, int id, int e)
{
    lfd_handle* h = V.h;
    if (!(V.flags & LFD_KERNEL_TIMES)) return LFD_OK;
    cudaStreamCaptureStatus cst = cudaStreamCaptureStatusNone;
    const bool capturing = cudaStreamIsCapturing(V.s, &cst) == cudaSuccess && cst == cudaStreamCaptureStatusActive;
    // under stream capture a plain record is a dependency marker, not a node: ask for an external record node
    CK(cudaEventRecordWithFlags(h->kb[h->cur_part][V.pass][id][e], V.s, capturing ? cudaEventRecordExternal : cudaEventRecordDefault));
    h->kb_used[h->cur_part][V.pass][id] = true;
    return LFD_OK;
}

// Sobel + NMS of the morphology plane into the candidate / strong edge masks; ntap: per-pixel class tap, or nullptr
static int launch_nms(const PassView& V, int low, int high, u8* ntap)
{
    lfd_handle* h = V.h;
    const Dims d = h->d; const int n = V.n;
    if ((d.W % 8) == 0) {        // k_nms_march stores only non-zero mask words
        CK(cudaMemsetAsync(V.cand, 0, (size_t)n * d.NW * sizeof(u32), V.s));
        CK(cudaMemsetAsync(V.strong, 0, (size_t)n * d.NW * sizeof(u32), V.s));
    }
    TRY(kb_mark(V, KB_NMS, 0));
    if ((d.W % 8) == 0) {
        const int nstrips = ((d.W >> 2) + MARCH_UW - 1) / MARCH_UW, nchunks = (d.H + NMS_R - 1) / NMS_R;
        const int nunits = nstrips * nchunks;
        dim3 gg((nunits + NMS_WPC - 1) / NMS_WPC, n);
        if (ntap) k_nms_march<true><<<gg, NMS_WPC * 32, 0, V.s>>>(V.morph, V.nz, V.cand, V.strong, ntap, V.C, V.pass, d, nstrips, nunits, low, high);
        else k_nms_march<false><<<gg, NMS_WPC * 32, 0, V.s>>>(V.morph, V.nz, V.cand, V.strong, ntap, V.C, V.pass, d, nstrips, nunits, low, high);
    } else {
        dim3 cg((d.W + CANNY_TW - 1) / CANNY_TW, (d.H + CANNY_TH - 1) / CANNY_TH, n);
        k_canny_nms<<<cg, 256, 0, V.s>>>(V.morph, V.nz, V.cand, V.strong, ntap, V.C, V.pass, d, low, high);
    }
    LAUNCH_CHECK();
    return kb_mark(V, KB_NMS, 1);
}

// Run labelling.  kind 0: the candidate edges, a component kept (hysteresis) and written to the edge mask where it holds
// a strong pixel (outer contours); kind 1: the background of the edge mask (holes).  k_ccl_extremes_flat is the caller's.
static int launch_labels(const PassView& V, int kind)
{
    lfd_handle* h = V.h;
    const Dims d = h->d; const int n = V.n;
    const int nbands = (d.H + CCL_BAND - 1) / CCL_BAND;
    const dim3 bands((n >= 16 && nbands > CCL_BAND_CTAS) ? CCL_BAND_CTAS : nbands, n), seams((nbands + CCL_WARPS - 1) / CCL_WARPS, n),
        flat(CCL_FLAT_CTAS, n);
    unsigned long long* const cnt = (unsigned long long*)h->counters_d;
    CclBuf* const ccl = V.ccl[kind];
    TRY(kb_mark(V, KB_CCL_BAND_FG + kind, 0));
    k_ccl_band<<<bands, 256, ccl_band_smem(d.WW), V.s>>>(kind ? V.edges : V.cand, ccl, V.C, V.pass, d, kind, h->cfg.max_runs, cnt); LAUNCH_CHECK();
    TRY(kb_mark(V, KB_CCL_BAND_FG + kind, 1));
    k_ccl_merge<<<seams, CCL_WARPS * 32, 0, V.s>>>(ccl, V.C, V.pass, d, kind); LAUNCH_CHECK();
    if (kind == 0) CK(cudaMemsetAsync(V.edges, 0, (size_t)n * d.NW * sizeof(u32), V.s));
    k_ccl_stats_flat<<<flat, 256, 0, V.s>>>(kind ? nullptr : V.strong, ccl, V.C, V.pass, d, kind); LAUNCH_CHECK();
    k_ccl_alloc_flat<<<flat, 256, 0, V.s>>>(ccl, kind ? nullptr : V.edges, V.comp, V.C, V.pass, d, kind); LAUNCH_CHECK();
    return LFD_OK;
}

// fit_minAreaRect's arguments (processfield.py:201); external: cv2.RETR_EXTERNAL, outermost outer borders only
struct ContourArgs { double minAreaRectMinLen, lwTresh; bool external; };

// Rectangles of both contour kinds + box image.  The screen rejects the contours whose aspect bound proves they cannot
// pass (most of them: the NMS rings around stars and their holes); only the survivors are fitted.  With `fit_all`
// every contour is fitted and the screen only records its verdicts, so that the RECTS tap holds every rectangle.
static int launch_contours(const PassView& V, const ContourArgs& a, bool fit_all)
{
    lfd_handle* h = V.h;
    const Dims d = h->d; const int n = V.n;
    unsigned long long* const cnt = (unsigned long long*)h->counters_d;
    int* const tasks = fit_all ? nullptr : h->rtasks[V.pass] + (size_t)V.f0 * 2 * h->cfg.max_components;
    TRY(kb_mark(V, KB_RECTS_SCREEN, 0));
    k_rects_screen<<<h->sm_count * 2, SCREEN_THREADS, screen_smem(n), V.s>>>(V.comp, V.rbuf, V.ccl[0], V.ccl[1], V.C, V.pass, n, d, a.lwTresh, tasks, cnt); LAUNCH_CHECK();
    TRY(kb_mark(V, KB_RECTS_SCREEN, 1));
    TRY(kb_mark(V, KB_RECTS, 0));
    k_rects_warp<<<h->sm_count * 16, RECT_WARPS * 32, rects_smem(n), V.s>>>(V.comp, V.rbuf, V.ccl[0], V.ccl[1], V.C, V.pass, n, d, a.minAreaRectMinLen, a.lwTresh, cnt, a.external ? 1 : 0, tasks); LAUNCH_CHECK();
    TRY(kb_mark(V, KB_RECTS, 1));
    CK(cudaMemsetAsync(V.box, 0, (size_t)n * d.NW * sizeof(u32), V.s));
    k_fill_boxes<<<dim3(16, n), 128, 0, V.s>>>(V.rbuf, V.box, V.C, V.pass, d); LAUNCH_CHECK();
    return LFD_OK;
}

// k_hough_vote of the segment lists of `nimg` images (of size d) into their accumulators
static int launch_hough_vote(lfd_handle* h, const HoughBufs& hb, Dims d, const uint2* segs, int* accum, const FrameCtl* C,
                             int pass, int nimg, cudaStream_t s)
{
    unsigned long long* const cnt = (unsigned long long*)h->counters_d;
    if (hough_magic_ok(d.H, d.W, hb.hc.rho))
        k_hough_vote<true><<<dim3(32, hb.hc.ngroups, nimg), HOUGH_THREADS, hb.smem, s>>>(segs, accum, hb.tabSin, hb.tabCos, C, pass, hb.hc, (size_t)d.NW, hb.accum_stride, cnt);
    else
        k_hough_vote<false><<<dim3(32, hb.hc.ngroups, nimg), HOUGH_THREADS, hb.smem, s>>>(segs, accum, hb.tabSin, hb.tabCos, C, pass, hb.hc, (size_t)d.NW, hb.accum_stride, cnt);
    LAUNCH_CHECK();
    return LFD_OK;
}

// the whole pass on frames [f0, f0 + n)
static int run_pass_kernels(lfd_handle* h, int f0, int n, int pass, int flags, cudaStream_t s, bool stage_events)
{
    const Dims d = h->d;
    const lfd_pass_params& pp = pass ? h->params.dim : h->params.bright;
    const PassView V = pass_view(h, f0, n, pass, flags, s);
    FrameCtl* const C = V.C;
    const size_t fN = (size_t)f0 * d.N;
    uint2* const v_segs = h->segs[pass] + (size_t)f0 * 2 * d.NW;
    lfd_result* const v_res = h->res_d + f0;
    const bool taps = flags & LFD_KEEP_TAPS;
    const int tbase = 2 + pass * (T_PER_PASS - 1);   // event index preceding this pass's first stage
    auto stage_event = [&](int i) -> int { if (stage_events) CK(cudaEventRecord(h->ev[tbase + i], s)); return LFD_OK; };
    HoughBufs& hb = h->hb[pass];

    // NMS tap (class per pixel) only with LFD_KEEP_TAPS
    u8* ntap = nullptr;
    if (taps) {
        if (!h->nms_tap[pass]) TRY(dev_alloc(h, &h->nms_tap[pass], (size_t)h->B * d.N));
        ntap = h->nms_tap[pass] + fN;
    }
    // LUT + morphology
    k_lut<<<dim3(n, 1), 256, 0, s>>>(h->hist + (size_t)f0 * 256, h->lut + (size_t)f0 * 256, C, h->B, d.N, pass); LAUNCH_CHECK();
    MorphCfg mc;
    mc.eh = pass ? pp.erode_h : 0; mc.ew = pass ? pp.erode_w : 0; mc.dh = pp.dilate_h; mc.dw = pp.dilate_w;
    u8* etap = nullptr;
    if (taps && pass == 1 && mc.eh > 0) {
        if (!h->eroded_tap) TRY(dev_alloc(h, &h->eroded_tap, (size_t)h->B * d.N));
        etap = h->eroded_tap + fN;
    }
    TRY(kb_mark(V, KB_MORPH, 0));
    {
        const u8* lutp = h->lut + ((size_t)pass * h->B + f0) * 256;
        const int nstrips = ((d.W >> 2) + MARCH_UW - 1) / MARCH_UW, nchunks = (d.H + MARCH_R - 1) / MARCH_R;
        const int nunits = nstrips * nchunks;
        dim3 gg((nunits + MARCH_WPC - 1) / MARCH_WPC, n);
        bool done = false;
        if (h->anyk_on[pass]) {     // erosion into the scratch plane, then dilation of it (or of gray)
            const dim3 ag((d.W + CHORD_SW - 1) / CHORD_SW, (d.H + CHORD_R - 1) / CHORD_R, n);
            auto chords = [](const lfd_handle::AnyElem& e) {
                return ChordSet{e.buf, reinterpret_cast<const u32*>(e.buf + e.kh + 1), e.kh, e.kw, e.kh / 2, e.kw / 2, e.nlev};
            };
            const lfd_handle::AnyElem &ee = h->anyk[pass][0], &de = h->anyk[pass][1];
            const u8* dsrc = V.gray;
            if (pass == 1 && ee.kh > 0) {
                u8* er = h->anyk_eroded + fN;
                k_morph_any<false><<<ag, CHORD_SW, chord_smem(ee.kh, ee.kw, ee.nlev), s>>>(V.gray, lutp, er, nullptr, etap, C,
                                                                                         pass, d, chords(ee));
                LAUNCH_CHECK();
                dsrc = er;
                etap = nullptr;
            }
            k_morph_any<true><<<ag, CHORD_SW, chord_smem(de.kh, de.kw, de.nlev), s>>>(dsrc, lutp, V.morph, V.nz, etap, C, pass,
                                                                                    d, chords(de));
            done = true;
        }
#define MORPH_CASE(EH_, EW_, DH_, DW_)                                                                              \
        if (!done && (d.W % 8) == 0 && mc.eh == EH_ && mc.ew == EW_ && mc.dh == DH_ && mc.dw == DW_) {                \
            k_morph_march<EH_, EW_, DH_, DW_><<<gg, MARCH_WPC * 32, 0, s>>>(V.gray, lutp, V.morph, V.nz, etap, \
                                                               C, pass, d, nstrips, nunits);                    \
            done = true;                                                                                             \
        }
        MORPH_CASE(0, 0, 4, 4)
        MORPH_CASE(3, 3, 9, 9)
        MORPH_CASE(3, 3, 15, 15)
        MORPH_CASE(0, 0, 9, 9)
        MORPH_CASE(0, 0, 3, 3)
#undef MORPH_CASE
        if (!done) {                // any other all-ones rectangle: shared-memory tile kernel
            dim3 mg((d.W + MORPH_TW - 1) / MORPH_TW, (d.H + MORPH_TH - 1) / MORPH_TH, n);
            k_morph<<<mg, 256, 0, s>>>(V.gray, lutp, V.morph, V.nz, etap, C, pass, d, mc);
        }
        LAUNCH_CHECK();
    }
    TRY(kb_mark(V, KB_MORPH, 1));
    TRY(stage_event(1));
    TRY(launch_nms(V, 0, 255, ntap));
    TRY(stage_event(2));
    for (int kind = 0; kind < 2; kind++) {
        TRY(launch_labels(V, kind));
        k_ccl_extremes_flat<<<dim3(CCL_FLAT_CTAS, n), 256, 0, s>>>(V.edges, V.ccl[kind], V.comp, C, pass, d, kind); LAUNCH_CHECK();
        TRY(stage_event(3 + kind));
    }
    TRY(launch_contours(V, {pp.minAreaRectMinLen, pp.lwTresh, pp.contoursMode == 0}, taps));
    TRY(stage_event(5));
    // Hough on the morphology output and on the box image
    int* const v_accum = hb.accum + (size_t)f0 * 2 * hb.accum_stride;
    u64* const v_keys = hb.keys + (size_t)f0 * 2 * hb.key_stride;
    CK(cudaMemsetAsync(v_accum, 0, (size_t)n * 2 * hb.accum_stride * sizeof(int), s));
    // a thread's iterations are a serial chain (load -> ballot -> slot atomic -> store): many CTAs, few iterations each
    k_hough_compact<<<dim3(128, n, 2), 256, 0, s>>>(V.nz, V.box, v_segs, C, pass, d, (size_t)d.NW); LAUNCH_CHECK();
    TRY(kb_mark(V, KB_HOUGH_VOTE, 0));
    TRY(launch_hough_vote(h, hb, d, v_segs, v_accum, C, pass, 2 * n, s));
    TRY(kb_mark(V, KB_HOUGH_VOTE, 1));
    int cells = hb.hc.numangle * hb.hc.numrho;
    int pblocks = (cells + 255) / 256; if (pblocks > 64) pblocks = 64;
    k_hough_peaks<<<dim3(pblocks, 2 * n), 256, 0, s>>>(v_accum, v_keys, C, pass, hb.hc, hb.accum_stride, hb.key_stride); LAUNCH_CHECK();
    k_hough_topk<<<dim3(2, n), 256, 0, s>>>(v_keys, v_res, C, pass, hb.hc, hb.key_stride, pp.nlinesInSet); LAUNCH_CHECK();
    if (flags & LFD_FULL_LINES) {
        if (!hb.lines) CK(cudaMalloc((void**)&hb.lines, (size_t)h->B * 2 * hb.line_stride * sizeof(float)));
        k_hough_sort<<<dim3(2, n), 1024, 0, s>>>(v_keys, hb.lines + (size_t)f0 * 2 * hb.line_stride, C, pass, hb.hc, hb.key_stride, hb.line_stride, hb.max_lines); LAUNCH_CHECK();
    }
    TRY(stage_event(6));
    k_check_theta<<<(n + 63) / 64, 64, 0, s>>>(v_res, C, pass, n, pp.nlinesInSet, pp.dro, pp.thetaTresh, pp.lineSetTresh,
                                              hb.hc.numangle, (unsigned long long*)h->counters_d); LAUNCH_CHECK();
    return stage_event(7);
}

// mode 0: whole-frame pipeline on h->in (un-flipped) ; mode 1/2: standalone bright/dim on frame slot 0
static int run_pipeline(lfd_handle* h, int n, int flags, int mode, bool want_clipped)
{
    const Dims d = h->d;
    cudaStream_t s = h->stream;
    if (!h->have_params) { h->err = "lfd_set_params has not been called"; return LFD_E_STATE; }
    h->inj_recorded = false;           // lfd_submit_injected sets it after this returns
    CK(cudaMemsetAsync(h->counters_d, 0, 16 * sizeof(int64_t), s));
    CK(cudaEventRecord(h->ev[0], s));
    lfd_handle::CachedGraph* cached = nullptr;
    for (auto& g : h->graphs) if (g.n == n && g.flags == flags) cached = &g;
    const bool replay = cached && h->use_graphs && mode == 0 &&
                        !(flags & (LFD_SERIAL_PASSES | LFD_KEEP_TAPS | LFD_FULL_LINES)) && !h->ktiming;
    if (!replay) memset(h->kb_used, 0, sizeof(h->kb_used));       // a replayed graph records the brackets of its capture again
    if (h->ktiming) { h->kn = 0; ktime_mark(h, 0); }
    k_ctl_init<<<(n + 127) / 128, 128, 0, s>>>(h->ctl, h->B, h->res_d, n, mode != 2, mode != 1, h->look, h->look_stride); LAUNCH_CHECK();
    CK(cudaMemsetAsync(h->hist, 0, (size_t)2 * h->B * 256 * sizeof(u32), s));
    if (mode == 0) {
        CK(cudaMemsetAsync(h->starmask, 0, (size_t)n * d.NW * sizeof(u32), s));
        const int total_rects = h->rect_off_h[n];
        if (total_rects > 0) { k_star_mask<<<(total_rects + 3) / 4, 128, 0, s>>>(h->rects_d, h->rect_off_d, n, total_rects, h->starmask, d); LAUNCH_CHECK(); }
    }
    float* clipped = nullptr;
    if (want_clipped) {
        if (!h->clipped) TRY(dev_alloc(h, &h->clipped, (size_t)d.N));
        clipped = h->clipped;
    }
    const lfd_pass_params& pd = h->params.dim;
    CK(cudaEventRecord(h->ev[1], s));
    const int be = (flags & LFD_INPUT_BIGENDIAN) ? 1 : 0;
    u32* hist1 = h->hist + (size_t)h->B * 256;
    if (clipped) {
        int pblocks = (d.N / 4 + 255) / 256; if (pblocks > 1184) pblocks = 1184;
        k_prep_generic<<<dim3(pblocks, n), 256, 0, s>>>(h->in, h->starmask, h->gray[0], h->gray[1], h->hist, hist1, clipped, d, mode,
                                                      (float)pd.minFlux, (float)pd.addFlux); LAUNCH_CHECK();
    } else {
        // one wave of resident CTAs spread over the frames of the batch (a second, partial wave would double the time)
        const float mf = (float)pd.minFlux, af = (float)pd.addFlux;
        // at most 16 frames in flight at a time (fewer concurrent DRAM streams: measured best of 16 / 24 / 32 / all
        // with profiles/lab/prep_lab.cu); the CTAs of the single resident wave walk the rest of the batch
        const int gy = n < 16 ? n : 16;
        int rb = h->prep_grid[mode] / gy; if (rb < 1) rb = 1;
        const int chunks = d.H * ((d.W * 4 + PR_CB - 1) / PR_CB);
        if (rb > (chunks + PR_WARPS - 1) / PR_WARPS) rb = (chunks + PR_WARPS - 1) / PR_WARPS;
        dim3 pg(rb, gy);
#define PREP_LAUNCH(M, E) k_prep<M, E><<<pg, PR_WARPS * 32, PR_SMEM, s>>>(h->in, h->starmask, h->gray[0], h->gray[1], h->hist, hist1, d, n, mf, af)
        if (mode == 0) { if (be) PREP_LAUNCH(0, true); else PREP_LAUNCH(0, false); }
        else if (mode == 1) PREP_LAUNCH(1, false);         // lfd_run_pass: native order only
        else PREP_LAUNCH(2, false);
#undef PREP_LAUNCH
        LAUNCH_CHECK();
    }
    CK(cudaEventRecord(h->ev[2], s));
    // The bright and the dim pass of a batch are independent until the verdict (the reference runs dim only
    // when bright finds nothing, detecttrails.py:125-129; here dim runs for every frame on a second stream and
    // k_finalize drops it where bright detected).  Most kernels after the morphology are latency-bound, so the
    // two passes overlap almost completely.  LFD_SERIAL_PASSES keeps one stream (clean per-stage timings).
    const bool overlap = mode == 0 && !(flags & LFD_SERIAL_PASSES) && !h->ktiming;
    const bool graph = overlap && h->use_graphs && !(flags & (LFD_KEEP_TAPS | LFD_FULL_LINES));
    h->stage_timings_valid = !graph;
    // everything from the fork to the result copies; captured into a CUDA graph when `graph`
    // with overlap and a batch of >= 16 frames the batch is also cut in LFD_BATCH_PARTS parts (two halves): 2 x nsplit
    // independent chains (bright / dim x part) keep the SMs busy through the latency-bound CCL / geometry phases
    const int nsplit = (overlap && n >= 16) ? LFD_BATCH_PARTS : 1;
    auto passes = [&](bool stage_events) -> int {
        if (overlap) {
            CK(cudaEventRecord(h->ev_fork, s));
            for (int k = 0; k < nsplit; k++)
                for (int p = 0; p < 2; p++)
                    if (k || p) CK(cudaStreamWaitEvent(h->xs[k][p], h->ev_fork, 0));
        }
        int fstart = 0;
        for (int k = 0; k < nsplit; k++) {
            const int cnt = (n - fstart + (nsplit - k) - 1) / (nsplit - k);     // first parts take the remainder
            cudaStream_t sb = overlap ? h->xs[k][0] : s, sd = overlap ? h->xs[k][1] : s;
            const bool ev = stage_events && k == 0;
            h->cur_part = k;
            if (mode != 2) TRY(run_pass_kernels(h, fstart, cnt, 0, flags, sb, ev));
            else if (k == 0) for (int i = 3; i <= T_PER_PASS + 1; i++) CK(cudaEventRecord(h->ev[i], s));
            if (mode != 1) TRY(run_pass_kernels(h, fstart, cnt, 1, flags, sd, ev));
            else if (k == 0) for (int i = T_PER_PASS + 2; i < N_TIMINGS; i++) CK(cudaEventRecord(h->ev[i], s));
            fstart += cnt;
        }
        if (overlap)
            for (int k = 0; k < nsplit; k++)
                for (int p = 0; p < 2; p++)
                    if (k || p) { CK(cudaEventRecord(h->xjoin[k][p], h->xs[k][p])); CK(cudaStreamWaitEvent(s, h->xjoin[k][p], 0)); }
        k_finalize<<<(n + 127) / 128, 128, 0, s>>>(h->ctl, h->B, h->res_d, n, mode, (unsigned long long*)h->counters_d); LAUNCH_CHECK();
        CK(cudaMemcpyAsync(h->res_h, h->res_d, (size_t)n * sizeof(lfd_result), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(h->ctl_h, h->ctl, (size_t)n * sizeof(FrameCtl), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(h->ctl_h + h->B, h->ctl + h->B, (size_t)n * sizeof(FrameCtl), cudaMemcpyDeviceToHost, s));
        CK(cudaMemcpyAsync(h->counters_h, h->counters_d, 16 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
        return LFD_OK;
    };
    if (graph) {
        if (!cached) {
            if ((int)h->graphs.size() >= GRAPH_CACHE) { cudaGraphExecDestroy(h->graphs.front().exec); h->graphs.erase(h->graphs.begin()); }
            const int64_t l0 = h->launches;
            CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
            const int rc = passes(false);
            cudaGraph_t g = nullptr;
            cudaError_t ce = cudaStreamEndCapture(s, &g);
            if (rc != LFD_OK) { if (g) cudaGraphDestroy(g); cudaGetLastError(); return rc; }
            if (ce != cudaSuccess) { h->err = std::string("cudaStreamEndCapture: ") + cudaGetErrorString(ce); return LFD_E_CUDA; }
            cudaGraphExec_t exec = nullptr;
            ce = cudaGraphInstantiate(&exec, g, 0);
            cudaGraphDestroy(g);
            if (ce != cudaSuccess) { h->err = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ce); return LFD_E_CUDA; }
            h->graphs.push_back({exec, n, flags, h->launches - l0});
            h->launches = l0;
            cached = &h->graphs.back();
        }
        CK(cudaGraphLaunch(cached->exec, s));
        h->launches += cached->launches;
    } else {
        TRY(passes(true));
    }
    CK(cudaEventRecord(h->ev[N_TIMINGS], s));
    h->last_n = n; h->last_flags = flags; h->pending = true;
    h->in_whole = mode == 0; h->in_be = be != 0;
    return LFD_OK;
}

static void CUDART_CB gate_release_cb(void* p) { flock((int)(intptr_t)p, LOCK_UN); }

// star-rectangle offsets of n frames: rect_offsets[0] == 0 and at most max_star_rects per frame
static int check_rect_offsets(lfd_handle* h, int n, const int32_t* rect_offsets)
{
    if (rect_offsets[0] != 0) { h->err = "rect_offsets[0] must be 0"; return LFD_E_ARG; }
    for (int f = 0; f < n; f++) {
        int c = rect_offsets[f + 1] - rect_offsets[f];
        if (c < 0 || c > h->cfg.max_star_rects) { h->err = "too many star rectangles for a frame (lfd_config.max_star_rects)"; return LFD_E_CAPACITY; }
    }
    return LFD_OK;
}

static int stage_rects(lfd_handle* h, int n, const int32_t* rects, const int32_t* rect_offsets)
{
    if (!rects || !rect_offsets) {
        for (int f = 0; f <= n; f++) h->rect_off_h[f] = 0;
    } else {
        TRY(check_rect_offsets(h, n, rect_offsets));
        memcpy(h->rect_off_h, rect_offsets, ((size_t)n + 1) * sizeof(int));
        memcpy(h->rects_h, rects, (size_t)rect_offsets[n] * sizeof(int4));
        CK(cudaMemcpyAsync(h->rects_d, h->rects_h, (size_t)rect_offsets[n] * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    }
    CK(cudaMemcpyAsync(h->rect_off_d, h->rect_off_h, ((size_t)n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    return LFD_OK;
}

extern "C" int lfd_upload(lfd_handle* h, const float* frames, int n, const int32_t* rects, const int32_t* rect_offsets, int flags)
{
    if (!h || n < 1 || n > h->B) { if (h) h->err = "bad batch size"; return LFD_E_ARG; }
    TRY(enter(h));
    TRY(stage_rects(h, n, rects, rect_offsets));
    const float* src = frames ? frames : h->frames_h;
    // Copy gate: wait (bounded) for this rank's slot of its host bridge, copy, and let a host callback on the stream free
    // the slot when the copy has completed.  With four GPUs behind one ~117 GB/s bridge the four concurrent 781 MB copies
    // are served unfairly (21-37 GB/s per GPU, profiles/h2d_lab_g8.txt) and the slowest rank sets the pace of a job that
    // gives every rank the same work; two copies at a time run at ~55 GB/s each and every rank gets the same share.
    bool held = false;
    if (h->gate_fd >= 0) {
        struct timespec t0, t1;
        clock_gettime(CLOCK_MONOTONIC, &t0);
        for (;;) {
            if (flock(h->gate_fd, LOCK_EX | LOCK_NB) == 0) { held = true; break; }
            clock_gettime(CLOCK_MONOTONIC, &t1);
            if ((t1.tv_sec - t0.tv_sec) * 1000.0 + (t1.tv_nsec - t0.tv_nsec) / 1e6 > 250.0) { h->gate_timeouts++; break; }   // never deadlock on a peer
            usleep(40);
        }
        h->gate_waits++;
    }
    cudaError_t ce = cudaMemcpyAsync(h->in, src, (size_t)n * h->d.N * sizeof(float), cudaMemcpyHostToDevice, h->stream);
    if (held) {
        if (ce != cudaSuccess || cudaLaunchHostFunc(h->stream, gate_release_cb, (void*)(intptr_t)h->gate_fd) != cudaSuccess)
            flock(h->gate_fd, LOCK_UN);
    }
    if (ce != cudaSuccess) { h->err = std::string("cudaMemcpyAsync(H2D): ") + cudaGetErrorString(ce); return LFD_E_CUDA; }
    h->last_flags = flags;
    h->in_whole = h->in_injected = false;
    return LFD_OK;
}

// Share the host->device copy slot named by `lock_path` (an advisory lock file, created if missing) with the other
// processes that name the same file; NULL or "" removes the gate.  See lfd_upload.
extern "C" int lfd_set_h2d_gate(lfd_handle* h, const char* lock_path)
{
    if (!h) return LFD_E_ARG;
    if (h->gate_fd >= 0) { flock(h->gate_fd, LOCK_UN); close(h->gate_fd); h->gate_fd = -1; }
    if (!lock_path || !lock_path[0]) return LFD_OK;
    int fd = open(lock_path, O_RDWR | O_CREAT | O_CLOEXEC, 0666);
    if (fd < 0) { h->err = std::string("lfd_set_h2d_gate: cannot open ") + lock_path; return LFD_E_ARG; }
    h->gate_fd = fd;
    return LFD_OK;
}

extern "C" int lfd_submit(lfd_handle* h, const float* frames, int n, const int32_t* rects, const int32_t* rect_offsets, int flags)
{
    TRY(lfd_upload(h, frames, n, rects, rect_offsets, flags));
    return run_pipeline(h, n, flags, 0, false);
}

extern "C" int lfd_run_resident(lfd_handle* h, int n, int flags)
{
    if (!h || n < 1 || n > h->B) { if (h) h->err = "bad batch size"; return LFD_E_ARG; }
    TRY(enter(h));
    return run_pipeline(h, n, flags, 0, false);
}

// ------------------------------------------------------------------------------------------------
// injection campaigns: resident bases + per-slot synthetic trails added on the device before k_prep
// ------------------------------------------------------------------------------------------------
// room for n_base bases and the per-slot trail buffers, allocated on first use by lfd_set_base / lfd_capture_bases;
// the current bases are dropped (n_base = 0) until the caller has replaced them
static int inj_reserve(lfd_handle* h, int n_base)
{
    h->n_base = 0;
    if (n_base > h->base_cap) {
        if (h->base_d) { cudaFree(h->base_d); h->base_d = nullptr; }
        h->base_cap = 0;
        CK(cudaMalloc((void**)&h->base_d, (size_t)n_base * h->d.N * sizeof(float)));
        h->base_cap = n_base;
    }
    if (!h->inj_trails_d) {
        TRY(dev_alloc(h, &h->inj_trails_d, (size_t)h->B * LFD_MAX_INJECT_TRAILS));
        TRY(dev_alloc(h, &h->inj_off_d, (size_t)h->B + 1));
        TRY(dev_alloc(h, &h->inj_base_d, (size_t)h->B));
        CK(cudaMallocHost((void**)&h->inj_trails_h, (size_t)h->B * LFD_MAX_INJECT_TRAILS * sizeof(InjTrail)));
        CK(cudaMallocHost((void**)&h->inj_off_h, ((size_t)h->B + 1) * sizeof(int)));
        CK(cudaMallocHost((void**)&h->inj_base_h, (size_t)h->B * sizeof(int)));
        for (int i = 0; i < 2; i++) { CK(cudaEventCreate(&h->ev_inj[i])); CK(cudaEventCreate(&h->ev_cap[i])); }
    }
    return LFD_OK;
}

extern "C" int lfd_set_base(lfd_handle* h, const float* frames, int n_base, const int32_t* rects, const int32_t* rect_offsets)
{
    if (!h) return LFD_E_ARG;
    if (!frames || n_base < 1) { h->err = "lfd_set_base: frames must be non-NULL and n_base >= 1"; return LFD_E_ARG; }
    TRY(enter(h));
    if (rects && rect_offsets) TRY(check_rect_offsets(h, n_base, rect_offsets));
    const size_t N = h->d.N;
    TRY(inj_reserve(h, n_base));
    CK(cudaMemcpyAsync(h->base_d, frames, (size_t)n_base * N * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));          // the caller may free `frames` on return
    h->base_rect_off.assign((size_t)n_base + 1, 0);
    h->base_rects.clear();
    if (rects && rect_offsets) {
        for (int f = 0; f <= n_base; f++) h->base_rect_off[f] = rect_offsets[f];
        h->base_rects.assign((const int4*)rects, (const int4*)rects + rect_offsets[n_base]);
    }
    h->n_base = n_base;
    return LFD_OK;
}

extern "C" int lfd_capture_bases(lfd_handle* h)
{
    if (!h) return LFD_E_ARG;
    TRY(enter(h));
    if (!h->in_whole || h->in_injected) {
        h->err = "lfd_capture_bases: the batch slots do not hold the input of a collected whole-frame batch"; return LFD_E_STATE;
    }
    const int n = h->last_n;
    TRY(inj_reserve(h, n));
    const size_t n16 = (size_t)n * h->d.N / 4;           // W % 4 == 0 (lfd_create)
    const size_t want = (n16 + 4 * CAP_THREADS - 1) / (4 * CAP_THREADS);
    const int grid = (int)(want < (size_t)h->sm_count * 8 ? want : (size_t)h->sm_count * 8);
    CK(cudaEventRecord(h->ev_cap[0], h->stream));
    if (h->in_be) k_capture_bases<true><<<grid, CAP_THREADS, 0, h->stream>>>((const uint4*)h->in, (uint4*)h->base_d, n16);
    else k_capture_bases<false><<<grid, CAP_THREADS, 0, h->stream>>>((const uint4*)h->in, (uint4*)h->base_d, n16);
    LAUNCH_CHECK();
    CK(cudaEventRecord(h->ev_cap[1], h->stream));
    h->cap_recorded = true;
    // the batch's star rectangles are still in the submit staging: every other writer of rects_h (lfd_submit_injected,
    // lfd_blot) also leaves the slots in a state this call refuses
    h->base_rect_off.assign(h->rect_off_h, h->rect_off_h + n + 1);
    h->base_rects.assign(h->rects_h, h->rects_h + h->rect_off_h[n]);
    h->n_base = n;
    return LFD_OK;
}

extern "C" int lfd_set_trail_tables(lfd_handle* h, const float* samples, int n_samples, const lfd_table* tables, int n_tables)
{
    if (!h) return LFD_E_ARG;
    TRY(enter(h));
    if (!samples || !tables || n_samples < 2 || n_tables < 1 || n_tables > LFD_MAX_TRAIL_TABLES) {
        h->err = "lfd_set_trail_tables: samples and tables must be non-NULL, n_samples >= 2, n_tables in 1..LFD_MAX_TRAIL_TABLES";
        return LFD_E_ARG;
    }
    for (int i = 0; i < n_samples; i++)
        if (!isfinite(samples[i])) { h->err = "trail table samples must be finite"; return LFD_E_ARG; }
    for (int k = 0; k < n_tables; k++) {
        const lfd_table& t = tables[k];
        if (t.n < 2 || t.n > LFD_MAX_TABLE_SAMPLES || t.offset < 0 || (int64_t)t.offset + t.n > n_samples) {
            h->err = "a trail table has n outside 2..LFD_MAX_TABLE_SAMPLES or lies outside the samples"; return LFD_E_ARG;
        }
        if (!isfinite(t.lo) || !isfinite(t.hi) || !(t.lo < t.hi) || fmaxf(fabsf(t.lo), fabsf(t.hi)) > 1024.f) {
            h->err = "a trail table needs finite lo < hi with max(|lo|, |hi|) <= 1024"; return LFD_E_ARG;
        }
    }
    if (n_samples > h->tab_cap) {
        if (h->tab_samples_d) { cudaFree(h->tab_samples_d); h->tab_samples_d = nullptr; }
        h->tab_cap = 0;
        h->tables.clear();
        CK(cudaMalloc((void**)&h->tab_samples_d, (size_t)n_samples * sizeof(float)));
        h->tab_cap = n_samples;
    }
    h->tables.clear();
    CK(cudaMemcpyAsync(h->tab_samples_d, samples, (size_t)n_samples * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));          // the caller may free `samples` on return
    h->tables.assign(tables, tables + n_tables);
    return LFD_OK;
}

extern "C" int lfd_submit_injected(lfd_handle* h, int n, const int32_t* base_index, const lfd_trail* trails,
                                   const int32_t* trail_offsets, int flags)
{
    return lfd_submit_injected_shaped(h, n, base_index, trails, nullptr, trail_offsets, flags);
}

extern "C" int lfd_submit_injected_shaped(lfd_handle* h, int n, const int32_t* base_index, const lfd_trail* trails,
                                          const lfd_trail_shape* shapes, const int32_t* trail_offsets, int flags)
{
    if (!h) return LFD_E_ARG;
    TRY(enter(h));
    if (h->n_base < 1) { h->err = "no base frames (call lfd_set_base)"; return LFD_E_STATE; }
    if (n < 1 || n > h->B || !base_index) { h->err = "bad batch size or base_index"; return LFD_E_ARG; }
    if (flags & LFD_INPUT_BIGENDIAN) { h->err = "injected frames are built in native byte order (LFD_INPUT_BIGENDIAN)"; return LFD_E_ARG; }
    if (!trails != !trail_offsets || (trail_offsets && trail_offsets[0] != 0)) { h->err = "bad trails / trail_offsets"; return LFD_E_ARG; }
    const int ntab = (int)h->tables.size();
    // validate everything before anything is staged or launched
    for (int f = 0; f < n; f++) {
        if (base_index[f] < 0 || base_index[f] >= h->n_base) { h->err = "base_index out of range"; return LFD_E_ARG; }
        if (!trail_offsets) continue;
        const int c = trail_offsets[f + 1] - trail_offsets[f];
        if (c < 0 || c > LFD_MAX_INJECT_TRAILS) { h->err = "a slot has more than LFD_MAX_INJECT_TRAILS trails"; return LFD_E_ARG; }
        for (int k = trail_offsets[f]; k < trail_offsets[f + 1]; k++) {
            const lfd_trail& t = trails[k];
            const lfd_trail_shape s = shapes ? shapes[k] : lfd_trail_shape{-1, -1};
            if (s.profile < -1 || s.lightcurve < -1) { h->err = "a trail table index is below -1"; return LFD_E_ARG; }
            if ((s.profile >= 0 || s.lightcurve >= 0) && ntab == 0) { h->err = "a trail names a table and no pool is set (call lfd_set_trail_tables)"; return LFD_E_STATE; }
            if (s.profile >= ntab || s.lightcurve >= ntab) { h->err = "a trail table index is not in the pool"; return LFD_E_ARG; }
            if (!isfinite(t.x0) || !isfinite(t.y0) || !isfinite(t.x1) || !isfinite(t.y1) || !isfinite(t.peak) ||
                (s.profile < 0 && !(isfinite(t.sigma) && t.sigma > 0.f))) {
                h->err = "trail values must be finite, with sigma > 0 for a Gaussian profile"; return LFD_E_ARG;
            }
        }
    }
    // per-slot star rectangles from the slot's base, into the lfd_submit staging
    int total = 0;
    for (int f = 0; f < n; f++) {
        const int b = base_index[f], c = h->base_rect_off[b + 1] - h->base_rect_off[b];
        h->rect_off_h[f] = total;
        if (c) memcpy(h->rects_h + total, h->base_rects.data() + h->base_rect_off[b], (size_t)c * sizeof(int4));
        total += c;
    }
    h->rect_off_h[n] = total;
    if (total) CK(cudaMemcpyAsync(h->rects_d, h->rects_h, (size_t)total * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->rect_off_d, h->rect_off_h, ((size_t)n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    // trails in the kernel's form: unit vector and length in double from the float32 end points, rounded to float32
    int nt = 0;
    for (int f = 0; f < n; f++) {
        h->inj_base_h[f] = base_index[f];
        h->inj_off_h[f] = nt;
        if (!trail_offsets) continue;
        for (int k = trail_offsets[f]; k < trail_offsets[f + 1]; k++) {
            const lfd_trail& t = trails[k];
            const double dx = (double)t.x1 - (double)t.x0, dy = (double)t.y1 - (double)t.y0, L = hypot(dx, dy);
            const lfd_trail_shape s = shapes ? shapes[k] : lfd_trail_shape{-1, -1};
            InjTrail& q = h->inj_trails_h[nt++];
            q.x0 = t.x0; q.y0 = t.y0; q.sigma = t.sigma; q.peak = t.peak;
            q.L = (float)L;
            q.ux = L > 0 ? (float)(dx / L) : 0.f;
            q.uy = L > 0 ? (float)(dy / L) : 0.f;
            if (L == 0) q.L = 0.f;
            if (s.profile < 0) {
                const float pad = (float)(ceil(5.0 * (double)t.sigma) + 1.0);
                q.dlo = -pad; q.dhi = pad; q.poff = q.pn = 0; q.inv = 0.f;
            } else {
                const lfd_table& p = h->tables[s.profile];
                q.dlo = p.lo; q.dhi = p.hi; q.poff = p.offset; q.pn = p.n;
                q.inv = (float)((double)(p.n - 1) / ((double)p.hi - (double)p.lo));
            }
            if (s.lightcurve < 0 || q.L == 0.f) {
                q.loff = q.lm = 0; q.c = 0.f;
            } else {
                const lfd_table& a = h->tables[s.lightcurve];
                q.loff = a.offset; q.lm = a.n;
                q.c = (float)((double)(a.n - 1) / (double)q.L);
            }
        }
    }
    h->inj_off_h[n] = nt;
    if (nt) CK(cudaMemcpyAsync(h->inj_trails_d, h->inj_trails_h, (size_t)nt * sizeof(InjTrail), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->inj_off_d, h->inj_off_h, ((size_t)n + 1) * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->inj_base_d, h->inj_base_h, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    CK(cudaEventRecord(h->ev_inj[0], h->stream));
    h->in_injected = true;
    k_inject<<<dim3((h->d.H + INJ_ROWS - 1) / INJ_ROWS, n), INJ_THREADS, 0, h->stream>>>(h->base_d, h->inj_base_d, h->inj_trails_d,
                                                                                       h->inj_off_d, h->tab_samples_d, h->in, h->d); LAUNCH_CHECK();
    CK(cudaEventRecord(h->ev_inj[1], h->stream));
    TRY(run_pipeline(h, n, flags, 0, false));
    h->inj_recorded = true;
    return LFD_OK;
}

extern "C" int lfd_wait(lfd_handle* h, lfd_result* out)
{
    if (!h) return LFD_E_ARG;
    cudaSetDevice(h->device);
    if (!h->pending) { h->err = "nothing submitted"; return LFD_E_STATE; }
    h->pending = false;
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < N_TIMINGS; i++) {
        float ms = 0.f;
        // in graph mode only the setup and k_prep brackets (recorded outside the graph) exist
        if (h->stage_timings_valid || i < 2)
            if (cudaEventElapsedTime(&ms, h->ev[i], h->ev[i + 1]) != cudaSuccess) { ms = 0.f; cudaGetLastError(); }
        h->timings[i] = ms;
    }
    memset(h->kb_ms, 0, sizeof(h->kb_ms));
    memset(h->kb_launches, 0, sizeof(h->kb_launches));
    for (int k = 0; k < LFD_BATCH_PARTS; k++)
        for (int p = 0; p < 2; p++)
            for (int b = 0; b < KB_COUNT; b++) {
                if (!h->kb_used[k][p][b]) continue;
                float ms = 0.f;
                if (cudaEventElapsedTime(&ms, h->kb[k][p][b][0], h->kb[k][p][b][1]) != cudaSuccess) { cudaGetLastError(); continue; }
                h->kb_ms[p][b] += ms;
                h->kb_launches[p][b]++;
            }
    h->inj_ms = 0.f;
    if (h->inj_recorded && cudaEventElapsedTime(&h->inj_ms, h->ev_inj[0], h->ev_inj[1]) != cudaSuccess) { h->inj_ms = 0.f; cudaGetLastError(); }
    h->cap_ms = 0.f; h->cap_launches = 0;
    if (h->cap_recorded) {
        h->cap_recorded = false;
        if (cudaEventElapsedTime(&h->cap_ms, h->ev_cap[0], h->ev_cap[1]) == cudaSuccess) h->cap_launches = 1;
        else { h->cap_ms = 0.f; cudaGetLastError(); }
    }
    if (out) memcpy(out, h->res_h, (size_t)h->last_n * sizeof(lfd_result));
    return LFD_OK;
}

// Bracketed kernels of the last collected batch: name, pass, summed duration over the batch parts and number of launches.
extern "C" int lfd_get_kernel_times(lfd_handle* h, int index, const char** name, int* pass, float* ms, int* launches)
{
    if (!h || index < 0 || index > 2 * KB_COUNT + 1) return LFD_E_ARG;
    if (index == 2 * KB_COUNT) {       // k_inject, bracketed on every lfd_submit_injected (outside the graph)
        const bool on = h->inj_recorded && !h->pending;
        if (name) *name = "k_inject";
        if (pass) *pass = 0;
        if (ms) *ms = on ? h->inj_ms : 0.f;
        if (launches) *launches = on ? 1 : 0;
        return LFD_OK;
    }
    if (index == 2 * KB_COUNT + 1) {   // k_capture_bases, bracketed on every lfd_capture_bases before this batch
        const bool on = h->cap_launches && !h->pending;
        if (name) *name = "k_capture_bases";
        if (pass) *pass = 0;
        if (ms) *ms = on ? h->cap_ms : 0.f;
        if (launches) *launches = on ? 1 : 0;
        return LFD_OK;
    }
    const int p = index / KB_COUNT, b = index % KB_COUNT;
    if (name) *name = k_bracket_names[b];
    if (pass) *pass = p;
    if (ms) *ms = h->kb_ms[p][b];
    if (launches) *launches = h->kb_launches[p][b];
    return LFD_OK;
}

extern "C" int lfd_run_pass(lfd_handle* h, int pass, float* img, int flags, int writeback, lfd_result* out)
{
    if (!h || !img || (pass != 0 && pass != 1)) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    TRY(enter(h));
    if (flags & LFD_INPUT_BIGENDIAN) { h->err = "lfd_run_pass reads and writes back native float32 (LFD_INPUT_BIGENDIAN)"; return LFD_E_ARG; }
    h->rect_off_h[0] = h->rect_off_h[1] = 0;
    CK(cudaMemcpyAsync(h->in, img, (size_t)h->d.N * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    TRY(run_pipeline(h, 1, flags, pass == 0 ? 1 : 2, writeback != 0));
    if (writeback) CK(cudaMemcpyAsync(img, h->clipped, (size_t)h->d.N * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    return lfd_wait(h, out);
}

// remove_stars' blot on a host image
__global__ void k_blot(float* img, const int4* rects, int nrects, Dims d)
{
    int ri = blockIdx.x;
    if (ri >= nrects) return;
    int4 r = rects[ri];
    int r0 = max(r.x, 0), r1 = min(r.y, d.H), c0 = max(r.z, 0), c1 = min(r.w, d.W);
    if (r0 >= r1 || c0 >= c1) return;
    int w = c1 - c0, total = (r1 - r0) * w;
    for (int i = threadIdx.x; i < total; i += blockDim.x) img[(size_t)(r0 + i / w) * d.W + c0 + i % w] = 0.0f;
}

extern "C" int lfd_blot(lfd_handle* h, float* img, const int32_t* rects, int nrects)
{
    if (!h || !img || nrects < 0 || (nrects > 0 && !rects)) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    TRY(enter(h));
    if (nrects > h->B * h->cfg.max_star_rects) { h->err = "too many rectangles"; return LFD_E_CAPACITY; }
    if (nrects == 0) return LFD_OK;
    memcpy(h->rects_h, rects, (size_t)nrects * sizeof(int4));
    CK(cudaMemcpyAsync(h->rects_d, h->rects_h, (size_t)nrects * sizeof(int4), cudaMemcpyHostToDevice, h->stream));
    h->in_whole = false;
    CK(cudaMemcpyAsync(h->in, img, (size_t)h->d.N * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    k_blot<<<nrects, 128, 0, h->stream>>>(h->in, h->rects_d, nrects, h->d); LAUNCH_CHECK();
    CK(cudaMemcpyAsync(img, h->in, (size_t)h->d.N * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// taps
// ------------------------------------------------------------------------------------------------
// entries of the RECTS / RECT_SCREEN taps: x outer contours then y holes, each kind's list at its own offset
static int2 rect_tap_counts(const lfd_handle* h, int frame, int pass)
{
    const FrameCtl& ch = h->ctl_h[(size_t)pass * h->B + frame];
    return make_int2(min(ch.ncomp_saved[pass][0], h->cfg.max_components), min(ch.ncomp_saved[pass][1], h->cfg.max_components));
}

extern "C" int lfd_get_stage_count(lfd_handle* h, int frame, int pass, int stage, int* count)
{
    if (!h || !count || frame < 0 || frame >= h->last_n || (pass != 0 && pass != 1)) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    cudaSetDevice(h->device);
    const HoughBufs& hb = h->hb[pass];
    switch (stage) {
    case LFD_STAGE_RECTS:
    case LFD_STAGE_RECT_SCREEN: {
        const int2 nc = rect_tap_counts(h, frame, pass);
        *count = nc.x + nc.y;
        return LFD_OK;
    }
    // the lines the tap holds: k_hough_sort keeps at most max_lines of them (n_lines in lfd_result is the full count)
    case LFD_STAGE_LINES_EQU: *count = min(h->res_h[frame].n_lines_equ[pass], hb.max_lines); return LFD_OK;
    case LFD_STAGE_LINES_BOX: *count = min(h->res_h[frame].n_lines_box[pass], hb.max_lines); return LFD_OK;
    case LFD_STAGE_ACCUM_EQU:
    case LFD_STAGE_ACCUM_BOX: *count = (int)hb.accum_stride; return LFD_OK;
    default: h->err = "stage has no count"; return LFD_E_ARG;
    }
}

extern "C" int lfd_get_stage(lfd_handle* h, int frame, int pass, int stage, void* host_out, size_t bytes)
{
    if (!h || !host_out || frame < 0 || frame >= h->last_n || (pass != 0 && pass != 1)) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    cudaSetDevice(h->device);
    if (h->pending) { h->err = "batch still pending (call lfd_wait)"; return LFD_E_STATE; }
    const Dims d = h->d;
    cudaStream_t s = h->stream;
    const size_t N = d.N;
    const void* src = nullptr;
    size_t need = N;
    HoughBufs& hb = h->hb[pass];
    switch (stage) {
    case LFD_STAGE_MASK:
    case LFD_STAGE_CANNY:
    case LFD_STAGE_BOX: {
        const u32* m = stage == LFD_STAGE_MASK ? h->starmask : stage == LFD_STAGE_CANNY ? h->edges[pass] : h->box[pass];
        k_expand_mask<<<dim3(256, 1), 256, 0, s>>>(m + (size_t)frame * d.NW, h->tap_u8, d); LAUNCH_CHECK();
        src = h->tap_u8; break;
    }
    case LFD_STAGE_GRAY: src = h->gray[pass] + (size_t)frame * N; break;
    case LFD_STAGE_EQU:
        k_apply_lut<<<dim3(256, 1), 256, 0, s>>>(h->gray[pass] + (size_t)frame * N, h->lut + ((size_t)pass * h->B + frame) * 256, h->tap_u8, d); LAUNCH_CHECK();
        src = h->tap_u8; break;
    case LFD_STAGE_ERODED:
        if (!h->eroded_tap || pass != 1) { h->err = "eroded tap not recorded (dim pass with LFD_KEEP_TAPS)"; return LFD_E_STATE; }
        src = h->eroded_tap + (size_t)frame * N; break;
    case LFD_STAGE_MORPH: src = h->morph[pass] + (size_t)frame * N; break;
    case LFD_STAGE_HIST: src = h->hist + ((size_t)pass * h->B + frame) * 256; need = 256 * sizeof(u32); break;
    case LFD_STAGE_LUT: src = h->lut + ((size_t)pass * h->B + frame) * 256; need = 256; break;
    case LFD_STAGE_NMS:
        if (!h->nms_tap[pass]) { h->err = "NMS tap not recorded (LFD_KEEP_TAPS)"; return LFD_E_STATE; }
        src = h->nms_tap[pass] + (size_t)frame * N; break;
    case LFD_STAGE_FG_LABELS:
    case LFD_STAGE_BG_LABELS: {
        if (!h->labels_tap) TRY(dev_alloc(h, &h->labels_tap, N));
        int kind = stage == LFD_STAGE_BG_LABELS;
        k_ccl_labels<<<(d.H + CCL_WARPS - 1) / CCL_WARPS, CCL_WARPS * 32, 0, s>>>(h->ccl_d[pass][kind], h->labels_tap, h->ctl + (size_t)pass * h->B, pass, d, kind, frame); LAUNCH_CHECK();
        src = h->labels_tap; need = N * sizeof(int); break;
    }
    case LFD_STAGE_RECTS:
    case LFD_STAGE_RECT_SCREEN: {
        const int2 nc = rect_tap_counts(h, frame, pass);
        const int n0 = nc.x, n1 = nc.y;
        const RectBuf& rb = h->rbuf_h[pass][frame];
        const bool rects = stage == LFD_STAGE_RECTS;
        const size_t esz = rects ? sizeof(lfd_rect) : sizeof(int);
        const char* list = rects ? (const char*)rb.rects : (const char*)rb.screened;
        need = (size_t)(n0 + n1) * esz;
        if (bytes < need) { h->err = "buffer too small"; return LFD_E_ARG; }
        if (n0) CK(cudaMemcpyAsync(host_out, list, (size_t)n0 * esz, cudaMemcpyDeviceToHost, s));
        if (n1) CK(cudaMemcpyAsync((char*)host_out + (size_t)n0 * esz, list + (size_t)h->cfg.max_components * esz, (size_t)n1 * esz, cudaMemcpyDeviceToHost, s));
        CK(cudaStreamSynchronize(s));
        return LFD_OK;
    }
    case LFD_STAGE_ACCUM_EQU:
    case LFD_STAGE_ACCUM_BOX:
        src = hb.accum + ((size_t)frame * 2 + (stage == LFD_STAGE_ACCUM_BOX)) * hb.accum_stride;
        need = hb.accum_stride * sizeof(int); break;
    case LFD_STAGE_LINES_EQU:
    case LFD_STAGE_LINES_BOX: {
        if (!hb.lines || !(h->last_flags & LFD_FULL_LINES)) { h->err = "full line lists not recorded (LFD_FULL_LINES)"; return LFD_E_STATE; }
        int which = stage == LFD_STAGE_LINES_BOX;
        int nl = which ? h->res_h[frame].n_lines_box[pass] : h->res_h[frame].n_lines_equ[pass];
        if (nl < 0) nl = 0;
        if (nl > hb.max_lines) nl = hb.max_lines;
        src = hb.lines + ((size_t)frame * 2 + which) * hb.line_stride;
        need = (size_t)nl * 2 * sizeof(float);
        if (need == 0) return LFD_OK;
        break;
    }
    case LFD_STAGE_CLIPPED:
        if (!h->clipped) { h->err = "clipped image not recorded"; return LFD_E_STATE; }
        src = h->clipped; need = N * sizeof(float); break;
    case LFD_STAGE_INPUT:
        if (!h->in_whole) { h->err = "the batch slots do not hold the frames of a whole-frame run"; return LFD_E_STATE; }
        src = h->in + (size_t)frame * N; need = N * sizeof(float); break;
    default: h->err = "unknown stage"; return LFD_E_ARG;
    }
    if (bytes < need) { h->err = "buffer too small"; return LFD_E_ARG; }
    CK(cudaMemcpyAsync(host_out, src, need, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    if (stage == LFD_STAGE_INPUT && h->in_be) {        // a raw FITS payload: back to native order
        uint32_t* w = (uint32_t*)host_out;
        for (size_t i = 0; i < N; i++) w[i] = __builtin_bswap32(w[i]);
    }
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// standalone cv2.HoughLines
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_hough_dims(int height, int width, double rho, double theta, int* numangle, int* numrho)
{
    if (!numangle || !numrho || !(rho > 0) || !(theta > 0)) return LFD_E_ARG;
    hough_dims_host(height, width, rho, theta, numangle, numrho);
    return LFD_OK;
}

extern "C" int lfd_hough_lines(lfd_handle* h, const uint8_t* img, int height, int width, double rho, double theta,
                               int threshold, float* lines, int max_lines, int* n_lines, int32_t* accum)
{
    if (!h || !img || height < 1 || width < 1 || height > 65535 || width > 65535 * 32) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    TRY(enter(h));
    cudaStream_t s = h->stream;
    Dims d; d.H = height; d.W = width; d.WW = (width + 31) / 32; d.N = height * width; d.NW = height * d.WW;
    HoughScratch& hs = h->hs;
    if (hs.H != height || hs.W != width) {
        hough_scratch_free(hs);
        CK(cudaMalloc((void**)&hs.img, (size_t)d.N));
        CK(cudaMalloc((void**)&hs.mask, (size_t)d.NW * sizeof(u32)));
        CK(cudaMalloc((void**)&hs.segs, (size_t)2 * d.NW * sizeof(uint2)));
        CK(cudaMalloc((void**)&hs.ctl, 2 * sizeof(FrameCtl)));
        CK(cudaMalloc((void**)&hs.res, sizeof(lfd_result)));
        hs.H = height; hs.W = width;
    }
    TRY(hough_setup(h, &hs.hb, height, width, rho, theta, threshold, 1, true, 0));
    HoughBufs& hb = hs.hb;
    CK(cudaMemcpyAsync(hs.img, img, (size_t)d.N, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(h->counters_d, 0, 16 * sizeof(int64_t), s));
    k_ctl_init<<<1, 32, 0, s>>>(hs.ctl, 1, hs.res, 1, 1, 0, nullptr, 0); LAUNCH_CHECK();
    // mark Hough as enabled for pass 0
    FrameCtl c; memset(&c, 0, sizeof(c)); c.active[0] = 1; c.hough[0] = 1;
    CK(cudaMemcpyAsync(hs.ctl, &c, sizeof(c), cudaMemcpyHostToDevice, s));
    // device times of the four phases -> lfd_get_timings entries 0..3 (pack+compact, vote, peaks, sort)
    CK(cudaEventRecord(h->ev[0], s));
    k_pack_mask<<<592, 256, 0, s>>>(hs.img, hs.mask, d); LAUNCH_CHECK();
    CK(cudaMemsetAsync(hb.accum, 0, (size_t)2 * hb.accum_stride * sizeof(int), s));
    // which = 0 only: pass the same mask twice and ignore slot 1
    k_hough_compact<<<dim3(64, 1, 1), 256, 0, s>>>(hs.mask, hs.mask, hs.segs, hs.ctl, 0, d, (size_t)d.NW); LAUNCH_CHECK();
    CK(cudaEventRecord(h->ev[1], s));
    TRY(launch_hough_vote(h, hb, d, hs.segs, hb.accum, hs.ctl, 0, 1, s));
    CK(cudaEventRecord(h->ev[2], s));
    long long cells = (long long)hb.hc.numangle * hb.hc.numrho;
    int pblocks = (int)((cells + 255) / 256); if (pblocks > 1184) pblocks = 1184;
    k_hough_peaks<<<dim3(pblocks, 1), 256, 0, s>>>(hb.accum, hb.keys, hs.ctl, 0, hb.hc, hb.accum_stride, hb.key_stride); LAUNCH_CHECK();
    CK(cudaEventRecord(h->ev[3], s));
    // the full sort is only needed when the caller wants the line list (n_lines and the accumulator do not depend on it)
    if (lines && max_lines > 0) { k_hough_sort<<<dim3(1, 1), 1024, 0, s>>>(hb.keys, hb.lines, hs.ctl, 0, hb.hc, hb.key_stride, hb.line_stride, hb.max_lines); LAUNCH_CHECK(); }
    CK(cudaEventRecord(h->ev[4], s));
    FrameCtl out;
    CK(cudaMemcpyAsync(&out, hs.ctl, sizeof(out), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h->counters_h, h->counters_d, 16 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memset(h->timings, 0, sizeof(h->timings));
    for (int i = 0; i < 4; i++)
        if (cudaEventElapsedTime(&h->timings[i], h->ev[i], h->ev[i + 1]) != cudaSuccess) { h->timings[i] = 0.f; cudaGetLastError(); }
    h->counters_h[0] = out.nnz[0];
    h->counters_h[2] = (int64_t)out.nnz[0] * hb.hc.numangle;
    int np = out.npeaks[0];
    if (n_lines) *n_lines = np;
    int ncopy = np < max_lines ? np : max_lines;
    if (ncopy > hb.max_lines) ncopy = hb.max_lines;
    if (lines && ncopy > 0) CK(cudaMemcpy(lines, hb.lines, (size_t)ncopy * 2 * sizeof(float), cudaMemcpyDeviceToHost));
    if (accum) CK(cudaMemcpy(accum, hb.accum, hb.accum_stride * sizeof(int), cudaMemcpyDeviceToHost));
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// standalone cv2.Canny (aperture 3, L1 gradient) on a host uint8 image of the handle's frame size
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_canny(lfd_handle* h, const uint8_t* img, int low, int high, uint8_t* edges_out)
{
    if (!h || !img || !edges_out || low < 0 || high < low) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    TRY(enter(h));
    const Dims d = h->d;
    cudaStream_t s = h->stream;
    const PassView V = pass_view(h, 0, 1, 0, 0, s);      // frame 0 of the bright pass
    CK(cudaMemcpyAsync(V.morph, img, (size_t)d.N, cudaMemcpyHostToDevice, s));
    k_ctl_init<<<1, 32, 0, s>>>(h->ctl, h->B, h->res_d, 1, 1, 0, h->look, h->look_stride); LAUNCH_CHECK();
    // device times -> lfd_get_timings entries 0..1 (Sobel + NMS incl. the input mask, hysteresis by run CCL)
    CK(cudaEventRecord(h->ev[0], s));
    k_pack_mask<<<592, 256, 0, s>>>(V.morph, V.nz, d); LAUNCH_CHECK();
    TRY(launch_nms(V, low, high, nullptr));
    CK(cudaEventRecord(h->ev[1], s));
    TRY(launch_labels(V, 0));
    CK(cudaEventRecord(h->ev[2], s));
    k_expand_mask<<<dim3(592, 1), 256, 0, s>>>(V.edges, h->tap_u8, d); LAUNCH_CHECK();
    FrameCtl out;
    CK(cudaMemcpyAsync(&out, V.C, sizeof(out), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(edges_out, h->tap_u8, (size_t)d.N, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    memset(h->timings, 0, sizeof(h->timings));
    for (int i = 0; i < 2; i++)
        if (cudaEventElapsedTime(&h->timings[i], h->ev[i], h->ev[i + 1]) != cudaSuccess) { h->timings[i] = 0.f; cudaGetLastError(); }
    if (out.status & LFD_FRAME_OVERFLOW) { h->err = "edge map has more runs than lfd_config.max_runs"; return LFD_E_CAPACITY; }
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// standalone fit_minAreaRect (processfield.py:201-263): Canny -> contours -> minAreaRect filter -> box image
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_fit_min_area_rect(lfd_handle* h, const uint8_t* img, int contoursMode, int contoursMethod,
                                     double minAreaRectMinLen, double lwTresh, uint8_t* box_out, int* detection)
{
    if (!h || !img || !box_out || !detection) { if (h) h->err = "bad argument"; return LFD_E_ARG; }
    TRY(enter(h));
    if (!h->have_params) { h->err = "lfd_set_params has not been called"; return LFD_E_STATE; }
    TRY(check_contours_args(h, contoursMode, contoursMethod));
    const Dims d = h->d;
    cudaStream_t s = h->stream;
    const PassView V = pass_view(h, 0, 1, 0, 0, s);      // frame 0 of the bright pass
    CK(cudaMemcpyAsync(V.morph, img, (size_t)d.N, cudaMemcpyHostToDevice, s));
    CK(cudaMemsetAsync(h->counters_d, 0, 16 * sizeof(int64_t), s));
    k_ctl_init<<<1, 32, 0, s>>>(h->ctl, h->B, h->res_d, 1, 1, 0, h->look, h->look_stride); LAUNCH_CHECK();
    k_pack_mask<<<592, 256, 0, s>>>(V.morph, V.nz, d); LAUNCH_CHECK();
    TRY(launch_nms(V, 0, 255, nullptr));
    for (int kind = 0; kind < 2; kind++) {
        TRY(launch_labels(V, kind));
        k_ccl_extremes_flat<<<dim3(CCL_FLAT_CTAS, 1), 256, 0, s>>>(V.edges, V.ccl[kind], V.comp, V.C, 0, d, kind); LAUNCH_CHECK();
    }
    // the box image is the call's output and its RECTS tap every rectangle: fit every contour
    TRY(launch_contours(V, {minAreaRectMinLen, lwTresh, contoursMode == 0}, true));
    k_expand_mask<<<dim3(592, 1), 256, 0, s>>>(V.box, h->tap_u8, d); LAUNCH_CHECK();
    FrameCtl out;
    CK(cudaMemcpyAsync(&out, V.C, sizeof(out), cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(box_out, h->tap_u8, (size_t)d.N, cudaMemcpyDeviceToHost, s));
    CK(cudaMemcpyAsync(h->counters_h, h->counters_d, 16 * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    // the RECTS tap of (frame 0, bright pass) reads its counts from the host copy of the frame's control block; no
    // k_check_theta runs here to save them, so save this call's own counts
    h->ctl_h[0].ncomp_saved[0][0] = out.ncomp[0];
    h->ctl_h[0].ncomp_saved[0][1] = out.ncomp[1];
    if (out.status & LFD_FRAME_OVERFLOW) { h->err = "per-frame work list overflow (lfd_config.max_runs / max_components)"; return LFD_E_CAPACITY; }
    *detection = out.hough[0] ? 1 : 0;
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// micro-benchmark: peak shared-memory atomic rate (denominator for the Hough vote kernel)
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_smem_atomic_peak(lfd_handle* h, double* gops)
{
    if (!h || !gops) return LFD_E_ARG;
    cudaSetDevice(h->device);
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, h->device));
    const int iters = 4096, blocks = prop.multiProcessorCount * 8;
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    k_smem_atomic_peak<<<blocks, 256, 0, h->stream>>>(64, (unsigned*)h->counters_d + 30); LAUNCH_CHECK();      // warm-up
    float best = 1e30f;
    for (int r = 0; r < 5; r++) {
        CK(cudaEventRecord(a, h->stream));
        k_smem_atomic_peak<<<blocks, 256, 0, h->stream>>>(iters, (unsigned*)h->counters_d + 30); LAUNCH_CHECK();
        CK(cudaEventRecord(b, h->stream));
        CK(cudaEventSynchronize(b));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, a, b));
        if (ms < best) best = ms;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    *gops = (double)blocks * 256.0 * 8.0 * iters / (best * 1e6);
    return LFD_OK;
}

// ------------------------------------------------------------------------------------------------
// introspection
// ------------------------------------------------------------------------------------------------
extern "C" int lfd_get_timings(lfd_handle* h, float* ms, int max_entries, int* n_entries)
{
    if (!h || !ms) return LFD_E_ARG;
    int n = N_TIMINGS < max_entries ? N_TIMINGS : max_entries;
    for (int i = 0; i < n; i++) ms[i] = h->timings[i];
    if (n_entries) *n_entries = n;
    return LFD_OK;
}

// caller-placed CUDA-event timestamps on the handle's stream (benchmark timing on the device)
extern "C" int lfd_timer_mark(lfd_handle* h, int slot)
{
    if (!h || slot < 0 || slot >= 4) return LFD_E_ARG;
    cudaSetDevice(h->device);
    CK(cudaEventRecord(h->mark[slot], h->stream));
    return LFD_OK;
}

extern "C" int lfd_timer_elapsed(lfd_handle* h, int slot_start, lfd_handle* h_end, int slot_end, float* ms)
{
    if (!h || !h_end || !ms || slot_start < 0 || slot_start >= 4 || slot_end < 0 || slot_end >= 4) return LFD_E_ARG;
    cudaSetDevice(h->device);
    CK(cudaEventSynchronize(h->mark[slot_start]));
    CK(cudaEventSynchronize(h_end->mark[slot_end]));
    CK(cudaEventElapsedTime(ms, h->mark[slot_start], h_end->mark[slot_end]));
    return LFD_OK;
}

// developer aid: per-launch device times of the last run when LFD_KTIMING=1 (source line of the launch, ms)
extern "C" int lfd_get_ktimings(lfd_handle* h, int* lines, float* ms, int max_entries, int* n_entries)
{
    if (!h || !lines || !ms || !n_entries) return LFD_E_ARG;
    int n = 0;
    for (int i = 1; i < h->kn && n < max_entries; i++) {
        float t = 0.f;
        if (cudaEventElapsedTime(&t, h->kev[i - 1], h->kev[i]) != cudaSuccess) { cudaGetLastError(); t = 0.f; }
        lines[n] = h->kline[i]; ms[n] = t; n++;
    }
    *n_entries = n;
    return LFD_OK;
}

extern "C" const char* lfd_timing_name(int i) { return (i >= 0 && i < N_TIMINGS) ? k_timing_names[i] : ""; }

extern "C" int64_t lfd_kernel_launches(const lfd_handle* h) { return h ? h->launches : 0; }

extern "C" int lfd_get_counters(lfd_handle* h, int64_t* out, int n)
{
    if (!h || !out) return LFD_E_ARG;
    for (int i = 0; i < n && i < 16; i++) out[i] = h->counters_h[i];
    return LFD_OK;
}
