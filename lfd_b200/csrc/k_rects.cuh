// k_rects.cuh - per-contour minAreaRect + length/width filter + boxPoints, and the fillPoly rasteriser
// that builds box_img (as a bit mask).
//
// Reference: fit_minAreaRect, /root/reference/lfd/detecttrails/processfield.py:248-261
//   rect = cv2.minAreaRect(cnt); length/width filter; box = int32(cv2.boxPoints(rect));
//   cv2.fillPoly(box_img, [box], 255); detection = True
#pragma once
#include "common.cuh"
#include "geom.cuh"
#include "k_ccl.cuh"

struct RectBuf {
    lfd_rect* rects;     // [2*maxcomp]  same indexing as CompBuf entries
    int* passing;        // [2*maxcomp]  entry indices of rectangles that passed
    int* screened;       // [2*maxcomp]  1 = k_rects_screen proved that the contour cannot pass (recorded in every mode)
    lfdgeom::Pt* hull;   // [hullcap]
    float* hullf;        // [3*hullcap]
};

// ---- production kernel -------------------------------------------------------------------------------
// Contours of ALL frames of the batch form one flat task list (prefix sums of the per-frame counts in
// shared memory), 32 consecutive tasks per warp:
//   * contours of up to RECT_T_ROWS rows (the bulk: noise blobs) run one-thread-per-contour, hull stack
//     and row extremes in lane-interleaved shared memory, edge vectors recomputed on the fly, so all 32
//     lanes of the warp do calipers at once;
//   * taller contours are then taken one at a time by the whole warp: every lane runs the monotone chain
//     over its slice of rows (both directions), lane 0 / lane 1 re-run the chain over the concatenated
//     partial chains (hull of hulls = the same strict hull in the same order), edge vectors and extreme
//     vertices are computed by all lanes and only the rotating loop is serial.
#define RECT_WARPS 4
#define RECT_SMALL_PTS 128          // hull capacity of the warp path's shared-memory tier
#define RECT_T_ROWS 64              // thread path: contours of at most this many rows ...
#define RECT_T_PTS 40               // ... whose monotone-chain stack never exceeds this (else: warp path)
#define RECT_TPW 8                  // thread-path contours per warp: the kernel is bound by the serial latency of one
                                    // contour, not by issue slots, so 8 busy lanes x 4 times as many warps beats 32 x 1
#define RECT_R_STRIDE (RECT_TPW + 1) // row-extreme staging [RECT_T_ROWS][RECT_TPW + 1]: conflict-free both ways
#define RECT_WARP_WORDS_T (RECT_T_PTS * RECT_TPW + RECT_T_ROWS * RECT_R_STRIDE)
#define RECT_WARP_WORDS_W (6 * RECT_SMALL_PTS + 8)                    // warp path: A, B, vect(2), inv, rows
#define RECT_TALL_PTS 448           // warp path, tall contours: capacity of each packed partial-chain list
#define RECT_WARP_WORDS (RECT_WARP_WORDS_T > RECT_WARP_WORDS_W ? RECT_WARP_WORDS_T : RECT_WARP_WORDS_W)

__host__ __device__ inline size_t rects_smem(int nframes) { return (size_t)RECT_WARPS * RECT_WARP_WORDS * 4 + ((size_t)nframes + 1) * 4; }

// Flat task numbering of the contours of a launch: pre[f] = contours of the active frames before f (fg entries of a
// frame first, then its bg entries).  Warp 0 of the block fills pre[0..nframes]; the caller synchronises.
__device__ __forceinline__ void rect_task_prefix(const CompBuf* __restrict__ comps, const FrameCtl* __restrict__ ctl, int pass,
                                                 int nframes, int* pre)
{
    const int lane = lane_id();
    if ((threadIdx.x >> 5) != 0) return;
    int carry = 0;
    for (int f0 = 0; f0 < nframes; f0 += 32) {
        int ff = f0 + lane, c = 0;
        if (ff < nframes && ctl[ff].active[pass]) {
            int mc = comps[ff].maxcomp;
            c = min(ctl[ff].ncomp[0], mc) + min(ctl[ff].ncomp[1], mc);
        }
        int inc = c;
        for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(FULLMASK, inc, o); if (lane >= o) inc += v; }
        if (ff < nframes) pre[ff + 1] = carry + inc;
        carry += __shfl_sync(FULLMASK, inc, 31);
    }
    if (lane == 0) pre[0] = 0;
}

// task -> (frame, entry, kind): the largest f with pre[f] <= task
__device__ __forceinline__ void rect_task_decode(const int* pre, int nframes, const CompBuf* __restrict__ comps,
                                                 const FrameCtl* __restrict__ ctl, int task, int* f, int* e, int* kind)
{
    int flo = 0, fhi = nframes;
    while (fhi - flo > 1) { int mid = (flo + fhi) >> 1; if (pre[mid] <= task) flo = mid; else fhi = mid; }
    const int i = task - pre[flo];
    const int mc = comps[flo].maxcomp;
    const int n0 = min(ctl[flo].ncomp[0], mc);
    *f = flo;
    *kind = i >= n0;
    *e = *kind ? mc + (i - n0) : i;
}

// ---- aspect screen -------------------------------------------------------------------------------------------------
// A contour passes only if length / width > lwTresh for its minimum-area rectangle.  With P the contour's points, every
// side of that rectangle is P's extent along some direction, so length <= diam(P) <= D (D^2 = bw^2 + bh^2, the squared
// diagonal of P's bounding box) and width >= w(P), the minimum width of P's hull.  The hull lies in a strip of width w(P)
// and length at most diam(P), so area(hull) <= w(P) * D; and the polygon through the row extremes of P (down the
// rowmin side, up the rowmax side) has its vertices in P, so its area A <= area(hull).  Hence
//   length / width <= D^2 / A,
// and a contour with D^2 < lwTresh * A cannot pass, whatever its hull.  2A = sum over consecutive non-empty rows of
// dy * (w_k + w_k+1) with w = rowmax - rowmin, an exact integer.  The test keeps a relative margin of 1e-4 for the float
// rounding of the fitted sides; lwTresh <= 1 or NaN rejects nothing (A <= bw * bh <= D^2 / 2).  It needs no minLen.
#define SCREEN_THREADS 256
#define SCREEN_MARGIN 1e-4

__host__ __device__ inline size_t screen_smem(int nframes) { return ((size_t)nframes + 1) * 4; }

// One thread per contour over the flat task list.  Every contour's verdict goes to rb.screened[e].  With `tasks`
// (production runs), a rejected contour gets its lfd_rect record here (kind 3, never passes) and the others are appended
// to tasks[0 .. ctl[0].nsurv) for k_rects_warp; without it (taps, the standalone fit) k_rects_warp fits every contour.
// counters[15] counts the rejected contours in every mode.
__global__ void __launch_bounds__(SCREEN_THREADS)
k_rects_screen(const CompBuf* __restrict__ comps, RectBuf* __restrict__ rbufs, const CclBuf* __restrict__ ccl0,
               const CclBuf* __restrict__ ccl1, FrameCtl* __restrict__ ctl, int pass, int nframes, Dims d, double lwTresh,
               int* __restrict__ tasks, unsigned long long* __restrict__ counters)
{
    extern __shared__ int spre[];      // [nframes + 1]
    rect_task_prefix(comps, ctl, pass, nframes, spre);
    __syncthreads();
    const int total = spre[nframes], lane = lane_id();
    for (int base = blockIdx.x * SCREEN_THREADS; base < total; base += gridDim.x * SCREEN_THREADS) {
        const int task = base + (int)threadIdx.x;
        const bool valid = task < total;
        bool drop = false;
        int f = 0, e = 0, kind = 0;
        if (valid) {
            rect_task_decode(spre, nframes, comps, ctl, task, &f, &e, &kind);
            const CompBuf& cb = comps[f];
            const int hh = cb.h[e], slot = cb.slot[e];
            const int* __restrict__ rmin = cb.rowmin + slot;
            const int* __restrict__ rmax = cb.rowmax + slot;
            int xlo = 0x7fffffff, xhi = -1, ylo = -1, py = -1, pw = 0;
            long long a2 = 0;
#pragma unroll 4
            for (int r = 0; r < hh; r++) {
                const int a = rmin[r], b = rmax[r];
                if (a > b) continue;                         // empty row
                xlo = min(xlo, a); xhi = max(xhi, b);
                const int w = b - a;
                if (py >= 0) a2 += (long long)(r - py) * (w + pw);
                else ylo = r;
                py = r; pw = w;
            }
            const long long bw = (long long)xhi - xlo, bh = (long long)py - ylo;
            drop = py >= 0 && (double)(bw * bw + bh * bh) * (1.0 + SCREEN_MARGIN) < lwTresh * (0.5 * (double)a2);
            rbufs[f].screened[e] = drop ? 1 : 0;
            if (drop && tasks) {
                lfd_rect o;
                memset(&o, 0, sizeof(o));
                o.kind = 3;                                  // screened: no fit, cannot pass
                Run rr = (kind ? ccl1[f] : ccl0[f]).runs[cb.root[e]];
                o.key = (int)rr.y * d.W + (int)rr.xs;
                rbufs[f].rects[e] = o;
            }
        }
        const unsigned dropped = __ballot_sync(FULLMASK, valid && drop);
        if (lane == 0 && dropped) atomicAdd(&counters[15], (unsigned long long)__popc(dropped));
        if (tasks) {
            const unsigned keep = __ballot_sync(FULLMASK, valid && !drop);
            int slot0 = 0;
            if (lane == 0 && keep) slot0 = atomicAdd(&ctl[0].nsurv, __popc(keep));
            slot0 = __shfl_sync(FULLMASK, slot0, 0);
            if (valid && !drop) tasks[slot0 + __popc(keep & ((1u << lane) - 1u))] = task;
        }
    }
}

__device__ __forceinline__ u32 pt_pack(int x, int y) { return (u32)(x & 0xffff) | ((u32)y << 16); }
__device__ __forceinline__ lfdgeom::Pt pt_unpack(u32 v) { lfdgeom::Pt p; p.x = (int)(v & 0xffffu); p.y = (int)(v >> 16); return p; }

// Monotone-chain stack (element j at st[j * stride]) with its two top entries cached in registers: the
// common case (no pop) touches memory only for the store.
struct Chain {
    u32* st; int k, stride; lfdgeom::Pt t1, t2;       // t1 = top, t2 = second
    __device__ __forceinline__ void init(u32* s, int stride_) { st = s; k = 0; stride = stride_; t1.x = t1.y = t2.x = t2.y = 0; }
    // pops are allowed while the stack holds at least `lo` entries (2 for a fresh chain)
    __device__ __forceinline__ void push(u32 pv, int lo)
    {
        lfdgeom::Pt p = pt_unpack(pv);
        while (k >= lo) {
            int cr = (t1.x - t2.x) * (p.y - t2.y) - (t1.y - t2.y) * (p.x - t2.x);
            if (cr > 0) break;
            k--;
            t1 = t2;
            if (k >= 2) t2 = pt_unpack(st[(k - 2) * stride]);
        }
        st[k * stride] = pv;
        k++;
        t2 = t1; t1 = p;
    }
};

struct PackedHull {
    const u32* a; int n, start, stride;
    __device__ __forceinline__ lfdgeom::Pt operator()(int i) const { int j = i + start; if (j >= n) j -= n; return pt_unpack(a[j * stride]); }
};

__device__ __forceinline__ u64 warp_max64(u64 v)
{
    for (int o = 16; o; o >>= 1) { u64 t = __shfl_xor_sync(FULLMASK, v, o); if (t > v) v = t; }
    return v;
}
__device__ __forceinline__ u64 warp_min64(u64 v)
{
    for (int o = 16; o; o >>= 1) { u64 t = __shfl_xor_sync(FULLMASK, v, o); if (t < v) v = t; }
    return v;
}

// filter (processfield.py:256-257), boxPoints + int32 (:259-260), bookkeeping
__device__ __forceinline__ void emit_rect(const lfdgeom::Rect& r, int e, int kind, int f, int pass, const CompBuf& cb, const RectBuf& rb,
                                          const CclBuf* ccl0, const CclBuf* ccl1, FrameCtl* ctl, Dims d, double minLen, double lwTresh)
{
    lfd_rect o;
    o.cx = r.cx; o.cy = r.cy; o.w = r.w; o.h = r.h; o.angle = r.angle;
    o.kind = kind;
    Run rr = (kind ? ccl1[f] : ccl0[f]).runs[cb.root[e]];   // raster-first run of the component / hole
    o.key = (int)rr.y * d.W + (int)rr.xs;
    float length = r.w > r.h ? r.w : r.h, width = r.w > r.h ? r.h : r.w;
    int passed = 0;
    if ((double)length > minLen && (double)width > minLen)
        if ((double)length / (double)width > lwTresh) passed = 1;
    o.passed = passed;
    float f8[8];
    lfdgeom::box_points(r, f8, o.box);
    rb.rects[e] = o;
    if (passed) {
        ctl[f].hough[pass] = 1;
        int pi = atomicAdd(&ctl[f].npass, 1);
        rb.passing[pi] = e;
    }
}

// one THREAD per contour; T = hull stack [RECT_T_PTS][32] (lane-interleaved), R = this lane's packed row
// extremes (rowmin | rowmax << 16, 0xffffffff = empty row) at stride RECT_R_STRIDE.  Returns false if the
// stack would overflow (the caller then gives the contour to the warp path).  `mask` = lanes running this
// path: the phases are separated by __syncwarp(mask) and there is no early return, so the lanes of a warp
// stay converged (a return inside the loops left them running one after the other).
__device__ __forceinline__ bool rect_thread_path(const u32* R, int hh, int y0, u32* T, u32 mask, lfdgeom::Rect* out)
{
    Chain ch; ch.init(T, RECT_TPW);
    bool ovf = false;
    for (int r = 0; r < hh; r++) {
        u32 v = R[r * RECT_R_STRIDE];
        if (v == 0xffffffffu || ovf) continue;
        int a = (int)(v & 0xffffu), b = (int)(v >> 16);
        if (ch.k + 2 > RECT_T_PTS) { ovf = true; continue; }
        ch.push(pt_pack(a, y0 + r), 2);
        if (b != a) ch.push(pt_pack(b, y0 + r), 2);
    }
    __syncwarp(mask);
    int n = ch.k;
    if (n > 1 && !ovf) {
        const int lo = n + 1;
        bool first = true;
        for (int r = hh - 1; r >= 0; r--) {
            u32 v = R[r * RECT_R_STRIDE];
            if (v == 0xffffffffu || ovf) continue;
            int a = (int)(v & 0xffffu), b = (int)(v >> 16);
            if (ch.k + 2 > RECT_T_PTS) { ovf = true; continue; }
            if (first) first = false;                          // the (y, x) maximum is already on the stack
            else ch.push(pt_pack(b, y0 + r), lo);
            if (a != b) ch.push(pt_pack(a, y0 + r), lo);
        }
        n = ch.k - 1;                                          // the last point equals T[0]
        if (n == 2 && T[0] == T[RECT_TPW]) n = 1;
    }
    if (ovf) n = 0;
    __syncwarp(mask);
    int start = 0, left = 0, bottom = 0, right = 0, top = 0;
    {
        u32 best = 0;
        int lx = 0, rx = 0, ty = 0, by = 0;
        for (int j = 0; j < n; j++) {
            u32 v = T[j * RECT_TPW];
            u32 key = ((v & 0xffffu) << 16) | (v >> 16);       // x, then y
            if (j == 0 || key > best) { best = key; start = j; }
        }
        // extremes in caliper order (index relative to start): first index of min x / max x / max y / min y
        for (int j = 0; j < n; j++) {
            int q = j + start; if (q >= n) q -= n;
            lfdgeom::Pt p = pt_unpack(T[q * RECT_TPW]);
            if (j == 0) { lx = rx = p.x; ty = by = p.y; }
            if (p.x < lx) { lx = p.x; left = j; }
            if (p.x > rx) { rx = p.x; right = j; }
            if (p.y > ty) { ty = p.y; top = j; }
            if (p.y < by) { by = p.y; bottom = j; }
        }
    }
    __syncwarp(mask);
    PackedHull hp; hp.a = T; hp.n = n; hp.start = start; hp.stride = RECT_TPW;
    if (n <= 2) {
        lfdgeom::Pt z; z.x = 0; z.y = 0;
        lfdgeom::min_area_rect_small(n, n > 0 ? hp(0) : z, n > 1 ? hp(1) : z, out);
    } else {
        lfdgeom::FlyEdges<PackedHull> ev; ev.hp = hp; ev.n = n;
        lfdgeom::min_area_rect_core(hp, n, ev, left, bottom, right, top, out);
    }
    __syncwarp(mask);
    return !ovf;
}

// the whole WARP on one contour; lane 0 returns the rectangle
__device__ __forceinline__ void rect_warp_path(const int* __restrict__ rmin, const int* __restrict__ rmax, int hh, int y0,
                                               u32* wsm, u32* gscratch, float* gscratchf, lfdgeom::Rect* out)
{
    const int lane = lane_id();
    // shared-memory tier layout inside the warp's buffer
    u32* sA = wsm; u32* sB = sA + RECT_SMALL_PTS;
    float* sV = reinterpret_cast<float*>(sB + RECT_SMALL_PTS);
    float* sI = sV + 2 * RECT_SMALL_PTS + 4;
    int* sRow = reinterpret_cast<int*>(sI + RECT_SMALL_PTS + 2);
    u32 *A, *B;
    float *vect, *inv;
    const bool tall = 2 * hh > RECT_SMALL_PTS;
    if (!tall) {
        A = sA; B = sB; vect = sV; inv = sI;
        for (int r = lane; r < hh; r += 32) { sRow[r] = rmin[r]; sRow[RECT_SMALL_PTS / 2 + r] = rmax[r]; }
        __syncwarp();
        rmin = sRow; rmax = sRow + RECT_SMALL_PTS / 2;
    } else {
        A = gscratch; B = A + 2 * hh;
        vect = gscratchf; inv = vect + 2 * (size_t)(2 * hh + 2);
    }
    // level 1: per-lane partial chains; B regions are mirrored so that level 2 can run in place
    const int c = (hh + 31) >> 5;
    const int r0 = min(lane * c, hh), r1 = min(r0 + c, hh);
    int ka, kb;
    {
        Chain ca; ca.init(A + 2 * r0, 1);
        for (int r = r0; r < r1; r++) {
            int a = rmin[r], b = rmax[r];
            if (a > b) continue;
            ca.push(pt_pack(a, y0 + r), 2);
            if (b != a) ca.push(pt_pack(b, y0 + r), 2);
        }
        ka = ca.k;
        Chain cbk; cbk.init(B + 2 * (hh - r1), 1);
        for (int r = r1 - 1; r >= r0; r--) {
            int a = rmin[r], b = rmax[r];
            if (a > b) continue;
            cbk.push(pt_pack(b, y0 + r), 2);
            if (a != b) cbk.push(pt_pack(a, y0 + r), 2);
        }
        kb = cbk.k;
    }
    __syncwarp();
    // level 2: lane 0 merges the ascending chains, lane 1 the descending ones (same instruction stream)
    int KA, KB;
    u32 *HA = A, *HB = B;
    bool compacted = false;
    if (tall) {
        // partial chains of a tall contour live in global scratch; they are short, so pack them into the warp's
        // shared memory first: the serial merge then runs at shared-memory latency
        int ia = ka, ib = kb;
        for (int o = 1; o < 32; o <<= 1) {
            int va = __shfl_up_sync(FULLMASK, ia, o), vb = __shfl_down_sync(FULLMASK, ib, o);
            if (lane >= o) ia += va;
            if (lane + o < 32) ib += vb;
        }
        const int suma = __shfl_sync(FULLMASK, ia, 31), sumb = __shfl_sync(FULLMASK, ib, 0);
        if (suma <= RECT_TALL_PTS && sumb <= RECT_TALL_PTS) {
            compacted = true;
            u32* SA = wsm; u32* SB = wsm + RECT_TALL_PTS;
            const u32* ga = A + 2 * r0; const u32* gb = B + 2 * (hh - r1);
            for (int j = 0; j < ka; j++) SA[ia - ka + j] = ga[j];
            for (int j = 0; j < kb; j++) SB[ib - kb + j] = gb[j];       // lanes 31..0 in this order
            __syncwarp();
            Chain cm; cm.init(lane == 1 ? SB : SA, 1);
            if (lane < 2) {
                const u32* src = lane ? SB : SA;
                const int cnt = lane ? sumb : suma;
                for (int j = 0; j < cnt; j++) cm.push(src[j], 2);
            }
            KA = __shfl_sync(FULLMASK, cm.k, 0); KB = __shfl_sync(FULLMASK, cm.k, 1);
            HA = SA; HB = SB;
        }
    }
    if (!compacted) {
        Chain cm; cm.init(lane == 1 ? B : A, 1);
        for (int t = 0; t < 32; t++) {
            int na_t = __shfl_sync(FULLMASK, ka, t), nb_t = __shfl_sync(FULLMASK, kb, 31 - t);
            if (lane < 2) {
                int L = lane ? 31 - t : t;
                int q0 = min(L * c, hh), q1 = min(q0 + c, hh);
                const u32* src = lane ? B + 2 * (hh - q1) : A + 2 * q0;
                int cnt = lane ? nb_t : na_t;
                for (int j = 0; j < cnt; j++) cm.push(src[j], 2);
            }
        }
        KA = __shfl_sync(FULLMASK, cm.k, 0); KB = __shfl_sync(FULLMASK, cm.k, 1);
    }
    const int n = (KA <= 1) ? KA : KA + KB - 2;
    __syncwarp();
    // gather the hull (A chain, then the interior of the B chain).  Hulls of up to RECT_SMALL_PTS vertices -
    // all but pathological ones - go to shared memory, so the serial caliper loop never waits on global memory.
    if (n <= RECT_SMALL_PTS) {
        u32 tmp[RECT_SMALL_PTS / 32];
#pragma unroll
        for (int k = 0; k < RECT_SMALL_PTS / 32; k++) {
            int j = lane + 32 * k;
            tmp[k] = j < n ? (j < KA ? HA[j] : HB[1 + j - KA]) : 0u;
        }
        __syncwarp();
#pragma unroll
        for (int k = 0; k < RECT_SMALL_PTS / 32; k++) {
            int j = lane + 32 * k;
            if (j < n) sA[j] = tmp[k];
        }
        A = sA; vect = sV; inv = sI;
    } else {
        // (only reachable for tall contours: A, vect, inv are the global scratch)
        if (compacted) { for (int j = lane; j < KA; j += 32) A[j] = HA[j]; }
        for (int j = lane; j < KB - 2; j += 32) A[KA + j] = HB[1 + j];
    }
    __syncwarp();
    // caliper start vertex: lexicographic maximum (x, then y)
    u64 bk = 0;
    for (int j = lane; j < n; j += 32) {
        u32 v = A[j];
        u64 k64 = ((u64)(((v & 0xffffu) << 16) | (v >> 16)) << 32) | (u32)j;
        if (k64 > bk) bk = k64;
    }
    bk = warp_max64(bk);
    PackedHull hp; hp.a = A; hp.n = n; hp.start = (int)(bk & 0xffffffffu); hp.stride = 1;
    if (n <= 2) {
        lfdgeom::Pt z; z.x = 0; z.y = 0;
        lfdgeom::min_area_rect_small(n, n > 0 ? hp(0) : z, n > 1 ? hp(1) : z, out);
        return;
    }
    u64 kl = ~0ull, kbm = ~0ull, kr = 0, kt = 0;       // first index of min x / min y / max x / max y
    for (int j = lane; j < n; j += 32) {
        lfdgeom::Pt p = hp(j), q = hp(j + 1 < n ? j + 1 : 0);
        lfdgeom::hull_edge(p, q, &vect[2 * j], &vect[2 * j + 1], &inv[j]);
        u64 lo = (u32)j, hi = 0xffffffffu - (u32)j;
        u64 a = ((u64)(u32)p.x << 32) | lo; if (a < kl) kl = a;
        a = ((u64)(u32)p.y << 32) | lo; if (a < kbm) kbm = a;
        a = ((u64)(u32)p.x << 32) | hi; if (a > kr) kr = a;
        a = ((u64)(u32)p.y << 32) | hi; if (a > kt) kt = a;
    }
    kl = warp_min64(kl); kbm = warp_min64(kbm); kr = warp_max64(kr); kt = warp_max64(kt);
    __syncwarp();
    if (lane == 0) {
        lfdgeom::ArrEdges ev; ev.vect = vect; ev.inv = inv;
        lfdgeom::min_area_rect_core(hp, n, ev, (int)(kl & 0xffffffffu), (int)(kbm & 0xffffffffu),
                                    (int)(0xffffffffu - (u32)(kr & 0xffffffffu)), (int)(0xffffffffu - (u32)(kt & 0xffffffffu)), out);
    }
}

// grid = (any, 1); dynamic smem = rects_smem(nframes).  `tasks`: the survivors of k_rects_screen (ctl[0].nsurv of them),
// one per warp; nullptr = every contour of the launch, RECT_TPW per warp.
__global__ void __launch_bounds__(RECT_WARPS * 32)
k_rects_warp(CompBuf* __restrict__ comps, RectBuf* __restrict__ rbufs, const CclBuf* __restrict__ ccl0,
             const CclBuf* __restrict__ ccl1, FrameCtl* __restrict__ ctl, int pass, int nframes,
             Dims d, double minLen, double lwTresh, unsigned long long* __restrict__ counters, int external_only,
             const int* __restrict__ tasks)
{
    extern __shared__ u32 rsm[];
    const int warp = threadIdx.x >> 5, lane = lane_id();
    u32* wsm = rsm + warp * RECT_WARP_WORDS;
    int* pre = reinterpret_cast<int*>(rsm + RECT_WARPS * RECT_WARP_WORDS);      // [nframes + 1]
    rect_task_prefix(comps, ctl, pass, nframes, pre);
    __syncthreads();
    const int ntasks = tasks ? ctl[0].nsurv : pre[nframes];
    // Survivors are few (a few % of the contours) and mostly the tall ones that take the serial warp path: one per warp,
    // so that they run side by side instead of up to RECT_TPW after one another in one warp.
    const int tpw = tasks ? 1 : RECT_TPW;
    for (int base = (blockIdx.x * RECT_WARPS + warp) * tpw; base < ntasks; base += gridDim.x * RECT_WARPS * tpw) {
        const bool valid = lane < tpw && base + lane < ntasks;
        int f = 0, e = 0, kind = 0, hh = 0, slot = 0, ho = 0, y0 = 0;
        if (valid) {
            const int task = tasks ? tasks[base + lane] : base + lane;
            rect_task_decode(pre, nframes, comps, ctl, task, &f, &e, &kind);
            const CompBuf& cbr = comps[f];
            hh = cbr.h[e]; slot = cbr.slot[e]; ho = cbr.hulloff[e]; y0 = cbr.y0[e];
        }
        bool valid2 = valid;
        if (valid && external_only) {
            // cv2.RETR_EXTERNAL: only outer borders whose surrounding region is the outside of the image.  The region
            // around an edge component is the background component of the pixel left of its raster-first pixel
            // (Suzuki's border following starts there); "outside" = that component reaches the frame border (or the
            // component itself starts in column 0).  Hole borders are never retrieved.
            bool keep = false;
            if (kind == 0) {
                const CclBuf& fg = ccl0[f];
                const CclBuf& bg = ccl1[f];
                Run rr = fg.runs[comps[f].root[e]];
                if (rr.xs == 0) keep = true;
                else {
                    int bid = run_at(bg, rr.y, (int)rr.xs - 1);
                    keep = (bg.flag[bg.parent[bid]] & 1) != 0;
                }
            }
            if (!keep) {
                lfd_rect o;
                memset(&o, 0, sizeof(o));
                o.kind = 2;                      // not retrieved in this contoursMode
                rbufs[f].rects[e] = o;
                valid2 = false;
            }
        }
        bool small = valid2 && hh <= RECT_T_ROWS;
        __syncwarp();
        // stage the row extremes of the 32 contours with coalesced loads: contour l -> column l of R
        u32* Rw = wsm + RECT_T_PTS * RECT_TPW;
        for (int l = 0; l < RECT_TPW; l++) {
            const int hl = __shfl_sync(FULLMASK, small ? hh : 0, l);
            if (hl == 0) continue;
            const int fl = __shfl_sync(FULLMASK, f, l), sl = __shfl_sync(FULLMASK, slot, l);
            const int* gmin = comps[fl].rowmin + sl;
            const int* gmax = comps[fl].rowmax + sl;
            for (int r = lane; r < hl; r += 32) {
                int a = gmin[r], b = gmax[r];
                Rw[r * RECT_R_STRIDE + l] = (a > b) ? 0xffffffffu : ((u32)a | ((u32)b << 16));
            }
        }
        __syncwarp();
        const u32 smask = __ballot_sync(FULLMASK, small);
        if (small) {
            lfdgeom::Rect r;
            small = rect_thread_path(Rw + lane, hh, y0, wsm + lane, smask, &r);
            if (!small) atomicAdd(&counters[12], 1ull);
            if (small) emit_rect(r, e, kind, f, pass, comps[f], rbufs[f], ccl0, ccl1, ctl, d, minLen, lwTresh);
        }
        u32 big = __ballot_sync(FULLMASK, valid2 && !small);
        if (lane == 0 && big) atomicAdd(&counters[11], (unsigned long long)__popc(big));
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1;
            const int bf = __shfl_sync(FULLMASK, f, src), be = __shfl_sync(FULLMASK, e, src), bkind = __shfl_sync(FULLMASK, kind, src);
            const int bhh = __shfl_sync(FULLMASK, hh, src), bslot = __shfl_sync(FULLMASK, slot, src);
            const int bho = __shfl_sync(FULLMASK, ho, src), by0 = __shfl_sync(FULLMASK, y0, src);
            CompBuf cb = comps[bf];
            RectBuf rb = rbufs[bf];
            lfdgeom::Rect r;
            __syncwarp();
            rect_warp_path(cb.rowmin + bslot, cb.rowmax + bslot, bhh, by0, wsm, reinterpret_cast<u32*>(rb.hull + bho),
                           rb.hullf + 3 * (size_t)bho, &r);
            if (lane == 0) emit_rect(r, be, bkind, bf, pass, cb, rb, ccl0, ccl1, ctl, d, minLen, lwTresh);
            __syncwarp();
        }
    }
}

// cv2.fillPoly(box_img, [box], 255) for every passing rectangle; one warp per rectangle.
__global__ void __launch_bounds__(128)
k_fill_boxes(RectBuf* __restrict__ rbufs, u32* __restrict__ box, const FrameCtl* __restrict__ ctl, int pass, Dims d)
{
    int f = blockIdx.y;
    if (!ctl[f].active[pass] || !ctl[f].hough[pass]) return;
    RectBuf rb = rbufs[f];
    u32* bm = box + (size_t)f * d.NW;
    int np = ctl[f].npass;
    int warps = (gridDim.x * blockDim.x) >> 5;
    int lane = lane_id();
    __shared__ lfdgeom::Edge sedge[4][4];
    int wslot = threadIdx.x >> 5;
    for (int pi = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; pi < np; pi += warps) {
        const lfd_rect& R = rb.rects[rb.passing[pi]];
        __syncwarp();
        if (lane < 4) {
            int i = lane, j = (lane + 3) & 3;
            int draw, x0, y0, x1, y1;
            lfdgeom::Edge e;
            lfdgeom::poly_edge(d.W, d.H, R.box[2 * j], R.box[2 * j + 1], R.box[2 * i], R.box[2 * i + 1], &e,
                               &draw, &x0, &y0, &x1, &y1);
            sedge[wslot][lane] = e;
            if (draw) {
                lfdgeom::LineIt it;
                it.init(x0, y0, x1, y1);
                for (int s = 0; s < it.count; s++) {
                    atomicOr(&bm[(size_t)it.y * d.WW + (it.x >> 5)], 1u << (it.x & 31));
                    it.next();
                }
            }
        }
        __syncwarp();
        lfdgeom::Edge e4[4];
        int ymin = 0x7fffffff, ymax = -0x7fffffff, nv = 0;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            e4[i] = sedge[wslot][i];
            if (e4[i].valid) { nv++; ymin = min(ymin, e4[i].y0); ymax = max(ymax, e4[i].y1); }
        }
        if (nv >= 2) {
            ymin = max(ymin, 0);
            ymax = min(ymax, d.H);
            for (int y = ymin + lane; y < ymax; y += 32) {
                int xs[4];
                int ns = lfdgeom::row_spans(e4, 4, y, d.W, xs);
                for (int s = 0; s < ns; s++) {
                    int x1 = xs[2 * s], x2 = xs[2 * s + 1];
                    for (int w = x1 >> 5; w <= (x2 >> 5); w++) {
                        int blo = max(x1 - (w << 5), 0), bhi = min(x2 - (w << 5), 31);
                        atomicOr(&bm[(size_t)y * d.WW + w], bit_range(blo, bhi));
                    }
                }
            }
        }
    }
}
