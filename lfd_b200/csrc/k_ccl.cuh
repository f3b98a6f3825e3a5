// k_ccl.cuh - run-based union-find connected components on bit masks.
//
// Replaces cv2.findContours(canny, RETR_LIST, CHAIN_APPROX_NONE)
// (/root/reference/lfd/detecttrails/processfield.py:241-246) by its structural equivalent
// (SURVEY.md 9.5, pinned in tests/test_oracle_cv.py::test_contour_sets_rects_box_img):
//   * one "outer" contour per 8-connected component of the edge map  -> kind 0 (fg)
//   * one "hole" contour per 4-connected background component that does not reach the frame border;
//     its points are the edge pixels 4-adjacent to the hole                                  -> kind 1 (bg)
// and doubles as Canny's hysteresis: the fg pass labels the NMS *candidates*; a component is an edge
// component iff it contains a strong pixel.
//
// Unit of work is a run (maximal horizontal span of set bits in one mask row), not a pixel: a
// 2048x1489 frame has ~10^5 runs against 3*10^6 pixels.  Runs get raster-order ids
// (row base + rank in row), so the root of a component (minimum id) is its raster-first run.
// Kernels are launched with one warp per mask row; lanes stride over the runs of the row.
#pragma once
#include "common.cuh"

struct CclBuf {
    Run* runs;        // [maxruns]
    int* parent;      // [maxruns]
    int* flag;        // [maxruns]  fg: bit0 = component holds a strong pixel; bg: bit0 = touches the border
    int* ymax;        // [maxruns]  valid at roots
    int* compidx;     // [maxruns]  valid at roots: contour index or -1
    int* rowbase;     // [H+1]
    unsigned* look;   // [1 + bands]  k_ccl_band's ticket, then one look-back word per band (zeroed by k_ctl_init)
};

// find with path halving (racy but safe: every store points a node at one of its ancestors)
__device__ __forceinline__ int uf_find(int* parent, int i)
{
    int cur = __ldcg(&parent[i]);
    if (cur != i) {
        int prev = i, next;
        while (cur > (next = __ldcg(&parent[cur]))) {
            parent[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

// read-only find: used where the caller then publishes parent[i] = root and later kernels rely on it
// (a concurrent path-halving store could otherwise replace the root by a mere ancestor)
__device__ __forceinline__ int uf_find_ro(const int* parent, int i)
{
    int p;
    while ((p = __ldcg(&parent[i])) != i) i = p;
    return i;
}

__device__ __forceinline__ void uf_union(int* parent, int a, int b)
{
    while (true) {
        a = uf_find(parent, a);
        b = uf_find(parent, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicMin(&parent[a], b);
        if (old == a) return;
        a = old;
    }
}

#define CCL_WARPS 8

// The runs of a row are sorted by xs and pairwise disjoint, so rows are searched by bisection over
// runs[rowbase[y] .. rowbase[y+1]) and the mask is never read again once the runs exist.

// index of the run of row y that contains pixel p (which must be set)
__device__ __forceinline__ int run_at(const CclBuf& b, int y, int p)
{
    int a = b.rowbase[y], e = b.rowbase[y + 1] - 1;          // last run with xs <= p
    while (a < e) {
        int mid = (a + e + 1) >> 1;
        if ((int)b.runs[mid].xs <= p) a = mid; else e = mid - 1;
    }
    return a;
}

// Linking two adjacent rows.  The overlap graph between the sorted run lists of rows y-1 and y is a
// staircase: every edge (r below, u above) is either "u is the first run above that r touches" or
// "r is the first run below that u touches".  So each run does exactly two lookups - first neighbour in
// the row above, first neighbour in the row below - instead of walking all of its neighbours; a
// frame-wide background run then costs the same as a one-pixel run.
__device__ __forceinline__ int first_touching(const CclBuf& b, int yy, Run r, int kind)
{
    const int c = kind ? 0 : 1;
    const int lo = (int)r.xs - c, hi = (int)r.xe + c;
    const int e1 = b.rowbase[yy + 1];
    int a = b.rowbase[yy], e = e1;                             // first run of row yy that ends at or after lo
    while (a < e) {
        int mid = (a + e) >> 1;
        if ((int)b.runs[mid].xe < lo) a = mid + 1; else e = mid;
    }
    return (a < e1 && (int)b.runs[a].xs <= hi) ? a : -1;
}

// link rows y-1 and y: work items [0, n_below) are runs of row y (look up), [n_below, n_below+n_above)
// are runs of row y-1 (look down)
__device__ __forceinline__ void link_rows(const CclBuf& b, int y, int kind, int first, int stride)
{
    int a0 = b.rowbase[y - 1], a1 = b.rowbase[y], b1 = b.rowbase[y + 1];
    int nb = b1 - a1, na = a1 - a0;
    for (int i = first; i < nb + na; i += stride) {
        bool below = i < nb;
        int id = below ? a1 + i : a0 + (i - nb);
        int j = first_touching(b, below ? y - 1 : y, b.runs[id], kind);
        if (j >= 0) uf_union(b.parent, id, j);
    }
}

#define CCL_BAND 32
#ifndef CCL_BAND_CTAS
#define CCL_BAND_CTAS 16          // CTAs per frame of k_ccl_band in launches of >= 16 frames
#endif

// ---- shared-memory union-find (band-local): same algorithm as uf_find / uf_union on a __shared__ array
__device__ __forceinline__ int suf_find(volatile int* p, int i)
{
    int cur = p[i];
    if (cur != i) {
        int prev = i, next;
        while (cur > (next = p[cur])) {
            p[prev] = next;
            prev = cur;
            cur = next;
        }
    }
    return cur;
}

__device__ __forceinline__ void suf_union(int* p, int a, int b)
{
    while (true) {
        a = suf_find(p, a);
        b = suf_find(p, b);
        if (a == b) return;
        if (a < b) { int t = a; a = b; b = t; }
        int old = atomicMin(&p[a], b);
        if (old == a) return;
        a = old;
    }
}

#define CCL_BAND_CAP 1536          // runs of one band kept in shared memory (12 B each = 18 KB)

// dynamic shared memory of k_ccl_band: CCL_BAND rows of mask words, then the band's parents and runs
// (+ its CCL_BAND + 1 band-local row bases and the run rank, within its row, of the first run start of every mask word, u16)
__host__ __device__ inline size_t ccl_band_smem(int WW)
{
    return (size_t)CCL_BAND * WW * 4 + (size_t)CCL_BAND_CAP * 12 + (size_t)(CCL_BAND + 2) * 4 + (size_t)CCL_BAND * WW * 2;
}

// Look-back words of k_ccl_band, CclBuf::look[1 + band]: 0 = nothing published yet, else a state in the top two bits
// over a run count: the band's own count (aggregate) or the count of bands 0 .. band (inclusive prefix).
#define CCL_LB_AGG (1u << 30)
#define CCL_LB_INC (2u << 30)
#define CCL_LB_VAL ((1u << 30) - 1u)
#define CCL_LB_SPIN (1 << 20)      // polls of one predecessor before the frame is given up (never reached when every claimed band publishes)

// exclusive prefix of `band` from its predecessors' look-back words (one thread); *stalled is set when a predecessor
// published nothing within CCL_LB_SPIN polls
__device__ __forceinline__ int ccl_lookback(const unsigned* look, int band, bool* stalled)
{
    int excl = 0;
    for (int j = band - 1; j >= 0; j--) {
        unsigned v;
        int spins = 0;
        while (((v = ((const volatile unsigned*)look)[1 + j]) >> 30) == 0u) {
            if (++spins > CCL_LB_SPIN) { *stalled = true; return excl; }
            __nanosleep(64);
        }
        excl += (int)(v & CCL_LB_VAL);
        if ((v & ~CCL_LB_VAL) == CCL_LB_INC) break;
    }
    return excl;
}

// The run-based labelling of one mask, one CCL_BAND-row band at a time: count the band's runs, materialise them, link
// all of its row pairs at once with a union-find that lives in shared memory, and publish band-local roots.
//   * The band's mask rows are staged in shared memory (complemented for kind 1), so counting, run ends and neighbour
//     lookups never go back to global memory.
//   * Run ids are raster-ordered: a band's runs are [base, base + nb), where base = runs of the bands above.  Everything
//     up to the publish works on band-local indices; base comes from a decoupled look-back over the bands' counts.
//   * Forward progress: bands are claimed in order from the frame's ticket (look[0]), so every band a CTA waits on is
//     held by a resident CTA, and every claimed band publishes its count before it waits on anything.  A CTA that
//     sees the frame inactive returns before its first claim; once it has claimed, it publishes whatever ctl says.
//   * The band that completes the frame writes rowbase[H] and nruns; a frame with more than maxruns runs is dropped
//     (LFD_FRAME_OVERFLOW, both passes' active flags cleared) and no band stores a run past maxruns.
//   * Bands with more runs than CCL_BAND_CAP use the global parent array with global ids, so they take their base
//     before the fill.
__global__ void __launch_bounds__(256)
k_ccl_band(const u32* __restrict__ mask, CclBuf* __restrict__ bufs, FrameCtl* __restrict__ ctl,
           int pass, Dims d, int kind, int maxruns, unsigned long long* __restrict__ counters)
{
    const int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    const u32* m = mask + (size_t)f * d.NW;
    CclBuf b = bufs[f];
    extern __shared__ u32 band_sm[];
    __shared__ int s_band, s_base;
    __shared__ bool s_stalled;
    const int WW = d.WW, nbands = (d.H + CCL_BAND - 1) / CCL_BAND;
    const int warp = threadIdx.x >> 5, lane = lane_id();
    u32* sw = band_sm;                                        // [CCL_BAND][WW]
    int* sp = (int*)(band_sm + CCL_BAND * WW);                // [CCL_BAND_CAP]
    Run* srun = (Run*)(sp + CCL_BAND_CAP);                    // [CCL_BAND_CAP]
    int* srb = (int*)(srun + CCL_BAND_CAP);                   // [CCL_BAND + 1] band-local row bases of rows y0 .. y1
    u16* swp = (u16*)(srb + CCL_BAND + 2);                    // [CCL_BAND][WW] run rank in its row of the word's first start
    // A CTA claims bands until the frame has none left: one band per CTA when a few frames are in the launch (shortest
    // latency), CCL_BAND_CTAS bands-looping CTAs per frame in big batches, where the per-CTA prologue (11 % of the
    // kernel's instructions with one band per CTA) is what counts (DESIGN.md section 7).
    for (;;) {
        __syncthreads();                                      // the previous band's shared state is consumed
        if (threadIdx.x == 0) { s_band = (int)atomicAdd(&b.look[0], 1u); s_stalled = false; }
        __syncthreads();
        const int band = s_band;
        if (band >= nbands) break;
        const int y0 = band * CCL_BAND, y1 = min(y0 + CCL_BAND, d.H), nr = y1 - y0;
        {
            // stage the band's mask rows (contiguous in global memory): four independent loads per thread and iteration
            const int tot = nr * WW;
            const u32* src = m + (size_t)y0 * WW;
            for (int i0 = threadIdx.x; i0 < tot; i0 += 4 * blockDim.x) {
                u32 v[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int i = i0 + k * blockDim.x;
                    v[k] = i < tot ? src[i] : 0u;
                }
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int i = i0 + k * blockDim.x;
                    if (i < tot) sw[i] = kind ? ~v[k] : v[k];
                }
            }
            __syncthreads();
            if (kind && (d.W & 31))                           // complemented rows: clear the bits past the frame edge
                for (int r = threadIdx.x; r < nr; r += blockDim.x) sw[r * WW + WW - 1] &= tail_mask(WW - 1, d.W);
        }
        __syncthreads();
        // count: one warp per row, 32 words at a time: run starts per word, warp scan -> rank of the word's first start
        for (int r = warp; r < nr; r += CCL_WARPS) {
            const u32* row = sw + r * WW;
            int base = 0;
            for (int w0 = 0; w0 < WW; w0 += 32) {
                const int w = w0 + lane;
                const u32 cur = w < WW ? row[w] : 0u, prev = (w && w <= WW) ? row[w - 1] : 0u;
                const u32 starts = cur & ~((cur << 1) | (prev >> 31));
                const int c = __popc(starts);
                int inc = c;
                if (__any_sync(FULLMASK, c != 0)) {
                    for (int o = 1; o < 32; o <<= 1) {
                        int v = __shfl_up_sync(FULLMASK, inc, o);
                        if (lane >= o) inc += v;
                    }
                }
                if (w < WW) swp[r * WW + w] = (u16)(base + inc - c);
                base += __shfl_sync(FULLMASK, inc, 31);
            }
            if (lane == 0) srb[r + 1] = base;
        }
        __syncthreads();
        if (warp == 0) {                                      // row counts -> band-local row bases (nr <= 32)
            const int c = lane < nr ? srb[lane + 1] : 0;
            int inc = c;
            for (int o = 1; o < 32; o <<= 1) {
                int v = __shfl_up_sync(FULLMASK, inc, o);
                if (lane >= o) inc += v;
            }
            if (lane < nr) srb[lane + 1] = inc;
            if (lane == 0) srb[0] = 0;
        }
        __syncthreads();
        const int nb = srb[nr];
        const bool insm = nb <= CCL_BAND_CAP;
        if (threadIdx.x == 0) {
            // publish the count before waiting on anything; band 0's count is already its inclusive prefix
            atomicExch(&b.look[1 + band], (band == 0 ? CCL_LB_INC : CCL_LB_AGG) | (unsigned)nb);
            if (!insm || band == 0) {
                bool st = false;
                const int ex = band ? ccl_lookback(b.look, band, &st) : 0;
                if (band) atomicExch(&b.look[1 + band], CCL_LB_INC | (unsigned)(ex + nb));
                s_base = ex; s_stalled = st;
            }
        }
        __syncthreads();
        // a dense band needs its global ids up front; a frame over maxruns stores no run past maxruns
        const bool fits_early = !insm && s_base + nb <= maxruns;
        // fill: one warp per row, rows strided over the 8 warps; ids are band-local
        if (insm || fits_early) {
            const int gb = insm ? 0 : s_base;
            for (int r = warp; r < nr; r += CCL_WARPS) {
                const int rb = srb[r];
                if (srb[r + 1] == rb) continue;                   // no run in this row (most rows of a sparse edge map)
                const u32* row = sw + r * WW;
                const int y = y0 + r;
                // words that are not all-ones, one ballot per 32-word chunk (W <= 4096 -> at most 4 chunks): a run
                // that leaves its word ends in the next such word, found with a bit scan instead of a serial walk
                // (the background of a sparse frame is one frame-wide run per row)
                u32 nf[4];
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    int w = c * 32 + lane;
                    nf[c] = __ballot_sync(FULLMASK, w >= WW || row[w] != 0xffffffffu);
                }
                for (int w = lane; w < WW; w += 32) {
                    u32 cur = row[w], prev = w ? row[w - 1] : 0u;
                    u32 starts = cur & ~((cur << 1) | (prev >> 31));
                    if (!starts) continue;
                    int id = rb + swp[r * WW + w];
                    while (starts) {
                        int s = __ffs(starts) - 1;
                        starts &= starts - 1;
                        u32 above = ~(cur >> s);
                        int t = above ? (__ffs(above) - 1) : 32;
                        int xe;
                        if (s + t < 32) {
                            xe = (w << 5) + s + t - 1;
                        } else {
                            int w2 = WW;                                   // first not-full word after w
                            const int c0 = w >> 5, pos = w & 31;
#pragma unroll
                            for (int c = 0; c < 4; c++) {
                                if (c < c0 || w2 < WW) continue;
                                u32 mbits = nf[c];
                                if (c == c0) mbits &= (pos == 31) ? 0u : (0xffffffffu << (pos + 1));
                                if (mbits) w2 = c * 32 + __ffs(mbits) - 1;
                            }
                            if (w2 >= WW) xe = (WW << 5) - 1;
                            else xe = (w2 << 5) + __ffs(~row[w2]) - 2;
                        }
                        Run run; run.xs = (u16)((w << 5) + s); run.xe = (u16)xe; run.y = (u16)y; run.pad = 0;
                        if (insm) { srun[id] = run; sp[id] = id; }
                        else {
                            b.runs[gb + id] = run;
                            b.flag[gb + id] = 0;
                            b.ymax[gb + id] = y;
                            b.compidx[gb + id] = -1;
                            b.parent[gb + id] = gb + id;
                        }
                        id++;
                    }
                }
            }
            __syncthreads();
            // link every run with the first run it touches in the row above and in the row below (staircase argument)
            const int c = kind ? 0 : 1;
            for (int i = threadIdx.x; i < nb; i += blockDim.x) {
                Run r = insm ? srun[i] : b.runs[gb + i];
                int lo = max((int)r.xs - c, 0), hi = min((int)r.xe + c, d.W - 1);
#pragma unroll
                for (int dy = -1; dy <= 1; dy += 2) {
                    int yy = (int)r.y + dy;
                    if (yy < y0 || yy >= y1) continue;
                    const u32* row = sw + (yy - y0) * WW;
                    int j = -1;
                    for (int w = lo >> 5; w <= (hi >> 5); w++) {
                        int blo = max(lo - (w << 5), 0), bhi = min(hi - (w << 5), 31);
                        u32 bits = row[w] & bit_range(blo, bhi);
                        if (bits) {
                            // band-local index of the run of row yy that contains pixel p
                            int bit = __ffs(bits) - 1;
                            u32 cur = row[w], prev = w ? row[w - 1] : 0u;
                            u32 starts = cur & ~((cur << 1) | (prev >> 31));
                            u32 upto = (bit == 31) ? 0xffffffffu : ((2u << bit) - 1u);
                            j = srb[yy - y0] + swp[(yy - y0) * WW + w] + __popc(starts & upto) - 1;
                            break;
                        }
                    }
                    if (j >= 0) { if (insm) suf_union(sp, i, j); else uf_union(b.parent, gb + i, gb + j); }
                }
            }
        }
        if (insm && band) {
            // the band's own work is done: now take the base (the predecessors have had all that time to publish)
            __syncthreads();
            if (threadIdx.x == 0) {
                bool st = false;
                const int ex = ccl_lookback(b.look, band, &st);
                atomicExch(&b.look[1 + band], CCL_LB_INC | (unsigned)(ex + nb));
                s_base = ex; s_stalled = st;
            }
        }
        __syncthreads();
        const int base = s_base;
        const bool fits = base + nb <= maxruns;
        if (insm && fits) {
            volatile int* vp = sp;
            for (int i = threadIdx.x; i < nb; i += blockDim.x) {
                int r = i, pr;
                while ((pr = vp[r]) != r) r = pr;
                const Run run = srun[i];
                b.runs[base + i] = run;
                b.flag[base + i] = 0;
                b.ymax[base + i] = run.y;
                b.compidx[base + i] = -1;
                b.parent[base + i] = base + r;
            }
        } else if (fits) {
            for (int i = threadIdx.x; i < nb; i += blockDim.x) b.parent[base + i] = uf_find_ro(b.parent, base + i);
        }
        if (threadIdx.x < nr) b.rowbase[y0 + threadIdx.x] = base + srb[threadIdx.x];
        if (threadIdx.x == 0) {
            const bool stalled = s_stalled;
            if (stalled) atomicAdd(&counters[14], 1ull);
            if (band == nbands - 1 || stalled) {
                int total = base + nb;
                if (band == nbands - 1) b.rowbase[d.H] = total;
                if (total > maxruns || stalled) {
                    // drop the frame (a stalled look-back leaves its run ids unknown): later kernels skip it
                    atomicOr(&ctl[f].status, LFD_FRAME_OVERFLOW);
                    ctl[f].active[0] = ctl[f].active[1] = 0;
                    total = 0;
                }
                if (band == nbands - 1) ctl[f].nruns[kind] = total;
            }
        }
    }
}

// 4b. stitch the bands: rows y = k * CCL_BAND against row y-1; one warp per seam
__global__ void __launch_bounds__(CCL_WARPS * 32)
k_ccl_merge(CclBuf* __restrict__ bufs, const FrameCtl* __restrict__ ctl, int pass, Dims d, int kind)
{
    int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    int y = (blockIdx.x * CCL_WARPS + (threadIdx.x >> 5) + 1) * CCL_BAND;
    if (y >= d.H) return;
    CclBuf b = bufs[f];
    if (ctl[f].nruns[kind] == 0) return;
    link_rows(b, y, kind, lane_id(), 32);
}

// Contour bookkeeping, one entry per selected component.
struct CompBuf {
    int* root;        // [2*maxcomp]  fg entries first, then bg
    int* y0;          // first row of the point set
    int* h;           // rows
    int* slot;        // offset into rowmin/rowmax
    int* hulloff;     // offset into the hull scratch
    int* rowmin;      // [slotcap]
    int* rowmax;      // [slotcap]
    int slotcap, hullcap, maxcomp;
};

// ---- steps 5-8: one thread per run ---------------------------------------------------------------------
// A frame has ~10-40 runs per row, so a warp-per-row grid leaves most lanes idle and launches ~1500 warps per
// frame that each wait on the same chain of dependent loads.  Runs are stored contiguously per frame
// (id = raster order), so these kernels simply stride over [0, nruns): full warps, 3x fewer of them.
#define CCL_FLAT_CTAS 48          // CTAs of 256 threads per frame (grid-stride over the frame's runs)

__global__ void __launch_bounds__(256)
k_ccl_stats_flat(const u32* __restrict__ strong, CclBuf* __restrict__ bufs, const FrameCtl* __restrict__ ctl,
                 int pass, Dims d, int kind)
{
    int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    const int nruns = ctl[f].nruns[kind];
    CclBuf b = bufs[f];
    const u32* sm = strong ? strong + (size_t)f * d.NW : nullptr;
    for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < nruns; id += gridDim.x * blockDim.x) {
        Run r = b.runs[id];
        const int y = r.y;
        int root = uf_find_ro(b.parent, id);
        b.parent[id] = root;
        int fl = 0;
        if (kind == 0) {
            for (int w = r.xs >> 5; w <= (r.xe >> 5); w++) {
                int blo = max((int)r.xs - (w << 5), 0), bhi = min((int)r.xe - (w << 5), 31);
                if (sm[(size_t)y * d.WW + w] & bit_range(blo, bhi)) { fl = 1; break; }
            }
        } else {
            fl = (y == 0 || y == d.H - 1 || r.xs == 0 || r.xe == d.W - 1) ? 1 : 0;
        }
        if (kind == 0) {
            // edge pass: many small components, neighbouring run ids rarely share one - plain atomics
            if (fl) atomicOr(&b.flag[root], 1);
            if (root != id) atomicMax(&b.ymax[root], y);
        } else {
            // hole pass: most runs belong to the frame-wide background, so consecutive run ids share a root: one
            // atomic per (warp, component) instead of one per run - thousands of same-address atomics serialise in
            // L2 and the kernel then waits for them at its exit (measured 35 -> 21 us; the same aggregation costs the
            // edge pass 20 %, its match groups are singletons)
            const unsigned peers = __match_any_sync(__activemask(), root);
            const int ymx = __reduce_max_sync(peers, y);
            const unsigned anyfl = __reduce_or_sync(peers, (unsigned)fl);
            if ((int)(__ffs(peers) - 1) == lane_id()) {
                if (anyfl) atomicOr(&b.flag[root], 1);
                if (!(root == id && __popc(peers) == 1)) atomicMax(&b.ymax[root], ymx);   // ymax[root] starts at the root's own row
            }
        }
    }
}

// fg: edge mask (pre-zeroed by the caller) + contour allocation ; bg: contour allocation only (edges == nullptr)
__global__ void __launch_bounds__(256)
k_ccl_alloc_flat(CclBuf* __restrict__ bufs, u32* __restrict__ edges, CompBuf* __restrict__ comps, FrameCtl* __restrict__ ctl,
                 int pass, Dims d, int kind)
{
    int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    const int nruns = ctl[f].nruns[kind];
    CclBuf b = bufs[f];
    CompBuf cb = comps[f];
    u32* em = edges ? edges + (size_t)f * d.NW : nullptr;
    for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < nruns; id += gridDim.x * blockDim.x) {
        const int root = b.parent[id];
        const int fl = b.flag[root] & 1;
        const bool sel = kind == 0 ? fl : !fl;          // fg: holds a strong pixel ; bg: does not touch the border
        if (!sel) continue;
        Run r = b.runs[id];
        const int y = r.y;
        if (kind == 0) {
            for (int w = r.xs >> 5; w <= (r.xe >> 5); w++) {
                int blo = max((int)r.xs - (w << 5), 0), bhi = min((int)r.xe - (w << 5), 31);
                atomicOr(&em[(size_t)y * d.WW + w], bit_range(blo, bhi));
            }
        }
        if (root != id) continue;
        int ci = atomicAdd(&ctl[f].ncomp[kind], 1);
        int hh = b.ymax[id] - y + 1 + (kind ? 2 : 0);
        int slot = atomicAdd(&ctl[f].nslots[0], hh);
        int ho = atomicAdd(&ctl[f].nhull[0], 2 * hh + 2);
        if (ci >= cb.maxcomp || slot + hh > cb.slotcap || ho + 2 * hh + 2 > cb.hullcap) {
            atomicOr(&ctl[f].status, LFD_FRAME_OVERFLOW);
            continue;
        }
        int e = kind * cb.maxcomp + ci;
        cb.root[e] = id;
        cb.y0[e] = y - (kind ? 1 : 0);
        cb.h[e] = hh;
        cb.slot[e] = slot;
        cb.hulloff[e] = ho;
        for (int i = 0; i < hh; i++) { cb.rowmin[slot + i] = 0x7fffffff; cb.rowmax[slot + i] = -1; }
        b.compidx[id] = e;
    }
}

__global__ void __launch_bounds__(256)
k_ccl_extremes_flat(const u32* __restrict__ edges, CclBuf* __restrict__ bufs, CompBuf* __restrict__ comps,
                    const FrameCtl* __restrict__ ctl, int pass, Dims d, int kind)
{
    int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    const int nruns = ctl[f].nruns[kind];
    CclBuf b = bufs[f];
    CompBuf cb = comps[f];
    const u32* em = edges + (size_t)f * d.NW;
    for (int id = blockIdx.x * blockDim.x + threadIdx.x; id < nruns; id += gridDim.x * blockDim.x) {
        int e = b.compidx[b.parent[id]];
        if (e < 0) continue;
        Run r = b.runs[id];
        const int y = r.y;
        int s = cb.slot[e] + (y - cb.y0[e]);
        if (kind == 0) {
            atomicMin(&cb.rowmin[s], (int)r.xs);
            atomicMax(&cb.rowmax[s], (int)r.xe);
        } else {
            // hole run [xs, xe] on row y (never on the frame border): edge pixels 4-adjacent to it
            atomicMin(&cb.rowmin[s], (int)r.xs - 1);
            atomicMax(&cb.rowmax[s], (int)r.xe + 1);
            for (int dy = -1; dy <= 1; dy += 2) {
                int yy = y + dy;
                int first = -1, last = -1;
                for (int w = r.xs >> 5; w <= (r.xe >> 5); w++) {
                    int blo = max((int)r.xs - (w << 5), 0), bhi = min((int)r.xe - (w << 5), 31);
                    u32 bits = em[(size_t)yy * d.WW + w] & bit_range(blo, bhi);
                    if (bits) {
                        if (first < 0) first = (w << 5) + __ffs(bits) - 1;
                        last = (w << 5) + 31 - __clz(bits);
                    }
                }
                if (first >= 0) {
                    atomicMin(&cb.rowmin[s + dy], first);
                    atomicMax(&cb.rowmax[s + dy], last);
                }
            }
        }
    }
}

// labels tap: int32 per pixel = raster-first pixel index of the component (fg) / hole (bg)
__global__ void __launch_bounds__(CCL_WARPS * 32)
k_ccl_labels(CclBuf* __restrict__ bufs, int* __restrict__ labels, const FrameCtl* __restrict__ ctl, int pass,
             Dims d, int kind, int frame)
{
    int f = frame;
    int y = blockIdx.x * CCL_WARPS + (threadIdx.x >> 5);
    if (y >= d.H) return;
    CclBuf b = bufs[f];
    int* out = labels + (size_t)y * d.W;
    for (int x = lane_id(); x < d.W; x += 32) out[x] = -1;
    __syncwarp();
    if (ctl[f].nruns[kind] == 0) return;
    int r0 = b.rowbase[y], r1 = b.rowbase[y + 1];
    for (int id = r0 + lane_id(); id < r1; id += 32) {
        int root = b.parent[id];
        Run r = b.runs[id], rr = b.runs[root];
        int lab;
        if (kind == 0) lab = (b.flag[root] & 1) ? (int)rr.y * d.W + (int)rr.xs : -1;
        else lab = (b.flag[root] & 1) ? -2 : (int)rr.y * d.W + (int)rr.xs;
        for (int x = r.xs; x <= r.xe; x++) out[x] = lab;
    }
}
