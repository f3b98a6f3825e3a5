// k_morph.cuh - erode / dilate fused with the equalisation LUT: all-ones rectangles (k_morph_march, k_morph) and flat
// structuring elements of any shape up to 255 x 255 (k_morph_any, chord decomposition).
//
// Reference: cv2.erode(equ, erodeKernel) processfield.py:464 ; cv2.dilate(., dilateKernel) :354, :471
// (paths under /root/reference/lfd/detecttrails/).  cv2 semantics: anchor = (kw/2, kh/2), window rows
// y-ay .. y-ay+kh-1, out-of-frame samples ignored.
//
// equalizeHist's LUT is monotone non-decreasing, so min/max filters commute with it:
// dilate(erode(lut[gray])) == lut[dilate(erode(gray))].  The kernel therefore filters the raw `gray`
// plane in shared memory and applies the LUT once on the way out; the equalised plane itself is only
// materialised for the debug tap.
//
// Tile: 128 x 16 output pixels per 256-thread CTA, 4 pixels (one 32-bit word) per thread and row,
// byte-wise SIMD min/max (__vminu4/__vmaxu4) with funnel shifts for the horizontal window.
#pragma once
#include "common.cuh"
#include "chords.cuh"

#define MORPH_TW 128                // tile width in pixels
#define MORPH_TWW (MORPH_TW / 4)    // in 4-pixel words
#define MORPH_TH 16
#define MORPH_PADW 4                // halo words each side (16 px)
#define MORPH_PADH 16               // halo rows each side
#define MORPH_SW (MORPH_TWW + 2 * MORPH_PADW)
#define MORPH_SH (MORPH_TH + 2 * MORPH_PADH)

struct MorphCfg {
    int eh, ew;     // erode kernel (0 = none)
    int dh, dw;     // dilate kernel (>= 1)
};

// horizontal window op over bytes: out byte x = op over x+lo .. x+hi of row `s` (word array with PADW halo)
template <bool IS_MAX>
__device__ __forceinline__ u32 hwin(const u32* s, int w, int lo, int hi)
{
    u32 acc = IS_MAX ? 0u : 0xffffffffu;
    for (int o = lo; o <= hi; o++) {
        int wi = w + (o >> 2);          // arithmetic shift = floor
        int b = o & 3;
        u32 v = __funnelshift_r(s[wi], s[wi + 1], 8 * b);
        acc = IS_MAX ? __vmaxu4(acc, v) : __vminu4(acc, v);
    }
    return acc;
}

// gray -> [erode] -> dilate -> lut -> morph (uint8) + nz (bit mask of morph != 0) [+ eroded tap (lut applied)]
__global__ void __launch_bounds__(256)
k_morph(const u8* __restrict__ gray, const u8* __restrict__ lut, u8* __restrict__ morph,
        u32* __restrict__ nz, u8* __restrict__ eroded_tap, const FrameCtl* __restrict__ ctl, int pass,
        Dims d, MorphCfg mc)
{
    int f = blockIdx.z;
    if (!ctl[f].active[pass]) return;
    __shared__ u32 A[MORPH_SH][MORPH_SW + 1];
    __shared__ u32 Bf[MORPH_SH][MORPH_SW + 1];
    __shared__ u8 slut[256];
    const int tx0w = blockIdx.x * MORPH_TWW;      // tile origin in words
    const int ty0 = blockIdx.y * MORPH_TH;
    const int Ww = d.W >> 2;
    const u32* g = reinterpret_cast<const u32*>(gray + (size_t)f * d.N);
    slut[threadIdx.x] = lut[(size_t)f * 256 + threadIdx.x];

    const bool has_e = mc.eh > 0;
    // window extents (relative offsets, inclusive)
    const int e_t = has_e ? -(mc.eh / 2) : 0, e_b = has_e ? mc.eh - 1 - mc.eh / 2 : 0;
    const int e_l = has_e ? -(mc.ew / 2) : 0, e_r = has_e ? mc.ew - 1 - mc.ew / 2 : 0;
    const int d_t = -(mc.dh / 2), d_b = mc.dh - 1 - mc.dh / 2;
    const int d_l = -(mc.dw / 2), d_r = mc.dw - 1 - mc.dw / 2;

    // 1. load rows [ty0 - PADH, ty0 + TH + PADH) x words [tx0w - PADW, tx0w + TWW + PADW); outside the
    //    frame -> identity of the FIRST filter
    const u32 ident_first = has_e ? 0xffffffffu : 0u;
    for (int i = threadIdx.x; i < MORPH_SH * MORPH_SW; i += blockDim.x) {
        int r = i / MORPH_SW, c = i - r * MORPH_SW;
        int y = ty0 - MORPH_PADH + r, w = tx0w - MORPH_PADW + c;
        u32 v = ident_first;
        if (y >= 0 && y < d.H && w >= 0 && w < Ww) v = g[(size_t)y * Ww + w];
        A[r][c] = v;
    }
    __syncthreads();

    if (has_e) {
        // 2a. vertical min: rows needed by the dilate = [ty0 + d_t, ty0 + TH - 1 + d_b]
        int r_lo = MORPH_PADH + d_t, r_hi = MORPH_PADH + MORPH_TH - 1 + d_b;
        int nrows = r_hi - r_lo + 1;
        for (int i = threadIdx.x; i < nrows * MORPH_SW; i += blockDim.x) {
            int r = r_lo + i / MORPH_SW, c = i % MORPH_SW;
            u32 acc = 0xffffffffu;
            for (int o = e_t; o <= e_b; o++) acc = __vminu4(acc, A[r + o][c]);
            Bf[r][c] = acc;
        }
        __syncthreads();
        // 2b. horizontal min into A; positions outside the frame become 0 (ignored by the dilate)
        // columns the dilate will read (host validates that the combined halo fits the padding)
        int c_lo = MORPH_PADW + (d_l >> 2), c_hi = MORPH_PADW + MORPH_TWW - 1 + ((d_r + 3) >> 2);
        for (int i = threadIdx.x; i < nrows * (c_hi - c_lo + 1); i += blockDim.x) {
            int r = r_lo + i / (c_hi - c_lo + 1), c = c_lo + i % (c_hi - c_lo + 1);
            int y = ty0 - MORPH_PADH + r, w = tx0w - MORPH_PADW + c;
            u32 v = 0u;
            if (y >= 0 && y < d.H && w >= 0 && w < Ww) v = hwin<false>(&Bf[r][0], c, e_l, e_r);
            A[r][c] = v;
        }
        __syncthreads();
        if (eroded_tap) {
            for (int i = threadIdx.x; i < MORPH_TH * MORPH_TWW; i += blockDim.x) {
                int r = i / MORPH_TWW, c = i % MORPH_TWW;
                int y = ty0 + r, w = tx0w + c;
                if (y < d.H && w < Ww) {
                    u32 v = A[MORPH_PADH + r][MORPH_PADW + c];
                    u32 o = slut[v & 255] | (slut[(v >> 8) & 255] << 8) | (slut[(v >> 16) & 255] << 16) | (slut[v >> 24] << 24);
                    reinterpret_cast<u32*>(eroded_tap + (size_t)f * d.N)[(size_t)y * Ww + w] = o;
                }
            }
        }
    }

    // 3a. vertical max over the output rows (all columns incl. halo)
    for (int i = threadIdx.x; i < MORPH_TH * MORPH_SW; i += blockDim.x) {
        int r = MORPH_PADH + i / MORPH_SW, c = i % MORPH_SW;
        u32 acc = 0u;
        for (int o = d_t; o <= d_b; o++) acc = __vmaxu4(acc, A[r + o][c]);
        Bf[r][c] = acc;
    }
    __syncthreads();
    // 3b. horizontal max + LUT + outputs.  One warp covers one tile row (32 words = 128 px).
    for (int i = threadIdx.x; i < MORPH_TH * MORPH_TWW; i += blockDim.x) {
        int r = i / MORPH_TWW, c = i % MORPH_TWW;   // c == lane
        int y = ty0 + r, w = tx0w + c;
        bool in = (y < d.H && w < Ww);
        u32 o = 0u;
        if (in) {
            u32 v = hwin<true>(&Bf[MORPH_PADH + r][0], MORPH_PADW + c, d_l, d_r);
            o = slut[v & 255] | (slut[(v >> 8) & 255] << 8) | (slut[(v >> 16) & 255] << 16) | (slut[v >> 24] << 24);
            reinterpret_cast<u32*>(morph + (size_t)f * d.N)[(size_t)y * Ww + w] = o;
        }
        // non-zero bit mask: 8 lanes x 4 px = one 32-bit mask word
        u32 b0 = __ballot_sync(FULLMASK, (o & 0x000000ffu) != 0);
        u32 b1 = __ballot_sync(FULLMASK, (o & 0x0000ff00u) != 0);
        u32 b2 = __ballot_sync(FULLMASK, (o & 0x00ff0000u) != 0);
        u32 b3 = __ballot_sync(FULLMASK, (o & 0xff000000u) != 0);
        int lane = lane_id();
        if (lane < 4) {
            u32 word = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                int l = lane * 8 + k;
                word |= ((b0 >> l) & 1u) << (4 * k);
                word |= ((b1 >> l) & 1u) << (4 * k + 1);
                word |= ((b2 >> l) & 1u) << (4 * k + 2);
                word |= ((b3 >> l) & 1u) << (4 * k + 3);
            }
            int mw = (tx0w * 4) / 32 + lane;      // mask word index in the row
            if (y < d.H && mw < d.WW) nz[(size_t)f * d.NW + (size_t)y * d.WW + mw] = word;
        }
    }
}

// ================================================================================================
// Register-marching variant (the production path for the kernel shapes instantiated below).
//
// A warp owns a strip of 64 4-pixel words (256 px: 224 useful + 16 px of halo per side) and marches
// down MARCH_R output rows.  Each lane holds 8 consecutive pixels of the current row as four u16x2
// registers, so every min/max is a native VIMNMX3.U16x2 (byte-wise __vmaxu4 is emulated with 7 ALU
// ops on sm_100a, the 16x2 three-input form is one).  Horizontal windows take neighbour pixels with
// warp shuffles, vertical windows are register rings indexed at compile time (the row loop is
// unrolled by lcm(EH, DH)), so the image is read once from global memory and nothing is staged in
// shared memory except the 256-byte LUT.
// ================================================================================================
#ifndef MARCH_R
#define MARCH_R 64            // output rows per warp
#endif
#define MARCH_UW 56           // useful words per strip (7 mask words)
#define MARCH_HW 4            // halo words per side (lanes 0,1 and 30,31)
#ifndef MARCH_WPC
#define MARCH_WPC 1           // warps (= strip units) per CTA
#endif

template <bool IS_MAX> __device__ __forceinline__ u32 mm2(u32 a, u32 b) { return IS_MAX ? __vmaxu2(a, b) : __vminu2(a, b); }
template <bool IS_MAX> __device__ __forceinline__ u32 mm3(u32 a, u32 b, u32 c)
{
    return IS_MAX ? __vimax3_u16x2(a, b, c) : __vimin3_u16x2(a, b, c);
}

// out pixel x = op over pixels x+LO .. x+HI of the row; p[i] = (px 2i, px 2i+1) of the lane's 8 pixels
template <bool IS_MAX, int LO, int HI>
__device__ __forceinline__ void hwin16(const u32 (&p)[4], u32 (&out)[4])
{
    constexpr int KL = (-LO + 1) / 2, KR = (HI + 1) / 2, NE = KL + 4 + KR;
    static_assert(KL <= 4 && KR <= 4, "horizontal reach exceeds one lane (8 px)");
    if (LO == 0 && HI == 0) {
#pragma unroll
        for (int i = 0; i < 4; i++) out[i] = p[i];
        return;
    }
    u32 E[NE];
#pragma unroll
    for (int i = 0; i < 4; i++) E[KL + i] = p[i];
#pragma unroll
    for (int j = 0; j < KL; j++) E[KL - 1 - j] = __shfl_up_sync(FULLMASK, p[3 - j], 1);
#pragma unroll
    for (int j = 0; j < KR; j++) E[KL + 4 + j] = __shfl_down_sync(FULLMASK, p[j], 1);
    u32 S[NE];      // S[j] = (px 2j+1, px 2j+2) of the extended row
#pragma unroll
    for (int j = 0; j + 1 < NE; j++) S[j] = __byte_perm(E[j], E[j + 1], 0x5432);
    S[NE - 1] = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        // term for offset o: even -> E[KL + i + o/2], odd -> S[KL + i + (o-1)/2]
        u32 acc = 0;
        bool first = true;
        u32 pend = 0;
        bool have_pend = false;
#pragma unroll
        for (int o = LO; o <= HI; o++) {
            int fl = (o >= 0) ? (o >> 1) : -((-o + 1) >> 1);        // floor(o / 2)
            u32 t = (o & 1) ? S[KL + i + fl] : E[KL + i + fl];
            if (first) { acc = t; first = false; }
            else if (!have_pend) { pend = t; have_pend = true; }
            else { acc = mm3<IS_MAX>(acc, pend, t); have_pend = false; }
        }
        if (have_pend) acc = mm2<IS_MAX>(acc, pend);
        out[i] = acc;
    }
}

template <bool IS_MAX, int K>
__device__ __forceinline__ u32 vreduce16(const u32 (&r)[K][4], int c)
{
    u32 acc = r[0][c];
    int k = 1;
#pragma unroll
    for (; k + 1 < K; k += 2) acc = mm3<IS_MAX>(acc, r[k][c], r[k + 1][c]);
    if (k < K) acc = mm2<IS_MAX>(acc, r[k][c]);
    return acc;
}

__host__ __device__ constexpr int morph_gcd(int a, int b) { return b == 0 ? a : morph_gcd(b, a % b); }

// four u16x2 pairs -> LUT -> two packed 4-pixel words
__device__ __forceinline__ void lut_pack(const u32 (&o)[4], const u8* slut, u32& w0, u32& w1)
{
    u32 r[4];
#pragma unroll
    for (int i = 0; i < 4; i++) r[i] = (u32)slut[o[i] & 0xffffu] | ((u32)slut[o[i] >> 16] << 16);
    w0 = __byte_perm(r[0], r[1], 0x6420);
    w1 = __byte_perm(r[2], r[3], 0x6420);
}

// bit k = byte k of w is non-zero
__device__ __forceinline__ u32 nzbits4(u32 w)
{
    u32 m = (((w & 0x7f7f7f7fu) + 0x7f7f7f7fu) | w) & 0x80808080u;
    return ((m >> 7) * 0x10204080u) >> 28;
}

#ifndef MARCH_MINB
#define MARCH_MINB 1          // __launch_bounds__ min CTAs per SM (register cap) of the marching morphology kernel
#endif
template <int EH, int EW, int DH, int DW>
__global__ void __launch_bounds__(MARCH_WPC * 32, MARCH_MINB)
k_morph_march(const u8* __restrict__ gray, const u8* __restrict__ lut, u8* __restrict__ morph, u32* __restrict__ nz,
              u8* __restrict__ eroded_tap, const FrameCtl* __restrict__ ctl, int pass, Dims d, int nstrips, int nunits)
{
    const int f = blockIdx.y;
    if (!ctl[f].active[pass]) return;
    __shared__ u8 slut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) slut[i] = lut[(size_t)f * 256 + i];
    __syncthreads();
    const int unit = blockIdx.x * MARCH_WPC + (threadIdx.x >> 5);
    if (unit >= nunits) return;
    const int chunk = unit / nstrips, s = unit - chunk * nstrips;
    constexpr bool HAS_E = EH > 0;
    constexpr int EHR = HAS_E ? EH : 1;
    constexpr int E_T = HAS_E ? -(EH / 2) : 0, E_B = HAS_E ? EH - 1 - EH / 2 : 0;
    constexpr int E_L = HAS_E ? -(EW / 2) : 0, E_R = HAS_E ? EW - 1 - EW / 2 : 0;
    constexpr int D_T = -(DH / 2), D_B = DH - 1 - DH / 2, D_L = -(DW / 2), D_R = DW - 1 - DW / 2;
    constexpr int U = EHR * DH / morph_gcd(EHR, DH);
    const int lane = lane_id();
    const int Ww = d.W >> 2;
    const int wx = s * MARCH_UW - MARCH_HW + 2 * lane;       // first of this lane's two words (even)
    const bool col_in = wx >= 0 && wx < Ww;
    const bool lane_out = lane >= 2 && lane < 30 && col_in;
    const int y0 = chunk * MARCH_R, y1 = min(y0 + MARCH_R, d.H);
    const int yfirst = y0 + D_T + E_T, ylast = y1 - 1 + D_B + E_B;
    const uint2* g = reinterpret_cast<const uint2*>(gray + (size_t)f * d.N);
    uint2* mo = reinterpret_cast<uint2*>(morph + (size_t)f * d.N);
    uint2* et = eroded_tap ? reinterpret_cast<uint2*>(eroded_tap + (size_t)f * d.N) : nullptr;
    const u32 lut0 = slut[0];
    // mask word of this lane's group: lanes 2..5 -> word 7s, 6..9 -> 7s+1, ...
    const int r = (lane - 2) & 31;
    const int mw = s * (MARCH_UW / 8) + (r >> 2);
    const int q8 = (r & 3) * 8;
    const int src1 = ((r ^ 1) + 2) & 31, src2 = ((r ^ 2) + 2) & 31;
    u32 eR[EHR][4], dR[DH][4];
#pragma unroll
    for (int k = 0; k < EHR; k++)
#pragma unroll
        for (int c = 0; c < 4; c++) eR[k][c] = 0;
#pragma unroll
    for (int k = 0; k < DH; k++)
#pragma unroll
        for (int c = 0; c < 4; c++) dR[k][c] = 0;

    // software pipeline: the U rows of the next block are requested before the current block is processed,
    // so the dependent min/max chain never waits on a global load (the kernel is latency-, not bandwidth-bound)
    // Pixels outside the frame are "ignored" by cv2: they are loaded as zeros (so that the all-zero test below sees
    // only frame pixels) and become the identity of the FIRST filter (255 for the erosion, 0 for the dilation) where a
    // row is actually filtered.  Row addresses are running element offsets (one 64-bit add per row instead of a
    // 64-bit multiply chain per access).
    //
    // All-zero rows are the common case on sky-subtracted frames (bright: everything but stars; dim: everything the
    // erosion removes): one warp vote per row skips the horizontal window, and the vertical reduction + LUT + mask
    // bits are skipped while every row of the dilation ring is zero (ezbits / dnz track the rings' all-zero rows).
    const long long rstep = Ww >> 1;                           // uint2 elements per image row
    long long ld_off = ((long long)yfirst * Ww + wx) >> 1;     // arithmetic shift: also right for rows above the frame
    uint2 nxt[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
        const int y = yfirst + u;
        nxt[u] = make_uint2(0u, 0u);
        if (y >= 0 && y < d.H && col_in) nxt[u] = __ldg(g + ld_off);
        ld_off += rstep;
    }
    long long st_off = ((long long)y0 * Ww + wx) >> 1;          // output rows are produced in order y0, y0+1, ...
    long long et_off = st_off;
    int nz_off = f * d.NW + y0 * d.WW + mw;
    u32 ezbits = (1u << EHR) - 1u;                             // erosion ring rows that are all-zero across the strip
    u32 dnz = 0;                                               // dilation ring rows that are NOT all-zero
    const bool lut0z = lut0 == 0u;
    const bool nz_lane = (r & 3) == 0 && lane >= 2 && lane < 30 && mw < d.WW;
    for (int yb = yfirst; yb <= ylast; yb += U) {
        uint2 cur[U];
#pragma unroll
        for (int u = 0; u < U; u++) cur[u] = nxt[u];
        if (yb + U <= ylast) {
#pragma unroll
            for (int u = 0; u < U; u++) {
                const int y = yb + U + u;
                nxt[u] = make_uint2(0u, 0u);
                if (y >= 0 && y < d.H && col_in) nxt[u] = __ldg(g + ld_off);
                ld_off += rstep;
            }
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int y = yb + u;
            uint2 v = cur[u];
            const bool yin = (unsigned)y < (unsigned)d.H;
            const bool in_zero = !__any_sync(FULLMASK, (v.x | v.y) != 0u);
            u32 e[4];
            bool e_zero;                                     // warp-uniform: the row entering the dilation is all-zero
            int ye = y;
            if (HAS_E) {
                ye = y - E_B;
                if (in_zero && yin) {                        // a frame row of zeros: every minimum that sees it is zero
                    if (!((ezbits >> (u % EHR)) & 1u)) {
#pragma unroll
                        for (int c = 0; c < 4; c++) eR[u % EHR][c] = 0;
                        ezbits |= 1u << (u % EHR);
                    }
                } else {
                    if (!(yin && col_in)) v = make_uint2(0xffffffffu, 0xffffffffu);
                    u32 p[4], hm[4];
                    p[0] = __byte_perm(v.x, 0, 0x4140); p[1] = __byte_perm(v.x, 0, 0x4342);
                    p[2] = __byte_perm(v.y, 0, 0x4140); p[3] = __byte_perm(v.y, 0, 0x4342);
                    hwin16<false, E_L, E_R>(p, hm);
#pragma unroll
                    for (int c = 0; c < 4; c++) eR[u % EHR][c] = hm[c];
                    ezbits &= ~(1u << (u % EHR));
                }
                if (ezbits != 0u) {                          // a zero row in the window: the minimum is zero
#pragma unroll
                    for (int c = 0; c < 4; c++) e[c] = 0u;
                    e_zero = true;
                } else {
                    const bool ein = col_in && ye >= 0 && ye < d.H;
#pragma unroll
                    for (int c = 0; c < 4; c++) e[c] = ein ? vreduce16<false, EHR>(eR, c) : 0u;
                    e_zero = !__any_sync(FULLMASK, (e[0] | e[1] | e[2] | e[3]) != 0u);
                }
                if (et && ye >= y0 && ye < y1) {
                    u32 w0, w1;
                    lut_pack(e, slut, w0, w1);
                    if (lane_out) et[et_off] = make_uint2(w0, w1);
                    et_off += rstep;
                }
            } else {
                e_zero = in_zero;
            }
            if (e_zero) {
                if ((dnz >> (u % DH)) & 1u) {
#pragma unroll
                    for (int c = 0; c < 4; c++) dR[u % DH][c] = 0;
                    dnz &= ~(1u << (u % DH));
                }
            } else {
                if (!HAS_E) {
                    e[0] = __byte_perm(v.x, 0, 0x4140); e[1] = __byte_perm(v.x, 0, 0x4342);
                    e[2] = __byte_perm(v.y, 0, 0x4140); e[3] = __byte_perm(v.y, 0, 0x4342);
                }
                u32 hd[4];
                hwin16<true, D_L, D_R>(e, hd);
#pragma unroll
                for (int c = 0; c < 4; c++) dR[u % DH][c] = hd[c];
                dnz |= 1u << (u % DH);
            }
            const int yo = ye - D_B;
            if (yo >= y0 && yo < y1) {                       // warp-uniform
                u32 w0 = 0, w1 = 0, bits = 0;
                if (dnz != 0u || !lut0z) {                   // (an all-zero window gives lut[0] == 0 everywhere)
                    u32 o[4];
#pragma unroll
                    for (int c = 0; c < 4; c++) o[c] = vreduce16<true, DH>(dR, c);
                    lut_pack(o, slut, w0, w1);
                    if (!lane_out) { w0 = 0; w1 = 0; }
                    if (__any_sync(FULLMASK, (w0 | w1) != 0u)) {
                        bits = (nzbits4(w0) | (nzbits4(w1) << 4)) << q8;
                        bits |= __shfl_sync(FULLMASK, bits, src1);
                        bits |= __shfl_sync(FULLMASK, bits, src2);
                    }
                }
                if (lane_out) mo[st_off] = make_uint2(w0, w1);
                st_off += rstep;
                if (nz_lane) nz[nz_off] = bits;
                nz_off += d.WW;
            }
        }
    }
}

// ================================================================================================
// Arbitrary flat structuring elements (cv2.getStructuringElement ellipses / crosses, rings, hand-made masks, all-ones
// rectangles past the tile halo), sides 1..CHORD_MAX_SIDE: the chord decomposition of chords.cuh, one launch per
// operation (erosion into a scratch plane, then dilation + LUT + mask bits).
//
// A CTA owns a strip of CHORD_SW output columns (one per thread) and a chunk of CHORD_R output rows.  It reads each
// input row the chunk needs once, with the element's horizontal reach on both sides, and builds that row's sparse-table
// levels P_0 .. P_{nlev-1} in shared memory.  Mask row i of the element folds its chords' result into output row
// y = r - (i - ay), held in a ring of kh partial rows; a row leaves the ring when mask row kh - 1 has contributed.
// Per output pixel that is 2 * #chords + 1 shared-memory loads per mask row plus nlev per input row, against |M| for
// the direct evaluation (DESIGN.md §3).  Out-of-frame samples are the identity (255 for min, 0 for max), so they are
// ignored as cv2 ignores them; an input row holding only the identity (all outside the frame, or a zero row of a
// dilation) contributes nothing and is skipped.
// ================================================================================================
#define CHORD_SW 256                   // strip width in pixels = threads per CTA
#define CHORD_R 64                     // output rows per chunk

struct ChordSet {
    const int* rowoff;                 // [kh + 1] first chord of each mask row (chords.cuh)
    const u32* code;                   // chord codes
    int kh, kw, ay, ax, nlev;          // nlev: sparse-table levels the chords read
};

__host__ __device__ inline int chord_lw(int kw) { return (CHORD_SW + kw - 1 + 3) & ~3; }

// dynamic smem: nlev level rows of chord_lw(kw) bytes, the kh-row ring, the LUT
__host__ __device__ inline size_t chord_smem(int kh, int kw, int nlev)
{
    return (size_t)nlev * chord_lw(kw) + (size_t)kh * CHORD_SW + 256;
}

template <bool IS_MAX> __device__ __forceinline__ u32 op8(u32 a, u32 b) { return IS_MAX ? max(a, b) : min(a, b); }

// IS_MAX = false: erosion of `src` into `dst` (raw values), eroded tap = lut[dst].
// IS_MAX = true: dilation of `src`, lut -> `dst` (the morphology plane) + nz; eroded_tap (runs without an erosion only)
// = lut[src], as the pass's eroded plane is then its input.
template <bool IS_MAX>
__global__ void __launch_bounds__(CHORD_SW)
k_morph_any(const u8* __restrict__ src, const u8* __restrict__ lut, u8* __restrict__ dst, u32* __restrict__ nz,
            u8* __restrict__ eroded_tap, const FrameCtl* __restrict__ ctl, int pass, Dims d, ChordSet cs)
{
    const int f = blockIdx.z;
    if (!ctl[f].active[pass]) return;
    extern __shared__ u32 chsm_[];
    const int LW = chord_lw(cs.kw), kh = cs.kh, ay = cs.ay;
    u8* lv = reinterpret_cast<u8*>(chsm_);
    u8* ring = lv + cs.nlev * LW;
    u8* slut = ring + kh * CHORD_SW;
    const int tx = threadIdx.x;
    slut[tx] = lut[(size_t)f * 256 + tx];
    const u32 ID = IS_MAX ? 0u : 255u;
    for (int i = 0; i < kh; i++) ring[i * CHORD_SW + tx] = (u8)ID;      // a thread's ring column is its own
    const int x0 = blockIdx.x * CHORD_SW, y0 = blockIdx.y * CHORD_R, y1 = min(y0 + CHORD_R, d.H);
    const int x = x0 + tx, xs = x0 - cs.ax;                              // xs: frame column of level column 0
    const bool xin = x < d.W;
    const u8* in = src + (size_t)f * d.N;
    u8* out = dst + (size_t)f * d.N;
    u8* et = eroded_tap ? eroded_tap + (size_t)f * d.N : nullptr;
    const int rlast = y1 - 1 + (kh - 1 - ay);
    for (int r = y0 - ay; r <= rlast; r++) {
        bool any = false;
        if (r >= 0 && r < d.H) {
            const u8* row = in + (size_t)r * d.W;
            for (int c = tx; c < LW; c += CHORD_SW) {
                const int xc = xs + c;
                const u32 v = (xc >= 0 && xc < d.W) ? row[xc] : ID;
                lv[c] = (u8)v;
                any |= v != ID;
            }
        }
        const bool busy = __syncthreads_or(any);
        if (IS_MAX && et && r >= y0 && r < y1 && xin) et[(size_t)r * d.W + x] = slut[lv[tx + cs.ax]];
        if (busy) {
            for (int k = 1; k < cs.nlev; k++) {
                const u8* p = lv + (k - 1) * LW;
                u8* q = lv + k * LW;
                const int s = 1 << (k - 1);
                for (int c = tx; c + 2 * s <= LW; c += CHORD_SW) q[c] = (u8)op8<IS_MAX>(p[c], p[c + s]);
                __syncthreads();
            }
            // mask rows i whose output row y = r - i + ay lies in the chunk; ring slot (y - y0) % kh
            const int ilo = max(0, r + ay - y1 + 1), ihi = min(kh - 1, r + ay - y0);
            int slot = (r + ay - ilo - y0) % kh;
            for (int i = ilo; i <= ihi; i++) {
                const int c0 = __ldg(cs.rowoff + i), c1 = __ldg(cs.rowoff + i + 1);
                if (c0 < c1) {
                    u32 acc = ID;
                    for (int c = c0; c < c1; c++) {
                        const u32 q = __ldg(cs.code + c);
                        const u8* P = lv + (q >> 16) * LW + tx;
                        acc = op8<IS_MAX>(acc, op8<IS_MAX>(P[q & 255u], P[(q >> 8) & 255u]));
                    }
                    u8* rv = ring + slot * CHORD_SW + tx;
                    *rv = (u8)op8<IS_MAX>(*rv, acc);
                }
                slot = slot == 0 ? kh - 1 : slot - 1;
            }
        }
        const int y = r - (kh - 1 - ay);                 // complete: mask row kh - 1 has contributed
        if (y >= y0) {
            u8* rv = ring + ((y - y0) % kh) * CHORD_SW + tx;
            const u32 v = *rv;
            *rv = (u8)ID;
            if (IS_MAX) {
                const u32 o = slut[v];
                if (xin) out[(size_t)y * d.W + x] = (u8)o;
                const u32 b = __ballot_sync(FULLMASK, xin && o != 0u);
                const int mw = (x0 >> 5) + (tx >> 5);
                if (lane_id() == 0 && mw < d.WW) nz[(size_t)f * d.NW + (size_t)y * d.WW + mw] = b;
            } else if (xin) {
                out[(size_t)y * d.W + x] = (u8)v;
                if (et) et[(size_t)y * d.W + x] = slut[v];
            }
        }
        __syncthreads();                                 // the next row overwrites the levels
    }
}
