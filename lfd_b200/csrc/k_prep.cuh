// k_prep.cuh - star mask rasterisation, fused blot+flip+clip+convertScaleAbs+histogram, equalisation LUT.
//
// Reference behaviour (paths under /root/reference/lfd/detecttrails/):
//   removestars.py:231      img[x-dxy:x+dxy, y-dxy:y+dxy].fill(0.0)  -> k_star_mask (+ applied in k_prep)
//   detecttrails.py:124     cv2.flip(img, 0)                          -> source row H-1-y in k_prep
//   processfield.py:342     img[img < 0] = 0                          -> bright clip
//   processfield.py:453-454 img[img < minFlux] = 0; img[img > 0] += addFlux
//   processfield.py:346,456 cv2.convertScaleAbs                       -> csa()
//   processfield.py:347,457 cv2.equalizeHist                          -> histogram here, LUT in k_lut
#pragma once
#include "common.cuh"

// rects: (r0, r1, c0, c1) half-open on the UN-flipped image; rect_off[n+1] indexes them per frame.
// mask: [n][H][WW] bit per pixel in the FLIPPED orientation (row H-1-r).
// One warp per rectangle over the flat list of ALL frames (the frame is found by bisection of rect_off),
// so the grid is proportional to the number of stars, not to frames x the densest frame.
__global__ void __launch_bounds__(128)
k_star_mask(const int4* __restrict__ rects, const int* __restrict__ rect_off, int nframes, int total,
            u32* __restrict__ mask, Dims d)
{
    const int ri = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (ri >= total) return;
    int flo = 0, fhi = nframes;                     // largest f with rect_off[f] <= ri
    while (fhi - flo > 1) { int mid = (flo + fhi) >> 1; if (rect_off[mid] <= ri) flo = mid; else fhi = mid; }
    const int4 r = rects[ri];
    int r0 = max(r.x, 0), r1 = min(r.y, d.H), c0 = max(r.z, 0), c1 = min(r.w, d.W);
    if (r0 >= r1 || c0 >= c1) return;
    int w0 = c0 >> 5, w1 = (c1 - 1) >> 5;
    int nw = w1 - w0 + 1;
    int totalw = (r1 - r0) * nw;
    u32* m = mask + (size_t)flo * d.NW;
    for (int i = lane_id(); i < totalw; i += 32) {
        int row = r0 + i / nw, w = w0 + i % nw;
        int lo = max(c0 - (w << 5), 0), hi = min(c1 - 1 - (w << 5), 31);
        atomicOr(&m[(size_t)(d.H - 1 - row) * d.WW + w], bit_range(lo, hi));
    }
}

// cv2.convertScaleAbs for alpha=1, beta=0: saturate_u8(rint(|v|)); NaN, inf and |v| >= 2^31 give 0
// (x86 cvtps2dq "integer indefinite" is negative and saturates to 0).
__device__ __forceinline__ u32 csa(float v)
{
    float a = fabsf(v);
    if (!(a < 2147483648.0f)) return 0u;
    int r = __float2int_rn(a);
    return (u32)min(r, 255);
}

__device__ __forceinline__ float bswapf(float v)
{
    return __uint_as_float(__byte_perm(__float_as_uint(v), 0, 0x0123));
}

// ---- generic variant: also emits the clipped float image (standalone pass functions with write-back).
// mode 0: whole-frame pipeline: mask + flip + bright clip -> gray0 ; + dim threshold/offset -> gray1
//         (the library runs k_prep<0, *> there; mode 0 is profiles/lab/prep_lab.cu's reference)
// mode 1: standalone bright on an already flipped frame (no mask, no flip) -> gray0
// mode 2: standalone dim on an already flipped frame (no bright clip)     -> gray1
// Each thread converts 4 consecutive pixels (W % 4 == 0).  hist: [2][n][256].
// clipped (optional): float image after the in-place clip of the selected standalone pass.
__global__ void __launch_bounds__(256)
k_prep_generic(const float* __restrict__ in, const u32* __restrict__ mask, u8* __restrict__ gray0,
       u8* __restrict__ gray1, u32* __restrict__ hist0, u32* __restrict__ hist1, float* __restrict__ clipped,
       Dims d, int mode, float minFlux, float addFlux)
{
    __shared__ u32 sh[2][256];
    int f = blockIdx.y;
    for (int i = threadIdx.x; i < 512; i += blockDim.x) (&sh[0][0])[i] = 0;
    __syncthreads();

    const float* src = in + (size_t)f * d.N;
    int quads = d.N >> 2;
    int wq = d.W >> 2;
    // bins 0..2 hold almost every pixel of a sky-subtracted frame (dim: |v + addFlux| rounds to 1 or 2);
    // they are counted in registers and merged once per warp, the rest goes to shared-memory atomics
    u32 z0[3] = {0, 0, 0}, z1[3] = {0, 0, 0};
    const int stride = gridDim.x * blockDim.x;
    for (int q0 = blockIdx.x * blockDim.x + threadIdx.x; q0 < quads; q0 += 2 * stride) {
        // two independent 16-byte loads in flight per thread
        float4 vv[2];
        int qq[2] = {q0, q0 + stride};
        int yy[2], xx[2];
#pragma unroll
        for (int u = 0; u < 2; u++) {
            int q = qq[u];
            if (q < quads) {
                yy[u] = q / wq; xx[u] = (q - yy[u] * wq) << 2;
                int sy = (mode == 0) ? (d.H - 1 - yy[u]) : yy[u];
                vv[u] = __ldcs(reinterpret_cast<const float4*>(src + (size_t)sy * d.W + xx[u]));
            }
        }
#pragma unroll
        for (int u = 0; u < 2; u++) {
            int q = qq[u];
            if (q >= quads) continue;
            int y = yy[u], x = xx[u];
            float4 v = vv[u];
            float a[4] = {v.x, v.y, v.z, v.w};
            u32 mbits = 0;
            if (mode == 0) mbits = (mask[(size_t)f * d.NW + (size_t)y * d.WW + (x >> 5)] >> (x & 31)) & 0xf;
            u32 g0 = 0, g1 = 0;
            float cl[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
                float t = a[k];
                if (mbits & (1u << k)) t = 0.0f;
                if (mode != 2) { if (t < 0.0f) t = 0.0f; }          // bright clip (NaN stays NaN)
                float b = t;
                if (mode != 1) {
                    if (b < minFlux) b = 0.0f;
                    if (b > 0.0f) b = __fadd_rn(b, addFlux);
                }
                u32 c0 = csa(t), c1 = csa(b);
                g0 |= c0 << (8 * k);
                g1 |= c1 << (8 * k);
                if (mode != 2) {
                    if (c0 < 3) { z0[0] += (c0 == 0); z0[1] += (c0 == 1); z0[2] += (c0 == 2); }
                    else atomicAdd(&sh[0][c0], 1u);
                }
                if (mode != 1) {
                    if (c1 < 3) { z1[0] += (c1 == 0); z1[1] += (c1 == 1); z1[2] += (c1 == 2); }
                    else atomicAdd(&sh[1][c1], 1u);
                }
                cl[k] = (mode == 2) ? b : t;
            }
            size_t o = (size_t)f * d.N + (size_t)y * d.W + x;
            if (mode != 2) *reinterpret_cast<u32*>(gray0 + o) = g0;
            if (mode != 1) *reinterpret_cast<u32*>(gray1 + o) = g1;
            if (clipped) *reinterpret_cast<float4*>(clipped + o) = make_float4(cl[0], cl[1], cl[2], cl[3]);
        }
    }
    // low bins: warp-aggregate before touching shared memory
#pragma unroll
    for (int k = 0; k < 3; k++) {
        for (int o = 16; o; o >>= 1) {
            z0[k] += __shfl_xor_sync(FULLMASK, z0[k], o);
            z1[k] += __shfl_xor_sync(FULLMASK, z1[k], o);
        }
        if (lane_id() == 0) {
            if (z0[k]) atomicAdd(&sh[0][k], z0[k]);
            if (z1[k]) atomicAdd(&sh[1][k], z1[k]);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        if (mode != 2 && sh[0][i]) atomicAdd(&hist0[(size_t)f * 256 + i], sh[0][i]);
        if (mode != 1 && sh[1][i]) atomicAdd(&hist1[(size_t)f * 256 + i], sh[1][i]);
    }
}


// ---- fast variant (no clipped output): the instruction-lean kernel of the batch pipeline -----------------
// saturate_u8(rint(|v|)) in three instructions: fabs (operand modifier), the >= 2^31 / NaN / inf -> 0
// select, and one cvt.rni.sat.u8.f32 (round-half-even + saturation in hardware; NaN converts to 0).
__device__ __forceinline__ u32 csa_fast(float v)
{
    float a = fabsf(v);
    a = (a < 2147483648.0f) ? a : 0.0f;
    u32 r;
    asm("cvt.rni.sat.u8.f32 %0, %1;" : "=r"(r) : "f"(a));
    return r;
}

// rint to u8 for 0 <= a < 256: a + 2^23 leaves round-half-even(a) in the low mantissa byte (FADD rounds to
// nearest even) - one full-rate FP32 instruction instead of a quarter-rate F2I.  The sum's bit pattern is
// 0x4B0000xx exactly when 0 <= a < 255.5; anything that needs saturation or special handling (a >= 255.5,
// |v| >= 2^31, inf - which cv2 maps to 0, not 255 -, NaN, and negative sums, whose sign bit makes them huge
// unsigned numbers) is above RINT_BITS_MAX as an unsigned integer and is redone exactly by the caller; a sum
// that rounds to just below 2^23 (a small negative a, only possible with a negative addFlux) is below
// RINT_BITS_MIN.
__device__ __forceinline__ u32 rint_bits(float a) { return __float_as_uint(__fadd_rn(a, 8388608.0f)); }
#define RINT_BITS_MIN 0x4B000000u
#define RINT_BITS_MAX 0x4B0000ffu
// true when any of the eight sums needs the exact path (a[]: never negative; b[]: negative only if addFlux < 0)
__device__ __forceinline__ bool rint_bits_special(const u32 (&a)[4], const u32 (&b)[4], bool b_may_be_negative)
{
    u32 m = __vimax3_u32(a[0], a[1], a[2]);
    m = __vimax3_u32(m, a[3], b[0]);
    m = __vimax3_u32(m, b[1], b[2]);
    m = max(m, b[3]);
    bool sp = m > RINT_BITS_MAX;
    if (b_may_be_negative) sp = sp || min(min(b[0], b[1]), min(b[2], b[3])) < RINT_BITS_MIN;
    return sp;
}

__device__ __forceinline__ u32 pack_low_bytes(u32 u0, u32 u1, u32 u2, u32 u3)
{
    return __byte_perm(__byte_perm(u0, u1, 0x0040), __byte_perm(u2, u3, 0x0040), 0x5410);
}

// one float4: mask, clips, both conversions.  t[] are the un-flipped-source pixels of 4 consecutive columns.
template <int MODE>
__device__ __forceinline__ void prep4(float4 v, u32 mb, float minFlux, float addFlux, u32& g0, u32& g1)
{
    if (MODE == 0 && mb) {
        if (mb & 1u) v.x = 0.0f;
        if (mb & 2u) v.y = 0.0f;
        if (mb & 4u) v.z = 0.0f;
        if (mb & 8u) v.w = 0.0f;
    }
    float t[4] = {v.x, v.y, v.z, v.w};
    u32 a[4] = {RINT_BITS_MIN, RINT_BITS_MIN, RINT_BITS_MIN, RINT_BITS_MIN}, b[4] = {RINT_BITS_MIN, RINT_BITS_MIN, RINT_BITS_MIN, RINT_BITS_MIN};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        float tt = t[k];
        if (MODE != 2) {
            tt = fmaxf(tt, 0.0f);              // v < 0 -> 0 ; NaN -> 0 (the reference keeps NaN, which converts to 0 too)
            a[k] = rint_bits(tt);
        }
        if (MODE != 1) {
            float bb = (tt < minFlux) ? 0.0f : tt;
            bb = (bb > 0.0f) ? __fadd_rn(bb, addFlux) : bb;
            if (MODE == 2) bb = fabsf(bb);     // standalone dim: negative input -> |v| ; NaN fails the overflow test below
            b[k] = rint_bits(bb);
        }
    }
    g0 = (MODE != 2) ? pack_low_bytes(a[0], a[1], a[2], a[3]) : 0u;
    g1 = (MODE != 1) ? pack_low_bytes(b[0], b[1], b[2], b[3]) : 0u;
    // exact redo of the rare pixels that need saturation / special values (MODE 2 converts |v|: never negative)
    if (rint_bits_special(a, b, MODE == 0 && !(addFlux >= 0.0f))) {
        g0 = 0; g1 = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            float tt = t[k];
            if (MODE != 2) { tt = fmaxf(tt, 0.0f); g0 |= csa_fast(tt) << (8 * k); }
            if (MODE != 1) {
                float bb = (tt < minFlux) ? 0.0f : tt;
                bb = (bb > 0.0f) ? __fadd_rn(bb, addFlux) : bb;
                g1 |= csa_fast(bb) << (8 * k);
            }
        }
    }
}

// ================================================================================================
// k_prep: the batch-pipeline kernel.  The float frames are staged through shared memory by the TMA engine.
// Every warp owns a ring of PR_S stages of PR_CB bytes (one stage = 512 consecutive pixels of a row) filled by
// 1-D bulk-async copies (cp.async.bulk -> UBLKCP) that complete on the warp's own mbarriers: lane 0 re-arms a
// stage as soon as the warp has consumed it, so the bytes in flight per SM (PR_WARPS x PR_S x 2 KB per CTA) no
// longer depend on registers or on how many warps are stalled, and no __syncthreads is needed in the loop.
// Per chunk a lane converts four float4 (q = lane + 32k: conflict-free LDS.128, 128-byte coalesced stores),
// the star-mask words of the chunk are fetched one chunk ahead (16 words, one per lane) and skipped with a
// single vote when the chunk holds no blotted pixel, and the histogram bookkeeping is per chunk: bin 1 by
// dp4a byte sums, one test for "any byte >= 2" over the eight output words.
// ================================================================================================
#define PR_WARPS 8
#define PR_S 2
#define PR_Q 4                              // float4 per lane per chunk
#define PR_CF4 (32 * PR_Q)                  // float4 per chunk
#define PR_CB (PR_CF4 * 16)                 // bytes per chunk
#define PR_SMEM (PR_WARPS * PR_S * PR_CB + 2 * 256 * 4 + PR_WARPS * PR_S * 8 + PR_WARPS * 2 * 256 * 4)

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(u32 bar, u32 count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory"); }
__device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes) { asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory"); }
__device__ __forceinline__ void bulk_g2s(u32 dst, const void* src, u32 bytes, u32 bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(u32 bar, u32 parity)
{
    asm volatile("{\n.reg .pred P1;\nLAB_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n@P1 bra DONE;\nbra LAB_WAIT;\nDONE:\n}"
                 :: "r"(bar), "r"(parity) : "memory");
}

// Pipeline-mode conversion of one float4 (mask + bright clip -> g0 ; + dim threshold/offset -> g1).
// After the bright clip t is never negative or NaN, so the two dim conditions "not (t < minFlux)" and "t > 0"
// (processfield.py:453-454) are the single compare t >= thr, thr = minFlux > 0 ? minFlux : smallest denormal.
template <bool BE>
__device__ __forceinline__ void prep4_pipe(float4 v, u32 mb, float thr, float minFlux, float addFlux, u32& g0, u32& g1)
{
    if (BE) { v.x = bswapf(v.x); v.y = bswapf(v.y); v.z = bswapf(v.z); v.w = bswapf(v.w); }
    if (mb) {
        if (mb & 1u) v.x = 0.0f;
        if (mb & 2u) v.y = 0.0f;
        if (mb & 4u) v.z = 0.0f;
        if (mb & 8u) v.w = 0.0f;
    }
    const float t[4] = {v.x, v.y, v.z, v.w};
    u32 a[4], b[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const float tt = fmaxf(t[k], 0.0f);              // v < 0 -> 0 ; NaN -> 0 (the reference keeps NaN, which converts to 0 too)
        a[k] = rint_bits(tt);
        const float s = __fadd_rn(tt, addFlux);
        b[k] = rint_bits((tt >= thr) ? s : 0.0f);
    }
    g0 = pack_low_bytes(a[0], a[1], a[2], a[3]);
    g1 = pack_low_bytes(b[0], b[1], b[2], b[3]);
    if (rint_bits_special(a, b, !(addFlux >= 0.0f))) {                                     // rare: exact redo
        g0 = 0; g1 = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const float tt = fmaxf(t[k], 0.0f);
            g0 |= csa_fast(tt) << (8 * k);
            float bb = (tt < minFlux) ? 0.0f : tt;
            bb = (bb > 0.0f) ? __fadd_rn(bb, addFlux) : bb;
            g1 |= csa_fast(bb) << (8 * k);
        }
    }
}

// Exact bookkeeping of one word that may hold bytes >= 2 (n1 already holds the word's dp4a byte sum): a SWAR test
// marks the bytes >= 2, those go to shared-memory atomics one by one (predicated, no nested branches), bin 1 is
// corrected to the number of bytes that are exactly 1.
__device__ __forceinline__ void hist4_fix(u32 g, u32& n1, u32& nbig, u32* sh)
{
    const u32 m2 = g & 0xfefefefeu;
    const u32 t = (((m2 & 0x7f7f7f7fu) + 0x7f7f7f7fu) | m2) & 0x80808080u;     // bit 7 of every byte that is >= 2
    if (t) {
        n1 += __popc(g & 0x01010101u & ~(t >> 7)) - __dp4a(g, 0x01010101u, 0u);
        nbig += __popc(t);
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (t & (0x80u << (8 * k))) atomicAdd(&sh[(g >> (8 * k)) & 0xffu], 1u);
    }
}

// Words with a byte >= 2 (star pixels) are not histogrammed where they are produced: a shared-memory atomic issued
// from the conversion loop with one or two active lanes costs the warp ~150 cycles each (measured: a dense field
// took 25 % longer than a sparse one for 1.4 % such words).  They are appended to a per-warp staging list instead
// (ballot + popc slot allocation, plain stores) and histogrammed 32 words at a time with all lanes active.
#define PR_STG 256                          // staging words per warp and plane; one chunk adds at most 128
__device__ __forceinline__ void stage_big(const u32 (&G)[PR_Q], u32* stg, int& base, int lane)
{
    const u32 lt = (1u << lane) - 1u;
#pragma unroll
    for (int k = 0; k < PR_Q; k++) {
        const bool big = (G[k] & 0xfefefefeu) != 0u;
        const u32 b = __ballot_sync(FULLMASK, big);
        if (big) stg[base + __popc(b & lt)] = G[k];
        base += __popc(b);
    }
}
__device__ __forceinline__ void drain_big(const u32* stg, int& base, u32& n1, u32& nbig, u32* sh, int lane)
{
    __syncwarp();
    for (int i = lane; i < base; i += 32) hist4_fix(stg[i], n1, nbig, sh);
    __syncwarp();
    base = 0;
}

// MODE 0: pipeline (mask + flip, both passes) ; 1: bright only ; 2: dim only (no bright clip).
// grid = (CTAs per frame, frames in flight), one resident wave; dynamic shared memory PR_SMEM bytes.
// MINB = 3 resident CTAs per SM (72 registers): measured 3-5 % faster than 4 CTAs of 64 registers.
template <int MODE, bool BE, int MINB = 3>
__global__ void __launch_bounds__(PR_WARPS * 32, MINB)
k_prep(const float* __restrict__ in, const u32* __restrict__ mask, u8* __restrict__ gray0, u8* __restrict__ gray1,
            u32* __restrict__ hist0, u32* __restrict__ hist1, Dims d, int nframes, float minFlux, float addFlux)
{
    static_assert(MODE == 0 || !BE, "the standalone passes (lfd_run_pass) read native float32 only");
    extern __shared__ __align__(128) unsigned char dsm[];
    float4* ring = reinterpret_cast<float4*>(dsm);                                       // [PR_WARPS][PR_S][PR_CF4]
    u32* sh = reinterpret_cast<u32*>(dsm + (size_t)PR_WARPS * PR_S * PR_CB);             // [2][256]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(sh + 512);          // [PR_WARPS][PR_S]
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    u32* stg0 = reinterpret_cast<u32*>(bars + PR_WARPS * PR_S) + (size_t)wid * 2 * PR_STG;   // [PR_WARPS][2][PR_STG]
    u32* stg1 = stg0 + PR_STG;
    int nst0 = 0, nst1 = 0;
    for (int i = threadIdx.x; i < 512; i += blockDim.x) sh[i] = 0;
    if (lane == 0)
        for (int s = 0; s < PR_S; s++) mbar_init(smem_u32(&bars[wid * PR_S + s]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    const int rowb = d.W * 4;                          // bytes per row (a multiple of 16: W % 4 == 0)
    const int cpr = (rowb + PR_CB - 1) / PR_CB;        // chunks per row
    const int total = d.H * cpr;
    const int stride = gridDim.x * PR_WARPS;
    const int dy = stride / cpr, dj = stride - dy * cpr;
    const float thr = (minFlux > 0.0f) ? minFlux : __int_as_float(1);
    const u32 ring0 = smem_u32(ring + (size_t)wid * PR_S * PR_CF4);
    const u32 bar0 = smem_u32(&bars[wid * PR_S]);

    // gridDim.y frames are in flight at a time (each frame read and written as three sequential streams: fewer
    // concurrent streams keep more DRAM pages open); a CTA walks the frames blockIdx.y, blockIdx.y + gridDim.y, ...
    int ps = 0, cs = 0; u32 cpar = 0;                  // ring stage of the producer / consumer, consumer phase parity
    for (int f = blockIdx.y; f < nframes; f += gridDim.y) {
    const char* src = reinterpret_cast<const char*>(in + (size_t)f * d.N);
    const u32* mf = mask + (size_t)f * d.NW;
    u32* o0 = reinterpret_cast<u32*>(gray0 + (size_t)f * d.N);
    u32* o1 = reinterpret_cast<u32*>(gray1 + (size_t)f * d.N);
    // producer state (next chunk to request) and consumer state (next chunk to convert)
    int pc = blockIdx.x * PR_WARPS + wid, py = pc / cpr, pj = pc - py * cpr;
    int cc = pc, cy = py, cj = pj;
    auto issue = [&]() {
        if (pc < total) {
            if (lane == 0) {
                const int sy = (MODE == 0) ? (d.H - 1 - py) : py;
                const u32 nb = (u32)min(PR_CB, rowb - pj * PR_CB);
                mbar_expect_tx(bar0 + 8 * ps, nb);
                bulk_g2s(ring0 + ps * PR_CB, src + (size_t)sy * rowb + (size_t)pj * PR_CB, nb, bar0 + 8 * ps);
            }
            pc += stride; py += dy; pj += dj; if (pj >= cpr) { pj -= cpr; py++; }
            ps = (ps + 1 == PR_S) ? 0 : ps + 1;
        }
    };
#pragma unroll
    for (int s = 0; s < PR_S; s++) issue();

    auto load_mask = [&](int y, int j) -> u32 {
        if (MODE != 0) return 0u;
        const int w = j * (4 * PR_Q) + lane;
        return (lane < 4 * PR_Q && w < d.WW) ? __ldg(mf + y * d.WW + w) : 0u;
    };
    u32 mword = (cc < total) ? load_mask(cy, cj) : 0u;
    u32 a1 = 0, abig = 0, b1 = 0, bbig = 0, nwords = 0;
    while (cc < total) {
        const int nf4 = min(PR_CF4, (rowb - cj * PR_CB) >> 4);
        const int xo = ((cy * d.W + cj * (PR_CB / 4)) >> 2) + lane;     // u32 index of this lane's first output word
        const u32 mcur = mword;
        cc += stride; cy += dy; cj += dj; if (cj >= cpr) { cj -= cpr; cy++; }
        if (cc < total) mword = load_mask(cy, cj);                      // next chunk's mask words, one chunk ahead
        mbar_wait(bar0 + 8 * cs, cpar);
        const float4* buf = ring + ((size_t)wid * PR_S + cs) * PR_CF4 + lane;
        float4 v[PR_Q];
#pragma unroll
        for (int k = 0; k < PR_Q; k++) v[k] = buf[32 * k];
        const bool anym = (MODE == 0) ? __any_sync(FULLMASK, mcur != 0u) : false;
        u32* p0 = o0 + xo; u32* p1 = o1 + xo;
        u32 G0[PR_Q], G1[PR_Q];
#pragma unroll
        for (int k = 0; k < PR_Q; k++) {
            u32 mb = 0;
            if (anym) mb = (__shfl_sync(FULLMASK, mcur, (lane >> 3) + 4 * k) >> ((lane & 7) << 2)) & 0xfu;
            if (MODE == 0) prep4_pipe<BE>(v[k], mb, thr, minFlux, addFlux, G0[k], G1[k]);
            else prep4<MODE>(v[k], 0u, minFlux, addFlux, G0[k], G1[k]);
        }
        if (nf4 == PR_CF4) {
#pragma unroll
            for (int k = 0; k < PR_Q; k++) {
                if (MODE != 2) p0[32 * k] = G0[k];
                if (MODE != 1) p1[32 * k] = G1[k];
            }
            nwords += PR_Q;
        } else {                                                        // last chunk of a row when 4W % PR_CB != 0
#pragma unroll
            for (int k = 0; k < PR_Q; k++) {
                if (lane + 32 * k < nf4) {
                    if (MODE != 2) p0[32 * k] = G0[k];
                    if (MODE != 1) p1[32 * k] = G1[k];
                    nwords++;
                } else { G0[k] = 0u; G1[k] = 0u; }
            }
        }
        // histogram: bin 1 = byte sums (exact while every byte is 0 or 1), bin 0 = remainder, anything else is rare
        u32 or0 = 0, or1 = 0;
#pragma unroll
        for (int k = 0; k < PR_Q; k++) {
            if (MODE != 2) { a1 = __dp4a(G0[k], 0x01010101u, a1); or0 |= G0[k]; }
            if (MODE != 1) { b1 = __dp4a(G1[k], 0x01010101u, b1); or1 |= G1[k]; }
        }
        if (MODE != 2 && __any_sync(FULLMASK, (or0 & 0xfefefefeu) != 0u)) {
            if (nst0 > PR_STG - 32 * PR_Q) drain_big(stg0, nst0, a1, abig, sh, lane);
            stage_big(G0, stg0, nst0, lane);
        }
        if (MODE != 1 && __any_sync(FULLMASK, (or1 & 0xfefefefeu) != 0u)) {
            if (nst1 > PR_STG - 32 * PR_Q) drain_big(stg1, nst1, b1, bbig, sh + 256, lane);
            stage_big(G1, stg1, nst1, lane);
        }
        __syncwarp();                                                   // every lane has consumed the stage
        issue();                                                        // ... so it can be refilled
        cs++; if (cs == PR_S) { cs = 0; cpar ^= 1u; }
    }
    if (MODE != 2) drain_big(stg0, nst0, a1, abig, sh, lane);
    if (MODE != 1) drain_big(stg1, nst1, b1, bbig, sh + 256, lane);
    u32 acc[4] = {a1, 4u * nwords - a1 - abig, b1, 4u * nwords - b1 - bbig};
#pragma unroll
    for (int k = 0; k < 4; k++) {
        u32 vsum = acc[k];
        for (int o = 16; o; o >>= 1) vsum += __shfl_xor_sync(FULLMASK, vsum, o);
        if (lane == 0 && vsum) atomicAdd(&sh[(k >> 1) * 256 + ((k & 1) ? 0 : 1)], vsum);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x) {
        if (MODE != 2 && sh[i]) atomicAdd(&hist0[(size_t)f * 256 + i], sh[i]);
        if (MODE != 1 && sh[256 + i]) atomicAdd(&hist1[(size_t)f * 256 + i], sh[256 + i]);
        sh[i] = 0; sh[256 + i] = 0;
    }
    __syncthreads();
    }   // frames
}

// cv2.equalizeHist's LUT from the 256-bin histogram; one 256-thread block per (frame, pass).
// grid = (n, 2): blockIdx.y selects hist/lut of pass 0/1 (pointers are [2][n][256] slabs).
__global__ void __launch_bounds__(256)
k_lut(const u32* __restrict__ hist, u8* __restrict__ lut, const FrameCtl* __restrict__ ctl, int n, int total,
      int pass_lo)
{
    int f = blockIdx.x, p = pass_lo + blockIdx.y;
    if (!ctl[f].active[p]) return;
    const u32* h = hist + ((size_t)p * n + f) * 256;
    u8* l = lut + ((size_t)p * n + f) * 256;
    __shared__ int s[256];
    __shared__ int i0s;
    int t = threadIdx.x;
    int hv = (int)h[t];
    if (t == 0) i0s = 256;
    __syncthreads();
    if (hv > 0) atomicMin(&i0s, t);
    __syncthreads();
    int i0 = i0s;
    if (i0 == 256 || (int)h[i0] == total) { l[t] = (u8)t; return; }   // constant image: dst = src
    s[t] = (t > i0) ? hv : 0;
    __syncthreads();
    for (int o = 1; o < 256; o <<= 1) {
        int v = (t >= o) ? s[t - o] : 0;
        __syncthreads();
        s[t] += v;
        __syncthreads();
    }
    float scale = 255.0f / (float)(total - (int)h[i0]);
    int val = 0;
    if (t > i0) {
        val = __float2int_rn(__fmul_rn((float)s[t], scale));
        val = min(max(val, 0), 255);
    }
    l[t] = (u8)val;
}

// expand a bit mask to a 0/255 uint8 plane (stage taps)
__global__ void k_expand_mask(const u32* __restrict__ mask, u8* __restrict__ out, Dims d)
{
    int f = blockIdx.y;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.N; i += gridDim.x * blockDim.x) {
        int y = i / d.W, x = i - y * d.W;
        u32 w = mask[(size_t)f * d.NW + (size_t)y * d.WW + (x >> 5)];
        out[(size_t)f * d.N + i] = ((w >> (x & 31)) & 1u) ? 255 : 0;
    }
}

// LUT applied to a plane (EQU tap: equalizeHist output before morphology)
__global__ void k_apply_lut(const u8* __restrict__ in, const u8* __restrict__ lut, u8* __restrict__ out, Dims d)
{
    int f = blockIdx.y;
    const u8* l = lut + (size_t)f * 256;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.N; i += gridDim.x * blockDim.x)
        out[(size_t)f * d.N + i] = l[in[(size_t)f * d.N + i]];
}
