// k_inject.cuh - on-device trail injection for completeness campaigns (lfd_set_base / lfd_submit_injected[_shaped]),
// and k_capture_bases, which makes a collected batch the injection bases (lfd_capture_bases).
//
// in[f] = base[base_index[f]] + the line segments of slot f (the checkers are oracle/inject_ref.py::render_trails and,
// for tabulated shapes, tests/inject_shapes_ref.py::render_trails).  Per pixel, in float32 and in
// lfd_b200/synth.py::_add_trail's operation order:
//   t = (x - x0) * ux + (y - y0) * uy,   d = -(x - x0) * uy + (y - y0) * ux
//   pixel += (peak * P(d)) * A(t)   iff 0 <= t <= L and dlo <= d <= dhi
// with ux, uy, L rounded to float32 from double on the host.  P is _add_trail's Gaussian expf(-0.5f * (d / sigma)^2)
// with [dlo, dhi] = [-pad, pad], pad = ceil(5 sigma) + 1, or the linear interpolation of a tabulated profile on
// [dlo, dhi]; A is 1 or the linear interpolation of a tabulated light curve over [0, L] (include/lfd_b200.h, lfd_table).
// Every product and sum is an explicit round-to-nearest intrinsic, so footprint membership and the tabulated shapes are
// bit-identical to the NumPy reference and only expf may differ in the last bits.
#pragma once
#include "common.cuh"

#define INJ_ROWS 8                  // frame rows per CTA
#define INJ_THREADS 256

// one trail as the kernel uses it (host-prepared from lfd_trail and lfd_trail_shape); L == 0 marks a zero-length trail
// (adds nothing).  pn == 0: Gaussian profile of sigma; else pn samples at poff on [dlo, dhi], inv = (pn - 1) / (dhi - dlo).
// lm == 0: no light curve; else lm samples at loff over [0, L], c = (lm - 1) / L.
struct InjTrail {
    float x0, y0, ux, uy, L, sigma, peak, dlo, dhi, inv, c;
    int poff, pn, loff, lm;
};

// Conservative x-range [lo, hi] of the pixels of row y the float32 test can accept: the exact interval of the rotated
// rectangle, widened by `slack` in t and d (far more than the float32 rounding of t and d) and by one pixel.
__device__ __forceinline__ int2 inj_row_range(const InjTrail& T, int y, int W)
{
    const double slack = 1e-5 * (fabs((double)T.x0) + fabs((double)T.y0) + (double)W + (double)y) + 1e-3;
    double lo = 0.0, hi = (double)(W - 1);
    const double yy = (double)y - (double)T.y0;
    // t(x) = ux * (x - x0) + yy * uy in [-slack, L + slack];  d(x) = -uy * (x - x0) + yy * ux in [dlo - slack, dhi + slack]
    const double c[2] = {(double)T.ux, -(double)T.uy};
    const double o[2] = {yy * (double)T.uy, yy * (double)T.ux};
    const double a[2] = {-slack, (double)T.dlo - slack};
    const double b[2] = {(double)T.L + slack, (double)T.dhi + slack};
    for (int k = 0; k < 2; k++) {
        if (c[k] == 0.0) {
            if (o[k] < a[k] || o[k] > b[k]) return make_int2(1, 0);
            continue;
        }
        double u = (a[k] - o[k]) / c[k] + (double)T.x0, v = (b[k] - o[k]) / c[k] + (double)T.x0;
        if (u > v) { double s = u; u = v; v = s; }
        lo = fmax(lo, u - 1.0);
        hi = fmin(hi, v + 1.0);
    }
    if (!(lo <= hi)) return make_int2(1, 0);
    return make_int2((int)floor(lo), (int)ceil(hi));
}

// a[i] + f * (a[i+1] - a[i]) at u >= 0, i = min(trunc(u), n - 2), f = u - i: the table value of lfd_table
__device__ __forceinline__ float inj_lerp(const float* __restrict__ a, int n, float u)
{
    const int i = min((int)u, n - 2);
    const float f = __fsub_rn(u, (float)i), a0 = __ldg(a + i), a1 = __ldg(a + i + 1);
    return __fadd_rn(a0, __fmul_rn(f, __fsub_rn(a1, a0)));
}

// grid (ceil(H / INJ_ROWS), n), INJ_THREADS threads; W % 4 == 0 (lfd_create)
__global__ void __launch_bounds__(INJ_THREADS)
k_inject(const float* __restrict__ base, const int* __restrict__ base_index, const InjTrail* __restrict__ trails,
         const int* __restrict__ trail_off, const float* __restrict__ samples, float* __restrict__ out, Dims d)
{
    __shared__ InjTrail st[LFD_MAX_INJECT_TRAILS];
    __shared__ int2 rng[INJ_ROWS][LFD_MAX_INJECT_TRAILS];
    __shared__ int2 urng[INJ_ROWS];           // union of the row's ranges: outside it a float4 is copied as is
    const int f = blockIdx.y, y0 = blockIdx.x * INJ_ROWS, tid = threadIdx.x;
    const int t0 = trail_off[f], nt = trail_off[f + 1] - t0;
    const int rows = min(INJ_ROWS, d.H - y0);
    if (tid < nt) st[tid] = trails[t0 + tid];
    __syncthreads();
    for (int i = tid; i < rows * nt; i += INJ_THREADS) {
        const int r = i / nt, k = i - r * nt;
        rng[r][k] = st[k].L > 0.f ? inj_row_range(st[k], y0 + r, d.W) : make_int2(1, 0);
    }
    __syncthreads();
    if (tid < rows) {
        int lo = d.W, hi = -1;
        for (int k = 0; k < nt; k++) { const int2 q = rng[tid][k]; if (q.x <= q.y) { lo = min(lo, q.x); hi = max(hi, q.y); } }
        urng[tid] = make_int2(lo, hi);
    }
    __syncthreads();
    const int W4 = d.W >> 2;
    const float4* src = reinterpret_cast<const float4*>(base + (size_t)base_index[f] * d.N + (size_t)y0 * d.W);
    float4* dst = reinterpret_cast<float4*>(out + (size_t)f * d.N + (size_t)y0 * d.W);
    const int total = rows * W4;
    // four independent 16-byte loads in flight per thread before any store
    for (int i0 = tid; i0 < total; i0 += 4 * INJ_THREADS) {
        float4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = i0 + j * INJ_THREADS;
            if (i < total) v[j] = __ldcs(src + i);
        }
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const int i = i0 + j * INJ_THREADS;
            if (i >= total) break;
            const int r = i / W4, x4 = (i - r * W4) << 2;
            const int2 u = urng[r];
            if (x4 + 3 >= u.x && x4 <= u.y) {
                const float yf = (float)(y0 + r);
                float* e = &v[j].x;
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    const int x = x4 + c;
                    const float xf = (float)x;
                    float acc = e[c];
                    for (int k = 0; k < nt; k++) {
                        const int2 q = rng[r][k];
                        if (x < q.x || x > q.y) continue;
                        const InjTrail& T = st[k];
                        const float ax = __fsub_rn(xf, T.x0), by = __fsub_rn(yf, T.y0);
                        const float t = __fadd_rn(__fmul_rn(ax, T.ux), __fmul_rn(by, T.uy));
                        const float dd = __fadd_rn(-__fmul_rn(ax, T.uy), __fmul_rn(by, T.ux));
                        if (t >= 0.f && t <= T.L && dd >= T.dlo && dd <= T.dhi) {
                            float p;
                            if (T.pn == 0) {
                                const float q2 = __fdiv_rn(dd, T.sigma);
                                p = expf(__fmul_rn(-0.5f, __fmul_rn(q2, q2)));
                            } else {
                                p = inj_lerp(samples + T.poff, T.pn, __fmul_rn(__fsub_rn(dd, T.dlo), T.inv));
                            }
                            float add = __fmul_rn(T.peak, p);
                            if (T.lm) add = __fmul_rn(add, inj_lerp(samples + T.loff, T.lm, __fmul_rn(t, T.c)));
                            acc = __fadd_rn(acc, add);
                        }
                    }
                    e[c] = acc;
                }
            }
            dst[i] = v[j];
        }
    }
}

#define CAP_THREADS 256

// lfd_capture_bases: the batch slots -> the injection bases, n16 16-byte words, each 4-byte word byte-swapped when the
// slots hold a raw FITS payload (BE).  Grid-stride, four independent loads in flight per thread; the slots are
// overwritten by k_inject next, so they are read with evict-first loads.
template <bool BE>
__global__ void __launch_bounds__(CAP_THREADS) k_capture_bases(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t n16)
{
    const size_t step = (size_t)gridDim.x * CAP_THREADS;
    for (size_t i0 = (size_t)blockIdx.x * CAP_THREADS + threadIdx.x; i0 < n16; i0 += 4 * step) {
        uint4 v[4];
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (i0 + j * step < n16) v[j] = __ldcs(src + i0 + j * step);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (i0 + j * step >= n16) break;
            if (BE) {
                v[j].x = __byte_perm(v[j].x, 0, 0x0123); v[j].y = __byte_perm(v[j].y, 0, 0x0123);
                v[j].z = __byte_perm(v[j].z, 0, 0x0123); v[j].w = __byte_perm(v[j].w, 0, 0x0123);
            }
            dst[i0 + j * step] = v[j];
        }
    }
}
