// common.cuh - shared device-side definitions for the lfd_b200 library (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lfd_b200.h"

typedef uint32_t u32;
typedef uint64_t u64;
typedef uint8_t u8;
typedef uint16_t u16;

#define LFD_WARP 32
#define FULLMASK 0xffffffffu

// Per-frame bookkeeping that kernels read and write (one per batch slot).
struct FrameCtl {
    int active[2];        // pass p runs on this frame
    int hough[2];         // a rectangle passed in pass p -> run Hough
    int nruns[2];         // fg / bg run count of the current pass
    int ncomp[2];         // fg / bg contour count
    int nslots[2];        // row-extreme slots used
    int nhull[2];         // hull scratch used
    int npass;            // passing rectangles (current pass)
    int nseg[2];          // non-zero mask words: [0] morph (equ) mask, [1] box mask
    int npeaks[2];        // Hough peaks: equ / box
    int nnz[2];           // non-zero pixels voted: equ / box
    int status;           // LFD_FRAME_* bits
    int detected;         // this pass accepted a line (k_check_theta)
    int ncomp_saved[2][2]; // [pass][kind] contour counts kept for the RECTS tap
    int nsurv;            // contours k_rects_screen kept in the rectangle launch whose first frame this is
};

// A run of set bits in one mask row.
struct Run { u16 xs, xe, y, pad; };

// Geometry of one frame batch, passed by value to kernels.
struct Dims {
    int H, W, WW;         // WW = words per mask row
    int N;                // H*W
    int NW;               // H*WW
};

struct HoughCfg {
    int numangle, numrho, RS;   // RS = numrho + 2
    int apc;                    // angles per CTA in the vote kernel
    int ngroups;                // ceil(numangle / apc)
    float rho, theta;
    int threshold;
};

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ u32 tail_mask(int w, int W)
{
    // valid-bit mask of mask word w for an image W pixels wide
    int rem = W - (w << 5);
    return rem >= 32 ? 0xffffffffu : (rem <= 0 ? 0u : ((1u << rem) - 1u));
}

__device__ __forceinline__ u32 bit_range(int lo, int hi)
{
    // bits lo..hi inclusive, 0 <= lo <= hi <= 31
    u32 a = 0xffffffffu << lo;
    u32 b = 0xffffffffu >> (31 - hi);
    return a & b;
}
