// chords.cuh - chord decomposition of a flat structuring element (Urbach & Wilkinson, "Efficient 2-D grayscale
// morphological transformations with arbitrary flat structuring elements", IEEE TIP 2008).
//
// Plain C++ with no CUDA dependency: lfd_b200.cu builds the chord lists with it, and tests/hostchords.cpp compiles it
// for the host so that the CPU suite checks the decomposition the library uploads.
//
// Each mask row i splits into maximal horizontal runs of members, the chords.  With cv2's default anchor
// (ax, ay) = (kw / 2, kh / 2), the chord starting at column a with length L stands for the offsets
// dy = i - ay, dx = a - ax .. a - ax + L - 1, and
//     out(y, x) = op over chords of T_L(y + dy, x + dx),   T_L(r, c) = op(in(r, c .. c + L - 1)).
// With the per-row sparse table P_k(r, c) = op(in(r, c .. c + 2^k - 1)), T_L = op(P_k(r, c), P_k(r, c + L - 2^k)) for
// k = floor(log2 L): the two windows overlap, which min and max do not mind.
//
// Encoding of one chord (u32): bits 0-7 the column of the first window (a), bits 8-15 the column of the second
// (a + L - 2^k), bits 16-19 the level k.  Columns are relative to the mask's left edge, so sides are limited to 256.
#pragma once
#include <stdint.h>

#define CHORD_MAX_SIDE 255                       // largest structuring element side

// chord count bound of a kh x kw mask: a row of kw columns holds at most ceil(kw / 2) runs
inline int chord_capacity(int kh, int kw) { return kh * ((kw + 1) / 2); }

inline int chord_level(int len)
{
    int k = 0;
    while ((2 << k) <= len) k++;
    return k;
}

inline uint32_t chord_code(int a, int len)
{
    const int k = chord_level(len);
    return (uint32_t)a | ((uint32_t)(a + len - (1 << k)) << 8) | ((uint32_t)k << 16);
}

// The chords of a row-major kh x kw mask (non-zero = member), row by row, left to right.  rowoff[kh + 1]: chords of
// row i are code[rowoff[i] .. rowoff[i + 1]); code holds chord_capacity(kh, kw) entries.  Returns the chord count and
// sets *nlev to the number of sparse-table levels the chords use (floor(log2 of the longest chord) + 1, 0 if none).
inline int chord_decompose(const uint8_t* mask, int kh, int kw, int* rowoff, uint32_t* code, int* nlev)
{
    int n = 0, lmax = 0;
    for (int i = 0; i < kh; i++) {
        rowoff[i] = n;
        const uint8_t* row = mask + (long)i * kw;
        for (int j = 0; j < kw;) {
            if (!row[j]) { j++; continue; }
            int e = j;
            while (e < kw && row[e]) e++;
            code[n++] = chord_code(j, e - j);
            if (e - j > lmax) lmax = e - j;
            j = e;
        }
    }
    rowoff[kh] = n;
    *nlev = lmax > 0 ? chord_level(lmax) + 1 : 0;
    return n;
}
