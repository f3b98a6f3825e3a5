// TEST-ONLY: compiles lfd_b200/csrc/chords.cuh for the host so the CPU suite can check the chord decomposition the
// library uploads for arbitrary structuring elements.  Never loaded by the product.
#include "../lfd_b200/csrc/chords.cuh"
extern "C" {
int hc_max_side(void) { return CHORD_MAX_SIDE; }
int hc_capacity(int kh, int kw) { return chord_capacity(kh, kw); }
int hc_decompose(const uint8_t* mask, int kh, int kw, int* rowoff, uint32_t* code, int* nlev)
{
    return chord_decompose(mask, kh, kw, rowoff, code, nlev);
}
}
