// host_ingest.cuh - host-side ingest of the two SDSS file kinds on the path (plain C++, no CUDA, no GPU needed).
//
// The batched drop-in driver (lfd_b200/detecttrails.py::compute_fields) is bound by per-frame interpreter time
// under the GIL once the kernels and the PCIe copy are out of the way.  These two entry points do the per-frame
// file work in native code, with the GIL released by ctypes for the whole call:
//
//   lfd_fits_load_frame   fitsio.read + fitsio.read_header of a frame file
//                         (/root/reference/lfd/detecttrails/detecttrails.py:113-114): the primary 2-D BITPIX=-32
//                         image is read as raw big-endian payload straight into the caller's (pinned) buffer - the
//                         first kernel byte-swaps - and the raw value text of the requested header cards is returned.
//   lfd_catalog_rects     read_photoObj + the object filter + the blot slices of remove_stars
//                         (/root/reference/lfd/detecttrails/removestars.py:96-130, 212-231), restated from
//                         lfd_b200/removestars.py::star_rects (which is pinned against the reference in
//                         tests/test_host_logic.py); tests/test_host_logic.py::test_native_ingest_equals_python pins
//                         this restatement against star_rects.
//
// Both are strict: anything outside the plain layout the reference's files have (other BITPIX / shape, missing
// cards, other column formats, non-finite catalog values - for which the Python code raises the reference's
// exceptions - or an I/O error) returns LFD_E_UNSUPPORTED / LFD_E_ARG and the driver takes its Python path for
// that frame, so error texts and exotic files behave exactly as before.
#pragma once
#include <errno.h>
#include <fcntl.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#if defined(__x86_64__)
#include <immintrin.h>
#endif

#include <atomic>
#include <string>
#include <thread>
#include <vector>

#include "../../include/lfd_b200.h"

namespace lfdhost {

static const int FITS_BLOCK = 2880, FITS_CARD = 80;

struct Card { char key[9]; char value[71]; };          // keyword (trimmed) and the raw text after "= "

// Reads header blocks from `off` until END.  Returns the data offset (first byte after the header) or -1.
static long read_header(int fd, long off, std::vector<Card>& cards)
{
    cards.clear();
    char block[FITS_BLOCK];
    for (int nblocks = 0; nblocks < 4096; nblocks++) {
        ssize_t got = pread(fd, block, FITS_BLOCK, off);
        if (got != FITS_BLOCK) return -1;
        off += FITS_BLOCK;
        for (int i = 0; i < FITS_BLOCK; i += FITS_CARD) {
            const char* c = block + i;
            int kl = 8;
            while (kl > 0 && c[kl - 1] == ' ') kl--;
            if (kl == 3 && memcmp(c, "END", 3) == 0) return off;
            if (kl == 0 || c[8] != '=' || c[9] != ' ') continue;
            Card cd;
            memcpy(cd.key, c, kl); cd.key[kl] = 0;
            memcpy(cd.value, c + 10, 70); cd.value[70] = 0;
            cards.push_back(cd);
        }
    }
    return -1;
}

static const Card* find(const std::vector<Card>& cards, const char* key)
{
    for (const Card& c : cards)
        if (strcmp(c.key, key) == 0) return &c;
    return nullptr;
}

// integer card value ("   -32 / comment"); false if the card is missing or not a plain integer
static bool card_int(const std::vector<Card>& cards, const char* key, long* out)
{
    const Card* c = find(cards, key);
    if (!c) return false;
    const char* p = c->value;
    while (*p == ' ') p++;
    char* end = nullptr;
    errno = 0;
    long v = strtol(p, &end, 10);
    if (end == p || errno) return false;
    while (*end == ' ') end++;
    if (*end != 0 && *end != '/') return false;
    *out = v;
    return true;
}

// string card value ('BINTABLE' / 'ROWC    '): text between the quotes, trailing blanks removed
static bool card_str(const std::vector<Card>& cards, const char* key, std::string* out)
{
    const Card* c = find(cards, key);
    if (!c) return false;
    const char* p = c->value;
    while (*p == ' ') p++;
    if (*p != '\'') return false;
    p++;
    std::string s;
    while (*p) {
        if (*p == '\'') { if (p[1] == '\'') { s.push_back('\''); p += 2; continue; } break; }
        s.push_back(*p++);
    }
    while (!s.empty() && s.back() == ' ') s.pop_back();
    *out = s;
    return true;
}

// numeric card value as a double ("1.0", "0.000000E+00", "1"); false if missing or not a number
static bool card_num(const std::vector<Card>& cards, const char* key, double* out)
{
    const Card* c = find(cards, key);
    if (!c) return false;
    const char* p = c->value;
    while (*p == ' ') p++;
    char buf[72];
    size_t n = 0;
    while (p[n] && p[n] != ' ' && p[n] != '/' && n + 1 < sizeof buf) { buf[n] = (p[n] == 'D' || p[n] == 'd') ? 'E' : p[n]; n++; }
    buf[n] = 0;
    char* end = nullptr;
    errno = 0;
    double v = strtod(buf, &end);
    if (end == buf || *end != 0 || errno) return false;
    *out = v;
    return true;
}

static long data_bytes(const std::vector<Card>& cards)
{
    long naxis = 0, bitpix = 0;
    if (!card_int(cards, "NAXIS", &naxis) || !card_int(cards, "BITPIX", &bitpix)) return -1;
    if (naxis == 0) return 0;
    long n = 1;
    for (long i = 1; i <= naxis; i++) {
        char k[32]; snprintf(k, sizeof k, "NAXIS%ld", i);
        long v; if (!card_int(cards, k, &v) || v < 0) return -1;
        n *= v;
    }
    long gcount = 1, pcount = 0;
    card_int(cards, "GCOUNT", &gcount); card_int(cards, "PCOUNT", &pcount);
    return labs(bitpix) / 8 * gcount * (pcount + n);
}

static inline float be_f32(const unsigned char* p)
{
    uint32_t u = ((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3];
    float f; memcpy(&f, &u, 4); return f;
}
static inline int32_t be_i32(const unsigned char* p)
{
    return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | (uint32_t)p[3]);
}

// slice.indices() of a bound for step 1: a negative bound counts from the end, then it is clamped to [0, length]
static inline long resolve(long v, long length)
{
    if (v < 0) v += length;
    return v < 0 ? 0 : (v > length ? length : v);
}

struct Fd { int fd; explicit Fd(const char* p) : fd(open(p, O_RDONLY | O_CLOEXEC)) {} ~Fd() { if (fd >= 0) close(fd); } };

// The payload copy, page cache -> (pinned) staging slot, is what bounds the drop-in once kernels and PCIe are out of the
// way: 12.2 MB per frame on every loader thread at once, i.e. the host's memory bus.  read() copies with ordinary stores,
// so every destination line is first read for ownership: 3 bytes over the bus per payload byte.  Mapping the file and
// copying with non-temporal stores moves 2 (profiles/lab/ingest_lab.cpp: +50-60 % frames/s at 8 threads); the H2D DMA
// reads the slot from DRAM either way.  Payloads under 1 MiB, and files that cannot be mapped, take the plain pread().
#if defined(__x86_64__)
__attribute__((target("avx2"))) static void stream_copy_avx2(char* dst, const char* src, size_t n)
{
    size_t i = 0;
    for (; i < n && ((uintptr_t)(dst + i) & 31); i++) dst[i] = src[i];
    for (; i + 128 <= n; i += 128) {
        __m256i a = _mm256_loadu_si256((const __m256i*)(src + i)), b = _mm256_loadu_si256((const __m256i*)(src + i + 32));
        __m256i c = _mm256_loadu_si256((const __m256i*)(src + i + 64)), d = _mm256_loadu_si256((const __m256i*)(src + i + 96));
        _mm256_stream_si256((__m256i*)(dst + i), a); _mm256_stream_si256((__m256i*)(dst + i + 32), b);
        _mm256_stream_si256((__m256i*)(dst + i + 64), c); _mm256_stream_si256((__m256i*)(dst + i + 96), d);
    }
    for (; i < n; i++) dst[i] = src[i];
    _mm_sfence();
}

static void stream_copy_sse2(char* dst, const char* src, size_t n)
{
    size_t i = 0;
    for (; i < n && ((uintptr_t)(dst + i) & 15); i++) dst[i] = src[i];
    for (; i + 64 <= n; i += 64) {
        __m128i a = _mm_loadu_si128((const __m128i*)(src + i)), b = _mm_loadu_si128((const __m128i*)(src + i + 16));
        __m128i c = _mm_loadu_si128((const __m128i*)(src + i + 32)), d = _mm_loadu_si128((const __m128i*)(src + i + 48));
        _mm_stream_si128((__m128i*)(dst + i), a); _mm_stream_si128((__m128i*)(dst + i + 16), b);
        _mm_stream_si128((__m128i*)(dst + i + 32), c); _mm_stream_si128((__m128i*)(dst + i + 48), d);
    }
    for (; i < n; i++) dst[i] = src[i];
    _mm_sfence();
}
#endif

static void stream_copy(char* dst, const char* src, size_t n)
{
#if defined(__x86_64__)
    static const bool avx2 = __builtin_cpu_supports("avx2");
    if (avx2) stream_copy_avx2(dst, src, n); else stream_copy_sse2(dst, src, n);
#else
    memcpy(dst, src, n);
#endif
}

// nbytes of the file at `off` into dest.  false: short file or I/O error.
static bool read_payload(int fd, long off, long nbytes, char* dest)
{
    struct stat st;
    if (fstat(fd, &st) != 0 || (long)st.st_size < off + nbytes) return false;    // (a mapping past the end would fault)
    if (nbytes >= (1 << 20)) {
        const long pg = sysconf(_SC_PAGESIZE), a0 = off & ~(pg - 1);
        void* m = mmap(nullptr, (size_t)(off - a0 + nbytes), PROT_READ, MAP_SHARED | MAP_POPULATE, fd, a0);
        if (m != MAP_FAILED) {
            stream_copy(dest, (const char*)m + (off - a0), (size_t)nbytes);
            munmap(m, (size_t)(off - a0 + nbytes));
            return true;
        }
    }
    long got = 0;
    while (got < nbytes) {
        ssize_t k = pread(fd, dest + got, (size_t)(nbytes - got), off + got);
        if (k <= 0) return false;
        got += k;
    }
    return true;
}

}  // namespace lfdhost

extern "C" int lfd_fits_load_frame(const char* path, void* dest, int height, int width, const char* const* keys,
                                   int nkeys, char* values)
{
    using namespace lfdhost;
    if (!path || !dest || height < 1 || width < 1 || nkeys < 0 || (nkeys > 0 && (!keys || !values))) return LFD_E_ARG;
    Fd f(path);
    if (f.fd < 0) return LFD_E_ARG;
    std::vector<Card> cards;
    long off = 0;
    for (int hdu = 0; hdu < 64; hdu++) {
        off = read_header(f.fd, off, cards);
        if (off < 0) return LFD_E_UNSUPPORTED;
        const long nbytes = data_bytes(cards);
        if (nbytes < 0) return LFD_E_UNSUPPORTED;
        if (nbytes == 0) continue;                       // like fitsio.read: the first HDU that has data
        long bitpix = 0, naxis = 0, n1 = 0, n2 = 0;
        if (!card_int(cards, "BITPIX", &bitpix) || !card_int(cards, "NAXIS", &naxis) || bitpix != -32 || naxis != 2) return LFD_E_UNSUPPORTED;
        if (!card_int(cards, "NAXIS1", &n1) || !card_int(cards, "NAXIS2", &n2) || n1 != width || n2 != height) return LFD_E_UNSUPPORTED;
        // scaled images (BSCALE != 1 or BZERO != 0): the Python reader applies the scaling; the trivial cards many
        // writers emit (BSCALE = 1, BZERO = 0) are plain payload
        {
            double bs = 1.0, bz = 0.0;
            if (find(cards, "BSCALE") && !card_num(cards, "BSCALE", &bs)) return LFD_E_UNSUPPORTED;
            if (find(cards, "BZERO") && !card_num(cards, "BZERO", &bz)) return LFD_E_UNSUPPORTED;
            if (bs != 1.0 || bz != 0.0) return LFD_E_UNSUPPORTED;
        }
        // the caller's slot holds exactly height * width 4-byte pixels: a header that claims more (PCOUNT / GCOUNT) is not
        // the plain layout
        if (nbytes != (long)height * (long)width * 4) return LFD_E_UNSUPPORTED;
        for (int k = 0; k < nkeys; k++) {
            const Card* c = find(cards, keys[k]);
            if (!c) return LFD_E_UNSUPPORTED;            // the Python path raises the KeyError the reference would
            memcpy(values + (size_t)k * 72, c->value, 71);
        }
        return read_payload(f.fd, off, nbytes, (char*)dest) ? LFD_OK : LFD_E_ARG;
    }
    return LFD_E_UNSUPPORTED;
}

extern "C" int lfd_catalog_rects(const char* path, int band, int height, int width, double cap, double maxmagdiff,
                                 double magcount, double pixscale, long long defaultxy, double maxxy, int32_t* rects,
                                 int max_rects, int* n_rects)
{
    using namespace lfdhost;
    if (!path || !rects || !n_rects || band < 0 || band > 4 || height < 1 || width < 1 || max_rects < 0) return LFD_E_ARG;
    if (!(pixscale > 0.0) || !isfinite(pixscale)) return LFD_E_UNSUPPORTED;
    Fd f(path);
    if (f.fd < 0) return LFD_E_ARG;
    std::vector<Card> cards;
    long off = 0;
    for (int hdu = 0; hdu < 64; hdu++) {
        off = read_header(f.fd, off, cards);
        if (off < 0) return LFD_E_UNSUPPORTED;
        const long nbytes = data_bytes(cards);
        if (nbytes < 0) return LFD_E_UNSUPPORTED;
        if (nbytes == 0) continue;
        std::string xt;
        if (!card_str(cards, "XTENSION", &xt) || xt != "BINTABLE") return LFD_E_UNSUPPORTED;
        long rowbytes = 0, nrows = 0, tfields = 0;
        if (!card_int(cards, "NAXIS1", &rowbytes) || !card_int(cards, "NAXIS2", &nrows) || !card_int(cards, "TFIELDS", &tfields)) return LFD_E_UNSUPPORTED;
        // byte offset of every column; the six on the path must have exactly the photoObj formats (5E / J)
        static const char* want[6] = {"ROWC", "COLC", "PSFMAG", "PETROTH90", "NOBSERVE", "NDETECT"};
        long offs[6] = {-1, -1, -1, -1, -1, -1};
        long pos = 0;
        for (long i = 1; i <= tfields; i++) {
            char k[32];
            std::string name, form;
            snprintf(k, sizeof k, "TTYPE%ld", i);
            if (!card_str(cards, k, &name)) return LFD_E_UNSUPPORTED;
            snprintf(k, sizeof k, "TFORM%ld", i);
            if (!card_str(cards, k, &form)) return LFD_E_UNSUPPORTED;
            const char* p = form.c_str();
            char* end = nullptr;
            long rep = strtol(p, &end, 10);
            if (end == p) rep = 1;
            const char code = *end;
            long sz;
            switch (code) {
                case 'L': case 'B': case 'A': sz = 1; break;
                case 'I': sz = 2; break;
                case 'J': case 'E': sz = 4; break;
                case 'K': case 'D': sz = 8; break;
                default: return LFD_E_UNSUPPORTED;       // bit arrays, complex, variable-length: not in the reader's set either
            }
            for (int c = 0; c < 6; c++) {
                if (name == want[c]) {
                    const bool ok = c < 4 ? (code == 'E' && rep == 5) : (code == 'J' && rep == 1);
                    if (!ok) return LFD_E_UNSUPPORTED;
                    offs[c] = pos;
                }
            }
            pos += rep * sz;
        }
        if (pos != rowbytes) return LFD_E_UNSUPPORTED;
        for (int c = 0; c < 6; c++) if (offs[c] < 0) return LFD_E_UNSUPPORTED;
        if (nrows * rowbytes > nbytes) return LFD_E_UNSUPPORTED;
        std::vector<unsigned char> tab((size_t)(nrows * rowbytes));
        long got = 0;
        while (got < (long)tab.size()) {
            ssize_t k = pread(f.fd, tab.data() + got, tab.size() - (size_t)got, off + got);
            if (k <= 0) return LFD_E_ARG;
            got += k;
        }
        // first pass: math.ceil of every band of the four float columns must be defined (removestars.py:113-130)
        for (long r = 0; r < nrows; r++) {
            const unsigned char* row = tab.data() + r * rowbytes;
            for (int c = 0; c < 4; c++)
                for (int b = 0; b < 5; b++)
                    if (!isfinite(be_f32(row + offs[c] + 4 * b))) return LFD_E_UNSUPPORTED;   // Python raises ValueError / OverflowError
        }
        const long H = height, W = width;
        int n = 0;
        for (long r = 0; r < nrows; r++) {
            const unsigned char* row = tab.data() + r * rowbytes;
            long long mags[5];
            for (int b = 0; b < 5; b++) mags[b] = (long long)ceil((double)be_f32(row + offs[2] + 4 * b));
            if (!((double)mags[band] < cap)) continue;                                       // :216
            int big = 0;
            for (int j = 0; j < 5; j++)
                for (int k = j + 1; k < 5; k++)
                    big += (double)llabs(mags[j] - mags[k]) > maxmagdiff;                    // :217-224
            if (!(magcount >= (double)big)) continue;
            if (be_i32(row + offs[4]) != be_i32(row + offs[5])) continue;                    // :230
            const long long x = (long long)ceil((double)be_f32(row + offs[1] + 4 * band));   // COLC -> axis 0 (sic, :231)
            const long long y = (long long)ceil((double)be_f32(row + offs[0] + 4 * band));   // ROWC -> axis 1
            const long long p90 = (long long)ceil((double)be_f32(row + offs[3] + 4 * band));
            long long dxy = defaultxy;
            if (p90 > 0) dxy = (long long)((double)p90 / pixscale) + 10;                     // :225-227, int() truncation
            if ((double)dxy > maxxy) dxy = defaultxy;                                        // :228-229
            const long r0 = resolve((long)(x - dxy), H), r1 = resolve((long)(x + dxy), H);
            const long c0 = resolve((long)(y - dxy), W), c1 = resolve((long)(y + dxy), W);
            if (!(r0 < r1 && c0 < c1)) continue;
            if (n >= max_rects) return LFD_E_CAPACITY;
            rects[4 * n + 0] = (int32_t)r0; rects[4 * n + 1] = (int32_t)r1;
            rects[4 * n + 2] = (int32_t)c0; rects[4 * n + 3] = (int32_t)c1;
            n++;
        }
        *n_rects = n;
        return LFD_OK;
    }
    return LFD_E_UNSUPPORTED;
}


// ---------------------------------------------------------------------------------------------------------------------
// lfd_ingest_batch: the two readers above for a whole batch of frames, on a pool of native threads.
// One call per GPU batch replaces 2 x n interpreter round trips of the drop-in driver (lfd_b200/detecttrails.py): the
// caller hands over the n frame / photoObj paths, the frames land in consecutive slots of `staging` (the handle's pinned
// host buffer: slot i = staging + i * height * width * 4 bytes) as raw big-endian payload, the blot rectangles in
// rects[i * max_rects ..], the header cards of the results line in values[(i * nkeys + k) * 72].  Every item reports its
// own status (LFD_OK, or the code that makes the caller take its general reader for THAT item only), so one odd file
// does not slow the batch down.  Work items (n frame reads, n catalog reads) are claimed from one atomic counter;
// the frame reads are what takes time (12.2 MB each from the page cache), so they are claimed first.
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int lfd_ingest_batch(void* staging, int height, int width, int n, const char* const* frame_paths,
                                const char* const* cat_paths, const int32_t* bands, const double* filter_caps,
                                double maxmagdiff, double magcount, double pixscale, long long defaultxy, double maxxy,
                                const char* const* keys, int nkeys, char* values, int32_t* rects, int max_rects,
                                int32_t* n_rects, int32_t* status_frame, int32_t* status_cat, int nthreads)
{
    if (!staging || n < 0 || !frame_paths || !cat_paths || !bands || !filter_caps || !rects || !n_rects || !status_frame ||
        !status_cat || height < 1 || width < 1 || max_rects < 0 || nkeys < 0 || (nkeys > 0 && (!keys || !values))) return LFD_E_ARG;
    if (n == 0) return LFD_OK;
    const size_t slot_bytes = (size_t)height * (size_t)width * 4;
    std::atomic<int> next(0);
    auto work = [&]() {
        for (;;) {
            const int t = next.fetch_add(1, std::memory_order_relaxed);
            if (t >= 2 * n) return;
            // nothing may propagate out of a worker thread (std::terminate): an item that throws (out of memory while
            // reading a table) is reported like any other item the caller has to read itself
            if (t < n) {
                const int i = t;
                try {
                    status_frame[i] = frame_paths[i] ? lfd_fits_load_frame(frame_paths[i], (char*)staging + (size_t)i * slot_bytes, height,
                                                                             width, keys, nkeys, values + (size_t)i * nkeys * 72)
                                                     : LFD_E_ARG;
                } catch (...) { status_frame[i] = LFD_E_ARG; }
            } else {
                const int i = t - n;
                n_rects[i] = 0;
                const int b = bands[i];
                try {
                    status_cat[i] = (cat_paths[i] && b >= 0 && b <= 4)
                                        ? lfd_catalog_rects(cat_paths[i], b, height, width, filter_caps[b], maxmagdiff, magcount, pixscale,
                                                            defaultxy, maxxy, rects + (size_t)i * max_rects * 4, max_rects, &n_rects[i])
                                        : LFD_E_ARG;
                } catch (...) { status_cat[i] = LFD_E_ARG; n_rects[i] = 0; }
            }
        }
    };
    int nt = nthreads > 0 ? nthreads : (int)std::thread::hardware_concurrency();
    if (nt < 1) nt = 1;
    if (nt > 2 * n) nt = 2 * n;
    if (nt > 64) nt = 64;
    std::vector<std::thread> pool;
    try {
        pool.reserve(nt - 1);
        for (int k = 1; k < nt; k++) pool.emplace_back(work);
    } catch (...) {
        // could not start (all of) the helpers: the calling thread and whoever did start finish the items
    }
    work();
    for (auto& th : pool) th.join();
    return LFD_OK;
}
