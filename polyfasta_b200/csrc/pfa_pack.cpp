// Host side of the ingest (north_star "FASTA ingest: ... encoded into a 2-bit-per-base packed alignment ... in pinned
// host memory"): one row of text -> 4 bases per byte, for the column chunks the CPU packs while the copy engine ships
// other chunks as raw text (pfa_ingest.cu).  This is data movement, not a CPU fallback of the scans: the packed rows
// are transposed into the site-major bit-planes on the GPU (pfa_encode_packed_kernel) and everything is counted there.
//
// Code of a base: t = (byte >> 1) & 3  ->  A 0, C 1, T 2, G 3 (upper or lower case: bit 5 is not looked at); base j
// of a byte sits at bits 2j..2j+1.  A row that holds anything but A/C/G/T/a/c/g/t is reported as dirty and the chunk
// travels as text instead (gaps, N, IUPAC codes need the validity plane and the exception list of K1).
#include <immintrin.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <atomic>
#include <thread>
#include <vector>

#include "pfa_host.h"

namespace {

struct Lut {
    uint8_t code[256];  // 0..3, or 0xff for a byte that is not A/C/G/T in either case
    Lut() {
        memset(code, 0xff, sizeof code);
        const char* up = "ACTG";
        for (int i = 0; i < 4; ++i) {
            code[(uint8_t)up[i]] = (uint8_t)i;
            code[(uint8_t)(up[i] | 0x20)] = (uint8_t)i;
        }
    }
};
const Lut g_lut;

int pack_scalar(const uint8_t* src, int64_t cols, uint8_t* dst) {
    unsigned bad = 0;
    int64_t i = 0;
    for (; i + 4 <= cols; i += 4) {
        const unsigned a = g_lut.code[src[i]], b = g_lut.code[src[i + 1]], c = g_lut.code[src[i + 2]], d = g_lut.code[src[i + 3]];
        bad |= a | b | c | d;
        dst[i >> 2] = (uint8_t)((a & 3) | ((b & 3) << 2) | ((c & 3) << 4) | ((d & 3) << 6));
    }
    if (i < cols) {
        unsigned x = 0;
        for (int j = 0; i + j < cols; ++j) {
            const unsigned a = g_lut.code[src[i + j]];
            bad |= a;
            x |= (a & 3) << (2 * j);
        }
        dst[i >> 2] = (uint8_t)x;
    }
    return (bad & 0x80) ? 1 : 0;
}

__attribute__((target("avx2"))) int pack_avx2(const uint8_t* src, int64_t cols, uint8_t* dst) {
    const __m256i three = _mm256_set1_epi8(3), fold = _mm256_set1_epi8((char)0xdf);
    // the upper-case letter each code must come from: A C T G (repeated per 128-bit lane)
    const __m256i letters = _mm256_setr_epi8('A', 'C', 'T', 'G', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 'A', 'C', 'T', 'G', 0, 0, 0, 0, 0, 0,
                                             0, 0, 0, 0, 0, 0);
    const __m256i w14 = _mm256_set1_epi16(0x0401), w116 = _mm256_set1_epi32(0x00100001);
    const __m256i gather = _mm256_setr_epi8(0, 4, 8, 12, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, -1, 0, 4, 8, 12, -1, -1, -1, -1, -1,
                                            -1, -1, -1, -1, -1, -1, -1);
    __m256i ok = _mm256_set1_epi8((char)0xff);
    int64_t i = 0;
    for (; i + 32 <= cols; i += 32) {
        const __m256i x = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(src + i));
        const __m256i code = _mm256_and_si256(_mm256_srli_epi16(x, 1), three);
        ok = _mm256_and_si256(ok, _mm256_cmpeq_epi8(_mm256_shuffle_epi8(letters, code), _mm256_and_si256(x, fold)));
        const __m256i n16 = _mm256_maddubs_epi16(code, w14);   // c0 + 4 c1 per 16-bit lane
        const __m256i n32 = _mm256_madd_epi16(n16, w116);      // + 16 (c2 + 4 c3) per 32-bit lane
        const __m256i b = _mm256_shuffle_epi8(n32, gather);    // low byte of every lane
        const uint32_t lo = (uint32_t)_mm256_extract_epi32(b, 0), hi = (uint32_t)_mm256_extract_epi32(b, 4);
        memcpy(dst + (i >> 2), &lo, 4);
        memcpy(dst + (i >> 2) + 4, &hi, 4);
    }
    int dirty = _mm256_movemask_epi8(ok) != -1;
    if (i < cols) dirty |= pack_scalar(src + i, cols - i, dst + (i >> 2));
    return dirty;
}

__attribute__((target("avx512f,avx512bw,avx512vl"))) int pack_avx512(const uint8_t* src, int64_t cols, uint8_t* dst) {
    const __m512i three = _mm512_set1_epi8(3), fold = _mm512_set1_epi8((char)0xdf);
    const __m512i letters = _mm512_broadcast_i32x4(_mm_setr_epi8('A', 'C', 'T', 'G', 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0));
    const __m512i w14 = _mm512_set1_epi16(0x0401), w116 = _mm512_set1_epi32(0x00100001);
    __mmask64 ok = ~0ull;
    int64_t i = 0;
    for (; i + 128 <= cols; i += 128) {  // two vectors per iteration: independent chains
        const __m512i x0 = _mm512_loadu_si512(src + i), x1 = _mm512_loadu_si512(src + i + 64);
        const __m512i c0 = _mm512_and_si512(_mm512_srli_epi16(x0, 1), three), c1 = _mm512_and_si512(_mm512_srli_epi16(x1, 1), three);
        ok &= _mm512_cmpeq_epi8_mask(_mm512_shuffle_epi8(letters, c0), _mm512_and_si512(x0, fold));
        ok &= _mm512_cmpeq_epi8_mask(_mm512_shuffle_epi8(letters, c1), _mm512_and_si512(x1, fold));
        const __m128i p0 = _mm512_cvtepi32_epi8(_mm512_madd_epi16(_mm512_maddubs_epi16(c0, w14), w116));
        const __m128i p1 = _mm512_cvtepi32_epi8(_mm512_madd_epi16(_mm512_maddubs_epi16(c1, w14), w116));
        _mm_storeu_si128(reinterpret_cast<__m128i*>(dst + (i >> 2)), p0);
        _mm_storeu_si128(reinterpret_cast<__m128i*>(dst + (i >> 2) + 16), p1);
    }
    for (; i + 64 <= cols; i += 64) {
        const __m512i x0 = _mm512_loadu_si512(src + i);
        const __m512i c0 = _mm512_and_si512(_mm512_srli_epi16(x0, 1), three);
        ok &= _mm512_cmpeq_epi8_mask(_mm512_shuffle_epi8(letters, c0), _mm512_and_si512(x0, fold));
        _mm_storeu_si128(reinterpret_cast<__m128i*>(dst + (i >> 2)),
                         _mm512_cvtepi32_epi8(_mm512_madd_epi16(_mm512_maddubs_epi16(c0, w14), w116)));
    }
    int dirty = ok != ~0ull;
    if (i < cols) dirty |= pack_scalar(src + i, cols - i, dst + (i >> 2));
    return dirty;
}

// ---- packer with a validity bitmap: gaps, N and ? travel packed too -------------------------------------------------------
// codes as the planes want them (A 0, C 1, G 2, T 3; '-' 0, 'N' 1, '?' 2 with validity 0), one validity BIT per base
// (bit s%8 of byte s/8).  Return value: bit 0 = the row holds '-', 'N' or '?', bit 1 = it holds any other byte (the chunk
// is dirty and travels as text: the exception list of K1 keeps the identity of such symbols).
struct Lut7 {
    alignas(64) uint8_t t[128];  // bits 0-1 code, bit 2 valid, bit 7 unknown symbol
    Lut7() {
        memset(t, 0x83, sizeof t);
        const char* b = "ACGT";
        for (int i = 0; i < 4; ++i) t[(uint8_t)b[i]] = t[(uint8_t)(b[i] | 0x20)] = (uint8_t)(4 | i);
        t[(uint8_t)'-'] = 0;
        t[(uint8_t)'N'] = t[(uint8_t)'n'] = 1;
        t[(uint8_t)'?'] = 2;
    }
};
const Lut7 g_lut7;

int pack3_scalar(const uint8_t* src, int64_t cols, uint8_t* codes, uint8_t* valid) {
    unsigned bad = 0, inval = 0;
    for (int64_t i = 0; i < cols; i += 8) {
        unsigned v = 0, c01 = 0, c23 = 0;
        const int lim = (int)std::min<int64_t>(8, cols - i);
        for (int j = 0; j < lim; ++j) {
            const unsigned x = src[i + j];
            const unsigned r = (x & 0x80) ? 0x83u : g_lut7.t[x];
            bad |= r;
            v |= ((r >> 2) & 1u) << j;
            if (j < 4) c01 |= (r & 3u) << (2 * j);
            else c23 |= (r & 3u) << (2 * (j - 4));
        }
        inval |= ~v & ((1u << lim) - 1u);
        valid[i >> 3] = (uint8_t)v;
        codes[i >> 2] = (uint8_t)c01;
        if (lim > 4) codes[(i >> 2) + 1] = (uint8_t)c23;
    }
    return ((bad & 0x80) ? 2 : 0) | (inval ? 1 : 0);
}

__attribute__((target("avx512f,avx512bw,avx512vl,avx512vbmi"))) int pack3_vbmi(const uint8_t* src, int64_t cols, uint8_t* codes,
                                                                                uint8_t* valid) {
    const __m512i lo = _mm512_load_si512(g_lut7.t), hi = _mm512_load_si512(g_lut7.t + 64);
    const __m512i three = _mm512_set1_epi8(3), four = _mm512_set1_epi8(4);
    const __m512i w14 = _mm512_set1_epi16(0x0401), w116 = _mm512_set1_epi32(0x00100001);
    __mmask64 bad = 0, inval = 0;
    int64_t i = 0;
    for (; i + 64 <= cols; i += 64) {
        const __m512i x = _mm512_loadu_si512(src + i);
        const __m512i r = _mm512_permutex2var_epi8(lo, x, hi);  // 128-entry table: bits 0-6 of the byte select the entry
        bad |= _mm512_movepi8_mask(r) | _mm512_movepi8_mask(x);  // unknown symbol, or a byte >= 0x80 (bit 7 is not looked up)
        const __mmask64 v = _mm512_test_epi8_mask(r, four);
        inval |= ~v;
        memcpy(valid + (i >> 3), &v, 8);
        const __m512i c = _mm512_and_si512(r, three);
        _mm_storeu_si128(reinterpret_cast<__m128i*>(codes + (i >> 2)),
                         _mm512_cvtepi32_epi8(_mm512_madd_epi16(_mm512_maddubs_epi16(c, w14), w116)));
    }
    int flags = (bad ? 2 : 0) | (inval ? 1 : 0);
    if (i < cols) flags |= pack3_scalar(src + i, cols - i, codes + (i >> 2), valid + (i >> 3));
    return flags;
}

bool have_vbmi() {
    __builtin_cpu_init();
    return __builtin_cpu_supports("avx512vbmi") && __builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl");
}
const bool g_vbmi = have_vbmi();

typedef int (*pack_fn)(const uint8_t*, int64_t, uint8_t*);

pack_fn choose() {
    __builtin_cpu_init();
    if (__builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl")) return pack_avx512;
    if (__builtin_cpu_supports("avx2")) return pack_avx2;
    return pack_scalar;
}
const pack_fn g_pack = choose();

}  // namespace

int pfa_pack2_row(const uint8_t* src, int64_t cols, uint8_t* dst) { return g_pack(src, cols, dst); }
bool pfa_pack3_fast() { return g_vbmi; }
int pfa_pack3_row(const uint8_t* src, int64_t cols, uint8_t* codes, uint8_t* valid) {
    return g_vbmi ? pack3_vbmi(src, cols, codes, valid) : pack3_scalar(src, cols, codes, valid);
}

extern "C" int pfa_host_pack3(const uint8_t* src, int64_t cols, uint8_t* codes, uint8_t* valid, int variant) {
    if (!src || !codes || !valid || cols < 0) return -1;
    if (variant == 1) return pack3_scalar(src, cols, codes, valid);
    if (variant == 4) return g_vbmi ? pack3_vbmi(src, cols, codes, valid) : -2;
    return pfa_pack3_row(src, cols, codes, valid);
}

extern "C" int pfa_host_pack2(const uint8_t* src, int64_t cols, uint8_t* dst, int variant) {
    if (!src || !dst || cols < 0) return -1;
    switch (variant) {
        case 1: return pack_scalar(src, cols, dst);
        case 2: return __builtin_cpu_supports("avx2") ? pack_avx2(src, cols, dst) : -2;
        case 3: return (__builtin_cpu_supports("avx512bw") && __builtin_cpu_supports("avx512vl")) ? pack_avx512(src, cols, dst) : -2;
        default: return g_pack(src, cols, dst);
    }
}

// rows [0, n) of a text matrix, packed with `threads` host threads (row blocks handed out dynamically); returns the number
// of dirty rows
extern "C" int64_t pfa_host_pack2_rows(const uint8_t* text, int64_t n, int64_t cols, int64_t ld, uint8_t* dst, int64_t ldp, int threads) {
    if (!text || !dst || n < 0 || cols < 0 || ld < cols || ldp < (cols + 3) / 4) return -1;
    if (threads < 1) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    std::atomic<int64_t> next(0), dirty(0);
    const int64_t block = 16;
    auto work = [&]() {
        int64_t d = 0;
        for (;;) {
            const int64_t r0 = next.fetch_add(block);
            if (r0 >= n) break;
            const int64_t r1 = std::min(n, r0 + block);
            for (int64_t r = r0; r < r1; ++r) d += g_pack(text + r * ld, cols, dst + r * ldp);
        }
        dirty += d;
    };
    if (threads == 1) {
        work();
    } else {
        std::vector<std::thread> th;
        for (int t = 0; t < threads; ++t) th.emplace_back(work);
        for (auto& t : th) t.join();
    }
    return dirty.load();
}
