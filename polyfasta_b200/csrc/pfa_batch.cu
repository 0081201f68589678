// Batched path for many small loci (the reference's --dir loop, PolyFastA.py:93-94,104): instead of one upload, three
// launches and several synchronisations PER FILE, a batch of loci is copied to the GPU as one pinned blob and processed by
// three segmented launches -- K1b encode, K2b site scan, K5b finalise -- with ONE synchronisation.  A locus keeps its own
// shape (n, L), populations and result slots; kernels find the locus of a tile / site group by binary search in a prefix
// table.  The arithmetic is the same device code as the single-alignment kernels (pfa_sites.cuh, pfa_finalize.cu).
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <cstdlib>
#include <cstring>
#include <new>
#include <thread>

#include "pfa_batch.cuh"
#include "pfa_host.h"
#include "pfa_sites.cuh"

// one locus as added on the host; the device layout (PfaLocusDesc / PfaPopSlot) is derived from these in pfa_batch_run
struct PfaBatchEntry {
    long long text_off = 0;
    int n = 0, L = 0, ld = 0, Wq = 0, k = 0;
    bool synthetic = false;  // the text is written on the device by the synthetic generator (benchmarks): nothing to upload
    uint64_t seed = 0;
    uint32_t p_seg_ppm = 0, tri_ppm = 0;
    std::vector<uint32_t> masks;    // [k][4*Wq]
    std::vector<long long> pop_n;   // [k]
};

// result buffer in pinned host memory (the device-to-host copies of a scan run asynchronously at full PCIe speed; into
// pageable vectors each of them was a staged, blocking copy: ~0.1 ms per batch of 2,500 loci)
template <typename T>
struct PfaPinned {
    T* p = nullptr;
    size_t cap = 0, n = 0;
    bool assign(size_t count, const T& v) {  // false: out of pinned memory
        if (count > cap) {
            if (p) cudaFreeHost(p);
            p = nullptr;
            cap = 0;
            const size_t want = std::max<size_t>(count + count / 4, 1024);
            if (cudaHostAlloc(reinterpret_cast<void**>(&p), want * sizeof(T), cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
            cap = want;
        }
        n = count;
        std::fill(p, p + count, v);
        return true;
    }
    // room for `count` elements, contents unspecified (about to be overwritten by a device-to-host copy): zero-filling
    // 4 MB of pinned results per 10,000-locus scan was 0.4 ms, as long as the scan kernel itself
    bool resize(size_t count) {
        if (count > cap && !assign(count, T())) return false;
        n = count;
        return true;
    }
    T* data() { return p; }
    const T* data() const { return p; }
    T& operator[](size_t i) { return p[i]; }
    const T& operator[](size_t i) const { return p[i]; }
    void release() {
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = n = 0;
    }
};

struct pfa_batch {
    pfa_ctx* ctx = nullptr;
    std::vector<PfaBatchEntry> entries;
    std::vector<PfaLocusDesc> desc;
    std::vector<PfaPopSlot> pops;
    std::vector<uint32_t> masks;  // per locus: k masks then the union, each 4*Wq words
    unsigned char* h_text = nullptr;  // pinned
    size_t h_text_cap = 0, h_text_used = 0;
    size_t synth_bytes = 0;  // device-only text of synthetic loci, laid out after the host text (host loci must be added first)
    long long n_sites = 0, n_tiles = 0, plane_u4 = 0, mask_u4 = 0, out_len = 0;
    int max_Wq = 0;
    long long n_ctiles = 0;
    // results (host)
    PfaPinned<int64_t> out;
    PfaPinned<pfa_final_out> fin;
    PfaPinned<int64_t> cds_out;         // [pops][PFA_CDS_LEN] (codon scan)
    PfaPinned<double> cds_ssites;       // [pops]
    PfaPinned<pfa_final_out> cds_fin;   // [pops][2]: synonymous, nonsynonymous
    bool ran = false, ran_cds = false;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};  // around K2b and around K4b of the last scan
    float site_ms = 0.f, cds_ms = 0.f;
    // device state between pfa_batch_stage and pfa_batch_release: the encoded planes of the whole batch and everything the
    // segmented kernels read
    struct Dev {
        uint8_t* text = nullptr;
        PfaLocusDesc* desc = nullptr;
        PfaPopSlot* pops = nullptr;
        long long *site_base = nullptr, *tile_base = nullptr, *ctile_base = nullptr, *out = nullptr, *cds_out = nullptr, *popn = nullptr;
        uint4 *planes = nullptr, *masks = nullptr;
        int* inv = nullptr;
        unsigned long long *count = nullptr, *keys = nullptr;
        pfa_final_in* fin_in = nullptr;
        pfa_final_out* fin_out = nullptr;
        double* ssites = nullptr;
        int64_t* heads = nullptr;
        int64_t n_heads = 0;
        unsigned long long n_exc = 0;
        size_t plane_bytes = 0;
        int any_invalid = 0;  // some locus of the batch holds a symbol outside A, C, G, T (count[1], read back with the exception count)
        bool staged = false;
    } dev;
};

static int grow_text(pfa_batch* b, size_t need) {
    if (need <= b->h_text_cap) return PFA_OK;
    size_t cap = std::max<size_t>(need, std::max<size_t>(b->h_text_cap * 2, 64u << 20));
    unsigned char* p = nullptr;
    if (cudaHostAlloc(&p, cap, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return pfa_fail(b->ctx, PFA_ERR_NOMEM, "cannot pin %zu bytes", cap);
    }
    if (b->h_text_used) memcpy(p, b->h_text, b->h_text_used);
    if (b->h_text) cudaFreeHost(b->h_text);
    b->h_text = p;
    b->h_text_cap = cap;
    return PFA_OK;
}

static inline int wq_of(int64_t n) {
    int wq = (int)((n + 127) / 128);
    if (wq >= 16 && (wq & 1)) wq++;
    return wq;
}

// ---- kernels ---------------------------------------------------------------------------------------------------

__device__ __forceinline__ unsigned pfa_classify_byte(unsigned c) {
    if (c >= 'a' && c <= 'z') c -= 32;
    switch (c) {
        case 'A': return 4 | 0;
        case 'C': return 4 | 1;
        case 'G': return 4 | 2;
        case 'T': return 4 | 3;
        case '-': return 0;
        case 'N': return 1;
        case '?': return 2;
        default: return 8 | 3;
    }
}

// K1b: one warp = 32 rows x 32 sites of one locus (see pfa_encode_kernel)
__global__ void __launch_bounds__(256) pfa_batch_encode_kernel(const uint8_t* __restrict__ text, const PfaLocusDesc* __restrict__ desc,
                                                               const long long* __restrict__ tile_base, int nloci, long long n_tiles,
                                                               uint32_t* __restrict__ b0, uint32_t* __restrict__ b1, uint32_t* __restrict__ v,
                                                               unsigned long long* __restrict__ exc_keys, unsigned long long* __restrict__ exc_count,
                                                               long long exc_cap, int* __restrict__ locus_invalid) {
    __shared__ uint8_t lut[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = (uint8_t)pfa_classify_byte(i);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long tile = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (tile >= n_tiles) return;
    const int li = pfa_find_locus(tile_base, nloci, tile);
    const PfaLocusDesc d = desc[li];
    const long long t = tile - d.tile_base;
    const int sgs = (d.L + 31) / 32;
    const int w = (int)(t / sgs);
    const long long c0 = (t % sgs) * 32;
    const long long row = (long long)w * 32 + lane;
    const bool live = row < d.n;
    uint32_t bytes[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) bytes[i] = 0x2d2d2d2du;
    if (live) {
        const uint8_t* src = text + d.text_off + row * d.ld + c0;
        if (c0 + 32 <= d.L) {
            const uint4* s4 = reinterpret_cast<const uint4*>(src);
            const uint4 a = __ldg(s4), b = __ldg(s4 + 1);
            bytes[0] = a.x; bytes[1] = a.y; bytes[2] = a.z; bytes[3] = a.w;
            bytes[4] = b.x; bytes[5] = b.y; bytes[6] = b.z; bytes[7] = b.w;
        } else {
            const int lim = (int)(d.L - c0);
            for (int i = 0; i < lim; ++i) {
                const uint32_t c = src[i];
                bytes[i >> 2] = (bytes[i >> 2] & ~(0xffu << (8 * (i & 3)))) | (c << (8 * (i & 3)));
            }
        }
    }
    uint32_t my0 = 0, my1 = 0, myv = 0;
    bool any_invalid = false;
#pragma unroll
    for (int s = 0; s < 32; ++s) {
        const unsigned c = (bytes[s >> 2] >> (8 * (s & 3))) & 0xffu;
        const unsigned code = live ? lut[c] : 0u;
        const uint32_t w0 = __ballot_sync(0xffffffffu, code & 1u);
        const uint32_t w1 = __ballot_sync(0xffffffffu, code & 2u);
        const uint32_t wv = __ballot_sync(0xffffffffu, code & 4u);
        if (lane == s) { my0 = w0; my1 = w1; myv = wv; }
        const bool in_range = c0 + s < d.L;
        if (live && in_range && !(code & 4u)) any_invalid = true;
        if (live && in_range && (code & 8u)) {
            const unsigned up = (c >= 'a' && c <= 'z') ? c - 32 : c;
            const unsigned long long slot = atomicAdd(exc_count, 1ull);
            if ((long long)slot < exc_cap)
                exc_keys[slot] = ((unsigned long long)(d.site_base + c0 + s) << 32) | ((unsigned long long)up << 24) | (unsigned long long)row;
        }
    }
    if (__any_sync(0xffffffffu, any_invalid) && lane == 0) {
        atomicOr(locus_invalid + li, 1);
        if (exc_count[1] == 0ull) atomicOr(exc_count + 1, 1ull);  // exc_count[1]: the batch holds a locus with invalid rows
    }
    if (c0 + lane < d.L) {
        const long long o = (d.plane_off + (c0 + lane) * d.Wq) * 4 + w;
        b0[o] = my0; b1[o] = my1; v[o] = myv;
    }
}

// pass 2 of one site of one locus on registers (class counts per population, group-reduced; the group's first lane books the
// variable columns into the batch result vector)
template <int LPS, int ITER>
__device__ __forceinline__ void pfa_batch_site_pass2(const PfaBatchArgs& a, const PfaLocusDesc& d, const uint4 (&x0)[ITER], const uint4 (&x1)[ITER],
                                                     const uint4 (&xv)[ITER], int sub, unsigned gmask) {
    const int Wq = d.Wq;
    for (int q = 0; q < d.k; ++q) {
        uint32_t c[PFA_NCLASS];
#pragma unroll
        for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
        const uint4* mq = a.masks + d.mask_off + (long long)q * Wq;
#pragma unroll
        for (int i = 0; i < ITER; ++i) {
            const int j = sub + LPS * i;
            const uint4 m4 = j < Wq ? __ldg(mq + j) : make_uint4(0, 0, 0, 0);
            const uint32_t mm[4] = {m4.x, m4.y, m4.z, m4.w}, w0[4] = {x0[i].x, x0[i].y, x0[i].z, x0[i].w},
                           w1[4] = {x1[i].x, x1[i].y, x1[i].z, x1[i].w}, wv[4] = {xv[i].x, xv[i].y, xv[i].z, xv[i].w};
#pragma unroll
            for (int w = 0; w < 4; ++w) {
                const uint32_t vm = wv[w] & mm[w];
                const uint32_t hi = vm & w1[w], lo = vm & ~w1[w];
                c[PFA_C_T] += __popc(hi & w0[w]);
                c[PFA_C_G] += __popc(hi & ~w0[w]);
                c[PFA_C_C] += __popc(lo & w0[w]);
                c[PFA_C_A] += __popc(lo & ~w0[w]);
                const uint32_t im = ~wv[w] & mm[w];
                const uint32_t ihi = im & w1[w];
                c[PFA_C_ESC] += __popc(ihi & w0[w]);
                c[PFA_C_Q] += __popc(ihi & ~w0[w]);
                c[PFA_C_N] += __popc(im & ~w1[w] & w0[w]);
            }
        }
        if (LPS > 1) {
#pragma unroll
            for (int i = 0; i < PFA_NCLASS; ++i) c[i] = pfa_group_add<LPS>(c[i], gmask);
        }
        if (sub != 0) continue;
        const PfaPopSlot ps = a.pops[d.pop_base + q];
        const PfaSiteResult r = pfa_site_result(c, ps.n, 0u, 0ull);
        if (r.has_escape || !r.isvar) continue;
        unsigned long long* o = reinterpret_cast<unsigned long long*>(a.out + ps.out_off);
        atomicAdd(o, 1ull);
        atomicAdd(o + 1, r.h);
        if (r.sfs_bin >= 0) atomicAdd(o + 2 + r.sfs_bin, 1ull);
    }
}

// second pass of the first `count` (<= 32) entries of a warp's queue (q: [PFA_BQ_WORDS][64] words), one lane each; a function of
// its own so that its registers do not weigh on the streaming loop
#define PFA_BQ_WORDS 13
__device__ __noinline__ void pfa_batch_drain(const PfaBatchArgs& a, const uint32_t* q, int count, int lane) {
    __syncwarp();
    const unsigned act = __ballot_sync(0xffffffffu, lane < count);
    if (lane < count) {
        uint4 y0[1], y1[1], yv[1];
        y0[0] = make_uint4(q[0 * 64 + lane], q[1 * 64 + lane], q[2 * 64 + lane], q[3 * 64 + lane]);
        y1[0] = make_uint4(q[4 * 64 + lane], q[5 * 64 + lane], q[6 * 64 + lane], q[7 * 64 + lane]);
        yv[0] = make_uint4(q[8 * 64 + lane], q[9 * 64 + lane], q[10 * 64 + lane], q[11 * 64 + lane]);
        const int li = (int)q[12 * 64 + lane];
        const PfaLocusDesc dq = a.desc[li];
        if (__match_any_sync(act, li) == act) {
            // the waiting sites are neighbours and nearly always belong to ONE locus: the lanes add up S and H (n <= 128 rows:
            // H of a site < 2^15) and one lane books them -- two atomics per population instead of two per site on the same
            // two words
            for (int p = 0; p < dq.k; ++p) {
                const uint4 m4 = __ldg(a.masks + dq.mask_off + p);
                const uint32_t mm[4] = {m4.x, m4.y, m4.z, m4.w}, w0[4] = {y0[0].x, y0[0].y, y0[0].z, y0[0].w},
                               w1[4] = {y1[0].x, y1[0].y, y1[0].z, y1[0].w}, wv[4] = {yv[0].x, yv[0].y, yv[0].z, yv[0].w};
                uint32_t c[PFA_NCLASS];
#pragma unroll
                for (int i = 0; i < PFA_NCLASS; ++i) c[i] = 0;
#pragma unroll
                for (int w = 0; w < 4; ++w) {
                    const uint32_t vm = wv[w] & mm[w];
                    const uint32_t hi = vm & w1[w], lo = vm & ~w1[w];
                    c[PFA_C_T] += __popc(hi & w0[w]);
                    c[PFA_C_G] += __popc(hi & ~w0[w]);
                    c[PFA_C_C] += __popc(lo & w0[w]);
                    c[PFA_C_A] += __popc(lo & ~w0[w]);
                    const uint32_t im = ~wv[w] & mm[w];
                    const uint32_t ihi = im & w1[w];
                    c[PFA_C_ESC] += __popc(ihi & w0[w]);
                    c[PFA_C_Q] += __popc(ihi & ~w0[w]);
                    c[PFA_C_N] += __popc(im & ~w1[w] & w0[w]);
                }
                const PfaPopSlot ps = a.pops[dq.pop_base + p];
                const PfaSiteResult r = pfa_site_result(c, ps.n, 0u, 0ull);
                const bool ok = !r.has_escape && r.isvar;
                const unsigned nS = (unsigned)__popc(__ballot_sync(act, ok));
                const unsigned hsum = __reduce_add_sync(act, ok ? (unsigned)r.h : 0u);
                unsigned long long* o = reinterpret_cast<unsigned long long*>(a.out + ps.out_off);
                if (nS && lane == __ffs(act) - 1) {
                    atomicAdd(o, (unsigned long long)nS);
                    atomicAdd(o + 1, (unsigned long long)hsum);
                }
                if (ok && r.sfs_bin >= 0) atomicAdd(o + 2 + r.sfs_bin, 1ull);
            }
        } else {
            pfa_batch_site_pass2<1, 1>(a, dq, y0, y1, yv, 0, 1u << lane);
        }
    }
    __syncwarp();
}

// K2b: a group of LPS lanes owns one site of one locus; same two passes as pfa_site_scan_reg_kernel, accumulators in global
// memory (only variable columns touch them).  A warp walks CONTIGUOUS chunks of PFA_BATCH_SCHUNK sites, 32 / LPS at a time: its
// loads stay coalesced and the locus of a site is found by one binary search per chunk plus a step forward now and then -- a
// search per site (12 dependent loads for 2,500 loci) held this kernel at 1.3 TB/s on the C5 shape.
// Records of one chunk handled by one lane (n <= 128 rows: LPS = ITER = 1, every lane of a warp its own site -- the shape of
// C1, C2 and C5): with 5 % of the sites variable, four passes out of five met one or two of them and the warp ran the whole
// second pass for those one or two lanes.  Here the variable sites go to a per-warp queue in shared memory (the 12 words of
// the record + the locus) and the second pass runs when 32 are waiting: one lane each, all lanes busy.
#define PFA_BATCH_SCHUNK 2048
template <int LPS, int ITER>
__global__ void __launch_bounds__(PFA_SITE_THREADS, (LPS == 1 && ITER == 1) ? 3 : 1) pfa_batch_site_kernel(const PfaBatchArgs a) {
    constexpr bool QUEUE = LPS == 1 && ITER == 1;
    __shared__ uint32_t sq[QUEUE ? PFA_SITE_THREADS / 32 : 1][QUEUE ? PFA_BQ_WORDS : 1][64];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int sub = lane & (LPS - 1);
    const unsigned gmask = LPS == 32 ? 0xffffffffu : (((1u << LPS) - 1u) << (lane - sub));
    constexpr int GW = 32 / LPS;
    int qn = 0;  // entries waiting in this warp's queue (QUEUE)
    auto drain = [&](int count) { pfa_batch_drain(a, &sq[wib][0][0], count, lane); };
    const long long nchunks = (a.n_sites + PFA_BATCH_SCHUNK - 1) / PFA_BATCH_SCHUNK;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long ch = warp0; ch < nchunks; ch += nwarps) {
      const long long g_lo = ch * PFA_BATCH_SCHUNK, g_hi = min(a.n_sites, g_lo + PFA_BATCH_SCHUNK);
      int li = pfa_find_locus(a.site_base, a.nloci, min(g_lo + lane / LPS, a.n_sites - 1));
      PfaLocusDesc d = a.desc[li];
      long long next_base = a.site_base[li + 1];
      if (QUEUE) {
        // four sites per lane and round: all their loads are issued before the first is looked at (one 16-byte record per
        // plane and site leaves little in flight otherwise: the kernel sat at 2 TB/s)
        constexpr int UN = 2;
        for (long long g0 = g_lo; g0 < g_hi; g0 += 32 * UN) {
            uint4 y0[UN], y1[UN], yv[UN], ym[UN];
            int yl[UN];
            bool act[UN];
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const long long g = g0 + 32 * u + lane;
                act[u] = g < g_hi;
                y0[u] = y1[u] = yv[u] = ym[u] = make_uint4(0, 0, 0, 0);
                yl[u] = li;
                if (act[u]) {
                    if (g >= next_base) {  // walked into a later locus
                        do {
                            ++li;
                            next_base = a.site_base[li + 1];
                        } while (g >= next_base);
                        d = a.desc[li];
                    }
                    yl[u] = li;
                    const long long o = d.plane_off + (g - d.site_base);  // Wq == 1
                    ym[u] = __ldg(a.masks + d.mask_off + d.k);
                    y0[u] = pfa_ld_stream(a.b0 + o);
                    y1[u] = pfa_ld_stream(a.b1 + o);
                    yv[u] = a.locus_invalid[li] ? pfa_ld_stream(a.v + o) : ym[u];
                }
            }
#pragma unroll
            for (int u = 0; u < UN; ++u) {
                const uint4 m = ym[u];
                const uint32_t o0 = (y0[u].x & m.x) | (y0[u].y & m.y) | (y0[u].z & m.z) | (y0[u].w & m.w);
                const uint32_t z0 = (~y0[u].x & m.x) | (~y0[u].y & m.y) | (~y0[u].z & m.z) | (~y0[u].w & m.w);
                const uint32_t o1 = (y1[u].x & m.x) | (y1[u].y & m.y) | (y1[u].z & m.z) | (y1[u].w & m.w);
                const uint32_t z1 = (~y1[u].x & m.x) | (~y1[u].y & m.y) | (~y1[u].z & m.z) | (~y1[u].w & m.w);
                const uint32_t ov = (yv[u].x & m.x) | (yv[u].y & m.y) | (yv[u].z & m.z) | (yv[u].w & m.w);
                const uint32_t zv = (~yv[u].x & m.x) | (~yv[u].y & m.y) | (~yv[u].z & m.z) | (~yv[u].w & m.w);
                const bool mono = !(o0 && z0) && !(o1 && z1) && !(ov && zv);
                const bool all_escape = o0 && o1 && !ov;
                const bool var = act[u] && !(mono && !all_escape);
                const unsigned vm = __ballot_sync(0xffffffffu, var);
                if (!vm) continue;
                if (var) {
                    const int pos = qn + __popc(vm & ((1u << lane) - 1u));
                    sq[wib][0][pos] = y0[u].x; sq[wib][1][pos] = y0[u].y; sq[wib][2][pos] = y0[u].z; sq[wib][3][pos] = y0[u].w;
                    sq[wib][4][pos] = y1[u].x; sq[wib][5][pos] = y1[u].y; sq[wib][6][pos] = y1[u].z; sq[wib][7][pos] = y1[u].w;
                    sq[wib][8][pos] = yv[u].x; sq[wib][9][pos] = yv[u].y; sq[wib][10][pos] = yv[u].z; sq[wib][11][pos] = yv[u].w;
                    sq[wib][12][pos] = (uint32_t)yl[u];
                }
                qn += __popc(vm);
                if (qn >= 32) {
                    drain(32);
                    const int rest = qn - 32;  // move the entries behind the first 32 to the front
                    uint32_t keep[PFA_BQ_WORDS];
                    if (lane < rest)
#pragma unroll
                        for (int w = 0; w < PFA_BQ_WORDS; ++w) keep[w] = sq[wib][w][32 + lane];
                    __syncwarp();
                    if (lane < rest)
#pragma unroll
                        for (int w = 0; w < PFA_BQ_WORDS; ++w) sq[wib][w][lane] = keep[w];
                    qn = rest;
                    __syncwarp();
                }
            }
        }
        continue;
      }
      for (long long g = g_lo + lane / LPS; g < g_hi; g += GW) {
        bool var = false;
        uint4 x0[ITER], x1[ITER], xv[ITER], m[ITER];
        {
            if (g >= next_base) {  // the group has walked into a later locus
                do {
                    ++li;
                    next_base = a.site_base[li + 1];
                } while (g >= next_base);
                d = a.desc[li];
            }
            const long long s = g - d.site_base;
            const int Wq = d.Wq;
            const bool hv = a.locus_invalid[li] != 0;
            const uint4* um = a.masks + d.mask_off + (long long)d.k * Wq;
            const uint4* p0 = a.b0 + d.plane_off + s * Wq;
            const uint4* p1 = a.b1 + d.plane_off + s * Wq;
            const uint4* pv = a.v + d.plane_off + s * Wq;
#pragma unroll
            for (int i = 0; i < ITER; ++i) {
                const int j = sub + LPS * i;
                x0[i] = x1[i] = xv[i] = m[i] = make_uint4(0, 0, 0, 0);
                if (j < Wq) {
                    m[i] = __ldg(um + j);
                    x0[i] = pfa_ld_stream(p0 + j);
                    x1[i] = pfa_ld_stream(p1 + j);
                    xv[i] = hv ? pfa_ld_stream(pv + j) : m[i];
                }
            }
            uint32_t o0 = 0, z0 = 0, o1 = 0, z1 = 0, ov = 0, zv = 0;
#pragma unroll
            for (int i = 0; i < ITER; ++i) {
                o0 |= (x0[i].x & m[i].x) | (x0[i].y & m[i].y) | (x0[i].z & m[i].z) | (x0[i].w & m[i].w);
                z0 |= (~x0[i].x & m[i].x) | (~x0[i].y & m[i].y) | (~x0[i].z & m[i].z) | (~x0[i].w & m[i].w);
                o1 |= (x1[i].x & m[i].x) | (x1[i].y & m[i].y) | (x1[i].z & m[i].z) | (x1[i].w & m[i].w);
                z1 |= (~x1[i].x & m[i].x) | (~x1[i].y & m[i].y) | (~x1[i].z & m[i].z) | (~x1[i].w & m[i].w);
                ov |= (xv[i].x & m[i].x) | (xv[i].y & m[i].y) | (xv[i].z & m[i].z) | (xv[i].w & m[i].w);
                zv |= (~xv[i].x & m[i].x) | (~xv[i].y & m[i].y) | (~xv[i].z & m[i].z) | (~xv[i].w & m[i].w);
            }
            unsigned f = (o0 ? 1u : 0u) | (z0 ? 2u : 0u) | (o1 ? 4u : 0u) | (z1 ? 8u : 0u) | (ov ? 16u : 0u) | (zv ? 32u : 0u);
            f = pfa_group_or<LPS>(f, gmask);
            const bool mono = ((f & 3u) != 3u) && ((f & 12u) != 12u) && ((f & 48u) != 48u);
            const bool all_escape = (f & 1u) && (f & 4u) && !(f & 16u);
            var = !(mono && !all_escape);
        }
        if (var) pfa_batch_site_pass2<LPS, ITER>(a, d, x0, x1, xv, sub, gmask);
      }
    }
    if (QUEUE && qn) drain(qn);
}

// K2b for batches in which EVERY locus fits one 128-row chunk (n <= 128: C1, C2, C5) -- the site records of the whole batch are
// then one contiguous array of 16-byte entries per plane (plane offset == global site number), and the kernel is the site
// scan's TMA design on it: one CTA of 512 threads per SM, every warp owns a shared-memory slot of PFA_BATCH_SLOT consecutive
// sites per plane fed by one cp.async.bulk per plane on the slot's mbarrier, refilled as soon as the last of its sites sits in
// registers.  pfa_batch_site_kernel's per-lane 16-byte loads left 50 KB per SM in flight (3.2 TB/s of padded bytes on the
// C5 shape).  With 16-byte records a slot holds MANY sites and scanning it takes as long as fetching it (one slot per warp:
// 4.7 TB/s), so every warp has two slots: one is scanned while the other is on its way.  HV = some locus of the batch holds a non-ACGT symbol: the validity plane is
// fetched too (for every locus; the planes of a clean locus say "all rows valid").  Lanes walk the loci as before (one
// binary search per slot, done while the slot's bytes are on their way); variable sites go to the warp's queue.
#define PFA_BATCH_SLOT 128     // sites per slot, two planes
#define PFA_BATCH_SLOT_HV 96   // sites per slot, three planes
#define PFA_BATCH_STAGES 2     // slots per warp: one is scanned while the other is on its way
template <bool HV>
__global__ void __launch_bounds__(512, 1) pfa_batch_site_tma_kernel(const PfaBatchArgs a) {
    constexpr int NW = 16, SB = HV ? PFA_BATCH_SLOT_HV : PFA_BATCH_SLOT, NPL = HV ? 3 : 2;
    extern __shared__ __align__(128) unsigned char dyn[];
    constexpr int ST = PFA_BATCH_STAGES;
    constexpr size_t SLOT_BYTES = (size_t)NPL * SB * 16;
    uint64_t* bars = reinterpret_cast<uint64_t*>(dyn + (size_t)NW * ST * SLOT_BYTES);  // [NW][ST]
    uint32_t* sqs = reinterpret_cast<uint32_t*>(bars + NW * ST);                      // [NW][PFA_BQ_WORDS][64]
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        for (int i = 0; i < NW * ST; ++i) pfa_mbar_init(&bars[i], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    unsigned char* ring = dyn + (size_t)wib * ST * SLOT_BYTES;
    uint64_t* bar = bars + wib * ST;
    uint32_t* sq = sqs + (size_t)wib * PFA_BQ_WORDS * 64;
    // every warp scans a CONTIGUOUS range of slots: its lanes walk the loci forward from one slot to the next, with one binary
    // search per warp (a search per slot -- 17 dependent loads -- took longer than the slot's bytes: ncu r2y, long scoreboard
    // 4.5 cycles per issue)
    const long long nblk = (a.n_sites + SB - 1) / SB;
    const long long nw = (long long)gridDim.x * NW, per = (nblk + nw - 1) / nw;
    long long blk = ((long long)blockIdx.x * NW + wib) * per;
    const long long blk_hi = min(nblk, blk + per);
    auto issue = [&](long long bnext, int stage) {  // all lanes
        __syncwarp();             // every lane has consumed its last values of the slot ...
        pfa_fence_proxy_async();  // ... and those generic-proxy reads come before the async-proxy writes of the copies
        if (lane == 0 && bnext < blk_hi) {
            const long long s0 = bnext * SB;
            const unsigned bytes = (unsigned)min((long long)SB, a.n_sites - s0) * 16u;
            unsigned char* dst = ring + (size_t)stage * SLOT_BYTES;
            pfa_mbar_expect_tx(bar + stage, NPL * bytes);
            pfa_bulk_load(dst, a.b0 + s0, bytes, bar + stage);
            pfa_bulk_load(dst + (size_t)SB * 16, a.b1 + s0, bytes, bar + stage);
            if (HV) pfa_bulk_load(dst + (size_t)2 * SB * 16, a.v + s0, bytes, bar + stage);
        }
    };
    int qn = 0;  // entries waiting in this warp's queue
#pragma unroll
    for (int st = 0; st < ST; ++st) issue(blk + st, st);
    // this lane's first site and its locus
    int li = blk < blk_hi ? pfa_find_locus(a.site_base, a.nloci, min(blk * SB + lane, a.n_sites - 1)) : 0;
    PfaLocusDesc d = a.desc[li];
    long long next_base = a.site_base[li + 1];
    uint4 m = __ldg(a.masks + d.mask_off + d.k);  // union of the locus' populations (Wq == 1)
    for (unsigned k = 0; blk < blk_hi; ++k, ++blk) {
        const long long g_lo = blk * SB, g_hi = min(a.n_sites, g_lo + SB);
        const int stage = (int)(k % ST);
        const uint4* slot = reinterpret_cast<const uint4*>(ring + (size_t)stage * SLOT_BYTES);
        pfa_mbar_wait(bar + stage, (k / ST) & 1u);
#pragma unroll 1
        for (int r = 0; r < SB / 32; ++r) {
            const long long g = g_lo + r * 32 + lane;
            const bool act = g < g_hi;
            if (act && g >= next_base) {  // walked into a later locus
                do {
                    ++li;
                    next_base = a.site_base[li + 1];
                } while (g >= next_base);
                d = a.desc[li];
                m = __ldg(a.masks + d.mask_off + d.k);
            }
            // sites beyond the end of the batch read what the slot held before: dropped (act)
            const uint4 y0 = slot[r * 32 + lane], y1 = slot[SB + r * 32 + lane];
            const uint4 yv = HV ? slot[2 * SB + r * 32 + lane] : m;
            const uint32_t o0 = (y0.x & m.x) | (y0.y & m.y) | (y0.z & m.z) | (y0.w & m.w);
            const uint32_t z0 = (~y0.x & m.x) | (~y0.y & m.y) | (~y0.z & m.z) | (~y0.w & m.w);
            const uint32_t o1 = (y1.x & m.x) | (y1.y & m.y) | (y1.z & m.z) | (y1.w & m.w);
            const uint32_t z1 = (~y1.x & m.x) | (~y1.y & m.y) | (~y1.z & m.z) | (~y1.w & m.w);
            const uint32_t ov = (yv.x & m.x) | (yv.y & m.y) | (yv.z & m.z) | (yv.w & m.w);
            const uint32_t zv = (~yv.x & m.x) | (~yv.y & m.y) | (~yv.z & m.z) | (~yv.w & m.w);
            const bool mono = !(o0 && z0) && !(o1 && z1) && !(ov && zv);
            const bool all_escape = o0 && o1 && !ov;
            const bool var = act && !(mono && !all_escape);
            const unsigned vm = __ballot_sync(0xffffffffu, var);  // every lane's record has been looked at
            if (r == SB / 32 - 1) issue(blk + ST, stage);
            if (!vm) continue;
            if (var) {
                const int pos = qn + __popc(vm & ((1u << lane) - 1u));
                sq[0 * 64 + pos] = y0.x; sq[1 * 64 + pos] = y0.y; sq[2 * 64 + pos] = y0.z; sq[3 * 64 + pos] = y0.w;
                sq[4 * 64 + pos] = y1.x; sq[5 * 64 + pos] = y1.y; sq[6 * 64 + pos] = y1.z; sq[7 * 64 + pos] = y1.w;
                sq[8 * 64 + pos] = yv.x; sq[9 * 64 + pos] = yv.y; sq[10 * 64 + pos] = yv.z; sq[11 * 64 + pos] = yv.w;
                sq[12 * 64 + pos] = (uint32_t)li;
            }
            qn += __popc(vm);
            if (qn >= 32) {
                pfa_batch_drain(a, sq, 32, lane);
                const int rest = qn - 32;  // move the entries behind the first 32 to the front
                uint32_t keep[PFA_BQ_WORDS];
                if (lane < rest)
#pragma unroll
                    for (int w = 0; w < PFA_BQ_WORDS; ++w) keep[w] = sq[w * 64 + 32 + lane];
                __syncwarp();
                if (lane < rest)
#pragma unroll
                    for (int w = 0; w < PFA_BQ_WORDS; ++w) sq[w * 64 + lane] = keep[w];
                qn = rest;
                __syncwarp();
            }
        }
    }
    if (qn) pfa_batch_drain(a, sq, qn, lane);
}

// sites with escape symbols: one warp per distinct (global) site of the sorted exception list
__global__ void __launch_bounds__(256) pfa_batch_escape_kernel(const PfaBatchArgs a, const unsigned long long* __restrict__ keys, long long n_exc,
                                                               const long long* __restrict__ heads, long long n_heads) {
    __shared__ unsigned int hist[8][256];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + wib;
    const long long nwarps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long h = wid; h < n_heads; h += nwarps) {
        const long long i0 = heads[h], i1 = (h + 1 < n_heads) ? heads[h + 1] : n_exc;
        const long long g = (long long)(keys[i0] >> 32);
        const int li = pfa_find_locus(a.site_base, a.nloci, g);
        const PfaLocusDesc d = a.desc[li];
        const long long s = g - d.site_base;
        const int Wq = d.Wq;
        for (int q = 0; q < d.k; ++q) {
            const uint4* mq = a.masks + d.mask_off + (long long)q * Wq;
            uint32_t c[PFA_NCLASS];
            pfa_class_counts<true>(a.b0 + d.plane_off + s * Wq, a.b1 + d.plane_off + s * Wq, a.v + d.plane_off + s * Wq, mq, Wq, lane, c);
            if (c[PFA_C_ESC] == 0) continue;
            for (int b = lane; b < 256; b += 32) hist[wib][b] = 0u;
            __syncwarp();
            const uint32_t* mw = reinterpret_cast<const uint32_t*>(mq);
            for (long long i = i0 + lane; i < i1; i += 32) {
                const unsigned long long key = keys[i];
                const uint32_t row = (uint32_t)(key & 0xffffffull);
                if ((mw[row >> 5] >> (row & 31)) & 1u) atomicAdd(&hist[wib][(key >> 24) & 0xffu], 1u);
            }
            __syncwarp();
            uint32_t distinct = 0;
            unsigned long long sq = 0;
            for (int b = lane; b < 256; b += 32) {
                const unsigned long long cnt = hist[wib][b];
                distinct += cnt ? 1u : 0u;
                sq += cnt * cnt;
            }
            for (int off = 16; off; off >>= 1) {
                distinct += __shfl_xor_sync(0xffffffffu, distinct, off);
                sq += __shfl_xor_sync(0xffffffffu, sq, off);
            }
            __syncwarp();
            if (lane != 0) continue;
            const PfaPopSlot ps = a.pops[d.pop_base + q];
            const PfaSiteResult r = pfa_site_result(c, ps.n, distinct, sq);
            if (!r.isvar) continue;
            unsigned long long* o = reinterpret_cast<unsigned long long*>(a.out + ps.out_off);
            atomicAdd(o, 1ull);
            atomicAdd(o + 1, r.h);
            if (r.sfs_bin >= 0) atomicAdd(o + 2 + r.sfs_bin, 1ull);
        }
    }
}

// K5b input straight from the device result vector: no host round trip between the scan and the finalisation
__global__ void pfa_batch_final_in_kernel(const PfaPopSlot* __restrict__ pops, const long long* __restrict__ out, int jc, long long n_pops,
                                          pfa_final_in* __restrict__ fin_in) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pops) return;
    const PfaPopSlot p = pops[i];
    pfa_final_in f;
    f.n = p.n;
    f.S = out[p.out_off];
    f.H = out[p.out_off + 1];
    f.seqlen = p.seqlen;
    f.jc = jc;
    f.pad = 0;
    fin_in[i] = f;
}


// ---- host --------------------------------------------------------------------------------------------------------

extern "C" {

int64_t pfa_mask_words_for(int64_t n) { return (int64_t)wq_of(n) * 4; }

int pfa_batch_create(pfa_ctx* ctx, pfa_batch** out) {
    if (!ctx || !out) return PFA_ERR_ARG;
    pfa_batch* b = new (std::nothrow) pfa_batch();
    if (!b) return PFA_ERR_NOMEM;
    b->ctx = ctx;
    *out = b;
    return PFA_OK;
}

int pfa_batch_clear(pfa_batch* b) {
    if (!b) return PFA_ERR_ARG;
    b->entries.clear();
    b->h_text_used = 0;
    b->synth_bytes = 0;
    b->ran = b->ran_cds = false;
    pfa_batch_release(b);
    return PFA_OK;
}

int pfa_batch_release(pfa_batch* b);

int pfa_batch_destroy(pfa_batch* b) {
    if (!b) return PFA_OK;
    pfa_batch_release(b);
    for (auto& e : b->ev) if (e) cudaEventDestroy(e);
    b->out.release(); b->fin.release(); b->cds_out.release(); b->cds_ssites.release(); b->cds_fin.release();
    if (b->h_text) cudaFreeHost(b->h_text);
    delete b;
    return PFA_OK;
}

int64_t pfa_batch_size(const pfa_batch* b) { return b ? (int64_t)b->entries.size() : 0; }
int64_t pfa_batch_text_bytes(const pfa_batch* b) { return b ? (int64_t)b->h_text_used : 0; }

}  // extern "C"

// trims the masks to n rows, counts the populations; false when one is empty
static bool entry_set_masks(PfaBatchEntry* e, const uint32_t* masks, int k) {
    const int64_t Wn = (int64_t)e->Wq * 4, n = e->n;
    e->k = k > 0 ? k : 1;
    e->masks.assign((size_t)(e->k * Wn), 0u);
    e->pop_n.assign((size_t)e->k, 0);
    for (int q = 0; q < e->k; ++q) {
        long long cnt = 0;
        for (int64_t w = 0; w < Wn; ++w) {
            uint32_t x = k > 0 ? masks[q * Wn + w] : 0xffffffffu;
            const int64_t lo = w * 32;
            if (lo >= n) x = 0;
            else if (lo + 32 > n) x &= (1u << (n - lo)) - 1u;
            e->masks[(size_t)(q * Wn + w)] = x;
            cnt += __builtin_popcount(x);
        }
        if (cnt == 0) return false;
        e->pop_n[(size_t)q] = cnt;
    }
    return true;
}

// device layout of the current entries
static void build_layout(pfa_batch* b) {
    b->desc.clear();
    b->pops.clear();
    b->masks.clear();
    b->n_sites = b->n_tiles = b->plane_u4 = b->mask_u4 = b->out_len = b->n_ctiles = 0;
    b->max_Wq = 0;
    for (size_t i = 0; i < b->entries.size(); ++i) {
        const PfaBatchEntry& e = b->entries[i];
        PfaLocusDesc d;
        d.text_off = e.text_off;
        d.plane_off = b->plane_u4;
        d.mask_off = b->mask_u4;
        d.site_base = b->n_sites;
        d.tile_base = b->n_tiles;
        d.pop_base = (long long)b->pops.size();
        d.n = e.n; d.L = e.L; d.ld = e.ld; d.Wq = e.Wq; d.k = e.k; d.pad = 0;
        const int64_t Wn = (int64_t)e.Wq * 4;
        const size_t m0 = b->masks.size();
        b->masks.resize(m0 + (size_t)((e.k + 1) * Wn), 0u);
        memcpy(b->masks.data() + m0, e.masks.data(), sizeof(uint32_t) * (size_t)(e.k * Wn));
        uint32_t* uni = b->masks.data() + m0 + (size_t)e.k * Wn;
        for (int q = 0; q < e.k; ++q) {
            for (int64_t w = 0; w < Wn; ++w) uni[w] |= e.masks[(size_t)(q * Wn + w)];
            PfaPopSlot ps;
            ps.n = e.pop_n[(size_t)q];
            ps.out_off = b->out_len;
            ps.locus = (long long)i;
            ps.seqlen = (double)e.L;
            b->pops.push_back(ps);
            b->out_len += 2 + ps.n / 2;
        }
        b->plane_u4 += (long long)e.L * e.Wq;
        b->mask_u4 += (long long)(e.k + 1) * e.Wq;
        b->n_sites += e.L;
        b->n_tiles += (long long)((e.n + 31) / 32) * ((e.L + 31) / 32);
        b->max_Wq = std::max(b->max_Wq, e.Wq);
        b->desc.push_back(d);
    }
}

#define PFA_BATCH_MAX_WQ 128

extern "C" {

int pfa_batch_add_rows(pfa_batch* b, const uint8_t* text, int64_t n, int64_t L, int64_t ld, const uint32_t* masks, int k, int64_t* index) {
    if (!b || n <= 0 || L < 0 || (L > 0 && (!text || ld < L)) || k < 0 || (k > 0 && !masks)) return PFA_ERR_ARG;
    if (L >= (1ll << 31) || wq_of(n) > PFA_BATCH_MAX_WQ) return pfa_fail(b->ctx, PFA_ERR_ARG, "locus too large for the batched path");
    if (b->synth_bytes) return pfa_fail(b->ctx, PFA_ERR_ARG, "host loci must be added before synthetic ones");
    PfaBatchEntry e;
    e.n = (int)n;
    e.L = (int)L;
    e.ld = (int)pfa_round_up(std::max<int64_t>(L, 1), 32);
    e.Wq = wq_of(n);
    if (!entry_set_masks(&e, masks, k)) return pfa_fail(b->ctx, PFA_ERR_ARG, "empty population in batch");
    e.text_off = (long long)pfa_round_up((int64_t)b->h_text_used, 256);
    const size_t need = (size_t)e.text_off + (size_t)n * e.ld;
    int rc = grow_text(b, need);
    if (rc) return rc;
    for (int64_t r = 0; r < n; ++r) memcpy(b->h_text + e.text_off + r * e.ld, text + r * ld, (size_t)L);
    b->h_text_used = need;
    if (index) *index = (int64_t)b->entries.size();
    b->entries.push_back(std::move(e));
    b->ran = false;
    return PFA_OK;
}

/* a locus of the synthetic generator (pfa_aln_synthetic's alignment, all columns): its text is produced on the device when the
 * batch is staged, so that benchmarks can hold many loci resident without 1 byte per base of host memory */
int pfa_batch_add_synthetic(pfa_batch* b, int64_t n, int64_t L, uint64_t seed, uint32_t p_seg_ppm, uint32_t tri_ppm, const uint32_t* masks, int k,
                            int64_t* index) {
    if (!b || n <= 0 || L < 0 || k < 0 || (k > 0 && !masks)) return PFA_ERR_ARG;
    if (L >= (1ll << 31) || wq_of(n) > PFA_BATCH_MAX_WQ) return pfa_fail(b->ctx, PFA_ERR_ARG, "locus too large for the batched path");
    PfaBatchEntry e;
    e.n = (int)n;
    e.L = (int)L;
    e.ld = (int)pfa_round_up(std::max<int64_t>(L, 1), 32);
    e.Wq = wq_of(n);
    e.synthetic = true;
    e.seed = seed;
    e.p_seg_ppm = p_seg_ppm;
    e.tri_ppm = tri_ppm;
    if (!entry_set_masks(&e, masks, k)) return pfa_fail(b->ctx, PFA_ERR_ARG, "empty population in batch");
    // synthetic loci occupy the device blob only: their offsets continue after the host text
    e.text_off = (long long)pfa_round_up((int64_t)(b->h_text_used + b->synth_bytes), 256);
    b->synth_bytes = (size_t)e.text_off + (size_t)n * e.ld - b->h_text_used;
    if (index) *index = (int64_t)b->entries.size();
    b->entries.push_back(std::move(e));
    b->ran = false;
    return PFA_OK;
}

int pfa_batch_add(pfa_batch* b, const pfa_fasta* f, const uint32_t* masks, int k, int64_t* index) {
    if (!b || !f) return PFA_ERR_ARG;
    if (f->seqlen < 0) return pfa_fail(b->ctx, PFA_ERR_RAGGED, "sequences do not have the same length");
    if (f->in_place) {  // a large file whose rows are slices of the file buffer: gather them into a matrix first (rare here)
        std::vector<uint8_t> mat((size_t)std::max<int64_t>(f->n * f->seqlen, 1));
        for (int64_t r = 0; r < f->n; ++r) {
            const uint8_t* src = f->data + f->row_off[(size_t)r];
            if (!f->wrap_w.empty() && f->wrap_w[(size_t)r] > 0)
                pfa_gather_wrapped(src, f->wrap_w[(size_t)r], f->wrap_gap[(size_t)r], 0, f->seqlen, mat.data() + r * f->seqlen);
            else
                memcpy(mat.data() + r * f->seqlen, src, (size_t)f->seqlen);
        }
        return pfa_batch_add_rows(b, mat.data(), f->n, f->seqlen, std::max<int64_t>(f->seqlen, 1), masks, k, index);
    }
    return pfa_batch_add_rows(b, f->data, f->n, f->seqlen, std::max<int64_t>(f->seqlen, 1), masks, k, index);
}

// --dir in one native call: read, parse (reference semantics), split by header-substring keys and append `count` files with
// `threads` host threads; rows are copied straight into the pinned blob.  Per file: status[i] (PFA_OK, PFA_ERR_NOT_FASTA,
// PFA_ERR_RAGGED, PFA_ERR_IO, PFA_ERR_NON_ASCII, or PFA_BATCH_TOO_BIG = not added, use the single-alignment path),
// shape[2i] = n, shape[2i+1] = L, locus[i] = its index in the batch or -1, hits[i*max(nkeys,1) + j] = rows matching key j
// (populations without a match are not added; with nkeys = 0 the one population is all rows).
int pfa_batch_add_files(pfa_batch* b, const char* const* paths, int count, const char* const* keys, int nkeys, int threads, int* status,
                        int64_t* shape, int64_t* locus, int64_t* hits) {
    if (!b || count < 0 || nkeys < 0 || (count > 0 && (!paths || !status || !shape || !locus || !hits)) || (nkeys > 0 && !keys))
        return PFA_ERR_ARG;
    if (count == 0) return PFA_OK;
    if (b->synth_bytes) return pfa_fail(b->ctx, PFA_ERR_ARG, "host loci must be added before synthetic ones");
    // size the blob once: the rows of a file never need more than its size plus the padding of every row to 32 bytes
    std::vector<size_t> fsize((size_t)count, 0);
    size_t bound = (size_t)pfa_round_up((int64_t)b->h_text_used, 256);
    for (int i = 0; i < count; ++i) {
        struct stat st;
        if (stat(paths[i], &st) == 0 && !S_ISDIR(st.st_mode)) fsize[(size_t)i] = (size_t)st.st_size;
        bound += fsize[(size_t)i] + fsize[(size_t)i] / 8 + 4096;
    }
    int rc = grow_text(b, bound);
    if (rc) return rc;
    if (threads < 1) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    threads = std::min(threads, count);
    const int nk = std::max(nkeys, 1);
    std::vector<PfaBatchEntry> slots((size_t)count);
    std::atomic<size_t> cursor((size_t)pfa_round_up((int64_t)b->h_text_used, 256));
    std::vector<size_t> klen((size_t)nkeys);
    for (int j = 0; j < nkeys; ++j) klen[(size_t)j] = strlen(keys[j]);
    // files whose padded rows did not fit the estimate (many short rows: every row is padded to 32 bytes) are staged in a
    // second round, after the blob has grown by their exact need
    std::vector<int> todo((size_t)count), deferred;
    for (int i = 0; i < count; ++i) todo[(size_t)i] = i;
    std::vector<char> overflow((size_t)count, 0);
    auto work = [&](int t) {
        std::vector<unsigned char> buf;
        PfaParsed parsed;
        for (size_t ii = (size_t)t; ii < todo.size(); ii += (size_t)threads) {
            const int i = todo[ii];
            locus[i] = -1;
            shape[2 * i] = shape[2 * i + 1] = 0;
            for (int j = 0; j < nk; ++j) hits[(size_t)i * nk + j] = 0;
            size_t len = 0;
            int st = pfa_read_file(paths[i], &buf, &len);
            if (!st) st = pfa_parse_lines(buf.data(), len, &parsed);
            if (st) { status[i] = st; continue; }
            const int64_t n = (int64_t)parsed.recs.size(), L = parsed.seqlen;
            shape[2 * i] = n;
            shape[2 * i + 1] = L;
            if (L < 0) { status[i] = PFA_ERR_RAGGED; continue; }
            PfaBatchEntry& e = slots[(size_t)i];
            e.n = (int)n; e.L = (int)L; e.Wq = wq_of(n);
            e.ld = (int)pfa_round_up(std::max<int64_t>(L, 1), 32);
            // populations: header substring match per key (PolyFastA.py:125), empty ones dropped
            const int64_t Wn = (int64_t)e.Wq * 4;
            std::vector<uint32_t> m;
            int kfound = 0;
            if (nkeys == 0) {
                hits[(size_t)i * nk] = n;
            } else {
                for (int j = 0; j < nkeys; ++j) {
                    std::vector<uint32_t> mj((size_t)Wn, 0u);
                    int64_t h = 0;
                    for (int64_t r = 0; r < n; ++r) {
                        const std::string& hd = parsed.recs[(size_t)r].header;
                        if (klen[(size_t)j] == 0 || (hd.size() >= klen[(size_t)j] && memmem(hd.data(), hd.size(), keys[j], klen[(size_t)j]))) {
                            mj[(size_t)(r >> 5)] |= 1u << (r & 31);
                            ++h;
                        }
                    }
                    hits[(size_t)i * nk + j] = h;
                    if (h) { m.insert(m.end(), mj.begin(), mj.end()); ++kfound; }
                }
                if (kfound == 0) { status[i] = PFA_OK; continue; }   // nothing to compute: every key prints its note
            }
            if (n >= (1ll << 24) || L >= (1ll << 31) || e.Wq > PFA_BATCH_MAX_WQ || (size_t)n * (size_t)e.ld > (64u << 20)) {
                status[i] = PFA_BATCH_TOO_BIG;
                continue;
            }
            const size_t need = (size_t)pfa_round_up((int64_t)((size_t)n * e.ld), 256);
            const size_t off = cursor.fetch_add(need);
            if (off + need > b->h_text_cap) {
                status[i] = PFA_BATCH_TOO_BIG;
                overflow[(size_t)i] = 1;
                continue;
            }
            bool ascii = true;
            for (int64_t r = 0; r < n; ++r) ascii &= pfa_copy_record(parsed.recs[(size_t)r], b->h_text + off + (size_t)r * e.ld);
            if (!ascii) { status[i] = PFA_ERR_NON_ASCII; continue; }
            e.text_off = (long long)off;
            entry_set_masks(&e, nkeys ? m.data() : nullptr, nkeys ? kfound : 0);
            locus[i] = 0;  // placeholder: numbered in file order below
            status[i] = PFA_OK;
        }
    };
    auto run_round = [&]() {
        const int nt = (int)std::min<size_t>((size_t)threads, todo.size());
        if (nt <= 1) {
            const int keep = threads;
            threads = 1;
            work(0);
            threads = keep;
        } else {
            const int keep = threads;
            threads = nt;
            std::vector<std::thread> th;
            for (int t = 0; t < nt; ++t) th.emplace_back(work, t);
            for (auto& x : th) x.join();
            threads = keep;
        }
    };
    run_round();
    size_t extra = 0;
    for (int i = 0; i < count; ++i)
        if (overflow[(size_t)i]) {
            deferred.push_back(i);
            extra += (size_t)pfa_round_up(shape[2 * i] * pfa_round_up(std::max<int64_t>(shape[2 * i + 1], 1), 32), 256);
        }
    if (!deferred.empty()) {
        // the first round's cursor may have run past the capacity: restart it at the end of what was really written
        size_t used = (size_t)pfa_round_up((int64_t)b->h_text_used, 256);
        for (int i = 0; i < count; ++i)
            if (locus[i] == 0) {
                const PfaBatchEntry& e = slots[(size_t)i];
                used = std::max(used, (size_t)e.text_off + (size_t)pfa_round_up((int64_t)((size_t)e.n * e.ld), 256));
            }
        b->h_text_used = used;  // grow_text copies this much
        rc = grow_text(b, used + extra);
        if (rc) return rc;
        cursor.store(used);
        todo = deferred;
        std::fill(overflow.begin(), overflow.end(), 0);
        run_round();
    }
    b->h_text_used = std::min(cursor.load(), b->h_text_cap);
    for (int i = 0; i < count; ++i)
        if (locus[i] == 0) {
            locus[i] = (int64_t)b->entries.size();
            b->entries.push_back(std::move(slots[(size_t)i]));
        }
    b->ran = false;
    return PFA_OK;
}

static void batch_free_dev(pfa_batch* b) {
    pfa_ctx* ctx = b->ctx;
    pfa_batch::Dev& d = b->dev;
    pfa_dfree(ctx, d.text); pfa_dfree(ctx, d.desc); pfa_dfree(ctx, d.pops); pfa_dfree(ctx, d.site_base); pfa_dfree(ctx, d.tile_base);
    pfa_dfree(ctx, d.ctile_base); pfa_dfree(ctx, d.out); pfa_dfree(ctx, d.cds_out); pfa_dfree(ctx, d.popn); pfa_dfree(ctx, d.planes);
    pfa_dfree(ctx, d.masks); pfa_dfree(ctx, d.inv); pfa_dfree(ctx, d.count); pfa_dfree(ctx, d.keys); pfa_dfree(ctx, d.fin_in);
    pfa_dfree(ctx, d.fin_out); pfa_dfree(ctx, d.ssites); pfa_dfree(ctx, d.heads);
    d = pfa_batch::Dev();
}

int pfa_batch_release(pfa_batch* b) {
    if (!b) return PFA_ERR_ARG;
    if (b->dev.staged) {
        cudaSetDevice(b->ctx->device);
        batch_free_dev(b);
    }
    return PFA_OK;
}

// ONE upload of the pinned blob + K1b: afterwards the planes of every locus of the batch are resident in HBM
int pfa_batch_stage(pfa_batch* b) {
    if (!b) return PFA_ERR_ARG;
    pfa_ctx* ctx = b->ctx;
    if (b->dev.staged) batch_free_dev(b);
    build_layout(b);
    const int nloci = (int)b->desc.size();
    const long long npops = (long long)b->pops.size();
    b->ran = b->ran_cds = false;
    b->dev.staged = true;
    if (nloci == 0) return PFA_OK;
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    std::vector<long long> site_base((size_t)nloci + 1), tile_base((size_t)nloci + 1), ctile_base((size_t)nloci + 1), popn((size_t)npops);
    long long ct = 0;
    for (int i = 0; i < nloci; ++i) {
        const PfaLocusDesc& dd = b->desc[(size_t)i];
        site_base[(size_t)i] = dd.site_base;
        tile_base[(size_t)i] = dd.tile_base;
        ctile_base[(size_t)i] = ct;
        // at least one tile per non-empty locus: it also books the trailing partial codon column
        if (dd.L > 0) ct += std::max<long long>(1, ((long long)(dd.L / 3) + PFA_BATCH_CTILE - 1) / PFA_BATCH_CTILE);
    }
    site_base[(size_t)nloci] = b->n_sites;
    tile_base[(size_t)nloci] = b->n_tiles;
    ctile_base[(size_t)nloci] = ct;
    b->n_ctiles = ct;
    for (long long i = 0; i < npops; ++i) popn[(size_t)i] = b->pops[(size_t)i].n;

    pfa_batch::Dev& d = b->dev;
    d.plane_bytes = (size_t)pfa_round_up(std::max<long long>(b->plane_u4, 1) * 16, 256);
    long long cap = std::max<long long>(1 << 16, (long long)((b->h_text_used + b->synth_bytes) / 64));
    if (b->h_text_used == 0) cap = 1 << 10;  // synthetic loci are pure ACGT
    if (const char* ev = getenv("PFA_BATCH_EXC_CAP")) cap = std::max<long long>(1, atoll(ev));  // tests: force the retry
    int rc = PFA_OK;
    cudaError_t e = cudaSuccess;
#define BR(call)                                                                       \
    do {                                                                               \
        if (e == cudaSuccess) e = (call);                                              \
    } while (0)
    const size_t text_bytes = b->h_text_used + b->synth_bytes;
    BR(pfa_dmalloc(ctx, &d.text, text_bytes));
    BR(pfa_dmalloc(ctx, &d.desc, sizeof(PfaLocusDesc) * (size_t)nloci));
    BR(pfa_dmalloc(ctx, &d.pops, sizeof(PfaPopSlot) * (size_t)npops));
    BR(pfa_dmalloc(ctx, &d.site_base, sizeof(long long) * ((size_t)nloci + 1)));
    BR(pfa_dmalloc(ctx, &d.tile_base, sizeof(long long) * ((size_t)nloci + 1)));
    BR(pfa_dmalloc(ctx, &d.ctile_base, sizeof(long long) * ((size_t)nloci + 1)));
    BR(pfa_dmalloc(ctx, &d.popn, sizeof(long long) * (size_t)npops));
    BR(pfa_dmalloc(ctx, &d.out, sizeof(long long) * (size_t)std::max<long long>(b->out_len, 1)));
    BR(pfa_dmalloc(ctx, &d.planes, 3 * d.plane_bytes));
    BR(pfa_dmalloc(ctx, &d.masks, sizeof(uint32_t) * std::max<size_t>(b->masks.size(), 4)));
    BR(pfa_dmalloc(ctx, &d.inv, sizeof(int) * (size_t)nloci));
    BR(pfa_dmalloc(ctx, &d.count, 2 * sizeof(unsigned long long)));  // [0] exceptions, [1] any locus with invalid rows
    BR(pfa_dmalloc(ctx, &d.keys, sizeof(unsigned long long) * (size_t)cap));
    BR(pfa_dmalloc(ctx, &d.fin_in, sizeof(pfa_final_in) * 2 * (size_t)npops));
    BR(pfa_dmalloc(ctx, &d.fin_out, sizeof(pfa_final_out) * 2 * (size_t)npops));
    BR(cudaMemcpyAsync(d.text, b->h_text, b->h_text_used, cudaMemcpyHostToDevice, st));
    if (e == cudaSuccess && b->synth_bytes)
        for (size_t i = 0; i < b->entries.size() && !rc; ++i) {
            const PfaBatchEntry& en = b->entries[i];
            if (en.synthetic && en.L > 0)
                rc = pfa_synth_text_device(ctx, d.text + en.text_off, en.ld, en.n, en.seed, en.p_seg_ppm, en.tri_ppm, 0, en.L);
        }
    BR(cudaMemcpyAsync(d.desc, b->desc.data(), sizeof(PfaLocusDesc) * (size_t)nloci, cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.pops, b->pops.data(), sizeof(PfaPopSlot) * (size_t)npops, cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.site_base, site_base.data(), sizeof(long long) * ((size_t)nloci + 1), cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.tile_base, tile_base.data(), sizeof(long long) * ((size_t)nloci + 1), cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.ctile_base, ctile_base.data(), sizeof(long long) * ((size_t)nloci + 1), cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.popn, popn.data(), sizeof(long long) * (size_t)npops, cudaMemcpyHostToDevice, st));
    BR(cudaMemcpyAsync(d.masks, b->masks.data(), sizeof(uint32_t) * b->masks.size(), cudaMemcpyHostToDevice, st));
    BR(cudaMemsetAsync(d.planes, 0, 3 * d.plane_bytes, st));
    BR(cudaMemsetAsync(d.inv, 0, sizeof(int) * (size_t)nloci, st));
    BR(cudaMemsetAsync(d.count, 0, 2 * sizeof(unsigned long long), st));
    d.any_invalid = 0;
    if (e == cudaSuccess && b->n_tiles > 0) {
        uint32_t* p0 = reinterpret_cast<uint32_t*>(d.planes);
        uint32_t* p1 = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(d.planes) + d.plane_bytes);
        uint32_t* pv = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(d.planes) + 2 * d.plane_bytes);
        for (int attempt = 0; attempt < 2 && e == cudaSuccess && !rc; ++attempt) {
            pfa_batch_encode_kernel<<<(unsigned)((b->n_tiles + 7) / 8), 256, 0, st>>>(d.text, d.desc, d.tile_base, nloci, b->n_tiles, p0, p1, pv, d.keys,
                                                                                    d.count, cap, d.inv);
            ctx->launches++;
            e = cudaGetLastError();
            // exception list: one small synchronisation per batch
            unsigned long long counts[2] = {0, 0};
            BR(cudaMemcpyAsync(counts, d.count, sizeof(counts), cudaMemcpyDeviceToHost, st));
            BR(cudaStreamSynchronize(st));
            if (e != cudaSuccess) break;
            const unsigned long long count = counts[0];
            d.any_invalid = counts[1] != 0;
            d.n_exc = count;
            if ((long long)count <= cap) break;
            // more symbols outside ACGT-N? than the list was sized for (dense IUPAC codes, '.', '*' ...: every character is an
            // allele in the reference, PolyFastA.py:256-258): encode once more with a list of the exact size
            if (attempt == 1) {
                rc = pfa_fail(ctx, PFA_ERR_CUDA, "batched path: the exception list changed between two encodes");
                break;
            }
            pfa_dfree(ctx, d.keys);
            d.keys = nullptr;
            cap = (long long)count;
            BR(pfa_dmalloc(ctx, &d.keys, sizeof(unsigned long long) * (size_t)cap));
            BR(cudaMemsetAsync(d.count, 0, 2 * sizeof(unsigned long long), st));
        }
        if (e == cudaSuccess && !rc && d.n_exc > 0) rc = pfa_sort_exceptions(ctx, &d.keys, (int64_t)d.n_exc, &d.heads, &d.n_heads);
    }
    // the text has done its duty
    pfa_dfree(ctx, d.text);
    d.text = nullptr;
#undef BR
    if (!rc && e != cudaSuccess) rc = pfa_fail(ctx, PFA_ERR_CUDA, "batched staging failed: %s", cudaGetErrorString(e));
    if (rc) batch_free_dev(b);
    return rc;
}

// per population of the batch: ssites, nsites and the two K5 inputs of the codon scan (PolyFastA.py:167,172-173)
__global__ void pfa_batch_final_in_cds_kernel(const PfaPopSlot* __restrict__ pops, const long long* __restrict__ cds, int jc, long long n_pops,
                                              pfa_final_in* __restrict__ fin_in, double* __restrict__ ssites) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pops) return;
    const PfaPopSlot p = pops[i];
    const long long* row = cds + i * PFA_CDS_LEN;
    double s = 0.0;
    for (int l = 1; l <= 64; ++l)
        if (row[PFA_CDS_SUM3 + l]) s = __dadd_rn(s, __ddiv_rn((double)row[PFA_CDS_SUM3 + l], __dmul_rn(3.0, (double)l)));
    ssites[i] = s;
    const double nsites = __dsub_rn(__dsub_rn(p.seqlen, (double)row[PFA_CDS_MISSING]), s);
    pfa_final_in f;
    f.n = p.n; f.S = row[PFA_CDS_SS]; f.H = row[PFA_CDS_HS]; f.seqlen = s; f.jc = jc; f.pad = 0;
    fin_in[2 * i] = f;
    f.S = row[PFA_CDS_SN]; f.H = row[PFA_CDS_HN]; f.seqlen = nsites;
    fin_in[2 * i + 1] = f;
}

// the segmented scans over the staged planes: K2b (+ escape sites), optionally K4b, K5b, ONE synchronisation
int pfa_batch_scan(pfa_batch* b, int jc, int cds) {
    if (!b || !b->dev.staged) return PFA_ERR_ARG;
    pfa_ctx* ctx = b->ctx;
    pfa_batch::Dev& d = b->dev;
    const int nloci = (int)b->desc.size();
    const long long npops = (long long)b->pops.size();
    // every element of these is written by the copies at the end of the scan (an empty batch has none)
    bool ok = b->out.resize((size_t)b->out_len) && b->fin.resize((size_t)npops);
    b->ran = b->ran_cds = false;  // results become readable when the scan has succeeded
    if (cds) ok = ok && b->cds_out.resize((size_t)npops * PFA_CDS_LEN) && b->cds_ssites.resize((size_t)npops) && b->cds_fin.resize((size_t)npops * 2);
    if (!ok) return pfa_fail(ctx, PFA_ERR_NOMEM, "cannot pin the result buffers of the batch");
    if (nloci == 0) {
        b->ran = true;
        b->ran_cds = cds != 0;
        return PFA_OK;
    }
    PFA_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    int rc = PFA_OK;
    cudaError_t e = cudaSuccess;
#define BR(call)                                                                       \
    do {                                                                               \
        if (e == cudaSuccess) e = (call);                                              \
    } while (0)
    if (cds && !d.cds_out) {
        BR(pfa_dmalloc(ctx, &d.cds_out, sizeof(long long) * (size_t)npops * PFA_CDS_LEN));
        BR(pfa_dmalloc(ctx, &d.ssites, sizeof(double) * (size_t)npops));
    }
    BR(cudaMemsetAsync(d.out, 0, sizeof(long long) * (size_t)std::max<long long>(b->out_len, 1), st));
    if (cds) BR(cudaMemsetAsync(d.cds_out, 0, sizeof(long long) * (size_t)npops * PFA_CDS_LEN, st));
    uint4* p0 = d.planes;
    uint4* p1 = reinterpret_cast<uint4*>(reinterpret_cast<char*>(d.planes) + d.plane_bytes);
    uint4* pv = reinterpret_cast<uint4*>(reinterpret_cast<char*>(d.planes) + 2 * d.plane_bytes);
    PfaBatchArgs args{p0, p1, pv, d.masks, d.desc, d.pops, d.site_base, d.inv, d.out, b->n_sites, nloci, d.ctile_base, b->n_ctiles, d.cds_out, d.popn};
    for (auto& ev : b->ev)
        if (!ev) BR(cudaEventCreate(&ev));
    BR(cudaEventRecord(b->ev[0], st));
    if (e == cudaSuccess && b->n_sites > 0) {
        int lps = 1;
        while (lps < 32 && (b->max_Wq + lps - 1) / lps > 4) lps *= 2;
        const int iter = (b->max_Wq + lps - 1) / lps;
        // every locus in one 128-row chunk: the TMA variant (PFA_BATCH_TMA=0 turns it off, =1 forces it).  Not for small batches:
        // its CTAs take a whole SM's shared memory, and in the --dir loop (chunks of 512 loci, two staging slots per GPU) a
        // scan then waits until the other slot's encode kernel has left the SMs -- 0.2 -> 2.4 ms per scan on average, 24 -> 33 us
        // per locus end to end (the per-lane kernel needs 0.2 ms for such a chunk either way)
        const char* tma_env = getenv("PFA_BATCH_TMA");
        const bool tma = b->max_Wq == 1 && b->plane_u4 == b->n_sites && !(tma_env && atoi(tma_env) == 0) &&
                         (b->n_sites >= ((long long)16 << 20) || (tma_env && atoi(tma_env) == 1));
        if (tma) {
            const bool hv = d.any_invalid != 0;
            const int sb = hv ? PFA_BATCH_SLOT_HV : PFA_BATCH_SLOT;
            const size_t dyn = (size_t)16 * PFA_BATCH_STAGES * (hv ? 3 : 2) * sb * 16 + 16 * PFA_BATCH_STAGES * sizeof(uint64_t) + (size_t)16 * PFA_BQ_WORDS * 64 * sizeof(uint32_t);
            const long long nblk = (b->n_sites + sb - 1) / sb;
            const unsigned grid = (unsigned)std::min<long long>(ctx->sm_count, (nblk + 15) / 16);
            if (hv) {
                BR(cudaFuncSetAttribute(pfa_batch_site_tma_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
                if (e == cudaSuccess) pfa_batch_site_tma_kernel<true><<<grid, 512, dyn, st>>>(args);
            } else {
                BR(cudaFuncSetAttribute(pfa_batch_site_tma_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
                if (e == cudaSuccess) pfa_batch_site_tma_kernel<false><<<grid, 512, dyn, st>>>(args);
            }
            pfa_note_kernel(ctx, "pfa_batch_site_tma_kernel<HV=%d> grid=%u block=512 slots=%d sites_per_slot=%d", (int)hv, grid, PFA_BATCH_STAGES, sb);
        } else
        {
        const long long chunks = (b->n_sites + PFA_BATCH_SCHUNK - 1) / PFA_BATCH_SCHUNK;   // one warp per chunk at a time
        long long blocks = (chunks + PFA_SITE_THREADS / 32 - 1) / (PFA_SITE_THREADS / 32);
        blocks = std::min<long long>(std::max<long long>(blocks, 1), (long long)ctx->sm_count * 8);
#define PFA_B_CASE(L_, I_) \
    if (lps == L_ && iter == I_) pfa_batch_site_kernel<L_, I_><<<(unsigned)blocks, PFA_SITE_THREADS, 0, st>>>(args); else
        PFA_B_CASE(1, 1) PFA_B_CASE(1, 2) PFA_B_CASE(1, 3) PFA_B_CASE(1, 4) PFA_B_CASE(2, 3) PFA_B_CASE(2, 4) PFA_B_CASE(4, 3) PFA_B_CASE(4, 4)
        PFA_B_CASE(8, 3) PFA_B_CASE(8, 4) PFA_B_CASE(16, 3) PFA_B_CASE(16, 4) PFA_B_CASE(32, 3) PFA_B_CASE(32, 4)
        rc = pfa_fail(ctx, PFA_ERR_ARG, "batched path: a locus has too many sequences (Wq=%d); use the single-alignment path", b->max_Wq);
#undef PFA_B_CASE
        if (!rc) pfa_note_kernel(ctx, "pfa_batch_site_kernel<LPS=%d,ITER=%d> grid=%u block=%d", lps, iter, (unsigned)blocks, PFA_SITE_THREADS);
        }
        ctx->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess && !rc && d.n_heads > 0) {
            long long eb = std::min<long long>((d.n_heads + 7) / 8, (long long)ctx->sm_count * 8);
            pfa_batch_escape_kernel<<<(unsigned)eb, 256, 0, st>>>(args, d.keys, (long long)d.n_exc, (const long long*)d.heads, d.n_heads);
            ctx->launches++;
            e = cudaGetLastError();
        }
    }
    BR(cudaEventRecord(b->ev[1], st));
    BR(cudaEventRecord(b->ev[2], st));
    if (e == cudaSuccess && !rc && cds)
        rc = pfa_launch_batch_cds(ctx, args, b->max_Wq, d.keys, (long long)d.n_exc, (const long long*)d.heads, d.n_heads);
    BR(cudaEventRecord(b->ev[3], st));
    if (e == cudaSuccess && !rc) {
        pfa_batch_final_in_kernel<<<(unsigned)((npops + 127) / 128), 128, 0, st>>>(d.pops, d.out, jc, npops, d.fin_in);
        ctx->launches++;
        e = cudaGetLastError();
        if (e == cudaSuccess) rc = pfa_launch_finalize(ctx, d.fin_in, d.fin_out, (int)npops);
        if (rc) e = cudaErrorUnknown;
        BR(cudaMemcpyAsync(b->out.data(), d.out, sizeof(long long) * (size_t)b->out_len, cudaMemcpyDeviceToHost, st));
        BR(cudaMemcpyAsync(b->fin.data(), d.fin_out, sizeof(pfa_final_out) * (size_t)npops, cudaMemcpyDeviceToHost, st));
        if (cds && e == cudaSuccess) {
            // the K5 outputs of the site scan are on their way to the host; the same buffers take the codon scan's entries next
            // (stream order keeps the copies ahead of the kernels)
            pfa_batch_final_in_cds_kernel<<<(unsigned)((npops + 127) / 128), 128, 0, st>>>(d.pops, d.cds_out, jc, npops, d.fin_in, d.ssites);
            ctx->launches++;
            e = cudaGetLastError();
            if (e == cudaSuccess) rc = pfa_launch_finalize(ctx, d.fin_in, d.fin_out, (int)(2 * npops));
            if (rc) e = cudaErrorUnknown;
            BR(cudaMemcpyAsync(b->cds_out.data(), d.cds_out, sizeof(long long) * (size_t)npops * PFA_CDS_LEN, cudaMemcpyDeviceToHost, st));
            BR(cudaMemcpyAsync(b->cds_ssites.data(), d.ssites, sizeof(double) * (size_t)npops, cudaMemcpyDeviceToHost, st));
            BR(cudaMemcpyAsync(b->cds_fin.data(), d.fin_out, sizeof(pfa_final_out) * 2 * (size_t)npops, cudaMemcpyDeviceToHost, st));
        }
        BR(cudaStreamSynchronize(st));
        if (e == cudaSuccess) {
            cudaEventElapsedTime(&b->site_ms, b->ev[0], b->ev[1]);
            cudaEventElapsedTime(&b->cds_ms, b->ev[2], b->ev[3]);
        }
    }
#undef BR
    if (rc) return rc;
    if (e != cudaSuccess) return pfa_fail(ctx, PFA_ERR_CUDA, "batched run failed: %s", cudaGetErrorString(e));
    b->ran = true;
    b->ran_cds = cds != 0;
    return PFA_OK;
}

/* device time of the segmented site scan (+ escape sites) and of the codon scan in the last pfa_batch_scan, ms (CUDA events) */
int pfa_batch_kernel_ms(const pfa_batch* b, double* site_ms, double* cds_ms) {
    if (!b) return PFA_ERR_ARG;
    if (site_ms) *site_ms = b->site_ms;
    if (cds_ms) *cds_ms = b->cds_ms;
    return PFA_OK;
}

/* bases (rows x sites summed over the loci) and bytes of the planes of the staged batch */
int pfa_batch_shape(const pfa_batch* b, int64_t* bases, int64_t* plane_bytes) {
    if (!b) return PFA_ERR_ARG;
    int64_t tot = 0;
    for (const auto& e : b->entries) tot += (int64_t)e.n * e.L;
    if (bases) *bases = tot;
    if (plane_bytes) *plane_bytes = (int64_t)b->plane_u4 * 16;
    return PFA_OK;
}

int pfa_batch_run(pfa_batch* b, int jc) {
    if (!b) return PFA_ERR_ARG;
    int rc = pfa_batch_stage(b);
    if (!rc) rc = pfa_batch_scan(b, jc, 0);
    pfa_batch_release(b);
    return rc;
}

int pfa_batch_run_cds(pfa_batch* b, int jc) {
    if (!b) return PFA_ERR_ARG;
    int rc = pfa_batch_stage(b);
    if (!rc) rc = pfa_batch_scan(b, jc, 1);
    pfa_batch_release(b);
    return rc;
}

/* codon-scan result of (locus, pop) after pfa_batch_run_cds / pfa_batch_scan(cds = 1): cds = int64[PFA_CDS_LEN], fin2 = the two K5
 * outputs (synonymous, nonsynonymous) */
int pfa_batch_result_cds(const pfa_batch* b, int64_t locus, int pop, int64_t* cds, double* ssites, void* fin2) {
    if (!b || !b->ran_cds || locus < 0 || locus >= (int64_t)b->desc.size()) return PFA_ERR_ARG;
    const PfaLocusDesc& d = b->desc[(size_t)locus];
    if (pop < 0 || pop >= d.k) return PFA_ERR_ARG;
    const size_t i = (size_t)(d.pop_base + pop);
    if (cds) memcpy(cds, b->cds_out.data() + i * PFA_CDS_LEN, sizeof(int64_t) * PFA_CDS_LEN);
    if (ssites) *ssites = b->cds_ssites[i];
    if (fin2) memcpy(fin2, b->cds_fin.data() + 2 * i, 2 * sizeof(pfa_final_out));
    return PFA_OK;
}

int pfa_batch_num_pops(const pfa_batch* b, int64_t locus) {
    return (b && locus >= 0 && locus < (int64_t)b->entries.size()) ? b->entries[(size_t)locus].k : -1;
}

/* result of (locus, pop): counts[0..2] = n, S, H ; sfs copied when sfs != NULL (n/2 bins); fin = K5 output */
int pfa_batch_result(const pfa_batch* b, int64_t locus, int pop, int64_t counts[3], int64_t* sfs, void* fin) {
    if (!b || !b->ran || locus < 0 || locus >= (int64_t)b->desc.size()) return PFA_ERR_ARG;
    const PfaLocusDesc& d = b->desc[(size_t)locus];
    if (pop < 0 || pop >= d.k) return PFA_ERR_ARG;
    const PfaPopSlot& ps = b->pops[(size_t)(d.pop_base + pop)];
    if (counts) {
        counts[0] = ps.n;
        counts[1] = b->out[(size_t)ps.out_off];
        counts[2] = b->out[(size_t)ps.out_off + 1];
    }
    if (sfs)
        for (long long i = 0; i < ps.n / 2; ++i) sfs[i] = b->out[(size_t)(ps.out_off + 2 + i)];
    if (fin) *static_cast<pfa_final_out*>(fin) = b->fin[(size_t)(d.pop_base + pop)];
    return PFA_OK;
}

}  // extern "C"
